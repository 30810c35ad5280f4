// Internal declarations shared by the host half (csic_params.cpp, csic_plan.cpp, csic_api.cu) and the kernels.
#ifndef CSIC_INTERNAL_H_
#define CSIC_INTERNAL_H_

#include <cstddef>
#include <cstdint>
#include <vector>

#include "../../include/csic.h"

namespace csic {

struct Geometry {
  int32_t out_w, out_h;
  size_t in_row_bytes, in_frame_bytes;
  size_t out_row_bytes, out_frame_bytes;
  int32_t out_px_bytes;      // 3 for YCC888/RGB888, slot bytes (1/2/4) for bundles
  int32_t in_px_bytes;       // 3 (RGB24) or 4 (RGBA32 / BGRA32, fourth byte ignored)
  bool chroma_first;         // ChromaSubsampling precedes SpatialSampling in op1..op3
  bool quant_first;          // ColorQuantization precedes SpatialSampling (only matters for AVERAGE)
  int32_t hf, vf;            // ChromaSubsampler.scala:26-27
  int32_t planar_hs, planar_vs, planar_cw, planar_ch;   // CSIC_OUT_PLANAR chroma decimation / plane size
};

int slot_bits(const csic_params& p);
Geometry geometry(const csic_params& p);

// Kernel-side output format after resolving the bundle slot width.
enum KFormat : int32_t { KF_YCC888 = 0, KF_RGB888 = 1, KF_SLOT8 = 2, KF_SLOT16 = 3, KF_SLOT32 = 4, KF_PLANAR = 5 };

// Everything a kernel needs, passed by value (lives in the constant bank).
struct KPlan {
  const uint8_t* in;
  uint8_t* out;
  uint64_t in_frame_bytes, out_frame_bytes;
  uint32_t in_row_bytes, out_row_bytes;  // row PITCHES in bytes (== dense row size unless the caller pitched the buffers)
  int32_t W, H, Wo, Ho;
  int32_t Wp;                            // row kernel: processing width in output pixels (Wo rounded up to 16)
  int32_t in_dense, out_dense, ragged;   // rows of a tile contiguous in memory (no pitch gap); Wp != Wo
  int32_t in_px_bytes;                   // 3 or 4
  uint32_t coef_y, coef_ncb, coef_ncr;   // dp4a coefficient words in the byte order of the input pixels
  int32_t f;
  int32_t hf, vf, last_sample_col;       // ((W-1)/hf)*hf : last chroma sample column of a line
  int32_t case_b;                        // spatial before chroma with f > 1 (misaligned counters)
  uint32_t caseb_row_add, caseb_col_bytes; // case B: held pixel = decimated-stream element (line-1)*W + last_sample_col
  int32_t quant_first, trunc, average;
  int32_t kformat, slot_bytes, slots_per_row;
  int32_t planar_hs, planar_vs, planar_cw, planar_ch;   // PLANAR: chroma decimation (output px) and plane size
  uint64_t planar_cb_off, planar_cr_off;                 // byte offsets of the Cb / Cr planes inside an output frame
  int32_t sy, scb, scr;                  // 8 - target bits
  int32_t cb_bits, cr_bits;
  int32_t row0, band_rows;               // output rows [row0, row0 + band_rows) of every frame
  int32_t compact;                       // input holds only the rows a DECIMATE pipeline reads (every f-th), densely
  int32_t row_step;                      // input rows between consecutive output rows: f, or 1 when compact
  uint32_t n_frames;
  // ---- TMA row kernel only ----
  int32_t hfe;                           // chroma hold width in *output* pixels inside a 4-pixel granule
  int32_t nsplit, tile_px;               // segments per output row, output pixels per row segment
  int32_t tile_rows;                     // output rows per tile (1 when nsplit > 1)
  uint32_t tiles_per_band;
  uint32_t tile_in_bytes, tile_out_bytes; // bytes of ONE row segment (input / output)
  uint32_t n_tiles;
  int32_t stages;
  int32_t block_threads;
  int32_t ctas_per_sm;
  int32_t ticketed;                      // row kernel: tiles dealt from a per-launch counter (TileDeal, csic_tma.cuh)
  uint32_t* tickets;                     // that counter pair: set per launch by csic_api.cu, one pair per stream
  uint32_t stage_stride, out_buf_off, out_buf_stride, meta_off, bar_off, smem_bytes;
  uint32_t qmask;                        // my | mcb<<8 | mcr<<16 (per-channel keep masks)
  int32_t tall_ho;                       // flex kernel: != 0 -> the batch is addressed as ONE image of n * Ho rows; rows per original frame
#ifdef CSIC_PROBE_WINDOW
  // row kernel drift probe (tools/rows_window_probe.py), null when off: n_tiles records {%globaltimer when the producer
  // takes the tile, CTA}, indexed by tile, then one record per CTA: {%globaltimer when it is done, 2^32 | CTA}
  uint64_t* probe;
#endif
};

// Constants shared by the planners (csic_plan.cpp) and the kernels.
constexpr uint32_t kRingBarBytes = 16;      // mbarrier bytes per stage of a TMA-staged kernel's ring (Ring, csic_tma.cuh)
constexpr int kDefaultBlockThreads = 256;   // row kernel: consumer threads; one producer warp is added at launch
constexpr int kMaxConsumerThreads = 512;
constexpr int kMaxTileRows = 64;        // rows per tile of the row kernel (small frames: 64 rows x 384 B still make a 24 KB tile; 256 rows
                                        // measured worse on 32x32 and 64x64 frames: the producer's per-row work, profiles/r2/rows_tall.txt)
constexpr uint32_t kTileMetaBytes = 32 + 4 * kMaxTileRows;   // sizeof(TileMeta) in csic_rows_kernel.cu
constexpr int kPoolMaxRows = 16;        // output rows per tile of the pooling kernel (each carries f input rows)
constexpr uint32_t kPoolMetaBytes = 32 + 4 * kPoolMaxRows;   // sizeof(PoolMeta) in csic_pool_kernel.cu
constexpr int kFlexMaxRows = 64;        // rows per tile of the flex kernel: the producer's lanes take two rows each
constexpr int kFlexConsumers = 256;                  // flex kernel default: 8 consumer warps (+ 1 producer warp)
constexpr int kFlexMaxThreads = 288;                 // 8 consumer warps + the producer warp
constexpr uint32_t kFlexTileBytes = 24u * 1024u;     // input bytes of one flex tile (B200 sweep: profiles/r1/sweep_flex.txt)
constexpr uint32_t kFlexDescBytes = 80u;             // sizeof(FlexDesc) in csic_flex_kernel.cu
constexpr int kDecConsumers = 256;        // PLANAR decoder: default consumer threads (+ the producer warp)
constexpr int kDecMaxConsumers = 512;
constexpr uint32_t kDecDescBytes = 48u;   // sizeof(DecDesc) in csic_decode_kernel.cu

// Parameters of the TMA-staged PLANAR decoder, passed by value (lives in the constant bank).
struct DecPlan {
  const uint8_t* planar;
  uint8_t* out;
  uint64_t frame_bytes, cb_off, cr_off;   // PLANAR frame layout: Y at 0, Cb / Cr planes at these offsets
  uint64_t lim_lo, lim_hi;                // byte range of the planar buffer (hull fetches are clipped to it)
  uint32_t Wo, Ho, A;                     // A = Wo * Ho pixels per frame
  uint32_t cw;                            // bytes per chroma plane row
  uint32_t hs_sh, vhold, last_c;          // log2 of the horizontal hold; odd lines replay sample last_c of the line above
  uint32_t tile_px, tiles_per_frame, n_tiles;
  uint32_t stages, y_slot, c_slot, stage_stride, out_off, out_stride, desc_off, bar_off;
  uint32_t to_rgb;
};

// ---- planning (csic_plan.cpp, host C++ only): every result depends on the arguments alone -------------------------
// Optional non-dense device layout: row pitches and frame strides in bytes (0 = dense).
struct Layout {
  size_t in_pitch = 0, in_frame = 0, out_pitch = 0, out_frame = 0;
  bool short_frames = false;   // the buffers hold only one row band of each frame (host band path)
};
// The kernel-independent part of a plan (geometry, layout, colour and quantiser constants) of output rows
// [row0, row0 + rows) of n_frames frames; returns a CSIC_* code.
int build_plan(const csic_params& p, const void* d_rgb, void* d_out, size_t n_frames, int32_t row0, int32_t rows,
               bool compact, const Layout& lay, KPlan& k);

struct DeviceLimits { int sm_count; size_t max_smem_optin; };
// csic_set_option's planner knobs; 0 = the planner's choice.  family: 0 automatic, 1 generic kernel only, 2 no TMA
// row / pooling kernel (CSIC_OPT_KERNEL_FAMILY).
struct PlanOptions { int family = 0, stages = 0; uint32_t tile_bytes = 0; int block_threads = 0, ctas_per_sm = 0; };
enum Family : int32_t { FAM_GENERIC = 1, FAM_ROWS = 2, FAM_POOL = 3, FAM_FLEX = 4 };   // as csic_last_kernel reports them
struct KernelChoice { int32_t family; KPlan k; unsigned grid; };   // grid = CTAs to launch, 0: nothing to do
// The first family whose planner takes `base`: TMA row kernel, pooling kernel, flex kernel, else the generic kernel, as
// opt.family allows.  Every candidate plans on its own copy of `base`.
KernelChoice select_kernel(const KPlan& base, const DeviceLimits& dev, const PlanOptions& opt);

// ---- host staging (csic_process_host / _band / csic_multi_process_host) --------------------------------------------
constexpr int kPipe = 3;   // chunks in flight, each with its own staging (and bounce) buffers
// Where row r of frame k of one buffer sits: byte off + k * frame + r * pitch; at(k): the same buffer from frame k on.
struct CopySide { size_t off, pitch, frame; CopySide at(size_t k) const { return {off + k * frame, pitch, frame}; } };
// One direction of the host pipeline: `rows` rows of `width` bytes per frame, as laid out in the caller's buffer, the
// pinned bounce buffer (pageable callers) and the device staging buffer (frame 0 = the chunk's first frame).
struct CopyShape { size_t width, rows; CopySide caller, bounce, staging; };
struct HostPlan {
  bool compact;                        // only every f-th input row is shipped (DECIMATE, f > 1)
  size_t first_stored;                 // the band's first stored row (an input row, or every f-th one when compact)
  Layout lay;                          // the staging layout run() is handed
  size_t in_pitch, out_pitch;          // staging row pitches the kernel sees
  size_t frames_per_chunk;
  CopyShape in, out;                   // in.rows: stored rows per frame; a PLANAR output frame is one row
};
// The host pipeline of output rows [row0, row0 + rows) of n_frames frames: ~chunk_bytes of staged input per chunk;
// full_frames ships whole frames even where compact rows would do; share_gpus: how many GPUs pull chunks from one
// shared cursor (0: none).  Returns a CSIC_* code.
int plan_host(const csic_params& p, int32_t row0, int32_t rows, size_t n_frames, const DeviceLimits& dev,
              const PlanOptions& opt, size_t chunk_bytes, bool full_frames, size_t share_gpus, HostPlan& h);
// One copy between two buffers, offsets from their bases; dst_pitch == 0: a 1-D copy of `width` bytes.
struct Copy { size_t dst, dst_pitch, src, src_pitch, width, height; };
// The copies that move nf frames of s: both sides dense, one 1-D copy; both sides' frames whole rows apart
// (frame == rows * pitch), one 2-D copy over all rows; otherwise one 2-D copy per frame.
std::vector<Copy> frame_copies(const CopyShape& s, const CopySide& dst, const CopySide& src, size_t nf);
// Output rows [r0, r1) of GPU i of G when every frame is cut into bands that start on an alignment unit, so that no
// band needs a row above it (sharding.band_plan); empty when r1 <= r0.
void band_split(const csic_params& p, size_t i, size_t G, int32_t& r0, int32_t& r1);

struct DecodeLaunch { DecPlan P; unsigned grid, threads; size_t smem; };
// The TMA-staged decoder of the PLANAR batch k.in -> k.out (tile_px: pixels per tile, 0 = the planner's choice).  False
// when the batch is outside that kernel (the LDG decoder runs instead): rows narrower than a granule, 2^30 or more
// pixels per frame, 2^32 or more tiles per launch, or chroma rows so wide that a stage does not fit.
bool plan_decode(const KPlan& k, int to_rgb, const DeviceLimits& dev, uint32_t tile_px, DecodeLaunch& d);

// ---- kernel instances and launches (kernel files); each int result is a cudaError_t --------------------------------
// One function per family (per factor where the build compiles one file per factor) maps a plan's run-time key to the
// kernel's template instance.  The launchers and set_kernel_attributes both go through them, and the setter enumerates
// every key, so no instance a plan can select runs without its dynamic shared-memory limit raised.
using KernelFn = void (*)(KPlan);
using DecodeFn = void (*)(DecPlan);
template <int F> KernelFn rows_kernel(int kformat, bool q8, bool trunc);   // csic_rows_kernel.cu, F = 1, 2, 4, 8
template <int F> KernelFn pool_kernel(int kformat, bool in4);              // csic_pool_kernel.cu, F = 2, 4, 8 (AVERAGE)
KernelFn flex_kernel(int kformat, bool trunc);                             // csic_flex_kernel.cu
DecodeFn decode_kernel(uint32_t hs_sh, bool vhold, bool to_rgb);           // csic_decode_kernel.cu
int launch(const KernelChoice& c, void* stream);                           // csic_kernels.cu: the chosen kernel
int set_kernel_attributes(size_t max_smem_optin);
int launch_expand_planar(const KPlan& k, int to_rgb, int sm_count, void* stream);   // LDG decoder of k.in -> k.out
int launch_decode_tma(const DecodeLaunch& d, void* stream);

}  // namespace csic

#endif  // CSIC_INTERNAL_H_
