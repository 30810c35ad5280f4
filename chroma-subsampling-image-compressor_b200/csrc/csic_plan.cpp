// Kernel planning and selection, host C++ only: kernel family, tile shape, ring depth, CTA size and CTAs per SM, the
// rules fitted to B200 sweeps.  The kernels only execute what a plan says; a plan depends on its arguments alone.
#include <algorithm>
#include <cstring>

#include "csic_internal.h"

namespace csic {

namespace {

// Shared memory of one SM that the residency estimates share out; the driver reserves another 1 KiB per CTA.
constexpr uint32_t kSmemPerSm = 227u * 1024u;

uint32_t up16(uint32_t v) { return (v + 15u) & ~15u; }
uint32_t up128(uint32_t v) { return (v + 127u) & ~127u; }
uint32_t ctas_by_smem(uint32_t smem) { return kSmemPerSm / (smem + 1024u); }   // CTAs of `smem` bytes one SM holds

// Persistent grid: `per_sm` CTAs per SM, never more than there are tiles.
unsigned persistent_grid(uint64_t n_tiles, int sm_count, uint32_t per_sm) {
  return (unsigned)std::min<uint64_t>(n_tiles, (uint64_t)(uint32_t)sm_count * per_sm);
}

// Spatial before chroma (case B): a counter line (W == f * Wo stream elements) must be whole output rows starting on a
// sample column (Wo % wo_unit == 0); the held pixel of an odd line is stream element (line-1) * W + lastSampleCol.
bool plan_case_b(KPlan& k, int wo_unit) {
  if (!k.case_b) return true;
  if (k.W % k.f != 0 || k.Wo % wo_unit != 0) return false;
  k.caseb_row_add = (uint32_t)k.last_sample_col / (uint32_t)k.Wo;
  k.caseb_col_bytes = ((uint32_t)k.last_sample_col % (uint32_t)k.Wo) * (uint32_t)k.in_px_bytes * (uint32_t)k.f;
  return true;
}

int32_t hold_width(const KPlan& k) { return k.case_b ? k.hf : std::max(1, k.hf / k.f); }   // in a granule, output px

// Segments per row: the fewest (at most max_n) of at most tile_max bytes that cut Wp into multiples of px_unit.
bool plan_segments(KPlan& k, uint32_t row_bytes, uint32_t tile_max, int px_unit, int max_n) {
  for (int n = (int)((row_bytes + tile_max - 1) / tile_max); n <= max_n; ++n)
    if (n >= 1 && k.Wp % (px_unit * n) == 0) { k.nsplit = n; k.tile_px = k.Wp / n; return true; }
  return false;
}

// Tiles of `rows` rows over `frames` bands of band_rows rows, nsplit segments each; false from 2^31 tiles on.
bool plan_tiles(KPlan& k, int rows, uint64_t frames, int band_rows) {
  k.tile_rows = rows;
  k.tiles_per_band = (uint32_t)((band_rows + rows - 1) / rows);
  const uint64_t n_tiles = frames * (uint64_t)k.tiles_per_band * (uint64_t)k.nsplit;
  k.n_tiles = (uint32_t)n_tiles;
  return n_tiles < (1ull << 31);
}

// "Tall image": every launch row is a whole frame row and frames lie back to back with one row stride inside and across
// frames, input AND output: the batch IS one image of n_frames * Ho rows, and a tile may span frames.
bool batch_is_tall(const KPlan& k) {
  const uint64_t stored_rows = (uint64_t)(uint32_t)k.Ho * (uint32_t)k.row_step;   // input rows from one frame's first row to the next frame's
  return k.nsplit == 1 && k.kformat != KF_PLANAR && k.n_frames > 1 && k.row0 == 0 && k.band_rows == k.Ho &&
         k.in_frame_bytes == stored_rows * k.in_row_bytes && k.out_frame_bytes == (uint64_t)(uint32_t)k.Ho * k.out_row_bytes &&
         (uint64_t)k.n_frames * (uint32_t)k.Ho < (1ull << 30) && (uint64_t)k.n_frames * (uint32_t)k.H < (1ull << 31);
}

void commit_tall(KPlan& k) {
  const int32_t rows = (int32_t)(k.n_frames * (uint32_t)k.Ho);
  k.in_frame_bytes *= k.n_frames; k.out_frame_bytes *= k.n_frames;
  k.H *= (int32_t)k.n_frames; k.Ho = rows; k.band_rows = rows; k.n_frames = 1;
}

// Whole rows of `row_bytes` per tile that fit the budget, at most max_rows; one more when the tile would stay under 70 %
// of the budget and within the slack (e.g. 15 KB RGBA 4K rows: one row leaves the ring too shallow, two are 30 KB).
int budget_rows(uint32_t row_bytes, uint32_t budget, uint32_t tile_max, int max_rows) {
  int rows = (int)std::min<uint32_t>((uint32_t)max_rows, std::max<uint32_t>(1u, budget / row_bytes));
  if ((uint32_t)rows * row_bytes < budget * 7u / 10u && (uint32_t)(rows + 1) * row_bytes <= tile_max && rows < max_rows) ++rows;
  return rows;
}

// Row and pooling kernels process Wp = Wo rounded up to 16 output pixels (of opx bytes) per row, in the row padding past
// Wo: both pitches must cover Wp (dense buffers: Wo % 16 == 0); rows, frames and bases keep 16-byte TMA granularity.
struct PaddedRows { int32_t Wp; uint64_t in, out; };   // Wp and the least input / output row bytes that cover it
PaddedRows padded_rows(int32_t Wo, int32_t f, int32_t ipb, uint32_t opx) {
  const int32_t Wp = (Wo + 15) & ~15;
  return {Wp, (uint64_t)Wp * (uint32_t)f * (uint32_t)ipb, (uint64_t)Wp * opx};
}

bool plan_padded_rows(KPlan& k, uint32_t opx) {
  const PaddedRows need = padded_rows(k.Wo, k.f, k.in_px_bytes, opx);
  k.Wp = need.Wp;
  if (k.in_row_bytes < need.in || k.out_row_bytes < need.out) return false;
  if ((k.in_row_bytes | k.out_row_bytes) & 15u) return false;
  if ((reinterpret_cast<uintptr_t>(k.in) | reinterpret_cast<uintptr_t>(k.out)) & 15u) return false;
  if ((k.in_frame_bytes | k.out_frame_bytes) & 15u) return false;
  k.ragged = k.Wp != k.Wo;
  k.in_dense = k.in_row_bytes == need.in;      // pooling: the f rows of a block row are contiguous
  k.out_dense = k.out_row_bytes == need.out;
  return true;
}

// Shared memory of the row and pooling kernels: input stages, two output buffers, tile metadata, full / empty mbarriers.
void ring_layout(KPlan& k, uint32_t stages, uint32_t meta_bytes) {
  k.out_buf_off = stages * k.stage_stride;
  k.meta_off = up128(k.out_buf_off + 2u * k.out_buf_stride);
  k.bar_off = up128(k.meta_off + stages * meta_bytes);
  k.smem_bytes = k.bar_off + stages * kRingBarBytes;
}

// Halves the rows per tile until there are ~4 tiles per SM: small batches still spread over the chip.
int spread_rows(int rows, uint64_t frames, int band_rows, int sm_count) {
  auto tiles_for = [&](int r) { return frames * (uint64_t)((band_rows + r - 1) / r); };
  while (rows > 1 && tiles_for(rows) < (uint64_t)sm_count * 4u) rows = (rows + 1) / 2;
  return rows;
}

// Equal tiles: the fewest rows per tile giving as many tiles as `rows` does.  CTAs take tiles round robin, so a short last
// tile per frame recurs with the frame's period (96 rows as 64 + 32: every other CTA got the 32-row tiles only and the
// row kernel ran at 0.71 of the copy peak where 64x64 and 128x128 frames reach 0.98 - 1.01).
int equal_tile_rows(int rows, int band_rows) {
  const int t = (band_rows + rows - 1) / rows;
  return (band_rows + t - 1) / t;
}

// ---- TMA-staged row kernel (csic_rows_kernel.cu) ---------------------------------------------------------------
bool plan_rows_kernel(KPlan& k, int sm_count, size_t max_smem_optin, int force_stages, uint32_t force_tile_bytes) {
  const bool auto_threads = k.block_threads <= 0;
  if (auto_threads) k.block_threads = kDefaultBlockThreads;
  if (k.block_threads > kMaxConsumerThreads) return false;
  const bool planar = k.kformat == KF_PLANAR;
  const uint32_t opx = planar ? 1u : (k.kformat <= KF_RGB888 ? 3u : (uint32_t)k.slot_bytes);
  if (!plan_padded_rows(k, opx) || !plan_case_b(k, 4)) return false;
  // PLANAR: three dense planes; chroma rows (Wo / hs bytes) must be 16-byte multiples too; bands start on a
  // chroma row
  if (planar && (k.ragged || !k.out_dense || k.Wo % (16 * k.planar_hs) != 0 || k.row0 % k.planar_vs != 0)) return false;
  k.hfe = hold_width(k);

  // 32-bit bundle slots at f == 1 leave through shared memory + TMA bulk stores like the 3-byte formats: there the
  // output is larger than the input (4 B per 3 B pixel) and per-warp 512-byte st.global bursts held the kernel at 0.90
  // of the copy peak (ncu: warps waiting on the store path, DRAM 70 % busy) -- 0.98 staged.  Narrower slots and f >= 2
  // keep the direct stores (16-bit slots at f == 1: 0.94 direct, 0.83 staged; cfg4: 1.03).  Must match kStaged in
  // csic_rows_kernel.cu.
  const bool staged = k.kformat <= KF_RGB888 || planar || (k.f == 1 && k.kformat == KF_SLOT32);
  // Tile budget: input bytes of one tile.  Staged formats also hold two output buffers per CTA.
  const uint32_t tile_budget = force_tile_bytes ? force_tile_bytes : 24u * 1024u;
  const uint32_t ipb = (uint32_t)k.in_px_bytes;
  const uint32_t row_in = (uint32_t)k.Wp * ipb * (uint32_t)k.f;  // bytes of one processed input row
  const uint32_t tile_max = tile_budget + tile_budget / 3;        // a tile may overshoot the budget by a third
  if (!plan_segments(k, row_in, tile_max, 16 * (planar ? k.planar_hs : 1), 64)) return false;
  k.tile_in_bytes = (uint32_t)k.tile_px * ipb * (uint32_t)k.f;    // one row segment
  k.tile_out_bytes = (uint32_t)k.tile_px * opx;
  // Tall image: 32x32 frames make 64-row tiles of two frames instead of one 3 KB tile per frame (0.74 -> 0.95 of the
  // copy peak).  The kernel does not change: the only rule that looks at a row index, "odd lines replay the line above"
  // (f == 1, 4:2:0 / 4:1:0), reads the same parity when frames have an even number of rows.
  const bool tall = batch_is_tall(k) && !k.case_b && !(k.vf == 2 && k.f == 1 && (k.Ho & 1));
  const uint32_t frames = tall ? 1u : k.n_frames;
  const int band_rows = tall ? (int)(k.n_frames * (uint32_t)k.Ho) : k.band_rows;
  // Rows per tile: whole rows only (so the tile's output is contiguous), as many as fit the budget, spread and equal.
  int rows = 1;
  if (k.nsplit == 1) {
    rows = std::min(budget_rows(k.tile_in_bytes, tile_budget, tile_max, kMaxTileRows), band_rows);
    rows = spread_rows(rows, frames, band_rows, sm_count);
    // staged 32-bit slots: a tile's two output buffers are larger than its input stages; keep two CTAs resident
    // (4096-pixel rows: two rows per tile left room for one CTA only -- 0.81 of the copy peak instead of 0.98)
    if (staged && !planar && k.kformat > KF_RGB888)
      while (rows > 1 && 2u * ((uint32_t)rows * (k.tile_in_bytes + 32u)) + 2u * ((uint32_t)rows * k.tile_out_bytes) + 2048u > kSmemPerSm / 2u - 1024u)
        --rows;
    // Equal tiles; even row counts keep a held line and its sample in one tile.
    int bal = equal_tile_rows(rows, band_rows);
    if ((k.vf == 2 || planar) && (bal & 1) && bal < rows) ++bal;
    rows = std::min(rows, bal);
    if (planar && rows > 1) rows &= ~(k.planar_vs - 1);          // tiles start on a chroma row
    if (rows < 1) rows = 1;
  }
  if (!plan_tiles(k, rows, frames, band_rows)) return false;
  // Tiny tiles (whole frames of a few KB: a tile never spans two frames): a granule per thread is all there is, so the
  // per-tile costs dominate -- half-size CTAs, as many as fit (32x32 frames: 0.74 of the copy peak vs 0.51;
  // profiles/r1/sweep_rows_v8.txt)
  const bool tiny = (uint32_t)rows * ((uint32_t)k.tile_px >> 2) <= 512u && k.n_tiles > (uint32_t)sm_count * 8u;
  if (tiny && auto_threads) k.block_threads = 128;

  k.stage_stride = up128((uint32_t)rows * (k.tile_in_bytes + 32u));
  k.out_buf_stride = staged ? up128((uint32_t)rows * k.tile_out_bytes) : 0u;
  if (planar)   // [Y rows][Cb rows][Cr rows]
    k.out_buf_stride = up128((uint32_t)rows * (uint32_t)k.tile_px +
                             2u * (uint32_t)((rows + k.planar_vs - 1) / k.planar_vs) * ((uint32_t)k.tile_px / (uint32_t)k.planar_hs));
  // Ring depth and residency, fitted to B200 sweeps (profiles/r1/exp_ctas_v4.txt): the kernel is fastest with
  // about four ~24 KB tiles in flight per SM -- 2 resident CTAs x 2 stages (cfg4 0.996 of the measured copy peak
  // vs 0.953 with 4 CTAs; cfg2 0.97 vs 0.94 with 6 tiles in flight).  Only when a tile carries little compute
  // per byte (f >= 4: one pixel in 16 is converted) does a third stage pay (cfg5 0.98 vs 0.92).
  auto need = [&](int s) {
    return (uint32_t)s * k.stage_stride + 2u * k.out_buf_stride + (uint32_t)s * kTileMetaBytes + (uint32_t)s * 16u + 384u;
  };
  auto ctas_for = [&](int s) {
    return std::min<uint32_t>(std::min<uint32_t>(ctas_by_smem(need(s)), 2048u / ((uint32_t)k.block_threads + 32u)), 8u);
  };
  int stages = force_stages >= 2 ? force_stages : (k.f >= 4 ? 3 : 2);
  while (force_stages < 2 && stages > 2 && ctas_for(stages) < 2) --stages;
  if (need(stages) > max_smem_optin || ctas_for(stages) < 1) return false;
  // f == 1 converts every byte it loads (issue slots 64 % busy with 16 warps): there more resident warps win
  // (PLANAR 1080p: 0.97 of the copy peak with 3 CTAs vs 0.84 with 2; 16-bit bundles: 0.93 with 4).
  k.ctas_per_sm = (int32_t)std::min<uint32_t>(ctas_for(stages), tiny ? 8u : (k.f == 1 ? 4u : 2u));
  k.stages = stages;
  if (tall) commit_tall(k);
  ring_layout(k, (uint32_t)stages, kTileMetaBytes);
  return true;
}

// ---- AVERAGE extension: TMA-staged pooling kernel (csic_pool_kernel.cu) -----------------------------------------
bool plan_pool_kernel(KPlan& k, int sm_count, size_t max_smem_optin) {
  // (csic_process_host re-pitches widths that break the padded-row rules, csic_process_device_pitched takes them as given)
  const bool staged = k.kformat <= KF_RGB888;
  const uint32_t opx = staged ? 3u : (uint32_t)k.slot_bytes;
  if (!plan_case_b(k, k.hf) || !plan_padded_rows(k, opx)) return false;
  // 4x4 / 8x8 pooling keeps more live registers per thread: 6 consumer warps leave room for one more CTA per SM
  // (B200 sweep, profiles/r1/sweep_pool_v8.txt: 8K 4x4 0.97 of the copy peak vs 0.92 with 8 warps)
  const bool auto_threads = k.block_threads <= 0;
  if (auto_threads) k.block_threads = k.f >= 4 ? 192 : kDefaultBlockThreads;
  if (k.block_threads > kMaxConsumerThreads) return false;

  const uint32_t f = (uint32_t)k.f, ipb = (uint32_t)k.in_px_bytes;
  const uint32_t budget = 24u * 1024u, tile_max = budget + budget / 3;   // (48 KB tiles for 8x8 pooling: 1080p +5 %, 4K / 8K -12 %)
  const uint32_t block_row_bytes = (uint32_t)k.Wp * f * f * ipb;          // the f input rows of one output row
  if (!plan_segments(k, block_row_bytes, tile_max, 16, 256)) return false;
  k.tile_in_bytes = (uint32_t)k.tile_px * f * f * ipb;                   // per output-row segment: f row parts
  k.tile_out_bytes = (uint32_t)k.tile_px * opx;
  int rows = 1;
  if (k.nsplit == 1) {
    // (e.g. 2560x1440 2x2 or 640x480 8x8: an output row carries 15 KB of input, a tile two rows)
    rows = budget_rows(k.tile_in_bytes, budget, tile_max, 1 << 30);
    rows = std::min(rows, (int)(2u * (uint32_t)kPoolMaxRows / f));      // held_addr[] holds rows * f/2 entries
    rows = std::min(rows, k.band_rows);
    if (!k.out_dense) rows = 1;                                           // a tile's output must be one contiguous range
    rows = spread_rows(rows, k.n_frames, k.band_rows, sm_count);
    rows = std::min(rows, equal_tile_rows(rows, k.band_rows));
  }
  if (!plan_tiles(k, rows, k.n_frames, k.band_rows)) return false;
  // 8x8 pooling is bound by the integer pipes, and a granule is 256 input pixels: a 15 KB tile has twenty of them, four
  // threads each -- 80 busy threads of 192 (1080p: 240 output pixels per row, split three ways).  Size the CTA to the
  // tile and let more of them be resident instead (1080p 8x8: 0.69-0.81 -> 0.78-0.91 of the copy peak).
  const uint32_t units = (uint32_t)rows * ((uint32_t)k.tile_px >> 2) * 4u;
  const bool small_cta = auto_threads && k.f == 8 && 2u * units <= (uint32_t)k.block_threads;   // (tiles that fill 2/3 of the CTA or more: 3-4 % slower this way)
  if (small_cta) k.block_threads = (int32_t)std::max(64u, (units + 31u) & ~31u);
  k.stage_stride = up128((uint32_t)rows * k.tile_in_bytes + (uint32_t)kPoolMaxRows * 32u);
  k.out_buf_stride = staged ? (uint32_t)(kMaxConsumerThreads / 32) * 384u / 2u : 0u;   // 2 x stride = one 384-byte slot per warp
  k.stages = 2;
  const uint32_t need = 2u * k.stage_stride + 2u * k.out_buf_stride + 2u * kPoolMetaBytes + 32u + 384u;
  if (need > max_smem_optin) return false;
  // pooling converts every input pixel: the kernel is issue-bound, so take all the warps that fit (measured:
  // 4 CTAs 0.79 of the copy peak on the 4K 2x2 case vs 0.73 with 2)
  const uint32_t threads = (uint32_t)k.block_threads + 32u;
  const uint32_t by_regs = 65536u / ((k.f == 2 ? 56u : 72u) * threads);     // __maxnreg__ of csic_pool_kernel
  k.ctas_per_sm = (int32_t)std::max<uint32_t>(1u, std::min<uint32_t>(std::min<uint32_t>(small_cta ? 8u : 4u, by_regs), ctas_by_smem(need)));
  ring_layout(k, 2u, kPoolMetaBytes);
  return true;
}

// ---- flex kernel: any width / pitch / alignment (csic_flex_kernel.cu) --------------------------------------------
bool plan_flex_kernel(KPlan& k, int sm_count, size_t max_smem_optin, int force_stages, uint32_t force_tile_bytes) {
  const uint32_t ipb = (uint32_t)k.in_px_bytes, f = (uint32_t)k.f, pxb = f * ipb;
  if (!plan_case_b(k, k.hf)) return false;
  k.hfe = hold_width(k);
  const bool planar = k.kformat == KF_PLANAR;
  const uint32_t unit = (k.kformat <= KF_RGB888) ? 12u : (planar ? 4u : 4u * (uint32_t)k.slot_bytes);
  const uint32_t S = (uint32_t)k.slots_per_row, Wo = (uint32_t)k.Wo;
  const uint32_t tile_bytes = force_tile_bytes ? std::max(1024u, force_tile_bytes) : kFlexTileBytes;
  const uint32_t tile_px_max = std::max(16u, (tile_bytes / pxb) & ~15u);
  k.tile_px = (int32_t)std::min(tile_px_max, (S + 15u) & ~15u);
  k.nsplit = (int32_t)((S + (uint32_t)k.tile_px - 1u) / (uint32_t)k.tile_px);
  const uint32_t len_in_max = ((std::min((uint32_t)k.tile_px, Wo) - 1u) * f + 1u) * ipb;
  // consecutive processed rows contiguous in memory?  (dense rows, every stored row is read)
  const bool contiguous = k.nsplit == 1 && k.row_step == 1 && k.in_row_bytes == (uint32_t)k.W * ipb;
  if (k.block_threads <= 0) k.block_threads = kFlexConsumers;
  k.block_threads = std::min(k.block_threads, kFlexMaxThreads - 32);
  const uint32_t stages = (uint32_t)std::min(std::max(force_stages, 2), 8);

  // Tall image: what batches of small frames need (a 96x96 frame at f = 8 is twelve 288-byte rows: one tile per frame
  // left the SMs waiting on 3 KB copies).  Only the held-line rule still looks at the row index inside its frame.
  const bool tall = batch_is_tall(k);
  const uint32_t frames = tall ? 1u : k.n_frames;
  const uint32_t band_rows = tall ? k.n_frames * (uint32_t)k.Ho : (uint32_t)k.band_rows;

  // Rows per tile (whole rows only).  What the B200 sweeps after the round-2 restructure show (profiles/r2/sweep_flex*.txt,
  // flex_rows_*.txt): throughput follows (a) the consumer warps that have work, summed over the resident CTAs -- it
  // saturates near 20 for the light formats and keeps growing to 32 for the fused RGB reconstruction, which is
  // issue-bound -- and (b) the granules per tile, over which ~110 warp-instructions of per-tile work and two CTA
  // barriers are spread; two resident CTAs instead of three or four cost another ~15 %.  The candidate that maximises
  // that product wins: 1366x768 f = 1 RGB888 -> 4 rows, 1080x1920 -> 7, 1918x1078 -> 4, 3838x2158 f = 2 -> 2.
  const uint32_t NW = (uint32_t)k.block_threads / 32u, gpr = (std::min((uint32_t)k.tile_px, S) + 3u) / 4u;
  const uint32_t row_in = up16((contiguous ? std::max(len_in_max, k.in_row_bytes) : len_in_max) + 15u) + 16u;
  uint32_t row_out = ((uint32_t)k.tile_px / 4u) * unit + 16u;
  if (planar) row_out += 2u * (uint32_t)k.tile_px;
  // resident CTAs: shared memory, threads, and the 56 registers per thread __launch_bounds__(288, 4) grants
  const uint32_t cta_cap = std::min<uint32_t>(std::min<uint32_t>(8u, 2048u / ((uint32_t)k.block_threads + 32u)),
                                              65536u / (56u * ((uint32_t)k.block_threads + 32u)));
  auto ctas_for = [&](uint32_t r) {
    const uint32_t smem = stages * (r * row_in + 32u) + r * row_out + 2048u;
    return std::min<uint32_t>(cta_cap, ctas_by_smem(smem));
  };
  int rows = 1;
  if (k.nsplit == 1) {
    const uint32_t rmax = std::min<uint32_t>((uint32_t)kFlexMaxRows, band_rows);
    auto tiles_for = [&](uint32_t r) { return (uint64_t)frames * (uint64_t)((band_rows + r - 1u) / r); };
    if (force_tile_bytes) {
      const uint32_t per_row = contiguous ? k.in_row_bytes : len_in_max;
      rows = (int)std::min<uint32_t>(rmax, std::max<uint32_t>(1u, tile_bytes / std::max(1u, per_row)));
    } else {
      // fraction of a CTA's consumer warps that get granules (flex_consume's modes 0 and 2); rows that deal unevenly
      // or are narrower than a warp run the flat loop: every thread busy, ~15 % more instructions per granule
      auto busy_frac = [&](uint32_t r) {
        const bool lanes_ok = gpr * 5u >= ((gpr + 31u) / 32u) * 32u * 4u;
        if (r <= NW) {
          const uint32_t parts = NW / r;
          const uint32_t lanes = parts * 32u, it = (gpr + lanes - 1u) / lanes;
          if ((parts & (parts - 1u)) == 0u && gpr * 5u >= it * lanes * 4u) return (double)(r * parts) / NW;
          return 0.85;
        }
        const uint32_t rounds = (r + NW - 1u) / NW;
        if (lanes_ok && r * 5u >= rounds * NW * 4u) return (double)r / (rounds * NW);
        return 0.85;
      };
      const double busy_cap = k.kformat == KF_RGB888 ? 32.0 : 20.0;
      double best_score = -1.0;
      for (uint32_t r = 1; r <= rmax; ++r) {
        const uint32_t c = ctas_for(r);
        if (c == 0u) break;
        if (r > 1u && tiles_for(r) < (uint64_t)sm_count * 8u) break;        // keep every SM supplied with several tiles
        const double gran = (double)r * gpr;
        // a short last tile per frame recurs with the frame's period under round-robin tile assignment: weigh by its fill
        const double fill = (double)band_rows / (double)(((band_rows + r - 1u) / r) * r);
        const double score = std::min(busy_cap, c * NW * busy_frac(r)) * gran / (gran + 400.0) * (c >= 3u ? 1.0 : 0.85) * fill;
        if (score >= best_score * 1.0001) { best_score = score; rows = (int)r; }
      }
    }
  }
  if (!plan_tiles(k, rows, frames, (int)band_rows)) return false;
  k.in_dense = (contiguous && rows > 1) ? 1 : 0;
  const uint32_t dense_out_row = planar ? Wo : S * (unit / 4u);
  k.out_dense = k.out_row_bytes == dense_out_row ? 1 : 0;

  k.stage_stride = row_in;
  const uint32_t in_bytes = stages * ((uint32_t)rows * k.stage_stride + 32u);   // + slack: pixel loads read one word ahead
  uint32_t stage_bytes = (uint32_t)rows * (((uint32_t)k.tile_px / 4u) * unit + 16u) + 16u;   // rows at their own offset mod 16
  if (planar) stage_bytes += 2u * (uint32_t)(rows / std::max(1, k.planar_vs) + 1) * (uint32_t)k.tile_px;
  k.out_buf_off = up128(in_bytes);
  k.out_buf_stride = up16(stage_bytes + 32u);                               // + slack: span_store reads one word ahead
  k.meta_off = k.out_buf_off + k.out_buf_stride;                            // held words of every stage
  k.bar_off = up128(k.meta_off + stages * (uint32_t)kFlexMaxRows * 4u);     // the ring's mbarriers, then S descriptors
  k.smem_bytes = k.bar_off + stages * (kRingBarBytes + kFlexDescBytes);
  if (k.smem_bytes > max_smem_optin) return false;
  k.tall_ho = tall ? k.Ho : 0;
  if (tall) commit_tall(k);
  k.stages = (int32_t)stages;
  // the grid is a whole number of RESIDENT CTAs per SM: a CTA that has to wait for a slot would run its share of the
  // tiles after everybody else (round 1 ignored the register limit here: small tiles launched 5-7 CTAs per SM where 4
  // fit, and the second wave doubled the run time -- 1080x1920 with 4-row tiles: 0.69 instead of 0.9)
  k.ctas_per_sm = (int32_t)std::max<uint32_t>(1u, std::min<uint32_t>(cta_cap, ctas_by_smem(k.smem_bytes)));
  return true;
}

// generic gather kernel (csic_kernels.cu): a warp per row (or per 32 / gpr rows under 32 granules), four per CTA
unsigned generic_grid(const KPlan& k, int sm_count) {
  const uint64_t n_rows = (uint64_t)k.n_frames * (uint64_t)k.band_rows;
  if (n_rows == 0 || k.slots_per_row == 0) return 0;
  const uint32_t gpr = ((uint32_t)k.slots_per_row + 3u) >> 2;
  const uint64_t groups = gpr < 32u ? (n_rows + 32u / gpr - 1u) / (32u / gpr) : n_rows;
  return (unsigned)std::min<uint64_t>((groups + 3u) / 4u, (uint64_t)sm_count * 16u);
}

}  // namespace

int build_plan(const csic_params& p, const void* d_rgb, void* d_out, size_t n_frames, int32_t row0,
               int32_t rows, bool compact, const Layout& lay, KPlan& k) {
  const Geometry g = geometry(p);
  std::memset(&k, 0, sizeof(k));
  k.in = static_cast<const uint8_t*>(d_rgb);
  k.out = static_cast<uint8_t*>(d_out);
  k.compact = compact ? 1 : 0;
  k.row_step = compact ? 1 : p.factor;
  k.in_frame_bytes = compact ? g.in_row_bytes * (size_t)g.out_h : g.in_frame_bytes;
  k.out_frame_bytes = g.out_frame_bytes;
  if (g.in_row_bytes > 0xFFFFFFFFull || g.out_row_bytes > 0xFFFFFFFFull) return CSIC_EINVAL_DIMS;
  if ((uint64_t)g.out_w * (uint64_t)g.out_h >= (1ull << 31) || (uint64_t)p.width * p.height >= (1ull << 31))
    return CSIC_EINVAL_DIMS;   // the reference's counters are far narrower; 2^31 pixels per frame is our limit
  k.in_row_bytes = (uint32_t)g.in_row_bytes;
  k.out_row_bytes = (uint32_t)g.out_row_bytes;
  if (lay.in_pitch) {
    if (lay.in_pitch < g.in_row_bytes || lay.in_pitch > 0xFFFFFFFFull) return CSIC_EINVAL_ARG;
    k.in_row_bytes = (uint32_t)lay.in_pitch;
    k.in_frame_bytes = (size_t)lay.in_pitch * (size_t)(compact ? g.out_h : p.height);
  }
  if (lay.in_frame) {
    if (lay.in_frame < k.in_frame_bytes && !lay.short_frames) return CSIC_EINVAL_ARG;
    k.in_frame_bytes = lay.in_frame;
  }
  if ((lay.out_pitch || lay.out_frame || lay.short_frames) && p.out_format == CSIC_OUT_PLANAR)
    return CSIC_EINVAL_MODE;   // three planes per frame: no pitched / banded host layout
  if (lay.out_pitch) {
    if (lay.out_pitch < g.out_row_bytes || lay.out_pitch > 0xFFFFFFFFull) return CSIC_EINVAL_ARG;
    k.out_row_bytes = (uint32_t)lay.out_pitch;
    k.out_frame_bytes = (size_t)lay.out_pitch * (size_t)g.out_h;
  }
  if (lay.out_frame) {
    if (lay.out_frame < k.out_frame_bytes && !lay.short_frames) return CSIC_EINVAL_ARG;
    k.out_frame_bytes = lay.out_frame;
  }
  k.in_px_bytes = g.in_px_bytes;
  auto swap_rb = [](uint32_t c) { return (c & 0xFF00FF00u) | ((c & 0xFFu) << 16) | ((c >> 16) & 0xFFu); };
  const bool bgr = p.in_format == CSIC_IN_BGRA32;
  k.coef_y = bgr ? swap_rb(0x001D964Du) : 0x001D964Du;      //  77, 150,  29, 0
  k.coef_ncb = bgr ? swap_rb(0x0080552Bu) : 0x0080552Bu;    //  43,  85,-128, 0  (negated Cb row)
  k.coef_ncr = bgr ? swap_rb(0x00156B80u) : 0x00156B80u;    //-128, 107,  21, 0  (negated Cr row)
  k.W = p.width;
  k.H = p.height;
  k.Wo = g.out_w;
  k.Ho = g.out_h;
  k.f = p.factor;
  k.hf = g.hf;
  k.vf = g.vf;
  k.last_sample_col = ((p.width - 1) / g.hf) * g.hf;
  // Spatial before chroma runs the chroma stage with misaligned counters (ImageCompressorTop.scala:52-58) -- which only
  // matters when that stage holds anything: with 4:4:4 (hf == vf == 1, the application's default) every element is its
  // own sample point whatever the counters say, so any width takes the fast kernels.
  k.case_b = (!g.chroma_first && p.factor > 1 && (g.hf > 1 || g.vf > 1)) ? 1 : 0;
  k.quant_first = g.quant_first ? 1 : 0;
  k.trunc = p.round_mode == CSIC_ROUND_TRUNC;
  k.average = (p.pool_mode == CSIC_POOL_AVERAGE && p.factor > 1) ? 1 : 0;
  if (p.out_format == CSIC_OUT_YCC888) k.kformat = KF_YCC888;
  else if (p.out_format == CSIC_OUT_RGB888) k.kformat = KF_RGB888;
  else if (p.out_format == CSIC_OUT_PLANAR) k.kformat = KF_PLANAR;
  else k.kformat = g.out_px_bytes == 1 ? KF_SLOT8 : (g.out_px_bytes == 2 ? KF_SLOT16 : KF_SLOT32);
  k.slot_bytes = g.out_px_bytes;
  k.slots_per_row = (k.kformat <= KF_RGB888 || k.kformat == KF_PLANAR)
                        ? g.out_w : (int32_t)(g.out_row_bytes / (size_t)g.out_px_bytes);
  k.planar_hs = g.planar_hs; k.planar_vs = g.planar_vs; k.planar_cw = g.planar_cw; k.planar_ch = g.planar_ch;
  k.planar_cb_off = (uint64_t)g.out_w * (uint64_t)g.out_h;
  k.planar_cr_off = k.planar_cb_off + (uint64_t)g.planar_cw * (uint64_t)g.planar_ch;
  k.sy = 8 - p.y_bits;
  k.scb = 8 - p.cb_bits;
  k.scr = 8 - p.cr_bits;
  k.cb_bits = p.cb_bits;
  k.cr_bits = p.cr_bits;
  k.qmask = ((0xFFu << k.sy) & 0xFFu) | (((0xFFu << k.scb) & 0xFFu) << 8) | (((0xFFu << k.scr) & 0xFFu) << 16);
  k.row0 = row0;
  k.band_rows = rows;
  if (n_frames > 0xFFFFFFFFull) return CSIC_EINVAL_ARG;
  k.n_frames = (uint32_t)n_frames;
  return CSIC_OK;
}

KernelChoice select_kernel(const KPlan& base, const DeviceLimits& dev, const PlanOptions& opt) {
  KernelChoice c;
  auto fresh = [&]() -> KPlan& { c.k = base; c.k.block_threads = opt.block_threads; return c.k; };
  const int sms = dev.sm_count;
  const size_t smem = dev.max_smem_optin;
  const bool rows = base.band_rows > 0 && base.n_frames > 0, avg = base.average && base.f > 1;   // avg: pooling kernel
  if (opt.family == 0 && rows && !avg && plan_rows_kernel(fresh(), sms, smem, opt.stages, opt.tile_bytes)) c.family = FAM_ROWS;
  else if (opt.family == 0 && avg && plan_pool_kernel(fresh(), sms, smem)) c.family = FAM_POOL;
  else if (opt.family != 1 && rows && !avg && plan_flex_kernel(fresh(), sms, smem, opt.stages, opt.tile_bytes)) c.family = FAM_FLEX;
  else {
    c.family = FAM_GENERIC;
    c.grid = generic_grid(fresh(), sms);
    return c;
  }
  c.grid = persistent_grid(c.k.n_tiles, sms, (uint32_t)(opt.ctas_per_sm > 0 ? opt.ctas_per_sm : std::max(1, c.k.ctas_per_sm)));
  return c;
}

// ---- TMA-staged PLANAR decoder (csic_decode_kernel.cu) -----------------------------------------------------------
bool plan_decode(const KPlan& k, int to_rgb, const DeviceLimits& dev, uint32_t tile_px, DecodeLaunch& d) {
  if (k.Wo < 4 || k.Ho < 1) return false;
  const uint64_t A = (uint64_t)k.Wo * (uint64_t)k.Ho;
  if (A >= (1ull << 30)) return false;
  DecPlan& P = d.P;
  std::memset(&P, 0, sizeof(P));
  P.planar = k.in; P.out = k.out;
  P.frame_bytes = k.out_frame_bytes; P.cb_off = k.planar_cb_off; P.cr_off = k.planar_cr_off;
  P.lim_lo = reinterpret_cast<uintptr_t>(k.in);
  P.lim_hi = P.lim_lo + (uint64_t)k.n_frames * k.out_frame_bytes;
  P.Wo = (uint32_t)k.Wo; P.Ho = (uint32_t)k.Ho; P.A = (uint32_t)A;
  P.cw = (uint32_t)k.planar_cw;
  P.hs_sh = k.planar_hs == 4 ? 2u : (k.planar_hs == 2 ? 1u : 0u);
  P.vhold = k.planar_vs == 2 ? 1u : 0u;                           // planar_vs == 2 <=> vf == 2 at f == 1: odd lines are held
  P.last_c = (uint32_t)((k.last_sample_col / k.f) / k.planar_hs);
  P.to_rgb = to_rgb ? 1u : 0u;
  const uint32_t vs = (uint32_t)k.planar_vs;
  // B200 sweeps (profiles/r2/decode_sweep.txt): 8192-pixel tiles; a frame of up to 12288 pixels is one tile.  A third
  // stage pays for the RGB reconstruction and on the 4-pixel paths (1080p 4:2:0 to RGB 0.83 -> 0.90, 333-pixel rows to
  // YCC 0.86 -> 0.93: the consumers otherwise wait for the next tile's loads) where it still leaves two CTAs per SM
  // their shared memory; where it does not (full-size chroma planes) two stages of 8192 pixels beat three of 4096, and
  // the 16-pixel path to YCC888 is fastest with two (0.945 vs 0.92).
  const bool w16 = (k.Wo & 15) == 0;
  uint32_t T = (tile_px ? tile_px : (A <= 12288u ? (uint32_t)((A + 15u) & ~(uint64_t)15) : 8192u)) & ~15u;
  if (T < 64u) T = 64u;
  auto layout = [&](uint32_t t, uint32_t S) {
    P.tile_px = (uint32_t)std::min<uint64_t>(t, (A + 15u) & ~(uint64_t)15);
    const uint32_t nr = std::min<uint32_t>(P.Ho, (P.tile_px + P.Wo - 2u) / P.Wo + 1u);       // rows a tile can touch
    const uint32_t ncr = vs == 2u ? nr / 2u + 1u : nr;
    P.stages = S;
    P.y_slot = (P.tile_px + 32u + 15u) & ~15u;
    P.c_slot = (ncr * P.cw + 48u + 15u) & ~15u;
    P.stage_stride = P.y_slot + 2u * P.c_slot;
    P.out_off = S * P.stage_stride;
    P.out_stride = (P.tile_px * 3u + 32u + 15u) & ~15u;
    P.desc_off = P.out_off + 2u * P.out_stride;
    P.bar_off = P.desc_off + S * kDecDescBytes;
    return (size_t)P.bar_off + S * kRingBarBytes;
  };
  uint32_t S = (to_rgb || !w16) ? 3u : 2u;
  size_t smem = layout(T, S);
  if (S == 3u && smem > dev.max_smem_optin / 2) { S = 2u; smem = layout(T, S); }
  while (smem > dev.max_smem_optin / 2 && T > 256u) { T = (T / 2u) & ~15u; smem = layout(T, S); }   // keep two CTAs per SM
  if (smem > dev.max_smem_optin) return false;
  P.tiles_per_frame = (uint32_t)((A + P.tile_px - 1u) / P.tile_px);
  P.tile_px = (uint32_t)((((A + P.tiles_per_frame - 1u) / P.tiles_per_frame) + 15u) & ~(uint64_t)15);   // equal tiles (never larger than planned)
  P.tiles_per_frame = (uint32_t)((A + P.tile_px - 1u) / P.tile_px);
  const uint64_t n_tiles = (uint64_t)k.n_frames * P.tiles_per_frame;
  if (n_tiles >= (1ull << 32)) return false;
  P.n_tiles = (uint32_t)n_tiles;
  // one consumer thread per 16-pixel group / 4-pixel granule of a tile, at most 256 (small frames: fewer idle warps)
  const uint32_t units = w16 ? P.tile_px >> 4 : P.tile_px >> 2;
  const uint32_t nc = std::max(64u, std::min<uint32_t>((uint32_t)kDecConsumers, (units + 31u) & ~31u));
  d.threads = nc + 32u;
  // (228 KiB per SM here, 227 KiB in kSmemPerSm: unifying the two would change decoder plans)
  const uint32_t per_sm = (uint32_t)std::max<size_t>(1, std::min<size_t>({(size_t)8, (size_t)(2048u / d.threads), (size_t)(228u * 1024u) / (smem + 1024u)}));
  d.grid = persistent_grid(n_tiles, dev.sm_count, per_sm);
  d.smem = smem;
  return true;
}

// ---- host staging (csic_api.cu's host pipeline) -------------------------------------------------------------------
namespace {

// Dense when the dense layout already satisfies a TMA kernel's 16-byte rules; otherwise the rows are re-pitched on the
// way in and out (the copies are 2-D anyway), so odd widths also avoid the generic kernel.
Layout staging_layout(const csic_params& p, const Geometry& g, bool compact, const DeviceLimits& dev,
                      const PlanOptions& opt) {
  auto eligible = [&](const Layout& l) {   // one frame at 4 KiB aligned bases
    KPlan k;
    if (build_plan(p, (void*)uintptr_t(4096), (void*)uintptr_t(4096), 1, 0, g.out_h, compact, l, k) != CSIC_OK) return false;
    const int family = select_kernel(k, dev, opt).family;
    return family == FAM_ROWS || family == FAM_POOL;
  };
  if (eligible(Layout()) || p.out_format == CSIC_OUT_PLANAR) return Layout();
  const PaddedRows need = padded_rows(g.out_w, p.factor, g.in_px_bytes, (uint32_t)g.out_px_bytes);
  Layout cand;
  cand.in_pitch = (std::max<size_t>(g.in_row_bytes, need.in) + 15) & ~(size_t)15;
  cand.out_pitch = (std::max<size_t>(g.out_row_bytes, need.out) + 15) & ~(size_t)15;
  return eligible(cand) ? cand : Layout();
}

}  // namespace

int plan_host(const csic_params& p, int32_t row0, int32_t rows, size_t n_frames, const DeviceLimits& dev,
              const PlanOptions& opt, size_t chunk_bytes, bool full_frames, size_t share_gpus, HostPlan& h) {
  const Geometry g = geometry(p);
  const bool band = !(row0 == 0 && rows == g.out_h);
  // A DECIMATE pipeline with f > 1 reads only every f-th input row, and when they sit at a uniform pitch across the
  // frames of a batch only those rows are shipped: 1/f of the H2D bytes.
  h.compact = p.pool_mode == CSIC_POOL_DECIMATE && p.factor > 1 && p.height % p.factor == 0 && !full_frames;
  int32_t in_row0 = 0, in_rows = p.height;
  if (band) {
    const int rc = csic_band_input_rows(&p, row0, rows, &in_row0, &in_rows);
    if (rc != CSIC_OK) return rc;
    if (p.out_format == CSIC_OUT_PLANAR) return CSIC_EINVAL_MODE;   // planes are not row bands
  }
  const size_t step = h.compact ? (size_t)p.factor : 1u;            // input rows per stored row
  h.first_stored = (size_t)in_row0 / step;
  const size_t rows_stored = h.compact ? (size_t)(row0 + rows) - h.first_stored : (size_t)in_rows;
  h.lay = staging_layout(p, g, h.compact, dev, opt);
  h.in_pitch = h.lay.in_pitch ? h.lay.in_pitch : g.in_row_bytes;
  h.out_pitch = h.lay.out_pitch ? h.lay.out_pitch : g.out_row_bytes;
  const size_t dev_in_frame = h.in_pitch * rows_stored;
  const size_t dev_out_frame = band ? h.out_pitch * (size_t)rows : std::max(h.out_pitch * (size_t)rows, g.out_frame_bytes);
  if (band) h.lay = {h.in_pitch, dev_in_frame, h.out_pitch, dev_out_frame, true};   // the device holds the band's rows only
  // Frames per chunk: ~chunk_bytes of input, at least one, at most all; several chunks per GPU that shares the cursor.
  h.frames_per_chunk = std::min(n_frames, std::max<size_t>(1, chunk_bytes / std::max<size_t>(1, dev_in_frame)));
  if (share_gpus)
    h.frames_per_chunk = std::min(h.frames_per_chunk, std::max<size_t>(1, n_frames / (share_gpus * (size_t)kPipe)));
  const size_t irb = g.in_row_bytes;
  h.in = {irb, rows_stored, {h.first_stored * step * irb, step * irb, g.in_frame_bytes}, {0, irb, irb * rows_stored},
          {0, h.in_pitch, dev_in_frame}};
  const bool planar = p.out_format == CSIC_OUT_PLANAR;
  const size_t orow = planar ? g.out_frame_bytes : g.out_row_bytes, orows = planar ? 1u : (size_t)rows;
  h.out = {orow, orows, {(size_t)row0 * orow, orow, g.out_frame_bytes}, {0, orow, orow * orows},
           {0, planar ? orow : h.out_pitch, dev_out_frame}};
  return CSIC_OK;
}

std::vector<Copy> frame_copies(const CopyShape& s, const CopySide& dst, const CopySide& src, size_t nf) {
  const size_t w = s.width, r = s.rows;
  auto dense = [&](const CopySide& x) { return x.pitch == w && x.frame == r * w; };
  auto whole_rows = [&](const CopySide& x) { return x.frame == r * x.pitch; };
  if (dense(dst) && dense(src)) return {{dst.off, 0, src.off, 0, nf * r * w, 1}};
  if (whole_rows(dst) && whole_rows(src)) return {{dst.off, dst.pitch, src.off, src.pitch, w, nf * r}};
  std::vector<Copy> v;
  for (size_t k = 0; k < nf; ++k) v.push_back({dst.off + k * dst.frame, dst.pitch, src.off + k * src.frame, src.pitch, w, r});
  return v;
}

void band_split(const csic_params& p, size_t i, size_t G, int32_t& r0, int32_t& r1) {
  const Geometry g = geometry(p);
  const bool case_b = !g.chroma_first && p.factor > 1;
  const int unit = case_b ? p.factor * g.vf : std::max(1, (p.factor % g.vf == 0 ? p.factor : p.factor * g.vf) / p.factor);
  const int units = (g.out_h + unit - 1) / unit;
  r0 = std::min(g.out_h, (int)(units * i / G) * unit);
  r1 = std::min(g.out_h, (int)(units * (i + 1) / G) * unit);
}

}  // namespace csic

extern "C" {

// Input rows a band of output rows reads: the rows it decimates / pools from, plus -- when the band
// starts on a line whose chroma is held from the line above -- the row holding that sample.
int csic_band_input_rows(const csic_params* p, int32_t out_row0, int32_t out_rows, int32_t* in_row0,
                         int32_t* in_rows) {
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  const csic::Geometry g = csic::geometry(*p);
  if (out_row0 < 0 || out_rows <= 0 || out_row0 + out_rows > g.out_h) return CSIC_EINVAL_ARG;
  const int f = p->factor;
  const bool avg = p->pool_mode == CSIC_POOL_AVERAGE && f > 1;
  int64_t lo = (int64_t)out_row0 * f;
  int64_t hi = (int64_t)(out_row0 + out_rows - 1) * f + (avg ? f - 1 : 0);   // inclusive
  const bool case_b = !g.chroma_first && f > 1;
  if (!case_b) {
    if (g.vf == 2 && (lo & 1)) lo -= 1;   // only possible for f == 1
  } else {
    // chroma runs on the decimated stream with full-size counters: walk the band's first and last
    // stream elements back to their sources (ImageCompressorTop.scala:52-58).
    const int64_t W = p->width, Wo = g.out_w;
    const int64_t last = ((W - 1) / g.hf) * g.hf;
    auto src_row = [&](int64_t m) {
      const int64_t col = m % W, line = (m / W) % p->height;
      const int64_t s = (g.vf == 2 && (line & 1)) ? (line - 1) * W + last : m - col % g.hf;
      return (s / Wo) * f;
    };
    lo = std::min(lo, src_row((int64_t)out_row0 * Wo));
    lo = std::min(lo, src_row((int64_t)out_row0 * Wo + Wo - 1));
  }
  hi = std::min<int64_t>(hi, p->height - 1);
  if (in_row0) *in_row0 = (int32_t)lo;
  if (in_rows) *in_rows = (int32_t)(hi - lo + 1);
  return CSIC_OK;
}

}  // extern "C"
