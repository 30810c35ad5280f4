// Dispatch of the pixel pipeline's kernels, written for sm_100a (B200), and the two kernels that are not TMA-staged.
// Every kernel is planned in csic_plan.cpp.  The staged kernels live in their own files:
//   csic_rows_kernel.cu    the hot path: packed RGB24 row segments through a shared-memory ring filled by the TMA engine
//                          (cp.async.bulk + mbarrier complete_tx), dp4a colour matrix, chroma hold inside the granule (or
//                          from one held pixel per row), quantise, pack, TMA bulk store.
//   csic_pool_kernel.cu    the AVERAGE extension, same machinery.
//   csic_flex_kernel.cu    DECIMATE for any width / pitch / alignment (hull fetch, staged span stores).
//   csic_decode_kernel.cu  the PLANAR decoder as flat tiles, any width.
// In this file:
//   csic_generic_kernel            a warp per output row, closed-form gather; any legal parameter set (odd sizes,
//                                  unaligned pointers, AVERAGE on dense odd widths, spatial-before-chroma shapes the
//                                  staged kernels exclude).  Not a fallback to the CPU: the independent second
//                                  implementation every other kernel is cross-checked against.
//   csic_expand_planar_any_kernel  LDG decoder for what csic_decode_kernel declines.
//
// Semantics (bit-exact with the reference; citations relative to its root, src/main/scala/jpeg/):
//   forward   RGB2YCbCr.scala:33-35,50-65,74-76 (FLOOR)   RGB2YCbCr.scala:95-121 (TRUNC)
//   chroma    ChromaSubsampler.scala:26-27,34-38,52-65      spatial  SpatialDownsampler.scala:17-55
//   quant     ColorQuantizer.scala:29-31,42-44              inverse  RGB2YCbCr.scala:123-132
//   order / misaligned counters   ImageCompressorTop.scala:43-58,83-114
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "csic_internal.h"
#include "csic_device_math.cuh"
#include "csic_tma.cuh"

namespace csic {

// ================================================================================================
// Generic gather kernel: any legal parameter set, any width, pitch and alignment
// ================================================================================================
// What runs when no staged kernel is eligible: spatial-before-chroma shapes whose counter lines are not whole output
// rows (e.g. W = 13, f = 2), the AVERAGE extension on shapes that break the pooling kernel's 16-byte rules -- and
// every parameter set when a test forces it (CSIC_OPT_KERNEL_FAMILY = 1), which makes it the independent second
// implementation the other kernels are cross-checked against.
//
// One WARP per output row (grid-stride) -- or, when a row has fewer than 32 granules, as many whole rows as fit its
// 32 lanes (a 96x96 frame pooled 8x8 has three granules per row: one row per CTA left 125 of 128 threads idle, 0.02 of
// the copy peak).  The frame / row split and, for case B, the split of the row into counter lines are the only
// divisions and happen once per row.  A thread computes one granule of four output slots:
//   load    every pixel is three bytes at an arbitrary address = two aligned LDG.32 and a funnel shift through L1 (the
//           second word never lies beyond the last word that holds a byte of the input); a thread's loads are all
//           independent, so a warp keeps 8 .. 200 of them in flight;
//   chroma  closed-form source maps of ChromaSubsampler.scala:52-65; case A resolves inside the granule (hold width
//           hfe divides 4), held lines replay one pixel per row; case B (ImageCompressorTop.scala:52-58) maps every
//           element through the full-size counters;
//   store   a warp's 32 granules are consecutive output bytes: staged in the warp's shared-memory slot at the output's
//           own offset modulo 16 and written as 16-byte st.global.cs aligned on the GLOBAL address (span_store); narrow
//           rows (several per warp) leave from registers with the widest stores their address allows (direct_store).
// Round 1's version -- one thread per slot, three divisions, byte loads and byte stores -- ran at 0.13 - 0.30 of the
// copy peak.

// A stored input row as the gather kernel addresses it: word-aligned base, byte phase of its first pixel, and the last
// word index a load may touch (the word holding the last byte this launch may read).  Set up once per row with 64-bit
// arithmetic; every pixel is then 32-bit offset arithmetic (round 2's first version did the 64-bit pointer math and
// the clamp per pixel: 382 warp-instructions per DECIMATE granule, now ~150).
struct GRow {
  const uint32_t* base;
  uint32_t a0, maxw;
};
__device__ __forceinline__ GRow grow_at(const uint8_t* p, const uint8_t* last_word) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  GRow r;
  r.base = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  r.a0 = (uint32_t)a & 3u;
  const uintptr_t lw = reinterpret_cast<uintptr_t>(last_word), ba = reinterpret_cast<uintptr_t>(r.base);
  r.maxw = lw >= ba ? (uint32_t)min((lw - ba) >> 2, (uintptr_t)0x3FFFFFFFu) : 0u;
  return r;
}
// three colour bytes (low three bytes of the result) at byte offset `off` of the row: two aligned LDG.32 through L1
// and a funnel shift; the second word is never fetched beyond GRow::maxw
__device__ __forceinline__ uint32_t grow_px(const GRow& r, uint32_t off) {
  const uint32_t o = r.a0 + off, wi = o >> 2;
  return __funnelshift_r(__ldg(r.base + wi), __ldg(r.base + min(wi + 1u, r.maxw)), (o & 3u) * 8u);
}

// Chroma source, in *output grid* coordinates, when the chroma stage runs on the downsampled stream
// but counts with the full W x H (ImageCompressorTop.scala:52-58).
__device__ __forceinline__ void chroma_src_case_b(const KPlan& P, int ro, int co, int& sro, int& sco) {
  const uint32_t m = (uint32_t)ro * (uint32_t)P.Wo + (uint32_t)co;
  const uint32_t line = m / (uint32_t)P.W;           // m < Wo * Ho <= W * H: the `% H` of the counters never wraps
  const uint32_t col = m - line * (uint32_t)P.W;
  uint32_t src;
  if (P.vf == 2 && (line & 1)) src = (line - 1) * (uint32_t)P.W + (uint32_t)P.last_sample_col;
  else src = m - (col % (uint32_t)P.hf);
  sro = (int)(src / (uint32_t)P.Wo);
  sco = (int)(src - (uint32_t)sro * (uint32_t)P.Wo);
}

constexpr uint32_t kGatherSlot = 32u * 16u + 32u;   // a warp's 32 granules of up to 16 bytes + alignment offset + read-ahead slack

// AF: 0 = DECIMATE (or f == 1); 2 / 4 / 8 = the AVERAGE extension with that factor (block loops unrolled)
template <bool TRUNC, int FMT, int AF>
__global__ void __launch_bounds__(128) csic_generic_kernel(const __grid_constant__ KPlan P) {
  __shared__ __align__(16) uint8_t stage[4][kGatherSlot];
  constexpr uint32_t kG = (FMT == KF_YCC888 || FMT == KF_RGB888) ? 12u : (FMT == KF_SLOT32 ? 16u : (FMT == KF_SLOT16 ? 8u : 4u));
  constexpr bool avg = AF > 1;
  constexpr uint32_t NR = avg ? (uint32_t)AF : 1u;                          // input rows per output row
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t Wo = (uint32_t)P.Wo, spr = (uint32_t)P.slots_per_row, gpr = (spr + 3u) >> 2;
  const uint32_t n_rows = P.n_frames * (uint32_t)P.band_rows;
  const uint32_t f = (uint32_t)P.f, ipb = (uint32_t)P.in_px_bytes, pxb = f * ipb;
  const uint32_t hfe = P.case_b ? 1u : (uint32_t)max(1, P.hf / P.f);         // case A: hold width inside a granule, in output pixels
  const uint32_t hfm = (uint32_t)P.hf - 1u;                                  // hf is 1, 2 or 4
  const uint32_t row_bytes = (FMT == KF_YCC888 || FMT == KF_RGB888) ? Wo * 3u : (FMT == KF_PLANAR ? Wo : spr * (uint32_t)P.slot_bytes);
  // last aligned word that still holds a byte this launch may read: the end of the band's last input row (the host
  // band path hands over buffers that hold only the band's rows)
  const uint32_t last_out_row = (uint32_t)(P.row0 + P.band_rows - 1);
  const uint32_t last_in_row = P.compact ? last_out_row : (avg ? (last_out_row + 1u) * f - 1u : last_out_row * f);
  const uint8_t* last_word = reinterpret_cast<const uint8_t*>(
      (reinterpret_cast<uintptr_t>(P.in) + (uint64_t)(P.n_frames - 1u) * P.in_frame_bytes + (uint64_t)last_in_row * P.in_row_bytes +
       (uint64_t)(uint32_t)P.W * ipb - 1u) & ~(uintptr_t)3);
  const uint32_t my = P.qmask & 0xFFu, mcb = (P.qmask >> 8) & 0xFFu, mcr = (P.qmask >> 16) & 0xFFu;
  const uint32_t sbase = smem_u32(stage[warp]);
  const int fsh = 31 - __clz(P.f);                                          // log2(f)

  // lanes -> (row of the warp's group, granule): wide rows take the whole warp, narrow ones share it
  const bool narrow = gpr < 32u;
  const uint32_t rpw = narrow ? 32u / gpr : 1u;                              // rows per warp and trip
  const uint32_t sub = narrow ? lane / gpr : 0u, gl = narrow ? lane - sub * gpr : lane;
  const uint32_t n_groups = (n_rows + rpw - 1u) / rpw, nwarps = blockDim.x >> 5;
  for (uint32_t grp = blockIdx.x * nwarps + warp; grp < n_groups; grp += gridDim.x * nwarps) {
    const uint32_t Rw = grp * rpw + sub;
    const bool row_ok = sub < rpw && Rw < n_rows;                            // lanes beyond the warp's last row idle (they still
    const uint32_t R = min(Rw, n_rows - 1u);                                 // compute, on a valid row, and store nothing)
    const uint32_t k = R / (uint32_t)P.band_rows, ro = (uint32_t)P.row0 + (R - k * (uint32_t)P.band_rows);
    const uint8_t* frame = P.in + (uint64_t)k * P.in_frame_bytes;
    uint8_t* fout = P.out + (uint64_t)k * P.out_frame_bytes;
    uint8_t* orow = fout + (uint64_t)ro * P.out_row_bytes;
    // stored row of a full-resolution row (KPlan::compact: only every f-th row is stored, DECIMATE reads no other)
    auto in_row = [&](uint32_t r) { return frame + (uint64_t)(P.compact ? (r >> fsh) : r) * P.in_row_bytes; };
    // the input rows of this output row: its own (DECIMATE) or the AF rows of its blocks (AVERAGE)
    GRow rows[NR];
#pragma unroll
    for (uint32_t dr = 0; dr < NR; ++dr) rows[dr] = grow_at(in_row(ro * f + dr), last_word);
    // Held chroma, one pixel per held line: DECIMATE case A on an odd full-resolution line of 4:2:0 / 4:1:0 (f == 1
    // only) replays the last sample point of the line above (ChromaSubsampler.scala:62-65); AVERAGE with the chroma
    // stage first does so for every odd line dr of the block rows.
    uint32_t hxb[NR / 2u + 1u], hxr[NR / 2u + 1u];
    const bool vheld = !P.case_b && P.vf == 2;
    const bool held_row = !avg && vheld && ((ro * f) & 1u);
#pragma unroll
    for (uint32_t h = 0; h < NR / 2u + 1u; ++h) { hxb[h] = 0u; hxr[h] = 0u; }
    if (held_row) {
      const GRow hr = grow_at(in_row(ro * f - 1u), last_word);
      const uint32_t hp = grow_px(hr, (uint32_t)P.last_sample_col * ipb);
      hxb[0] = fwd_nc16<TRUNC>(hp, P.coef_ncb); hxr[0] = fwd_nc16<TRUNC>(hp, P.coef_ncr);
    }
    if (avg && vheld) {
#pragma unroll
      for (int h = 0; h < (int)(NR / 2u); ++h) {                             // odd line 2h + 1 replays (2h, lastSampleCol)
        const uint32_t hp = grow_px(rows[2u * h], (uint32_t)P.last_sample_col * ipb);
        hxb[h] = fwd_nc16<TRUNC>(hp, P.coef_ncb); hxr[h] = fwd_nc16<TRUNC>(hp, P.coef_ncr);
      }
    }
    // Case B (spatial before chroma, DECIMATE): the chroma stage walks the DECIMATED stream with the full-size counters
    // (ImageCompressorTop.scala:52-58), so a counter line is W stream elements = W / Wo output rows, and an output row
    // lies in at most two lines (W >= Wo).  Per row: the column where the second line starts, and for each of the two
    // lines either its held pair (odd line, vf == 2: element (line-1) * W + lastSampleCol) or the phase of its hold
    // groups.  Per pixel nothing is divided any more.
    uint32_t cb_split = 0xFFFFFFFFu, cb_ph[1] = {0u}, cb_hxb[2] = {0u, 0u}, cb_hxr[2] = {0u, 0u};
    bool cb_held[2] = {false, false};
    GRow prev_row = rows[0];
    if (!avg && P.case_b) {
      const uint32_t m0 = ro * Wo, line0 = m0 / (uint32_t)P.W, col0 = m0 - line0 * (uint32_t)P.W;
      cb_split = (uint32_t)P.W - col0;                                       // first column of the row that lies in line0 + 1
#pragma unroll
      for (int l = 0; l < 2; ++l) {
        const uint32_t line = line0 + (uint32_t)l;
        if (l == 0) cb_ph[0] = col0 & hfm;                                   // (column in its line) mod hf of the row's first pixel; 0 for the second line
        if (P.vf == 2 && (line & 1u) && (l == 0 || cb_split < Wo)) {
          const uint32_t src = (line - 1u) * (uint32_t)P.W + (uint32_t)P.last_sample_col, sro = src / Wo, sco = src - sro * Wo;
          const GRow hr = grow_at(in_row(sro * f), last_word);
          const uint32_t hp = grow_px(hr, sco * pxb);
          cb_hxb[l] = fwd_nc16<TRUNC>(hp, P.coef_ncb); cb_hxr[l] = fwd_nc16<TRUNC>(hp, P.coef_ncr);
          cb_held[l] = true;
        }
      }
      if (ro > 0u) prev_row = grow_at(in_row((ro - 1u) * f), last_word);    // a hold group may start at the end of the row above
    }
    for (uint32_t g0 = 0; g0 < gpr; g0 += 32u) {                             // warp uniform; one trip when the rows are narrow
      const uint32_t g = narrow ? gl : g0 + lane, c0 = 4u * g;
      uint8_t* og = orow + (size_t)g0 * kG;                                  // first output byte of this warp's group
      const uint32_t st = sbase + ((uint32_t)reinterpret_cast<uintptr_t>(og) & 12u);
      if (g < gpr) {
        uint32_t y[4], cb[4], cr[4];                                         // final channel values (quantised)
        if (!avg) {
          uint32_t p[4], xb[4], xr[4];
          if (pxb == 3u && c0 + 3u < Wo) {                                   // f == 1, RGB24: twelve consecutive bytes
            const uint32_t o = rows[0].a0 + c0 * 3u, wi = o >> 2, sh = (o & 3u) * 8u;
            const uint32_t w0 = __ldg(rows[0].base + wi), w1 = __ldg(rows[0].base + wi + 1u), w2 = __ldg(rows[0].base + wi + 2u);
            const uint32_t w3 = __ldg(rows[0].base + min(wi + 3u, rows[0].maxw));
            const uint32_t v0 = __funnelshift_r(w0, w1, sh), v1 = __funnelshift_r(w1, w2, sh), v2 = __funnelshift_r(w2, w3, sh);
            p[0] = v0; p[1] = __funnelshift_r(v0, v1, 24); p[2] = __funnelshift_r(v1, v2, 16); p[3] = v2 >> 8;
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) p[j] = grow_px(rows[0], min(c0 + j, Wo - 1u) * pxb);
          }
          if (held_row) {
#pragma unroll
            for (int j = 0; j < 4; ++j) { xb[j] = hxb[0]; xr[j] = hxr[0]; }
          } else if (!P.case_b) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {                                    // sample where j % hfe == 0, hold in between
              if (j == 0 || ((uint32_t)j & (hfe - 1u)) == 0u) { xb[j] = fwd_nc16<TRUNC>(p[j], P.coef_ncb); xr[j] = fwd_nc16<TRUNC>(p[j], P.coef_ncr); }
              else { xb[j] = xb[j - 1]; xr[j] = xr[j - 1]; }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t co = min(c0 + j, Wo - 1u);
              const bool l = co >= cb_split;                                 // which of the row's two counter lines
              if (l ? cb_held[1] : cb_held[0]) {
                xb[j] = l ? cb_hxb[1] : cb_hxb[0]; xr[j] = l ? cb_hxr[1] : cb_hxr[0];
              } else {
                // sampled line: the pixel replays the first element of its hold group, (col - col % hf); the group may
                // begin in the row above (never further back: hf - 1 <= 3 elements; rows narrower than that divide)
                const uint32_t back = (l ? co - cb_split : co + cb_ph[0]) & hfm;
                uint32_t pc;
                if (back == 0u) pc = p[j];
                else if (back <= co) pc = grow_px(rows[0], (co - back) * pxb);
                else if (Wo + co >= back) pc = grow_px(prev_row, (Wo + co - back) * pxb);
                else {
                  int sro, sco;
                  chroma_src_case_b(P, (int)ro, (int)co, sro, sco);
                  pc = grow_px(grow_at(in_row((uint32_t)sro * f), last_word), (uint32_t)sco * pxb);
                }
                xb[j] = fwd_nc16<TRUNC>(pc, P.coef_ncb); xr[j] = fwd_nc16<TRUNC>(pc, P.coef_ncr);
              }
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            y[j] = (fwd_y16(p[j], P.coef_y) >> 8) & my;
            cb[j] = (~(xb[j] >> 8)) & mcb;
            cr[j] = (~(xr[j] >> 8)) & mcr;
          }
        } else {
          // AVERAGE extension: mean over the AF x AF block of the stream entering the spatial stage, round half up;
          // the quantiser before or after the mean as op[] says
          const uint32_t qy = P.quant_first ? my : 0xFFu, qb = P.quant_first ? mcb : 0xFFu, qr = P.quant_first ? mcr : 0xFFu;
          constexpr uint32_t half = (uint32_t)(AF * AF) >> 1, sh = AF == 2 ? 2u : (AF == 4 ? 4u : 6u);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t co = min(c0 + j, Wo - 1u), col0 = co * NR;
            uint32_t sy = 0, sb = 0, sr = 0;
            if (!P.case_b) {
#pragma unroll
              for (uint32_t dr = 0; dr < NR; ++dr) {
                const bool hl = vheld && (dr & 1u);       // nothing is sampled on an odd line: it replays the held pair
                uint32_t xb = hxb[dr >> 1], xr = hxr[dr >> 1];
                if (!hl && (col0 & hfm) != 0u) {          // the block starts inside a hold group (hf > AF): its sample lies to the left
                  const uint32_t pc = grow_px(rows[dr], (col0 & ~hfm) * ipb);
                  xb = fwd_nc16<TRUNC>(pc, P.coef_ncb); xr = fwd_nc16<TRUNC>(pc, P.coef_ncr);
                }
#pragma unroll
                for (uint32_t dc = 0; dc < NR; ++dc) {
                  const uint32_t pv = grow_px(rows[dr], (col0 + dc) * ipb);
                  sy += (fwd_y16(pv, P.coef_y) >> 8) & qy;
                  if (!hl && ((col0 + dc) & hfm) == 0u) { xb = fwd_nc16<TRUNC>(pv, P.coef_ncb); xr = fwd_nc16<TRUNC>(pv, P.coef_ncr); }
                  sb += (~(xb >> 8)) & qb; sr += (~(xr >> 8)) & qr;
                }
              }
            } else {
              // pooling first: the chroma stage then samples the POOLED stream with the full-size counters, i.e. this
              // pixel takes the pooled chroma of block (bro, bco) (ImageCompressorTop.scala:52-58)
              int bro, bco;
              chroma_src_case_b(P, (int)ro, (int)co, bro, bco);
#pragma unroll
              for (uint32_t dr = 0; dr < NR; ++dr) {
                const GRow cr_ = grow_at(in_row((uint32_t)bro * f + dr), last_word);
#pragma unroll
                for (uint32_t dc = 0; dc < NR; ++dc) {
                  sy += (fwd_y16(grow_px(rows[dr], (col0 + dc) * ipb), P.coef_y) >> 8) & qy;
                  const uint32_t pc = grow_px(cr_, ((uint32_t)bco * NR + dc) * ipb);
                  sb += (~(fwd_nc16<TRUNC>(pc, P.coef_ncb) >> 8)) & qb; sr += (~(fwd_nc16<TRUNC>(pc, P.coef_ncr) >> 8)) & qr;
                }
              }
            }
            y[j] = (sy + half) >> sh; cb[j] = (sb + half) >> sh; cr[j] = (sr + half) >> sh;
            if (!P.quant_first) { y[j] &= my; cb[j] &= mcb; cr[j] &= mcr; }
          }
        }
        // ---- pack the granule: into the warp's staging slot, or (narrow rows) straight to global memory ----
        const uint32_t so = st + kG * lane;
        uint8_t* gp = orow + (size_t)g * kG;
        const uint32_t gbytes = min(kG, row_bytes - g * kG);                  // the row's last granule may be partial
        uint32_t ww[kG / 4u];
        if (FMT == KF_YCC888 || FMT == KF_RGB888) {
          uint32_t v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            v[j] = FMT == KF_RGB888 ? inverse_rgb((int)y[j], (int)cb[j], (int)cr[j]) : (y[j] | (cb[j] << 8) | (cr[j] << 16));
          pack_rgb_granule(v, ww[0], ww[1], ww[2]);
        } else if (FMT == KF_PLANAR) {
          ww[0] = y[0] | (y[1] << 8) | (y[2] << 16) | (y[3] << 24);
          if (row_ok && ro % (uint32_t)P.planar_vs == 0u) {                  // surviving chroma sample points of this row
            const size_t crow = (size_t)(ro / (uint32_t)P.planar_vs) * (size_t)P.planar_cw;
#pragma unroll
            for (uint32_t j = 0; j < 4u; ++j)
              if ((j & ((uint32_t)P.planar_hs - 1u)) == 0u && c0 + j < Wo) {
                fout[P.planar_cb_off + crow + (c0 + j) / (uint32_t)P.planar_hs] = (uint8_t)cb[j];
                fout[P.planar_cr_off + crow + (c0 + j) / (uint32_t)P.planar_hs] = (uint8_t)cr[j];
              }
          }
        } else {
          uint32_t v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            v[j] = (c0 + j < Wo) ? ((y[j] >> P.sy) << (P.cb_bits + P.cr_bits)) | ((cb[j] >> P.scb) << P.cr_bits) | (cr[j] >> P.scr)
                                 : 0u;                                        // BUNDLE row padding: zero slots
          if (FMT == KF_SLOT32) { ww[0] = v[0]; ww[kG / 4u > 1u ? 1 : 0] = v[1]; ww[kG / 4u > 2u ? 2 : 0] = v[2]; ww[kG / 4u > 3u ? 3 : 0] = v[3]; }
          else if (FMT == KF_SLOT16) { ww[0] = v[0] | (v[1] << 16); ww[kG / 4u > 1u ? 1 : 0] = v[2] | (v[3] << 16); }
          else ww[0] = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
        }
        if (narrow) {
          if (row_ok) direct_store(gp, ww, gbytes);
        } else {
#pragma unroll
          for (uint32_t i = 0; i < kG / 4u; ++i) sts32(so + 4u * i, ww[i]);
        }
      }
      if (narrow) break;                                                     // the rows of this trip are done
      __syncwarp();
      span_store(og, st, min(32u * kG, row_bytes - g0 * kG), lane, 32u);   // the row's last granule may be partial
      __syncwarp();
    }
  }
}

// Decoder of the PLANAR format for ANY width and any alignment of the planes and of the output: chroma fetched with the
// reference's replay rule (ChromaSubsampler.scala:52-65) expressed in output coordinates (chroma before spatial, or
// f == 1).  One CTA per output row segment of up to 4096 pixels; the only division (frame / row split) and everything
// row-dependent happen once per row.
//   load   a thread takes up to four granules of four pixels and issues ALL their loads first (Y word, Cb and Cr
//          samples: aligned LDG.32 pairs + funnel shifts on per-row word bases, 32-bit offsets), so a warp keeps ~24
//          loads in flight instead of 3;
//   store  the whole segment is staged in shared memory at the output's own offset modulo 16 (rounded down to a
//          word) and leaves as 16-byte st.global.cs aligned on the GLOBAL address (span_store): one head and one tail
//          of < 16 bytes per row instead of one per 384 bytes.
// Round 1: one thread per pixel, three divisions, three byte loads and three byte stores each -- 0.10 of the copy
// peak; the first round-2 version (one granule per thread and trip, per-warp staging) 0.22; this one 0.4 - 0.5.  Since
// the TMA-staged decoder (csic_decode_kernel.cu: 0.6 - 0.95) it only runs what that kernel declines, and under
// CSIC_DEC_NO_TMA in the tests.
constexpr uint32_t kExpandSeg = 4096u;   // pixels per staged segment: 12 KB of shared memory

__global__ void __launch_bounds__(128) csic_expand_planar_any_kernel(const __grid_constant__ KPlan P, const uint8_t* __restrict__ planar,
                                                                     uint8_t* __restrict__ out, int to_rgb) {
  __shared__ __align__(16) uint8_t stage[kExpandSeg * 3u + 48u];      // + alignment offset + read-ahead slack of span_store
  const uint32_t Wo = (uint32_t)P.Wo, tid = threadIdx.x, NT = blockDim.x;
  const uint32_t n_rows = P.n_frames * (uint32_t)P.Ho;
  const uint32_t last_c = (uint32_t)((P.last_sample_col / P.f) / P.planar_hs);   // plane column of a line's last sample point
  const uint32_t hs_sh = P.planar_hs == 4 ? 2u : (P.planar_hs == 2 ? 1u : 0u), vs_sh = P.planar_vs == 2 ? 1u : 0u;
  const uint32_t csel = hs_sh == 0 ? 0x3210u : (hs_sh == 1 ? 0x1100u : 0x0000u);   // sample bytes -> the four pixels of a granule
  const bool vhold = P.vf == 2 && P.f == 1;                         // odd lines replay the line above (f == 1 only)
  // last aligned word that still holds a byte of the planar buffer (loads never go past it)
  const uint8_t* last_word = reinterpret_cast<const uint8_t*>(
      (reinterpret_cast<uintptr_t>(planar) + (uint64_t)P.n_frames * P.out_frame_bytes - 1u) & ~(uintptr_t)3);
  const uint32_t sbase = smem_u32(stage);
  for (uint32_t R = blockIdx.x; R < n_rows; R += gridDim.x) {
    const uint32_t k = R / (uint32_t)P.Ho, ro = R - k * (uint32_t)P.Ho;
    const uint8_t* fr = planar + (uint64_t)k * P.out_frame_bytes;
    const bool held = vhold && (ro & 1u);
    const size_t crow = (size_t)((held ? ro - 1u : ro) >> vs_sh) * (size_t)P.planar_cw;
    const GRow yr = grow_at(fr + (size_t)ro * Wo, last_word);
    const GRow br = grow_at(fr + P.planar_cb_off + crow, last_word), rr = grow_at(fr + P.planar_cr_off + crow, last_word);
    uint8_t* orow = out + (uint64_t)R * Wo * 3u;
    uint32_t hcb = 0, hcr = 0;
    if (held) { hcb = (grow_px(br, last_c) & 0xFFu) * 0x01010101u; hcr = (grow_px(rr, last_c) & 0xFFu) * 0x01010101u; }
    for (uint32_t seg0 = 0; seg0 < Wo; seg0 += kExpandSeg) {
      const uint32_t npx = min(kExpandSeg, Wo - seg0), ngr = (npx + 3u) >> 2;
      uint8_t* og = orow + (size_t)seg0 * 3u;
      const uint32_t st = sbase + ((uint32_t)reinterpret_cast<uintptr_t>(og) & 12u);
      for (uint32_t g0 = tid; g0 < ngr; g0 += 4u * NT) {
        // All the loads of up to four granules first, as bare LDGs on clamped indices: no branch and no dependent
        // instruction between them (a funnel shift right behind its two loads stalls the warp -- the GPU issues in
        // order -- and the next granule's loads with it: ncu showed 11.7 long-scoreboard stalls per issue that way).
        uint32_t yl[4], yh[4], bl[4], bh[4], rl[4], rh[4];
        const uint32_t oc0 = seg0 >> hs_sh;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t g = min(g0 + (uint32_t)u * NT, ngr - 1u);
          const uint32_t wy = (yr.a0 + seg0 + 4u * g) >> 2;
          yl[u] = __ldg(yr.base + wy); yh[u] = __ldg(yr.base + min(wy + 1u, yr.maxw));
        }
        if (!held) {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t g = min(g0 + (uint32_t)u * NT, ngr - 1u), cs = oc0 + ((4u * g) >> hs_sh);
            const uint32_t wb = (br.a0 + cs) >> 2, wr = (rr.a0 + cs) >> 2;
            bl[u] = __ldg(br.base + wb); bh[u] = __ldg(br.base + min(wb + 1u, br.maxw));
            rl[u] = __ldg(rr.base + wr); rh[u] = __ldg(rr.base + min(wr + 1u, rr.maxw));
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t g = g0 + (uint32_t)u * NT;
          if (g < ngr) {
            const uint32_t cs = oc0 + ((4u * g) >> hs_sh);
            const uint32_t yw = __funnelshift_r(yl[u], yh[u], ((yr.a0 + seg0 + 4u * g) & 3u) * 8u);
            uint32_t cbw = hcb, crw = hcr;
            if (!held) {
              cbw = __byte_perm(__funnelshift_r(bl[u], bh[u], ((br.a0 + cs) & 3u) * 8u), 0, csel);
              crw = __byte_perm(__funnelshift_r(rl[u], rh[u], ((rr.a0 + cs) & 3u) * 8u), 0, csel);
            }
            uint32_t w0, w1, w2;
            decode_granule(yw, cbw, crw, held ? 2u : hs_sh, to_rgb, w0, w1, w2);
            sts32(st + 12u * g, w0); sts32(st + 12u * g + 4u, w1); sts32(st + 12u * g + 8u, w2);
          }
        }
      }
      __syncthreads();
      span_store(og, st, npx * 3u, tid, NT);                           // the row's last granule may hold fewer than four pixels
      __syncthreads();
    }
  }
}

int launch_expand_planar(const KPlan& k, int to_rgb, int sm_count, void* stream) {
  const uint64_t total = (uint64_t)k.n_frames * (uint64_t)k.Ho * (uint64_t)k.Wo;
  if (total == 0) return (int)cudaSuccess;
  const uint64_t n_rows = (uint64_t)k.n_frames * (uint64_t)k.Ho;
  if (n_rows >= (1ull << 32)) return (int)cudaErrorInvalidValue;
  const unsigned threads = (unsigned)std::min<uint32_t>(128u, ((((uint32_t)k.Wo + 3u) >> 2) + 31u) & ~31u);
  const unsigned blocks = (unsigned)std::min<uint64_t>(n_rows, (uint64_t)sm_count * (2048u / threads));
  csic_expand_planar_any_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(k, k.in, k.out, to_rgb);
  return (int)cudaGetLastError();
}

namespace {
template <int FMT, int AF>
KernelFn generic_by_trunc(bool trunc) { return trunc ? csic_generic_kernel<true, FMT, AF> : csic_generic_kernel<false, FMT, AF>; }
template <int FMT>
KernelFn generic_by_af(int af, bool trunc) {
  switch (af) {
    case 2: return generic_by_trunc<FMT, 2>(trunc);
    case 4: return generic_by_trunc<FMT, 4>(trunc);
    case 8: return generic_by_trunc<FMT, 8>(trunc);
    default: return generic_by_trunc<FMT, 0>(trunc);
  }
}
// af: the AVERAGE factor, 0 for DECIMATE (see csic_generic_kernel)
KernelFn generic_kernel(int kformat, int af, bool trunc) {
  switch (kformat) {
    case KF_YCC888: return generic_by_af<KF_YCC888>(af, trunc);
    case KF_RGB888: return generic_by_af<KF_RGB888>(af, trunc);
    case KF_SLOT8: return generic_by_af<KF_SLOT8>(af, trunc);
    case KF_SLOT16: return generic_by_af<KF_SLOT16>(af, trunc);
    case KF_PLANAR: return generic_by_af<KF_PLANAR>(af, trunc);
    default: return generic_by_af<KF_SLOT32>(af, trunc);
  }
}

// the per-factor instances of the row and pooling kernels (compiled one file per factor)
KernelFn rows_for(int f, int kformat, bool q8, bool trunc) {
  switch (f) {
    case 1: return rows_kernel<1>(kformat, q8, trunc);
    case 2: return rows_kernel<2>(kformat, q8, trunc);
    case 4: return rows_kernel<4>(kformat, q8, trunc);
    default: return rows_kernel<8>(kformat, q8, trunc);
  }
}

KernelFn pool_for(int f, int kformat, bool in4) {
  switch (f) {
    case 2: return pool_kernel<2>(kformat, in4);
    case 4: return pool_kernel<4>(kformat, in4);
    default: return pool_kernel<8>(kformat, in4);
  }
}
}  // namespace

int launch(const KernelChoice& c, void* stream) {
  const KPlan& k = c.k;
  KernelFn fn;
  unsigned threads = (unsigned)k.block_threads + 32u;   // + producer warp
  size_t smem = k.smem_bytes;
  switch (c.family) {
    case FAM_ROWS: fn = rows_for(k.f, k.kformat, k.sy == 0 && k.scb == 0 && k.scr == 0, k.trunc != 0); break;
    case FAM_POOL: fn = pool_for(k.f, k.kformat, k.in_px_bytes == 4); break;
    case FAM_FLEX: fn = flex_kernel(k.kformat, k.trunc != 0); break;
    default:
      if (c.grid == 0) return (int)cudaSuccess;
      if ((uint64_t)k.n_frames * (uint64_t)k.band_rows >= (1ull << 32)) return (int)cudaErrorInvalidValue;
      fn = generic_kernel(k.kformat, k.average && k.f > 1 ? k.f : 0, k.trunc != 0);
      threads = 128u;   // four warps per CTA
      smem = 0;
  }
  fn<<<c.grid, threads, smem, (cudaStream_t)stream>>>(k);
  return (int)cudaGetLastError();
}

// Raises the dynamic shared-memory limit of every instance of the TMA-staged kernels (the generic and LDG kernels use
// static shared memory only).  Keys that select the same instance set it twice.
int set_kernel_attributes(size_t max_smem_optin) {
  cudaError_t e = cudaSuccess;
  auto set = [&](auto fn) {
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem_optin);
  };
  for (int fmt = KF_YCC888; fmt <= KF_PLANAR; ++fmt)
    for (const bool a : {false, true}) {
      for (const bool b : {false, true})
        for (const int f : {1, 2, 4, 8}) set(rows_for(f, fmt, a, b));
      for (const int f : {2, 4, 8}) set(pool_for(f, fmt, a));
      set(flex_kernel(fmt, a));
    }
  for (uint32_t hs_sh = 0; hs_sh < 3; ++hs_sh)
    for (const bool vhold : {false, true})
      for (const bool to_rgb : {false, true}) set(decode_kernel(hs_sh, vhold, to_rgb));
  return (int)e;
}

}  // namespace csic
