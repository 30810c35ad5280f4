// The TMA-staged row kernel and its launchers for ONE spatial factor F = CSIC_ROWS_F.
// build.sh compiles this file four times (F = 1, 2, 4, 8) in parallel.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "csic_internal.h"
#include "csic_device_math.cuh"
#include "csic_tma.cuh"

#ifndef CSIC_ROWS_F
#error "compile with -DCSIC_ROWS_F=1|2|4|8"
#endif

namespace csic {

// ================================================================================================
// TMA-staged row kernel
// ================================================================================================
// IN4: 4-byte input pixels (RGBA32 / BGRA32); every pixel is an aligned word, the fourth byte meets a zero
// coefficient.  Granule = 16F bytes.
template <int F, bool IN4>
__device__ __forceinline__ void load_granule(uint32_t a, uint32_t (&p)[4]) {
  if (IN4) {
    if (F == 1) {
      const uint4 v = lds128(a);
      p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
    } else if (F == 2) {
      const uint4 v = lds128(a), w = lds128(a + 16);
      p[0] = v.x; p[1] = v.z; p[2] = w.x; p[3] = w.z;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) p[j] = lds32(a + j * 4u * F);
    }
    return;
  }
  if (F == 1) {                                  // 12 bytes; word stride 3 across lanes: conflict free
    const uint32_t w0 = lds32(a), w1 = lds32(a + 4), w2 = lds32(a + 8);
    p[0] = w0;
    p[1] = __funnelshift_r(w0, w1, 24);
    p[2] = __funnelshift_r(w1, w2, 16);
    p[3] = w2 >> 8;
  } else if (F == 2) {                           // 24 bytes, 8-byte aligned; conflict free per half warp
    const uint2 u0 = lds64(a), u1 = lds64(a + 8), u2 = lds64(a + 16);
    p[0] = u0.x;                                 // bytes 0..2
    p[1] = __funnelshift_r(u0.y, u1.x, 16);      // bytes 6..8
    p[2] = u1.y;                                 // bytes 12..14
    p[3] = __funnelshift_r(u2.x, u2.y, 16);      // bytes 18..20
  } else {                                       // pixels sit on word boundaries
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = lds32(a + j * 3u * F);
  }
}

// Per-stage tile descriptor: written by the producer thread before it arms the stage's mbarrier
// (release), read by every thread after the barrier's phase flips (acquire).
struct TileMeta {
  uint64_t out_base;                 // global address of the tile's first output byte
  uint32_t n_granules;               // rows * granules per row segment
  uint32_t any_held_col0;            // bit 31: some row replays a held chroma pair; bits 0..30: first output column
  uint64_t cb_base, cr_base;         // PLANAR: global address of the tile's first Cb / Cr row (bits 24.. of n_granules: #rows)
  uint32_t held_addr[kMaxTileRows];  // per row: 0, or shared address of the RGB pixel whose chroma the row replays
};
static_assert(sizeof(TileMeta) == kTileMetaBytes, "kTileMetaBytes out of sync");

// Runtime constants of the inner loop, hoisted into registers once per kernel.
struct LoopConst {
  uint32_t qm0, qm1, qm2;            // YCC888: quantiser keep-masks over the three packed words
  uint32_t my, mcb, mcr;             // RGB888
  int shy, shb, shr, ly, lb;         // bundles
  uint32_t coef_y, coef_ncb, coef_ncr;       // dp4a coefficient words (byte order of the input pixels)
  uint32_t gran_per_row;
  uint32_t out_pitch, out_dense, ragged, Wo;  // pitched / padded output rows (see KPlan)
  uint32_t pl_cb_off, pl_cr_off, pl_crow_bytes, pl_vs_shift;   // PLANAR staging: region offsets, bytes per chroma row
  uint32_t nthreads;                         // consumer threads per CTA
  uint32_t row0_of_thread, rem0_of_thread;   // threadIdx.x / gran_per_row, threadIdx.x % gran_per_row
  uint32_t drow, drem;                       // blockDim.x / gran_per_row, blockDim.x % gran_per_row
};

// One tile: a flat loop over its granules.  Rows are packed back to back in the stage (and, for the
// staged formats, in the output buffer), so granule q lives at  base + q * granule_bytes  and the row
// index is only needed to look up a held chroma pair (HELD tiles).
//   HFE   chroma hold width inside a granule, in output pixels (1, 2 or 4)
//   HELD  the tile may contain rows that replay a held pair (odd 4:2:0 / 4:1:0 lines)
//   Q8    8/8/8 bits in a 32-bit slot: pure byte permutes
template <int F, int FMT, int HFE, bool HELD, bool Q8, bool TRUNC, bool IN4>
__device__ __forceinline__ void tile_loop(uint32_t in_s, uint32_t out_s, uint8_t* __restrict__ out_g,
                                          const TileMeta* __restrict__ meta, const LoopConst& C) {
  const uint32_t n = meta->n_granules & 0x00FFFFFFu;
  uint32_t row = C.row0_of_thread, rem = C.rem0_of_thread;   // row of granule q, tracked without a division
  for (uint32_t q = threadIdx.x; q < n; q += C.nthreads) {
    uint32_t p[4];
    load_granule<F, IN4>(in_s + q * ((IN4 ? 16u : 12u) * F), p);
    uint32_t dy[4], xb[4], xr[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) dy[j] = fwd_y16(p[j], C.coef_y);
    uint32_t haddr = 0;
    if (HELD) haddr = meta->held_addr[row];
    // byte offset of this granule's output inside the tile: rows are back to back unless the output is pitched
    const uint32_t orow = row, orem = rem;
    row += C.drow;
    rem += C.drem;
    if (rem >= C.gran_per_row) { rem -= C.gran_per_row; ++row; }
    if (FMT == KF_RGB888) {
      // fused reconstruction: the chroma-only part of YCbCr2RGB is computed per chroma SAMPLE inside each branch
      // (once per granule on a held row, every HFE-th pixel otherwise), the per-pixel part in emit()
      const uint32_t my8 = C.my << 8, mcb8 = C.mcb << 8, mcr8 = C.mcr << 8;
      const uint32_t a = out_s + q * 12u;
      // the chroma terms are chosen inside the branch, the per-pixel part runs once behind it: warps of narrow frames
      // straddle a held and a sampled row, and would otherwise execute the (long) per-pixel part twice
      InvChroma t[4];
      if (HELD && haddr != 0) {
        const uint32_t hp = lds8(haddr) | (lds8(haddr + 1) << 8) | (lds8(haddr + 2) << 16);
        t[0] = inv_chroma_terms(fwd_nc16<TRUNC>(hp, C.coef_ncb), fwd_nc16<TRUNC>(hp, C.coef_ncr), mcb8, mcr8);
        t[1] = t[0]; t[2] = t[0]; t[3] = t[0];
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j % HFE == 0) t[j] = inv_chroma_terms(fwd_nc16<TRUNC>(p[j], C.coef_ncb), fwd_nc16<TRUNC>(p[j], C.coef_ncr), mcb8, mcr8);
          else t[j] = t[j - 1];
        }
      }
      uint32_t w0, w1, w2;
      inv_granule(dy, my8, t[0], t[1], t[2], t[3], w0, w1, w2);
      sts32(a, w0); sts32(a + 4, w1); sts32(a + 8, w2);
      continue;
    }
    if (HELD && haddr != 0) {
      const uint32_t hp = lds8(haddr) | (lds8(haddr + 1) << 8) | (lds8(haddr + 2) << 16);
      const uint32_t hb = fwd_nc16<TRUNC>(hp, C.coef_ncb), hr = fwd_nc16<TRUNC>(hp, C.coef_ncr);
#pragma unroll
      for (int j = 0; j < 4; ++j) { xb[j] = hb; xr[j] = hr; }
    } else {
      // sample where j % HFE == 0, hold in between (ChromaSubsampler.scala:57-65)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j % HFE == 0) {
          xb[j] = fwd_nc16<TRUNC>(p[j], C.coef_ncb);
          xr[j] = fwd_nc16<TRUNC>(p[j], C.coef_ncr);
        } else {
          xb[j] = xb[j - 1];
          xr[j] = xr[j - 1];
        }
      }
    }

    if (FMT == KF_PLANAR) {
      // Y plane: four Y bytes per granule.  Chroma planes: only sampled lines contribute, 4/HFE samples each.
      const uint32_t my4 = C.my * 0x01010101u, mb4 = C.mcb * 0x01010101u, mr4 = C.mcr * 0x01010101u;
      const uint32_t yw = __byte_perm(__byte_perm(dy[0], dy[1], 0x0051), __byte_perm(dy[2], dy[3], 0x0051), 0x5410) & my4;
      sts32(out_s + q * 4u, yw);
      if (!(HELD && haddr != 0)) {
        const uint32_t crow = (orow >> C.pl_vs_shift) * C.pl_crow_bytes;
        if (HFE == 1) {
          const uint32_t bw = ~__byte_perm(__byte_perm(xb[0], xb[1], 0x0051), __byte_perm(xb[2], xb[3], 0x0051), 0x5410) & mb4;
          const uint32_t rw = ~__byte_perm(__byte_perm(xr[0], xr[1], 0x0051), __byte_perm(xr[2], xr[3], 0x0051), 0x5410) & mr4;
          sts32(out_s + C.pl_cb_off + crow + orem * 4u, bw);
          sts32(out_s + C.pl_cr_off + crow + orem * 4u, rw);
        } else if (HFE == 2) {
          const uint32_t bw = ~__byte_perm(xb[0], xb[2], 0x0051) & mb4 & 0xFFFFu;
          const uint32_t rw = ~__byte_perm(xr[0], xr[2], 0x0051) & mr4 & 0xFFFFu;
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(out_s + C.pl_cb_off + crow + orem * 2u), "h"((unsigned short)bw) : "memory");
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(out_s + C.pl_cr_off + crow + orem * 2u), "h"((unsigned short)rw) : "memory");
        } else {
          const uint32_t bw = (~(xb[0] >> 8)) & C.mcb, rw = (~(xr[0] >> 8)) & C.mcr;
          asm volatile("st.shared.u8 [%0], %1;" ::"r"(out_s + C.pl_cb_off + crow + orem), "r"(bw) : "memory");
          asm volatile("st.shared.u8 [%0], %1;" ::"r"(out_s + C.pl_cr_off + crow + orem), "r"(rw) : "memory");
        }
      }
    } else if (FMT == KF_YCC888) {
      // byte 1 of dy is Y, byte 1 of xb/xr is ~Cb/~Cr: gather with PRMT, flip and quantise per word.
      uint32_t t, u;
      t = __byte_perm(dy[0], xb[0], 0x0051); u = __byte_perm(xr[0], dy[1], 0x0051);
      const uint32_t w0 = (__byte_perm(t, u, 0x5410) ^ 0x00FFFF00u) & C.qm0;
      t = __byte_perm(xb[1], xr[1], 0x0051); u = __byte_perm(dy[2], xb[2], 0x0051);
      const uint32_t w1 = (__byte_perm(t, u, 0x5410) ^ 0xFF00FFFFu) & C.qm1;
      t = __byte_perm(xr[2], dy[3], 0x0051); u = __byte_perm(xb[3], xr[3], 0x0051);
      const uint32_t w2 = (__byte_perm(t, u, 0x5410) ^ 0xFFFF00FFu) & C.qm2;
      const uint32_t a = out_s + q * 12u;
      sts32(a, w0); sts32(a + 4, w1); sts32(a + 8, w2);
    } else {
      // bundle slots go straight to global memory: one coalesced 4/8/16-byte store per granule
      uint32_t v[4];
      if (Q8) {
#pragma unroll
        for (int j = 0; j < 4; ++j)   // (Cr, Cb, Y, 0): dy < 65536 so its byte 3 is the zero pad
          v[j] = __byte_perm(__byte_perm(xr[j], xb[j], 0x0051), dy[j], 0x7510) ^ 0x0000FFFFu;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          v[j] = ((dy[j] >> C.shy) << C.ly) | (((xb[j] ^ 0xFFFFu) >> C.shb) << C.lb) | ((xr[j] ^ 0xFFFFu) >> C.shr);
      }
      if (C.ragged) {                 // padded columns (>= Wo) are the row's zero pad slots
        const uint32_t co = (meta->any_held_col0 & 0x7FFFFFFFu) + orem * 4u;
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (co + j < C.Wo) ? v[j] : 0u;
      }
      constexpr uint32_t kG = (FMT == KF_SLOT32) ? 16u : (FMT == KF_SLOT16 ? 8u : 4u);
      if (F == 1 && FMT == KF_SLOT32) {   // staged like the 3-byte formats: rows back to back in the output buffer, TMA store per tile
        const uint32_t a = out_s + q * kG;
        if (FMT == KF_SLOT32) asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
        else if (FMT == KF_SLOT16) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(v[0] | (v[1] << 16)), "r"(v[2] | (v[3] << 16)) : "memory");
        else sts32(a, v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24));
        continue;
      }
      uint8_t* dst = out_g + (C.out_dense ? q * kG : orow * C.out_pitch + orem * kG);
      if (FMT == KF_SLOT32) __stcs(reinterpret_cast<uint4*>(dst), make_uint4(v[0], v[1], v[2], v[3]));
      else if (FMT == KF_SLOT16) __stcs(reinterpret_cast<uint2*>(dst), make_uint2(v[0] | (v[1] << 16), v[2] | (v[3] << 16)));
      else __stcs(reinterpret_cast<uint32_t*>(dst), v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24));
    }
  }
}

// Per-tile specialisation: hold width, held rows, input pixel size.
template <int F, int FMT, bool Q8, bool TRUNC, bool IN4>
__device__ __forceinline__ void tile_dispatch(bool held, int hfe, uint32_t in_s, uint32_t out_s, uint8_t* out_g,
                                              const TileMeta* m, const LoopConst& C) {
  if (held) {
    if (hfe == 1) tile_loop<F, FMT, 1, true, Q8, TRUNC, IN4>(in_s, out_s, out_g, m, C);
    else if (hfe == 2) tile_loop<F, FMT, 2, true, Q8, TRUNC, IN4>(in_s, out_s, out_g, m, C);
    else tile_loop<F, FMT, 4, true, Q8, TRUNC, IN4>(in_s, out_s, out_g, m, C);
  } else {
    if (hfe == 1) tile_loop<F, FMT, 1, false, Q8, TRUNC, IN4>(in_s, out_s, out_g, m, C);
    else if (hfe == 2) tile_loop<F, FMT, 2, false, Q8, TRUNC, IN4>(in_s, out_s, out_g, m, C);
    else tile_loop<F, FMT, 4, false, Q8, TRUNC, IN4>(in_s, out_s, out_g, m, C);
  }
}

template <int F, int FMT, bool Q8, bool TRUNC>
__global__ void __launch_bounds__(kMaxConsumerThreads + 32) csic_rows_kernel(const __grid_constant__ KPlan P) {
  extern __shared__ __align__(128) uint8_t smem[];
  // output leaves through smem + TMA store: the 3-byte formats, PLANAR, and 32-bit bundle slots at F == 1 (plan_rows_kernel)
  constexpr bool kStaged = (FMT == KF_YCC888 || FMT == KF_RGB888 || FMT == KF_PLANAR) || (F == 1 && FMT == KF_SLOT32);
  constexpr uint32_t kGranOut = (FMT == KF_PLANAR || FMT == KF_SLOT8) ? 4u : (FMT == KF_SLOT16 ? 8u : (FMT == KF_SLOT32 ? 16u : 12u));
  const uint32_t tid = threadIdx.x;
  const uint32_t NC = blockDim.x - 32u;        // consumer threads; the last warp is the producer
  const uint32_t sbase = smem_u32(smem);
  const uint64_t pol = policy_evict_first();   // every byte is touched exactly once: do not keep it in L2
  const Ring ring(sbase + P.bar_off, (uint32_t)P.stages, P.n_tiles);
  ring.init(NC / 32u);                          // one arrive per consumer warp

  // ============================== producer warp ==============================================
  // Walks this CTA's tiles S deep ahead of the consumers.  All lanes track the geometry; the per-row work of a tile
  // (where a held row finds its chroma, the row's own bulk copy when rows are not contiguous) is spread over the
  // lanes -- a tile of small frames has up to 64 rows -- and every lane announces its copies on the stage's mbarrier
  // (expect_tx); lane 0 describes the tile in TileMeta and arrives once for the warp.
  if (tid >= NC) {
    const uint32_t lane = tid - NC;
    const uint32_t ipb = (uint32_t)P.in_px_bytes;
    const bool one_copy = P.row_step == 1 && P.nsplit == 1 && P.in_dense;   // consecutive rows are contiguous in memory
    for (uint32_t i = 0; i < ring.n_my; ++i) {
      const Ring::Pos pos = ring.at(i);
      ring.wait_empty(pos, i);
      const RowTile t = row_tile(P, blockIdx.x + i * gridDim.x);
      const uint32_t s = pos.s, seg = t.seg, k = t.k, ro0 = t.ro0, nrows = t.nrows;
      const uint8_t* frame = P.in + (uint64_t)k * P.in_frame_bytes;
      const uint32_t bar = ring.full(s);
      const uint32_t dst = sbase + s * P.stage_stride;
      const uint32_t aux = dst + (uint32_t)P.tile_rows * P.tile_in_bytes;    // 32-byte window per row
      TileMeta* m = reinterpret_cast<TileMeta*>(smem + P.meta_off) + s;
      const uint8_t* src = frame + (uint64_t)(ro0 * (uint32_t)P.row_step) * P.in_row_bytes + (uint64_t)seg * P.tile_in_bytes;

      // Which rows replay a held chroma pair, and from where?  (KPlan::hfe covers the in-row hold.)
      uint32_t any = 0;
      for (uint32_t j = lane; j < nrows; j += 32u) {
        if (P.vf == 2) {
          const uint32_t ro = ro0 + j;
          uint32_t h = 0;
          const uint8_t* hp = nullptr;
          if (!P.case_b) {
            if (F == 1 && (ro & 1)) {          // odd line at full resolution: last sample point of the line above
              if (j > 0 && P.nsplit == 1) h = dst + (j - 1) * P.tile_in_bytes + (uint32_t)P.last_sample_col * ipb;   // in this tile
              else hp = frame + (uint64_t)(ro - 1) * P.in_row_bytes + (uint32_t)P.last_sample_col * ipb;
            }
          } else {
            const uint32_t line = ro / F;      // W == F * Wo: one counter line spans F output rows
            if (line & 1) {                    // held from (line-1, lastSampleCol) of the decimated stream
              const uint32_t srow = (line - 1) * F + P.caseb_row_add;
              hp = frame + (uint64_t)(srow * (uint32_t)P.row_step) * P.in_row_bytes + P.caseb_col_bytes;
            }
          }
          if (hp) {                            // a 32-byte TMA-fetched window around the pixel
            const uint64_t a = reinterpret_cast<uint64_t>(hp);
            h = aux + j * 32u + (uint32_t)(a & 15u);
            mbar_expect_tx_only(bar, 32u);
            tma_load_1d(aux + j * 32u, reinterpret_cast<const uint8_t*>(a & ~(uint64_t)15), 32u, bar, pol);
          }
          m->held_addr[j] = h;
          any |= h;
        }
        if (!one_copy) {
          mbar_expect_tx_only(bar, P.tile_in_bytes);
          tma_load_1d(dst + j * P.tile_in_bytes, src + (uint64_t)j * (uint32_t)P.row_step * P.in_row_bytes, P.tile_in_bytes, bar, pol);
        }
      }
      any = __reduce_or_sync(0xFFFFFFFFu, any);
      if (lane == 0) {
        m->any_held_col0 = (any ? 0x80000000u : 0u) | (seg * (uint32_t)P.tile_px);
        m->n_granules = nrows * ((uint32_t)P.tile_px >> 2);
        m->out_base = reinterpret_cast<uint64_t>(P.out) + (uint64_t)k * P.out_frame_bytes + (uint64_t)ro0 * P.out_row_bytes +
                      (uint64_t)seg * P.tile_out_bytes;
        if (FMT == KF_PLANAR) {
          // chroma rows of this tile: output rows with (ro % vs == 0); tiles of more than one row start on one
          const uint32_t vs = (uint32_t)P.planar_vs, hs = (uint32_t)P.planar_hs;
          const uint32_t nrc = (ro0 % vs == 0) ? (nrows + vs - 1) / vs : 0u;
          const uint64_t coff = (uint64_t)(ro0 / vs) * (uint32_t)P.planar_cw + (uint64_t)seg * ((uint32_t)P.tile_px / hs);
          const uint64_t fbase = reinterpret_cast<uint64_t>(P.out) + (uint64_t)k * P.out_frame_bytes;
          m->cb_base = fbase + P.planar_cb_off + coff;
          m->cr_base = fbase + P.planar_cr_off + coff;
          m->n_granules |= nrc << 24;
        }
        if (one_copy) {                        // one bulk copy for the whole tile
          mbar_expect_tx_only(bar, nrows * P.tile_in_bytes);
          tma_load_1d(dst, src, nrows * P.tile_in_bytes, bar, pol);
        }
      }
      __syncwarp();
      // meta is published by the release of this arrive and observed after the consumers' acquire-wait; the phase
      // completes when the last announced byte has landed
      if (lane == 0) mbar_arrive(bar);
    }
    return;
  }

  // ============================== consumer warps =============================================
  LoopConst C;
  {
    const uint32_t my = P.qmask & 0xFFu, mcb = (P.qmask >> 8) & 0xFFu, mcr = (P.qmask >> 16) & 0xFFu;
    C.qm0 = my | (mcb << 8) | (mcr << 16) | (my << 24);
    C.qm1 = mcb | (mcr << 8) | (my << 16) | (mcb << 24);
    C.qm2 = mcr | (my << 8) | (mcb << 16) | (mcr << 24);
    C.my = my; C.mcb = mcb; C.mcr = mcr;
    C.shy = 8 + P.sy; C.shb = 8 + P.scb; C.shr = 8 + P.scr;
    C.ly = P.cb_bits + P.cr_bits; C.lb = P.cr_bits;
    C.coef_y = P.coef_y; C.coef_ncb = P.coef_ncb; C.coef_ncr = P.coef_ncr;
    C.gran_per_row = (uint32_t)P.tile_px >> 2;
    C.out_pitch = P.out_row_bytes; C.out_dense = (uint32_t)P.out_dense; C.ragged = (uint32_t)P.ragged; C.Wo = (uint32_t)P.Wo;
    C.pl_cb_off = (uint32_t)P.tile_rows * (uint32_t)P.tile_px;
    C.pl_crow_bytes = (uint32_t)P.tile_px / (uint32_t)max(1, P.planar_hs);
    C.pl_cr_off = C.pl_cb_off + (uint32_t)((P.tile_rows + P.planar_vs - 1) / max(1, P.planar_vs)) * C.pl_crow_bytes;
    C.pl_vs_shift = P.planar_vs == 2 ? 1u : 0u;
    C.nthreads = NC;
    C.row0_of_thread = tid / C.gran_per_row;
    C.rem0_of_thread = tid % C.gran_per_row;
    C.drow = NC / C.gran_per_row;
    C.drem = NC % C.gran_per_row;
  }
  const int hfe = P.hfe;
  const bool in4 = P.in_px_bytes == 4;

  for (uint32_t i = 0; i < ring.n_my; ++i) {
    const Ring::Pos pos = ring.at(i);
    const uint32_t s = pos.s;
    ring.wait_full(pos);

    const uint32_t in_s = sbase + s * P.stage_stride;
    const uint32_t out_s = sbase + P.out_buf_off + (i & 1u) * P.out_buf_stride;
    const TileMeta* m = reinterpret_cast<const TileMeta*>(smem + P.meta_off) + s;
    uint8_t* out_g = reinterpret_cast<uint8_t*>(m->out_base);
    const uint32_t ngr = m->n_granules & 0x00FFFFFFu, nrc = m->n_granules >> 24;
    const uint32_t out_bytes = ngr * kGranOut;
    const uint64_t cb_g = m->cb_base, cr_g = m->cr_base;
    if (in4) tile_dispatch<F, FMT, Q8, TRUNC, true>((m->any_held_col0 >> 31) != 0, hfe, in_s, out_s, out_g, m, C);
    else tile_dispatch<F, FMT, Q8, TRUNC, false>((m->any_held_col0 >> 31) != 0, hfe, in_s, out_s, out_g, m, C);

    if (kStaged) {
      // Hand the tile to the TMA engine.  Generic-proxy writes must be fenced before the async proxy
      // reads them; the staging buffer used two tiles ago must have been read out before it is reused.
      // The store is issued BEFORE the stage goes back to the producer, so that it sits ahead of the
      // refill's bulk copies in the TMA queue (measured: +6 % on tiles made of many short rows).
      fence_proxy_async_smem();
      if (tid == 0) tma_store_wait_read0();
      consumer_barrier(NC);
      if (tid == 0) {
        if (FMT == KF_PLANAR) {
          tma_store_1d(out_g, out_s, out_bytes, pol);
          if (nrc) {
            tma_store_1d(reinterpret_cast<void*>(cb_g), out_s + C.pl_cb_off, nrc * C.pl_crow_bytes, pol);
            tma_store_1d(reinterpret_cast<void*>(cr_g), out_s + C.pl_cr_off, nrc * C.pl_crow_bytes, pol);
          }
        } else if (P.out_dense) {
          tma_store_1d(out_g, out_s, out_bytes, pol);
        } else {                       // pitched output rows: one bulk store per row of the tile
          const uint32_t nrows = out_bytes / P.tile_out_bytes;
          for (uint32_t j = 0; j < nrows; ++j)
            tma_store_1d(out_g + (uint64_t)j * P.out_row_bytes, out_s + j * P.tile_out_bytes, P.tile_out_bytes, pol);
        }
        tma_store_commit();
      }
    }
    // This warp is done with stage s and its meta: give it back to the producer.
    __syncwarp();
    if ((tid & 31u) == 0) mbar_arrive(ring.empty(s));
  }
  if (kStaged && tid == 0) tma_store_wait_all();
}


namespace {
constexpr int kF = CSIC_ROWS_F;
template <int FMT, bool Q8>
KernelFn by_trunc(bool trunc) { return trunc ? csic_rows_kernel<kF, FMT, Q8, true> : csic_rows_kernel<kF, FMT, Q8, false>; }
}  // namespace

// q8: the bundle's slots keep all 8 bits of every channel (only KF_SLOT32 has an instance for it)
template <>
KernelFn rows_kernel<kF>(int kformat, bool q8, bool trunc) {
  switch (kformat) {
    case KF_YCC888: return by_trunc<KF_YCC888, false>(trunc);
    case KF_RGB888: return by_trunc<KF_RGB888, false>(trunc);
    case KF_SLOT8: return by_trunc<KF_SLOT8, false>(trunc);
    case KF_SLOT16: return by_trunc<KF_SLOT16, false>(trunc);
    case KF_PLANAR: return by_trunc<KF_PLANAR, false>(trunc);
    default: return q8 ? by_trunc<KF_SLOT32, true>(trunc) : by_trunc<KF_SLOT32, false>(trunc);
  }
}

}  // namespace csic
