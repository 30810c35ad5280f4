// csic_pool_kernel<F, FMT, IN4> -- TMA-staged kernel for the AVERAGE pooling extension (pool_mode = AVERAGE,
// chroma stage before the spatial stage).  Not reference behaviour: the reference's SpatialDownsampler is point
// decimation (SpatialDownsampler.scala:33-55); README.md:44 only *says* "average pooling".  Semantics are the
// oracle's: mean of the f x f block of the stream entering the spatial stage, per channel, round half up.
//
// Same machinery as csic_rows_kernel (producer warp + full/empty mbarriers + TMA bulk copies), but a tile needs
// ALL f input rows of every output row, so the f x f block resolves on chip:
//   stage layout   row part (j*F + dr) of the tile at  (j*F + dr) * seg_row_bytes      (j: output row, dr: 0..F-1)
//   granule        4 output pixels = F rows x 4F input pixels
//   chroma hold    in-row: sample at i % hf == 0 inside the 4F-pixel span; odd lines of 4:2:0 / 4:1:0 replay the
//                  last sample of the line above, which is the previous row part of the same block
//                  (ChromaSubsampler.scala:52-65); when rows are split into segments it is TMA-fetched instead.
// Pooling BEFORE the chroma stage (SQC / SCQ / QSC: the application's default order, ImageCompressorTopApp.scala:170-173)
// runs here too when a counter line is whole output rows starting on a sample column (ceil(W/f) % hf == 0): every
// channel is pooled first, the chroma stage then samples the pooled stream with the full-size counters
// (ImageCompressorTop.scala:52-58) -- in-row hold between output pixels, and on odd counter lines every pixel replays
// the pooled chroma of ONE block of the line above, which the producer warp reduces itself (f x f pixels, lanes = pixels).
// Compiled once per F = CSIC_POOL_F (2, 4, 8).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "csic_internal.h"
#include "csic_device_math.cuh"
#include "csic_tma.cuh"

#ifndef CSIC_POOL_F
#error "compile with -DCSIC_POOL_F=2|4|8"
#endif

namespace csic {

struct PoolMeta {
  uint64_t out_base;
  uint32_t n_granules;
  uint32_t col0;                      // first output column of the tile (row segments)
  uint32_t pad[4];
  uint32_t held_addr[kPoolMaxRows];   // index j * (F/2) + dr/2: shared address of the pixel an odd line replays
};
static_assert(sizeof(PoolMeta) == kPoolMetaBytes, "kPoolMetaBytes out of sync");

struct PoolConst {
  uint32_t coef_y, coef_ncb, coef_ncr;
  uint32_t pre_y, pre_cb, pre_cr;     // quantiser keep-masks applied BEFORE pooling (0xFF when quant follows)
  uint32_t pre_y4;                    // pre_y replicated into the four bytes of a word
  uint32_t post_y, post_cb, post_cr;  // ... and AFTER pooling (0xFF when quant came first)
  int sy, scb, scr, ly, lb;           // bundle slot shifts
  uint32_t gran_per_row, nthreads, row0_of_thread, rem0_of_thread, drow, drem;
  uint32_t seg_row_bytes;
  uint32_t Wo, ragged;                // pitched rows wider than the frame: bundle slots of columns >= Wo are the row's zero pad
  bool trunc, vhold;
  bool linear_y;                      // ... same for Y: byte 1 of each dp4a result is accumulated by a second dp4a
  bool linear;                        // no quantiser in front of the pooling: chroma sums in the complement domain
  bool pool_first;                    // pooling precedes the chroma stage: held_addr[] holds pooled pairs, not addresses
};

// 4F consecutive input pixels of one row part, each as a word whose low three bytes are the colour bytes.
template <int F, bool IN4>
__device__ __forceinline__ void load_row_part(uint32_t a, uint32_t (&p)[4 * F]) {
  if (IN4) {
#pragma unroll
    for (int k = 0; k < F; ++k) {
      const uint4 v = lds128(a + 16u * k);
      p[4 * k] = v.x; p[4 * k + 1] = v.y; p[4 * k + 2] = v.z; p[4 * k + 3] = v.w;
    }
  } else {
    uint32_t w[3 * F];
    if (F == 2) {                      // 24 bytes, 8-byte aligned
#pragma unroll
      for (int k = 0; k < 3; ++k) { const uint2 v = lds64(a + 8u * k); w[2 * k] = v.x; w[2 * k + 1] = v.y; }
    } else {                           // 48 / 96 bytes, 16-byte aligned
#pragma unroll
      for (int k = 0; k < 3 * F / 4; ++k) {
        const uint4 v = lds128(a + 16u * k);
        w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
      }
    }
#pragma unroll
    for (int i = 0; i < 4 * F; ++i) {
      const int k = (3 * i) >> 2, sh = ((3 * i) & 3) * 8;
      p[i] = (sh == 0) ? w[k] : ((k + 1 < 3 * F) ? __funnelshift_r(w[k], w[k + 1], sh) : (w[k] >> sh));
    }
  }
}

// MODE resolves the per-launch flags at compile time for the common pipelines, so that the inner loop carries no
// uniform branches on them (ncu, 4K 2x2: 27 of the 325 warp-instructions per granule were such branches and their
// predicate logic):  0 = every flag read at run time (quantiser in front of the pooling, or TRUNC rounding);
// 1..3 = no quantiser in front (complement-domain sums): 1 chroma stage first, 4:2:0 / 4:1:0 (odd lines replay a
// held pair); 2 chroma stage first, no vertical hold; 3 pooling first (the application's default order).
template <int F, int FMT, bool IN4, int HF, bool TRUNC, int MODE>
__device__ __forceinline__ void pool_tile(uint32_t in_s, uint32_t out_s, uint8_t* __restrict__ out_g,
                                          const PoolMeta* __restrict__ meta, const PoolConst& CC) {
  struct Flags {
    bool linear, linear_y, pool_first, vhold;
  };
  const Flags C_f = MODE == 0 ? Flags{CC.linear, CC.linear_y, CC.pool_first, CC.vhold}
                              : Flags{true, F == 2, MODE == 3, MODE == 1};
  const PoolConst& C = CC;
  constexpr uint32_t kGranBytes = (IN4 ? 16u : 12u) * F;     // one row part of a granule
  constexpr int kShift = (F == 2) ? 2 : (F == 4 ? 4 : 6);    // log2(F*F)
  constexpr int kHalf = (F * F) / 2;
  constexpr int kH = (F == 8) ? 2 : 1;                       // chunks per row part
  constexpr int NO = 4 / kH;                                 // output pixels per chunk
  const uint32_t n = meta->n_granules;
  uint32_t row = C.row0_of_thread, rem = C.rem0_of_thread;
  constexpr bool kStagedFmt = (FMT == KF_YCC888 || FMT == KF_RGB888);
  // 12-byte formats: whole warps iterate together (lanes past the tile's last granule idle through the body), because
  // a warp's 32 granules are 384 consecutive output bytes which leave through the warp's own staging slot as 16-byte
  // stores -- no CTA-wide barrier, no TMA store: the kernel is bound by the integer pipes, a barrier per tile cost 10 %
  // 8x8 pooling: a granule is 256 input pixels, so a 24 KB tile has only ~32 of them -- four threads share one, two
  // row parts each (in two 16-pixel halves: 56 registers instead of 96), and add their partial sums up with two
  // shfl.xor steps (1080p 0.27 -> 0.63, 4K 0.36 -> 0.82 of the copy peak; eight threads per granule measured worse).
  constexpr uint32_t kSplit = (F == 8) ? 4u : 1u;      // threads per granule
  constexpr uint32_t kGpw = 32u / kSplit;              // granules per warp and iteration
  const uint32_t sub = threadIdx.x % kSplit;
  const uint32_t n_loop = (kStagedFmt || kSplit > 1u) ? (n + kGpw - 1u) / kGpw * kGpw : n;
  for (uint32_t q = threadIdx.x / kSplit; q < n_loop; q += C.nthreads / kSplit) {
    uint32_t w0 = 0, w1 = 0, w2 = 0;
    int ay[4] = {0, 0, 0, 0}, ab[4] = {0, 0, 0, 0}, ar[4] = {0, 0, 0, 0};
    uint32_t held_pair = 0;
    if (q < n) {
    const uint32_t base = in_s + row * (F * C.seg_row_bytes) + rem * kGranBytes;
    held_pair = C_f.pool_first ? meta->held_addr[row] : 0u;   // bit 31 | pooled Cb << 8 | pooled Cr
    // two row parts per trip: `dr & 1` (is this an odd, i.e. held, line?) is then a compile-time value
#pragma unroll 2
    for (int dr = (int)(sub * (F / kSplit)); dr < (int)((sub + 1u) * (F / kSplit)); ++dr) {
      // 8x8: the row part is taken in two halves of two output pixels each (16 pixels in registers instead of 32)
#pragma unroll
      for (int hh = 0; hh < kH; ++hh) {
      const int ob = hh * NO;          // first output pixel of this chunk
      uint32_t p[NO * F];
      load_row_part<F / kH, IN4>(base + (uint32_t)dr * C.seg_row_bytes + (uint32_t)hh * (NO * F * (IN4 ? 4u : 3u)), p);
      // Y: byte 1 of each dp4a result is the pixel's Y.  Gather the F bytes of an output pixel's row part into
      // words with PRMT (byte 3 of a result is zero: the pad), mask once, and let dp4a add the bytes up.
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        uint32_t d[F];
#pragma unroll
        for (int i = 0; i < F; ++i) d[i] = fwd_y16(p[o * F + i], C.coef_y);
        if (C_f.linear_y) {          // no quantiser in front: byte 1 of every result goes straight into the sum (FMA pipe)
#pragma unroll
          for (int i = 0; i < F; ++i) ay[ob + o] = (int)dp4a_uu(d[i], 1u << 8, (uint32_t)ay[ob + o]);
        } else if (F == 2) {
          const uint32_t w = __byte_perm(d[0], d[1], 0x3351) & C.pre_y4;
          ay[ob + o] = (int)dp4a_uu(w, 0x01010101u, (uint32_t)ay[ob + o]);
        } else {
#pragma unroll
          for (int h = 0; h < F / 4; ++h) {
            const uint32_t lo = __byte_perm(d[4 * h], d[4 * h + 1], 0x3351), hi = __byte_perm(d[4 * h + 2], d[4 * h + 3], 0x3351);
            const uint32_t w = __byte_perm(lo, hi, 0x5410) & C.pre_y4;
            ay[ob + o] = (int)dp4a_uu(w, 0x01010101u, (uint32_t)ay[ob + o]);
          }
        }
      }
      if (C_f.linear) {
        // No quantiser in front of the pooling: the chroma value is 255 - byte1(x) (x = fwd_nc16 < 65536), so the sums are
        // taken in the complement domain -- weight * byte1(x) accumulated by ONE dp4a per sample and channel (coefficient
        // `weight` on byte 1), on the FMA pipe instead of four ALU-pipe instructions -- and flipped once after the loop.
        if (C_f.pool_first) {
          // every pixel's own chroma is pooled; only output pixels on a sample column are needed (the others replay
          // them after the pooling), and rows of an odd counter line replay a pooled pair the producer supplies
          if (!held_pair) {
#pragma unroll
            for (int i = 0; i < NO * F; ++i) {
              if ((ob + i / F) % HF == 0) {
                ab[ob + i / F] = (int)dp4a_uu(fwd_nc16<TRUNC>(p[i], C.coef_ncb), 1u << 8, (uint32_t)ab[ob + i / F]);
                ar[ob + i / F] = (int)dp4a_uu(fwd_nc16<TRUNC>(p[i], C.coef_ncr), 1u << 8, (uint32_t)ar[ob + i / F]);
              }
            }
          }
        } else if (C_f.vhold && (dr & 1)) {
          // nothing is sampled on an odd line: every pixel replays the last sample of the line above
          if (hh == 0) {
          const uint32_t ha = meta->held_addr[row * (F / 2) + (uint32_t)(dr >> 1)];
          const uint32_t hp = lds8(ha) | (lds8(ha + 1) << 8) | (lds8(ha + 2) << 16);
          const uint32_t xb = fwd_nc16<TRUNC>(hp, C.coef_ncb), xr = fwd_nc16<TRUNC>(hp, C.coef_ncr);
#pragma unroll
          for (int o = 0; o < 4; ++o) {
            ab[o] = (int)dp4a_uu(xb, (uint32_t)F << 8, (uint32_t)ab[o]);
            ar[o] = (int)dp4a_uu(xr, (uint32_t)F << 8, (uint32_t)ar[o]);
          }
          }
        } else {
#pragma unroll
          for (int i = 0; i < NO * F; i += HF) {   // sample points; each is held for HF pixels (ChromaSubsampler.scala:57-65)
            const uint32_t xb = fwd_nc16<TRUNC>(p[i], C.coef_ncb), xr = fwd_nc16<TRUNC>(p[i], C.coef_ncr);
            if (HF <= F) {                        // the HF pixels lie inside one output pixel
              ab[ob + i / F] = (int)dp4a_uu(xb, (uint32_t)HF << 8, (uint32_t)ab[ob + i / F]);
              ar[ob + i / F] = (int)dp4a_uu(xr, (uint32_t)HF << 8, (uint32_t)ar[ob + i / F]);
            } else {                              // ... or cover HF / F whole output pixels
#pragma unroll
              for (int o = ob + i / F; o < ob + (i + HF) / F; ++o) {
                ab[o] = (int)dp4a_uu(xb, (uint32_t)F << 8, (uint32_t)ab[o]);
                ar[o] = (int)dp4a_uu(xr, (uint32_t)F << 8, (uint32_t)ar[o]);
              }
            }
          }
        }
      } else if (C_f.pool_first) {
        if (!held_pair) {
#pragma unroll
          for (int i = 0; i < NO * F; ++i) {
            if ((ob + i / F) % HF == 0) {
              ab[ob + i / F] += (int)(((fwd_nc16<TRUNC>(p[i], C.coef_ncb) ^ 0xFFFFu) >> 8) & C.pre_cb);
              ar[ob + i / F] += (int)(((fwd_nc16<TRUNC>(p[i], C.coef_ncr) ^ 0xFFFFu) >> 8) & C.pre_cr);
            }
          }
        }
      } else if (C_f.vhold && (dr & 1)) {
        if (hh == 0) {
        const uint32_t ha = meta->held_addr[row * (F / 2) + (uint32_t)(dr >> 1)];
        const uint32_t hp = lds8(ha) | (lds8(ha + 1) << 8) | (lds8(ha + 2) << 16);
        const int hb = (int)(((fwd_nc16<TRUNC>(hp, C.coef_ncb) ^ 0xFFFFu) >> 8) & C.pre_cb) * F;
        const int hr = (int)(((fwd_nc16<TRUNC>(hp, C.coef_ncr) ^ 0xFFFFu) >> 8) & C.pre_cr) * F;
#pragma unroll
        for (int o = 0; o < 4; ++o) { ab[o] += hb; ar[o] += hr; }
        }
      } else {
        int cb = 0, cr = 0;
#pragma unroll
        for (int i = 0; i < NO * F; ++i) {
          if (i % HF == 0) {          // sample point; held for the next HF-1 pixels (ChromaSubsampler.scala:57-65)
            cb = (int)(((fwd_nc16<TRUNC>(p[i], C.coef_ncb) ^ 0xFFFFu) >> 8) & C.pre_cb);
            cr = (int)(((fwd_nc16<TRUNC>(p[i], C.coef_ncr) ^ 0xFFFFu) >> 8) & C.pre_cr);
          }
          ab[ob + i / F] += cb;
          ar[ob + i / F] += cr;
        }
      }
      }   // hh
    }
    }   // q < n: accumulation
    if (kSplit > 1u) {                 // partial sums of the threads that share the granule (adjacent lanes)
#pragma unroll
      for (int o = 0; o < 4; ++o) {
#pragma unroll
        for (uint32_t d = 1; d < kSplit; d <<= 1) {
          ay[o] += __shfl_xor_sync(0xFFFFFFFFu, ay[o], d);
          ab[o] += __shfl_xor_sync(0xFFFFFFFFu, ab[o], d);
          ar[o] += __shfl_xor_sync(0xFFFFFFFFu, ar[o], d);
        }
      }
    }
    if (q < n && sub == 0u) {
    if (C_f.linear) {                    // back from the complement domain: F*F samples of weight 1 each
#pragma unroll
      for (int o = 0; o < 4; ++o) { ab[o] = 255 * F * F - ab[o]; ar[o] = 255 * F * F - ar[o]; }
    }
    uint32_t y[4], cb[4], cr[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) {      // round half up, then the quantiser if it follows the pooling
      y[o] = (uint32_t)((ay[o] + kHalf) >> kShift) & C.post_y;
      cb[o] = (uint32_t)((ab[o] + kHalf) >> kShift) & C.post_cb;
      cr[o] = (uint32_t)((ar[o] + kHalf) >> kShift) & C.post_cr;
    }
    if (C_f.pool_first) {                // the chroma stage on the pooled stream (ChromaSubsampler.scala:57-65)
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        if (held_pair) { cb[o] = (held_pair >> 8) & 0xFFu & C.post_cb; cr[o] = held_pair & 0xFFu & C.post_cr; }
        else if (o % HF != 0) { cb[o] = cb[o - o % HF]; cr[o] = cr[o - o % HF]; }
      }
    }
    if (FMT == KF_YCC888 || FMT == KF_RGB888) {
      if (FMT == KF_YCC888) {
        // bytes packed with multiply-adds (one IMAD per byte on the FMA pipe) rather than shift + OR on the ALU pipe
        w0 = ((y[1] * 256u + cr[0]) * 256u + cb[0]) * 256u + y[0];
        w1 = ((cb[2] * 256u + y[2]) * 256u + cr[1]) * 256u + cb[1];
        w2 = ((cr[3] * 256u + cb[3]) * 256u + y[3]) * 256u + cr[2];
      } else {
        uint32_t v[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) v[o] = inverse_rgb((int)y[o], (int)cb[o], (int)cr[o]);
        w0 = v[1] * 0x1000000u + v[0];
        w1 = v[2] * 0x10000u + (v[1] >> 8);
        w2 = v[3] * 0x100u + (v[2] >> 16);
      }
    } else {
      uint32_t v[4];
#pragma unroll
      for (int o = 0; o < 4; ++o) v[o] = ((y[o] >> C.sy) << C.ly) | ((cb[o] >> C.scb) << C.lb) | (cr[o] >> C.scr);
      if (C.ragged) {
        const uint32_t co = meta->col0 + rem * 4u;
#pragma unroll
        for (int o = 0; o < 4; ++o) v[o] = (co + o < C.Wo) ? v[o] : 0u;
      }
      if (FMT == KF_SLOT32) __stcs(reinterpret_cast<uint4*>(out_g) + q, make_uint4(v[0], v[1], v[2], v[3]));
      else if (FMT == KF_SLOT16) __stcs(reinterpret_cast<uint2*>(out_g) + q, make_uint2(v[0] | (v[1] << 16), v[2] | (v[3] << 16)));
      else __stcs(reinterpret_cast<uint32_t*>(out_g) + q, v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24));
    }
    }   // q < n && sub == 0: finalise
    if (kStagedFmt) {
      const uint32_t lane = threadIdx.x & 31u, g = lane / kSplit, slot = out_s + (threadIdx.x >> 5) * 384u;
      if (sub == 0u) { sts32(slot + g * 12u, w0); sts32(slot + g * 12u + 4u, w1); sts32(slot + g * 12u + 8u, w2); }
      __syncwarp();
      const uint32_t q0 = q - g;                                      // the warp's first granule: 96 / 384-byte aligned output
      const uint32_t valid = min(kGpw, n - q0) * 12u;                 // bytes of this group that exist
      uint8_t* o = out_g + (size_t)q0 * 12u;
      if (lane < kGpw * 12u / 16u) {
        if ((lane + 1u) * 16u <= valid) {
          __stcs(reinterpret_cast<uint4*>(o) + lane, lds128(slot + lane * 16u));
        } else {
          for (uint32_t wd = lane * 4u; wd < lane * 4u + 4u; ++wd)
            if ((wd + 1u) * 4u <= valid) __stcs(reinterpret_cast<uint32_t*>(o) + wd, lds32(slot + wd * 4u));
        }
      }
      __syncwarp();
    }
    row += C.drow;
    rem += C.drem;
    if (rem >= C.gran_per_row) { rem -= C.gran_per_row; ++row; }
  }
}

// Register budget instead of launch bounds: four CTAs per SM of 288 threads (2x2) need <= 56 registers, of 224 threads
// (4x4, 8x8: six consumer warps) <= 73.  With __launch_bounds__(544) alone ptxas settled on 56 for every factor and
// spilled 24-60 bytes per thread in the 4x4 / 8x8 loops; at 72 nothing spills.
template <int F, int FMT, bool IN4>
__global__ void __maxnreg__(F == 2 ? 56 : 72) csic_pool_kernel(const __grid_constant__ KPlan P) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t tid = threadIdx.x;
  const uint32_t NC = blockDim.x - 32u;
  const uint32_t sbase = smem_u32(smem);
  const uint64_t pol = policy_evict_first();
  const uint32_t seg_row_bytes = P.tile_in_bytes / F;          // one input row part of a segment
  const Ring ring(sbase + P.bar_off, (uint32_t)P.stages, P.n_tiles);
  ring.init(NC / 32u);                                          // one arrive per consumer warp

  // ============================== producer warp ==============================================
  if (tid >= NC) {
    const bool pool_first = P.case_b != 0;
    const uint32_t lane = tid - NC;
    if (lane != 0 && !pool_first) return;        // chroma-first orders: one lane feeds the TMA engine
    const uint32_t ipb = (uint32_t)P.in_px_bytes;
    uint32_t cached_line = 0xFFFFFFFFu, cached_frame = 0xFFFFFFFFu, cached_pair = 0;   // the last block this warp reduced
    for (uint32_t i = 0; i < ring.n_my; ++i) {
      const Ring::Pos pos = ring.at(i);
      ring.wait_empty(pos, i);
      const RowTile t = row_tile(P, blockIdx.x + i * gridDim.x);
      const uint32_t s = pos.s, seg = t.seg, k = t.k, ro0 = t.ro0, nrows = t.nrows;
      const uint8_t* frame = P.in + (uint64_t)k * P.in_frame_bytes;
      const uint32_t bar = ring.full(s);
      const uint32_t dst = sbase + s * P.stage_stride;
      const uint32_t aux = dst + (uint32_t)P.tile_rows * P.tile_in_bytes;    // kPoolMaxRows windows of 32 bytes
      PoolMeta* m = reinterpret_cast<PoolMeta*>(smem + P.meta_off) + s;

      uint32_t n_aux = 0;
      const uint8_t* aux_src[kPoolMaxRows];
      if (pool_first) {
        // Rows of an odd counter line (a line = F output rows, W == F * Wo) replay the pooled chroma of the block at
        // stream element (line-1) * W + lastSampleCol of the pooled stream.  The warp reduces that block itself:
        // lane l takes pixels l, l + 32 of the F x F block.
        constexpr int kShift = (CSIC_POOL_F == 2) ? 2 : (CSIC_POOL_F == 4 ? 4 : 6);
        const uint32_t mcb = P.quant_first ? (P.qmask >> 8) & 0xFFu : 0xFFu, mcr = P.quant_first ? (P.qmask >> 16) & 0xFFu : 0xFFu;
        for (uint32_t j = 0; j < nrows; ++j) {
          const uint32_t line = (ro0 + j) / F;
          uint32_t pair = 0;
          if (P.vf == 2 && (line & 1u)) {
            if (line != cached_line || k != cached_frame) {        // (a CTA's consecutive tiles are often the same line of DIFFERENT frames)
              const uint8_t* blk = frame + (uint64_t)(((line - 1u) * F + P.caseb_row_add) * F) * P.in_row_bytes + P.caseb_col_bytes;
              int sb = 0, sr = 0;
              for (uint32_t e = lane; e < F * F; e += 32u) {
                const uint8_t* px = blk + (uint64_t)(e / F) * P.in_row_bytes + (e % F) * ipb;
                const uint32_t v = (uint32_t)__ldg(px) | ((uint32_t)__ldg(px + 1) << 8) | ((uint32_t)__ldg(px + 2) << 16);
                const uint32_t xb = P.trunc ? fwd_nc16<true>(v, P.coef_ncb) : fwd_nc16<false>(v, P.coef_ncb);
                const uint32_t xr = P.trunc ? fwd_nc16<true>(v, P.coef_ncr) : fwd_nc16<false>(v, P.coef_ncr);
                sb += (int)(((xb ^ 0xFFFFu) >> 8) & mcb);
                sr += (int)(((xr ^ 0xFFFFu) >> 8) & mcr);
              }
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) { sb += __shfl_xor_sync(0xFFFFFFFFu, sb, o); sr += __shfl_xor_sync(0xFFFFFFFFu, sr, o); }
              cached_pair = 0x80000000u | ((uint32_t)((sb + (F * F) / 2) >> kShift) << 8) | (uint32_t)((sr + (F * F) / 2) >> kShift);
              cached_line = line;
              cached_frame = k;
            }
            pair = cached_pair;
          }
          if (lane == 0) m->held_addr[j] = pair;
        }
        __syncwarp();
        if (lane != 0) continue;                  // the rest is lane 0's: describe the tile, feed the TMA engine
      } else if (P.vf == 2) {
        for (uint32_t j = 0; j < nrows; ++j)
          for (uint32_t h = 0; h < F / 2; ++h) {       // odd input line dr = 2h+1 replays (dr-1, lastSampleCol)
            const uint32_t e = j * (F / 2) + h;
            if (P.nsplit == 1) {
              m->held_addr[e] = dst + (j * F + 2 * h) * seg_row_bytes + (uint32_t)P.last_sample_col * ipb;
              aux_src[e] = nullptr;
            } else {
              const uint8_t* hp = frame + (uint64_t)((ro0 + j) * F + 2 * h) * P.in_row_bytes + (uint32_t)P.last_sample_col * ipb;
              const uint64_t a = reinterpret_cast<uint64_t>(hp);
              m->held_addr[e] = aux + e * 32u + (uint32_t)(a & 15u);
              aux_src[e] = reinterpret_cast<const uint8_t*>(a & ~(uint64_t)15);
              ++n_aux;
            }
          }
      }
      m->n_granules = nrows * ((uint32_t)P.tile_px >> 2);
      m->col0 = seg * (uint32_t)P.tile_px;
      m->out_base = reinterpret_cast<uint64_t>(P.out) + (uint64_t)k * P.out_frame_bytes + (uint64_t)ro0 * P.out_row_bytes +
                    (uint64_t)seg * P.tile_out_bytes;
      mbar_expect_tx(bar, nrows * P.tile_in_bytes + n_aux * 32u);
      const uint8_t* src = frame + (uint64_t)(ro0 * F) * P.in_row_bytes + (uint64_t)seg * seg_row_bytes;
      if (P.nsplit == 1 && P.in_dense) {     // whole dense rows: the F*nrows input rows are one contiguous range
        tma_load_1d(dst, src, nrows * P.tile_in_bytes, bar, pol);
      } else {
        for (uint32_t r = 0; r < nrows * F; ++r)
          tma_load_1d(dst + r * seg_row_bytes, src + (uint64_t)r * P.in_row_bytes, seg_row_bytes, bar, pol);
      }
      if (n_aux) {
        for (uint32_t e = 0; e < nrows * (F / 2); ++e)
          if (aux_src[e]) tma_load_1d(aux + e * 32u, aux_src[e], 32u, bar, pol);
      }
    }
    return;
  }

  // ============================== consumer warps =============================================
  PoolConst C;
  {
    const uint32_t my = P.qmask & 0xFFu, mcb = (P.qmask >> 8) & 0xFFu, mcr = (P.qmask >> 16) & 0xFFu;
    C.coef_y = P.coef_y; C.coef_ncb = P.coef_ncb; C.coef_ncr = P.coef_ncr;
    C.pre_y = P.quant_first ? my : 0xFFu;   C.pre_cb = P.quant_first ? mcb : 0xFFu;   C.pre_cr = P.quant_first ? mcr : 0xFFu;
    C.pre_y4 = C.pre_y * 0x01010101u;
    C.post_y = P.quant_first ? 0xFFu : my;  C.post_cb = P.quant_first ? 0xFFu : mcb;  C.post_cr = P.quant_first ? 0xFFu : mcr;
    C.sy = P.sy; C.scb = P.scb; C.scr = P.scr;
    C.ly = P.cb_bits + P.cr_bits; C.lb = P.cr_bits;
    C.gran_per_row = (uint32_t)P.tile_px >> 2;
    C.nthreads = NC;
    constexpr uint32_t kSplit = (F == 8) ? 4u : 1u;      // threads per granule (see pool_tile)
    C.row0_of_thread = (tid / kSplit) / C.gran_per_row;
    C.rem0_of_thread = (tid / kSplit) % C.gran_per_row;
    C.drow = (NC / kSplit) / C.gran_per_row;
    C.drem = (NC / kSplit) % C.gran_per_row;
    C.seg_row_bytes = seg_row_bytes;
    C.Wo = (uint32_t)P.Wo; C.ragged = (uint32_t)P.ragged;
    C.trunc = P.trunc != 0;
    C.vhold = P.vf == 2;
    C.pool_first = P.case_b != 0;
    C.linear = C.pre_cb == 0xFFu && C.pre_cr == 0xFFu;
    C.linear_y = F == 2 && C.pre_y == 0xFFu;   // B200: pays for 2x2 only (4x4: the PRMT gather + one dp4a is cheaper)
  }
  const int hf = P.hf;
  // which specialisation of pool_tile (see its MODE parameter)
  const int mode = C.trunc ? 4 : ((C.linear && C.pre_y == 0xFFu) ? (C.pool_first ? 3 : (C.vhold ? 1 : 2)) : 0);

  for (uint32_t i = 0; i < ring.n_my; ++i) {
    const Ring::Pos pos = ring.at(i);
    const uint32_t s = pos.s;
    ring.wait_full(pos);
    const uint32_t in_s = sbase + s * P.stage_stride;
    const uint32_t out_s = sbase + P.out_buf_off;     // 12-byte formats: one 384-byte staging slot per consumer warp
    const PoolMeta* m = reinterpret_cast<const PoolMeta*>(smem + P.meta_off) + s;
    uint8_t* out_g = reinterpret_cast<uint8_t*>(m->out_base);
    switch (mode) {
#define CSIC_POOL_HF(TR, MD)                                                            \
      if (hf == 1) pool_tile<F, FMT, IN4, 1, TR, MD>(in_s, out_s, out_g, m, C);         \
      else if (hf == 2) pool_tile<F, FMT, IN4, 2, TR, MD>(in_s, out_s, out_g, m, C);    \
      else pool_tile<F, FMT, IN4, 4, TR, MD>(in_s, out_s, out_g, m, C);                 \
      break;
      case 1: CSIC_POOL_HF(false, 1)
      case 2: CSIC_POOL_HF(false, 2)
      case 3: CSIC_POOL_HF(false, 3)
      case 4: CSIC_POOL_HF(true, 0)
      default: CSIC_POOL_HF(false, 0)
#undef CSIC_POOL_HF
    }

    __syncwarp();
    if ((tid & 31u) == 0) mbar_arrive(ring.empty(s));
  }
}

template <>
KernelFn pool_kernel<CSIC_POOL_F>(int kformat, bool in4) {
  constexpr int F = CSIC_POOL_F;
  switch (kformat) {
    case KF_YCC888: return in4 ? csic_pool_kernel<F, KF_YCC888, true> : csic_pool_kernel<F, KF_YCC888, false>;
    case KF_RGB888: return in4 ? csic_pool_kernel<F, KF_RGB888, true> : csic_pool_kernel<F, KF_RGB888, false>;
    case KF_SLOT8: return in4 ? csic_pool_kernel<F, KF_SLOT8, true> : csic_pool_kernel<F, KF_SLOT8, false>;
    case KF_SLOT16: return in4 ? csic_pool_kernel<F, KF_SLOT16, true> : csic_pool_kernel<F, KF_SLOT16, false>;
    default: return in4 ? csic_pool_kernel<F, KF_SLOT32, true> : csic_pool_kernel<F, KF_SLOT32, false>;
  }
}

}  // namespace csic
