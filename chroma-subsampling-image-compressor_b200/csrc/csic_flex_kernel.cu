// csic_flex_kernel<FMT, TRUNC> -- the DECIMATE pipeline for buffers the TMA row kernel's 16-byte rules exclude:
// any frame width, any row pitch, any base-pointer alignment (dense odd-width frames on the device, sub-views of a
// larger buffer, bundle rows with pad slots).  Same arithmetic and the same closed-form source maps as
// csic_rows_kernel; what differs is how bytes move:
//
//   load     a tile = up to 16 whole output rows (or one row segment).  Every input row span lands in shared memory
//            at the SAME offset modulo 16 it has in global memory, so its 16-byte-aligned hull can be fetched by the
//            TMA engine (one cp.async.bulk per span, mbarrier complete_tx) although neither the span's start nor its
//            length is aligned.  The hull brings along < 16 bytes of the neighbouring pixels / rows of the same
//            buffer on each side; only at the two ends of the byte range the launch may touch is the hull clipped and
//            the edge bytes copied one by one, so the kernel is exact on sub-buffers.  A dedicated producer warp walks
//            the CTA's tiles ahead of the consumer warps (two input stages, full / empty mbarriers), fetches the
//            pixel a held row replays, and publishes a small descriptor per tile so that nobody else does geometry
//            arithmetic.
//   compute  one thread per granule of 4 output pixels; pixels at arbitrary byte addresses are aligned LDS.32 words
//            re-aligned with funnel shifts.  dp4a colour matrix, in-granule chroma hold, held rows from one pixel per
//            row (ChromaSubsampler.scala:52-65), quantise, pack -- into a staging area whose rows sit at the output's
//            own offset modulo 16 (to the word).
//   store    the staging area leaves as 16-byte st.global.cs words aligned on the GLOBAL address (LDS.128 plus at
//            most one extra word and four funnel shifts), head / tail bytes with byte stores: coalesced whatever the
//            row size.
//
// Reference semantics as in csic_kernels.cu's header (RGB2YCbCr.scala:33-76, ChromaSubsampler.scala:26-65,
// SpatialDownsampler.scala:17-55, ColorQuantizer.scala:29-44, RGB2YCbCr.scala:123-132, ImageCompressorTop.scala:43-58).
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "csic_internal.h"
#include "csic_device_math.cuh"
#include "csic_tma.cuh"

namespace csic {

namespace {

constexpr uint32_t kCtaWideSpan = 2048u;             // row spans at least this long are stored by the whole CTA
constexpr uint32_t kDirectRowBytes = 257u;           // output rows shorter than this that cannot be packed leave from registers (B200 map:
                                                     // 75-250-byte rows 1.3x faster direct, 375-1000-byte rows up to 2x faster staged)

__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
// issued where it is written (never sunk towards its use): the value is consumed a whole tile later
__device__ __forceinline__ uint32_t ldg8_now(const uint8_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// n and m powers of two, n <= m  (no division: this runs once per tile in every thread)
__device__ __forceinline__ bool pow2_divides(uint32_t n, uint32_t m) {
  return n != 0u && (n & (n - 1u)) == 0u && (m & (m - 1u)) == 0u && n <= m;
}

// `n` row spans of `len` bytes: long ones share the warps (or go one after the other with the whole CTA when their
// number does not divide the warps), short ones take one warp each.
template <typename F>
__device__ __forceinline__ void for_each_span(uint32_t n, uint32_t len, uint32_t NC, F&& fn) {
  const uint32_t tid = threadIdx.x, NW = NC >> 5;
  if ((len >= kCtaWideSpan || n == 1) && pow2_divides(n, NW)) {      // few long spans: NW / n warps each, set up once per warp
    const uint32_t sh = 31u - __clz(NW) - (31u - __clz(n));                // log2(NW / n): both powers of two
    const uint32_t parts = 1u << sh, j = (tid >> 5) >> sh, part = (tid >> 5) & (parts - 1u);
    fn(j, part * 32u + (tid & 31u), parts * 32u);
  } else if (len >= kCtaWideSpan || n == 1) {
    for (uint32_t j = 0; j < n; ++j) fn(j, tid, NC);
  } else {
    for (uint32_t j = tid >> 5; j < n; j += NW) fn(j, tid & 31u, 32u);
  }
}

// three colour bytes at an arbitrary shared-memory address (low three bytes of the result)
__device__ __forceinline__ uint32_t lds_px(uint32_t a) {
  const uint32_t b = a & ~3u;
  return __funnelshift_r(lds32(b), lds32(b + 4), (a & 3u) * 8u);
}

// The four sampled pixels of a whole granule: input pixels at a, a + pxb, a + 2 pxb, a + 3 pxb (pxb = bytes between
// sampled pixels: 3, 6, 12, 24 for RGB24 at f = 1, 2, 4, 8; 4, 8, 16, 32 for the 4-byte formats).
template <uint32_t PXB>   // 3, 6, or 0 = any multiple of four (passed at run time)
__device__ __forceinline__ void load_granule_any(uint32_t a, uint32_t pxb, uint32_t (&p)[4]) {
  const uint32_t b = a & ~3u, sh = (a & 3u) * 8u;
  if (PXB == 3u) {             // 12 consecutive bytes: word stride 3 across lanes, conflict free
    const uint32_t w0 = lds32(b), w1 = lds32(b + 4), w2 = lds32(b + 8), w3 = lds32(b + 12);
    const uint32_t v0 = __funnelshift_r(w0, w1, sh), v1 = __funnelshift_r(w1, w2, sh), v2 = __funnelshift_r(w2, w3, sh);
    p[0] = v0;
    p[1] = __funnelshift_r(v0, v1, 24);
    p[2] = __funnelshift_r(v1, v2, 16);
    p[3] = v2 >> 8;
  } else if (PXB == 6u) {      // 21 bytes inside six words
    const uint32_t w0 = lds32(b), w1 = lds32(b + 4), w2 = lds32(b + 8), w3 = lds32(b + 12), w4 = lds32(b + 16), w5 = lds32(b + 20);
    p[0] = __funnelshift_r(w0, w1, sh);                                                          // bytes 0..2
    p[1] = __funnelshift_r(__funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), 16);        // bytes 6..8
    p[2] = __funnelshift_r(w3, w4, sh);                                                          // bytes 12..14
    p[3] = __funnelshift_r(__funnelshift_r(w4, w5, sh), w5 >> sh, 16);                           // bytes 18..20
  } else {                     // pxb % 4 == 0: every pixel has the same byte phase
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = __funnelshift_r(lds32(b + j * pxb), lds32(b + j * pxb + 4), sh);
  }
}

template <int FMT> struct FlexFmt {
  // staging bytes per granule of four slots
  static constexpr uint32_t kUnit = (FMT == KF_YCC888 || FMT == KF_RGB888) ? 12u : (FMT == KF_SLOT32 ? 16u : (FMT == KF_SLOT16 ? 8u : 4u));
};

// Everything the consumer warps need to know about a tile, computed by the producer warp (which has the time: it
// only issues a few bulk copies per tile) and written to shared memory before it arms the stage's mbarrier; read by
// every thread after the barrier's phase flips as five vector loads.  Round 1 had each of the 256 consumer threads
// redo this arithmetic (64-bit output address, row assignment mode, a `% stages` division) for every tile: about 200
// of the 770 warp-instructions a 16 KB tile cost (ncu, 1366x768).
struct FlexDesc {
  uint32_t k, ro0, nrows, col0;            // frame, first output row, rows, first slot
  uint32_t npx, a0, gpr, last_px;          // pixels (>= 1), (address of the first input byte) & 15, granules per row, npx - 1
  uint32_t obase_lo, obase_hi, st_mul, st_add;   // global address of the first output byte; staging row j sits at
                                           //   out_s + j * st_mul + ((obase_lo + j * st_add) & 12)
  uint32_t mode, sh, magic, n_gran;        // how granules are dealt to threads (flex_consume), log2(warps per row), 2^32 / gpr
  uint32_t row_out, out_one, ncols, direct; // output bytes per row, "whole dense rows: one packed span", slots (pad slots incl.),
                                           // "narrow rows: granules go straight to global memory" (direct_store)
};
static_assert(sizeof(FlexDesc) == kFlexDescBytes, "kFlexDescBytes out of sync");

}  // namespace

// The consumer warps' loop over this CTA's tiles.
template <int FMT, bool TRUNC, uint32_t HFE, uint32_t PXB, bool DIRECT>
__device__ __forceinline__ void flex_consume(const KPlan& P, uint8_t* smem, const Ring& ring) {
  constexpr uint32_t kUnit = FlexFmt<FMT>::kUnit;
  const uint32_t tid = threadIdx.x, NC = blockDim.x - 32u, NW = NC >> 5;
  const uint32_t sbase = smem_u32(smem), out_s = sbase + P.out_buf_off, held_base = sbase + P.meta_off;
  const uint32_t desc0 = sbase + P.bar_off + kRingBarBytes * ring.S;
  const uint32_t in_stage = P.stage_stride * (uint32_t)P.tile_rows + 32u;     // bytes of one input stage
  const uint32_t ipb = (uint32_t)P.in_px_bytes, pxb = (uint32_t)P.f * ipb;
  const uint32_t nsplit = (uint32_t)P.nsplit;
  const bool vhold = P.vf == 2;
  const uint32_t my = P.qmask & 0xFFu, mcb = (P.qmask >> 8) & 0xFFu, mcr = (P.qmask >> 16) & 0xFFu;
  const uint32_t qm0 = my | (mcb << 8) | (mcr << 16) | (my << 24);
  const uint32_t qm1 = mcb | (mcr << 8) | (my << 16) | (mcb << 24);
  const uint32_t qm2 = mcr | (my << 8) | (mcb << 16) | (mcr << 24);
  const int shy = 8 + P.sy, shb = 8 + P.scb, shr = 8 + P.scr, ly = P.cb_bits + P.cr_bits, lb = P.cr_bits;
  const bool q8 = FMT == KF_SLOT32 && P.sy == 0 && P.scb == 0 && P.scr == 0;
  const uint32_t vs_sh = P.planar_vs == 2 ? 1u : 0u, hs_sh = P.planar_hs == 4 ? 2u : (P.planar_hs == 2 ? 1u : 0u);
  // Input rows of a tile land in stage s at  in(s) + j * rs_mul + ((a0 + j * rs_add) & 15),  a0 = src0 & 15.
  const uint32_t rs_mul = P.in_dense ? P.in_row_bytes : P.stage_stride;
  const uint32_t rs_add = P.in_dense ? 0u : (((uint32_t)P.row_step * P.in_row_bytes) & 15u);

  // How the granules of a tile are dealt to the threads (FlexDesc::mode, chosen by the producer):
  //   0  no more rows than warps: a power-of-two number of warps per row (NW / nrows rounded down), everything
  //      row-dependent set up once per warp -- taken when at least 4/5 of the lanes of a row's warps get a granule
  //   1  very wide rows: row by row with the whole CTA          2  more rows than warps: one row per warp and round
  //   3  one flat loop over the tile's granules (rows that deal unevenly)
  Ring::Pos pos;
  for (uint32_t it = 0; it < ring.n_my; ++it, pos.next(ring.S)) {
    const uint32_t s = pos.s;
    ring.wait_full(pos);
    const uint32_t da = desc0 + s * kFlexDescBytes;
    const uint4 d0 = lds128(da), d1 = lds128(da + 16u), d2 = lds128(da + 32u), d3 = lds128(da + 48u);
    const uint4 d4 = lds128(da + 64u);   // row_out, out_one, ncols, direct
    const uint32_t Dk = d0.x, Dro0 = d0.y, Dnrows = d0.z, Dcol0 = d0.w, Dnpx = d1.x, Da0 = d1.y;
    constexpr bool direct = DIRECT;      // launch-wide (every tile of a launch has the same row geometry when nsplit == 1)
    consumer_barrier(NC);          // the previous tile has left the staging area

    // ---- compute -------------------------------------------------------------------------------------------
    const uint32_t in_s = sbase + s * in_stage, held_s = held_base + s * (uint32_t)kFlexMaxRows * 4u;
    const uint32_t gpr = d1.z, last_px = d1.w;
    uint8_t* obase = reinterpret_cast<uint8_t*>((uint64_t)d2.x | ((uint64_t)d2.y << 32));
    // staging row j sits at  out_s + j * st_mul + ((oa0 + j * st_add) & 12):  the output row's own offset modulo 16,
    // rounded down to a word
    const uint32_t oa0 = d2.x, st_mul = d2.z, st_add = d2.w;
    // PLANAR: chroma rows of the tile are the output rows with ro % vs == 0
    uint8_t* fout = P.out + (uint64_t)Dk * P.out_frame_bytes;
    const uint32_t c_first = (Dro0 + (1u << vs_sh) - 1u) >> vs_sh;
    const uint32_t c_last1 = ((Dro0 + Dnrows - 1u) >> vs_sh) + 1u;
    const uint32_t nrc = (FMT == KF_PLANAR && c_last1 > c_first) ? c_last1 - c_first : 0u;
    const uint32_t ccols = (Dnpx + (1u << hs_sh) - 1u) >> hs_sh;
    const uint32_t cb_s = out_s + Dnrows * st_mul + 16u, cr_s = cb_s + nrc * ccols;

    // one granule: (row, g) of the tile; rs = shared address of the row's first input byte, so_row = of its staging
    // row, hv = the row's held pixel (0: the row samples its own chroma)
    auto granule = [&](uint32_t row, uint32_t g, uint32_t rs, uint32_t so_row, uint32_t hv) {
      const uint32_t c = g * 4u;
      uint32_t p[4], dy[4], xb[4], xr[4];
      if (c + 3u <= last_px) {
        load_granule_any<PXB>(rs + c * pxb, pxb, p);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) p[j] = lds_px(rs + min(c + j, last_px) * pxb);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) dy[j] = fwd_y16(p[j], P.coef_y);
      const uint32_t so = so_row + g * kUnit;
      // direct mode: this granule's first output byte in global memory and how many of its bytes exist in the row
      uint8_t* gp = obase + (uint64_t)row * P.out_row_bytes + g * kUnit;
      const uint32_t gbytes = min(kUnit, d4.x - g * kUnit);
      if (FMT == KF_RGB888) {
        // fused reconstruction: the chroma-only part of YCbCr2RGB per chroma SAMPLE (once per granule on a held row,
        // every HFE-th pixel otherwise), the per-pixel part in emit()
        const uint32_t my8 = my << 8, mcb8 = mcb << 8, mcr8 = mcr << 8;
        auto emit = [&](const InvChroma& t0, const InvChroma& t1, const InvChroma& t2, const InvChroma& t3) {
          uint32_t w0, w1, w2;
        inv_granule(dy, my8, t0, t1, t2, t3, w0, w1, w2);
          if (direct) { const uint32_t ww[3] = {w0, w1, w2}; direct_store(gp, ww, gbytes); }
          else { sts32(so, w0); sts32(so + 4, w1); sts32(so + 8, w2); }
        };
        if (hv) {
          const InvChroma t = inv_chroma_terms(fwd_nc16<TRUNC>(hv & 0x00FFFFFFu, P.coef_ncb), fwd_nc16<TRUNC>(hv & 0x00FFFFFFu, P.coef_ncr), mcb8, mcr8);
          emit(t, t, t, t);
        } else {
          InvChroma t[4];
#pragma unroll
          for (int j = 0; j < 4; j += (int)HFE) t[j] = inv_chroma_terms(fwd_nc16<TRUNC>(p[j], P.coef_ncb), fwd_nc16<TRUNC>(p[j], P.coef_ncr), mcb8, mcr8);
          emit(t[0], t[1 - 1 % HFE], t[2 - 2 % HFE], t[3 - 3 % HFE]);
        }
        return;
      }
      if (hv) {
        const uint32_t hb = fwd_nc16<TRUNC>(hv & 0x00FFFFFFu, P.coef_ncb), hr = fwd_nc16<TRUNC>(hv & 0x00FFFFFFu, P.coef_ncr);
#pragma unroll
        for (int j = 0; j < 4; ++j) { xb[j] = hb; xr[j] = hr; }
      } else {
        // sample where j % HFE == 0, hold in between (ChromaSubsampler.scala:57-65)
        xb[0] = fwd_nc16<TRUNC>(p[0], P.coef_ncb); xr[0] = fwd_nc16<TRUNC>(p[0], P.coef_ncr);
        if (HFE == 1) { xb[1] = fwd_nc16<TRUNC>(p[1], P.coef_ncb); xr[1] = fwd_nc16<TRUNC>(p[1], P.coef_ncr); }
        else { xb[1] = xb[0]; xr[1] = xr[0]; }
        if (HFE <= 2) { xb[2] = fwd_nc16<TRUNC>(p[2], P.coef_ncb); xr[2] = fwd_nc16<TRUNC>(p[2], P.coef_ncr); }
        else { xb[2] = xb[0]; xr[2] = xr[0]; }
        if (HFE == 1) { xb[3] = fwd_nc16<TRUNC>(p[3], P.coef_ncb); xr[3] = fwd_nc16<TRUNC>(p[3], P.coef_ncr); }
        else { xb[3] = xb[2]; xr[3] = xr[2]; }
      }
      if (FMT == KF_YCC888) {
        // byte 1 of dy is Y, byte 1 of xb/xr is ~Cb/~Cr: gather with PRMT, flip and quantise per word
        uint32_t t, u, ww[3];
        t = __byte_perm(dy[0], xb[0], 0x0051); u = __byte_perm(xr[0], dy[1], 0x0051);
        ww[0] = (__byte_perm(t, u, 0x5410) ^ 0x00FFFF00u) & qm0;
        t = __byte_perm(xb[1], xr[1], 0x0051); u = __byte_perm(dy[2], xb[2], 0x0051);
        ww[1] = (__byte_perm(t, u, 0x5410) ^ 0xFF00FFFFu) & qm1;
        t = __byte_perm(xr[2], dy[3], 0x0051); u = __byte_perm(xb[3], xr[3], 0x0051);
        ww[2] = (__byte_perm(t, u, 0x5410) ^ 0xFFFF00FFu) & qm2;
        if (direct) direct_store(gp, ww, gbytes);
        else { sts32(so, ww[0]); sts32(so + 4, ww[1]); sts32(so + 8, ww[2]); }
      } else if (FMT == KF_PLANAR) {
        const uint32_t my4 = my * 0x01010101u;
        sts32(so, __byte_perm(__byte_perm(dy[0], dy[1], 0x0051), __byte_perm(dy[2], dy[3], 0x0051), 0x5410) & my4);
        if (!hv) {               // a sampled line: its sample points go to the chroma planes (hs == HFE here)
          const uint32_t crow = (((Dro0 + row) >> vs_sh) - c_first) * ccols + (c >> hs_sh);
          if (HFE == 1) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (c + j <= last_px) { sts8(cb_s + crow + j, (~(xb[j] >> 8)) & mcb); sts8(cr_s + crow + j, (~(xr[j] >> 8)) & mcr); }
          } else if (HFE == 2) {
            sts8(cb_s + crow, (~(xb[0] >> 8)) & mcb); sts8(cr_s + crow, (~(xr[0] >> 8)) & mcr);
            if (c + 2 <= last_px) { sts8(cb_s + crow + 1, (~(xb[2] >> 8)) & mcb); sts8(cr_s + crow + 1, (~(xr[2] >> 8)) & mcr); }
          } else {
            sts8(cb_s + crow, (~(xb[0] >> 8)) & mcb); sts8(cr_s + crow, (~(xr[0] >> 8)) & mcr);
          }
        }
      } else {
        uint32_t v[4];
        if (q8) {
#pragma unroll
          for (int j = 0; j < 4; ++j)   // (Cr, Cb, Y, 0): dy < 65536 so its byte 3 is the zero pad
            v[j] = __byte_perm(__byte_perm(xr[j], xb[j], 0x0051), dy[j], 0x7510) ^ 0x0000FFFFu;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            v[j] = ((dy[j] >> shy) << ly) | (((xb[j] ^ 0xFFFFu) >> shb) << lb) | ((xr[j] ^ 0xFFFFu) >> shr);
        }
        if (c + 3u > last_px) {        // the row's zero pad slots
#pragma unroll
          for (int j = 0; j < 4; ++j) if (c + j > last_px) v[j] = 0u;
        }
        if (direct) {
          if (FMT == KF_SLOT32) direct_store(gp, v, gbytes);
          else if (FMT == KF_SLOT16) { const uint32_t ww[2] = {v[0] | (v[1] << 16), v[2] | (v[3] << 16)}; direct_store(gp, ww, gbytes); }
          else { const uint32_t ww[1] = {v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24)}; direct_store(gp, ww, gbytes); }
        } else if (FMT == KF_SLOT32) {
          if ((so & 15u) == 0) sts128(so, v[0], v[1], v[2], v[3]);
          else if ((so & 7u) == 0) { sts64(so, v[0], v[1]); sts64(so + 8, v[2], v[3]); }
          else { sts32(so, v[0]); sts32(so + 4, v[1]); sts32(so + 8, v[2]); sts32(so + 12, v[3]); }
        } else if (FMT == KF_SLOT16) {
          if ((so & 7u) == 0) sts64(so, v[0] | (v[1] << 16), v[2] | (v[3] << 16));
          else { sts32(so, v[0] | (v[1] << 16)); sts32(so + 4, v[2] | (v[3] << 16)); }
        } else {
          sts32(so, v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24));
        }
      }
    };
    auto row_in = [&](uint32_t row) { return in_s + row * rs_mul + ((Da0 + row * rs_add) & 15u); };
    auto row_st = [&](uint32_t row) { return out_s + row * st_mul + ((oa0 + row * st_add) & 12u); };
    if (d3.x == 0u) {
      const uint32_t parts = 1u << d3.y, row = (tid >> 5) >> d3.y, part = (tid >> 5) & (parts - 1u);
      if (row < Dnrows) {          // 3, 5, 6 or 7 rows on 8 warps leave the last warps without one
        const uint32_t rs = row_in(row), so_row = row_st(row), hv = vhold ? lds32(held_s + row * 4u) : 0u;
        for (uint32_t g = part * 32u + (tid & 31u); g < gpr; g += parts * 32u) granule(row, g, rs, so_row, hv);
      }
    } else if (d3.x == 1u) {     // very wide rows: row by row, nothing row-dependent inside the loop
      for (uint32_t row = 0; row < Dnrows; ++row) {
        const uint32_t rs = row_in(row), so_row = row_st(row), hv = vhold ? lds32(held_s + row * 4u) : 0u;
        for (uint32_t g = tid; g < gpr; g += NC) granule(row, g, rs, so_row, hv);
      }
    } else if (d3.x == 2u) {     // narrow rows that fill whole warps, a whole number of rows per warp: row by row per warp
      for (uint32_t row = tid >> 5; row < Dnrows; row += NW) {
        const uint32_t rs = row_in(row), so_row = row_st(row), hv = vhold ? lds32(held_s + row * 4u) : 0u;
        for (uint32_t g = tid & 31u; g < gpr; g += 32u) granule(row, g, rs, so_row, hv);
      }
    } else {                       // narrow rows: one flat loop over the tile's granules
      for (uint32_t q = tid; q < d3.w; q += NC) {
        const uint32_t row = gpr > 1u ? __umulhi(q, d3.z) : q, g = q - row * gpr;
        granule(row, g, row_in(row), row_st(row), vhold ? lds32(held_s + row * 4u) : 0u);
      }
    }
    consumer_barrier(NC);          // staging complete; every read of input stage s, its held words and descriptor is done
    if (tid == 0) mbar_arrive(ring.empty(s));

    // ---- store ---------------------------------------------------------------------------------------------
    if (direct) {
      // nothing staged: the granules went out from registers
    } else if (d4.y) {
      span_store(obase, out_s + (oa0 & 12u), Dnrows * d4.x, tid, NC);
    } else {
      for_each_span(Dnrows, d4.x, NC, [&](uint32_t j, uint32_t t, uint32_t n) {
        span_store(obase + (uint64_t)j * P.out_row_bytes, out_s + j * st_mul + ((oa0 + j * st_add) & 12u), d4.x, t, n);
      });
    }
    if (FMT == KF_PLANAR && nrc) {
      const uint64_t coff = (uint64_t)c_first * (uint32_t)P.planar_cw + (Dcol0 >> hs_sh);
      uint8_t* cb_g = fout + P.planar_cb_off + coff;
      uint8_t* cr_g = fout + P.planar_cr_off + coff;
      if (nsplit == 1) {                                       // ccols == planar_cw: chroma rows are contiguous
        span_store(cb_g, cb_s, nrc * ccols, tid, NC);
        span_store(cr_g, cr_s, nrc * ccols, tid, NC);
      } else {
        for_each_span(nrc, ccols, NC, [&](uint32_t j, uint32_t t, uint32_t n) {
          span_store(cb_g + (uint64_t)j * (uint32_t)P.planar_cw, cb_s + j * ccols, ccols, t, n);
          span_store(cr_g + (uint64_t)j * (uint32_t)P.planar_cw, cr_s + j * ccols, ccols, t, n);
        });
      }
    }
  }
}

template <int FMT, bool TRUNC>
__global__ void __launch_bounds__(kFlexMaxThreads, 4) csic_flex_kernel(const __grid_constant__ KPlan P) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr uint32_t kUnit = FlexFmt<FMT>::kUnit, kOpx = kUnit / 4u;
  const uint32_t tid = threadIdx.x, NT = blockDim.x;
  const uint32_t sbase = smem_u32(smem), held_base = sbase + P.meta_off;
  const uint32_t in_stage = P.stage_stride * (uint32_t)P.tile_rows + 32u;     // bytes of one input stage
  const uint32_t ipb = (uint32_t)P.in_px_bytes, f = (uint32_t)P.f, pxb = f * ipb;
  const uint32_t nsplit = (uint32_t)P.nsplit;
  const uint32_t hfe = (uint32_t)P.hfe;
  const bool vhold = P.vf == 2;
  const uint64_t rstep = (uint64_t)(uint32_t)P.row_step * P.in_row_bytes;
  const Ring ring(sbase + P.bar_off, (uint32_t)P.stages, P.n_tiles);
  if (ring.n_my == 0) return;
  // Input rows of a tile land in stage s at  in(s) + j * rs_mul + ((a0 + j * rs_add) & 15),  a0 = src0 & 15.
  const uint32_t rs_mul = P.in_dense ? P.in_row_bytes : P.stage_stride;
  const uint32_t NC = NT - 32u;    // consumer threads; the last warp is the producer
  ring.init(1);                    // one consumer's arrive, behind the consumers' barrier

  // ============================== producer warp ==============================================================
  // Walks this CTA's tiles up to S stages ahead of the consumers.  All lanes track the geometry; lane 0 describes the
  // tile, lanes 0..nrows-1 hand one row span each to the TMA engine and fetch the pixel a held row replays.
  if (tid >= NC) {
    const uint32_t lane = tid - NC;
    const uint64_t pol = policy_evict_first();
    const uint32_t t2 = blockIdx.x / nsplit, g2 = gridDim.x / nsplit;
    uint32_t pseg = blockIdx.x - t2 * nsplit, pk = t2 / P.tiles_per_band, ptb = t2 - pk * P.tiles_per_band;
    const uint32_t dseg = gridDim.x - g2 * nsplit, dk = g2 / P.tiles_per_band, dtb = g2 - dk * P.tiles_per_band;
    // the byte range of the input this launch may touch (see span_fetch)
    const uintptr_t lim_lo = reinterpret_cast<uintptr_t>(P.in) + (uint64_t)((uint32_t)P.row0 * (uint32_t)P.row_step) * P.in_row_bytes;
    const uintptr_t lim_hi = reinterpret_cast<uintptr_t>(P.in) + (uint64_t)(P.n_frames - 1u) * P.in_frame_bytes +
                             (uint64_t)((uint32_t)(P.row0 + P.band_rows - 1) * (uint32_t)P.row_step) * P.in_row_bytes +
                             ((uint32_t)P.Wo - 1u) * pxb + ipb;
    Ring::Pos pos;
    for (uint32_t j = 0; j < ring.n_my; ++j, pos.next(ring.S)) {
      const uint32_t s = pos.s, bar = ring.full(s), in_s = sbase + s * in_stage;
      ring.wait_empty(pos, j);
      FlexDesc* d = reinterpret_cast<FlexDesc*>(smem + P.bar_off + kRingBarBytes * ring.S) + s;
      const uint32_t ro0 = (uint32_t)P.row0 + ptb * (uint32_t)P.tile_rows;
      const uint32_t nrows = min((uint32_t)P.tile_rows, (uint32_t)(P.row0 + P.band_rows) - ro0);
      const uint32_t col0 = pseg * (uint32_t)P.tile_px;
      const uint32_t ncols = min((uint32_t)P.tile_px, (uint32_t)P.slots_per_row - col0);
      const uint32_t npx = min((uint32_t)P.Wo, col0 + ncols) - col0;
      const uint32_t len_in = (npx - 1u) * pxb + ipb;  // first byte of the first .. last byte of the last sampled pixel
      const uint8_t* frame = P.in + (uint64_t)pk * P.in_frame_bytes;
      const uint8_t* src0 = frame + (uint64_t)(ro0 * (uint32_t)P.row_step) * P.in_row_bytes + (uint64_t)col0 * pxb;
      // the pixel whose chroma a held row replays (ChromaSubsampler.scala:62-65): loads first, used after the TMA issue.
      // Lanes take rows lane and lane + 32.  In a tall-image launch (KPlan::tall_ho) the held-line rule looks at the row
      // index inside the row's own frame.
      uint32_t hw[kFlexMaxRows / 32];
#pragma unroll
      for (uint32_t u = 0; u < (uint32_t)kFlexMaxRows / 32u; ++u) {
        const uint32_t j = lane + 32u * u;
        uint32_t h0 = 0, h1 = 0, h2 = 0, hvalid = 0;
        if (vhold && j < nrows) {
          const uint32_t ro = ro0 + j;
          uint32_t rf = ro, fr0 = 0;                 // row inside its frame, first launch row of its frame
          if (P.tall_ho) { const uint32_t kf = ro / (uint32_t)P.tall_ho; fr0 = kf * (uint32_t)P.tall_ho; rf = ro - fr0; }
          const uint8_t* hp = nullptr;
          if (!P.case_b) {
            if (f == 1 && (rf & 1u)) hp = frame + (uint64_t)(ro - 1u) * P.in_row_bytes + (uint32_t)P.last_sample_col * ipb;
          } else {
            const uint32_t line = rf >> (31u - __clz(f));   // rf / f (f is 1, 2, 4 or 8); W == f * Wo: one counter line spans f output rows
            if (line & 1u) {
              const uint32_t srow = fr0 + (line - 1u) * f + P.caseb_row_add;
              hp = frame + (uint64_t)(srow * (uint32_t)P.row_step) * P.in_row_bytes + P.caseb_col_bytes;
            }
          }
          if (hp) { h0 = ldg8_now(hp); h1 = ldg8_now(hp + 1); h2 = ldg8_now(hp + 2); hvalid = 0x80000000u; }
        }
        hw[u] = hvalid ? (hvalid | h0 | (h1 << 8) | (h2 << 16)) : 0u;
      }
      if (lane == 0) {
        const uint32_t NWc = NC >> 5, gpr = (ncols + 3u) >> 2, srow = gpr * kUnit, row_out = ncols * kOpx;
        const uint64_t ob = reinterpret_cast<uint64_t>(P.out) + (uint64_t)pk * P.out_frame_bytes + (uint64_t)ro0 * P.out_row_bytes +
                            (uint64_t)col0 * kOpx;
        const uint32_t out_one = (P.out_dense && nsplit == 1u && row_out == srow) ? 1u : 0u;   // whole dense rows: one packed span
        // how the granules are dealt to the consumer threads (flex_consume)
        const uint32_t parts = nrows <= NWc ? NWc / nrows : 0u;                 // warps per row when the rows fit the warps
        uint32_t mode = 3u, sh = 0u;
        if (parts && (parts & (parts - 1u)) == 0u) {
          sh = 31u - __clz(parts);
          const uint32_t lsh = sh + 5u, iters = (gpr + (1u << lsh) - 1u) >> lsh;   // lanes per row = 1 << lsh
          if (gpr * 5u >= (iters << lsh) * 4u) mode = 0u;                       // at least 4/5 of those lanes get a granule
        }
        if (mode != 0u) {
          const uint32_t rounds = (nrows + NWc - 1u) / NWc, li = (gpr + 31u) >> 5;
          if (gpr >= 4u * NC) mode = 1u;
          else if (nrows > NWc && nrows * 5u >= rounds * NWc * 4u && gpr * 5u >= li * 32u * 4u) mode = 2u;
        }
        d->k = pk; d->ro0 = ro0; d->nrows = nrows; d->col0 = col0;
        d->npx = npx; d->a0 = (uint32_t)reinterpret_cast<uintptr_t>(src0) & 15u; d->gpr = gpr; d->last_px = npx - 1u;
        d->obase_lo = (uint32_t)ob; d->obase_hi = (uint32_t)(ob >> 32);
        d->st_mul = out_one ? srow : srow + 16u; d->st_add = out_one ? 0u : P.out_row_bytes;
        d->mode = mode; d->sh = sh; d->magic = gpr > 1u ? 0xFFFFFFFFu / gpr + 1u : 0u;   // q / gpr == umulhi(q, magic) for q < 65536
        d->n_gran = nrows * gpr;
        d->row_out = row_out; d->out_one = out_one; d->ncols = ncols;
        d->direct = 0u;   // (the consumers decide launch-wide: see the dispatch at the end of the kernel)
      }
      if (P.in_dense) {            // consecutive rows are contiguous in memory: one span
        if (lane == 0) span_fetch(in_s, src0, (nrows - 1u) * P.in_row_bytes + len_in, bar, pol, lim_lo, lim_hi);
      } else {                     // one lane per row span: 64 short rows do not queue up behind one thread
        for (uint32_t j = lane; j < nrows; j += 32u)
          span_fetch(in_s + j * rs_mul, src0 + (uint64_t)j * rstep, len_in, bar, pol, lim_lo, lim_hi);
      }
      if (vhold) {
#pragma unroll
        for (uint32_t u = 0; u < (uint32_t)kFlexMaxRows / 32u; ++u)
          sts32(held_base + (s * (uint32_t)kFlexMaxRows + lane + 32u * u) * 4u, hw[u]);
      }
      __syncwarp();
      // releases the descriptor, the held words and the hand-copied edge bytes; the phase completes with the last TMA byte
      if (lane == 0) mbar_arrive(bar);
      // advance by gridDim.x tiles in (frame, row tile, segment) coordinates
      pseg += dseg;
      uint32_t c = pseg >= nsplit ? 1u : 0u;
      pseg -= c * nsplit;
      ptb += dtb + c;
      c = ptb >= P.tiles_per_band ? 1u : 0u;
      ptb -= c * P.tiles_per_band;
      pk += dk + c;
    }
    return;
  }

  // ============================== consumer warps =============================================================
  // One specialisation per (chroma hold width, pixel stride class), chosen once per CTA: no per-tile dispatch, and a
  // CTA only ever runs one copy of the loop (the nine copies used to thrash the instruction cache: ncu showed
  // `no_instruction` stalls of 1.3 per issue on 1366x768 f = 2).
  // narrow output rows that cannot be packed into one span leave from registers (direct_store): a separate
  // specialisation, so that the staged one carries none of its code and registers
  const uint32_t row_out_full = min((uint32_t)P.tile_px, (uint32_t)P.slots_per_row) * kOpx;
  const bool out_one_full = P.out_dense && nsplit == 1u && row_out_full == ((min((uint32_t)P.tile_px, (uint32_t)P.slots_per_row) + 3u) >> 2) * kUnit;
  const bool direct = FMT != KF_PLANAR && nsplit == 1u && !out_one_full && row_out_full < kDirectRowBytes;
  auto run = [&](auto hfe_tag) {
    constexpr uint32_t H = decltype(hfe_tag)::value;
    if (direct) {
      if (pxb == 3u) flex_consume<FMT, TRUNC, H, 3u, true>(P, smem, ring);
      else if (pxb == 6u) flex_consume<FMT, TRUNC, H, 6u, true>(P, smem, ring);
      else flex_consume<FMT, TRUNC, H, 0u, true>(P, smem, ring);
    } else if (pxb == 3u) flex_consume<FMT, TRUNC, H, 3u, false>(P, smem, ring);          // RGB24, f = 1
    else if (pxb == 6u) flex_consume<FMT, TRUNC, H, 6u, false>(P, smem, ring);     // RGB24, f = 2
    else flex_consume<FMT, TRUNC, H, 0u, false>(P, smem, ring);                    // sampled pixels on a common byte phase
  };
  if (hfe == 1u) run(std::integral_constant<uint32_t, 1u>{});
  else if (hfe == 2u) run(std::integral_constant<uint32_t, 2u>{});
  else run(std::integral_constant<uint32_t, 4u>{});
}

KernelFn flex_kernel(int kformat, bool trunc) {
  switch (kformat) {
    case KF_YCC888: return trunc ? csic_flex_kernel<KF_YCC888, true> : csic_flex_kernel<KF_YCC888, false>;
    case KF_RGB888: return trunc ? csic_flex_kernel<KF_RGB888, true> : csic_flex_kernel<KF_RGB888, false>;
    case KF_SLOT8: return trunc ? csic_flex_kernel<KF_SLOT8, true> : csic_flex_kernel<KF_SLOT8, false>;
    case KF_SLOT16: return trunc ? csic_flex_kernel<KF_SLOT16, true> : csic_flex_kernel<KF_SLOT16, false>;
    case KF_PLANAR: return trunc ? csic_flex_kernel<KF_PLANAR, true> : csic_flex_kernel<KF_PLANAR, false>;
    default: return trunc ? csic_flex_kernel<KF_SLOT32, true> : csic_flex_kernel<KF_SLOT32, false>;
  }
}

}  // namespace csic
