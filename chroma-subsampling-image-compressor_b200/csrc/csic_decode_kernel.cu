// csic_decode_kernel -- the PLANAR decoder (Y plane + subsampled Cb / Cr planes -> interleaved YCC888, or RGB888 through
// the reference's YCbCr2RGB, RGB2YCbCr.scala:123-132) as a TMA-staged kernel for ANY frame width and base alignment.
//
// The decoder's two sides are both flat byte streams: a frame's Y plane is Wo * Ho consecutive bytes and its output
// 3 * Wo * Ho consecutive bytes, whatever the width.  So a tile is a run of `tile_px` consecutive pixels of ONE frame
// (a multiple of 16, not a number of rows), and the row structure only matters for finding a pixel's chroma sample:
//
//   load     producer warp, S stages, full / empty mbarriers: one bulk copy for the tile's Y bytes, one each for the
//            stretch of the Cb and the Cr plane its rows sample (first to last sample needed, trimmed inside the first
//            and last chroma row).  Spans keep their offset modulo 16 in shared memory, so the 16-byte hull goes to
//            the TMA engine whatever the alignment (span_fetch, csic_tma.cuh).
//   compute  (row, col) of a thread's pixels are tracked without divisions; three paths, chosen per tile:
//            * rows a multiple of 16 pixels wide with every plane on its 16-byte phase: SIXTEEN pixels per thread -- one
//              LDS.128 of Y, one LDS.128 / .64 / .32 per chroma plane, three STS.128; the hold pattern of each of the four
//              granules is a compile-time constant, so the YCC interleave is 8 PRMTs per granule and the RGB
//              reconstruction computes the chroma terms once per distinct sample (decode_granule_idx);
//            * rows a multiple of 4 pixels: one granule of 4 pixels per thread, samples as one unaligned word (two LDS.32 +
//              funnel shift), compile-time pattern;
//            * any other width: the same with the pattern chosen by the granule's column phase (constant along a row);
//              granules that contain a row end are skipped by the main loop and decoded afterwards, one thread per row
//              end, sample by sample -- one warp pays for the slow lookup instead of every warp that meets a row end.
//            Odd lines of a 4:2:0 / 4:1:0 stream replay the LAST sample of the line above (ChromaSubsampler.scala:52-65):
//            one byte broadcast, chroma terms once per 16 pixels.
//   store    12 bytes per granule into a double-buffered staging area, which leaves as ONE bulk store per tile when the
//            tile's first output byte is word aligned (head / tail bytes up to the next 16-byte boundary by hand), else
//            through span_store.
//
// Algorithmic bytes per output pixel: 1 (Y) + 2 / (hs * vs) (chroma) read, 3 written.
#include <cuda_runtime.h>

#include <cstdint>

#include "csic_internal.h"
#include "csic_device_math.cuh"
#include "csic_tma.cuh"

namespace csic {

namespace {

// Written by the producer before it arms the stage, read by the consumers after the phase flips.
struct DecDesc {
  uint64_t out_g;        // global address of the tile's first output byte
  uint32_t npx;          // pixels in this tile
  uint32_t y_s;          // shared address of the tile's first Y byte
  uint32_t cb_s, cr_s;   // shared address of sample (0, 0) of the frame's chroma planes (biased: sample (r, c) is at + r * cw + c)
  uint32_t r0, col0;     // row and column of the tile's first pixel
  uint32_t nrows;        // rows the tile touches
  uint32_t pad[3];
};
static_assert(sizeof(DecDesc) == kDecDescBytes, "kDecDescBytes out of sync");

// up to four bytes at an arbitrary shared address
__device__ __forceinline__ uint32_t lds_un(uint32_t a) {
  const uint32_t b = a & ~3u;
  return __funnelshift_r(lds32(b), lds32(b + 4), (a & 3u) * 8u);
}

// ---- consumer side: one tile ------------------------------------------------------------------------------------
struct DecTile {
  uint32_t npx, y_s, cb_s, cr_s, r0, col0, nrows, out_s;
};
// How a thread walks the rows: (row, col) of its first group of `px` pixels relative to a tile start, and the step to
// its next group.  Computed once per kernel (four divisions), never per tile.
struct DecWalk {
  uint32_t row_t, col_t, drow, dcol;
};
__device__ __forceinline__ DecWalk make_walk(uint32_t px, uint32_t tid, uint32_t NC, uint32_t Wo) {
  DecWalk w;
  w.row_t = (px * tid) / Wo; w.col_t = px * tid - w.row_t * Wo;
  w.drow = (px * NC) / Wo;   w.dcol = px * NC - w.drow * Wo;
  return w;
}

// Sixteen pixels per thread: rows are a multiple of 16 pixels wide and every plane keeps its 16-byte phase, so a thread's
// Y bytes are one LDS.128, its chroma samples one LDS.128 / .64 / .32 per plane, and its 48 output bytes three STS.128
// (lane stride 48 bytes: conflict free).  The hold pattern of every granule is a compile-time constant.
template <int HS, bool VHOLD, bool RGB>
__device__ __forceinline__ void tile_wide(const DecTile& T, const DecWalk& K, uint32_t Wo, uint32_t cw, uint32_t last_c, uint32_t tid,
                                          uint32_t NC) {
  const uint32_t n16 = T.npx >> 4;
  const uint32_t drow = K.drow, dcol = K.dcol;
  uint32_t row = T.r0 + K.row_t, col = T.col0 + K.col_t;
  if (col >= Wo) { col -= Wo; ++row; }
  for (uint32_t u = tid; u < n16; u += NC) {
    const uint4 yv = lds128(T.y_s + 16u * u);
    const uint32_t yw[4] = {yv.x, yv.y, yv.z, yv.w};
    uint32_t o[12];
    const bool held = VHOLD && (row & 1u);
    const uint32_t cbase = (VHOLD ? (row >> 1) : row) * cw;
    if (held) {
      const uint32_t hb = lds8(T.cb_s + cbase + last_c), hr = lds8(T.cr_s + cbase + last_c);
      if (RGB) {
        const InvChroma t = dec_terms(hb, hr, 0);
#pragma unroll
        for (int i = 0; i < 4; ++i) rgb_granule_terms(yw[i], t, t, t, t, o[3 * i], o[3 * i + 1], o[3 * i + 2]);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) decode_granule_idx<false>(yw[i], hb, hr, 0, 0, 0, 0, o[3 * i], o[3 * i + 1], o[3 * i + 2]);
      }
    } else {
      const uint32_t a = cbase + (col >> HS);
      uint32_t cb[4], cr[4];
      if (HS == 0) {
        const uint4 b = lds128(T.cb_s + a), r = lds128(T.cr_s + a);
        cb[0] = b.x; cb[1] = b.y; cb[2] = b.z; cb[3] = b.w; cr[0] = r.x; cr[1] = r.y; cr[2] = r.z; cr[3] = r.w;
      } else if (HS == 1) {
        const uint2 b = lds64(T.cb_s + a), r = lds64(T.cr_s + a);
        cb[0] = b.x; cb[1] = b.y; cr[0] = r.x; cr[1] = r.y;
      } else {
        cb[0] = lds32(T.cb_s + a); cr[0] = lds32(T.cr_s + a);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t wi = HS == 0 ? i : (HS == 1 ? i >> 1 : 0);                    // chroma word of granule i
        const uint32_t k0 = HS == 0 ? 0u : (HS == 1 ? 2u * (i & 1) : (uint32_t)i);     // its first sample's byte
        const uint32_t s1 = HS == 0 ? 1u : 0u, s2 = HS == 2 ? 0u : (HS == 1 ? 1u : 2u), s3 = HS == 2 ? 0u : (HS == 1 ? 1u : 3u);
        decode_granule_idx<RGB>(yw[i], cb[wi], cr[wi], k0, k0 + s1, k0 + s2, k0 + s3, o[3 * i], o[3 * i + 1], o[3 * i + 2]);
      }
    }
    const uint32_t oa = T.out_s + 48u * u;
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(oa), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(oa + 16u), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(oa + 32u), "r"(o[8]), "r"(o[9]), "r"(o[10]), "r"(o[11]) : "memory");
    col += dcol; row += drow;
    if (col >= Wo) { col -= Wo; ++row; }
  }
}

// One granule (4 flat pixels starting at pixel 4q of the tile = (row, col) of the frame) that lies inside one row: its
// <= 4 samples are one unaligned word, the hold pattern follows the column phase (AL4: rows are a multiple of 4 pixels,
// every granule starts on a sample, the pattern is a compile-time constant).
template <int HS, bool VHOLD, bool RGB, bool AL4>
__device__ __forceinline__ void granule_in_row(const DecTile& T, uint32_t q, uint32_t row, uint32_t col, uint32_t cw, uint32_t last_c) {
  const uint32_t yw = AL4 && (T.y_s & 3u) == 0u ? lds32(T.y_s + 4u * q) : lds_un(T.y_s + 4u * q);
  uint32_t w0, w1, w2;
  const bool held = VHOLD && (row & 1u);
  const uint32_t cbase = (VHOLD ? (row >> 1) : row) * cw;
  if (held) {
    decode_granule_idx<RGB>(yw, lds8(T.cb_s + cbase + last_c), lds8(T.cr_s + cbase + last_c), 0, 0, 0, 0, w0, w1, w2);
  } else {
    const uint32_t a = cbase + (col >> HS);
    const uint32_t cbw = lds_un(T.cb_s + a), crw = lds_un(T.cr_s + a);
    const uint32_t ph = AL4 ? 0u : (col & 3u);
    if (HS == 0) {
      decode_granule_idx<RGB>(yw, cbw, crw, 0, 1, 2, 3, w0, w1, w2);
    } else if (HS == 1) {
      if (ph & 1u) decode_granule_idx<RGB>(yw, cbw, crw, 0, 1, 1, 2, w0, w1, w2);
      else decode_granule_idx<RGB>(yw, cbw, crw, 0, 0, 1, 1, w0, w1, w2);
    } else {
      if (ph == 0u) decode_granule_idx<RGB>(yw, cbw, crw, 0, 0, 0, 0, w0, w1, w2);
      else if (ph == 1u) decode_granule_idx<RGB>(yw, cbw, crw, 0, 0, 0, 1, w0, w1, w2);
      else if (ph == 2u) decode_granule_idx<RGB>(yw, cbw, crw, 0, 0, 1, 1, w0, w1, w2);
      else decode_granule_idx<RGB>(yw, cbw, crw, 0, 1, 1, 1, w0, w1, w2);
    }
  }
  const uint32_t a = T.out_s + q * 12u;
  sts32(a, w0); sts32(a + 4, w1); sts32(a + 8, w2);
}

// A granule that runs over its row's end (or the frame's): four samples looked up one by one.
template <int HS, bool VHOLD, bool RGB>
__device__ __forceinline__ void granule_over_row_end(const DecTile& T, uint32_t q, uint32_t row, uint32_t col, uint32_t Wo, uint32_t cw,
                                                     uint32_t last_c) {
  const uint32_t yw = lds_un(T.y_s + 4u * q);
  uint32_t cbw = 0, crw = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t c = col + j, r = row;
    if (c >= Wo) { c -= Wo; ++r; }
    if (4u * q + j >= T.npx) { c = col; r = row; }            // past the frame's last pixel: never stored
    const bool held = VHOLD && (r & 1u);
    const uint32_t idx = (VHOLD ? (r >> 1) : r) * cw + (held ? last_c : c >> HS);
    cbw |= lds8(T.cb_s + idx) << (8 * j);
    crw |= lds8(T.cr_s + idx) << (8 * j);
  }
  uint32_t w0, w1, w2;
  decode_granule_idx<RGB>(yw, cbw, crw, 0, 1, 2, 3, w0, w1, w2);
  const uint32_t a = T.out_s + q * 12u;
  sts32(a, w0); sts32(a + 4, w1); sts32(a + 8, w2);
}

// Four pixels per thread, any width.  Granules that contain a row end are left out of the main loop and decoded
// afterwards, one thread per row end: one warp pays for the slow lookup instead of every warp that meets a row end
// (1918-pixel rows: every fourth warp; 333-pixel rows: every third).
template <int HS, bool VHOLD, bool RGB, bool AL4>
__device__ __forceinline__ void tile_granules(const DecTile& T, const DecWalk& K, uint32_t Wo, uint32_t cw, uint32_t last_c, uint32_t tid,
                                              uint32_t NC) {
  const uint32_t n_gran = (T.npx + 3u) >> 2;
  const uint32_t drow = K.drow, dcol = K.dcol;
  uint32_t row = T.r0 + K.row_t, col = T.col0 + K.col_t;
  if (col >= Wo) { col -= Wo; ++row; }
  for (uint32_t q = tid; q < n_gran; q += NC) {
    if (AL4 || col + 3u < Wo) granule_in_row<HS, VHOLD, RGB, AL4>(T, q, row, col, cw, last_c);
    col += dcol; row += drow;
    if (col >= Wo) { col -= Wo; ++row; }
  }
  if (!AL4) {
    // row end number bi sits at tile pixel e = (bi + 1) * Wo - col0; it cuts a granule unless e is a multiple of 4
    const uint32_t nb = T.nrows;                                  // rows the tile touches
    for (uint32_t bi = tid; bi < nb; bi += NC) {
      const uint32_t e = (bi + 1u) * Wo - T.col0;
      if (e <= T.npx && (e & 3u) != 0u) {
        const uint32_t q = e >> 2;
        granule_over_row_end<HS, VHOLD, RGB>(T, q, T.r0 + bi, Wo - (e - 4u * q), Wo, cw, last_c);
      }
    }
  }
}

template <int HS, bool VHOLD, bool RGB>
__global__ void __launch_bounds__(kDecMaxConsumers + 32) csic_decode_kernel(const __grid_constant__ DecPlan P) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t tid = threadIdx.x;
  const uint32_t NC = blockDim.x - 32u;          // consumer threads; the last warp is the producer
  const uint32_t sbase = smem_u32(smem);
  const uint64_t pol = policy_evict_first();
  const Ring ring(sbase + P.bar_off, P.stages, P.n_tiles);
  ring.init(NC / 32u);                           // one arrive per consumer warp

  // ============================== producer warp ==============================================
  if (tid >= NC) {
    const uint32_t lane = tid - NC;
    Ring::Pos pos;
    for (uint32_t i = 0; i < ring.n_my; ++i, pos.next(ring.S)) {
      const uint32_t s = pos.s;
      ring.wait_empty(pos, i);
      if (lane < 3u) {
        const uint32_t tile = blockIdx.x + i * gridDim.x;
        const uint32_t k = tile / P.tiles_per_frame, tt = tile - k * P.tiles_per_frame;
        const uint32_t p0 = tt * P.tile_px, npx = min(P.tile_px, P.A - p0), p1 = p0 + npx - 1u;
        const uint32_t r0 = p0 / P.Wo, col0 = p0 - r0 * P.Wo, r1 = p1 / P.Wo, col1 = p1 - r1 * P.Wo;
        const uint8_t* frame = P.planar + (uint64_t)k * P.frame_bytes;
        const uint32_t bar = ring.full(s);
        const uint32_t slot = sbase + s * P.stage_stride;
        DecDesc* d = reinterpret_cast<DecDesc*>(smem + P.desc_off) + s;
        if (lane == 0) {
          const uint8_t* y = frame + p0;
          span_fetch(slot, y, npx, bar, pol, (uintptr_t)P.lim_lo, (uintptr_t)P.lim_hi);
          d->out_g = reinterpret_cast<uint64_t>(P.out) + ((uint64_t)k * P.A + p0) * 3u;
          d->npx = npx;
          d->y_s = slot + ((uint32_t)reinterpret_cast<uintptr_t>(y) & 15u);
          d->r0 = r0;
          d->col0 = col0;
          d->nrows = r1 - r0 + 1u;
        } else {
          // first and last sample this tile reads: odd (held) lines read sample last_c of the chroma row they share with
          // the line above, which -- when that line is in the tile too -- is read to its end
          const bool h0 = VHOLD && (r0 & 1u), h1 = VHOLD && (r1 & 1u);
          const uint32_t first = (VHOLD ? r0 >> 1 : r0) * P.cw + (h0 ? P.last_c : col0 >> HS);
          const uint32_t last = (VHOLD ? r1 >> 1 : r1) * P.cw + (h1 ? (r1 > r0 ? P.cw - 1u : P.last_c) : col1 >> HS);
          const uint8_t* plane = frame + (lane == 1u ? P.cb_off : P.cr_off);
          const uint32_t cslot = slot + P.y_slot + (lane - 1u) * P.c_slot;
          span_fetch(cslot, plane + first, last - first + 1u, bar, pol, (uintptr_t)P.lim_lo, (uintptr_t)P.lim_hi);
          const uint32_t bias = cslot + ((uint32_t)reinterpret_cast<uintptr_t>(plane + first) & 15u) - first;
          if (lane == 1u) d->cb_s = bias; else d->cr_s = bias;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(ring.full(s));
    }
    return;
  }

  // ============================== consumer warps =============================================
  const uint32_t Wo = P.Wo, cw = P.cw, last_c = P.last_c;
  const bool w16 = (Wo & 15u) == 0u, w4 = (Wo & 3u) == 0u;
  const DecWalk walk16 = make_walk(16u, tid, NC, Wo), walk4 = make_walk(4u, tid, NC, Wo);
  Ring::Pos pos;
  for (uint32_t i = 0; i < ring.n_my; ++i, pos.next(ring.S)) {
    const uint32_t s = pos.s;
    ring.wait_full(pos);
    const DecDesc* d = reinterpret_cast<const DecDesc*>(smem + P.desc_off) + s;
    DecTile T;
    T.npx = d->npx; T.y_s = d->y_s; T.cb_s = d->cb_s; T.cr_s = d->cr_s; T.r0 = d->r0; T.col0 = d->col0; T.nrows = d->nrows;
    uint8_t* out_g = reinterpret_cast<uint8_t*>(d->out_g);
    const uint32_t galign = (uint32_t)d->out_g & 15u;
    // staging: byte b of the tile at out_s + b, out_s = buffer + (address of the first output byte mod 16, to the word)
    T.out_s = sbase + P.out_off + (i & 1u) * P.out_stride + (galign & 12u);
    // every plane on its 16-byte phase: the 16-pixel path
    const bool wide = w16 && (galign & 12u) == 0u && (T.y_s & 15u) == 0u && ((T.cb_s | T.cr_s) & ((16u >> HS) - 1u)) == 0u;
    if (wide) tile_wide<HS, VHOLD, RGB>(T, walk16, Wo, cw, last_c, tid, NC);
    else if (w4) tile_granules<HS, VHOLD, RGB, true>(T, walk4, Wo, cw, last_c, tid, NC);
    else tile_granules<HS, VHOLD, RGB, false>(T, walk4, Wo, cw, last_c, tid, NC);
    // inputs consumed: the stage goes back to the producer
    __syncwarp();
    if ((tid & 31u) == 0) mbar_arrive(ring.empty(s));

    const uint32_t len = T.npx * 3u;
    if ((galign & 3u) == 0u) {
      // word-aligned output: the staging offset equals the global offset modulo 16, so the 16-byte interior is one
      // bulk store; up to 15 head and 15 tail bytes by hand
      fence_proxy_async_smem();
      if (tid == 0) tma_store_wait_read0();
      consumer_barrier(NC);
      const uint32_t head = min(len, (16u - galign) & 15u), body = (len - head) & ~15u, tail = len - head - body;
      if (tid == 0 && body) {
        tma_store_1d(out_g + head, T.out_s + head, body, pol);
        tma_store_commit();
      }
      if (tid >= 32u && tid < 32u + head) out_g[tid - 32u] = (uint8_t)lds8(T.out_s + tid - 32u);           // NC >= 64
      if (tid >= 48u && tid < 48u + tail) out_g[head + body + tid - 48u] = (uint8_t)lds8(T.out_s + head + body + tid - 48u);
    } else {
      if (tid == 0) tma_store_wait_read0();
      consumer_barrier(NC);
      span_store(out_g, T.out_s, len, tid, NC);
    }
  }
  if (tid == 0) tma_store_wait_all();
}

template <int HS, bool VHOLD>
DecodeFn by_rgb(bool to_rgb) { return to_rgb ? csic_decode_kernel<HS, VHOLD, true> : csic_decode_kernel<HS, VHOLD, false>; }
template <bool VHOLD>
DecodeFn by_hs(uint32_t hs_sh, bool to_rgb) {
  return hs_sh == 0 ? by_rgb<0, VHOLD>(to_rgb) : (hs_sh == 1 ? by_rgb<1, VHOLD>(to_rgb) : by_rgb<2, VHOLD>(to_rgb));
}

}  // namespace

DecodeFn decode_kernel(uint32_t hs_sh, bool vhold, bool to_rgb) {
  return vhold ? by_hs<true>(hs_sh, to_rgb) : by_hs<false>(hs_sh, to_rgb);
}

int launch_decode_tma(const DecodeLaunch& d, void* stream) {
  decode_kernel(d.P.hs_sh, d.P.vhold, d.P.to_rgb)<<<d.grid, d.threads, d.smem, (cudaStream_t)stream>>>(d.P);
  return (int)cudaGetLastError();
}

}  // namespace csic
