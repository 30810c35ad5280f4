// TMA / mbarrier / shared-memory PTX wrappers shared by the TMA-staged kernels (sm_100a), and their common skeleton: the
// stage ring and the row tiles.
#ifndef CSIC_TMA_CUH_
#define CSIC_TMA_CUH_
#include <cuda_runtime.h>
#include <cstdint>

#include "csic_internal.h"

namespace csic {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// adds to the transaction count without arriving: several lanes can each announce their own bulk copy, one of them
// arrives afterwards (behind a __syncwarp)
__device__ __forceinline__ void mbar_expect_tx_only(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// named barrier 1 over the consumer threads only (the producer warp never joins it)
__device__ __forceinline__ void consumer_barrier(uint32_t n_threads) {
  asm volatile("bar.sync 1, %0;" ::"r"(n_threads) : "memory");
}
// Blocks until the barrier's phase with the given parity completes.  try_wait suspends the warp in hardware; the
// suspend-time hint keeps it asleep until the phase flips instead of returning early to spin (ncu showed the
// retry loop -- BRA / SYNCS.TRYWAIT / YIELD -- taking ~30 % of the issued instructions of the pooling kernel).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "CSIC_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra CSIC_DONE_%=;\n\t"
      "bra CSIC_WAIT_%=;\n\t"
      "CSIC_DONE_%=:\n\t}"
      ::"r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
}
// global -> shared bulk copy performed by the TMA engine; completion counted in bytes on `bar`.
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(pol)
      : "memory");
}
// shared -> global bulk copy (bulk async-group completion).
__device__ __forceinline__ void tma_store_1d(void* dst, uint32_t src, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src),
               "r"(bytes), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// The S-stage ring of a TMA-staged kernel.  The producer warp fills stage s and arrives on full(s) (its bulk copies add
// their bytes to that phase); the consumers wait on full(s), use the stage and arrive on empty(s), on which the producer
// waits before it refills the stage.  Barriers at `bar`: full[S], then empty[S] (kRingBarBytes per stage).  A CTA
// walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... of n_tiles: n_my of them.
struct Ring {
  uint32_t bar, ebar, S, n_my;
  // Stage of a tile and the parity of the barrier phase it waits for, which flips each lap of the ring.
  struct Pos {
    uint32_t s = 0, ph = 0;
    __device__ __forceinline__ void next(uint32_t S) {
      if (++s == S) { s = 0; ph ^= 1u; }
    }
  };
  __device__ __forceinline__ Ring(uint32_t bar_, uint32_t stages, uint32_t n_tiles)
      : bar(bar_), ebar(bar_ + stages * 8u), S(stages),
        n_my(n_tiles > blockIdx.x ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0) {}
  // the position of this CTA's i-th tile, for loops that would rather divide than carry a Pos (the row and pooling
  // kernels: counters there cost registers)
  __device__ __forceinline__ Pos at(uint32_t i) const {
    Pos p;
    p.s = i % S;
    p.ph = (i / S) & 1u;
    return p;
  }
  __device__ __forceinline__ uint32_t full(uint32_t s) const { return bar + s * 8u; }
  __device__ __forceinline__ uint32_t empty(uint32_t s) const { return ebar + s * 8u; }
  // full[] counts the producer's one arrive, empty[] `empty_arrivals` consumer arrives; every thread of the CTA calls it
  __device__ __forceinline__ void init(uint32_t empty_arrivals) const {
    if (threadIdx.x == 0) {
      for (uint32_t s = 0; s < S; ++s) {
        mbar_init(full(s), 1);
        mbar_init(empty(s), empty_arrivals);
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  // producer, before it fills the i-th tile's stage: from the second lap on, the consumers must have drained its last use
  __device__ __forceinline__ void wait_empty(const Pos& p, uint32_t i) const {
    if (i >= S) mbar_wait(empty(p.s), p.ph ^ 1u);
  }
  // consumers: the stage's bytes have landed and the producer's shared-memory writes are visible
  __device__ __forceinline__ void wait_full(const Pos& p) const { mbar_wait(full(p.s), p.ph); }
};
static_assert(kRingBarBytes == 2u * 8u, "a ring stage has one 8-byte full and one 8-byte empty mbarrier");

// Ticket dealing of a persistent grid's tiles (the row kernel in a ticketed plan, KPlan::ticketed): a CTA's first tile is
// blockIdx.x, each further one gridDim.x + the next value of a counter every CTA of the launch draws from, so that CTAs
// that run ahead take more tiles and the grid stays on one narrow band of the batch instead of drifting apart over a
// static round robin (cfg4 on a B200: 1.3 frames in flight at the median instead of 82, profiles/r3/README.md).
// `ctr` is a pair of words that is zero when the launch starts: [0] tickets drawn, [1] CTAs done drawing.  A CTA calls
// leave() once, after its last take(); the last one to leave has seen every take() of the launch and zeroes the pair,
// so the next launch in stream order finds it zero again -- no memset, no host bookkeeping.  Launches that share a pair
// must therefore never overlap (csic_api.cu: one pair per stream, none for launches captured into a graph).
struct TileDeal {
  uint32_t* ctr;
  __device__ __forceinline__ uint32_t take() const { return gridDim.x + atomicAdd(ctr, 1u); }
  __device__ __forceinline__ void leave() const {
    if (atomicAdd(ctr + 1, 1u) == gridDim.x - 1u) {
      atomicExch(ctr, 0u);
      atomicExch(ctr + 1, 0u);
    }
  }
};

// Tile `tile` of the row and pooling kernels: segment seg of row tile tb of frame k (tile = (k * tiles_per_band + tb) *
// nsplit + seg), output rows [ro0, ro0 + nrows).
struct RowTile {
  uint32_t seg, k, ro0, nrows;
};
__device__ __forceinline__ RowTile row_tile(const KPlan& P, uint32_t tile) {
  RowTile t;
  const uint32_t t2 = tile / (uint32_t)P.nsplit;
  t.seg = tile - t2 * (uint32_t)P.nsplit;
  t.k = t2 / P.tiles_per_band;
  const uint32_t tb = t2 - t.k * P.tiles_per_band;
  t.ro0 = (uint32_t)P.row0 + tb * (uint32_t)P.tile_rows;
  t.nrows = min((uint32_t)P.tile_rows, (uint32_t)(P.row0 + P.band_rows) - t.ro0);
  return t;
}

__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds8(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

__device__ __forceinline__ void sts8(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// Producer side (one thread per span).  global [g, g+len) -> shared, byte i at  slot + (g & 15) + i  (slot 16-byte aligned):
// the 16-byte hull of the span goes to the TMA engine; where the hull would leave [lo, hi) -- the byte range this
// launch may touch -- it is clipped and the < 16 edge bytes are copied by hand (first / last span of a launch only).
__device__ __forceinline__ void span_fetch(uint32_t slot, const uint8_t* __restrict__ g, uint32_t len, uint32_t bar, uint64_t pol,
                                           uintptr_t lo, uintptr_t hi) {
  const uintptr_t A = reinterpret_cast<uintptr_t>(g), B = A + len, base = A & ~(uintptr_t)15;
  uintptr_t start = base, end = (B + 15) & ~(uintptr_t)15;
  if (start < lo) start += 16;                   // then start > A: head bytes [A, min(start, B)) by hand
  if (end > hi) end -= 16;                       // then end < B: tail bytes by hand
  if (end > start) {
    const uint32_t n = (uint32_t)(end - start);
    mbar_expect_tx_only(bar, n);
    tma_load_1d(slot + (uint32_t)(start - base), reinterpret_cast<const void*>(start), n, bar, pol);
  }
  if (start > A || end < B) {
    const uint8_t* gb = reinterpret_cast<const uint8_t*>(base);
    const uintptr_t h1 = start > A ? (start < B ? start : B) : A;          // head is [A, h1)
    const uintptr_t t0 = end < B ? (end > h1 ? end : h1) : B;              // tail is [t0, B)
    for (uintptr_t x = A; x < h1; ++x) sts8(slot + (uint32_t)(x - base), __ldg(gb + (x - base)));
    for (uintptr_t x = t0; x < B; ++x) sts8(slot + (uint32_t)(x - base), __ldg(gb + (x - base)));
  }
}

// The four sampled pixels of a granule, each as a word whose low three bytes are R,G,B.
// A granule is 4 consecutive output pixels = 4 input pixels at a stride of F pixels (3F bytes);
// `a` is the shared-memory address of its first byte.
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}

// shared [ssrc, ssrc+len) -> global [g, g+len): 16-byte stores aligned on the global address.  The staging rows are
// laid out so that (ssrc & 12) == (g & 12): the shared side of a chunk is then one LDS.128, plus one word when the
// low two address bits differ.
__device__ __forceinline__ void span_store(uint8_t* __restrict__ g, uint32_t ssrc, uint32_t len, uint32_t t,
                                           uint32_t nthr) {
  const uint32_t head = min(len, (16u - ((uint32_t)reinterpret_cast<uintptr_t>(g) & 15u)) & 15u);
  const uint32_t nchunk = (len - head) >> 4;
  const uint32_t tail = len - head - (nchunk << 4);
  const uint32_t s0 = ssrc + head, sa = s0 & ~3u, sh = (s0 & 3u) * 8u;
  if (sh == 0 && (sa & 15u) == 0) {
    for (uint32_t c = t; c < nchunk; c += nthr) __stcs(reinterpret_cast<uint4*>(g + head + (c << 4)), lds128(sa + (c << 4)));
  } else if ((sa & 15u) == 12u) {
    for (uint32_t c = t; c < nchunk; c += nthr) {
      const uint32_t a = sa + (c << 4);
      const uint32_t w0 = lds32(a);
      const uint4 v = lds128(a + 4);
      __stcs(reinterpret_cast<uint4*>(g + head + (c << 4)),
             make_uint4(__funnelshift_r(w0, v.x, sh), __funnelshift_r(v.x, v.y, sh), __funnelshift_r(v.y, v.z, sh),
                        __funnelshift_r(v.z, v.w, sh)));
    }
  } else {
    for (uint32_t c = t; c < nchunk; c += nthr) {
      const uint32_t a = sa + (c << 4);
      const uint32_t w0 = lds32(a), w1 = lds32(a + 4), w2 = lds32(a + 8), w3 = lds32(a + 12), w4 = lds32(a + 16);
      __stcs(reinterpret_cast<uint4*>(g + head + (c << 4)),
             make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                        __funnelshift_r(w3, w4, sh)));
    }
  }
  for (uint32_t i = nthr - 1u - t; i < head + tail; i += nthr) {
    const uint32_t off = i < head ? i : len - tail + (i - head);
    g[off] = (uint8_t)lds8(ssrc + off);
  }
}


// A granule's output bytes straight from registers to global memory (rows too narrow for the staged path to pay: there
// every 150-byte row costs a warp ~120 instructions of span_store set-up, head and tail).  `w` holds the granule's
// little-endian words, `nbytes` of which exist (the row's last granule may be partial); the widest stores the address
// allows -- words, half words or bytes.  Rows are contiguous in memory and written by one CTA within microseconds, so
// L2 merges the partial sectors before they reach HBM.
template <int NW_>
__device__ __forceinline__ void direct_store(uint8_t* __restrict__ gp, const uint32_t (&w)[NW_], uint32_t nbytes) {
  const uint32_t al = (uint32_t)reinterpret_cast<uintptr_t>(gp) & 3u;
  if (al == 0u) {
#pragma unroll
    for (int i = 0; i < NW_; ++i) {
      if (4u * i + 4u <= nbytes) __stcs(reinterpret_cast<uint32_t*>(gp) + i, w[i]);
      else {
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if (4u * i + b < nbytes) gp[4 * i + b] = (uint8_t)(w[i] >> (8 * b));
      }
    }
  } else if (al == 2u) {
#pragma unroll
    for (int i = 0; i < 2 * NW_; ++i) {
      const uint32_t h = (w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu;
      if (2u * i + 2u <= nbytes) __stcs(reinterpret_cast<unsigned short*>(gp) + i, (unsigned short)h);
      else if (2u * i < nbytes) gp[2 * i] = (uint8_t)h;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4 * NW_; ++i)
      if ((uint32_t)i < nbytes) gp[i] = (uint8_t)(w[i >> 2] >> (8 * (i & 3)));
  }
}

}  // namespace csic
#endif  // CSIC_TMA_CUH_
