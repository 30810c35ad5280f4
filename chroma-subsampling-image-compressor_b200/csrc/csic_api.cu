// Device half of the C ABI: contexts, the device / band / host entry points (plans come from csic_plan.cpp).
// No CPU compute path exists here: every process call ends in a kernel launch or an error code.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "csic_internal.h"

namespace {

thread_local std::string g_last_error;

int cuda_fail(cudaError_t e, const char* what) {
  g_last_error = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInitializationError)
             ? CSIC_ENODEVICE
             : (e == cudaErrorMemoryAllocation ? CSIC_ENOMEM : CSIC_ECUDA);
}

#define CSIC_CUDA(call)                                   \
  do {                                                    \
    cudaError_t e__ = (call);                             \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

using csic::kPipe;
// Input bytes per pipelined chunk.  B200 + PCIe 5 x16, 4K batches (profiles/r2/e2e_chunk_sweep.txt): 16 MB 32.6 k MP/s,
// 32 MB 32.3 k, 64 MB (round 1) 31.9 k, 128 MB 31.3 k -- the pipeline's fill and drain cost one chunk each per call.
constexpr size_t kDefaultChunkBytes = 16u << 20;

// No C++ exception may cross the C ABI (the caller is a JVM, Python or C): std::thread / std::vector / std::string can
// throw system_error or bad_alloc inside the host pipeline.
template <typename F>
int guarded(const char* where, F&& body) {
  try {
    return body();
  } catch (const std::bad_alloc&) {
    g_last_error = std::string(where) + ": out of host memory";
    return CSIC_ENOMEM;
  } catch (const std::exception& e) {
    g_last_error = std::string(where) + ": " + e.what();
    return CSIC_ECUDA;
  } catch (...) {
    g_last_error = std::string(where) + ": unknown C++ exception";
    return CSIC_ECUDA;
  }
}

}  // namespace

struct csic_ctx {
  int device = 0;
  csic::DeviceLimits dev = {};
  cudaStream_t stream = nullptr;             // default compute stream
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  struct Ring { void* buf[kPipe] = {}; size_t cap = 0; } d_in, d_out;   // device staging: kPipe buffers of cap bytes
  Ring h_in, h_out;                          // pinned bounce buffers for pageable callers
  cudaEvent_t ev_h2d[kPipe] = {}, ev_k[kPipe] = {}, ev_d2h[kPipe] = {};
  int opt_no_bounce = 0;
  int last_family = 0;
  int64_t launches = 0;
  csic::PlanOptions opt;                     // csic_set_option's planner knobs
  size_t opt_chunk_bytes = kDefaultChunkBytes;
  int opt_no_compact = 0;
  uint64_t h2d_bytes = 0;    // bytes csic_process_host has shipped host -> device so far
};

namespace {

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int run(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t n_frames, void* d_out, int32_t row0,
        int32_t rows, void* cuda_stream, bool compact = false, const csic::Layout& lay = csic::Layout()) {
  if (!ctx || !p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  if (n_frames == 0 || rows == 0) return CSIC_OK;
  if (!d_rgb || !d_out) return CSIC_EINVAL_ARG;
  csic::KPlan base;
  rc = csic::build_plan(*p, d_rgb, d_out, n_frames, row0, rows, compact, lay, base);
  if (rc != CSIC_OK) return rc;
  if (row0 < 0 || rows < 0 || row0 + rows > base.Ho) return CSIC_EINVAL_ARG;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  const csic::KernelChoice c = csic::select_kernel(base, ctx->dev, ctx->opt);
  const int err = csic::launch(c, st);
  ctx->last_family = c.family;
  ctx->launches += 1;
  if (err != (int)cudaSuccess) return cuda_fail((cudaError_t)err, "kernel launch");
  return CSIC_OK;
}

// Grows one ring of staging buffers (device or pinned: alloc / release) to at least `bytes` each.
template <typename Alloc, typename Release>
int grow_ring(csic_ctx::Ring& r, size_t bytes, Alloc alloc, Release release) {
  if (bytes <= r.cap) return CSIC_OK;
  for (void*& b : r.buf) { if (b) release(b); b = nullptr; }
  r.cap = 0;
  for (void*& b : r.buf) CSIC_CUDA(alloc(&b, bytes));
  r.cap = bytes;
  return CSIC_OK;
}

}  // namespace

extern "C" {

const char* csic_last_error(void) { return g_last_error.c_str(); }

int csic_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cuda_fail(e, "cudaGetDeviceCount");
    return CSIC_ENODEVICE;
  }
  return n;
}

int csic_create(int device, csic_ctx** out) {
  if (!out) return CSIC_EINVAL_ARG;
  *out = nullptr;
  int n = csic_device_count();
  if (n <= 0) return CSIC_ENODEVICE;
  if (device < 0 || device >= n) return CSIC_EINVAL_ARG;
  csic_ctx* c = new (std::nothrow) csic_ctx();
  if (!c) return CSIC_ENOMEM;
  c->device = device;
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { delete c; return cuda_fail(e, "cudaGetDeviceProperties"); }
  if (prop.major < 10) {   // the row kernel is written for sm_100a only; there is no other build
    delete c;
    g_last_error = "device is not sm_100 (Blackwell B200); this library is built for sm_100a only";
    return CSIC_ENODEVICE;
  }
  c->dev = {prop.multiProcessorCount, prop.sharedMemPerBlockOptin};
  // keep the FIRST failing call's own error code (cudaGetLastError may already read cudaSuccess again), and tear down
  // whatever was created before it
  cudaError_t err = cudaSuccess;
  auto step = [&](cudaError_t r) { if (err == cudaSuccess) err = r; return err == cudaSuccess; };
  step(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) &&
      step(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking)) &&
      step(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
  for (int i = 0; err == cudaSuccess && i < kPipe; ++i)
    step(cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming)) &&
        step(cudaEventCreateWithFlags(&c->ev_k[i], cudaEventDisableTiming)) &&
        step(cudaEventCreateWithFlags(&c->ev_d2h[i], cudaEventDisableTiming));
  if (err == cudaSuccess) step((cudaError_t)csic::set_kernel_attributes(c->dev.max_smem_optin));
  if (err != cudaSuccess) {
    const int rc = cuda_fail(err, "csic_create");
    const std::string keep = g_last_error;
    cudaGetLastError();
    csic_destroy(c);
    g_last_error = keep;
    return rc;
  }
  *out = c;
  return CSIC_OK;
}

int csic_destroy(csic_ctx* ctx) {
  if (!ctx) return CSIC_OK;
  DeviceGuard guard(ctx->device);
  for (cudaStream_t st : {ctx->stream, ctx->s_h2d, ctx->s_d2h})
    if (st) cudaStreamSynchronize(st);
  for (int i = 0; i < kPipe; ++i) {
    if (ctx->d_in.buf[i]) cudaFree(ctx->d_in.buf[i]);
    if (ctx->d_out.buf[i]) cudaFree(ctx->d_out.buf[i]);
    if (ctx->h_in.buf[i]) cudaFreeHost(ctx->h_in.buf[i]);
    if (ctx->h_out.buf[i]) cudaFreeHost(ctx->h_out.buf[i]);
    if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]);
    if (ctx->ev_k[i]) cudaEventDestroy(ctx->ev_k[i]);
    if (ctx->ev_d2h[i]) cudaEventDestroy(ctx->ev_d2h[i]);
  }
  for (cudaStream_t st : {ctx->stream, ctx->s_h2d, ctx->s_d2h})
    if (st) cudaStreamDestroy(st);
  delete ctx;
  return CSIC_OK;
}

int csic_set_option(csic_ctx* ctx, int option, int64_t value) {
  if (!ctx) return CSIC_EINVAL_ARG;
  switch (option) {
    case CSIC_OPT_KERNEL_FAMILY:
      if (value < 0 || value > 2) return CSIC_EINVAL_ARG;
      ctx->opt.family = (int)value;
      return CSIC_OK;
    case CSIC_OPT_HOST_CHUNK_BYTES:
      if (value < 0) return CSIC_EINVAL_ARG;
      ctx->opt_chunk_bytes = value == 0 ? kDefaultChunkBytes : (size_t)value;
      return CSIC_OK;
    case CSIC_OPT_GRID_CTAS_PER_SM:
      if (value < 0 || value > 32) return CSIC_EINVAL_ARG;
      ctx->opt.ctas_per_sm = (int)value;
      return CSIC_OK;
    case CSIC_OPT_STAGES:
      if (value < 0 || value > 16 || value == 1) return CSIC_EINVAL_ARG;
      ctx->opt.stages = (int)value;
      return CSIC_OK;
    case CSIC_OPT_BLOCK_THREADS:
      if (value < 0 || value > 512 || (value % 32) != 0) return CSIC_EINVAL_ARG;
      ctx->opt.block_threads = (int)value;
      return CSIC_OK;
    case CSIC_OPT_HOST_FULL_FRAMES:
      ctx->opt_no_compact = value != 0;
      return CSIC_OK;
    case CSIC_OPT_HOST_NO_BOUNCE:
      ctx->opt_no_bounce = value != 0;
      return CSIC_OK;
    case CSIC_OPT_TILE_BYTES:
      if (value < 0 || value > (200 << 10)) return CSIC_EINVAL_ARG;
      ctx->opt.tile_bytes = (uint32_t)value;
      return CSIC_OK;
    default:
      return CSIC_EINVAL_ARG;
  }
}

int csic_process_device(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t n_frames, void* d_out,
                        void* cuda_stream) {
  if (!p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  const csic::Geometry g = csic::geometry(*p);
  return run(ctx, p, d_rgb, n_frames, d_out, 0, g.out_h, cuda_stream);
}

int csic_process_device_pitched(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t in_pitch_bytes,
                                size_t in_frame_stride, size_t n_frames, void* d_out, size_t out_pitch_bytes,
                                size_t out_frame_stride, void* cuda_stream) {
  if (!p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  const csic::Geometry g = csic::geometry(*p);
  const csic::Layout lay{in_pitch_bytes, in_frame_stride, out_pitch_bytes, out_frame_stride};
  return run(ctx, p, d_rgb, n_frames, d_out, 0, g.out_h, cuda_stream, false, lay);
}

int csic_expand_planar_device(csic_ctx* ctx, const csic_params* p, const void* d_planar, size_t n_frames, void* d_out,
                              int32_t expand_format, void* cuda_stream) {
  if (!ctx || !p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  if (p->out_format != CSIC_OUT_PLANAR || (expand_format != CSIC_OUT_YCC888 && expand_format != CSIC_OUT_RGB888))
    return CSIC_EINVAL_MODE;
  if (n_frames == 0) return CSIC_OK;
  if (!d_planar || !d_out) return CSIC_EINVAL_ARG;
  const csic::Geometry g = csic::geometry(*p);
  csic::KPlan k;
  rc = csic::build_plan(*p, d_planar, d_out, n_frames, 0, g.out_h, false, csic::Layout(), k);
  if (rc != CSIC_OK) return rc;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  const int to_rgb = expand_format == CSIC_OUT_RGB888;
  // test switches, read per call: the LDG decoder instead of the TMA-staged one; pixels per tile
  const bool no_tma = std::getenv("CSIC_DEC_NO_TMA") != nullptr;
  const char* tile = std::getenv("CSIC_DEC_TILE");
  const long tile_px = tile ? std::strtol(tile, nullptr, 10) : 0;
  // what the TMA-staged decoder declines (rows narrower than a granule, chroma rows too wide for a stage) runs on LDG
  csic::DecodeLaunch d;
  const int err = !no_tma && csic::plan_decode(k, to_rgb, ctx->dev, tile_px > 0 ? (uint32_t)tile_px : 0u, d)
                      ? csic::launch_decode_tma(d, st)
                      : csic::launch_expand_planar(k, to_rgb, ctx->dev.sm_count, st);
  ctx->launches += 1;
  if (err != (int)cudaSuccess) return cuda_fail((cudaError_t)err, "expand kernel launch");
  return CSIC_OK;
}

int csic_process_band(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t n_frames, void* d_out,
                      int32_t out_row0, int32_t out_rows, void* cuda_stream) {
  return run(ctx, p, d_rgb, n_frames, d_out, out_row0, out_rows, cuda_stream);
}

namespace {

bool is_pageable(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

// One copy of csic::frame_copies between host buffers, on several host threads: a pageable caller's rows are gathered
// into / scattered from the pinned bounce buffers at host memory speed instead of the driver's single-threaded staging.
void host_copy(uint8_t* dst, const uint8_t* src, const csic::Copy& c) {
  const size_t total = c.width * c.height;
  unsigned T = std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency() / 2));
  if (total < (4u << 20)) T = 1;
  const bool contiguous = !c.dst_pitch || (c.dst_pitch == c.width && c.src_pitch == c.width);
  // contiguous ranges are cut by bytes (a "row" may be a whole frame), strided ones by rows
  const size_t units = contiguous ? total : c.height;
  auto work = [=](size_t u0, size_t u1) {
    if (contiguous) {
      std::memcpy(dst + c.dst + u0, src + c.src + u0, u1 - u0);
    } else {
      for (size_t r = u0; r < u1; ++r) std::memcpy(dst + c.dst + r * c.dst_pitch, src + c.src + r * c.src_pitch, c.width);
    }
  };
  if (T == 1) { work(0, units); return; }
  std::vector<std::thread> th;
  for (unsigned t = 1; t < T; ++t) th.emplace_back(work, units * t / T, units * (t + 1) / T);
  work(0, units / T);
  for (std::thread& x : th) x.join();
}

// Issues the copies of csic::frame_copies between host and device buffers (or back) on `st`.
int device_copies(uint8_t* dst, const uint8_t* src, const std::vector<csic::Copy>& cs, cudaMemcpyKind dir,
                  cudaStream_t st) {
  for (const csic::Copy& c : cs)
    CSIC_CUDA(c.dst_pitch ? cudaMemcpy2DAsync(dst + c.dst, c.dst_pitch, src + c.src, c.src_pitch, c.width, c.height, dir, st)
                          : cudaMemcpyAsync(dst + c.dst, src + c.src, c.width, dir, st));
  return CSIC_OK;
}

}  // namespace

// Host buffers in, host buffers out, for output rows [row0, row0+rows) of every frame (the whole frame or one
// row band).  Frames are cut into chunks that flow through a kPipe-deep ring of device buffers on three streams.
// Only what the band needs crosses PCIe: its input rows (every f-th one under DECIMATE) and its output rows; the
// device buffers hold just those rows and the kernel is handed *virtual* frame bases (buffer - first_row * pitch).
// `share` (optional): a cursor several contexts (GPUs) pull their chunks from, so that a batch is divided by how fast
// each GPU's host link turns out to be (csic_multi_process_host) instead of evenly.
struct ChunkShare {
  std::atomic<size_t> next{0};
  size_t gpus = 1;
};

static int host_pipeline_run(csic_ctx* ctx, const csic_params* p, const uint8_t* rgb, size_t n_frames, uint8_t* out,
                             int32_t row0, int32_t rows, ChunkShare* share) {
  DeviceGuard guard(ctx->device);
  csic::HostPlan h;
  int rc = csic::plan_host(*p, row0, rows, n_frames, ctx->dev, ctx->opt, ctx->opt_chunk_bytes, ctx->opt_no_compact,
                           share ? share->gpus : 0, h);
  if (rc != CSIC_OK) return rc;
  const size_t per = h.frames_per_chunk;
  auto dev_alloc = [](void** b, size_t n) { return cudaMalloc(b, n); };
  rc = grow_ring(ctx->d_in, per * h.in.staging.frame, dev_alloc, cudaFree);
  if (rc == CSIC_OK) rc = grow_ring(ctx->d_out, per * h.out.staging.frame, dev_alloc, cudaFree);
  if (rc != CSIC_OK) return rc;

  // The chunks this context processes, in order: consecutive ones when it owns the whole batch, otherwise whatever
  // it pulls from the shared cursor (all contexts use the same `per`: same parameters, same chunk-size option).
  std::vector<std::pair<size_t, size_t>> mine;   // (first frame, frames)
  mine.reserve((n_frames + per - 1) / per + 1);  // never reallocates: the drain thread reads entries while this one appends
  auto next_chunk = [&]() -> bool {
    const size_t f0 = share ? share->next.fetch_add(per, std::memory_order_relaxed) : mine.size() * per;
    if (f0 >= n_frames) return false;
    mine.emplace_back(f0, std::min(per, n_frames - f0));
    return true;
  };
  const size_t n_chunks = share ? (size_t)-1 : (n_frames + per - 1) / per;
  // Pageable caller buffers (a JVM heap, malloc): cudaMemcpyAsync would fall back to the driver's synchronous,
  // single-threaded staging (measured 5 k MP/s vs 31 k MP/s pinned on cfg4).  Gather the needed rows into pinned
  // bounce buffers on several host threads instead, overlapped with the DMA of the neighbouring chunks.
  const bool bounce =
      !ctx->opt_no_bounce && n_frames * h.in.staging.frame >= (8u << 20) && (is_pageable(rgb) || is_pageable(out));
  if (bounce) {
    auto pinned = [](void** b, size_t n) { return cudaHostAlloc(b, n, cudaHostAllocDefault); };
    rc = grow_ring(ctx->h_in, per * h.in.bounce.frame, pinned, cudaFreeHost);
    if (rc == CSIC_OK) rc = grow_ring(ctx->h_out, per * h.out.bounce.frame, pinned, cudaFreeHost);
    if (rc != CSIC_OK) return rc;
  }
  // scatters chunk j's result from its bounce buffer to the caller once its D2H has landed
  auto drain = [&](size_t j) -> int {
    const int bj = (int)(j % kPipe);
    CSIC_CUDA(cudaEventSynchronize(ctx->ev_d2h[bj]));
    for (const csic::Copy& x : csic::frame_copies(h.out, h.out.caller.at(mine[j].first), h.out.bounce, mine[j].second))
      host_copy(out, static_cast<const uint8_t*>(ctx->h_out.buf[bj]), x);
    return CSIC_OK;
  };
  // The scatter of chunk j runs on its own host thread, so that it overlaps the gather of chunk j + kPipe - 1 on this
  // one (each side fans out over host_copy's workers).  Joined before its bounce buffer is refilled.
  struct AsyncDrain {
    std::thread th;
    int rc = CSIC_OK;
    std::string err;
    int join() {
      if (th.joinable()) th.join();
      if (rc != CSIC_OK) g_last_error = err;
      const int r = rc;
      rc = CSIC_OK;
      return r;
    }
    ~AsyncDrain() { if (th.joinable()) th.join(); }
  } adrain;
  const int device = ctx->device;
  auto start_drain = [&](size_t j) {
    adrain.th = std::thread([&adrain, &drain, device, j] {
      cudaSetDevice(device);
      adrain.rc = guarded("csic_process_host drain", [&] { return drain(j); });
      if (adrain.rc != CSIC_OK) adrain.err = g_last_error;
    });
  };
  // One chunk (small batches, single images): nothing to overlap, so issue copy-in, kernel and copy-out on ONE
  // stream and synchronise once -- no cross-stream events on the latency path.
  const bool single = n_chunks == 1 && !bounce;
  cudaStream_t s_in = single ? ctx->stream : ctx->s_h2d, s_out = single ? ctx->stream : ctx->s_d2h;
  for (size_t c = 0; next_chunk(); ++c) {
    const int b = (int)(c % kPipe);
    const size_t f0 = mine[c].first, nf = mine[c].second;
    if (c >= (size_t)kPipe) {
      // buffer reuse: the kernel that read d_in[b] and the copy that drained d_out[b] must be done
      CSIC_CUDA(cudaStreamWaitEvent(ctx->s_h2d, ctx->ev_k[b], 0));
      CSIC_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_d2h[b], 0));
    }
    uint8_t* d_in = static_cast<uint8_t*>(ctx->d_in.buf[b]);
    uint8_t* d_out = static_cast<uint8_t*>(ctx->d_out.buf[b]);
    if (bounce) {
      if (c >= (size_t)kPipe) CSIC_CUDA(cudaEventSynchronize(ctx->ev_h2d[b]));   // bounce_in[b] has been shipped
      uint8_t* hb = static_cast<uint8_t*>(ctx->h_in.buf[b]);
      for (const csic::Copy& x : csic::frame_copies(h.in, h.in.bounce, h.in.caller.at(f0), nf)) host_copy(hb, rgb, x);
      rc = device_copies(d_in, hb, csic::frame_copies(h.in, h.in.staging, h.in.bounce, nf), cudaMemcpyHostToDevice, s_in);
    } else {
      rc = device_copies(d_in, rgb, csic::frame_copies(h.in, h.in.staging, h.in.caller.at(f0), nf),
                         cudaMemcpyHostToDevice, s_in);
    }
    if (rc != CSIC_OK) return rc;
    ctx->h2d_bytes += nf * h.in.rows * h.in.width;
    if (!single) {
      CSIC_CUDA(cudaEventRecord(ctx->ev_h2d[b], s_in));
      CSIC_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_h2d[b], 0));
    }
    // virtual frame bases: row r of the frame sits at base + r * pitch; only the band's rows are ever touched
    rc = run(ctx, p, d_in - h.first_stored * h.in_pitch, nf, d_out - (size_t)row0 * h.out_pitch, row0, rows, ctx->stream,
             h.compact, h.lay);
    if (rc != CSIC_OK) return rc;
    if (!single) {
      CSIC_CUDA(cudaEventRecord(ctx->ev_k[b], ctx->stream));
      CSIC_CUDA(cudaStreamWaitEvent(s_out, ctx->ev_k[b], 0));
    }
    if (bounce) {
      rc = adrain.join();                  // chunk c - kPipe has left h_out[b]
      if (rc == CSIC_OK)
        rc = device_copies(static_cast<uint8_t*>(ctx->h_out.buf[b]), d_out,
                           csic::frame_copies(h.out, h.out.bounce, h.out.staging, nf), cudaMemcpyDeviceToHost, s_out);
    } else {
      rc = device_copies(out, d_out, csic::frame_copies(h.out, h.out.caller.at(f0), h.out.staging, nf),
                         cudaMemcpyDeviceToHost, s_out);
    }
    if (rc != CSIC_OK) return rc;
    if (!single) CSIC_CUDA(cudaEventRecord(ctx->ev_d2h[b], s_out));
    if (bounce && c + 1 >= (size_t)kPipe) start_drain(c + 1 - (size_t)kPipe);   // the chunk issued kPipe-1 iterations ago
  }
  if (bounce) {
    rc = adrain.join();
    if (rc != CSIC_OK) return rc;
    const size_t n_mine = mine.size();
    for (size_t j = n_mine >= (size_t)kPipe ? n_mine - ((size_t)kPipe - 1) : 0; j < n_mine; ++j) {
      rc = drain(j);
      if (rc != CSIC_OK) return rc;
    }
  }
  if (single) {
    CSIC_CUDA(cudaStreamSynchronize(ctx->stream));
    return CSIC_OK;
  }
  CSIC_CUDA(cudaStreamSynchronize(ctx->s_d2h));
  CSIC_CUDA(cudaStreamSynchronize(ctx->stream));
  CSIC_CUDA(cudaStreamSynchronize(ctx->s_h2d));
  return CSIC_OK;
}

// An error in the middle of the pipeline must not leave copies in flight on the caller's buffers or on the staging
// ring: drain the three streams before reporting it.
static int host_pipeline(csic_ctx* ctx, const csic_params* p, const uint8_t* rgb, size_t n_frames, uint8_t* out,
                         int32_t row0, int32_t rows, ChunkShare* share = nullptr) {
  const int rc = host_pipeline_run(ctx, p, rgb, n_frames, out, row0, rows, share);
  if (rc != CSIC_OK) {
    const std::string keep = g_last_error;
    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->s_h2d);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->s_d2h);
    cudaGetLastError();
    g_last_error = keep;
  }
  return rc;
}

int csic_process_host(csic_ctx* ctx, const csic_params* p, const uint8_t* rgb, size_t n_frames, uint8_t* out) {
  if (!ctx || !p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  if (n_frames == 0) return CSIC_OK;
  if (!rgb || !out) return CSIC_EINVAL_ARG;
  return guarded("csic_process_host", [&] { return host_pipeline(ctx, p, rgb, n_frames, out, 0, csic::geometry(*p).out_h); });
}

int csic_process_host_band(csic_ctx* ctx, const csic_params* p, const uint8_t* rgb, size_t n_frames, uint8_t* out,
                           int32_t out_row0, int32_t out_rows) {
  if (!ctx || !p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  if (n_frames == 0 || out_rows == 0) return CSIC_OK;
  if (!rgb || !out) return CSIC_EINVAL_ARG;
  if (out_row0 < 0 || out_rows < 0 || out_row0 + out_rows > csic::geometry(*p).out_h) return CSIC_EINVAL_ARG;
  return guarded("csic_process_host_band", [&] { return host_pipeline(ctx, p, rgb, n_frames, out, out_row0, out_rows); });
}

// ---- one process, several GPUs ------------------------------------------------------------------
// The reference's host is one JVM process.  csic_multi owns one context per GPU and one host thread per
// context; a batch is split by frames (E1) -- or, when there are fewer frames than GPUs, every frame is cut into
// aligned row bands (E2).  No data moves between GPUs.
struct csic_multi {
  std::vector<csic_ctx*> ctx;
  bool static_split = false;
};

int csic_multi_create(const int* devices, int n_devices, csic_multi** out) {
  if (!out) return CSIC_EINVAL_ARG;
  *out = nullptr;
  const int avail = csic_device_count();
  if (avail <= 0) return CSIC_ENODEVICE;
  if (n_devices <= 0) { n_devices = avail; devices = nullptr; }
  csic_multi* m = new (std::nothrow) csic_multi();
  if (!m) return CSIC_ENOMEM;
  for (int i = 0; i < n_devices; ++i) {
    csic_ctx* c = nullptr;
    int rc = csic_create(devices ? devices[i] : i, &c);
    if (rc != CSIC_OK) {
      for (csic_ctx* x : m->ctx) csic_destroy(x);
      delete m;
      return rc;
    }
    m->ctx.push_back(c);
  }
  *out = m;
  return CSIC_OK;
}

int csic_multi_destroy(csic_multi* m) {
  if (!m) return CSIC_OK;
  for (csic_ctx* c : m->ctx) csic_destroy(c);
  delete m;
  return CSIC_OK;
}

int csic_multi_size(const csic_multi* m) { return m ? (int)m->ctx.size() : CSIC_EINVAL_ARG; }

int csic_multi_set_option(csic_multi* m, int option, int64_t value) {
  if (!m) return CSIC_EINVAL_ARG;
  if (option == CSIC_OPT_MULTI_STATIC_SPLIT) {
    m->static_split = value != 0;
    return CSIC_OK;
  }
  for (csic_ctx* c : m->ctx) {
    const int rc = csic_set_option(c, option, value);
    if (rc != CSIC_OK) return rc;
  }
  return CSIC_OK;
}

int csic_multi_host_bytes(const csic_multi* m, uint64_t* h2d_per_device, int n) {
  if (!m || !h2d_per_device || n < (int)m->ctx.size()) return CSIC_EINVAL_ARG;
  for (size_t i = 0; i < m->ctx.size(); ++i) h2d_per_device[i] = m->ctx[i]->h2d_bytes;
  return CSIC_OK;
}

static int multi_process_host_impl(csic_multi* m, const csic_params* p, const uint8_t* rgb, size_t n_frames, uint8_t* out) {
  if (!m || !p) return CSIC_EINVAL_ARG;
  int rc = csic_validate(p, nullptr, 0);
  if (rc != CSIC_OK) return rc;
  if (n_frames == 0) return CSIC_OK;
  if (!rgb || !out) return CSIC_EINVAL_ARG;
  const csic::Geometry g = csic::geometry(*p);
  const size_t G = m->ctx.size();
  std::vector<int> rcs(G, CSIC_OK);
  std::vector<std::string> errs(G);
  struct Joiner {   // an exception while spawning must not leave joinable threads behind (std::terminate)
    std::vector<std::thread> v;
    ~Joiner() { for (std::thread& t : v) if (t.joinable()) t.join(); }
  } joiner;
  std::vector<std::thread>& th = joiner.v;
  ChunkShare share;
  share.gpus = G;
  if (n_frames >= G || p->out_format == CSIC_OUT_PLANAR) {
    // Frames are independent: every GPU's pipeline pulls its next chunk of frames from one shared cursor, so the batch
    // divides itself by what each GPU's host link delivers (on the 8-GPU boxes of this pool four of the links are
    // 1.4x slower than the other four when all run at once: profiles/r2/pcie_ceiling.json) instead of evenly.
    const int32_t out_h = g.out_h;
    for (size_t i = 0; i < G; ++i) {
      const size_t lo = n_frames * i / G, hi = n_frames * (i + 1) / G;
      if (m->static_split && hi == lo) continue;
      th.emplace_back([=, &rcs, &errs, &share] {
        cudaSetDevice(m->ctx[i]->device);   // this thread's device from the start: no context is made on device 0
        rcs[i] = guarded("csic_multi_process_host worker", [&] {
          return m->static_split   // the even split of round 1, kept for comparison (CSIC_OPT_MULTI_STATIC_SPLIT)
                     ? host_pipeline(m->ctx[i], p, rgb + lo * g.in_frame_bytes, hi - lo, out + lo * g.out_frame_bytes, 0, out_h)
                     : host_pipeline(m->ctx[i], p, rgb, n_frames, out, 0, out_h, &share);
        });
        if (rcs[i] != CSIC_OK) errs[i] = g_last_error;
      });
    }
  } else {
    // fewer frames than GPUs: aligned row bands of every frame (zero halo; SURVEY.md section 8(e) E2)
    for (size_t i = 0; i < G; ++i) {
      int32_t r0, r1;
      csic::band_split(*p, i, G, r0, r1);
      if (r1 <= r0) continue;
      th.emplace_back([=, &rcs, &errs] {
        cudaSetDevice(m->ctx[i]->device);
        rcs[i] = csic_process_host_band(m->ctx[i], p, rgb, n_frames, out, r0, r1 - r0);   // guarded inside
        if (rcs[i] != CSIC_OK) errs[i] = g_last_error;
      });
    }
  }
  for (std::thread& t : th) t.join();
  for (size_t i = 0; i < G; ++i)
    if (rcs[i] != CSIC_OK) {
      g_last_error = errs[i];
      return rcs[i];
    }
  return CSIC_OK;
}

int csic_multi_process_host(csic_multi* m, const csic_params* p, const uint8_t* rgb, size_t n_frames, uint8_t* out) {
  return guarded("csic_multi_process_host", [&] { return multi_process_host_impl(m, p, rgb, n_frames, out); });
}

int csic_host_alloc(size_t bytes, void** out) {
  if (!out) return CSIC_EINVAL_ARG;
  *out = nullptr;
  if (csic_device_count() <= 0) return CSIC_ENODEVICE;
  CSIC_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
  return CSIC_OK;
}

int csic_host_free(void* p) {
  if (!p) return CSIC_OK;
  CSIC_CUDA(cudaFreeHost(p));
  return CSIC_OK;
}

int csic_synchronize(csic_ctx* ctx) {
  if (!ctx) return CSIC_EINVAL_ARG;
  DeviceGuard guard(ctx->device);
  CSIC_CUDA(cudaStreamSynchronize(ctx->stream));
  return CSIC_OK;
}

int csic_host_bytes(const csic_ctx* ctx, uint64_t* h2d_total) {
  if (!ctx) return CSIC_EINVAL_ARG;
  if (h2d_total) *h2d_total = ctx->h2d_bytes;
  return CSIC_OK;
}

int csic_last_kernel(const csic_ctx* ctx, int32_t* family, int64_t* launches_total) {
  if (!ctx) return CSIC_EINVAL_ARG;
  if (family) *family = ctx->last_family;
  if (launches_total) *launches_total = ctx->launches;
  return CSIC_OK;
}

}  // extern "C"
