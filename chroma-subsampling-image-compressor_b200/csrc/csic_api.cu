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

constexpr int kPipe = 3;   // chunks in flight in csic_process_host
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
  void* d_in[kPipe] = {nullptr, nullptr, nullptr};
  void* d_out[kPipe] = {nullptr, nullptr, nullptr};
  size_t d_in_cap = 0, d_out_cap = 0;
  cudaEvent_t ev_h2d[kPipe] = {}, ev_k[kPipe] = {}, ev_d2h[kPipe] = {};
  void* h_in[kPipe] = {nullptr, nullptr, nullptr};    // pinned bounce buffers for pageable callers
  void* h_out[kPipe] = {nullptr, nullptr, nullptr};
  size_t h_in_cap = 0, h_out_cap = 0;
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

// True when a DECIMATE pipeline reads only every f-th input row and those rows sit at a uniform pitch
// across the frames of a batch: then csic_process_host ships just those rows over PCIe.
bool can_compact(const csic_params& p) {
  return p.pool_mode == CSIC_POOL_DECIMATE && p.factor > 1 && p.height % p.factor == 0;
}

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
  int err;
  switch (c.family) {
    case csic::FAM_ROWS: err = csic::launch_rows(c.k, c.grid, st); break;
    case csic::FAM_POOL: err = csic::launch_pool(c.k, c.grid, st); break;
    case csic::FAM_FLEX: err = csic::launch_flex(c.k, c.grid, st); break;
    default: err = csic::launch_generic(c.k, c.grid, st); break;
  }
  ctx->last_family = c.family;
  ctx->launches += 1;
  if (err != (int)cudaSuccess) return cuda_fail((cudaError_t)err, "kernel launch");
  return CSIC_OK;
}

int ensure_staging(csic_ctx* ctx, size_t in_bytes, size_t out_bytes) {
  if (in_bytes > ctx->d_in_cap) {
    for (int i = 0; i < kPipe; ++i) {
      if (ctx->d_in[i]) cudaFree(ctx->d_in[i]);
      ctx->d_in[i] = nullptr;
    }
    ctx->d_in_cap = 0;
    for (int i = 0; i < kPipe; ++i) CSIC_CUDA(cudaMalloc(&ctx->d_in[i], in_bytes));
    ctx->d_in_cap = in_bytes;
  }
  if (out_bytes > ctx->d_out_cap) {
    for (int i = 0; i < kPipe; ++i) {
      if (ctx->d_out[i]) cudaFree(ctx->d_out[i]);
      ctx->d_out[i] = nullptr;
    }
    ctx->d_out_cap = 0;
    for (int i = 0; i < kPipe; ++i) CSIC_CUDA(cudaMalloc(&ctx->d_out[i], out_bytes));
    ctx->d_out_cap = out_bytes;
  }
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
  if (err == cudaSuccess) step((cudaError_t)csic::rows_kernel_set_attributes(c->dev.max_smem_optin));
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
    if (ctx->d_in[i]) cudaFree(ctx->d_in[i]);
    if (ctx->d_out[i]) cudaFree(ctx->d_out[i]);
    if (ctx->h_in[i]) cudaFreeHost(ctx->h_in[i]);
    if (ctx->h_out[i]) cudaFreeHost(ctx->h_out[i]);
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
  csic::Layout lay;
  lay.in_pitch = in_pitch_bytes;
  lay.in_frame = in_frame_stride;
  lay.out_pitch = out_pitch_bytes;
  lay.out_frame = out_frame_stride;
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

namespace {

bool is_pageable(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

int ensure_bounce(csic_ctx* ctx, size_t in_bytes, size_t out_bytes) {
  if (in_bytes > ctx->h_in_cap) {
    for (int i = 0; i < kPipe; ++i) {
      if (ctx->h_in[i]) cudaFreeHost(ctx->h_in[i]);
      ctx->h_in[i] = nullptr;
    }
    ctx->h_in_cap = 0;
    for (int i = 0; i < kPipe; ++i) CSIC_CUDA(cudaHostAlloc(&ctx->h_in[i], in_bytes, cudaHostAllocDefault));
    ctx->h_in_cap = in_bytes;
  }
  if (out_bytes > ctx->h_out_cap) {
    for (int i = 0; i < kPipe; ++i) {
      if (ctx->h_out[i]) cudaFreeHost(ctx->h_out[i]);
      ctx->h_out[i] = nullptr;
    }
    ctx->h_out_cap = 0;
    for (int i = 0; i < kPipe; ++i) CSIC_CUDA(cudaHostAlloc(&ctx->h_out[i], out_bytes, cudaHostAllocDefault));
    ctx->h_out_cap = out_bytes;
  }
  return CSIC_OK;
}

// Copies `n_rows` rows of `row_bytes` from src (row stride src_step) to dst (row stride dst_step) on several
// host threads: a pageable caller's rows are gathered into / scattered from the pinned bounce buffers at host
// memory speed instead of the driver's single-threaded staging.
void parallel_rows_copy(uint8_t* dst, size_t dst_step, const uint8_t* src, size_t src_step, size_t row_bytes, size_t n_rows) {
  const size_t total = row_bytes * n_rows;
  unsigned T = std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency() / 2));
  if (total < (4u << 20)) T = 1;
  const bool contiguous = dst_step == row_bytes && src_step == row_bytes;
  // contiguous ranges are cut by bytes (a "row" may be a whole frame), strided ones by rows
  const size_t units = contiguous ? total : n_rows;
  auto work = [=](size_t u0, size_t u1) {
    if (contiguous) {
      std::memcpy(dst + u0, src + u0, u1 - u0);
    } else {
      for (size_t r = u0; r < u1; ++r) std::memcpy(dst + r * dst_step, src + r * src_step, row_bytes);
    }
  };
  if (T == 1) { work(0, units); return; }
  std::vector<std::thread> th;
  for (unsigned t = 1; t < T; ++t) th.emplace_back(work, units * t / T, units * (t + 1) / T);
  work(0, units / T);
  for (std::thread& x : th) x.join();
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
  const csic::Geometry g = csic::geometry(*p);
  DeviceGuard guard(ctx->device);
  const bool band = !(row0 == 0 && rows == g.out_h);

  // DECIMATE with f > 1 reads only every f-th row: ship only those (a strided 2-D copy), 1/f of the H2D bytes.
  const bool compact = can_compact(*p) && !ctx->opt_no_compact;
  int32_t in_row0 = 0, in_rows = p->height;
  if (band) {
    int rc = csic_band_input_rows(p, row0, rows, &in_row0, &in_rows);
    if (rc != CSIC_OK) return rc;
  }
  // rows kept on the device, in stored-row units (a stored row is an input row, or every f-th one when compact)
  const size_t first_stored = compact ? (size_t)(in_row0 / p->factor) : (size_t)in_row0;
  const size_t rows_stored = compact ? (size_t)(row0 + rows) - first_stored : (size_t)in_rows;

  // Staging layout.  Dense when the dense layout already satisfies a TMA kernel's 16-byte rules; otherwise the
  // rows are re-pitched on the way in and out (the copies are 2-D anyway), so odd widths also avoid the
  // generic kernel.
  auto eligible = [&](const csic::Layout& l) {
    csic::KPlan probe;
    if (csic::build_plan(*p, reinterpret_cast<const void*>(uintptr_t(4096)), reinterpret_cast<void*>(uintptr_t(4096)), 1, 0,
                         g.out_h, compact, l, probe) != CSIC_OK)
      return false;
    const int family = csic::select_kernel(probe, ctx->dev, ctx->opt).family;
    return family == csic::FAM_ROWS || family == csic::FAM_POOL;
  };
  csic::Layout lay;
  if (!eligible(csic::Layout()) && p->out_format != CSIC_OUT_PLANAR) {
    const size_t wp = ((size_t)g.out_w + 15) & ~(size_t)15;
    csic::Layout cand;
    cand.in_pitch = (std::max(g.in_row_bytes, wp * (size_t)p->factor * (size_t)g.in_px_bytes) + 15) & ~(size_t)15;
    cand.out_pitch = (std::max(g.out_row_bytes, wp * (size_t)g.out_px_bytes) + 15) & ~(size_t)15;
    if (eligible(cand)) lay = cand;
  }
  const size_t in_pitch = lay.in_pitch ? lay.in_pitch : g.in_row_bytes;
  const size_t out_pitch = lay.out_pitch ? lay.out_pitch : g.out_row_bytes;
  const size_t dev_frame_bytes = in_pitch * rows_stored;
  if (band && p->out_format == CSIC_OUT_PLANAR) return CSIC_EINVAL_MODE;   // planes are not row bands
  const size_t dev_out_frame_bytes = band ? out_pitch * (size_t)rows : std::max(out_pitch * (size_t)rows, g.out_frame_bytes);
  const size_t host_row_step = g.in_row_bytes * (size_t)(compact ? p->factor : 1);
  if (band) {   // the device holds only the band's rows: frames are dev_*_frame_bytes apart
    lay.in_pitch = in_pitch;
    lay.out_pitch = out_pitch;
    lay.in_frame = dev_frame_bytes;
    lay.out_frame = dev_out_frame_bytes;
    lay.short_frames = true;
  }
  // Frames per chunk: ~opt_chunk_bytes of input, at least one frame, at most what is there.
  size_t per = std::max<size_t>(1, ctx->opt_chunk_bytes / std::max<size_t>(1, dev_frame_bytes));
  per = std::min(per, n_frames);
  if (share) per = std::min(per, std::max<size_t>(1, n_frames / (share->gpus * (size_t)kPipe)));   // several chunks per GPU
  int rc = ensure_staging(ctx, per * dev_frame_bytes, per * dev_out_frame_bytes);
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
  const bool bounce = !ctx->opt_no_bounce && n_frames * dev_frame_bytes >= (8u << 20) && (is_pageable(rgb) || is_pageable(out));
  const size_t bounce_in_frame = g.in_row_bytes * rows_stored, bounce_out_frame = band ? g.out_row_bytes * (size_t)rows : g.out_frame_bytes;
  if (bounce) {
    rc = ensure_bounce(ctx, per * bounce_in_frame, per * bounce_out_frame);
    if (rc != CSIC_OK) return rc;
  }
  // scatters chunk j's result from its bounce buffer to the caller once its D2H has landed
  auto drain = [&](size_t j) -> int {
    const int bj = (int)(j % kPipe);
    const size_t jf0 = mine[j].first, jnf = mine[j].second;
    CSIC_CUDA(cudaEventSynchronize(ctx->ev_d2h[bj]));
    const uint8_t* hb = static_cast<const uint8_t*>(ctx->h_out[bj]);
    if (band) {
      for (size_t k = 0; k < jnf; ++k)
        parallel_rows_copy(out + (jf0 + k) * g.out_frame_bytes + (size_t)row0 * g.out_row_bytes, g.out_row_bytes,
                           hb + k * bounce_out_frame, g.out_row_bytes, g.out_row_bytes, (size_t)rows);
    } else {
      parallel_rows_copy(out + jf0 * g.out_frame_bytes, bounce_out_frame, hb, bounce_out_frame, bounce_out_frame, jnf);
    }
    return CSIC_OK;
  };
  // The scatter of chunk j runs on its own host thread, so that it overlaps the gather of chunk j + kPipe - 1 on this
  // one (each side fans out over parallel_rows_copy's workers).  Joined before its bounce buffer is refilled.
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
    uint8_t* d_in = static_cast<uint8_t*>(ctx->d_in[b]);
    uint8_t* d_out = static_cast<uint8_t*>(ctx->d_out[b]);
    if (bounce) {
      if (c >= (size_t)kPipe) CSIC_CUDA(cudaEventSynchronize(ctx->ev_h2d[b]));   // bounce_in[b] has been shipped
      uint8_t* hb = static_cast<uint8_t*>(ctx->h_in[b]);
      if (!band) {                          // only the rows that are read, densely; uniform stride across frames
        parallel_rows_copy(hb, g.in_row_bytes, rgb + f0 * g.in_frame_bytes, host_row_step, g.in_row_bytes, nf * rows_stored);
      } else {
        for (size_t k = 0; k < nf; ++k)
          parallel_rows_copy(hb + k * bounce_in_frame, g.in_row_bytes,
                             rgb + (f0 + k) * g.in_frame_bytes + first_stored * host_row_step, host_row_step,
                             g.in_row_bytes, rows_stored);
      }
      if (in_pitch != g.in_row_bytes) {
        CSIC_CUDA(cudaMemcpy2DAsync(d_in, in_pitch, hb, g.in_row_bytes, g.in_row_bytes, nf * rows_stored,
                                    cudaMemcpyHostToDevice, s_in));
      } else {
        CSIC_CUDA(cudaMemcpyAsync(d_in, hb, nf * bounce_in_frame, cudaMemcpyHostToDevice, s_in));
      }
    } else if (band) {
      // one strided copy per frame: rows [first_stored, first_stored + rows_stored) of that frame
      for (size_t k = 0; k < nf; ++k)
        CSIC_CUDA(cudaMemcpy2DAsync(d_in + k * dev_frame_bytes, in_pitch,
                                    rgb + (f0 + k) * g.in_frame_bytes + first_stored * host_row_step, host_row_step,
                                    g.in_row_bytes, rows_stored, cudaMemcpyHostToDevice, s_in));
    } else if (compact || lay.in_pitch) {
      CSIC_CUDA(cudaMemcpy2DAsync(d_in, in_pitch, rgb + f0 * g.in_frame_bytes, host_row_step, g.in_row_bytes,
                                  nf * rows_stored, cudaMemcpyHostToDevice, s_in));
    } else {
      CSIC_CUDA(cudaMemcpyAsync(d_in, rgb + f0 * g.in_frame_bytes, nf * g.in_frame_bytes, cudaMemcpyHostToDevice,
                                s_in));
    }
    ctx->h2d_bytes += nf * rows_stored * g.in_row_bytes;
    if (!single) {
      CSIC_CUDA(cudaEventRecord(ctx->ev_h2d[b], s_in));
      CSIC_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_h2d[b], 0));
    }
    // virtual frame bases: row r of the frame sits at base + r * pitch; only the band's rows are ever touched
    rc = run(ctx, p, d_in - first_stored * in_pitch, nf, d_out - (size_t)row0 * out_pitch, row0, rows, ctx->stream,
             compact, lay);
    if (rc != CSIC_OK) return rc;
    if (!single) {
      CSIC_CUDA(cudaEventRecord(ctx->ev_k[b], ctx->stream));
      CSIC_CUDA(cudaStreamWaitEvent(s_out, ctx->ev_k[b], 0));
    }
    if (bounce) {
      rc = adrain.join();                  // chunk c - kPipe has left h_out[b]
      if (rc != CSIC_OK) return rc;
      uint8_t* hb = static_cast<uint8_t*>(ctx->h_out[b]);
      if (band || lay.out_pitch) {
        CSIC_CUDA(cudaMemcpy2DAsync(hb, g.out_row_bytes, d_out, out_pitch, g.out_row_bytes, nf * (size_t)rows,
                                    cudaMemcpyDeviceToHost, s_out));
      } else {
        CSIC_CUDA(cudaMemcpyAsync(hb, d_out, nf * g.out_frame_bytes, cudaMemcpyDeviceToHost, s_out));
      }
    } else if (band) {
      for (size_t k = 0; k < nf; ++k)
        CSIC_CUDA(cudaMemcpy2DAsync(out + (f0 + k) * g.out_frame_bytes + (size_t)row0 * g.out_row_bytes, g.out_row_bytes,
                                    d_out + k * dev_out_frame_bytes, out_pitch, g.out_row_bytes, (size_t)rows,
                                    cudaMemcpyDeviceToHost, s_out));
    } else if (lay.out_pitch) {
      CSIC_CUDA(cudaMemcpy2DAsync(out + f0 * g.out_frame_bytes, g.out_row_bytes, d_out, out_pitch, g.out_row_bytes,
                                  nf * (size_t)g.out_h, cudaMemcpyDeviceToHost, s_out));
    } else {
      CSIC_CUDA(cudaMemcpyAsync(out + f0 * g.out_frame_bytes, d_out, nf * g.out_frame_bytes, cudaMemcpyDeviceToHost,
                                s_out));
    }
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
    const bool case_b = !g.chroma_first && p->factor > 1;
    const int unit = case_b ? p->factor * g.vf : std::max(1, (p->factor % g.vf == 0 ? p->factor : p->factor * g.vf) / p->factor);
    const int units = (g.out_h + unit - 1) / unit;
    for (size_t i = 0; i < G; ++i) {
      const int r0 = std::min(g.out_h, (int)(units * i / G) * unit), r1 = std::min(g.out_h, (int)(units * (i + 1) / G) * unit);
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
