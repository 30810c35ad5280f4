/*
 * csic.h -- C ABI of the B200-native pixel pipeline (libcsic.so).
 *
 * Drop-in boundary for the hot path of Andurdur/Chroma-Subsampling-Image-Compressor:
 *   RGB2YCbCr -> {ChromaSubsampler, SpatialDownsampler, ColorQuantizer in any order} -> pack / YCbCr2RGB.
 * The reference has no FFI of its own; its seam is the Scala constructor surface of
 * `ImageCompressorTop` / `ImageProcessorParams` plus a raster pixel stream.  Every entry point below
 * names the reference interface it replaces (paths relative to the reference root).
 * INTEGRATION.md shows the Scala (Panama / JNI) binding a maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++ / torch types cross this boundary;
 *   - the caller owns every buffer; the library never allocates an output;
 *   - every function returns CSIC_OK (0) or a negative csic_status; the reference signals the same
 *     conditions with Scala `require` -> IllegalArgumentException at construction time;
 *   - there is NO CPU fallback: without a usable CUDA device the process/create calls return
 *     CSIC_ENODEVICE.  (The CPU oracle lives in oracle/ and is test infrastructure only.)
 */
#ifndef CSIC_H_
#define CSIC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSIC_ABI_VERSION 1

#if defined(__GNUC__)
#define CSIC_API __attribute__((visibility("default")))
#else
#define CSIC_API
#endif

/* ProcessingStep ids -- src/main/scala/jpeg/ImageCompressorTop.scala:7-9 (ChiselEnum declaration order). */
enum csic_step {
  CSIC_STEP_NOOP = 0,              /* exists in the enum, rejected by the top (:27-31) */
  CSIC_STEP_SPATIAL = 1,           /* SpatialSampling   */
  CSIC_STEP_COLOR = 2,             /* ColorQuantization */
  CSIC_STEP_CHROMA = 3             /* ChromaSubsampling */
};

/* Forward-transform rounding.  FLOOR = RTL `>> 8` (src/main/scala/jpeg/RGB2YCbCr.scala:50-52,
 * ReferenceModel.scala:15-17) -- what ImageCompressorTop / ImageProcessor compute.
 * TRUNC = Scala `/ 256` of YCbCrUtils.rgbToYCbCr (RGB2YCbCr.scala:111-118) used by the stage benches. */
enum csic_round_mode { CSIC_ROUND_FLOOR = 0, CSIC_ROUND_TRUNC = 1 };

/* SpatialDownsampler behaviour.  DECIMATE = the reference (SpatialDownsampler.scala:33-55: forward the
 * pixel at row%f==0 && col%f==0 unchanged).  AVERAGE = documented extension (README.md:44 prose only;
 * "parity unpinned"): mean of the f x f block, round half up; requires W%f==0 && H%f==0. */
enum csic_pool_mode { CSIC_POOL_DECIMATE = 0, CSIC_POOL_AVERAGE = 1 };

/* Output wire format.
 *  YCC888    3 bytes/pixel Y,Cb,Cr            = PixelYCbCrBundle fields (PixelBundle.scala:11-15); parity layout.
 *  RGB888    3 bytes/pixel R,G,B after YCbCrUtils.ycbcr2rgb (RGB2YCbCr.scala:123-132) fused as last stage
 *            (replaces the host call at src/test/scala/jpeg/ImageCompressorTopApp.scala:118).
 *  BUNDLE64 / BUNDLE128   build-defined packed words (the reference has no multi-pixel packing):
 *            slot = 8/16/32 bits for y_bits+cb_bits+cr_bits <= 8 / <= 16 / <= 24; pixel k of a row sits in
 *            bits [k*slot,(k+1)*slot) of a little-endian 64/128-bit word stream; inside a slot
 *            value = (Y>>sy) << (cb_bits+cr_bits) | (Cb>>scb) << cr_bits | (Cr>>scr), zero padded above;
 *            each output row is padded with zero slots to a whole word.
 *  PLANAR    build-defined (SURVEY.md 8(f) N3): what a downstream JPEG / video encoder wants.  Per frame three
 *            planes back to back: Y [out_h x out_w], Cb [ch x cw], Cr [ch x cw], one byte per sample, quantised.
 *            The chroma planes hold ONLY the sample points that survive: cw = ceil(out_w / hs), ch = ceil(out_h / vs),
 *            hs = max(1, (4/a)/f), vs = max(1, vf/f); Cb[rc][cc] is the chroma of output pixel (rc*vs, cc*hs).
 *            The reference replays held chroma at full rate (3 bytes/pixel); 4:2:0 at f=1 is 1.5 bytes/pixel here.
 *            csic_expand_planar_* re-applies the reference's replay rule and returns the YCC888 / RGB888 stream.
 *            Needs ChromaSubsampling before SpatialSampling (or f == 1) and DECIMATE. */
enum csic_out_format { CSIC_OUT_YCC888 = 0, CSIC_OUT_RGB888 = 1, CSIC_OUT_BUNDLE64 = 2, CSIC_OUT_BUNDLE128 = 3,
                       CSIC_OUT_PLANAR = 4 };

/* Input pixel layout.  RGB24 = 3 bytes R,G,B (pixel.red/green/blue, ImageCompressorTopApp.scala:86-89).
 * RGBA32 / BGRA32 = 4 bytes per pixel with the fourth ignored, exactly as the reference ignores alpha;
 * BGRA32 is the in-memory layout of a little-endian Java / AWT / scrimage ARGB int (0xAARRGGBB), so a JVM host
 * can pass its pixel array without repacking (SURVEY.md section 8(f) N1). */
enum csic_in_format { CSIC_IN_RGB24 = 0, CSIC_IN_RGBA32 = 1, CSIC_IN_BGRA32 = 2 };

/* Legacy enums (removed from the reference's HEAD, recovered from its committed outputs; SURVEY.md F4). */
enum csic_chroma_mode { CSIC_CHROMA_444 = 0, CSIC_CHROMA_422 = 1, CSIC_CHROMA_420 = 2 };
enum csic_quant_mode { CSIC_Q_24BIT = 0, CSIC_Q_16BIT = 1, CSIC_Q_8BIT = 2 };

typedef enum csic_status {
  CSIC_OK = 0,
  CSIC_EINVAL_DIMS = -1,      /* "Width and height must be positive" (SpatialDownsampler.scala:7, ImageProcessor.scala:22-23) */
  CSIC_EINVAL_FACTOR = -2,    /* "Factor must be 1, 2, 4, or 8" (SpatialDownsampler.scala:8, ImageProcessor.scala:24) */
  CSIC_EINVAL_DIVISIBLE = -3, /* "Image dimensions must be divisible by spatial downsampling factor." (ImageProcessor.scala:25) */
  CSIC_EINVAL_CHROMA_A = -4,  /* "param_a must be 4, 2, or 1. Got $a" (ChromaSubsampler.scala:17) */
  CSIC_EINVAL_CHROMA_B = -5,  /* "param_b must be equal to param_a ($a) or 0. Got $b" (ChromaSubsampler.scala:18) */
  CSIC_EINVAL_QBITS = -6,     /* "Y target bits must be between 1 and 8. Got $n" (ColorQuantizer.scala:13-15) */
  CSIC_EINVAL_OPS = -7,       /* "op1, op2, and op3 types must be distinct and form a permutation." (ImageCompressorTop.scala:28-31) */
  CSIC_EINVAL_MODE = -8,      /* round_mode / pool_mode / out_format / legacy enum out of range */
  CSIC_EINVAL_ARG = -9,       /* NULL pointer, bad band, bad device index */
  CSIC_ENODEVICE = -10,       /* no CUDA device / driver: there is no CPU fallback */
  CSIC_ECUDA = -11,           /* a CUDA call failed; csic_last_error() has the text */
  CSIC_ENOMEM = -12
} csic_status;

/* The parameter surface of `class ImageCompressorTop(width, height, chroma_param_a_config,
 * chroma_param_b_config, yTargetQuantBitsConfig, cbTargetQuantBitsConfig, crTargetQuantBitsConfig,
 * downFactorConfig, op1Type, op2Type, op3Type)` -- ImageCompressorTop.scala:11-25 -- plus three
 * build-side selectors.  POD, 16 x int32. */
typedef struct csic_params {
  int32_t width, height;            /* input frame, pixels */
  int32_t chroma_a, chroma_b;       /* J:a:b with J = 4 */
  int32_t y_bits, cb_bits, cr_bits; /* ColorQuantizer target bits, 1..8 */
  int32_t factor;                   /* SpatialDownsampler factor 1,2,4,8 */
  int32_t op[3];                    /* csic_step, a permutation of {1,2,3} */
  int32_t round_mode;               /* csic_round_mode */
  int32_t pool_mode;                /* csic_pool_mode */
  int32_t out_format;               /* csic_out_format */
  int32_t in_format;                /* csic_in_format (0 = RGB24, the reference's pixel stream) */
  int32_t reserved;                 /* must be 0 */
} csic_params;

typedef struct csic_ctx csic_ctx;   /* one per (host thread, GPU); not thread-safe */

/* ---- parameter helpers (host only, no device needed) ------------------------------------------ */

/* Defaults of `ImageCompressionApp` (ImageCompressorTopApp.scala:164-173): a=b=4, 8/8/8 bits, sf=8,
 * spatial -> color -> chroma; FLOOR, DECIMATE, YCC888. */
CSIC_API int csic_params_default(int32_t width, int32_t height, csic_params* out);

/* `ImageProcessorParams(width,height,factor,chromaParamA,chromaParamB)` + `class ImageProcessor`
 * (ImageProcessor.scala:15-63): fixed order toYC -> chroma -> spatial, no quantiser (8/8/8), and the
 * extra divisibility requirement (:25); checks in the case class's order (:22-28: width, height, factor,
 * divisibility, chromaParamA, chromaParamB). */
CSIC_API int csic_params_from_image_processor(int32_t width, int32_t height, int32_t factor, int32_t chroma_a,
                                     int32_t chroma_b, csic_params* out);

/* Legacy surface `ImageCompressorTop(w,h,ChromaSubsamplingMode,QuantizationMode,factor)` (SURVEY.md F4):
 * CHROMA_444/422/420 -> (4,4)/(2,2)/(2,0); Q_24BIT/Q_16BIT/Q_8BIT -> (8,8,8)/(6,5,5)/(3,3,2);
 * order chroma -> color -> spatial. */
CSIC_API int csic_params_from_legacy(int32_t width, int32_t height, int32_t chroma_mode, int32_t quant_mode,
                            int32_t factor, csic_params* out);

/* All `require(...)` predicates of ChromaSubsampler.scala:13-18, ColorQuantizer.scala:12-15,
 * SpatialDownsampler.scala:7-8, ImageCompressorTop.scala:27-31, evaluated in the ORDER the Scala constructor
 * evaluates them (ops :28-31 -> SpatialDownsampler :45 -> ColorQuantizer :46-51 -> ChromaSubsampler :53-59), so a
 * parameter set that is invalid in several ways reports the same first failure as `new ImageCompressorTop(...)`.
 * On failure writes the reference's message text (NUL terminated, truncated to n) into msg when msg != NULL. */
CSIC_API int csic_validate(const csic_params* p, char* msg, size_t n);

/* Output geometry.  out_w x out_h = ceil(W/f) x ceil(H/f): what the DUT emits
 * (SpatialDownsamplerSpec.scala:120-123); bytes_per_frame includes BUNDLE row padding. */
CSIC_API int csic_out_shape(const csic_params* p, int32_t* out_w, int32_t* out_h, size_t* out_row_bytes,
                   size_t* out_bytes_per_frame);

/* Geometry of CSIC_OUT_PLANAR: chroma plane size and the byte offsets of the Cb / Cr planes inside a frame. */
CSIC_API int csic_planar_shape(const csic_params* p, int32_t* chroma_w, int32_t* chroma_h, size_t* cb_offset,
                               size_t* cr_offset);

/* `ImageCompressionApp.parseProcessingStep` (ImageCompressorTopApp.scala:154-161): case-insensitive
 * "spatial"|"spatialsampling" -> 1, "color"|"colorquantization" -> 2, "chroma"|"chromasubsampling" -> 3,
 * anything else -> CSIC_EINVAL_OPS. */
CSIC_API int csic_parse_step(const char* name);

CSIC_API const char* csic_strerror(int status);
CSIC_API const char* csic_last_error(void);  /* thread-local text of the last CSIC_ECUDA */
CSIC_API int csic_abi_version(void);

/* ---- device side ------------------------------------------------------------------------------ */

CSIC_API int csic_device_count(void);        /* >= 0, or CSIC_ENODEVICE */

/* Binds a context to one GPU; owns a stream, events and the staging buffers of csic_process_host. */
CSIC_API int csic_create(int device, csic_ctx** out);
CSIC_API int csic_destroy(csic_ctx* ctx);

/* The hot path.  Replaces the body `chiseltest.RawTester.test(new ImageCompressorTop(...)){...}` of
 * ImageCompressionApp.processImage (ImageCompressorTopApp.scala:53-131) for n_frames independent frames
 * (the reference builds a fresh DUT per image, :53).  d_rgb: n_frames x H x W x (3|4) bytes per in_format,
 * raster order (pixel.red/green/blue, :86-89).  d_out: n_frames x bytes_per_frame.  Both device
 * pointers on ctx's GPU.  Asynchronous on `cuda_stream` (a cudaStream_t; NULL = the context's own
 * non-blocking stream -- pass cudaStreamLegacy (0x1) / cudaStreamPerThread (0x2) to name a default
 * stream); no hidden synchronisation. */
CSIC_API int csic_process_device(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t n_frames,
                        void* d_out, void* cuda_stream);

/* Same, for pitched buffers (cudaMallocPitch-style): rows start every *_pitch_bytes, frames every *_frame_stride
 * bytes (0 = dense).  When both pitches are multiples of 16 and cover the width rounded up to 16 output pixels
 * (in: that many x factor x bytes-per-pixel; out: that many x 3 or slot bytes) ANY frame width takes the TMA row
 * kernel; columns beyond the frame are read from / written into the row padding.  Dense buffers take it when
 * ceil(W/f) % 16 == 0 and the input row size is a multiple of 16 bytes.  Every other DECIMATE layout -- any width,
 * pitch or base-pointer alignment -- runs the flex kernel (TMA hull fetch + shifted 16-byte stores); only AVERAGE on
 * unaligned shapes and spatial-before-chroma shapes whose counter lines are not whole output rows use the
 * generic gather kernel (AVERAGE: the TMA pooling kernel on 16-byte-aligned shapes, any stage order). */
CSIC_API int csic_process_device_pitched(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t in_pitch_bytes,
                                         size_t in_frame_stride, size_t n_frames, void* d_out, size_t out_pitch_bytes,
                                         size_t out_frame_stride, void* cuda_stream);

/* Decoder of CSIC_OUT_PLANAR: replays the planes with the reference's sample-and-hold rule
 * (ChromaSubsampler.scala:52-65) into the YCC888 (expand_format 0) or RGB888 (1) stream, byte for byte what
 * csic_process_device would have produced with that out_format.  p->out_format must be CSIC_OUT_PLANAR. */
CSIC_API int csic_expand_planar_device(csic_ctx* ctx, const csic_params* p, const void* d_planar, size_t n_frames,
                                       void* d_out, int32_t expand_format, void* cuda_stream);

/* Row-band shard of ONE frame layout: processes output rows [out_row0, out_row0+out_rows) of every
 * frame, reading d_rgb / writing d_out at their whole-frame offsets (so bands of one frame may be
 * issued on different streams, or -- with per-GPU copies of the rows a band needs -- on different
 * GPUs).  csic_band_input_rows() tells which input rows a band reads. */
CSIC_API int csic_process_band(csic_ctx* ctx, const csic_params* p, const void* d_rgb, size_t n_frames,
                      void* d_out, int32_t out_row0, int32_t out_rows, void* cuda_stream);
CSIC_API int csic_band_input_rows(const csic_params* p, int32_t out_row0, int32_t out_rows, int32_t* in_row0,
                         int32_t* in_rows);

/* Host buffers in, host buffers out: H2D + kernel + D2H, chunked and double-buffered on the
 * context's streams, synchronous on return.  This is the call a Scala `processImage` replacement
 * makes (ImageCompressorTopApp.scala:23-145 minus PNG I/O).  rgb/out may be pageable or pinned; pageable
 * buffers (a JVM heap, malloc) are gathered into / scattered from pinned bounce buffers on several host threads.
 * With DECIMATE and f > 1 (and H % f == 0) only the input rows the pipeline reads -- every f-th -- are
 * copied to the device (strided 2-D copy); the result is identical.  Widths that break the TMA kernels' 16-byte
 * rules are re-pitched in the staging buffers, so they take the TMA row kernel too. */
CSIC_API int csic_process_host(csic_ctx* ctx, const csic_params* p, const uint8_t* rgb, size_t n_frames,
                      uint8_t* out);

/* Row band of every frame, host buffers (whole frames on the host): only the band's input rows go to the device
 * and only its output rows come back.  Lets several GPUs share ONE frame with no exchange (SURVEY.md 8(e) E2). */
CSIC_API int csic_process_host_band(csic_ctx* ctx, const csic_params* p, const uint8_t* rgb, size_t n_frames,
                                    uint8_t* out, int32_t out_row0, int32_t out_rows);

/* One host process, several GPUs (the reference's host is a single JVM process -- ImageCompressorTopApp.scala:149-190
 * drives one DUT from one `main`): one context and one host thread per device.  devices == NULL or n_devices <= 0 ->
 * every visible GPU.  csic_multi_process_host divides the batch by frames -- every GPU's chunk pipeline pulls its next
 * chunk from one shared cursor, so GPUs behind faster host links take more of the batch -- or, with fewer frames than
 * GPUs, cuts every frame into aligned row bands; no collective, no peer traffic.
 * csic_multi_set_option applies a csic_option to every context; CSIC_OPT_MULTI_STATIC_SPLIT = 1 restores the even
 * frame split.  csic_multi_host_bytes reports the bytes each device has received so far (n >= csic_multi_size). */
typedef struct csic_multi csic_multi;
CSIC_API int csic_multi_create(const int* devices, int n_devices, csic_multi** out);
CSIC_API int csic_multi_destroy(csic_multi* m);
CSIC_API int csic_multi_size(const csic_multi* m);
CSIC_API int csic_multi_process_host(csic_multi* m, const csic_params* p, const uint8_t* rgb, size_t n_frames,
                                     uint8_t* out);
CSIC_API int csic_multi_set_option(csic_multi* m, int option, int64_t value);
CSIC_API int csic_multi_host_bytes(const csic_multi* m, uint64_t* h2d_per_device, int n);

/* Pinned host memory helpers for callers that want the fast H2D/D2H path. */
CSIC_API int csic_host_alloc(size_t bytes, void** out);
CSIC_API int csic_host_free(void* p);

CSIC_API int csic_synchronize(csic_ctx* ctx);

/* Tuning / test knobs (never change results).  KERNEL_FAMILY: 0 = automatic (TMA row / pooling kernel whenever
 * the shape satisfies its 16-byte alignment rules, else the flex kernel, else the generic gather kernel), 1 = always
 * the generic gather kernel, 2 = never the aligned TMA kernels and no re-pitching in the host path (flex kernel
 * whenever it is eligible).  HOST_CHUNK_BYTES: input bytes per pipelined chunk of csic_process_host.
 * GRID_CTAS_PER_SM / STAGES / TILE_BYTES: overrides for the row kernel's persistent grid, ring depth and
 * input bytes per tile (0 = auto; STAGES / TILE_BYTES / BLOCK_THREADS also steer the flex kernel); HOST_FULL_FRAMES: 1 = csic_process_host copies whole frames even when a
 * DECIMATE pipeline reads only every f-th row (default 0: ship only the rows that are read); HOST_NO_BOUNCE: 1 =
 * do not stage pageable caller buffers through the context's pinned bounce buffers; BLOCK_THREADS: threads per CTA of the row kernel (multiple of 32, <= 512). */
enum csic_option { CSIC_OPT_KERNEL_FAMILY = 0, CSIC_OPT_HOST_CHUNK_BYTES = 1, CSIC_OPT_GRID_CTAS_PER_SM = 2,
                   CSIC_OPT_STAGES = 3, CSIC_OPT_TILE_BYTES = 4, CSIC_OPT_BLOCK_THREADS = 5, CSIC_OPT_HOST_FULL_FRAMES = 6, CSIC_OPT_HOST_NO_BOUNCE = 7,
                   CSIC_OPT_MULTI_STATIC_SPLIT = 100 /* csic_multi_set_option only */ };
CSIC_API int csic_set_option(csic_ctx* ctx, int option, int64_t value);

/* Diagnostics: total bytes csic_process_host has copied host -> device on this context. */
CSIC_API int csic_host_bytes(const csic_ctx* ctx, uint64_t* h2d_total);

/* Diagnostics: which kernel family the last process call on this ctx used (0 none, 1 generic gather
 * kernel, 2 TMA-staged row kernel, 3 TMA-staged pooling kernel of the AVERAGE extension, 4 any-alignment flex
 * kernel) and how many kernels it launched. */
CSIC_API int csic_last_kernel(const csic_ctx* ctx, int32_t* family, int64_t* launches_total);

/* Diagnostics: 1 when the last process call's row kernel dealt its tiles from a ticket counter, 0 when its CTAs walked
 * them round robin (or another kernel ran).  The planner deals by ticket where that measured faster (direct bundle
 * stores at f >= 2).  The counter is a pair of words the context keeps per stream (for its first 64 streams), which
 * every launch leaves zeroed; only launches enqueued directly on that stream use it, so they never overlap.  A launch
 * captured into a CUDA graph walks round robin and holds no context memory: graphs may be replayed on any stream, at
 * the same time as other work, and after csic_destroy. */
CSIC_API int csic_last_walk(const csic_ctx* ctx, int32_t* ticketed);

#ifdef __cplusplus
}
#endif
#endif /* CSIC_H_ */
