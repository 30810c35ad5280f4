"""Thin Python layer over the C ABI: parameter objects, error mapping, the per-GPU context.

Error behaviour mirrors the reference: a Scala `require(...)` failure raises
IllegalArgumentException at construction; here the same predicates (evaluated inside libcsic's
csic_validate, with the reference's message text) raise `IllegalArgumentException(ValueError)`.
"""
import ctypes
import enum

import numpy as np

from . import _ffi
from ._ffi import CsicParams


class IllegalArgumentException(ValueError):
    """What the reference throws from `require` (e.g. SpatialDownsamplerSpec.scala:147-151)."""
    def __init__(self, status, message):
        super().__init__(f"requirement failed: {message}")
        self.status = status


class CsicError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"csic status {status}: {message}")
        self.status = status


class ProcessingStep(enum.IntEnum):
    """object ProcessingStep extends ChiselEnum -- ImageCompressorTop.scala:7-9."""
    NoOp = 0
    SpatialSampling = 1
    ColorQuantization = 2
    ChromaSubsampling = 3


class RoundMode(enum.IntEnum):
    FLOOR = 0
    TRUNC = 1


class PoolMode(enum.IntEnum):
    DECIMATE = 0
    AVERAGE = 1


class InFormat(enum.IntEnum):
    """Input pixel layout; BGRA32 == a little-endian Java/AWT/scrimage ARGB int (alpha ignored)."""
    RGB24 = 0
    RGBA32 = 1
    BGRA32 = 2


class OutFormat(enum.IntEnum):
    YCC888 = 0
    RGB888 = 1
    BUNDLE64 = 2
    BUNDLE128 = 3
    PLANAR = 4


class ChromaSubsamplingMode(enum.IntEnum):
    """Legacy enum (SURVEY.md F4)."""
    CHROMA_444 = 0
    CHROMA_422 = 1
    CHROMA_420 = 2


class QuantizationMode(enum.IntEnum):
    """Legacy enum (SURVEY.md F4); mapping pinned by goldens G11-G13, G27."""
    Q_24BIT = 0
    Q_16BIT = 1
    Q_8BIT = 2


_EINVAL = range(-9, 0)
CSIC_ENODEVICE = -10


def check(rc, msg=None):
    if rc == 0:
        return
    L = _ffi.lib()
    text = msg or L.csic_strerror(rc).decode()
    if rc in _EINVAL:
        raise IllegalArgumentException(rc, text)
    if rc == -11:
        text = L.csic_last_error().decode() or text
    raise CsicError(rc, text)


def validate(p):
    buf = ctypes.create_string_buffer(256)
    rc = _ffi.lib().csic_validate(ctypes.byref(p), buf, len(buf))
    check(rc, buf.value.decode() or None)
    return p


def parse_processing_step(name):
    """ImageCompressionApp.parseProcessingStep -- ImageCompressorTopApp.scala:154-161."""
    rc = _ffi.lib().csic_parse_step(str(name).encode())
    if rc < 0:
        raise IllegalArgumentException(rc, f"Unknown processing step: {name}. Use 'spatial', 'color', or 'chroma'.")
    return ProcessingStep(rc)


def make_params(width, height, a=4, b=4, y_bits=8, cb_bits=8, cr_bits=8, factor=1,
                ops=(ProcessingStep.ChromaSubsampling, ProcessingStep.SpatialSampling, ProcessingStep.ColorQuantization),
                round_mode=RoundMode.FLOOR, pool_mode=PoolMode.DECIMATE, out_format=OutFormat.YCC888,
                in_format=InFormat.RGB24):
    p = CsicParams()
    p.width, p.height, p.chroma_a, p.chroma_b = int(width), int(height), int(a), int(b)
    p.y_bits, p.cb_bits, p.cr_bits, p.factor = int(y_bits), int(cb_bits), int(cr_bits), int(factor)
    p.op[0], p.op[1], p.op[2] = (int(o) for o in ops)
    p.round_mode, p.pool_mode, p.out_format = int(round_mode), int(pool_mode), int(out_format)
    p.in_format = int(in_format)
    return validate(p)


def params_from_legacy(width, height, chroma_mode, quant_mode, factor=1):
    p = CsicParams()
    check(_ffi.lib().csic_params_from_legacy(width, height, int(chroma_mode), int(quant_mode), factor, ctypes.byref(p)))
    return p


def out_shape(p):
    """(out_w, out_h, row_bytes, bytes_per_frame)."""
    w, h = ctypes.c_int32(), ctypes.c_int32()
    rb, fb = ctypes.c_size_t(), ctypes.c_size_t()
    check(_ffi.lib().csic_out_shape(ctypes.byref(p), ctypes.byref(w), ctypes.byref(h), ctypes.byref(rb), ctypes.byref(fb)))
    return w.value, h.value, rb.value, fb.value


def planar_shape(p):
    """(chroma_w, chroma_h, cb_offset, cr_offset) of the PLANAR output format."""
    w, h = ctypes.c_int32(), ctypes.c_int32()
    ob, orr = ctypes.c_size_t(), ctypes.c_size_t()
    check(_ffi.lib().csic_planar_shape(ctypes.byref(p), ctypes.byref(w), ctypes.byref(h), ctypes.byref(ob), ctypes.byref(orr)))
    return w.value, h.value, ob.value, orr.value


def band_input_rows(p, out_row0, out_rows):
    r0, n = ctypes.c_int32(), ctypes.c_int32()
    check(_ffi.lib().csic_band_input_rows(ctypes.byref(p), out_row0, out_rows, ctypes.byref(r0), ctypes.byref(n)))
    return r0.value, n.value


def device_count():
    return max(0, _ffi.lib().csic_device_count())


class PinnedBuffer:
    """Page-locked host memory from csic_host_alloc, viewed as a NumPy uint8 array."""
    def __init__(self, nbytes):
        self._ptr = ctypes.c_void_p()
        check(_ffi.lib().csic_host_alloc(nbytes, ctypes.byref(self._ptr)))
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(ctypes.cast(self._ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(max(nbytes, 1),))[:nbytes]

    def free(self):
        if self._ptr:
            self.array = None
            _ffi.lib().csic_host_free(self._ptr)
            self._ptr = ctypes.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _host_args(p, rgb, out):
    """Shape / dtype / size checks shared by every host entry point: a wrong array must raise here, not become an
    out-of-bounds native read or write.  -> (rgb [n,H,W,C] contiguous uint8, n, out [n*bytes_per_frame])."""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    if rgb.ndim == 3:
        rgb = rgb[None]
    ch = 3 if p.in_format == InFormat.RGB24 else 4
    if rgb.ndim != 4 or rgb.shape[1:] != (p.height, p.width, ch):
        raise IllegalArgumentException(-9, f"rgb must be [n,{p.height},{p.width},{ch}], got {rgb.shape}")
    n = rgb.shape[0]
    fb = out_shape(p)[3]
    if out is None:
        out = np.empty((n, fb), dtype=np.uint8)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.uint8 and out.flags.c_contiguous and out.flags.writeable
              and out.size == n * fb):
        raise IllegalArgumentException(-9, f"out must be a writable C-contiguous uint8 array of {n * fb} bytes")
    return rgb, n, out


class Context:
    """`csic_ctx`: one per (host thread, GPU)."""
    KERNEL_AUTO, KERNEL_GENERIC, KERNEL_NO_ALIGNED_TMA = 0, 1, 2

    def __init__(self, device=0):
        self._h = ctypes.c_void_p()
        check(_ffi.lib().csic_create(int(device), ctypes.byref(self._h)))
        self.device = int(device)

    def close(self):
        if self._h:
            _ffi.lib().csic_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_option(self, option, value):
        check(_ffi.lib().csic_set_option(self._h, int(option), int(value)))

    def synchronize(self):
        check(_ffi.lib().csic_synchronize(self._h))

    def host_bytes(self):
        n = ctypes.c_uint64()
        check(_ffi.lib().csic_host_bytes(self._h, ctypes.byref(n)))
        return n.value

    def last_kernel(self):
        fam, n = ctypes.c_int32(), ctypes.c_int64()
        check(_ffi.lib().csic_last_kernel(self._h, ctypes.byref(fam), ctypes.byref(n)))
        return fam.value, n.value

    def last_walk(self):
        """1: the last call's row kernel dealt its tiles from a ticket counter; 0: round robin or another kernel."""
        t = ctypes.c_int32()
        check(_ffi.lib().csic_last_walk(self._h, ctypes.byref(t)))
        return t.value

    # -- raw device pointers (ints); asynchronous on `stream` (int cudaStream_t handle, 0/None = ctx stream)
    def process_device(self, p, d_rgb, n_frames, d_out, stream=None):
        check(_ffi.lib().csic_process_device(self._h, ctypes.byref(p), d_rgb, n_frames, d_out, stream or None))

    def process_device_pitched(self, p, d_rgb, in_pitch, in_frame_stride, n_frames, d_out, out_pitch, out_frame_stride,
                               stream=None):
        check(_ffi.lib().csic_process_device_pitched(self._h, ctypes.byref(p), d_rgb, in_pitch, in_frame_stride, n_frames,
                                                     d_out, out_pitch, out_frame_stride, stream or None))

    def process_band(self, p, d_rgb, n_frames, d_out, out_row0, out_rows, stream=None):
        check(_ffi.lib().csic_process_band(self._h, ctypes.byref(p), d_rgb, n_frames, d_out, out_row0, out_rows,
                                           stream or None))

    # -- host buffers: NumPy uint8 in, NumPy uint8 out (H2D + kernel + D2H inside)
    def process_host(self, p, rgb, out=None):
        rgb, n, out = _host_args(p, rgb, out)
        check(_ffi.lib().csic_process_host(self._h, ctypes.byref(p), rgb.ctypes.data, n, out.ctypes.data))
        return out

    def expand_planar_torch(self, p, planar, to_rgb=False):
        """Decoder of OutFormat.PLANAR on the device: torch uint8 [n, bytes_per_frame] -> [n, out_h, out_w, 3]."""
        import torch
        assert planar.is_cuda and planar.dtype == torch.uint8 and planar.is_contiguous()
        w, h, _, fb = out_shape(p)
        n = planar.numel() // fb
        out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=planar.device)
        stream = torch.cuda.current_stream(planar.device).cuda_stream or 1
        check(_ffi.lib().csic_expand_planar_device(self._h, ctypes.byref(p), planar.data_ptr(), n, out.data_ptr(),
                                                   1 if to_rgb else 0, stream))
        return out

    def process_host_band(self, p, rgb, out, out_row0, out_rows):
        """Whole frames in host arrays; computes output rows [out_row0, out_row0+out_rows) of every frame in place
        in `out` ([n, bytes_per_frame]); other rows of `out` are left untouched."""
        if out is None:
            raise IllegalArgumentException(-9, "process_host_band writes a band of an existing output array: out is required")
        rgb, n, out = _host_args(p, rgb, out)
        oh = out_shape(p)[1]
        if not (0 <= int(out_row0) and 0 <= int(out_rows) and int(out_row0) + int(out_rows) <= oh):
            raise IllegalArgumentException(-9, f"band [{out_row0}, {out_row0}+{out_rows}) is outside 0..{oh}")
        check(_ffi.lib().csic_process_host_band(self._h, ctypes.byref(p), rgb.ctypes.data, n, out.ctypes.data,
                                                out_row0, out_rows))
        return out

    # -- torch CUDA tensors (plumbing only: torch owns the memory and the stream)
    def process_torch(self, p, rgb, out=None, out_row0=None, out_rows=None):
        import torch
        if not (rgb.is_cuda and rgb.dtype == torch.uint8 and rgb.is_contiguous()):
            raise IllegalArgumentException(-9, "rgb must be a contiguous CUDA uint8 tensor")
        frame = p.height * p.width * (3 if p.in_format == InFormat.RGB24 else 4)
        if rgb.numel() % frame != 0:
            raise IllegalArgumentException(-9, f"rgb holds {rgb.numel()} bytes, not a multiple of the {frame}-byte frame")
        n = rgb.numel() // frame
        _, oh, _, fb = out_shape(p)
        if out is None:
            out = torch.empty((n, fb), dtype=torch.uint8, device=rgb.device)
        elif not (out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == n * fb
                  and out.device == rgb.device):
            raise IllegalArgumentException(-9, f"out must be a contiguous CUDA uint8 tensor of {n * fb} bytes on {rgb.device}")
        if out_row0 is not None and not (0 <= int(out_row0) and 0 <= int(out_rows) and int(out_row0) + int(out_rows) <= oh):
            raise IllegalArgumentException(-9, f"band [{out_row0}, {out_row0}+{out_rows}) is outside 0..{oh}")
        # torch's default stream has handle 0, which the C ABI reads as "the context's own stream":
        # name it explicitly as cudaStreamLegacy (0x1) so the launch is ordered with torch's work.
        stream = torch.cuda.current_stream(rgb.device).cuda_stream or 1
        if out_row0 is None:
            self.process_device(p, rgb.data_ptr(), n, out.data_ptr(), stream)
        else:
            self.process_band(p, rgb.data_ptr(), n, out.data_ptr(), out_row0, out_rows, stream)
        return out


class MultiContext:
    """`csic_multi`: one process driving several GPUs (frames split across them, or row bands of each frame when
    there are fewer frames than GPUs)."""

    def __init__(self, devices=None):
        self._h = ctypes.c_void_p()
        if devices is None:
            check(_ffi.lib().csic_multi_create(None, 0, ctypes.byref(self._h)))
        else:
            arr = (ctypes.c_int * len(devices))(*devices)
            check(_ffi.lib().csic_multi_create(arr, len(devices), ctypes.byref(self._h)))

    def __len__(self):
        return _ffi.lib().csic_multi_size(self._h)

    def close(self):
        if self._h:
            _ffi.lib().csic_multi_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    STATIC_SPLIT = 100

    def set_option(self, option, value):
        check(_ffi.lib().csic_multi_set_option(self._h, int(option), int(value)))

    def host_bytes(self):
        """Bytes each device has received host -> device so far (shows how the shared cursor divided the batches)."""
        n = len(self)
        arr = (ctypes.c_uint64 * n)()
        check(_ffi.lib().csic_multi_host_bytes(self._h, arr, n))
        return list(arr)

    def process_host(self, p, rgb, out=None):
        rgb, n, out = _host_args(p, rgb, out)
        check(_ffi.lib().csic_multi_process_host(self._h, ctypes.byref(p), rgb.ctypes.data, n, out.ctypes.data))
        return out
