"""ctypes binding of the C ABI (include/cvs_b200.h) and a Python mirror of the reference's
diff::cuda::CUDACore interface (server/include/kernels.cuh:13-43).

No torch types cross the boundary: device buffers are passed as integer addresses (e.g.
``tensor.data_ptr()``), CUDA streams as integer handles (``torch.cuda.current_stream().cuda_stream``).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("CVS_B200_LIB") or os.path.join(_HERE, "libcvs_b200.so")  # override: experiments only

MODE_NONE, MODE_HEAT_MAP, MODE_RED_BLACK, MODE_RED_OVERLAP = 0, 1, 2, 3
MODE_GRAY_WEIGHTED, MODE_BINARIZE, MODE_GRAY_AVERAGE, MODE_BINARIZE_AVERAGE = 4, 5, 6, 7
MAX_BATCH = 64  # CVS_MAX_BATCH
YUV_YUYV, YUV_NV12, YUV_I420 = 1, 2, 3  # cvs_yuv_format
BAYER_BGGR, BAYER_GBRG, BAYER_GRBG, BAYER_RGGB = 1, 2, 3, 4  # cvs_bayer_pattern (V4L2 sensor order)

CHARS_STR = "0123456789BFPSWbkps :/"  # server/include/common.h:13

_STATUS = {0: "CVS_OK", 1: "CVS_ERR_INVALID", 2: "CVS_ERR_CUDA", 3: "CVS_ERR_NOMEM", 4: "CVS_ERR_ALIGN",
           5: "CVS_ERR_CAPACITY", 6: "CVS_ERR_NODEVICE", 7: "CVS_ERR_INTERNAL"}


class CVSError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{_STATUS.get(status, status)}: {message}")
        self.status = status


class _Config(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("threshold", C.c_int), ("mode", C.c_int),
                ("noise_filter", C.c_int), ("ksize", C.c_int), ("kweights", C.POINTER(C.c_float)),
                ("device", C.c_int), ("base_frame", C.POINTER(C.c_uint8)), ("glyphs", C.POINTER(C.c_uint8)),
                ("glyph_w", C.c_int), ("glyph_h", C.c_int), ("glyph_chars", C.c_char_p),
                ("max_sequence", C.c_int)]


_u8p, _i32p, _u32p, _f32p = (C.POINTER(C.c_uint8), C.POINTER(C.c_int), C.POINTER(C.c_uint),
                             C.POINTER(C.c_float))
_vp, _sz = C.c_void_p, C.c_size_t

# every symbol include/cvs_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "cvs_last_error": (C.c_char_p, []),
    "cvs_abi_version": (C.c_int, []),
    "cvs_device_count": (C.c_int, []),
    "cvs_config_default": (None, [C.POINTER(_Config)]),
    "cvs_create": (C.c_int, [C.POINTER(_Config), C.POINTER(_vp)]),
    "cvs_destroy": (C.c_int, [_vp]),
    "cvs_reset": (C.c_int, [_vp, _u8p]),
    "cvs_alloc_host": (C.c_int, [C.POINTER(_vp), _sz]),
    "cvs_free_host": (C.c_int, [_vp]),
    "cvs_exec": (C.c_int, [_vp, _vp, _vp, C.c_char_p, _u32p, _vp]),
    "cvs_submit": (C.c_int, [_vp, _vp, _vp, C.c_char_p, _vp, _vp, C.POINTER(C.c_uint64)]),
    "cvs_wait": (C.c_int, [_vp, C.c_uint64]),
    "cvs_submit_io": (C.c_int, [_vp, _vp, _vp, _vp, C.c_char_p, _vp, _vp, C.POINTER(C.c_uint64)]),
    "cvs_get_timing": (C.c_int, [_vp, _f32p, _f32p, _f32p]),
    "cvs_get_reference": (C.c_int, [_vp, _vp]),
    "cvs_reference_device": (C.c_int, [_vp, C.POINTER(_vp)]),
    "cvs_run_sequence_device": (C.c_int, [_vp, _vp, _sz, C.c_int, _vp, _vp, _vp, _sz, _vp, _sz, C.c_char_p, _vp]),
    "cvs_sequence_status": (C.c_int, [_vp]),
    "cvs_launch_count": (C.c_uint64, [_vp]),
    "cvs_run_batch_device": (C.c_int, [C.POINTER(_vp), C.c_int, C.POINTER(_vp), _vp, _vp, _vp, _sz, _vp, _sz,
                                       C.POINTER(C.c_char_p), _vp]),
    "cvs_submit_io_batch": (C.c_int, [C.POINTER(_vp), C.c_int, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                      C.POINTER(C.c_char_p), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_uint64)]),
    "cvs_heat_map_device": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    "cvs_red_map_device": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "cvs_grayscale_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    "cvs_binarize_device": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    "cvs_noise_filter_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _f32p, _vp]),
    "cvs_client_apply_device": (C.c_int, [_vp, _vp, _vp, _vp, _sz, _vp]),
    "cvs_wire_bound": (_sz, [C.c_int, C.c_int]),
    "cvs_wire_size": (_sz, [_vp]),
    "cvs_submit_wire": (C.c_int, [_vp, _vp, _vp, _vp, C.c_char_p, C.POINTER(C.c_uint64)]),
    "cvs_wire_encode_device": (C.c_int, [_vp, _vp, _vp, _sz, C.c_int, C.c_int, _vp, _vp, _vp]),
    "cvs_wire_decode_device": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    "cvs_wire_decode_status": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "cvs_submit_jpeg": (C.c_int, [_vp, _vp, _sz, _vp, _vp, C.c_char_p, _vp, _vp, C.POINTER(C.c_uint64)]),
    "cvs_submit_jpeg_wire": (C.c_int, [_vp, _vp, _sz, _vp, _vp, C.c_char_p, C.POINTER(C.c_uint64)]),
    "cvs_decode_jpeg_device": (C.c_int, [_vp, _vp, _sz, _vp, _vp]),
    "cvs_yuv_frame_bytes": (_sz, [C.c_int, C.c_int, C.c_int]),
    "cvs_submit_yuv": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_char_p, _vp, _vp, C.POINTER(C.c_uint64)]),
    "cvs_submit_yuv_wire": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_char_p, C.POINTER(C.c_uint64)]),
    "cvs_yuv_to_bgr_device": (C.c_int, [C.c_int, C.POINTER(_vp), C.POINTER(_sz), _vp, C.c_int, C.c_int, _vp]),
    "cvs_submit_bayer": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_char_p, _vp, _vp, C.POINTER(C.c_uint64)]),
    "cvs_submit_bayer_wire": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_char_p, C.POINTER(C.c_uint64)]),
    "cvs_bayer_to_bgr_device": (C.c_int, [C.c_int, _vp, _sz, _vp, C.c_int, C.c_int, _vp]),
    "cvs_synth_base_device": (C.c_int, [_vp, C.c_int, C.c_int, C.c_uint64, _vp]),
    "cvs_synth_next_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32, _vp]),
}

_lib = None


def library_path() -> str:
    return _LIB_PATH


def load_library() -> C.CDLL:
    """Loads libcvs_b200.so.  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError(f"{_LIB_PATH} is missing: build it with `python -m cudavideostream_b200.build` "
                               "(__graft_entry__.build()); there is no CPU fallback")
        lib = C.CDLL(_LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(status: int) -> None:
    if status != 0:
        raise CVSError(status, load_library().cvs_last_error().decode(errors="replace"))


def device_count() -> int:
    return load_library().cvs_device_count()


class HostBuffer:
    """Pinned host memory from cvs_alloc_host (replaces CUDACore::alloc_arrays, kernels.cu:531-536)."""

    def __init__(self, nbytes: int):
        self._ptr = _vp()
        _check(load_library().cvs_alloc_host(C.byref(self._ptr), nbytes))
        self.nbytes = nbytes
        self.ptr = self._ptr.value

    def array(self, dtype=np.uint8) -> np.ndarray:
        n = self.nbytes // np.dtype(dtype).itemsize
        return np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(np.ctypeslib.as_ctypes_type(dtype))), shape=(n,))

    def free(self):
        if self.ptr:
            load_library().cvs_free_host(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def alloc_host(nbytes: int) -> HostBuffer:
    return HostBuffer(nbytes)


def yuv_frame_bytes(fmt: int, width: int, height: int) -> int:
    """cvs_yuv_frame_bytes: bytes of one packed YUV frame (0 if the format is unknown or the size odd where it forbids)."""
    return int(load_library().cvs_yuv_frame_bytes(fmt, width, height))


class Stream:
    """One camera stream = one cvs_handle (reference-frame state on one GPU)."""

    def __init__(self, width: int, height: int, base_frame: np.ndarray, threshold: int = 20, mode: int = 0,
                 noise_filter: bool = False, ksize: int = 3, kweights=None, device: int = 0, glyphs=None,
                 glyph_w: int = 0, glyph_h: int = 0, glyph_chars: str = CHARS_STR, max_sequence: int = 512):
        lib = load_library()
        self.width, self.height, self.total = width, height, 3 * width * height
        self.mode, self.device = mode, device
        cfg = _Config()
        lib.cvs_config_default(C.byref(cfg))
        cfg.width, cfg.height, cfg.threshold, cfg.mode = width, height, threshold, mode
        cfg.noise_filter, cfg.ksize, cfg.device, cfg.max_sequence = int(bool(noise_filter)), ksize, device, max_sequence
        self._base = np.ascontiguousarray(base_frame, dtype=np.uint8).reshape(-1)
        if self._base.size != self.total:
            raise ValueError("base_frame must hold 3*width*height bytes")
        cfg.base_frame = self._base.ctypes.data_as(_u8p)
        self._k = None
        if kweights is not None:
            self._k = np.ascontiguousarray(kweights, dtype=np.float32).reshape(-1)
            cfg.kweights = self._k.ctypes.data_as(_f32p)
        self._glyphs = None
        self._chars = glyph_chars.encode()
        if glyphs is not None:
            self._glyphs = np.ascontiguousarray(glyphs, dtype=np.uint8).reshape(-1)
            cfg.glyphs = self._glyphs.ctypes.data_as(_u8p)
            cfg.glyph_w, cfg.glyph_h, cfg.glyph_chars = glyph_w, glyph_h, self._chars
        self._h = _vp()
        _check(lib.cvs_create(C.byref(cfg), C.byref(self._h)))

    # -- drop-in path ------------------------------------------------------------------------------
    def exec_raw(self, frame_ptr: int, show_ptr, text: str, pos_ptr, xs_ptr: int) -> None:
        _check(load_library().cvs_exec(self._h, frame_ptr, show_ptr, text.encode(), pos_ptr, xs_ptr))

    def submit_raw(self, frame_ptr: int, show_ptr, text: str, pos_ptr: int, xs_ptr: int) -> int:
        t = C.c_uint64(0)
        _check(load_library().cvs_submit(self._h, frame_ptr, show_ptr, text.encode(), pos_ptr, xs_ptr, C.byref(t)))
        return t.value

    def submit_io_raw(self, frame_ptr: int, diff_ptr: int, show_ptr, text: str, pos_ptr: int, xs_ptr: int) -> int:
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_io(self._h, frame_ptr, diff_ptr, show_ptr, text.encode(), pos_ptr, xs_ptr,
                                            C.byref(t)))
        return t.value

    def submit_wire_raw(self, frame_ptr: int, wire_ptr: int, show_ptr, text: str) -> int:
        """cvs_submit_wire: the payload comes back as one compact CVW1 frame in wire_ptr (see cudavideostream_b200.wire)."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_wire(self._h, frame_ptr, wire_ptr, show_ptr, text.encode(), C.byref(t)))
        return t.value

    def submit_jpeg_raw(self, jpeg_ptr: int, jpeg_bytes: int, diff_ptr: int, show_ptr, text: str, pos_ptr: int, xs_ptr: int) -> int:
        """cvs_submit_jpeg: the frame arrives as the camera's JPEG bitstream and is decoded on the GPU (the library's own
        kernels: OpenCV's pixels bit for bit)."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_jpeg(self._h, jpeg_ptr, jpeg_bytes, diff_ptr, show_ptr, text.encode(), pos_ptr, xs_ptr,
                                              C.byref(t)))
        return t.value

    def submit_jpeg_wire_raw(self, jpeg_ptr: int, jpeg_bytes: int, wire_ptr: int, show_ptr, text: str) -> int:
        """cvs_submit_jpeg_wire: JPEG bitstream in, one compact CVW1 frame out."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_jpeg_wire(self._h, jpeg_ptr, jpeg_bytes, wire_ptr, show_ptr, text.encode(), C.byref(t)))
        return t.value

    def submit_yuv_raw(self, fmt: int, yuv_ptr: int, diff_ptr: int, show_ptr, text: str, pos_ptr: int, xs_ptr: int) -> int:
        """cvs_submit_yuv: the frame arrives in the camera's packed YUV layout (YUV_YUYV / YUV_NV12 / YUV_I420,
        yuv_frame_bytes bytes) and is converted to BGR on the GPU (cv2.cvtColor's pixels bit for bit)."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_yuv(self._h, fmt, yuv_ptr, diff_ptr, show_ptr, text.encode(), pos_ptr, xs_ptr,
                                             C.byref(t)))
        return t.value

    def submit_yuv_wire_raw(self, fmt: int, yuv_ptr: int, wire_ptr: int, show_ptr, text: str) -> int:
        """cvs_submit_yuv_wire: packed YUV frame in, one compact CVW1 frame out."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_yuv_wire(self._h, fmt, yuv_ptr, wire_ptr, show_ptr, text.encode(), C.byref(t)))
        return t.value

    def submit_bayer_raw(self, pattern: int, raw_ptr: int, diff_ptr: int, show_ptr, text: str, pos_ptr: int,
                         xs_ptr: int) -> int:
        """cvs_submit_bayer: the frame arrives as the camera's 8-bit Bayer mosaic (BAYER_BGGR / _GBRG / _GRBG / _RGGB,
        width * height bytes) and is demosaiced to BGR on the GPU (cv2.cvtColor's pixels bit for bit)."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_bayer(self._h, pattern, raw_ptr, diff_ptr, show_ptr, text.encode(), pos_ptr,
                                               xs_ptr, C.byref(t)))
        return t.value

    def submit_bayer_wire_raw(self, pattern: int, raw_ptr: int, wire_ptr: int, show_ptr, text: str) -> int:
        """cvs_submit_bayer_wire: Bayer mosaic in, one compact CVW1 frame out."""
        t = C.c_uint64(0)
        _check(load_library().cvs_submit_bayer_wire(self._h, pattern, raw_ptr, wire_ptr, show_ptr, text.encode(),
                                                    C.byref(t)))
        return t.value

    def decode_jpeg_device(self, jpeg: bytes, d_out: int, cuda_stream: int = 0) -> None:
        buf = (C.c_uint8 * len(jpeg)).from_buffer_copy(jpeg)
        _check(load_library().cvs_decode_jpeg_device(self._h, C.addressof(buf), len(jpeg), d_out, cuda_stream or None))

    def wait(self, ticket: int) -> None:
        _check(load_library().cvs_wait(self._h, ticket))

    def exec(self, frame: np.ndarray, text: str = "", want_show: bool = True):
        """cvs_exec on numpy buffers.  Returns (pos, xs[pos], diff[pos], show or None)."""
        f = np.ascontiguousarray(frame, dtype=np.uint8).reshape(-1).copy()
        if f.size != self.total:
            raise ValueError("frame must hold 3*width*height bytes")
        xs = np.empty(self.total, dtype=np.int32)
        show = np.zeros(self.total, dtype=np.uint8) if (self.mode and want_show) else None
        pos = C.c_uint(0)
        _check(load_library().cvs_exec(self._h, f.ctypes.data, show.ctypes.data if show is not None else None,
                                       text.encode(), C.byref(pos), xs.ctypes.data))
        n = pos.value
        return n, xs[:n].copy(), f[:n].copy(), show

    def timing(self):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        _check(load_library().cvs_get_timing(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"h2d_us": a.value, "kernel_us": b.value, "d2h_us": c.value}

    # -- state --------------------------------------------------------------------------------------
    def reference(self) -> np.ndarray:
        out = np.empty(self.total, dtype=np.uint8)
        _check(load_library().cvs_get_reference(self._h, out.ctypes.data))
        return out

    def reference_device(self) -> int:
        p = _vp()
        _check(load_library().cvs_reference_device(self._h, C.byref(p)))
        return p.value

    def reset(self, base_frame: np.ndarray) -> None:
        b = np.ascontiguousarray(base_frame, dtype=np.uint8).reshape(-1)
        _check(load_library().cvs_reset(self._h, b.ctypes.data_as(_u8p)))

    # -- device-resident sequence ---------------------------------------------------------------------
    def run_sequence_device(self, d_frames: int, frame_stride: int, nframes: int, d_pos: int, d_xs: int,
                            d_diff: int, capacity: int, d_show: int = 0, show_stride: int = 0, text: str = "",
                            cuda_stream: int = 0) -> None:
        _check(load_library().cvs_run_sequence_device(self._h, d_frames, frame_stride, nframes, d_pos, d_xs,
                                                      d_diff, capacity, d_show or None, show_stride,
                                                      text.encode(), cuda_stream or None))

    def sequence_status(self) -> None:
        _check(load_library().cvs_sequence_status(self._h))

    def launch_count(self) -> int:
        return int(load_library().cvs_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            load_library().cvs_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ptrs(values):
    """n addresses (None / 0 = NULL) as a C array of void*, or NULL for None."""
    return None if values is None else (_vp * len(values))(*[v or None for v in values])


def _texts(texts):
    return None if texts is None else (C.c_char_p * len(texts))(*[None if t is None else t.encode() for t in texts])


def run_batch_device(streams, d_frames, d_pos: int, d_xs: int, d_diff: int, capacity: int, d_show: int = 0,
                     show_stride: int = 0, texts=None, cuda_stream: int = 0) -> None:
    """cvs_run_batch_device: one device-resident frame of each stream (d_frames[i] for streams[i]) in one stream-kernel
    launch; outputs laid out like a sequence indexed by camera.  texts: None or one entry (str or None) per stream."""
    n = len(streams)
    hs = (_vp * n)(*[s._h.value for s in streams])
    _check(load_library().cvs_run_batch_device(hs, n, _ptrs(d_frames), d_pos, d_xs, d_diff, capacity, d_show or None,
                                               show_stride, _texts(texts), cuda_stream or None))


def submit_io_batch(streams, frames, diff_out, pos, xs, show=None, texts=None) -> list:
    """cvs_submit_io_batch: one frame of each stream; returns the tickets (tickets[i] is completed by streams[i].wait).
    frames, diff_out, pos, xs (and show, None entries allowed) are lists of host addresses, one per stream."""
    n = len(streams)
    hs = (_vp * n)(*[s._h.value for s in streams])
    tk = (C.c_uint64 * n)()
    _check(load_library().cvs_submit_io_batch(hs, n, _ptrs(frames), _ptrs(diff_out), _ptrs(show), _texts(texts),
                                              _ptrs(pos), _ptrs(xs), tk))
    return list(tk)


class matsz:
    """diff::utils::matsz (server/include/utils.hpp:7-16)."""

    def __init__(self, height: int = 0, width: int = 0):
        self.height, self.width = height, width

    def area(self) -> int:
        return self.height * self.width


class CUDACore:
    """Python mirror of diff::cuda::CUDACore (server/include/kernels.cuh:38-41): same member names, argument
    order and meaning; compile-time switches of common.h are keyword arguments."""

    def __init__(self, charsPx, charsSz: matsz, k, total: int, sampleMatData, frameSz: matsz, *,
                 noise_visualizer: int = 0, noise_filter: bool = False, K: int = 3, lr_thresholds: int = 20,
                 chars_str: str = CHARS_STR, device: int = 0):
        if total != 3 * frameSz.area():
            raise ValueError("total must be 3 * frameSz.area()")
        self.frameSz, self.total = frameSz, total
        self._s = Stream(frameSz.width, frameSz.height, sampleMatData, threshold=lr_thresholds,
                         mode=noise_visualizer, noise_filter=noise_filter, ksize=K, kweights=k, device=device,
                         glyphs=charsPx, glyph_w=charsSz.width if charsSz else 0,
                         glyph_h=charsSz.height if charsSz else 0, glyph_chars=chars_str)

    @staticmethod
    def alloc_arrays(r: int, c: int):
        """Returns (h_frame, n_frame, o_frame, h_xs) as pinned HostBuffers (kernels.cu:531-536)."""
        n = 3 * r * c
        return alloc_host(n + 32), alloc_host(n + 32), alloc_host(n + 32), alloc_host(4 * n + 32)

    def exec_core(self, frameData: HostBuffer, showReadyNData, text: str, h_xs: HostBuffer) -> int:
        """Runs one frame; frameData[0:pos] becomes the diff bytes, h_xs[0:pos] the indices.  Returns h_pos."""
        pos = C.c_uint(0)
        self._s.exec_raw(frameData.ptr, showReadyNData.ptr if showReadyNData is not None else None, text,
                         C.byref(pos), h_xs.ptr)
        return pos.value

    def chunkt_size(self) -> int:
        return 32

    @property
    def stream(self) -> Stream:
        return self._s
