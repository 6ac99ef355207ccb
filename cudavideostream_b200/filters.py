"""Stand-alone display filters of the C ABI on device buffers (integer device addresses)."""
from __future__ import annotations

import numpy as np

from .api import _check, _f32p, _sz, _vp, load_library


def heat_map(d_prev: int, d_cur: int, d_out: int, width: int, height: int, stream: int = 0) -> None:
    _check(load_library().cvs_heat_map_device(d_prev, d_cur, d_out, width, height, stream or None))


def red_map(d_prev: int, d_cur: int, d_out: int, width: int, height: int, threshold: int = 20,
            stream: int = 0) -> None:
    _check(load_library().cvs_red_map_device(d_prev, d_cur, d_out, width, height, threshold, stream or None))


def grayscale(d_frame: int, d_out: int, width: int, height: int, weighted: bool, channels: int,
              stream: int = 0) -> None:
    _check(load_library().cvs_grayscale_device(d_frame, d_out, width, height, int(weighted), channels,
                                               stream or None))


def binarize(d_frame: int, d_out: int, d_gray: int, d_hist_thr: int, width: int, height: int, weighted: bool,
             clamp_lo: int = 50, clamp_hi: int = 200, stream: int = 0) -> None:
    _check(load_library().cvs_binarize_device(d_frame, d_out, d_gray, d_hist_thr, width, height, int(weighted),
                                              clamp_lo, clamp_hi, stream or None))


def noise_filter(d_frame: int, d_out: int, width: int, height: int, ksize: int, weights, stream: int = 0) -> None:
    w = np.ascontiguousarray(weights, dtype=np.float32).reshape(-1)
    _check(load_library().cvs_noise_filter_device(d_frame, d_out, width, height, ksize, w.ctypes.data_as(_f32p),
                                                  stream or None))


def client_apply(d_frame: int, d_xs: int, d_diff: int, d_pos: int, capacity: int, stream: int = 0) -> None:
    _check(load_library().cvs_client_apply_device(d_frame, d_xs, d_diff, d_pos, capacity, stream or None))


def yuv_to_bgr(fmt: int, planes, pitches, d_out: int, width: int, height: int, stream: int = 0) -> None:
    """cvs_yuv_to_bgr_device: a raw YUV frame in device memory -> packed BGR24 (cv2.cvtColor's pixels).  planes: the
    device addresses of the format's planes (YUYV: 1; NV12: Y, UV; I420: Y, U, V), pitches: their row pitches in bytes."""
    # three entries whatever the format: missing planes arrive as NULL and are refused, never read past the array
    _check(load_library().cvs_yuv_to_bgr_device(fmt, (_vp * 3)(*planes), (_sz * 3)(*pitches), d_out, width, height,
                                                stream or None))


def bayer_to_bgr(pattern: int, d_raw: int, pitch: int, d_out: int, width: int, height: int, stream: int = 0) -> None:
    """cvs_bayer_to_bgr_device: an 8-bit Bayer mosaic in device memory (rows `pitch` bytes apart) -> packed BGR24
    (cv2.cvtColor's pixels)."""
    _check(load_library().cvs_bayer_to_bgr_device(pattern, d_raw, pitch, d_out, width, height, stream or None))
