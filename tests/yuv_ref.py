"""numpy reference of the raw camera YUV -> BGR24 conversion (cvs_yuv_to_bgr_device, cvs_submit_yuv), plus the frames the
YUV tests feed it.  Test infrastructure only; pinned to cv2.cvtColor by tests/test_yuv_oracle.py, which also checks
that nothing under cudavideostream_b200/ refers to it.  It lives beside its only users, the YUV tests, rather than in
oracle/: the oracle package is the fixed reference the existing suites measure the library against, and this change
adds to the library without changing that reference.

Formats as include/cvs_b200.h packs them (rows without padding):
    YUYV  Y0 U Y1 V per pixel pair, 2W bytes per row
    NV12  Y plane (W x H), then U V interleaved (W bytes x H/2 rows)
    I420  Y plane (W x H), then the U plane and the V plane (W/2 x H/2 each)
"""
import numpy as np

YUYV, NV12, I420 = 1, 2, 3
NAMES = {YUYV: "yuyv", NV12: "nv12", I420: "i420"}


def frame_bytes(fmt, w, h):
    return 2 * w * h if fmt == YUYV else w * h * 3 // 2


def planes(fmt, buf, w, h):
    """(Y [h, w], U [hc, w/2], V [hc, w/2]) views of a packed frame; hc = h (YUYV) or h/2."""
    b = np.ascontiguousarray(buf, dtype=np.uint8).reshape(-1)[:frame_bytes(fmt, w, h)]
    if fmt == YUYV:
        q = b.reshape(h, w // 2, 4)
        return q[:, :, [0, 2]].reshape(h, w), q[:, :, 1], q[:, :, 3]
    y = b[:w * h].reshape(h, w)
    if fmt == NV12:
        uv = b[w * h:].reshape(h // 2, w // 2, 2)
        return y, uv[:, :, 0], uv[:, :, 1]
    c = (w // 2) * (h // 2)
    return y, b[w * h:w * h + c].reshape(h // 2, w // 2), b[w * h + c:].reshape(h // 2, w // 2)


def yuv_to_bgr(fmt, buf, w, h):
    """OpenCV's fixed-point BT.601 limited-range conversion with nearest-neighbour chroma: [h, w, 3] uint8 BGR."""
    Y, U, V = planes(fmt, buf, w, h)
    U = np.repeat(U, 2, axis=1)
    V = np.repeat(V, 2, axis=1)
    if fmt != YUYV:
        U = np.repeat(U, 2, axis=0)
        V = np.repeat(V, 2, axis=0)
    y = np.maximum(Y.astype(np.int32) - 16, 0) * 1220542 + (1 << 19)
    u = U.astype(np.int32) - 128
    v = V.astype(np.int32) - 128
    out = np.empty((h, w, 3), dtype=np.uint8)
    out[:, :, 0] = np.clip((y + 2116026 * u) >> 20, 0, 255)
    out[:, :, 1] = np.clip((y - 409993 * u - 852492 * v) >> 20, 0, 255)
    out[:, :, 2] = np.clip((y + 1673527 * v) >> 20, 0, 255)
    return out


def pack(fmt, Y, U, V):
    """Packed frame from full-resolution Y and subsampled U, V planes."""
    Y, U, V = (np.ascontiguousarray(a, dtype=np.uint8) for a in (Y, U, V))
    h, w = Y.shape
    if fmt == YUYV:
        q = np.empty((h, w // 2, 4), dtype=np.uint8)
        q[:, :, 0], q[:, :, 1], q[:, :, 2], q[:, :, 3] = Y[:, 0::2], U, Y[:, 1::2], V
        return q.reshape(-1)
    if fmt == NV12:
        return np.concatenate([Y.reshape(-1), np.stack([U, V], axis=2).reshape(-1)])
    return np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)])


def from_bgr(fmt, bgr, w, h):
    """A camera-like packed frame of a BGR picture (integer BT.601 encoder, chroma averaged over its pixels).  Any YUV
    bytes are valid input; this only makes synthetic sequences look like what a camera sends."""
    f = np.ascontiguousarray(bgr, dtype=np.uint8).reshape(h, w, 3).astype(np.int32)
    B, G, R = f[:, :, 0], f[:, :, 1], f[:, :, 2]
    Y = ((66 * R + 129 * G + 25 * B + 128) >> 8) + 16
    U = ((-38 * R - 74 * G + 112 * B + 128) >> 8) + 128
    V = ((112 * R - 94 * G - 18 * B + 128) >> 8) + 128
    ry = 1 if fmt == YUYV else 2
    U = U.reshape(h // ry, ry, w // 2, 2).sum(axis=(1, 3)) // (2 * ry)
    V = V.reshape(h // ry, ry, w // 2, 2).sum(axis=(1, 3)) // (2 * ry)
    return pack(fmt, np.clip(Y, 0, 255), np.clip(U, 0, 255), np.clip(V, 0, 255))


def exhaustive(fmt):
    """A 4096 x 4096 frame in which every (Y, U, V) triple occurs: (U, V) pair k of 2^16 is carried by 64 chroma
    samples of 2 x 2 pixels (NV12, I420) or 128 of 2 x 1 pixels (YUYV), whose pixels take the 256 values of Y once each."""
    S = 4096
    if fmt == YUYV:
        m = np.arange(S * S // 2, dtype=np.int64).reshape(S, S // 2)  # pixel pair index
        U, V, g = m & 255, (m >> 8) & 255, m >> 16                     # g: 0..127
        Y = np.empty((S, S), dtype=np.int64)
        Y[:, 0::2], Y[:, 1::2] = 2 * g, 2 * g + 1
    else:
        m = np.arange((S // 2) ** 2, dtype=np.int64).reshape(S // 2, S // 2)  # chroma sample index
        U, V, g = m & 255, (m >> 8) & 255, m >> 16                           # g: 0..63
        Y = np.empty((S, S), dtype=np.int64)
        for dy in (0, 1):
            for dx in (0, 1):
                Y[dy::2, dx::2] = 4 * g + 2 * dy + dx
    return pack(fmt, Y, U, V), S, S


def cv2_code(cv2, fmt):
    return {YUYV: cv2.COLOR_YUV2BGR_YUYV, NV12: cv2.COLOR_YUV2BGR_NV12, I420: cv2.COLOR_YUV2BGR_I420}[fmt]


def cv2_convert(cv2, fmt, buf, w, h):
    """cv2.cvtColor of a packed frame: [h, w, 3] BGR."""
    b = np.ascontiguousarray(buf, dtype=np.uint8).reshape(-1)[:frame_bytes(fmt, w, h)]
    src = b.reshape(h, w, 2) if fmt == YUYV else b.reshape(h * 3 // 2, w)
    return cv2.cvtColor(src, cv2_code(cv2, fmt))
