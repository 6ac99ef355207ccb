"""numpy reference of the 8-bit Bayer demosaic (cvs_bayer_to_bgr_device, cvs_submit_bayer), plus the mosaics the Bayer
tests feed it.  Test infrastructure only; pinned to cv2.cvtColor by tests/test_bayer_oracle.py, which also checks that
nothing under cudavideostream_b200/ refers to it.  Like tests/yuv_ref.py it lives beside its only users rather than in
oracle/, the fixed reference the existing suites measure the library against.

The rule (OpenCV's default bilinear demosaic, COLOR_Bayer<P>2BGR):
    W < 3 or H < 3: all zero.
    otherwise out(y, x) = I(clamp(y, 1, H-2), clamp(x, 1, W-2)), where at an interior pixel of mosaic colour c
      channel c                 = raw[y][x]
      c = G: horizontal colour   = (left + right + 1) >> 1,   vertical colour = (up + down + 1) >> 1
      c = R or B: G              = (left + right + up + down + 2) >> 2,
                  opposite colour = (four diagonals + 2) >> 2
Pattern P names the sensor's top-left 2x2 in V4L2 order (BGGR: row 0 B G B G ..., row 1 G R G R ...); P at (y, x) is
BGGR at (y + py, x + px).
"""
import numpy as np

BGGR, GBRG, GRBG, RGGB = 1, 2, 3, 4
PATTERNS = [BGGR, GBRG, GRBG, RGGB]
NAMES = {BGGR: "bggr", GBRG: "gbrg", GRBG: "grbg", RGGB: "rggb"}


def parity(pattern):
    """(py, px): the pattern's offset into BGGR."""
    k = pattern - 1
    return k >> 1, k & 1


def colours(pattern, h, w):
    """[h, w] channel index (0 B, 1 G, 2 R) the mosaic holds at each pixel."""
    py, px = parity(pattern)
    Y = (np.arange(h)[:, None] + py) & 1
    X = (np.arange(w)[None, :] + px) & 1
    return np.where((Y == 0) & (X == 0), 0, np.where((Y == 1) & (X == 1), 2, 1))


def bayer_to_bgr(pattern, raw):
    """[h, w] uint8 mosaic (any strides) -> [h, w, 3] uint8 BGR."""
    raw = np.asarray(raw, dtype=np.uint8)
    h, w = raw.shape
    out = np.zeros((h, w, 3), dtype=np.uint8)
    if h < 3 or w < 3:
        return out
    r = raw.astype(np.int32)
    c = r[1:-1, 1:-1]
    left, right, up, down = r[1:-1, :-2], r[1:-1, 2:], r[:-2, 1:-1], r[2:, 1:-1]
    diag = r[:-2, :-2] + r[:-2, 2:] + r[2:, :-2] + r[2:, 2:]
    hor, ver = (left + right + 1) >> 1, (up + down + 1) >> 1
    cross, diag = (left + right + up + down + 2) >> 2, (diag + 2) >> 2
    py, px = parity(pattern)
    Y = (np.arange(1, h - 1)[:, None] + py) & 1
    X = (np.arange(1, w - 1)[None, :] + px) & 1
    at_b, at_r = (Y == 0) & (X == 0), (Y == 1) & (X == 1)
    g_brow = (Y == 0) & (X == 1)  # G between B's horizontally, R's vertically
    g_rrow = (Y == 1) & (X == 0)  # G between R's horizontally, B's vertically
    B = np.select([at_b, at_r, g_brow, g_rrow], [c, diag, hor, ver])
    G = np.select([at_b | at_r], [cross], c)
    R = np.select([at_r, at_b, g_brow, g_rrow], [c, diag, ver, hor])
    inner = np.stack([B, G, R], axis=2).astype(np.uint8)
    yi = np.clip(np.arange(h), 1, h - 2) - 1
    xi = np.clip(np.arange(w), 1, w - 2) - 1
    return inner[yi][:, xi]


def mosaic(bgr, pattern):
    """The camera-like mosaic of a [h, w, 3] (or flat 3wh with h, w taken from its shape) BGR frame: each pixel keeps the
    one channel the pattern's colour filter passes there."""
    f = np.asarray(bgr, dtype=np.uint8)
    h, w = f.shape[:2]
    ch = colours(pattern, h, w)
    return np.take_along_axis(f, ch[:, :, None], axis=2)[:, :, 0].copy()


def cv2_code(cv2, pattern):
    """The four-letter OpenCV codes, named in sensor order like V4L2 (never the shifted two-letter aliases)."""
    return {BGGR: cv2.COLOR_BayerBGGR2BGR, GBRG: cv2.COLOR_BayerGBRG2BGR, GRBG: cv2.COLOR_BayerGRBG2BGR,
            RGGB: cv2.COLOR_BayerRGGB2BGR}[pattern]


def cv2_demosaic(cv2, pattern, raw):
    """cv2.cvtColor of a [h, w] mosaic: [h, w, 3] BGR."""
    return cv2.cvtColor(np.asarray(raw, dtype=np.uint8), cv2_code(cv2, pattern))
