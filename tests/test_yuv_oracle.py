"""The raw-YUV conversion's reference (tests/yuv_ref.py) is cv2.cvtColor's COLOR_YUV2BGR_YUYV / _NV12 / _I420, on every
(Y, U, V) triple and on random frames of camera and odd-multiple sizes; the library's frame sizes and argument checks
agree with what cv2 accepts.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

import yuv_ref as Y

FORMATS = [Y.YUYV, Y.NV12, Y.I420]
SIZES = [(2, 2), (6, 4), (34, 10), (1918, 1078), (1920, 1080), (3840, 2160)]


@pytest.mark.parametrize("fmt", FORMATS, ids=Y.NAMES.get)
def test_every_triple_matches_cv2(fmt):
    cv2 = pytest.importorskip("cv2")
    buf, w, h = Y.exhaustive(fmt)
    Yp, U, V = Y.planes(fmt, buf, w, h)
    # the frame does hold all 2^24 triples
    ry = 1 if fmt == Y.YUYV else 2
    key = (Yp.astype(np.int64) << 16) | (np.repeat(np.repeat(U, 2, 1), ry, 0).astype(np.int64) << 8) | \
        np.repeat(np.repeat(V, 2, 1), ry, 0)
    assert np.bincount(key.reshape(-1), minlength=1 << 24).min() >= 1
    want = Y.cv2_convert(cv2, fmt, buf, w, h)
    got = Y.yuv_to_bgr(fmt, buf, w, h)
    bad = np.flatnonzero((got != want).any(axis=2))
    assert bad.size == 0, f"{bad.size} pixels differ from cv2, first at {bad[:5]}"


@pytest.mark.parametrize("fmt", FORMATS, ids=Y.NAMES.get)
@pytest.mark.parametrize("w,h", SIZES)
def test_random_frames_match_cv2(fmt, w, h):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(w * 7919 + h * 31 + fmt)
    buf = rng.integers(0, 256, size=Y.frame_bytes(fmt, w, h), dtype=np.uint8)
    assert np.array_equal(Y.yuv_to_bgr(fmt, buf, w, h), Y.cv2_convert(cv2, fmt, buf, w, h))


@pytest.mark.parametrize("fmt", FORMATS, ids=Y.NAMES.get)
def test_packing_round_trip(fmt):
    """pack / planes are inverse, and from_bgr gives the layout's size: the GPU tests build their frames with them."""
    rng = np.random.default_rng(fmt)
    w, h = 10, 6
    ry = 1 if fmt == Y.YUYV else 2
    Yp = rng.integers(0, 256, (h, w), dtype=np.uint8)
    U, V = (rng.integers(0, 256, (h // ry, w // 2), dtype=np.uint8) for _ in range(2))
    buf = Y.pack(fmt, Yp, U, V)
    assert buf.size == Y.frame_bytes(fmt, w, h)
    for a, b in zip(Y.planes(fmt, buf, w, h), (Yp, U, V)):
        assert np.array_equal(a, b)
    assert Y.from_bgr(fmt, rng.integers(0, 256, 3 * w * h, dtype=np.uint8), w, h).size == buf.size


def test_frame_bytes_and_odd_sizes_as_cv2(cvs):
    """cvs_yuv_frame_bytes is 2WH / 3WH/2, and 0 exactly for the sizes cv2.cvtColor refuses (YUYV: odd width; NV12 /
    I420: odd width or odd height)."""
    cv2 = pytest.importorskip("cv2")
    for fmt in FORMATS:
        for w in range(1, 9):
            for h in range(1, 9):
                shape = (h, w, 2) if fmt == Y.YUYV else (h * 3 // 2, w)
                try:
                    cv2.cvtColor(np.zeros(shape, np.uint8), Y.cv2_code(cv2, fmt))
                    ok = True
                except cv2.error:
                    ok = False
                got = cvs.yuv_frame_bytes(fmt, w, h)
                assert got == (Y.frame_bytes(fmt, w, h) if ok else 0), (fmt, w, h, got, ok)
    assert cvs.yuv_frame_bytes(Y.NV12, 1920, 1080) == 3110400
    assert cvs.yuv_frame_bytes(Y.YUYV, 1920, 1080) == 4147200
    assert cvs.yuv_frame_bytes(Y.I420, 3840, 2160) == 12441600
    for fmt in (0, 4, -1):
        assert cvs.yuv_frame_bytes(fmt, 64, 64) == 0
    assert cvs.yuv_frame_bytes(Y.NV12, 0, 64) == cvs.yuv_frame_bytes(Y.YUYV, 64, -2) == 0


def test_device_conversion_refuses_bad_arguments_without_a_device(cvs):
    """cvs_yuv_to_bgr_device checks its arguments before it looks for a device: unknown format, odd size, NULL or short
    pitch -> CVS_ERR_INVALID; a plane, pitch or output not 16-byte aligned -> CVS_ERR_ALIGN."""
    lib = cvs.load_library()
    P = C.c_void_p * 3
    Z = C.c_size_t * 3
    a = 1 << 20  # any 16-byte aligned address: a refusal touches nothing

    def call(fmt, planes, pitches, out=a, w=64, h=32):
        return lib.cvs_yuv_to_bgr_device(fmt, P(*planes), Z(*pitches), out, w, h, None)

    good = {Y.YUYV: ([a], [128]), Y.NV12: ([a, a], [64, 64]), Y.I420: ([a, a, a], [64, 32, 32])}
    for fmt, (pl, pi) in good.items():
        assert call(0, pl, pi) == 1 and call(7, pl, pi) == 1
        assert call(fmt, pl, pi, w=63) == 1
        assert call(fmt, pl, pi, out=None) == 1
        for i in range(len(pl)):
            q = list(pl)
            q[i] = None
            assert call(fmt, q, pi) == 1
            r = list(pi)
            r[i] -= 16
            assert call(fmt, pl, r) == 1, (fmt, i)
            q = list(pl)
            q[i] += 8
            assert call(fmt, q, pi) == 4
            r = list(pi)
            r[i] += 8
            assert call(fmt, pl, r) == 4
        assert call(fmt, pl, pi, out=a + 4) == 4
    assert call(Y.NV12, [a, a], [64, 64], h=31) == 1
    assert lib.cvs_yuv_to_bgr_device(Y.NV12, None, Z(64, 64, 0), a, 64, 32, None) == 1
    assert lib.cvs_yuv_to_bgr_device(Y.NV12, P(a, a), None, a, 64, 32, None) == 1


def test_conversion_kernel_is_integer_only_with_wide_accesses(cvs):
    """Each k_yuv_to_bgr<FORMAT> in the built library: 16-byte loads and three 16-byte stores on its fast path, no
    floating-point arithmetic, nothing in local memory."""
    import re
    import shutil
    import subprocess
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        sass = subprocess.run([tool, "-sass", cvs.library_path()], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError) as e:
        pytest.skip(f"cuobjdump unavailable: {e}")
    blocks = re.split(r"(?=\n\s*Function : )", sass)
    for fmt in FORMATS:
        hit = [b for b in blocks if re.search(r"Function : \S*k_yuv_to_bgrILi%dE" % fmt, b)]
        assert len(hit) == 1, f"k_yuv_to_bgr<{fmt}> missing from the library"
        k = hit[0]
        assert len(re.findall(r"\bSTG\.E\.128\b", k)) == 3, Y.NAMES[fmt]
        assert re.search(r"\bLDG\.E\.(128|64)", k), Y.NAMES[fmt]
        # the pixel arithmetic is integer; the one conversion pair is the reciprocal of the row / group division
        assert len(re.findall(r"\bI2F\b", k)) <= 1 and len(re.findall(r"\bF2I\b", k)) <= 1, Y.NAMES[fmt]
        assert not re.search(r"\b(FFMA|FADD|FMUL|DFMA|DADD|DMUL)\b", k), f"{Y.NAMES[fmt]}: integer arithmetic only"
        assert not re.search(r"\b(LDL|STL)\b", k), f"{Y.NAMES[fmt]}: spills"


def test_product_never_uses_the_yuv_reference():
    """tests/yuv_ref.py is test infrastructure, like oracle/: the library's conversion must not lean on it."""
    import os
    import re
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cudavideostream_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                with open(os.path.join(dirpath, f), errors="replace") as fh:
                    assert not re.search(r"\byuv_ref\b", fh.read()), f"{f} refers to the test reference"
