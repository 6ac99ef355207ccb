"""The Bayer demosaic's reference (tests/bayer_ref.py) is cv2.cvtColor's COLOR_Bayer<P>2BGR for all four patterns, on
random and 0/255 frames from 1x1 to 3840x2160 and on non-contiguous sources; the device entry's argument checks need no
device; the kernel is integer-only with wide accesses.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

import bayer_ref as B

# (H, W): the degenerate sizes OpenCV zeroes, the smallest interiors, widths around one 16-pixel group, camera sizes and
# their odd neighbours
SIZES = [(1, 1), (1, 8), (2, 2), (2, 9), (9, 2), (3, 1), (3, 3), (4, 5), (6, 16), (6, 17), (6, 18),
         (1079, 1919), (1080, 1920), (1081, 1921), (2160, 3840)]


def _frames(h, w, seed):
    rng = np.random.default_rng(seed)
    return {"random": rng.integers(0, 256, (h, w), dtype=np.uint8),
            "0/255": rng.integers(0, 2, (h, w), dtype=np.uint8) * np.uint8(255)}


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
@pytest.mark.parametrize("h,w", SIZES)
def test_reference_matches_cv2(pattern, h, w):
    cv2 = pytest.importorskip("cv2")
    for kind, raw in _frames(h, w, h * 7919 + w * 31 + pattern).items():
        want = B.cv2_demosaic(cv2, pattern, raw)
        got = B.bayer_to_bgr(pattern, raw)
        bad = np.argwhere((got != want).any(axis=2))
        assert bad.size == 0, f"{kind}: {len(bad)} pixels differ from cv2, first at {bad[:5].tolist()}"


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
def test_reference_matches_cv2_on_a_non_contiguous_source(pattern):
    """A mosaic cut out of a wider buffer (rows farther apart than the width): both sides read it through its strides."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(pattern)
    big = rng.integers(0, 256, (1090, 1950), dtype=np.uint8)
    raw = big[3:1083, 7:1927]
    assert not raw.flags.c_contiguous
    assert np.array_equal(B.bayer_to_bgr(pattern, raw), B.cv2_demosaic(cv2, pattern, raw))
    assert np.array_equal(B.bayer_to_bgr(pattern, raw), B.bayer_to_bgr(pattern, np.ascontiguousarray(raw)))


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
def test_flat_white_stays_white_and_tiny_frames_are_black(pattern):
    assert np.all(B.bayer_to_bgr(pattern, np.full((7, 9), 255, np.uint8)) == 255)
    assert np.all(B.bayer_to_bgr(pattern, np.full((1080, 1920), 255, np.uint8)) == 255)
    for h, w in [(1, 1), (2, 2), (2, 9), (9, 2), (1, 100), (100, 1), (2, 1920)]:
        assert np.all(B.bayer_to_bgr(pattern, np.full((h, w), 200, np.uint8)) == 0), (h, w)


def test_legacy_two_letter_names_are_shifted():
    """OpenCV's two-letter codes name the second row's middle, not the sensor's top-left 2x2: BG is RGGB, RG is BGGR,
    GB is GRBG, GR is GBRG.  The library, its tests and its documents use the four-letter (V4L2-order) names only."""
    cv2 = pytest.importorskip("cv2")
    assert cv2.COLOR_BayerBG2BGR == cv2.COLOR_BayerRGGB2BGR == 46
    assert cv2.COLOR_BayerGB2BGR == cv2.COLOR_BayerGRBG2BGR == 47
    assert cv2.COLOR_BayerRG2BGR == cv2.COLOR_BayerBGGR2BGR == 48
    assert cv2.COLOR_BayerGR2BGR == cv2.COLOR_BayerGBRG2BGR == 49


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
def test_mosaic_samples_the_pattern(pattern):
    """mosaic() keeps the channel the sensor's filter passes: a flat-colour frame gives the pattern's 2x2 in V4L2 order."""
    bgr = np.zeros((4, 6, 3), np.uint8)
    bgr[:, :] = (10, 20, 30)  # B G R
    m = B.mosaic(bgr, pattern)
    order = {B.BGGR: "BGGR", B.GBRG: "GBRG", B.GRBG: "GRBG", B.RGGB: "RGGB"}[pattern]
    val = {"B": 10, "G": 20, "R": 30}
    assert [int(v) for v in m[:2, :2].reshape(-1)] == [val[c] for c in order]
    assert np.array_equal(m[2:, :], m[:2, :]) and np.array_equal(m[:, 2:4], m[:, :2])


def test_device_demosaic_refuses_bad_arguments_without_a_device(cvs):
    """cvs_bayer_to_bgr_device checks its arguments before it looks for a device: unknown pattern, size not positive,
    NULL pointers or a pitch below the width -> CVS_ERR_INVALID; d_raw, pitch or d_out not 16-byte aligned ->
    CVS_ERR_ALIGN."""
    lib = cvs.load_library()
    a = 1 << 20  # any 16-byte aligned address: a refusal touches nothing

    def call(pattern=B.BGGR, raw=a, pitch=64, out=a, w=64, h=32):
        return lib.cvs_bayer_to_bgr_device(pattern, raw, pitch, out, w, h, None)

    for bad in (0, 5, -1):
        assert call(pattern=bad) == 1
    for w, h in [(0, 32), (64, 0), (-16, 32)]:
        assert call(w=w, h=h) == 1
    assert call(raw=None) == 1 and call(out=None) == 1
    assert call(pitch=48) == 1 and call(pitch=63, w=64) == 1
    assert call(raw=a + 1) == 4 and call(raw=a + 8) == 4
    assert call(pitch=72) == 4 and call(w=65, pitch=65) == 4
    assert call(out=a + 4) == 4


def test_submit_refuses_bad_arguments_without_a_device(cvs):
    """A NULL handle is refused by both submit forms before anything else is looked at."""
    lib = cvs.load_library()
    tk = C.c_uint64(7)
    a = 1 << 20
    assert lib.cvs_submit_bayer(None, B.BGGR, a, a, None, b"", a, a, C.byref(tk)) == 1
    assert lib.cvs_submit_bayer_wire(None, B.RGGB, a, a, None, b"", C.byref(tk)) == 1
    assert tk.value == 7


def test_demosaic_kernel_is_integer_only_with_wide_accesses(cvs):
    """k_bayer_to_bgr in the built library: 16-byte loads and three 16-byte stores on its fast path, no floating-point
    arithmetic, nothing in local memory."""
    import re
    import shutil
    import subprocess
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        sass = subprocess.run([tool, "-sass", cvs.library_path()], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError) as e:
        pytest.skip(f"cuobjdump unavailable: {e}")
    blocks = re.split(r"(?=\n\s*Function : )", sass)
    hit = [b for b in blocks if re.search(r"Function : \S*k_bayer_to_bgr", b)]
    assert len(hit) == 1, "k_bayer_to_bgr missing from the library"
    k = hit[0]
    assert len(re.findall(r"\bSTG\.E\.128\b", k)) == 3
    assert len(re.findall(r"\bLDG\.E\.128\.CONSTANT\b|\bLDG\.E\.128\b", k)) == 3
    # the pixel arithmetic is integer; the one conversion pair is the reciprocal of the row / group division
    assert len(re.findall(r"\bI2F\b", k)) <= 1 and len(re.findall(r"\bF2I\b", k)) <= 1
    assert not re.search(r"\b(FFMA|FADD|FMUL|DFMA|DADD|DMUL)\b", k), "integer arithmetic only"
    assert not re.search(r"\b(LDL|STL)\b", k), "spills"


def test_product_never_uses_the_bayer_reference():
    """tests/bayer_ref.py is test infrastructure, like oracle/: the library's demosaic must not lean on it."""
    import os
    import re
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cudavideostream_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                with open(os.path.join(dirpath, f), errors="replace") as fh:
                    assert not re.search(r"\bbayer_ref\b", fh.read()), f"{f} refers to the test reference"
