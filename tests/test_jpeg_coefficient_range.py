"""The JPEG decoder's IDCT at the edges of the coefficient range, against OpenCV.

In natural pictures the IDCT output of a block stays within about [-384, 639].  A camera, an encoder with unusual
quantisation tables or a stream built on purpose goes far beyond, and such a stream is still a well-formed baseline JPEG
whose pixels must be OpenCV's.  OpenCV's bundled libjpeg-turbo does not run jidctint.c's int32 C code there: on x86-64 it
runs its SIMD islow IDCT, which computes in 16-bit lanes with saturating packs.  `_reference_idct` states that arithmetic
in exact integers and is checked against cv2.imdecode as a black box; the oracle (oracle/jpeg_oracle.c idct_islow) and
the GPU's k_idct must give its pixels.  The rules, each with a test of its own below:

  1. dequantisation wraps to int16: coef * q mod 2**16;
  2. in both passes, in0+in4, in0-in4, in7+in3 and in5+in1 wrap to int16; every other sum and product is exact;
  3. pass 1 saturates its descaled outputs to int16;
  4. a block whose quantised coefficient rows 1..7 are all zero skips pass 1: every workspace row is the dequantised row 0
     times 4, wrapped to int16 (not saturated);
  5. pass 2's descaled output x becomes min(max(x, -128), 127) + 128: a plain clamp, where jidctint.c's range-limit table
     maps x & 1023 (so a large positive overshoot comes out black there).

The designed streams are golden cases' headers with chosen quantised coefficients, written by tests/util.transcode_huffman:
DC-only sweeps across every boundary of the old range-limit table, one AC coefficient at each zig-zag position at +-1023
and where it crosses the 16-bit and 32-bit limits, pairs, blocks where only one pass leaves its range, dense random blocks
at +-1023 -- on gray, 4:4:4, 4:2:2 and 4:2:0 sources, with their own quantisation tables and with every entry 255."""
import functools
import os

import numpy as np
import pytest

from util import _ZIGZAG, transcode_huffman

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
ZZ = np.array(_ZIGZAG)  # zig-zag index -> natural index
SOURCES = ("q90_gray_123x77", "q85_444_161x97", "q90_422_320x240", "q10_420_128x128", "q100_420_37x29")
# consecutive centred samples DC*q0/8 on either side of each boundary of jidctint.c's range-limit table (x & 1023)
TABLE_BOUNDARIES = ((-897, -896), (-513, -512), (-129, -128), (127, 128), (511, 512), (895, 896))


def _golden(name):
    return np.load(os.path.join(GOLDEN, "jpeg_cases.npz"))[name + "/jpg"].tobytes()


# ---- headers -------------------------------------------------------------------------------------------------------

def _segments(jpg):
    """(marker, payload offset, payload length) of every segment before the scan."""
    i = 2
    while True:
        m, ln = jpg[i + 1], (jpg[i + 2] << 8) | jpg[i + 3]
        yield m, i + 4, ln - 2
        if m == 0xDA:
            return
        i += 2 + ln


def _header(jpg):
    """Geometry and the quantisation table (zig-zag order) of each component."""
    tables, sof = {}, None
    for m, p, n in _segments(jpg):
        if m == 0xDB:
            o = p
            while o < p + n:
                assert jpg[o] >> 4 == 0, "8-bit tables only"
                tables[jpg[o] & 15] = np.frombuffer(jpg, np.uint8, 64, o + 1).astype(np.int64)
                o += 65
        elif m == 0xC0:
            sof = p
    h, w, nc = (jpg[sof + 1] << 8) | jpg[sof + 2], (jpg[sof + 3] << 8) | jpg[sof + 4], jpg[sof + 5]
    hs, vs = (jpg[sof + 7] >> 4, jpg[sof + 7] & 15) if nc == 3 else (1, 1)
    q = [tables[jpg[sof + 8 + 3 * c]] for c in range(nc)]
    bpm = hs * vs + (2 if nc == 3 else 0)
    nmcu = -(-w // (8 * hs)) * -(-h // (8 * vs))
    comp = np.array([0 if nc == 1 or j < hs * vs else j - hs * vs + 1 for j in range(bpm)] * nmcu)
    return dict(w=w, h=h, hs=hs, vs=vs, ncomp=nc, bpm=bpm, q=q, comp=comp)


def _with_q255(jpg):
    """The same stream with every quantisation table entry rewritten to 255."""
    j = bytearray(jpg)
    for m, p, n in _segments(jpg):
        if m == 0xDB:
            for o in range(p, p + n, 65):
                j[o + 1:o + 65] = b"\xff" * 64
    return bytes(j)


def _with_gray_blocks(jpg, nblocks, qzz):
    """A one-component header of nblocks blocks side by side (8*nblocks x 8 pixels) with quantisation table qzz."""
    j = bytearray(jpg)
    for m, p, n in _segments(jpg):
        if m == 0xC0:
            assert j[p + 5] == 1
            j[p + 1:p + 5] = (8).to_bytes(2, "big") + (8 * nblocks).to_bytes(2, "big")
        elif m == 0xDB:
            assert n == 65
            j[p + 1:p + 65] = bytes(int(v) for v in qzz)
    return bytes(j)


def _bound_dc(coef, hd, restart_interval=0):
    """Replaces each block's DC (a target) by the nearest value its component's predictor can reach with a difference of
    at most 2047 (category 11, the largest a baseline DC difference can be), in scan order; prediction restarts from 0 at
    every restart interval."""
    pred = [0, 0, 0]
    for b in range(coef.shape[0]):
        if restart_interval and b % (hd["bpm"] * restart_interval) == 0:
            pred = [0, 0, 0]
        c = hd["comp"][b]
        pred[c] += int(np.clip(int(coef[b, 0]) - pred[c], -2047, 2047))
        coef[b, 0] = pred[c]
    return coef


def _stream(jpg, hd, coef, restart_interval=0):
    return transcode_huffman(jpg, coef, hd["hs"], hd["vs"], hd["ncomp"], 12, 12, restart_interval)


# ---- the reference IDCT --------------------------------------------------------------------------------------------

def _w16(x):
    return ((x + 32768) & 0xFFFF) - 32768


def _pass(v, shift, wrap_sums, wrapped):
    """jpeg_idct_islow's 1-D transform along the last axis of v, descaled by shift, with the products grouped as
    libjpeg-turbo's SIMD code groups them (pmaddwd pairs of jidctint.c's FIX_x constants).  Appends to `wrapped` where one
    of the four 16-bit sums left int16."""
    s04, d04, s73, s51 = v[..., 0] + v[..., 4], v[..., 0] - v[..., 4], v[..., 7] + v[..., 3], v[..., 5] + v[..., 1]
    wrapped.append((s04 != _w16(s04)) | (d04 != _w16(d04)) | (s73 != _w16(s73)) | (s51 != _w16(s51)))
    W = _w16 if wrap_sums else (lambda x: x)
    tmp3 = v[..., 2] * (4433 + 6270) + v[..., 6] * 4433
    tmp2 = v[..., 2] * 4433 + v[..., 6] * (4433 - 15137)
    tmp0, tmp1 = W(s04) * 8192, W(d04) * 8192
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    z3, z4 = W(s73), W(s51)
    Z3, Z4 = z3 * (9633 - 16069) + z4 * 9633, z3 * 9633 + z4 * (9633 - 3196)
    o0 = v[..., 7] * (2446 - 7373) + v[..., 1] * -7373 + Z3
    o3 = v[..., 7] * -7373 + v[..., 1] * (12299 - 7373) + Z4
    o1 = v[..., 5] * (16819 - 20995) + v[..., 3] * -20995 + Z4
    o2 = v[..., 5] * -20995 + v[..., 3] * (25172 - 20995) + Z3
    out = np.stack([t10 + o3, t11 + o2, t12 + o1, t13 + o0, t13 - o0, t12 - o1, t11 - o2, t10 - o3], axis=-1)
    return (out + (1 << (shift - 1))) >> shift


def _reference_idct(coef, qzz, wrap_dequant=True, wrap_sums=True, saturate_pass1=True, skip_pass1=True):
    """Pixels [n, 8, 8] of quantised blocks coef [n, 64] (natural order) under table qzz (zig-zag order), and a trace of
    which rule each block reached.  int64 holds every value exactly (none reaches 2**40), so this is integer arithmetic
    without overflow; the keyword arguments switch one rule off, to show that cv2 needs it."""
    q = np.zeros(64, np.int64)
    q[ZZ] = np.asarray(qzz, np.int64)
    c = np.asarray(coef, np.int64).reshape(-1, 64)
    dq = c * q
    t = {"dequant_wrap": np.any(dq != _w16(dq), axis=1), "skip": ~np.any(c[:, 8:] != 0, axis=1)}
    dq = (_w16(dq) if wrap_dequant else dq).reshape(-1, 8, 8)
    wrapped = []
    p1 = _pass(np.swapaxes(dq, 1, 2), 11, wrap_sums, wrapped)  # [block, column, row]
    t["p1_sat"] = ~t["skip"] & np.any((p1 < -32768) | (p1 > 32767), axis=(1, 2))
    t["p1_wrap"] = ~t["skip"] & np.any(wrapped[0], axis=1)
    if saturate_pass1:
        p1 = np.clip(p1, -32768, 32767)
    if skip_pass1:
        p1 = np.where(t["skip"][:, None, None], _w16(dq[:, 0, :] * 4)[:, :, None], p1)
    x = _pass(np.swapaxes(p1, 1, 2), 18, wrap_sums, wrapped)  # [block, row, column]
    t["p2_wrap"] = np.any(wrapped[1], axis=1)
    t["clamped"] = np.any((x < -128) | (x > 127), axis=(1, 2))
    t["x"] = x
    return (np.clip(x, -128, 127) + 128).astype(np.uint8), t


# ---- designed coefficient sets -------------------------------------------------------------------------------------

def _dc_sweep(q0):
    """DC-only blocks, DC ascending from -32767 to 32767 in steps a DC difference can take: around every table boundary
    of the centred sample DC*q0/8, around the 16-bit limits of DC*q0*4 and DC*q0, and at +-2047 and +-32767."""
    pts = {0, -2047, 2047, -32767, 32767}
    for lo, hi in TABLE_BOUNDARIES:
        pts.update(range(8 * hi // q0 - 2, 8 * hi // q0 + 3))
    for lim in (8192, 32768):
        pts.update(s * (lim // q0 + d) for s in (-1, 1) for d in (-1, 0, 1))
    pts.update(range(-2047, 2048, 89))
    dc = []
    for v in sorted(p for p in pts if abs(p) <= 32767):
        while dc and v - dc[-1] > 2047:
            dc.append(dc[-1] + 2047)
        dc.append(v)
    b = np.zeros((len(dc), 64), np.int64)
    b[:, 0] = dc
    return b


def _edge_values(q):
    """AC values (1..1023) at which coef*q crosses 2**15 (dequantisation wraps) or coef*q*FIX_3_072711026 crosses 2**31
    (jidctint.c's int32 products overflow), and 1023."""
    vals = {1023}
    for lim in (32768, 2 ** 31 / 25172):
        v = int(np.ceil(lim / q))
        vals.update((v - 1, v))
    return sorted(v for v in vals if 1 <= v <= 1023)


def _ac_singles(qzz):
    """One AC coefficient per block: every zig-zag position, both signs, at its edge values."""
    out = []
    for k in range(1, 64):
        for v in _edge_values(int(qzz[k])):
            for s in (-1, 1):
                b = np.zeros(64, np.int64)
                b[ZZ[k]] = s * v
                out.append(b)
    return np.array(out)


def _pairs(qzz, rng, n=96):
    """Two non-zero coefficients (the DC among the candidates) at edge values or random ones."""
    out = np.zeros((n, 64), np.int64)
    for i in range(n):
        for k in rng.choice(64, 2, replace=False):
            e = _edge_values(int(qzz[k]))
            v = int(rng.choice(e)) if rng.random() < 0.5 else int(rng.integers(1, 1024))
            out[i, ZZ[k]] = int(rng.choice((-1, 1))) * v
    return out


def _one_pass_out_of_range(qzz, rng, per_kind=32):
    """Random sparse blocks picked by the reference's trace: pass 1 in range (no saturation, no 16-bit wrap) while pass 2
    clamps; pass 1 saturates while pass 2 stays in range; pass 2 wraps while pass 1 does not saturate; pass 1 saturates
    while pass 2 does not wrap.  Each kind as far as the table admits it."""
    n = 3000
    c = np.zeros((n, 64), np.int64)
    for i in range(n):
        k = int(rng.integers(2, 7))
        c[i, rng.choice(np.arange(1, 64), k, replace=False)] = rng.integers(-1023, 1024, k)
    c[:, 8] = np.where(np.any(c[:, 8:] != 0, axis=1), c[:, 8], 1)  # keep pass 1
    c[:, 0] = rng.integers(-2047, 2048, n)
    _, t = _reference_idct(c, qzz)
    kinds = (~t["p1_sat"] & ~t["p1_wrap"] & ~t["dequant_wrap"] & t["clamped"], t["p1_sat"] & ~t["clamped"],
             ~t["p1_sat"] & t["p2_wrap"], t["p1_sat"] & ~t["p2_wrap"])
    return np.concatenate([c[np.flatnonzero(k)[:per_kind]] for k in kinds])


def _dense(rng, n=48):
    """Every coefficient random in -1023..1023, and every coefficient +-1023."""
    a = rng.integers(-1023, 1024, (n, 64))
    b = 1023 * rng.choice((-1, 1), (n, 64))
    d = np.concatenate([a, b]).astype(np.int64)
    d[:, 0] = rng.integers(-2047, 2048, 2 * n)
    return d


def _design(qzz, seed=0):
    rng = np.random.default_rng(seed)
    return np.concatenate([_dc_sweep(int(qzz[0])), _ac_singles(qzz), _pairs(qzz, rng), _one_pass_out_of_range(qzz, rng),
                           _dense(rng)])


@functools.lru_cache(maxsize=None)
def _designed_streams(name, q255=False, restart_interval=0):
    """The designed sets of each component's table, block by block in the component's places in scan order, as many
    streams of the source's header as they fill.  Returns [(stream, coefficients as written)]."""
    jpg = _golden(name)
    if q255:
        jpg = _with_q255(jpg)
    hd = _header(jpg)
    comp = hd["comp"]
    sets = {c: _design(hd["q"][c], seed=c) for c in range(hd["ncomp"])}
    slots = {c: np.flatnonzero(comp == c) for c in sets}
    nstreams = max(-(-len(sets[c]) // len(slots[c])) for c in sets)
    out = []
    for s in range(nstreams):
        coef = np.zeros((comp.size, 64), np.int64)
        for c, d in sets.items():
            chunk = d[s * len(slots[c]):(s + 1) * len(slots[c])]
            coef[slots[c][:len(chunk)]] = chunk
        _bound_dc(coef, hd, restart_interval)
        out.append((_stream(jpg, hd, coef, restart_interval), coef))
    return hd, out


def _gray_decode(cv2, blocks, qzz):
    """Blocks [n, 64] as an 8*n x 8 gray image with table qzz (DC reached by bounded differences): the coefficients as
    written and cv2's pixels [n, 8, 8]."""
    blocks = np.asarray(blocks, np.int64)
    jpg = _with_gray_blocks(_golden("q90_gray_123x77"), len(blocks), qzz)
    hd = _header(jpg)
    coef = _bound_dc(blocks.copy(), hd)
    img = cv2.imdecode(np.frombuffer(_stream(jpg, hd, coef), np.uint8), cv2.IMREAD_GRAYSCALE)
    assert img is not None and img.shape == (8, 8 * len(blocks))
    return coef, img.reshape(8, -1, 8).transpose(1, 0, 2)


def _table(v):
    return np.full(64, v, np.int64)


# ---- CPU: the reference against cv2, rule by rule ------------------------------------------------------------------

@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


@pytest.mark.parametrize("q", [1, 3, 16, 100, 255])
def test_reference_matches_opencv_on_single_coefficient_8x8_images(cv2, q):
    """One gray 8x8 image per coefficient: the DC sweep (within +-2047, reachable from 0) and every AC position at its
    edge values."""
    jpg = _with_gray_blocks(_golden("q90_gray_123x77"), 1, _table(q))
    hd = _header(jpg)
    blocks = np.concatenate([_dc_sweep(q), _ac_singles(_table(q))])
    blocks = blocks[np.abs(blocks[:, 0]) <= 2047]
    want, _ = _reference_idct(blocks, _table(q))
    for b, w in zip(blocks, want):
        img = cv2.imdecode(np.frombuffer(_stream(jpg, hd, b[None].copy()), np.uint8), cv2.IMREAD_GRAYSCALE)
        assert np.array_equal(img, w), f"q={q}, coefficients {dict((int(i), int(b[i])) for i in np.flatnonzero(b))}"


@pytest.mark.parametrize("q", [3, 50, 255])
def test_reference_matches_opencv_on_pairs_and_sweeps(cv2, q):
    coef, got = _gray_decode(cv2, _design(_table(q), seed=q), _table(q))
    want, _ = _reference_idct(coef, _table(q))
    bad = np.flatnonzero(np.any(got != want, axis=(1, 2)))
    assert bad.size == 0, f"{bad.size} of {len(coef)} blocks differ, first {coef[bad[0]][coef[bad[0]] != 0]}"


def _rule_blocks(cv2, blocks, qzz, **off):
    """cv2 agrees with the reference on blocks, and disagrees with the reference without the rule `off` switches off."""
    coef, got = _gray_decode(cv2, blocks, qzz)
    want, t = _reference_idct(coef, qzz)
    assert np.array_equal(got, want)
    without, _ = _reference_idct(coef, qzz, **off)
    assert not np.array_equal(got, without), f"the blocks do not tell {off} apart"
    return coef, got, t


def test_rule_dequantisation_wraps_to_16_bits(cv2):
    # one coefficient at zig-zag 2 or 9 (natural rows 1 and 3: pass 1 runs) with coef*q up to and past 2**15
    qzz = _table(255)
    b = np.zeros((8, 64), np.int64)
    for i, v in enumerate((128, 129, 1023, -129)):
        b[i, ZZ[2]] = v      # zig-zag 2 is natural 8: row 1
        b[4 + i, ZZ[9]] = v
    _, _, t = _rule_blocks(cv2, b, qzz, wrap_dequant=False)
    assert t["dequant_wrap"][[1, 2, 3, 5, 6, 7]].all()


def test_rule_paired_sums_wrap_to_16_bits(cv2):
    # in0 + in4 of pass 1 past 2**15 in each column, both halves in range: rows 0 and 4 at +-(2**14 + 2**13)
    qzz = _table(32)
    b = np.zeros((4, 64), np.int64)
    b[0, [0, 32]] = 768
    b[1, [1, 33]] = -768
    b[2, [8 + 3, 40 + 3]] = 768   # rows 1 and 5: in5 + in1 of the odd part
    b[3, [24 + 6, 56 + 6]] = -768  # rows 3 and 7: in7 + in3
    b[0, 8] = b[1, 8] = 1
    _, _, t = _rule_blocks(cv2, b, qzz, wrap_sums=False)
    assert t["p1_wrap"].all()


def test_rule_pass_1_saturates_to_16_bits(cv2):
    qzz = _table(255)
    b = np.zeros((3, 64), np.int64)
    b[0, [0, 8, 16, 24]] = 120           # one column, four rows: pass 1 far past 2**15, no 16-bit sum wraps
    b[1, [2, 10, 18]] = -127
    b[2, [0, 8]] = 127
    _, _, t = _rule_blocks(cv2, b, qzz, saturate_pass1=False)
    assert t["p1_sat"].all() and not t["p1_wrap"].any() and not t["dequant_wrap"].any()


def test_rule_blocks_with_zero_rows_skip_pass_1_with_a_wrapping_shift(cv2):
    # row 0 only: dequantised values past 2**13, so that times 4 they wrap -- the full pass 1 would saturate instead
    qzz = _table(255)
    b = np.zeros((4, 64), np.int64)
    b[0, 0] = 40
    b[1, 0] = -100
    b[2, [1, 5]] = (50, -60)
    b[3, [0, 7]] = (33, 64)
    _, _, t = _rule_blocks(cv2, b, qzz, skip_pass1=False)
    assert t["skip"].all()
    # the test for zero rows looks at the quantised coefficients: 512 * 128 = 2**16 dequantises to 0 but keeps pass 1
    q = _table(128)
    b = np.zeros((2, 64), np.int64)
    b[:, 0] = 100
    b[1, 8] = 512
    coef, got = _gray_decode(cv2, b, q)
    assert np.array_equal(got, _reference_idct(coef, q)[0])
    assert not np.array_equal(got[0], got[1]), "a row of zeros after dequantisation still runs pass 1"


def test_rule_output_is_clamped_then_centred(cv2):
    """Rule 5 on the DC sweep: clamp(x, -128, 127) + 128, where jidctint.c's table maps x & 1023 (0..127 -> 128+i,
    128..511 -> 255, 512..895 -> 0, 896..1023 -> i-896)."""
    qzz = _table(16)
    coef, got = _gray_decode(cv2, _dc_sweep(16), qzz)
    want, t = _reference_idct(coef, qzz)
    assert np.array_equal(got, want)
    i = np.asarray(t["x"]) & 1023
    table = np.where(i < 128, 128 + i, np.where(i < 512, 255, np.where(i < 896, 0, i - 896)))
    assert np.any(table != got), "the sweep must reach the samples where the table and the clamp disagree"
    s = t["x"][:, 0, 0]
    for lo, hi in TABLE_BOUNDARIES:
        assert np.any((s[:-1] <= lo) & (s[1:] >= hi)), f"the sweep does not cross {lo}/{hi}"


# ---- CPU: the oracle -----------------------------------------------------------------------------------------------

def test_designed_sets_reach_every_rule():
    """The designed streams are not vacuous: across the sources they reach every rule and both one-pass-only kinds."""
    seen = {k: 0 for k in ("dequant_wrap", "skip", "p1_sat", "p1_wrap", "p2_wrap", "clamped", "p1_in_range_p2_clamped",
                           "p1_sat_p2_in_range")}
    for name in SOURCES:
        for q255 in (False, True):
            hd, streams = _designed_streams(name, q255)
            for _, coef in streams:
                for c in range(hd["ncomp"]):
                    _, t = _reference_idct(coef[hd["comp"] == c], hd["q"][c])
                    for k in ("dequant_wrap", "skip", "p1_sat", "p1_wrap", "p2_wrap", "clamped"):
                        seen[k] += int(t[k].sum())
                    seen["p1_in_range_p2_clamped"] += int((~t["skip"] & ~t["p1_sat"] & ~t["p1_wrap"] & t["clamped"]).sum())
                    seen["p1_sat_p2_in_range"] += int((t["p1_sat"] & ~t["clamped"]).sum())
    assert all(v >= 20 for v in seen.values()), seen


def test_oracle_matches_the_reference_on_gray_streams(oracle):
    for q255 in (False, True):
        hd, streams = _designed_streams("q90_gray_123x77", q255)
        for s, (jpg, coef) in enumerate(streams):
            want, _ = _reference_idct(coef, hd["q"][0])
            nbx = -(-hd["w"] // 8)
            plane = want.reshape(-1, nbx, 8, 8).transpose(0, 2, 1, 3).reshape(-1, nbx * 8)[:hd["h"], :hd["w"]]
            got = oracle.jpeg_decode_bgr(jpg)
            assert np.array_equal(got[:, :, 0], plane) and np.array_equal(got[:, :, 2], plane), f"q255={q255} stream {s}"


@pytest.mark.parametrize("q255", [False, True], ids=["own_tables", "q255"])
@pytest.mark.parametrize("name", SOURCES)
def test_oracle_matches_opencv_on_designed_streams(oracle, cv2, name, q255):
    _, streams = _designed_streams(name, q255)
    for s, (jpg, _) in enumerate(streams):
        ref = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_COLOR)
        got = oracle.jpeg_decode_bgr(jpg)
        bad = np.flatnonzero(got.reshape(-1) != ref.reshape(-1))
        assert bad.size == 0, f"stream {s}: {bad.size} of {ref.size} bytes differ"


@pytest.mark.parametrize("name,interval", [("q90_gray_123x77", 1), ("q85_444_161x97", 5), ("q10_420_128x128", 3)])
def test_oracle_matches_opencv_with_restart_intervals(oracle, cv2, name, interval):
    _, streams = _designed_streams(name, True, interval)
    for s, (jpg, _) in enumerate(streams):
        assert b"\xff\xdd" in jpg[:400]
        ref = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_COLOR)
        assert np.array_equal(oracle.jpeg_decode_bgr(jpg), ref), f"stream {s}"


# ---- GPU: k_idct -----------------------------------------------------------------------------------------------------

@pytest.fixture
def own_decoder(monkeypatch):
    monkeypatch.setenv("CVS_JPEG_DECODER", "own")


def _gpu_vs_opencv_and_oracle(cvs, oracle, cv2, streams, hd, label):
    from test_jpeg_ingest import _decode  # checks the guard band behind the frame
    for s, (jpg, _) in enumerate(streams):
        ref = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_COLOR).reshape(-1)
        assert np.array_equal(oracle.jpeg_decode_bgr(jpg).reshape(-1), ref), f"{label} stream {s}: oracle vs cv2"
        g = _decode(cvs, jpg, hd["w"], hd["h"])
        bad = np.flatnonzero(g != ref)
        assert bad.size == 0, f"{label} stream {s}: {bad.size} of {ref.size} bytes differ from cv2, first at {bad[:5]}"


@pytest.mark.gpu
@pytest.mark.parametrize("q255", [False, True], ids=["own_tables", "q255"])
@pytest.mark.parametrize("name", SOURCES)
def test_gpu_decodes_designed_streams_like_opencv(cvs, oracle, cv2, own_decoder, name, q255):
    hd, streams = _designed_streams(name, q255)
    _gpu_vs_opencv_and_oracle(cvs, oracle, cv2, streams, hd, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name,interval", [("q90_gray_123x77", 1), ("q85_444_161x97", 5), ("q10_420_128x128", 3)])
def test_gpu_restart_interval_streams_like_opencv(cvs, oracle, cv2, own_decoder, name, interval):
    """Restart intervals send the stream through k_entropy_restart; the IDCT's range must not depend on it."""
    hd, streams = _designed_streams(name, True, interval)
    _gpu_vs_opencv_and_oracle(cvs, oracle, cv2, streams, hd, f"{name} interval {interval}")


@pytest.mark.gpu
def test_submit_jpeg_camera_frame_with_sweep_blocks(cvs, oracle, cv2, own_decoder):
    """The reference's camera frame with every fourth MCU replaced by designed blocks, through cvs_submit_jpeg: the
    payload is the oracle's diff of the oracle's pixels, and those are cv2's."""
    import ctypes as C
    with open(os.path.join(GOLDEN, "k1_f1.jpg"), "rb") as f:
        j1 = f.read()
    hd = _header(j1)
    coef = oracle.jpeg_coefficients(j1).astype(np.int64)
    mixed = np.flatnonzero((np.arange(coef.shape[0]) // hd["bpm"]) % 4 == 1)
    for c in range(hd["ncomp"]):
        d = _design(hd["q"][c], seed=c)
        at = mixed[hd["comp"][mixed] == c]
        coef[at] = d[np.arange(len(at)) % len(d)]
    j2 = _stream(j1, hd, _bound_dc(coef, hd))
    w, h, n = hd["w"], hd["h"], 3 * hd["w"] * hd["h"]
    g1, g2 = oracle.jpeg_decode_bgr(j1).reshape(-1), oracle.jpeg_decode_bgr(j2).reshape(-1)
    assert np.array_equal(g2, cv2.imdecode(np.frombuffer(j2, np.uint8), cv2.IMREAD_COLOR).reshape(-1))
    s = cvs.Stream(w, h, g1)
    dout, xout, pb = cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()
    oref = g1
    try:
        for cur, j in ((g2, j2), (g1, j1), (g2, j2)):
            jb = cvs.alloc_host(len(j) + 64)
            jb.array()[:len(j)] = np.frombuffer(j, dtype=np.uint8)
            s.wait(s.submit_jpeg_raw(jb.ptr, len(j), dout.ptr, None, "", C.addressof(pb), xout.ptr))
            opos, oxs, odiff, oref, _ = oracle.diff_compact(cur, oref, 20)
            assert opos > 0 and pb[0] == opos
            assert np.array_equal(dout.array()[:opos], odiff) and np.array_equal(xout.array(np.int32)[:opos], oxs)
            assert np.array_equal(s.reference(), oref)
    finally:
        s.close()
