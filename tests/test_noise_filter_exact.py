"""The noise filter, bit for bit, on every kernel variant launch_conv picks and at the edges where they go wrong.

The expected bytes come from an independent numpy model of what the filter promises (include/cvs_b200.h): per output
byte, fp32 accumulation with one correctly rounded fused multiply-add per tap in row-major tap order over a zero-padded
frame, then (uint8_t)acc as x86-64 converts it (cvttss2si: 0x80000000 for NaN and anything outside [-2^31, 2^31), then
the low byte).  The model is checked against the C oracle on the CPU, and the library against the model on the GPU.

The weights reach both sides of every choice launch_conv makes: non-negative with a float sum <= 16384 (the FADD.RZ
truncation) or not (F2I), accumulators that wrap below 0 and above 255, at and above 2^31, NaN and +inf, and a set
whose result depends on the order of the taps."""
import functools

import numpy as np
import pytest

# ------------------------------------------------------------------------------------------------
# the model
# ------------------------------------------------------------------------------------------------


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _rn32(s, e):
    """fp32 rounding (to nearest, ties to even) of the exact sum s + e, where s = fl64(a + b) and e is its error."""
    f = s.astype(np.float32)
    fd = f.astype(np.float64)
    # np.float32(s) rounds s, not s + e: the two differ only when s is a float32 midpoint and e != 0
    g = np.nextafter(f, np.where(s > fd, np.float32(np.inf), np.float32(-np.inf)))
    tie = np.isfinite(s) & (fd != s) & (s == (fd + g.astype(np.float64)) * 0.5) & (e != 0)
    if tie.any():
        f = np.where(tie, np.where(e > 0, np.maximum(f, g), np.minimum(f, g)), f)
    return f


def _cvtt_byte(acc):
    a = acc.astype(np.float64)
    ok = (a >= -2.0 ** 31) & (a < 2.0 ** 31)  # False for NaN
    v = np.where(ok, np.trunc(np.where(ok, a, 0.0)), -2.0 ** 31).astype(np.int64)
    return (v & 0xFF).astype(np.uint8)


def _padded_taps(image, width, height, K, k, order):
    """(weight, shifted zero-padded frame) per tap, in the given tap order ("row" or "col")."""
    R = K // 2
    pad = np.zeros((height + 2 * R, width + 2 * R, 3), dtype=np.float64)
    pad[R:R + height, R:R + width] = np.asarray(image, dtype=np.uint8).reshape(height, width, 3)
    k = np.asarray(k, dtype=np.float32).reshape(K, K)
    taps = [(i, j) for i in range(K) for j in range(K)]
    if order == "col":
        taps = [(i, j) for j in range(K) for i in range(K)]
    for i, j in taps:
        yield np.float64(k[i, j]), pad[i:i + height, j:j + width]


def noise_filter_model(image, width, height, K, k, order="row"):
    """acc = RN32(k * p + acc) per tap (k * p is exact in float64: 24 x 8 bits), then the cvttss2si byte."""
    acc = np.zeros((height, width, 3), dtype=np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for kw, p in _padded_taps(image, width, height, K, k, order):
            s, e = _two_sum(kw * p, acc.astype(np.float64))
            acc = _rn32(s, e)
    return _cvtt_byte(acc).reshape(-1)


def noise_filter_f64(image, width, height, K, k):
    """The same taps summed in float64 and rounded once: what a filter that ignores the fp32 order would give."""
    acc = np.zeros((height, width, 3), dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        for kw, p in _padded_taps(image, width, height, K, k, "row"):
            acc = acc + kw * p
        return _cvtt_byte(acc.astype(np.float32)).reshape(-1)


def _f32_sum(k):
    s = np.float32(0.0)
    with np.errstate(over="ignore", invalid="ignore"):
        for v in np.asarray(k, dtype=np.float32):
            s = np.float32(s + v)
    return s


def conv_variant(width, K, k, in_stride, out_stride):
    """The kernel launch_conv (cvs_api.cu) runs for these arguments (16-byte aligned buffers)."""
    rowbytes = 3 * width
    fast = rowbytes % 4 == 0 and in_stride % 4 == 0 and out_stride % 4 == 0 and K in (1, 3, 5)
    if fast and K in (3, 5):
        k = np.asarray(k, dtype=np.float32)
        nonneg = bool(np.all(k >= 0)) and bool(_f32_sum(k) <= 16384)
        wide = K == 3 and rowbytes % 8 == 0 and in_stride % 8 == 0 and out_stride % 8 == 0
        return "k_conv_strip<%d,%s,%d>" % (K, "true" if nonneg else "false", 2 if wide else 1)
    return "k_conv_rows4<1>" if fast else "k_conv_bytes"


ALL_VARIANTS = {"k_conv_strip<3,true,2>", "k_conv_strip<3,false,2>", "k_conv_strip<3,true,1>", "k_conv_strip<3,false,1>",
                "k_conv_strip<5,true,1>", "k_conv_strip<5,false,1>", "k_conv_rows4<1>", "k_conv_bytes"}

# ------------------------------------------------------------------------------------------------
# weights: name -> K -> float32[K*K]
# ------------------------------------------------------------------------------------------------


def _gauss(K):
    c = (K - 1) / 2.0
    y, x = np.mgrid[0:K, 0:K] - c
    g = np.exp(-(x * x + y * y) / (2.0 * (K * K / 6.0) ** 2))
    return (g / g.sum()).astype(np.float32).reshape(-1)


def _sum16384(K):
    """Positive weights whose float sum, taken in order as launch_conv takes it, is exactly 16384."""
    rng = np.random.default_rng(40 + K)
    u = rng.uniform(0.5, 1.5, K * K)
    k = (u / u.sum() * 16384.0).astype(np.float32)
    head = _f32_sum(k[:-1])
    k[-1] = np.float32(16384.0) - head
    while _f32_sum(k) > 16384:
        k[-1] = np.nextafter(k[-1], np.float32(0))
    while _f32_sum(k) < 16384:
        k[-1] = np.nextafter(k[-1], np.float32(np.inf))
    assert _f32_sum(k) == 16384 and np.all(k > 0)
    return k


def _over16384(K):
    """The same weights with the last one nudged until the float sum is just above 16384."""
    k = _sum16384(K)
    while _f32_sum(k) <= 16384:
        k[-1] = np.nextafter(k[-1], np.float32(np.inf))
    return k


def _inf(K):
    k = _gauss(K)
    k[0] = np.inf  # top-left tap: inf * 0 = NaN at zero pixels and in the padding, +inf elsewhere
    return k


def _order(K):
    # +-1e4 next to 1.0001 and 0.3: the fp32 accumulator is rounded at a different magnitude after every tap, so
    # another tap order (or a float64 sum) changes some bytes -- shown by test_order_fixture_detects_reordering
    t = np.arange(K * K)
    return np.where(t % 3 == 0, np.where((t // 3) % 2 == 0, 1e4, -1e4), np.where(t % 3 == 1, 1.0001, 0.3)).astype(np.float32)


WEIGHTS = {
    "gauss": _gauss,                                                                  # NONNEG
    "mean": lambda K: np.full(K * K, 1.0 / (K * K), dtype=np.float32),               # NONNEG (the K2 answer's filter)
    "sharpen": lambda K: np.where(np.arange(K * K) == K * K // 2, K * K, -1.0).astype(np.float32),  # !NONNEG, wraps both ways
    "random": lambda K: np.random.default_rng(K).uniform(-2.0, 2.0, K * K).astype(np.float32),       # !NONNEG
    "sum16384": _sum16384,                                                            # NONNEG, accumulators up to 4.2 M
    "over16384": _over16384,                                                          # !NONNEG
    "big": lambda K: np.full(K * K, 1e7, dtype=np.float32),                          # !NONNEG, accumulators >= 2^31
    "inf": _inf,                                                                      # !NONNEG, +inf and NaN
    "order": _order,                                                                  # !NONNEG, tap-order sensitive
}

# (width, height, K): every variant, its x tail (W = 344 and 684: the last x-block holds one thread), its row tail
# (H % 8 in {0, 1, 7}), frames lower (H < K) and narrower (W < K) than the filter
SHAPES = [
    (64, 8, 3), (64, 9, 3), (344, 7, 3), (344, 17, 3),   # K = 3, W % 8 == 0: two words per thread
    (68, 16, 3), (684, 9, 3), (684, 7, 3),               # K = 3, W % 8 == 4: one word per thread
    (64, 1, 3), (64, 2, 3), (68, 2, 3),                  # H < K
    (37, 9, 3), (250, 7, 3), (1, 5, 3), (2, 3, 3),       # W % 4 != 0: the byte kernel (W < K included)
    (64, 16, 5), (100, 15, 5), (44, 17, 5),              # K = 5, W % 4 == 0
    (64, 1, 5), (8, 2, 5), (4, 9, 5), (4, 4, 5),         # H < K, W < K on the strip kernel
    (37, 9, 5), (2, 7, 5),                               # K = 5 byte kernel
    (64, 9, 1), (37, 7, 1),                              # K = 1: one-row kernel / byte kernel
    (64, 9, 7), (5, 3, 7), (40, 17, 9), (3, 2, 9),       # K = 7, 9: byte kernel
]
FULL_SIZE = [(1920, 1080, 3, "random"), (1920, 1080, 5, "random")]  # mixed-sign weights at full size

CASES = [(w, h, K, name) for (w, h, K) in SHAPES for name in WEIGHTS] + FULL_SIZE


def _case_id(c):
    w, h, K, name = c
    return f"{w}x{h}-K{K}-{name}"


def frame(width, height, seed):
    """Random bytes with zero runs (inf * 0 inside the frame) and saturated bytes."""
    rng = np.random.default_rng(seed)
    n = 3 * width * height
    f = rng.integers(0, 256, size=n, dtype=np.uint8)
    f[rng.random(n) < 0.1] = 0
    f[rng.random(n) < 0.05] = 255
    return f


@functools.lru_cache(maxsize=None)
def _expected(width, height, K, name):
    img = frame(width, height, width * 131 + height * 7 + K)
    return img, WEIGHTS[name](K), noise_filter_model(img, width, height, K, WEIGHTS[name](K))


# ------------------------------------------------------------------------------------------------
# CPU: the model, the oracle and the fixtures themselves
# ------------------------------------------------------------------------------------------------


def test_model_reproduces_the_k2_known_answer():
    # REPORT/report.tex:2351-2378 (also pinned for the oracle in test_oracle_kat.py): 3x3 mean filter on matrix A
    A = np.array([[120, 131, 112], [112, 101, 82], [44, 106, 65]], dtype=np.uint8)
    img = np.repeat(A.reshape(3, 3, 1), 3, axis=2)
    got = noise_filter_model(img, 3, 3, 3, WEIGHTS["mean"](3)).reshape(3, 3, 3)
    for ch in range(3):
        assert np.array_equal(got[:, :, ch], [[51, 73, 47], [68, 96, 66], [40, 56, 39]])


def test_model_rounding_and_conversion_corners():
    # a float32 midpoint reached by float64 rounding: 2^24 + 1 is a tie, 2^24 + 1 + 2^-30 is not
    s, e = _two_sum(np.array([2.0 ** 24]), np.array([1.0 + 2.0 ** -30]))
    assert e[0] != 0 and _rn32(s, e)[0] == np.float32(2.0 ** 24 + 2)
    s, e = _two_sum(np.array([2.0 ** 24]), np.array([1.0]))
    assert _rn32(s, e)[0] == np.float32(2.0 ** 24)  # exact tie: to even
    acc = np.array([-1.5, 255.9, 256.0, -256.5, 2.0 ** 31 - 128, 2.0 ** 31, -2.0 ** 31, -2.0 ** 32, np.inf, -np.inf, np.nan],
                   dtype=np.float32)
    assert _cvtt_byte(acc).tolist() == [0xFF, 0xFF, 0x00, 0x00, 0x80, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00]


def test_fixtures_reach_every_kernel_variant():
    seen = {}
    for w, h, K, name in CASES:
        n = 3 * w * h
        seen.setdefault(conv_variant(w, K, WEIGHTS[name](K), n, n), []).append((w, h, K, name))
    assert set(seen) == ALL_VARIANTS, set(seen) ^ ALL_VARIANTS
    # the weights take the branch their comment names
    for K in (3, 5):
        for name in WEIGHTS:
            want = name in ("gauss", "mean", "sum16384")
            assert ("true" in conv_variant(64, K, WEIGHTS[name](K), 3 * 64, 3 * 64)) == want, (K, name)


def test_fixtures_leave_the_byte_range():
    # the accumulators really leave [0, 255] the way each fixture says (so the conversion is what is tested)
    img = frame(64, 9, 1)
    for name, want in (("sharpen", (-1, 256)), ("random", (-1, 256)), ("sum16384", (None, 2 ** 21)),
                       ("big", (None, 2 ** 31)), ("order", (-2 ** 20, 2 ** 20))):
        acc = sum(kw * p for kw, p in _padded_taps(img, 64, 9, 3, WEIGHTS[name](3), "row"))
        lo, hi = want
        assert lo is None or acc.min() <= lo, name
        assert acc.max() >= hi, name
    with np.errstate(invalid="ignore"):
        out = noise_filter_model(img, 64, 9, 3, WEIGHTS["inf"](3))
        acc = sum(kw * p for kw, p in _padded_taps(img, 64, 9, 3, WEIGHTS["inf"](3), "row"))
    assert np.isnan(acc).any() and np.isposinf(acc).any() and not out.any()


@pytest.mark.parametrize("K", [3, 5, 7, 9])
def test_order_fixture_detects_reordering(K):
    w, h = 40, 9
    img = frame(w, h, 77 + K)
    k = WEIGHTS["order"](K)
    row = noise_filter_model(img, w, h, K, k)
    assert np.count_nonzero(row != noise_filter_model(img, w, h, K, k, order="col")) > 0
    assert np.count_nonzero(row != noise_filter_f64(img, w, h, K, k)) > 0


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_model_matches_oracle(oracle, case):
    w, h, K, name = case
    img, k, want = _expected(w, h, K, name)
    assert np.array_equal(oracle.noise_filter(img, w, h, K, k), want)


@pytest.mark.parametrize("ksize", [-1, 0, 2, 4, 10, 11, None])
def test_create_rejects_bad_filter_arguments(cvs, ksize):
    # checked before the library looks for a device: runs wherever the library loads
    base = np.zeros(3 * 16 * 16, dtype=np.uint8)
    kw = dict(ksize=3, kweights=None) if ksize is None else dict(ksize=ksize, kweights=np.ones(121, dtype=np.float32))
    with pytest.raises(cvs.CVSError) as e:
        cvs.Stream(16, 16, base, noise_filter=True, **kw)
    assert e.value.status == 1  # CVS_ERR_INVALID


# ------------------------------------------------------------------------------------------------
# GPU: the three entry points against the model and the oracle
# ------------------------------------------------------------------------------------------------
G = 4096


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_standalone_filter_matches_model(cvs, case):
    import torch
    w, h, K, name = case
    img, k, want = _expected(w, h, K, name)
    n = img.size
    d_in = torch.from_numpy(img).cuda()
    raw = torch.full((n + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
    d_out = raw[G:G + n]
    cvs.filters.noise_filter(d_in.data_ptr(), d_out.data_ptr(), w, h, K, k, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, (f"{conv_variant(w, K, k, n, n)}: {bad.size} bytes differ, first at {bad[0]}: "
                           f"0x{got[bad[0]]:02x}, expected 0x{want[bad[0]]:02x}")
    assert bool((raw[:G] == 0xA5).all()) and bool((raw[G + n:] == 0xA5).all()), "write outside out[0, N)"
    assert np.array_equal(d_in.cpu().numpy(), img), "the input frame was modified"


@pytest.mark.gpu
def test_standalone_filter_rejects_bad_arguments(cvs):
    import torch
    w, h = 16, 8
    d_in = torch.zeros(3 * w * h, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(3 * w * h, dtype=torch.uint8, device="cuda")
    k = np.ones(121, dtype=np.float32)
    for ksize in (-1, 0, 2, 4, 10, 11):
        with pytest.raises(cvs.CVSError) as e:
            cvs.filters.noise_filter(d_in.data_ptr(), d_out.data_ptr(), w, h, ksize, k)
        assert e.value.status == 1, ksize
    lib = cvs.load_library()
    assert lib.cvs_noise_filter_device(d_in.data_ptr(), d_out.data_ptr(), w, h, 3, None, None) == 1  # NULL weights
    with pytest.raises(cvs.CVSError) as e:
        cvs.filters.noise_filter(d_in.data_ptr(), d_in.data_ptr(), w, h, 3, k)  # in place
    assert e.value.status == 1
    torch.cuda.synchronize()
    assert not bool(d_out.any()) and not bool(d_in.any())


# the pipeline entry points: one shape per variant, weights that leave the byte range
PIPE_CASES = [(64, 9, 3, "sharpen"), (68, 7, 3, "big"), (684, 9, 3, "inf"), (64, 16, 5, "order"), (44, 17, 5, "over16384"),
              (37, 9, 3, "random"), (64, 9, 1, "big"), (40, 17, 9, "sharpen"), (64, 8, 3, "sum16384")]


def _pipe_frames(w, h, nframes, seed):
    return [frame(w, h, seed + t) for t in range(nframes)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PIPE_CASES, ids=_case_id)
def test_drop_in_exec_with_filter(cvs, oracle, case):
    # cvs_exec, binarising display mode: payload, binarised frame and reference against OracleCore; the payload of the
    # first frame also against the model's filtered frame
    w, h, K, name = case
    k = WEIGHTS[name](K)
    frames = _pipe_frames(w, h, 3, 500 + w + K)
    base = frame(w, h, 499)
    s = cvs.Stream(w, h, base, mode=5, noise_filter=True, ksize=K, kweights=k)
    oc = oracle.OracleCore(w, h, base, mode=5, noise_filter=1, K=K, k=k)
    for t, f in enumerate(frames):
        pos, xs, diff, show = s.exec(f)
        opos, oxs, odiff, oshow, _ = oc.exec_core(f)
        if t == 0:
            filt = noise_filter_model(f, w, h, K, k).astype(np.int64)
            want = np.flatnonzero(np.abs(filt - base) > 20)
            assert np.array_equal(oxs, want) and np.array_equal(odiff, (filt - base)[want].astype(np.uint8))
        assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff), f"frame {t}"
        assert np.array_equal(show, oshow), f"frame {t}: binarised frame"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", PIPE_CASES, ids=_case_id)
def test_sequence_with_filter_in_pieces(cvs, oracle, case):
    # a device sequence longer than max_sequence (pieces of 2 frames: the filter runs with gridDim.z = 2 and 1) whose
    # frames sit 48 bytes further apart than a 16-byte rounded frame (input stride != N)
    import torch
    w, h, K, name = case
    k = WEIGHTS[name](K)
    nframes, n = 5, 3 * w * h
    stride = (n + 15) // 16 * 16 + 48
    frames = _pipe_frames(w, h, nframes, 700 + w + K)
    base = frame(w, h, 699)
    d_frames = torch.zeros(nframes * stride, dtype=torch.uint8, device="cuda")
    for t in range(nframes):
        d_frames[t * stride:t * stride + n] = torch.from_numpy(frames[t]).cuda()
    cap = (n + 3) // 4 * 4
    d_pos = torch.zeros(nframes, dtype=torch.int32, device="cuda")
    d_xs = torch.empty(nframes * cap, dtype=torch.int32, device="cuda")
    d_diff = torch.empty(nframes * cap, dtype=torch.uint8, device="cuda")
    s = cvs.Stream(w, h, base, noise_filter=True, ksize=K, kweights=k, max_sequence=2)
    s.run_sequence_device(d_frames.data_ptr(), stride, nframes, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(), cap,
                          cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s.sequence_status()
    oc = oracle.OracleCore(w, h, base, noise_filter=1, K=K, k=k)
    pos = d_pos.cpu().numpy()
    for t in range(nframes):
        opos, oxs, odiff, _, _ = oc.exec_core(frames[t])
        assert pos[t] == opos, f"frame {t}"
        assert np.array_equal(d_xs[t * cap:t * cap + opos].cpu().numpy(), oxs), f"frame {t}"
        assert np.array_equal(d_diff[t * cap:t * cap + opos].cpu().numpy(), odiff), f"frame {t}"
        assert np.array_equal(d_frames[t * stride:t * stride + n].cpu().numpy(), frames[t]), "input modified"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()
