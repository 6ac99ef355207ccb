"""Every stream-kernel variant against the CPU oracle, on frames that sit on the edges of the byte compare.

The hot path is compiled into 48 functions: k_stream<MODE, HI> (frames walked in several segments, the reference
through L2), k_stream_ws<MODE, HI> (a frame or a band of it in one pass, the reference in registers) and
k_stream_ws_batch<MODE, HI>.  MODE 0..7 is the display filter, HI the form of the carry-free byte compare (thresholds
of 128 and above).  The host picks one from the call, the frame size and the number of frames.  Each GPU test below
takes one route through that choice for every mode at low and high thresholds and compares the count, xs, diff, every
display byte, the reference afterwards and the guard bytes behind the display buffer with OracleCore.  It also records
with torch.profiler which kernels it launched and asserts that its route reached the whole family it is meant to
reach, so a routing change that sends a case to another function fails here instead of passing on the wrong one.  The CPU test at the end pins the library's inventory of those functions.

The frames (checked on the CPU by the tests without a gpu mark):
  pairs         every (reference, current) byte pair in each of the four byte lanes of a 32-bit word, laid out by seeded
                permutations; a 3840x2160 frame is tiled with independently permuted copies
  next frames   built from the reference the frame before left: every byte moves by exactly thr or thr + 1, in either
                direction where that fits, or takes a random value
  heat pixels   channel differences summing to every index 0..765 of the heat-map table, channel order and sign permuted
  single pixels exactly one channel (B, G, R in turn) moves by thr + 1, the other two by thr
  binarisation  (modes 5 / 7 at 3840x2160) the first and last sixteenth of the rows hold one gray value each, so the
                two-max threshold moves if either is left out of the histogram
"""
import ctypes as C
import functools
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
from util import kernel_id, launched

LO = (-1, 0, 20, 127)
HI = (128, 200, 254, 255)
THRESHOLDS = LO + HI
SMALL = (514, 173)    # 266,766 bytes: every pair in every lane; N % 96 = 78 and N % 48 = 30 (a partial last group)
UHD = (3840, 2160)    # several segments / several bands
GUARD = 64            # bytes behind every display frame (multiple of 16: strides stay aligned)
FILL = 0xA5
NPAIRS = 256 * 256
HEAT = 766            # heat-map indices 0..765
SEED = 20

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def _r16(n):
    return (n + 15) // 16 * 16


def _r4(n):
    return (n + 3) // 4 * 4


def _hi(thr):
    return int(thr >= 128)


# ---------------------------------------------------------------------------------------------------------------------
# frames
# ---------------------------------------------------------------------------------------------------------------------
def _moves(rng, mag):
    """(reference, current) bytes with |current - reference| == mag, the sign random where both fit."""
    up = rng.random(mag.shape) < 0.5
    ref = np.where(up, rng.integers(0, 256 - mag), rng.integers(mag, 256))
    cur = np.where(up, ref + mag, ref - mag)
    return ref.astype(np.uint8), cur.astype(np.uint8)


@functools.lru_cache(maxsize=None)
def layout(w, h, seed):
    """Where the special pixels sit and which pair each other byte carries.
    Returns (heat pixel indices, single-channel pixel indices, pair index per byte or -1)."""
    npix, n = w * h, 3 * w * h
    rng = np.random.default_rng((seed, 1))
    big = n > 4_000_000
    nheat = HEAT * (16 if big else 1)
    nsingle = 3 * (64 if big else 8)
    special = rng.choice(npix, nheat + nsingle, replace=False)
    free = np.ones(n, dtype=bool)
    free[(3 * special[:, None] + np.arange(3)).reshape(-1)] = False
    pos = np.flatnonzero(free)
    pairs = np.full(n, -1, dtype=np.int32)
    for lane in range(4):
        pl = pos[pos % 4 == lane]
        copies = pl.size // NPAIRS
        assert copies >= 1, f"{w}x{h}: lane {lane} has room for {pl.size} of {NPAIRS} pairs"
        # copy c takes the next NPAIRS free bytes of the lane (a contiguous stretch of the frame) in its own order
        order = np.argsort(rng.random((copies, NPAIRS), dtype=np.float32), axis=1)
        pairs[pl[:copies * NPAIRS]] = order.reshape(-1)
    return special[:nheat], special[nheat:], pairs


@functools.lru_cache(maxsize=4)
def _first_common(w, h, seed):
    heat_px, _, pairs = layout(w, h, seed)
    n = 3 * w * h
    rng = np.random.default_rng((seed, 2))
    base = rng.integers(0, 256, n, dtype=np.uint8)
    cur = rng.integers(0, 256, n, dtype=np.uint8)
    m = pairs >= 0
    base[m] = (pairs[m] >> 8).astype(np.uint8)
    cur[m] = (pairs[m] & 255).astype(np.uint8)
    # heat pixels: sum s split into three channel differences of at most 255 each, in a random channel order
    s = rng.permuted(np.tile(np.arange(HEAT), heat_px.size // HEAT))
    lo0, hi0 = np.maximum(0, s - 510), np.minimum(255, s)
    d0 = rng.integers(lo0, hi0 + 1)
    lo1, hi1 = np.maximum(0, s - d0 - 255), np.minimum(255, s - d0)
    d1 = rng.integers(lo1, hi1 + 1)
    d = rng.permuted(np.stack([d0, d1, s - d0 - d1], axis=1), axis=1)
    r, c = _moves(rng, d)
    idx = 3 * heat_px[:, None] + np.arange(3)
    base[idx], cur[idx] = r, c
    base.flags.writeable = cur.flags.writeable = False
    return base, cur


def first_frame(w, h, thr, seed):
    """Base frame and first frame: every pair, the heat pixels and the single-channel pixels for thr."""
    base, cur = _first_common(w, h, seed)
    base, cur = base.copy(), cur.copy()
    _, single_px, _ = layout(w, h, seed)
    rng = np.random.default_rng((seed, 3, thr + 1))
    mags = np.full((single_px.size, 3), min(max(thr, 0), 255))
    mags[np.arange(single_px.size), np.arange(single_px.size) % 3] = min(max(thr + 1, 0), 255)
    r, c = _moves(rng, mags)
    idx = 3 * single_px[:, None] + np.arange(3)
    base[idx], cur[idx] = r, c
    return base, cur


def next_frame(ref, thr, seed, t):
    """Every byte moves by exactly thr or thr + 1 from the reference (either direction where it fits) or is random."""
    n = ref.size
    rng = np.random.default_rng((seed, 4, t, thr + 1))
    r = ref.astype(np.int16)
    kind = rng.integers(0, 3, n, dtype=np.int8)
    mag = np.where(kind == 0, min(max(thr, 0), 255), min(max(thr + 1, 0), 255)).astype(np.int16)
    up, down = r + mag, r - mag
    go_up = (up <= 255) & ((rng.random(n, dtype=np.float32) < 0.5) | (down < 0))
    rand = rng.integers(0, 256, n, dtype=np.int16)
    cur = np.where(go_up, up, np.where(down >= 0, down, rand))
    return np.where(kind == 2, rand, cur).astype(np.uint8)


def after(ref, cur, thr):
    """The reference after a frame: changed bytes take the frame's value (negative feedback)."""
    return np.where(np.abs(cur.astype(np.int16) - ref) > thr, cur, ref)


def binarising_rows(frame, w, h, t):
    """The first sixteenth of the rows one gray value A, the last sixteenth (plus 8 middle rows) another one B > A:
    the two-max threshold is (A + B) / 2, and it moves if either sixteenth is missing from the histogram."""
    img = frame.copy().reshape(h, w, 3)
    k = h // 16
    a, b = 80 + 4 * t, 170 - 6 * t
    img[:k] = a
    img[h - k:] = b
    img[h // 2:h // 2 + 8] = b
    return img.reshape(-1)


def scenario(w, h, thr, nframes, seed, binarise=False):
    """(base, frames[nframes]): the first frame, then frames built from the reference each one leaves."""
    base, cur = first_frame(w, h, thr, seed)
    frames = np.empty((nframes, base.size), dtype=np.uint8)
    ref = base
    for t in range(nframes):
        f = cur if t == 0 else next_frame(ref, thr, seed, t)
        frames[t] = binarising_rows(f, w, h, t) if binarise else f
        ref = after(ref, frames[t], thr)
    return base, frames


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the frames have the properties the GPU matrix relies on
# ---------------------------------------------------------------------------------------------------------------------
def _pair_codes(base, cur):
    return base.astype(np.int32) * 256 + cur


@pytest.mark.parametrize("size", [SMALL, UHD], ids=["small", "uhd"])
def test_every_pair_in_every_lane(size):
    w, h = size
    base, cur = first_frame(w, h, 20, SEED)
    code = _pair_codes(base, cur)
    n = code.size
    # the whole frame, and at 3840x2160 every quarter (the drop-in kernel's segments) and every band of one grid pass
    windows = [(0, n)]
    if n > 4_000_000:
        q = n // 4
        band = 148 * 512 * 96
        windows += [(i * q, (i + 1) * q) for i in range(4)] + [(o, min(o + band, n)) for o in range(0, n, band)]
    for lo, hi in windows:
        for lane in range(4):
            start = lo + (lane - lo) % 4
            seen = np.bincount(code[start:hi:4], minlength=NPAIRS)
            assert (seen > 0).all(), f"bytes [{lo}, {hi}) lane {lane}: {int((seen == 0).sum())} pairs missing"
    # the permutations move pairs across channels and positions in the 48-byte pixel group
    i = np.flatnonzero(code == 0x80FF)
    assert len(set(i % 3)) == 3 and len(set(i % 48)) >= 4


@pytest.mark.parametrize("size", [SMALL, UHD], ids=["small", "uhd"])
def test_heat_pixels_cover_the_table(size):
    w, h = size
    base, cur = first_frame(w, h, 20, SEED)
    heat_px, _, _ = layout(w, h, SEED)
    d = np.abs(cur.reshape(-1, 3)[heat_px].astype(np.int32) - base.reshape(-1, 3)[heat_px])
    sums = d.sum(axis=1)
    assert (np.bincount(sums, minlength=HEAT) == heat_px.size // HEAT).all(), "every sum 0..765 once per copy"
    # the largest differences sit in every channel, and both signs occur
    assert len(set(np.argmax(d, axis=1)[sums > 300])) == 3
    sd = cur.reshape(-1, 3)[heat_px].astype(np.int32) - base.reshape(-1, 3)[heat_px]
    assert (sd > 100).any() and (sd < -100).any()


@pytest.mark.parametrize("thr", [t for t in THRESHOLDS if 0 <= t <= 254])
def test_single_channel_pixels(thr):
    w, h = SMALL
    base, cur = first_frame(w, h, thr, SEED)
    _, single_px, _ = layout(w, h, SEED)
    d = np.abs(cur.reshape(-1, 3)[single_px].astype(np.int32) - base.reshape(-1, 3)[single_px])
    crossing = d > thr
    assert (crossing.sum(axis=1) == 1).all(), "exactly one channel over the threshold"
    assert (d[crossing] == thr + 1).all() and (d[~crossing] == thr).all()
    assert set(np.argmax(crossing, axis=1)) == {0, 1, 2}, "B, G and R each take their turn"


@pytest.mark.parametrize("thr", THRESHOLDS)
def test_moves_on_the_threshold_in_both_directions(oracle, thr):
    """Frame 1 against the base and frame 2 against the reference frame 1 left -- the oracle's -- both hold differences
    of exactly thr and thr + 1, up and down."""
    w, h = SMALL
    base, frames = scenario(w, h, thr, 2, SEED)
    oc = oracle.OracleCore(w, h, base, thr=thr)
    oc.exec_core(frames[0])
    ref1 = oc.reference()
    oc.close()
    assert np.array_equal(ref1, after(base, frames[0], thr))
    for t, (ref, f) in enumerate([(base, frames[0]), (ref1, frames[1])]):
        d = f.astype(np.int16) - ref
        for m in {thr, thr + 1} & set(range(1, 256)):
            assert (d == m).any() and (d == -m).any(), f"frame {t + 1}: |d| = {m} missing in one direction"
        if thr <= 0:
            assert (d == 0).any()


@pytest.mark.parametrize("mode", [5, 7])
def test_binarisation_threshold_needs_the_first_and_last_rows(oracle, mode):
    w, h = UHD
    k = h // 16
    gray = oracle.gray_weighted1 if mode == 5 else oracle.gray_avg1
    _, frames = scenario(w, h, 200, 2, SEED, binarise=True)
    for t, f in enumerate(frames):
        g = gray(f, w, h).reshape(h, w)
        full = oracle.histogram1(g)
        head, tail = oracle.histogram1(g[:k]), oracle.histogram1(g[h - k:])
        thr = [oracle.threshold_twomax(x, 50, 200) for x in (full, full - head, full - tail)]
        assert len(set(thr)) == 3, f"frame {t}: thresholds full / without the first / without the last rows {thr}"


# ---------------------------------------------------------------------------------------------------------------------
# which kernels ran
# ---------------------------------------------------------------------------------------------------------------------
def family(kernel, modes=range(8)):
    return {f"{kernel}<{m},{hi}>" for m in modes for hi in (0, 1)}


# ---------------------------------------------------------------------------------------------------------------------
# comparisons (collected, so one run reports every case that disagrees and where)
# ---------------------------------------------------------------------------------------------------------------------
def _where(idx, n):
    idx = np.asarray(idx, dtype=np.int64)
    return (f"{idx.size} bytes, first {idx[:4].tolist()}, by lane {np.bincount(idx % 4, minlength=4).tolist()}, "
            f"by channel {np.bincount(idx % 3, minlength=3).tolist()}, by quarter {np.bincount(idx * 4 // n, minlength=4).tolist()}")


def _compare(errors, tag, oc, frame, pos, xs, diff, show, guard):
    opos, oxs, odiff, oshow, _ = oc.exec_core(frame)
    if pos != opos:
        errors.append(f"{tag}: count {pos}, oracle {opos}")
    m = min(pos, opos)
    bad = np.flatnonzero(xs[:m] != oxs[:m])
    if bad.size:
        errors.append(f"{tag}: xs differ at {bad.size} entries, first {bad[0]} ({xs[bad[0]]}, oracle {oxs[bad[0]]})")
    bad = np.flatnonzero(diff[:m] != odiff[:m])
    if bad.size:
        errors.append(f"{tag}: diff differs at {_where(oxs[bad], frame.size)}")
    if oshow is not None:
        bad = np.flatnonzero(show != oshow)
        if bad.size:
            errors.append(f"{tag}: display differs at {_where(bad, frame.size)}")
    if guard is not None and (guard != FILL).any():
        errors.append(f"{tag}: {int((guard != FILL).sum())} guard bytes behind the display frame written")


def _compare_ref(errors, tag, ref, oref):
    bad = np.flatnonzero(ref != oref)
    if bad.size:
        errors.append(f"{tag}: reference differs at {_where(bad, ref.size)}")


def _report(errors, seen, expected):
    assert seen == expected, f"missing {sorted(expected - seen)}, unexpected {sorted(seen - expected)}"
    assert not errors, f"{len(errors)} disagreements:\n" + "\n".join(errors[:40])


# ---------------------------------------------------------------------------------------------------------------------
# the routes
# ---------------------------------------------------------------------------------------------------------------------
def _exec_frames(cvs, w, h, base, frames, thr, mode):
    """cvs_exec frame by frame into host buffers with a guard behind the display frame."""
    n = 3 * w * h
    s = cvs.Stream(w, h, base, threshold=thr, mode=mode)
    out = []
    for f in frames:
        buf = f.copy()
        xs = np.empty(n, dtype=np.int32)
        show = np.full(n + GUARD, FILL, dtype=np.uint8)
        pos = C.c_uint(0)
        s.exec_raw(buf.ctypes.data, show.ctypes.data if mode else None, "", C.byref(pos), xs.ctypes.data)
        p = pos.value
        out.append((p, xs[:p], buf[:p], show[:n] if mode else None, show[n:]))
    ref = s.reference()
    s.close()
    return out, ref


def _sequence(cvs, w, h, base, frames, thr, mode):
    """cvs_run_sequence_device over all frames at once; display frames GUARD bytes apart."""
    import torch
    nf, n = frames.shape
    fstride, cap, sstride = _r16(n), _r4(n), _r16(n) + GUARD
    host = np.zeros((nf, fstride), dtype=np.uint8)
    host[:, :n] = frames
    d_frames = torch.from_numpy(host).cuda().reshape(-1)
    d_pos = torch.zeros(nf, dtype=torch.int32, device="cuda")
    d_xs = torch.full((nf * cap,), -7, dtype=torch.int32, device="cuda")
    d_diff = torch.zeros(nf * cap, dtype=torch.uint8, device="cuda")
    d_show = torch.full((nf * sstride,), FILL, dtype=torch.uint8, device="cuda") if mode else None
    s = cvs.Stream(w, h, base, threshold=thr, mode=mode)
    s.run_sequence_device(d_frames.data_ptr(), fstride, nf, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(), cap,
                          d_show.data_ptr() if mode else 0, sstride if mode else 0,
                          cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s.sequence_status()
    pos = d_pos.cpu().numpy()
    xs, diff = d_xs.cpu().numpy().reshape(nf, cap), d_diff.cpu().numpy().reshape(nf, cap)
    show = d_show.cpu().numpy().reshape(nf, sstride) if mode else None
    out = [(int(pos[t]), xs[t, :pos[t]], diff[t, :pos[t]], show[t, :n] if mode else None,
            show[t, n:] if mode else None) for t in range(nf)]
    ref = s.reference()
    s.close()
    return out, ref


def _run_case(cvs, oracle, errors, seen, runner, w, h, thr, mode, nframes, expected, binarise=False, seed=SEED):
    tag = f"{w}x{h} mode {mode} thr {thr}"
    base, frames = scenario(w, h, thr, nframes, seed, binarise)
    (out, ref), names = launched(lambda: runner(cvs, w, h, base, frames, thr, mode))
    seen |= names
    if names != {expected}:
        errors.append(f"{tag}: launched {sorted(names)}, expected {expected}")
    oc = oracle.OracleCore(w, h, base, thr=thr, mode=mode)
    for t, r in enumerate(out):
        _compare(errors, f"{tag} frame {t}", oc, frames[t], *r)
    _compare_ref(errors, tag, ref, oc.reference())
    oc.close()


def _uhd_cases(modes=range(8)):
    """At 3840x2160 every mode runs at one low and one high threshold; over the eight modes every threshold runs."""
    return [(m, t) for m in modes for t in (LO[m % 4], HI[m % 4])]


def _seq_kmode(mode):
    return 0 if mode in (5, 7) else mode  # sequences binarise with k_gray_hist_seq in front of the plain kernel


_FRESH = "CVS_TEST_FRESH_PROCESS"


@pytest.mark.gpu
def test_standalone_red_and_heat_maps(cvs, oracle):
    """cvs_red_map_device at every threshold (k_filter<1, hi>) and cvs_heat_map_device over the 766 sums
    (k_filter<0, false>), at a size whose last pixel group is partial, with guard bands on both sides of the output.
    The checks run in a fresh interpreter of their own.  On a B200 with torch 2.11, a process that has already run about
    two minutes of other GPU tests still gets the cudaLaunchKernel calls of these few-microsecond kernels from the
    profiler, but no longer the kernels themselves.  That happens whichever tests ran before, so the kernel names could
    not be checked in the same process."""
    if os.environ.get(_FRESH) != "1":
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", "-p", "no:cacheprovider",
                            os.path.abspath(__file__) + "::test_standalone_red_and_heat_maps"],
                           cwd=root, env=dict(os.environ, **{_FRESH: "1"}), stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, timeout=600)
        out = r.stdout.decode()
        assert r.returncode == 0 and re.search(r"\b1 passed\b", out), out[-4000:]
        return
    import torch
    from cudavideostream_b200 import filters
    errors, seen = [], set()
    w, h = SMALL
    n = 3 * w * h
    assert n % 48
    for op in ["heat"] + list(THRESHOLDS):
        base, cur = first_frame(w, h, 20 if op == "heat" else op, SEED)
        d_prev, d_cur = torch.from_numpy(base).cuda(), torch.from_numpy(cur).cuda()
        raw = torch.full((n + 2 * GUARD,), FILL, dtype=torch.uint8, device="cuda")
        out = raw[GUARD:GUARD + n]
        if op == "heat":
            got, names = launched(lambda: (filters.heat_map(d_prev.data_ptr(), d_cur.data_ptr(), out.data_ptr(), w, h),
                                           raw.cpu().numpy())[1])
            want, wname = oracle.heat_map(base, cur, w, h), "k_filter<0,0>"
        else:
            got, names = launched(lambda: (filters.red_map(d_prev.data_ptr(), d_cur.data_ptr(), out.data_ptr(), w, h, op),
                                           raw.cpu().numpy())[1])
            want, wname = oracle.red_map(base, cur, w, h, op), f"k_filter<1,{_hi(op)}>"
        seen |= names
        if names != {wname}:
            errors.append(f"{op}: launched {sorted(names)}, expected {wname}")
        bad = np.flatnonzero(got[GUARD:GUARD + n] != want)
        if bad.size:
            errors.append(f"{op}: output differs at {_where(bad, n)}")
        if (got[:GUARD] != FILL).any() or (got[GUARD + n:] != FILL).any():
            errors.append(f"{op}: guard bytes written")
    _report(errors, seen, {"k_filter<0,0>", "k_filter<1,0>", "k_filter<1,1>"})


@pytest.mark.gpu
def test_dropin_small(cvs, oracle):
    """cvs_exec at 514x173: one pass, reference in registers -- k_stream_ws<m, hi>."""
    errors, seen = [], set()
    w, h = SMALL
    for mode in range(8):
        for thr in THRESHOLDS:
            _run_case(cvs, oracle, errors, seen, _exec_frames, w, h, thr, mode, 2, f"k_stream_ws<{mode},{_hi(thr)}>")
    _report(errors, seen, family("k_stream_ws"))


@pytest.mark.gpu
def test_sequence_small(cvs, oracle):
    """Three frames in one cvs_run_sequence_device -- k_stream_ws<kmode, hi>, kmode 0 for modes 5 / 7."""
    errors, seen = [], set()
    w, h = SMALL
    for mode in range(8):
        for thr in THRESHOLDS:
            _run_case(cvs, oracle, errors, seen, _sequence, w, h, thr, mode, 3,
                      f"k_stream_ws<{_seq_kmode(mode)},{_hi(thr)}>")
    _report(errors, seen, family("k_stream_ws", modes=(0, 1, 2, 3, 4, 6)))


@pytest.mark.gpu
def test_batch_small(cvs, oracle):
    """Three cameras per cvs_run_batch_device, two batches in a row -- k_stream_ws_batch<m, hi>."""
    import torch
    errors, seen = [], set()
    w, h = SMALL
    n = 3 * w * h
    cap, sstride = _r4(n), _r16(n) + GUARD
    cs = torch.cuda.current_stream().cuda_stream
    for mode in range(8):
        for thr in THRESHOLDS:
            tag = f"batch mode {mode} thr {thr}"
            cams = [scenario(w, h, thr, 2, SEED + i) for i in range(3)]
            streams = [cvs.Stream(w, h, b, threshold=thr, mode=mode) for b, _ in cams]
            orcs = [oracle.OracleCore(w, h, b, thr=thr, mode=mode) for b, _ in cams]
            for t in range(2):
                def batch():
                    d_frames = []
                    for _, frames in cams:
                        buf = np.zeros(_r16(n) + 16, dtype=np.uint8)
                        buf[:n] = frames[t]
                        d_frames.append(torch.from_numpy(buf).cuda())
                    d_pos = torch.zeros(3, dtype=torch.int32, device="cuda")
                    d_xs = torch.full((3 * cap,), -7, dtype=torch.int32, device="cuda")
                    d_diff = torch.zeros(3 * cap, dtype=torch.uint8, device="cuda")
                    d_show = torch.full((3 * sstride,), FILL, dtype=torch.uint8, device="cuda") if mode else None
                    cvs.run_batch_device(streams, [f.data_ptr() for f in d_frames], d_pos.data_ptr(), d_xs.data_ptr(),
                                         d_diff.data_ptr(), cap, d_show.data_ptr() if mode else 0,
                                         sstride if mode else 0, cuda_stream=cs)
                    torch.cuda.synchronize()
                    for s in streams:
                        s.sequence_status()
                    return (d_pos.cpu().numpy(), d_xs.cpu().numpy().reshape(3, cap), d_diff.cpu().numpy().reshape(3, cap),
                            d_show.cpu().numpy().reshape(3, sstride) if mode else None)
                (pos, xs, diff, show), names = launched(batch)
                seen |= names
                want = f"k_stream_ws_batch<{mode},{_hi(thr)}>"
                if names != {want}:
                    errors.append(f"{tag} step {t}: launched {sorted(names)}, expected {want}")
                for i, (_, frames) in enumerate(cams):
                    p = int(pos[i])
                    _compare(errors, f"{tag} step {t} camera {i}", orcs[i], frames[t], p, xs[i, :p], diff[i, :p],
                             show[i, :n] if mode else None, show[i, n:] if mode else None)
            for i in range(3):
                _compare_ref(errors, f"{tag} camera {i}", streams[i].reference(), orcs[i].reference())
                streams[i].close()
                orcs[i].close()
    _report(errors, seen, family("k_stream_ws_batch"))


@pytest.mark.gpu
def test_dropin_uhd(cvs, oracle):
    """cvs_exec at 3840x2160: several segments, reference through L2 -- k_stream<m, hi>.  In modes 5 / 7 the
    block histograms gather all segments of the frame."""
    errors, seen = [], set()
    w, h = UHD
    for mode, thr in _uhd_cases():
        _run_case(cvs, oracle, errors, seen, _exec_frames, w, h, thr, mode, 2, f"k_stream<{mode},{_hi(thr)}>",
                  binarise=mode in (5, 7))
    _report(errors, seen, family("k_stream"))


@pytest.mark.gpu
def test_short_sequence_uhd(cvs, oracle):
    """Two 3840x2160 frames in one sequence (too few for bands): k_stream<kmode, hi>, several frames x several
    segments, the look-back carrying totals across both."""
    errors, seen = [], set()
    w, h = UHD
    for mode, thr in _uhd_cases():
        _run_case(cvs, oracle, errors, seen, _sequence, w, h, thr, mode, 2, f"k_stream<{_seq_kmode(mode)},{_hi(thr)}>",
                  binarise=mode in (5, 7))
    _report(errors, seen, family("k_stream", modes=(0, 1, 2, 3, 4, 6)))


@pytest.mark.gpu
def test_banded_sequence_uhd(cvs, oracle):
    """Five 3840x2160 frames: walked band by band, k_stream_ws<m, hi> per band."""
    errors, seen = [], set()
    w, h = UHD
    modes = (1, 2, 3, 4, 6)
    for mode, thr in _uhd_cases(modes):
        _run_case(cvs, oracle, errors, seen, _sequence, w, h, thr, mode, 5, f"k_stream_ws<{mode},{_hi(thr)}>")
    _report(errors, seen, family("k_stream_ws", modes=modes))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the library holds exactly the functions the matrix above runs
# ---------------------------------------------------------------------------------------------------------------------
def test_library_inventory_matches_the_matrix():
    """All 48 stream-kernel functions, and the 7 k_filter ones (ops 2..5 are run by test_standalone_filters).  A new
    template parameter or mode fails here until the GPU tests above reach it."""
    import cudavideostream_b200 as cvs
    try:
        res = subprocess.run([CUOBJDUMP, "-res-usage", cvs.library_path()], capture_output=True, text=True,
                             check=True).stdout
    except (OSError, subprocess.CalledProcessError) as e:
        pytest.skip(f"cuobjdump unavailable: {e}")
    names = [kernel_id(f) for f in re.findall(r"Function (\S+):", res)]
    stream = sorted(k for k in names if k and k.startswith("k_stream"))
    assert len(stream) == len(set(stream)) == 48, len(stream)
    assert set(stream) == family("k_stream") | family("k_stream_ws") | family("k_stream_ws_batch")
    filt = sorted(k for k in names if k and k.startswith("k_filter"))
    assert filt == sorted({"k_filter<0,0>", "k_filter<1,0>", "k_filter<1,1>"} | {f"k_filter<{op},0>" for op in range(2, 6)})
