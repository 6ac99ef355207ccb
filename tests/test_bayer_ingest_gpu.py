"""Raw Bayer cameras on the GPU: cvs_bayer_to_bgr_device is cv2.cvtColor byte for byte (all four patterns, degenerate,
odd and camera sizes, pitched mosaics, nothing written outside the frame), and cvs_submit_bayer / cvs_submit_bayer_wire
deliver what cvs_submit_io / cvs_submit_wire deliver for the demosaiced frames -- and what the CPU oracle computes -- in
every display mode, with the noise filter and the overlay, from pinned and pageable memory, interleaved with raw, YUV
and JPEG tickets, at 3840x2160 and at 2x2.  Refused submissions leave the handle as it was."""
import ctypes as C
import os

import numpy as np
import pytest

import bayer_ref as B
import yuv_ref as Y
from util import CHARS_STR, glyph_atlas

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
GUARD = 64


def _device_demosaic(cvs, torch, pattern, raw, extra_pitch=0):
    """The mosaic at a pitch of the width rounded up to 16 (+ extra_pitch), the padding filled with garbage; the output
    between two guard bands.  Returns the frame [h, w, 3]."""
    h, w = raw.shape
    pitch = (w + 15) // 16 * 16 + extra_pitch
    src = torch.full((h, pitch), 0x5A, dtype=torch.uint8, device="cuda")
    src[:, :w] = torch.from_numpy(np.ascontiguousarray(raw)).cuda()
    n = 3 * w * h
    out = torch.full((n + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
    cvs.filters.bayer_to_bgr(pattern, src.data_ptr(), pitch, out.data_ptr() + GUARD, w, h,
                             torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert np.all(o[:GUARD] == 0xA5) and np.all(o[GUARD + n:] == 0xA5), "the demosaic wrote outside the frame"
    return o[GUARD:GUARD + n].reshape(h, w, 3)


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
def test_device_demosaic_is_cv2(cvs, pattern):
    cv2 = pytest.importorskip("cv2")
    import torch
    rng = np.random.default_rng(pattern)
    for w, h in [(1, 1), (2, 2), (2, 9), (9, 2), (3, 3), (17, 5), (18, 6), (1918, 1078), (1919, 1079), (1920, 1080),
                 (3840, 2160)]:
        raw = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
        want = B.cv2_demosaic(cv2, pattern, raw)
        for extra in (0, 48):  # tight (rounded to 16) and wider pitches
            got = _device_demosaic(cvs, torch, pattern, raw, extra)
            bad = np.argwhere((got != want).any(axis=2))
            assert bad.size == 0, f"{w}x{h} pitch +{extra}: {len(bad)} pixels differ, first at {bad[:5].tolist()}"


def _synth_bayer(oracle, pattern, w, h, nframes, density_ppm, seed):
    """Mosaics of a synthetic sequence's frames, and the BGR frames cv2.cvtColor makes of them (base first)."""
    base, frames = oracle.synth_sequence(w, h, nframes, density_ppm, seed)
    raws = [B.mosaic(f.reshape(h, w, 3), pattern).reshape(-1) for f in [base] + list(frames)]
    bgr = [B.bayer_to_bgr(pattern, r.reshape(h, w)).reshape(-1) for r in raws]
    return raws, bgr


def _outs(cvs, n, pinned):
    if pinned:
        return [(cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), cvs.alloc_host(n + 32), (C.c_uint * 1)()) for _ in range(4)]
    return [(np.zeros(n + 32, np.uint8), np.zeros(n + 8, np.int32), np.zeros(n + 32, np.uint8), (C.c_uint * 1)()) for _ in range(4)]


def _ptr(b):
    return b.ctypes.data if isinstance(b, np.ndarray) else b.ptr


def _arr(b, dtype=np.uint8):
    return b.view(dtype) if isinstance(b, np.ndarray) else b.array(dtype)


def _host(cvs, a, pinned):
    if not pinned:
        return a.copy()
    hb = cvs.alloc_host(a.size + 64)
    hb.array()[:a.size] = a
    return hb


def _run(s, frames, submit, n, pinned, mode, text, cvs):
    """Submits every frame with four tickets in flight; returns [(pos, xs, diff, show)] in order."""
    outs, res, pending = _outs(cvs, n, pinned), [], []

    def drain():
        tk, (d, x, sh, pb) = pending.pop(0)
        s.wait(tk)
        p = pb[0]
        res.append((p, _arr(x, np.int32)[:p].copy(), _arr(d)[:p].copy(), _arr(sh)[:n].copy() if mode else None))

    for i, f in enumerate(frames):
        if len(pending) == 4:
            drain()
        d, x, sh, pb = outs[i % 4]
        pending.append((submit(f, _ptr(d), _ptr(sh) if mode else None, text, C.addressof(pb), _ptr(x)), outs[i % 4]))
    while pending:
        drain()
    return res


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
@pytest.mark.parametrize("mode", range(8))
def test_submit_bayer_is_submit_io_of_the_demosaiced_frames(cvs, oracle, pattern, mode):
    """323x181: odd W and H, 3W % 16 != 0 and a packed mosaic whose rows are not 16-byte aligned, so the demosaic takes
    both its vector stores and its byte path.  Across the eight modes every combination of noise filter, overlay text
    and pinned / pageable buffers occurs once per pattern."""
    cv2 = pytest.importorskip("cv2")
    w, h, nframes = 323, 181, 7
    n = 3 * w * h
    noise, text, pinned = mode % 2 == 1, "FPS: 30" if mode % 4 < 2 else "", mode < 4
    raws, bgr = _synth_bayer(oracle, pattern, w, h, nframes, 60000, seed=11 * mode + pattern)
    for r, f in zip(raws, bgr):  # the frames the raw side uploads are cv2's
        assert np.array_equal(B.cv2_demosaic(cv2, pattern, r.reshape(h, w)).reshape(-1), f)
    k = oracle.gaussian_kernel(3, 1.2)
    g = glyph_atlas()
    cfg = dict(mode=mode, glyphs=g, glyph_w=7, glyph_h=5, glyph_chars=CHARS_STR)
    if noise:
        cfg.update(noise_filter=True, ksize=3, kweights=k)
    sb, sr = cvs.Stream(w, h, bgr[0], **cfg), cvs.Stream(w, h, bgr[0], **cfg)
    ins = [_host(cvs, r, pinned) for r in raws[1:]]
    frames = [_host(cvs, f, pinned) for f in bgr[1:]]
    got = _run(sb, ins, lambda f, d, sh, t, p, x: sb.submit_bayer_raw(pattern, _ptr(f), d, sh, t, p, x), n, pinned, mode,
               text, cvs)
    want = _run(sr, frames, lambda f, d, sh, t, p, x: sr.submit_io_raw(_ptr(f), d, sh, t, p, x), n, pinned, mode, text, cvs)
    oc = oracle.OracleCore(w, h, bgr[0], mode=mode, noise_filter=int(noise), K=3, k=k, glyphs=g, gw=7, gh=5, chars=CHARS_STR)
    for t in range(nframes):
        opos, oxs, odiff, oshow, _ = oc.exec_core(bgr[t + 1], text)
        for name, r in (("bayer", got[t]), ("raw", want[t])):
            assert r[0] == opos, f"{name} frame {t}: pos {r[0]} vs {opos}"
            assert np.array_equal(r[1], oxs) and np.array_equal(r[2], odiff), f"{name} frame {t}: payload"
            if mode:
                assert np.array_equal(r[3], oshow), f"{name} frame {t}: display frame"
    assert opos > 0
    assert np.array_equal(sb.reference(), oc.reference()) and np.array_equal(sr.reference(), oc.reference())
    tm = sb.timing()
    assert tm["h2d_us"] > 0 and tm["kernel_us"] > 0
    sb.close()
    sr.close()


@pytest.mark.parametrize("pattern", B.PATTERNS, ids=B.NAMES.get)
def test_submit_bayer_wire_is_submit_wire_of_the_demosaiced_frames(cvs, oracle, pattern):
    from cudavideostream_b200 import wire
    w, h = 1920, 1080
    n = 3 * w * h
    raws, bgr = _synth_bayer(oracle, pattern, w, h, 4, 40000, seed=5 + pattern)
    sb, sr = cvs.Stream(w, h, bgr[0]), cvs.Stream(w, h, bgr[0])
    wb, wr = cvs.alloc_host(wire.bound(w, h) + 64), cvs.alloc_host(wire.bound(w, h) + 64)
    inp, raw = cvs.alloc_host(w * h + 64), cvs.alloc_host(n + 64)
    pageable = np.zeros(wire.bound(w, h) + 64, np.uint8)
    for t in range(1, 5):
        inp.array()[:w * h] = raws[t]
        raw.array()[:n] = bgr[t]
        # (the Bayer side alternates between a pinned and a pageable output buffer: pushed by the device / copied in
        # cvs_wait)
        out, optr = (wb.array(), wb.ptr) if t % 2 else (pageable, pageable.ctypes.data)
        sb.wait(sb.submit_bayer_wire_raw(pattern, inp.ptr, optr, None, ""))
        sr.wait(sr.submit_wire_raw(raw.ptr, wr.ptr, None, ""))
        a, b = out, wr.array()
        size = wire.size_of(b)
        assert size > 16 and wire.size_of(a) == size and np.array_equal(a[:size], b[:size]), f"frame {t}"
    assert np.array_equal(sb.reference(), sr.reference())
    sb.close()
    sr.close()


def test_bayer_raw_yuv_and_jpeg_tickets_interleave(cvs, oracle, monkeypatch):
    """One handle, tickets of every ingest form in flight together: each delivers what the oracle computes on the BGR
    frame it stands for, in submission order."""
    monkeypatch.setenv("CVS_JPEG_DECODER", "own")
    z = np.load(os.path.join(GOLDEN, "jpeg_cases.npz"))
    name = "q90_422_320x240"
    jpg = z[name + "/jpg"].tobytes()
    w, h = (int(v) for v in z[name + "/wh"])
    n = 3 * w * h
    jb = cvs.alloc_host(len(jpg) + 64)
    jb.array()[:len(jpg)] = np.frombuffer(jpg, dtype=np.uint8)
    jbgr = oracle.jpeg_decode_bgr(jpg).reshape(-1)
    rg, bg = _synth_bayer(oracle, B.RGGB, w, h, 6, 50000, seed=8)
    rb, bb = _synth_bayer(oracle, B.GBRG, w, h, 6, 50000, seed=9)
    base, frames = oracle.synth_sequence(w, h, 6, 50000, 10)
    yn = [Y.from_bgr(Y.NV12, f, w, h) for f in frames]
    bn = [Y.yuv_to_bgr(Y.NV12, b, w, h).reshape(-1) for b in yn]
    seq = []  # (kind, pattern or format, input, the BGR frame it stands for), in submission order
    for t in range(1, 7):
        seq += [("bayer", B.RGGB, rg[t], bg[t]), ("raw", 0, None, bb[t]), ("yuv", Y.NV12, yn[t - 1], bn[t - 1]),
                ("jpeg", 0, None, jbgr), ("bayer", B.GBRG, rb[t], bb[t])]
    s = cvs.Stream(w, h, bg[0])
    oc = oracle.OracleCore(w, h, bg[0])
    bufs = [(cvs.alloc_host(n + 64), cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()) for _ in range(4)]
    pending = []

    def check(tk, d, x, pb, ff):
        s.wait(tk)
        opos, oxs, odiff, _, _ = oc.exec_core(ff)
        assert pb[0] == opos and np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs)

    for i, (kind, code, src, f) in enumerate(seq):
        if len(pending) == 4:
            tk, (_, d, x, pb), ff = pending.pop(0)
            check(tk, d, x, pb, ff)
        ib, d, x, pb = bufs[i % 4]
        if kind == "raw":
            ib.array()[:n] = f
            tk = s.submit_io_raw(ib.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        elif kind == "jpeg":
            tk = s.submit_jpeg_raw(jb.ptr, len(jpg), d.ptr, None, "", C.addressof(pb), x.ptr)
        elif kind == "yuv":
            ib.array()[:src.size] = src
            tk = s.submit_yuv_raw(code, ib.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        else:
            ib.array()[:src.size] = src
            tk = s.submit_bayer_raw(code, ib.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        pending.append((tk, bufs[i % 4], f))
    for tk, (_, d, x, pb), ff in pending:
        check(tk, d, x, pb, ff)
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_4k_stream(cvs, oracle):
    """3840x2160 does not fit one pass of the stream kernel: the single-frame path walks it in segments."""
    w, h = 3840, 2160
    n = 3 * w * h
    raws, bgr = _synth_bayer(oracle, B.GRBG, w, h, 3, 20000, seed=4)
    s = cvs.Stream(w, h, bgr[0], mode=cvs.MODE_HEAT_MAP)
    oc = oracle.OracleCore(w, h, bgr[0], mode=1)
    inp = cvs.alloc_host(w * h + 64)
    d, x, sh, pb = cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), cvs.alloc_host(n + 32), (C.c_uint * 1)()
    for t in range(1, 4):
        inp.array()[:w * h] = raws[t]
        s.wait(s.submit_bayer_raw(B.GRBG, inp.ptr, d.ptr, sh.ptr, "", C.addressof(pb), x.ptr))
        opos, oxs, odiff, oshow, _ = oc.exec_core(bgr[t])
        assert pb[0] == opos > 0, f"frame {t}"
        assert np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs), f"frame {t}"
        assert np.array_equal(sh.array()[:n], oshow), f"frame {t}: heat map"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_2x2_stream_gets_black_frames(cvs, oracle):
    """Below 3x3 OpenCV's demosaic is all zero: a 2x2 stream whose reference holds other pixels sees black frames."""
    w, h = 2, 2
    n = 3 * w * h
    base = np.arange(n, dtype=np.uint8) * np.uint8(20) + np.uint8(30)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    inp = cvs.alloc_host(64)
    d, x, pb = cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()
    for t, pattern in enumerate(B.PATTERNS):
        inp.array()[:w * h] = np.array([255, 7, 90, 200], np.uint8) + np.uint8(t)
        s.wait(s.submit_bayer_raw(pattern, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr))
        opos, oxs, odiff, _, _ = oc.exec_core(np.zeros(n, np.uint8))
        assert pb[0] == opos and np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs)
        assert (opos > 0) == (t == 0)
    assert np.all(s.reference() == 0) and np.array_equal(s.reference(), oc.reference())
    s.close()


def test_refusals_leave_the_handle_as_it_was(cvs, oracle):
    lib = cvs.load_library()
    w, h = 64, 48
    n = 3 * w * h
    raws, bgr = _synth_bayer(oracle, B.BGGR, w, h, 3, 80000, seed=2)
    s = cvs.Stream(w, h, bgr[0])
    oc = oracle.OracleCore(w, h, bgr[0])
    inp, d, x, pb = cvs.alloc_host(n), cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()
    tk = C.c_uint64(0)
    wout = cvs.alloc_host(cvs.wire.bound(w, h) + 64)

    def good(t):
        inp.array()[:w * h] = raws[t]
        ticket = s.submit_bayer_raw(B.BGGR, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        s.wait(ticket)
        opos, oxs, odiff, _, _ = oc.exec_core(bgr[t])
        assert pb[0] == opos and np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs)
        return ticket

    last = good(1)
    ref = s.reference()
    h_ = s._h
    P = B.BGGR
    refusals = [
        lib.cvs_submit_bayer(h_, 0, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_bayer(h_, 5, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_bayer(h_, P, None, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_bayer(h_, P, inp.ptr, None, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_bayer(h_, P, inp.ptr, d.ptr, None, b"", None, x.ptr, C.byref(tk)),
        lib.cvs_submit_bayer(h_, P, inp.ptr, d.ptr, None, b"", C.addressof(pb), None, C.byref(tk)),
        lib.cvs_submit_bayer(h_, P, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, None),
        lib.cvs_submit_bayer(None, P, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_bayer_wire(h_, 0, inp.ptr, wout.ptr, None, b"", C.byref(tk)),
        lib.cvs_submit_bayer_wire(h_, 5, inp.ptr, wout.ptr, None, b"", C.byref(tk)),
        lib.cvs_submit_bayer_wire(h_, B.RGGB, None, wout.ptr, None, b"", C.byref(tk)),
        lib.cvs_submit_bayer_wire(h_, B.RGGB, inp.ptr, None, None, b"", C.byref(tk)),
        lib.cvs_submit_bayer_wire(h_, B.RGGB, inp.ptr, wout.ptr, None, b"", None),
        lib.cvs_submit_bayer_wire(None, B.RGGB, inp.ptr, wout.ptr, None, b"", C.byref(tk)),
    ]
    assert refusals == [1] * len(refusals)
    assert np.array_equal(s.reference(), ref)
    assert good(2) == last + 1  # no ticket was consumed
    # a fifth ticket while four are outstanding
    tks = []
    inp.array()[:w * h] = raws[3]
    outs = [(cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()) for _ in range(4)]
    for dd, xx, pp in outs:
        tks.append(s.submit_bayer_raw(B.BGGR, inp.ptr, dd.ptr, None, "", C.addressof(pp), xx.ptr))
    with pytest.raises(cvs.CVSError) as e:
        s.submit_bayer_raw(B.BGGR, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
    assert e.value.status == 1
    for t, (dd, xx, pp) in zip(tks, outs):
        s.wait(t)
        opos, oxs, odiff, _, _ = oc.exec_core(bgr[3])
        assert pp[0] == opos and np.array_equal(dd.array()[:opos], odiff)
    assert tks == [last + 2 + i for i in range(4)]
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_device_demosaic_alignment_and_pitch(cvs):
    """Refusals of the device entry on real device buffers, then a good call on the same buffers."""
    import torch
    w, h = 64, 32
    buf = torch.zeros(2 * w * h + 64, dtype=torch.uint8, device="cuda")
    out = torch.zeros(3 * w * h + 64, dtype=torch.uint8, device="cuda")
    a, o = buf.data_ptr(), out.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    cases = [((a + 8, w, o), 4), ((a, w + 4, o), 4), ((a, w, o + 4), 4), ((a, w - 16, o), 1), ((a, w, 0), 1),
             ((0, w, o), 1)]
    for (raw, pitch, dst), status in cases:
        with pytest.raises(cvs.CVSError) as e:
            cvs.filters.bayer_to_bgr(B.RGGB, raw, pitch, dst, w, h, st)
        assert e.value.status == status
    for bad in (0, 5):
        with pytest.raises(cvs.CVSError) as e:
            cvs.filters.bayer_to_bgr(bad, a, w, o, w, h, st)
        assert e.value.status == 1
    buf[:w * h] = torch.from_numpy(np.random.default_rng(3).integers(0, 256, w * h, dtype=np.uint8)).cuda()
    cvs.filters.bayer_to_bgr(B.RGGB, a, w, o, w, h, st)
    torch.cuda.synchronize()
    want = B.bayer_to_bgr(B.RGGB, buf[:w * h].cpu().numpy().reshape(h, w)).reshape(-1)
    assert np.array_equal(out[:3 * w * h].cpu().numpy(), want)
