"""Raw YUV cameras on the GPU: cvs_yuv_to_bgr_device is cv2.cvtColor byte for byte (every (Y, U, V) triple, camera and odd
sizes, pitched planes, nothing written outside the frame), and cvs_submit_yuv / cvs_submit_yuv_wire deliver what
cvs_submit_io / cvs_submit_wire deliver for the converted frames -- and what the CPU oracle computes -- in every display
mode, with the noise filter and the overlay, from pinned and pageable memory, interleaved with raw and JPEG tickets, and
at 3840x2160.  Refused submissions leave the handle as it was."""
import ctypes as C
import os

import numpy as np
import pytest

import yuv_ref as Y
from util import CHARS_STR, glyph_atlas

pytestmark = pytest.mark.gpu
FORMATS = [Y.YUYV, Y.NV12, Y.I420]
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
GUARD = 64


def _row_bytes(fmt, w):
    return [2 * w] if fmt == Y.YUYV else ([w, w] if fmt == Y.NV12 else [w, w // 2, w // 2])


def _device_convert(cvs, torch, fmt, buf, w, h, extra_pitch=0):
    """Each plane in an allocation of its own, rows at a pitch of the row bytes rounded up to 16 (+ extra_pitch), the
    padding filled with garbage; the output between two guard bands.  Returns the frame [h, w, 3]."""
    Yp, U, V = Y.planes(fmt, buf, w, h)
    if fmt == Y.YUYV:
        srcs = [buf[:2 * w * h].reshape(h, 2 * w)]
    elif fmt == Y.NV12:
        srcs = [Yp, np.stack([U, V], axis=2).reshape(h // 2, w)]
    else:
        srcs = [Yp, U, V]
    planes, pitches, keep = [], [], []
    for src, rb in zip(srcs, _row_bytes(fmt, w)):
        pitch = (rb + 15) // 16 * 16 + extra_pitch
        t = torch.full((src.shape[0], pitch), 0x5A, dtype=torch.uint8, device="cuda")
        t[:, :rb] = torch.from_numpy(np.ascontiguousarray(src)).cuda()
        keep.append(t)
        planes.append(t.data_ptr())
        pitches.append(pitch)
    n = 3 * w * h
    out = torch.full((n + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
    cvs.filters.yuv_to_bgr(fmt, planes, pitches, out.data_ptr() + GUARD, w, h, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert np.all(o[:GUARD] == 0xA5) and np.all(o[GUARD + n:] == 0xA5), "the conversion wrote outside the frame"
    return o[GUARD:GUARD + n].reshape(h, w, 3)


@pytest.mark.parametrize("fmt", FORMATS, ids=Y.NAMES.get)
def test_device_conversion_is_cv2(cvs, fmt):
    cv2 = pytest.importorskip("cv2")
    import torch
    buf, w, h = Y.exhaustive(fmt)
    want = Y.cv2_convert(cv2, fmt, buf, w, h)
    got = _device_convert(cvs, torch, fmt, buf, w, h)
    bad = np.flatnonzero((got != want).any(axis=2))
    assert bad.size == 0, f"all triples: {bad.size} pixels differ, first at {bad[:5]}"
    rng = np.random.default_rng(fmt)
    for w, h in [(2, 2), (6, 4), (34, 10), (1918, 1078), (1920, 1080), (3840, 2160)]:
        buf = rng.integers(0, 256, size=Y.frame_bytes(fmt, w, h), dtype=np.uint8)
        want = Y.cv2_convert(cv2, fmt, buf, w, h)
        for extra in (0, 48):  # tight (rounded to 16) and wider pitches
            got = _device_convert(cvs, torch, fmt, buf, w, h, extra)
            bad = np.flatnonzero((got != want).any(axis=2))
            assert bad.size == 0, f"{w}x{h} pitch +{extra}: {bad.size} pixels differ, first at {bad[:5]}"


def _synth_yuv(oracle, fmt, w, h, nframes, density_ppm, seed):
    """Camera-like YUV frames of a synthetic sequence, and the BGR frames cv2.cvtColor makes of them (base first)."""
    base, frames = oracle.synth_sequence(w, h, nframes, density_ppm, seed)
    yuv = [Y.from_bgr(fmt, f, w, h) for f in [base] + list(frames)]
    bgr = [Y.yuv_to_bgr(fmt, b, w, h).reshape(-1) for b in yuv]
    return yuv, bgr


def _outs(cvs, n, pinned):
    if pinned:
        return [(cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), cvs.alloc_host(n + 32), (C.c_uint * 1)()) for _ in range(4)]
    return [(np.zeros(n + 32, np.uint8), np.zeros(n + 8, np.int32), np.zeros(n + 32, np.uint8), (C.c_uint * 1)()) for _ in range(4)]


def _ptr(b):
    return b.ctypes.data if isinstance(b, np.ndarray) else b.ptr


def _arr(b, dtype=np.uint8):
    return b.view(dtype) if isinstance(b, np.ndarray) else b.array(dtype)


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


@pytest.mark.parametrize("fmt", FORMATS, ids=Y.NAMES.get)
@pytest.mark.parametrize("mode", range(8))
def test_submit_yuv_is_submit_io_of_the_converted_frames(cvs, oracle, fmt, mode):
    """322x182: 3W % 16 != 0, so rows of the conversion take both its vector and its byte path.  Across the eight modes
    every combination of noise filter, overlay text and pinned / pageable buffers occurs once per format."""
    w, h, nframes = 322, 182, 7
    n = 3 * w * h
    noise, text, pinned = mode % 2 == 1, "FPS: 30" if mode % 4 < 2 else "", mode < 4
    yuv, bgr = _synth_yuv(oracle, fmt, w, h, nframes, 60000, seed=11 * mode + fmt)
    k = oracle.gaussian_kernel(3, 1.2)
    g = glyph_atlas()
    cfg = dict(mode=mode, glyphs=g, glyph_w=7, glyph_h=5, glyph_chars=CHARS_STR)
    if noise:
        cfg.update(noise_filter=True, ksize=3, kweights=k)
    sy, sr = cvs.Stream(w, h, bgr[0], **cfg), cvs.Stream(w, h, bgr[0], **cfg)
    ins = []
    for b in yuv[1:]:
        if pinned:
            hb = cvs.alloc_host(b.size + 64)
            hb.array()[:b.size] = b
            ins.append(hb)
        else:
            ins.append(b.copy())
    raws = []
    for f in bgr[1:]:
        if pinned:
            hb = cvs.alloc_host(n + 64)
            hb.array()[:n] = f
            raws.append(hb)
        else:
            raws.append(f.copy())
    got = _run(sy, ins, lambda f, d, sh, t, p, x: sy.submit_yuv_raw(fmt, _ptr(f), d, sh, t, p, x), n, pinned, mode, text, cvs)
    want = _run(sr, raws, lambda f, d, sh, t, p, x: sr.submit_io_raw(_ptr(f), d, sh, t, p, x), n, pinned, mode, text, cvs)
    oc = oracle.OracleCore(w, h, bgr[0], mode=mode, noise_filter=int(noise), K=3, k=k, glyphs=g, gw=7, gh=5, chars=CHARS_STR)
    for t in range(nframes):
        opos, oxs, odiff, oshow, _ = oc.exec_core(bgr[t + 1], text)
        for name, r in (("yuv", got[t]), ("raw", want[t])):
            assert r[0] == opos, f"{name} frame {t}: pos {r[0]} vs {opos}"
            assert np.array_equal(r[1], oxs) and np.array_equal(r[2], odiff), f"{name} frame {t}: payload"
            if mode:
                assert np.array_equal(r[3], oshow), f"{name} frame {t}: display frame"
    assert opos > 0
    assert np.array_equal(sy.reference(), oc.reference()) and np.array_equal(sr.reference(), oc.reference())
    tm = sy.timing()
    assert tm["h2d_us"] > 0 and tm["kernel_us"] > 0
    sy.close()
    sr.close()


@pytest.mark.parametrize("fmt", FORMATS, ids=Y.NAMES.get)
def test_submit_yuv_wire_is_submit_wire_of_the_converted_frames(cvs, oracle, fmt):
    from cudavideostream_b200 import wire
    w, h = 1920, 1080
    n = 3 * w * h
    yuv, bgr = _synth_yuv(oracle, fmt, w, h, 4, 40000, seed=5 + fmt)
    sy, sr = cvs.Stream(w, h, bgr[0]), cvs.Stream(w, h, bgr[0])
    wy, wr = cvs.alloc_host(wire.bound(w, h) + 64), cvs.alloc_host(wire.bound(w, h) + 64)
    inp, raw = cvs.alloc_host(2 * w * h + 64), cvs.alloc_host(n + 64)
    pageable = np.zeros(wire.bound(w, h) + 64, np.uint8)
    for t in range(1, 5):
        inp.array()[:yuv[t].size] = yuv[t]
        raw.array()[:n] = bgr[t]
        # (the YUV side alternates between a pinned and a pageable output buffer: pushed by the device / copied in cvs_wait)
        out, optr = (wy.array(), wy.ptr) if t % 2 else (pageable, pageable.ctypes.data)
        sy.wait(sy.submit_yuv_wire_raw(fmt, inp.ptr, optr, None, ""))
        sr.wait(sr.submit_wire_raw(raw.ptr, wr.ptr, None, ""))
        a, b = out, wr.array()
        size = wire.size_of(b)
        assert size > 16 and wire.size_of(a) == size and np.array_equal(a[:size], b[:size]), f"frame {t}"
    assert np.array_equal(sy.reference(), sr.reference())
    sy.close()
    sr.close()


def test_yuv_raw_and_jpeg_tickets_interleave(cvs, oracle, monkeypatch):
    """One handle, tickets of all three ingest forms in flight together: each delivers what the oracle computes on the
    BGR frame it stands for, in submission order."""
    monkeypatch.setenv("CVS_JPEG_DECODER", "own")
    z = np.load(os.path.join(GOLDEN, "jpeg_cases.npz"))
    name = "q90_422_320x240"
    jpg = z[name + "/jpg"].tobytes()
    w, h = (int(v) for v in z[name + "/wh"])
    n = 3 * w * h
    jb = cvs.alloc_host(len(jpg) + 64)
    jb.array()[:len(jpg)] = np.frombuffer(jpg, dtype=np.uint8)
    jbgr = oracle.jpeg_decode_bgr(jpg).reshape(-1)
    yn, bn = _synth_yuv(oracle, Y.NV12, w, h, 6, 50000, seed=8)
    yy, by = _synth_yuv(oracle, Y.YUYV, w, h, 6, 50000, seed=9)
    yi, bi = _synth_yuv(oracle, Y.I420, w, h, 6, 50000, seed=10)
    seq = []  # in submission order
    for t in range(1, 7):
        seq += [("nv12", yn[t], bn[t]), ("raw", None, by[t]), ("jpeg", None, jbgr), ("yuyv", yy[t], by[t]), ("i420", yi[t], bi[t])]
    s = cvs.Stream(w, h, bn[0])
    oc = oracle.OracleCore(w, h, bn[0])
    bufs = [(cvs.alloc_host(n + 64), cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()) for _ in range(4)]
    pending = []
    for i, (kind, yb, f) in enumerate(seq):
        if len(pending) == 4:
            tk, (_, d, x, pb), ff = pending.pop(0)
            s.wait(tk)
            opos, oxs, odiff, _, _ = oc.exec_core(ff)
            assert pb[0] == opos and np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs)
        ib, d, x, pb = bufs[i % 4]
        if kind == "raw":
            ib.array()[:n] = f
            tk = s.submit_io_raw(ib.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        elif kind == "jpeg":
            tk = s.submit_jpeg_raw(jb.ptr, len(jpg), d.ptr, None, "", C.addressof(pb), x.ptr)
        else:
            ib.array()[:yb.size] = yb
            tk = s.submit_yuv_raw({"nv12": Y.NV12, "yuyv": Y.YUYV, "i420": Y.I420}[kind], ib.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        pending.append((tk, bufs[i % 4], f))
    for tk, (_, d, x, pb), ff in pending:
        s.wait(tk)
        opos, oxs, odiff, _, _ = oc.exec_core(ff)
        assert pb[0] == opos and np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs)
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


@pytest.mark.parametrize("fmt", [Y.NV12, Y.YUYV], ids=Y.NAMES.get)
def test_4k_stream(cvs, oracle, fmt):
    """3840x2160 does not fit one pass of the stream kernel: the single-frame path walks it in segments."""
    w, h = 3840, 2160
    n = 3 * w * h
    yuv, bgr = _synth_yuv(oracle, fmt, w, h, 3, 20000, seed=4)
    s = cvs.Stream(w, h, bgr[0], mode=cvs.MODE_HEAT_MAP)
    oc = oracle.OracleCore(w, h, bgr[0], mode=1)
    inp = cvs.alloc_host(yuv[1].size + 64)
    d, x, sh, pb = cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), cvs.alloc_host(n + 32), (C.c_uint * 1)()
    for t in range(1, 4):
        inp.array()[:yuv[t].size] = yuv[t]
        s.wait(s.submit_yuv_raw(fmt, inp.ptr, d.ptr, sh.ptr, "", C.addressof(pb), x.ptr))
        opos, oxs, odiff, oshow, _ = oc.exec_core(bgr[t])
        assert pb[0] == opos > 0, f"frame {t}"
        assert np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs), f"frame {t}"
        assert np.array_equal(sh.array()[:n], oshow), f"frame {t}: heat map"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_refusals_leave_the_handle_as_it_was(cvs, oracle):
    lib = cvs.load_library()
    w, h = 64, 48
    n = 3 * w * h
    yuv, bgr = _synth_yuv(oracle, Y.NV12, w, h, 3, 80000, seed=2)
    s = cvs.Stream(w, h, bgr[0])
    oc = oracle.OracleCore(w, h, bgr[0])
    inp, d, x, pb = cvs.alloc_host(2 * n), cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()
    tk = C.c_uint64(0)
    wout = cvs.alloc_host(cvs.wire.bound(w, h) + 64)

    def good(t):
        inp.array()[:yuv[t].size] = yuv[t]
        ticket = s.submit_yuv_raw(Y.NV12, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
        s.wait(ticket)
        opos, oxs, odiff, _, _ = oc.exec_core(bgr[t])
        assert pb[0] == opos and np.array_equal(d.array()[:opos], odiff) and np.array_equal(x.array(np.int32)[:opos], oxs)
        return ticket

    last = good(1)
    ref = s.reference()
    h_ = s._h
    refusals = [
        lib.cvs_submit_yuv(h_, 0, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_yuv(h_, 4, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_yuv(h_, Y.NV12, None, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_yuv(h_, Y.NV12, inp.ptr, None, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_yuv(h_, Y.NV12, inp.ptr, d.ptr, None, b"", None, x.ptr, C.byref(tk)),
        lib.cvs_submit_yuv(h_, Y.NV12, inp.ptr, d.ptr, None, b"", C.addressof(pb), None, C.byref(tk)),
        lib.cvs_submit_yuv(h_, Y.NV12, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, None),
        lib.cvs_submit_yuv(None, Y.NV12, inp.ptr, d.ptr, None, b"", C.addressof(pb), x.ptr, C.byref(tk)),
        lib.cvs_submit_yuv_wire(h_, 9, inp.ptr, wout.ptr, None, b"", C.byref(tk)),
        lib.cvs_submit_yuv_wire(h_, Y.I420, None, wout.ptr, None, b"", C.byref(tk)),
        lib.cvs_submit_yuv_wire(h_, Y.I420, inp.ptr, None, None, b"", C.byref(tk)),
        lib.cvs_submit_yuv_wire(h_, Y.I420, inp.ptr, wout.ptr, None, b"", None),
    ]
    assert refusals == [1] * len(refusals)
    assert np.array_equal(s.reference(), ref)
    assert good(2) == last + 1  # no ticket was consumed
    # sizes a format forbids: odd width (every format), odd height (the 4:2:0 ones)
    for (ww, hh), bad in (((63, 48), FORMATS), ((64, 47), [Y.NV12, Y.I420])):
        so = cvs.Stream(ww, hh, np.zeros(3 * ww * hh, np.uint8))
        for fmt in bad:
            with pytest.raises(cvs.CVSError) as e:
                so.submit_yuv_raw(fmt, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
            assert e.value.status == 1
        if (ww, hh) == (64, 47):  # YUYV takes an odd height
            so.wait(so.submit_yuv_raw(Y.YUYV, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr))
        so.close()
    # a fifth ticket while four are outstanding
    tks = []
    inp.array()[:yuv[3].size] = yuv[3]
    outs = [(cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()) for _ in range(4)]
    for dd, xx, pp in outs:
        tks.append(s.submit_yuv_raw(Y.NV12, inp.ptr, dd.ptr, None, "", C.addressof(pp), xx.ptr))
    with pytest.raises(cvs.CVSError) as e:
        s.submit_yuv_raw(Y.NV12, inp.ptr, d.ptr, None, "", C.addressof(pb), x.ptr)
    assert e.value.status == 1
    for t, (dd, xx, pp) in zip(tks, outs):
        s.wait(t)
        opos, oxs, odiff, _, _ = oc.exec_core(bgr[3])
        assert pp[0] == opos and np.array_equal(dd.array()[:opos], odiff)
    assert tks == [last + 2 + i for i in range(4)]
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_device_conversion_alignment_and_pitch(cvs):
    """Refusals of the device entry on real device buffers, then a good call on the same buffers."""
    import torch
    w, h = 64, 32
    buf = torch.zeros(4 * w * h + 64, dtype=torch.uint8, device="cuda")
    out = torch.zeros(3 * w * h + 64, dtype=torch.uint8, device="cuda")
    a, o = buf.data_ptr(), out.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    cases = [((Y.NV12, [a + 8, a + w * h], [w, w]), 4), ((Y.NV12, [a, a + w * h], [w + 4, w]), 4),
             ((Y.I420, [a, a + w * h, a + w * h + 512], [w, 16, 32]), 1), ((Y.YUYV, [a], [2 * w - 16]), 1)]
    for (fmt, pl, pi), status in cases:
        with pytest.raises(cvs.CVSError) as e:
            cvs.filters.yuv_to_bgr(fmt, pl, pi, o, w, h, st)
        assert e.value.status == status
    with pytest.raises(cvs.CVSError) as e:
        cvs.filters.yuv_to_bgr(Y.YUYV, [a], [2 * w], o + 4, w, h, st)
    assert e.value.status == 4
    cvs.filters.yuv_to_bgr(Y.I420, [a, a + w * h, a + w * h + 512], [w, 32, 32], o, w, h, st)
    torch.cuda.synchronize()
    want = Y.yuv_to_bgr(Y.I420, np.zeros(Y.frame_bytes(Y.I420, w, h), np.uint8), w, h).reshape(-1)
    assert np.array_equal(out[:3 * w * h].cpu().numpy(), want)
