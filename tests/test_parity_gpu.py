"""Parity of the CUDA path (through the C ABI) against the CPU oracle: bit-exact change mask, payload order
and values, new reference, and every display filter.  Needs a B200."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from util import CHARS_STR, glyph_atlas, random_sequence

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

# sizes: pixel-group tail (N % 48 != 0), rows not a multiple of 4 bytes, exactly one group, tiny, multi-block
SIZES = [(7, 5), (16, 1), (1, 1), (33, 9), (64, 48), (250, 130), (641, 359)]


def _check_frames(cvs, oracle, w, h, base, frames, text="", **cfg):
    okw = dict(thr=cfg.get("threshold", 20), mode=cfg.get("mode", 0), noise_filter=int(cfg.get("noise_filter", 0)),
               K=cfg.get("ksize", 3), k=cfg.get("kweights"), glyphs=cfg.get("glyphs"), gw=cfg.get("glyph_w", 0),
               gh=cfg.get("glyph_h", 0), chars=CHARS_STR if cfg.get("glyphs") is not None else "")
    core = oracle.OracleCore(w, h, base, **okw)
    s = cvs.Stream(w, h, base, **cfg)
    try:
        for t, f in enumerate(frames):
            pos, xs, diff, show, _ = core.exec_core(f, text)
            gpos, gxs, gdiff, gshow = s.exec(f, text)
            assert gpos == pos, f"frame {t}: pos {gpos} != {pos}"
            assert np.array_equal(gxs, xs), f"frame {t}: xs differ"
            assert np.array_equal(gdiff, diff), f"frame {t}: diff bytes differ"
            if cfg.get("mode", 0):
                bad = np.flatnonzero(gshow != show)
                assert bad.size == 0, f"frame {t}: show differs at {bad[:8]} ({gshow[bad[:8]]} vs {show[bad[:8]]})"
            assert np.array_equal(s.reference(), core.reference()), f"frame {t}: reference differs"
    finally:
        s.close()
        core.close()


@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("density", [0.0, 0.01, 0.5, 1.0])
def test_diff_compact_small(cvs, oracle, w, h, density):
    base, frames = random_sequence(w, h, 4, density, seed=w * 1000 + h)
    _check_frames(cvs, oracle, w, h, base, frames)


def test_threshold_edges(cvs, oracle):
    # df = +-20 unchanged, +-21 changed; wrap cases 0 vs 255
    w, h = 16, 2
    base = np.full(3 * w * h, 100, dtype=np.uint8)
    f = base.copy()
    f[0], f[1], f[2], f[3] = 120, 121, 80, 79
    base[4], f[4] = 255, 0
    base[5], f[5] = 0, 255
    _check_frames(cvs, oracle, w, h, base, [f, f, base])
    s = cvs.Stream(w, h, base)
    pos, xs, diff, _ = s.exec(f)
    assert xs.tolist() == [1, 3, 4, 5] and diff.tolist() == [21, 235, 1, 255]
    s.close()


@pytest.mark.parametrize("thr", [-1, 0, 1, 20, 127, 128, 200, 254, 255])
def test_threshold_values(cvs, oracle, thr):
    base, frames = random_sequence(40, 30, 2, 0.3, seed=thr + 7)
    frames[1] = np.random.default_rng(thr + 1).integers(0, 256, size=frames[1].size, dtype=np.uint8)
    _check_frames(cvs, oracle, 40, 30, base, frames, threshold=thr)


@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5, 6, 7])
@pytest.mark.parametrize("w,h", [(7, 5), (64, 48), (250, 130)])
def test_display_modes(cvs, oracle, mode, w, h):
    base, frames = random_sequence(w, h, 3, 0.1, seed=mode)
    _check_frames(cvs, oracle, w, h, base, frames, mode=mode)


def test_gray_weighted_exact_products(cvs, oracle):
    # pixels whose weighted sum is an exact integer in real arithmetic (114B+587G+299R = 0 mod 1000) are
    # where double rounding decides the truncation
    px = [(b, g, r) for b in range(256) for g in range(0, 256, 5) for r in range(0, 256, 3)
          if (114 * b + 587 * g + 299 * r) % 1000 == 0]
    px = np.array(px, dtype=np.uint8)
    n = (len(px) // 16) * 16
    w, h = 16, n // 16
    frame = px[:n].reshape(-1)
    base = np.zeros_like(frame)
    _check_frames(cvs, oracle, w, h, base, [frame], mode=4)
    _check_frames(cvs, oracle, w, h, base, [frame], mode=5)


@pytest.mark.parametrize("kind", ["gauss", "mean"])
@pytest.mark.parametrize("w,h", [(3, 3), (33, 9), (64, 48), (250, 130)])
def test_noise_filter_then_diff(cvs, oracle, kind, w, h):
    k = oracle.gaussian_kernel(3, 1.5) if kind == "gauss" else oracle.mean_kernel(3)
    base, frames = random_sequence(w, h, 3, 0.2, seed=5)
    _check_frames(cvs, oracle, w, h, base, frames, noise_filter=True, ksize=3, kweights=k)


@pytest.mark.parametrize("K", [1, 5, 7, 9])
def test_noise_filter_other_k(cvs, oracle, K):
    k = oracle.gaussian_kernel(K, K * K / 6.0)
    base, frames = random_sequence(64, 40, 2, 0.2, seed=K)
    _check_frames(cvs, oracle, 64, 40, base, frames, noise_filter=True, ksize=K, kweights=k, mode=5)


def test_k2_report_matrices_on_gpu(cvs):
    # REPORT/report.tex:2351-2378 through the CUDA noise filter
    import torch
    A = np.array([[120, 131, 112], [112, 101, 82], [44, 106, 65]], dtype=np.uint8)
    want = np.array([[51, 73, 47], [68, 96, 66], [40, 56, 39]], dtype=np.uint8)
    img = np.repeat(A.reshape(3, 3, 1), 3, axis=2).reshape(-1)
    d_in = torch.zeros(64, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(64, dtype=torch.uint8, device="cuda")
    d_in[:27] = torch.from_numpy(img).cuda()
    cvs.filters.noise_filter(d_in.data_ptr(), d_out.data_ptr(), 3, 3, 3, np.full(9, 1.0 / 9, dtype=np.float32),
                             torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = d_out[:27].cpu().numpy().reshape(3, 3, 3)
    for ch in range(3):
        assert np.array_equal(got[:, :, ch], want)


def test_text_overlay(cvs, oracle):
    gw, gh = 7, 5
    atlas = glyph_atlas(gw, gh)
    w, h = 64, 48
    base, frames = random_sequence(w, h, 3, 0.05, seed=9)
    for text in ["FPS 26", "0123456789", "zz?FPS", "BW:12/3 kbps WWWWWWWWWWWWWWWWWWWW"]:
        _check_frames(cvs, oracle, w, h, base, frames, text=text, glyphs=atlas, glyph_w=gw, glyph_h=gh, mode=4)


def test_cudacore_mirror_inplace_semantics(cvs, oracle):
    # exec_core overwrites the head of the frame buffer with the diff bytes and leaves the tail alone
    # (kernels.cu:522); buffers come from alloc_arrays (pinned)
    from cudavideostream_b200.api import CUDACore, matsz
    w, h = 96, 64
    base, frames = random_sequence(w, h, 3, 0.1, seed=11)
    core = CUDACore(None, None, None, 3 * w * h, base, matsz(h, w))
    oc = oracle.OracleCore(w, h, base)
    h_frame, n_frame, o_frame, h_xs = CUDACore.alloc_arrays(h, w)
    for f in frames:
        h_frame.array()[: f.size] = f
        pos = core.exec_core(h_frame, None, "", h_xs)
        opos, oxs, odiff, _, after = oc.exec_core(f)
        assert pos == opos
        assert np.array_equal(h_frame.array()[: f.size], after)
        assert np.array_equal(h_xs.array(np.int32)[:pos], oxs)
    assert core.chunkt_size() == 32


def test_submit_wait_pipeline(cvs, oracle):
    w, h = 200, 120
    base, frames = random_sequence(w, h, 7, 0.1, seed=13)
    n = 3 * w * h
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    bufs = [(cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()) for _ in range(2)]
    tickets = []
    for t, f in enumerate(frames):
        fb, xb, pb = bufs[t % 2]
        if len(tickets) == 2:
            tk, tt = tickets.pop(0)
            s.wait(tk)
            ofb, oxb, opb = bufs[tt % 2]
            opos, oxs, odiff, _, _ = oc.exec_core(frames[tt])
            assert opb[0] == opos
            assert np.array_equal(ofb.array()[:opos], odiff) and np.array_equal(oxb.array(np.int32)[:opos], oxs)
        fb.array()[:n] = f
        tickets.append((s.submit_raw(fb.ptr, None, "", C.addressof(pb), xb.ptr), t))
    for tk, tt in tickets:
        s.wait(tk)
        ofb, oxb, opb = bufs[tt % 2]
        opos, oxs, odiff, _, _ = oc.exec_core(frames[tt])
        assert opb[0] == opos
        assert np.array_equal(ofb.array()[:opos], odiff) and np.array_equal(oxb.array(np.int32)[:opos], oxs)
    assert np.array_equal(s.reference(), oc.reference())
    tm = s.timing()
    assert tm["h2d_us"] > 0 and tm["kernel_us"] > 0
    s.close()


class _Pageable:
    """Ordinary host memory with HostBuffer's interface: not mapped, so the payload arrives by copies."""

    def __init__(self, nbytes):
        self.buf = np.zeros(nbytes, dtype=np.uint8)
        self.ptr = self.buf.ctypes.data

    def array(self, dtype=np.uint8):
        return self.buf.view(dtype)


@pytest.mark.parametrize("buffers", ["pinned", "pageable"])
def test_submit_io_jumping_density(cvs, oracle, buffers):
    """cvs_submit_io keeps the input frame intact and copies a PREDICTED payload size behind the count: frames whose
    count jumps far above / falls far below the prediction must still deliver exactly [0, pos).  Outside the prediction
    window the payload is pushed into pinned buffers by a kernel, and copied in cvs_wait into pageable ones."""
    w, h = 320, 180
    n = 3 * w * h
    rng = np.random.default_rng(77)
    base = rng.integers(0, 256, n, dtype=np.uint8)
    # the predicted copy is used when the previous count lies in [N/64, N/4]: 0.05 -> 0.9 under-predicts (remainder
    # copy), 0.1 -> 0.0 over-predicts, 0.05 -> 0.06 is the normal case
    dens = [0.001, 0.05, 0.9, 0.0, 0.1, 0.0, 0.3, 1.0, 0.05, 0.06, 0.2, 0.002, 0.6, 0.05, 0.0, 0.45]
    frames, cur = [], base.copy()
    for d in dens:
        nxt = cur.copy()
        idx = np.flatnonzero(rng.random(n) < d)
        nxt[idx] = (nxt[idx].astype(np.int64) + rng.integers(40, 200, idx.size)).astype(np.uint8)
        frames.append(nxt)
        cur = nxt
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    ring = cvs.alloc_host(len(frames) * n)
    for t, f in enumerate(frames):
        ring.array()[t * n:(t + 1) * n] = f
    alloc = cvs.alloc_host if buffers == "pinned" else _Pageable
    bufs = [(alloc(n + 32), alloc(4 * n + 32), (C.c_uint * 1)()) for _ in range(4)]

    def check(tt):
        ofb, oxb, opb = bufs[tt % 4]
        opos, oxs, odiff, _, _ = oc.exec_core(frames[tt])
        assert opb[0] == opos, f"frame {tt}: pos {opb[0]} != {opos}"
        assert np.array_equal(ofb.array()[:opos], odiff), f"frame {tt}: diff bytes differ"
        assert np.array_equal(oxb.array(np.int32)[:opos], oxs), f"frame {tt}: xs differ"

    tickets = []
    for t in range(len(frames)):
        if len(tickets) == 4:
            tk, tt = tickets.pop(0)
            s.wait(tk)
            check(tt)
        fb, xb, pb = bufs[t % 4]
        tickets.append((s.submit_io_raw(ring.ptr + t * n, fb.ptr, None, "", C.addressof(pb), xb.ptr), t))
    for tk, tt in tickets:
        s.wait(tk)
        check(tt)
    # the captured frames were not touched
    for t, f in enumerate(frames):
        assert np.array_equal(ring.array()[t * n:(t + 1) * n], f)
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_golden_real_camera_crop(cvs):
    # 128x72 crop of the reference's own fixture frames f1.jpg/f2.jpg with the oracle payload recorded in the
    # build container (tests/golden/make_golden.py)
    g = np.load(os.path.join(GOLDEN, "k1_crop.npz"))
    f1, f2 = g["f1"], g["f2"]
    s = cvs.Stream(128, 72, f1)
    pos, xs, diff, _ = s.exec(f2)
    with open(os.path.join(GOLDEN, "k1_f1_f2.json")) as f:
        assert pos == json.load(f)["crop"]["changed_bytes"]
    assert np.array_equal(xs, g["xs"]) and np.array_equal(diff, g["diff"])
    assert np.array_equal(s.reference(), g["new_reference"])
    s.close()


@pytest.mark.parametrize("w,h", [(1, 1), (5, 1), (3, 3)])
def test_submit_io_tiny_frames_stay_inside_the_buffers(cvs, oracle, w, h):
    # N not a multiple of 4: neither the push nor a speculative copy may touch anything past N bytes / N ints of
    # the caller's buffers (guard words behind them must survive), first frame and later frames alike
    n = 3 * w * h
    rng = np.random.default_rng(n)
    base = rng.integers(0, 256, n, dtype=np.uint8)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    fin = cvs.alloc_host(n + 64)
    dout = cvs.alloc_host(n + 64)
    xout = cvs.alloc_host(4 * n + 64)
    pb = (C.c_uint * 1)()
    for t in range(6):
        f = rng.integers(0, 256, n, dtype=np.uint8)
        fin.array()[:n] = f
        dout.array()[:] = 0xA5
        xout.array()[:] = 0xA5
        tk = s.submit_io_raw(fin.ptr, dout.ptr, None, "", C.addressof(pb), xout.ptr)
        s.wait(tk)
        opos, oxs, odiff, _, _ = oc.exec_core(f)
        assert pb[0] == opos
        assert np.array_equal(dout.array()[:opos], odiff) and np.array_equal(xout.array(np.int32)[:opos], oxs)
        assert bool((dout.array()[n:] == 0xA5).all()), f"frame {t}: write past diff_out[N]"
        assert bool((xout.array()[4 * n:] == 0xA5).all()), f"frame {t}: write past xs[N]"
        assert np.array_equal(fin.array()[:n], f)
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


def test_long_sequence_is_walked_in_pieces(cvs, oracle):
    # nframes > max_sequence: the whole chain (noise filter + overlay pre-pass, stream kernel, binarisation pass 2)
    # runs piece by piece on scratch sized by the piece
    import torch
    w, h, T = 64, 48, 11
    n = 3 * w * h
    stride = (n + 15) // 16 * 16
    k = oracle.gaussian_kernel(3, 1.5)
    atlas = glyph_atlas(7, 5)
    base, frames = random_sequence(w, h, T, 0.1, seed=4)
    d_frames = torch.zeros(T * stride + 64, dtype=torch.uint8, device="cuda")
    for t in range(T):
        d_frames[t * stride:t * stride + n] = torch.from_numpy(frames[t]).cuda()
    cap = (n + 3) // 4 * 4
    d_pos = torch.zeros(T, dtype=torch.int32, device="cuda")
    d_xs = torch.empty(T * cap, dtype=torch.int32, device="cuda")
    d_diff = torch.empty(T * cap, dtype=torch.uint8, device="cuda")
    d_show = torch.zeros(T * stride, dtype=torch.uint8, device="cuda")
    s = cvs.Stream(w, h, base, mode=5, noise_filter=True, ksize=3, kweights=k, glyphs=atlas, glyph_w=7, glyph_h=5,
                   max_sequence=4)
    s.run_sequence_device(d_frames.data_ptr(), stride, T, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(), cap,
                          d_show.data_ptr(), stride, text="FPS 12", cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s.sequence_status()
    oc = oracle.OracleCore(w, h, base, mode=5, noise_filter=1, K=3, k=k, glyphs=atlas, gw=7, gh=5, chars=CHARS_STR)
    for t in range(T):
        opos, oxs, odiff, oshow, _ = oc.exec_core(frames[t], "FPS 12")
        assert int(d_pos[t]) == opos, f"frame {t}"
        assert np.array_equal(d_xs[t * cap:t * cap + opos].cpu().numpy(), oxs), f"frame {t}"
        assert np.array_equal(d_diff[t * cap:t * cap + opos].cpu().numpy(), odiff), f"frame {t}"
        assert np.array_equal(d_show[t * stride:t * stride + n].cpu().numpy(), oshow), f"frame {t}: show"
        # the caller's frames are never modified (the overlay goes into a private copy)
        assert np.array_equal(d_frames[t * stride:t * stride + n].cpu().numpy(), frames[t])
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
