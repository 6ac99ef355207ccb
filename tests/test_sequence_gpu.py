"""Device-resident sequences (the path bench.py times), full-size frames and size-independent properties."""
import numpy as np
import pytest

from util import random_sequence

pytestmark = pytest.mark.gpu


def _run_sequence(cvs, torch, w, h, base, frames_np=None, d_frames=None, nframes=None, cap=None, mode=0, **cfg):
    n = 3 * w * h
    stride = (n + 15) // 16 * 16
    if d_frames is None:
        nframes = frames_np.shape[0]
        d_frames = torch.zeros(nframes * stride + 64, dtype=torch.uint8, device="cuda")
        for t in range(nframes):
            d_frames[t * stride: t * stride + n] = torch.from_numpy(frames_np[t]).cuda()
    cap = cap or (n + 3) // 4 * 4
    d_pos = torch.zeros(nframes, dtype=torch.int32, device="cuda")
    d_xs = torch.empty(nframes * cap, dtype=torch.int32, device="cuda")
    d_diff = torch.empty(nframes * cap, dtype=torch.uint8, device="cuda")
    d_show = torch.zeros(nframes * stride, dtype=torch.uint8, device="cuda") if mode else None
    s = cvs.Stream(w, h, base, mode=mode, **cfg)
    s.run_sequence_device(d_frames.data_ptr(), stride, nframes, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(),
                          cap, d_show.data_ptr() if mode else 0, stride,
                          cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return s, d_pos, d_xs, d_diff, d_show, cap, stride


@pytest.mark.parametrize("w,h,nframes", [(7, 5, 5), (64, 48, 9), (641, 359, 6)])
@pytest.mark.parametrize("mode", [0, 1, 3, 5])
def test_sequence_matches_oracle(cvs, oracle, w, h, nframes, mode):
    import torch
    base, frames = random_sequence(w, h, nframes, 0.08, seed=w + mode)
    s, d_pos, d_xs, d_diff, d_show, cap, stride = _run_sequence(cvs, torch, w, h, base, frames, mode=mode)
    s.sequence_status()
    oc = oracle.OracleCore(w, h, base, mode=mode)
    pos = d_pos.cpu().numpy()
    n = 3 * w * h
    for t in range(nframes):
        opos, oxs, odiff, oshow, _ = oc.exec_core(frames[t])
        assert pos[t] == opos, f"frame {t}"
        assert np.array_equal(d_xs[t * cap: t * cap + opos].cpu().numpy(), oxs), f"frame {t}"
        assert np.array_equal(d_diff[t * cap: t * cap + opos].cpu().numpy(), odiff), f"frame {t}"
        if mode:
            assert np.array_equal(d_show[t * stride: t * stride + n].cpu().numpy(), oshow), f"frame {t}"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


@pytest.mark.parametrize("form", ["split", "fused"])
@pytest.mark.parametrize("w,h,nframes,mode,noise", [(7, 5, 4, 5, False), (250, 130, 5, 7, False), (641, 359, 4, 5, True),
                                                    (333, 77, 3, 7, True)])
def test_binarising_sequences_split_and_fused(cvs, oracle, form, w, h, nframes, mode, noise):
    """Modes 5 / 7: a sequence computes gray + histogram in k_gray_hist_seq in front of the plain stream kernel (split),
    a single frame inside the stream kernel (fused).  The same frames as one sequence or one by one through cvs_exec:
    same payload, same binarised frames (server.cpp:96-135 behind the optional noise filter of kernels.cu:457-459)."""
    import torch
    k = oracle.gaussian_kernel(3, 1.5)
    cfg = dict(noise_filter=True, ksize=3, kweights=k) if noise else {}
    ocfg = dict(noise_filter=1, K=3, k=k) if noise else {}
    base, frames = random_sequence(w, h, nframes, 0.1, seed=3 * w + mode)
    n = 3 * w * h
    if form == "split":
        s, d_pos, d_xs, d_diff, d_show, cap, stride = _run_sequence(cvs, torch, w, h, base, frames, mode=mode, **cfg)
        s.sequence_status()
        pos = d_pos.cpu().numpy()
        got = [(int(pos[t]), d_xs[t * cap: t * cap + pos[t]].cpu().numpy(), d_diff[t * cap: t * cap + pos[t]].cpu().numpy(),
                d_show[t * stride: t * stride + n].cpu().numpy()) for t in range(nframes)]
    else:
        s = cvs.Stream(w, h, base, mode=mode, **cfg)
        got = [s.exec(f) for f in frames]
    oc = oracle.OracleCore(w, h, base, mode=mode, **ocfg)
    for t in range(nframes):
        opos, oxs, odiff, oshow, _ = oc.exec_core(frames[t])
        gpos, gxs, gdiff, gshow = got[t]
        assert gpos == opos, f"frame {t}"
        assert np.array_equal(gxs, oxs), f"frame {t}"
        assert np.array_equal(gdiff, odiff), f"frame {t}"
        assert np.array_equal(gshow, oshow), f"frame {t}: binarised frame"
    assert np.array_equal(s.reference(), oc.reference())
    # the split form is one launch more per piece (noise filter?, gray + histogram, stream kernel, threshold, binarize)
    # than the fused form is per frame (noise filter?, stream kernel, threshold, binarize)
    assert s.launch_count() == (4 + int(noise) if form == "split" else nframes * (3 + int(noise)))
    s.close()


def test_sequence_capacity_overflow_is_reported(cvs):
    import torch
    w, h = 64, 48
    base, frames = random_sequence(w, h, 3, 0.5, seed=2)
    s, d_pos, *_ = _run_sequence(cvs, torch, w, h, base, frames, cap=64)
    with pytest.raises(cvs.CVSError) as e:
        s.sequence_status()
    assert e.value.status == 5  # CVS_ERR_CAPACITY
    assert int(d_pos[0]) > 64   # the true count is still reported
    s.sequence_status()         # sticky bit cleared after being reported
    s.close()


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160), (1919, 1079)])
def test_full_size_pair_matches_oracle(cvs, oracle, w, h):
    # BASELINE.json configs[0]: one synthetic frame pair at full size, CUDA vs the CPU oracle
    base = cvs.synth.base_frame(w, h)
    f1 = cvs.synth.next_frame(base, cvs.synth.DEFAULT_SEED, 0, 100000)
    f2 = cvs.synth.next_frame(f1, cvs.synth.DEFAULT_SEED, 1, 10000)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    for f in (f1, f2):
        pos, xs, diff, _ = s.exec(f)
        opos, oxs, odiff, _, _ = oc.exec_core(f)
        assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff)
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


@pytest.mark.parametrize("mode", [1, 2, 4, 5])
def test_full_size_display_modes(cvs, oracle, mode):
    w, h = 1920, 1080
    base = cvs.synth.base_frame(w, h)
    f1 = cvs.synth.next_frame(base, 7, 0, 100000)
    s = cvs.Stream(w, h, base, mode=mode)
    oc = oracle.OracleCore(w, h, base, mode=mode)
    pos, xs, diff, show = s.exec(f1)
    opos, oxs, odiff, oshow, _ = oc.exec_core(f1)
    assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff)
    assert np.array_equal(show, oshow)
    s.close()


def test_full_size_noise_filter_binarize(cvs, oracle):
    # BASELINE.json configs[2]: noise filter -> diff, weighted gray -> binarize, at 1080p
    w, h = 1920, 1080
    k = oracle.gaussian_kernel(3, 1.5)
    base = cvs.synth.base_frame(w, h)
    f1 = cvs.synth.next_frame(base, 9, 0, 100000)
    s = cvs.Stream(w, h, base, mode=5, noise_filter=True, ksize=3, kweights=k)
    oc = oracle.OracleCore(w, h, base, mode=5, noise_filter=1, K=3, k=k)
    pos, xs, diff, show = s.exec(f1)
    opos, oxs, odiff, oshow, _ = oc.exec_core(f1)
    assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff)
    assert np.array_equal(show, oshow)
    s.close()


def test_synth_device_twin(cvs):
    import torch
    w, h = 250, 130
    n = 3 * w * h
    d0 = torch.empty(n, dtype=torch.uint8, device="cuda")
    d1 = torch.empty(n, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    cvs.synth.base_frame_device(d0.data_ptr(), w, h, 1234, st)
    cvs.synth.next_frame_device(d0.data_ptr(), d1.data_ptr(), w, h, 1234, 5, 100000, st)
    torch.cuda.synchronize()
    b = cvs.synth.base_frame(w, h, 1234)
    assert np.array_equal(d0.cpu().numpy(), b)
    assert np.array_equal(d1.cpu().numpy(), cvs.synth.next_frame(b, 1234, 5, 100000))


def test_full_sequence_client_round_trip(cvs):
    # size-independent property at BASELINE's full size (configs[1]): applying every frame's payload to the base
    # frame on the client side (client/opencv.cpp:64-66) reproduces the server's reference frame exactly, the
    # indices of every frame are strictly ascending, and every transmitted value is a real change (> T).
    import torch
    w, h, T = 1920, 1080, 24
    n = 3 * w * h
    stride = n
    st = torch.cuda.current_stream().cuda_stream
    d_frames = torch.empty((T + 1) * stride, dtype=torch.uint8, device="cuda")
    cvs.synth.base_frame_device(d_frames.data_ptr(), w, h, 99, st)
    for t in range(T):
        dens = (10000, 100000, 500000)[t % 3]
        cvs.synth.next_frame_device(d_frames.data_ptr() + t * stride, d_frames.data_ptr() + (t + 1) * stride,
                                    w, h, 99, t, dens, st)
    torch.cuda.synchronize()
    base = d_frames[:n].cpu().numpy()
    s, d_pos, d_xs, d_diff, _, cap, _ = _run_sequence(cvs, torch, w, h, base, d_frames=d_frames[stride:], nframes=T)
    s.sequence_status()
    client = d_frames[:n].clone()
    pos = d_pos.cpu().numpy()
    for t in range(T):
        assert pos[t] > 0
        xs = d_xs[t * cap: t * cap + int(pos[t])]
        assert bool((xs[1:] > xs[:-1]).all()) and int(xs[0]) >= 0 and int(xs[-1]) < n
        before = client[xs.long()].to(torch.int16)
        cvs.filters.client_apply(client.data_ptr(), d_xs.data_ptr() + 4 * t * cap, d_diff.data_ptr() + t * cap,
                                 d_pos.data_ptr() + 4 * t, cap, st)
        torch.cuda.synchronize()
        after = client[xs.long()].to(torch.int16)
        assert bool(((after - before).abs() > 20).all())
    ref = torch.from_numpy(s.reference()).cuda()
    assert bool((client == ref).all())
    # and the reference never drifts more than T away from the last frame
    last = d_frames[T * stride: T * stride + n].to(torch.int16)
    assert int((last - ref.to(torch.int16)).abs().max()) <= 20
    s.close()


def test_standalone_filters(cvs, oracle):
    import torch
    w, h = 250, 130
    n, p = 3 * w * h, w * h
    base, frames = random_sequence(w, h, 1, 0.2, seed=21)
    pad = lambda a, m: torch.cat([torch.from_numpy(a).cuda(), torch.zeros(m, dtype=torch.uint8, device="cuda")])
    d_a, d_b = pad(base, 64), pad(frames[0], 64)
    d_o = torch.zeros(n + 64, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    cvs.filters.heat_map(d_a.data_ptr(), d_b.data_ptr(), d_o.data_ptr(), w, h, st)
    assert np.array_equal(d_o[:n].cpu().numpy(), oracle.heat_map(base, frames[0], w, h))
    cvs.filters.red_map(d_a.data_ptr(), d_b.data_ptr(), d_o.data_ptr(), w, h, 20, st)
    assert np.array_equal(d_o[:n].cpu().numpy(), oracle.red_map(base, frames[0], w, h, 20))
    cvs.filters.grayscale(d_b.data_ptr(), d_o.data_ptr(), w, h, True, 3, st)
    assert np.array_equal(d_o[:n].cpu().numpy(), oracle.gray_weighted3(frames[0]))
    cvs.filters.grayscale(d_b.data_ptr(), d_o.data_ptr(), w, h, False, 3, st)
    assert np.array_equal(d_o[:n].cpu().numpy(), oracle.gray_avg3(frames[0]))
    cvs.filters.grayscale(d_b.data_ptr(), d_o.data_ptr(), w, h, True, 1, st)
    assert np.array_equal(d_o[:p].cpu().numpy(), oracle.gray_weighted1(frames[0], w, h))
    cvs.filters.grayscale(d_b.data_ptr(), d_o.data_ptr(), w, h, False, 1, st)
    assert np.array_equal(d_o[:p].cpu().numpy(), oracle.gray_avg1(frames[0], w, h))
    # tests/binarization/cpu.cu variant: weighted gray, clamp "< 20 -> 20" only
    d_g = torch.zeros(p + 64, dtype=torch.uint8, device="cuda")
    d_ht = torch.zeros(257, dtype=torch.int32, device="cuda")
    cvs.filters.binarize(d_b.data_ptr(), d_o.data_ptr(), d_g.data_ptr(), d_ht.data_ptr(), w, h, True, 20, 255, st)
    g1 = oracle.gray_weighted1(frames[0], w, h)
    hist = oracle.histogram1(g1)
    thr = oracle.threshold_twomax(hist, 20, 255)
    ht = d_ht.cpu().numpy()
    assert np.array_equal(ht[:256], hist) and ht[256] == thr
    assert np.array_equal(d_o[:n].cpu().numpy(), oracle.binarize(np.repeat(g1, 3), thr))


@pytest.mark.parametrize("th", [-1, 0, 1, 50, 127, 128, 129, 200, 254, 255, 300])
def test_binarize_pass_at_every_kind_of_threshold(cvs, oracle, th):
    """k_binarize_expand compares four gray bytes at once (carry-free byte compare, two forms for th < 128 and th >= 128);
    clamp_lo = clamp_hi = th forces the frame's threshold: out = gray > th ? 255 : 0 per channel (server.cpp:129-135)."""
    import torch
    w, h = 253, 67  # a tail group (253 * 67 = 16,951 pixels = 1,059 groups + 7 pixels)
    n, p = 3 * w * h, w * h
    rng = np.random.default_rng(100 + th)
    frame = rng.integers(0, 256, size=n, dtype=np.uint8)
    frame[:3 * 256] = np.repeat(np.arange(256, dtype=np.uint8), 3)  # every gray value once (gray of (v, v, v) is v ...
    d_f = torch.cat([torch.from_numpy(frame).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    d_o = torch.full((n + 64,), 0x5A, dtype=torch.uint8, device="cuda")
    d_g = torch.zeros(p + 64, dtype=torch.uint8, device="cuda")
    d_ht = torch.zeros(257, dtype=torch.int32, device="cuda")
    cvs.filters.binarize(d_f.data_ptr(), d_o.data_ptr(), d_g.data_ptr(), d_ht.data_ptr(), w, h, False, th, th,
                         torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    g1 = oracle.gray_avg1(frame, w, h)
    assert np.array_equal(d_g[:p].cpu().numpy(), g1)
    assert int(d_ht[256].item()) == th
    want = np.where(np.repeat(g1, 3).astype(np.int64) > th, 255, 0).astype(np.uint8)
    got = d_o.cpu().numpy()
    assert np.array_equal(got[:n], want)
    assert np.all(got[n:] == 0x5A)


@pytest.mark.parametrize("w,h,mode", [(1919, 1079, 0), (641, 359, 1), (250, 130, 5), (7, 5, 3)])
def test_no_write_outside_the_buffers(cvs, w, h, mode):
    # compute-sanitizer is closed on the pool, so out-of-bounds writes are caught with guard bands: every output
    # buffer of the sequence API sits inside a larger allocation filled with a pattern that must survive.  (The
    # reference's kernel2 over-writes 5,120 bytes past its buffers, SURVEY section 2a -- this one must not.)
    import torch
    G = 4096
    nframes, n = 3, 3 * w * h
    stride = (n + 15) // 16 * 16
    cap = (n + 3) // 4 * 4
    base, frames = random_sequence(w, h, nframes, 1.0, seed=5)   # every byte changes: payload fills the capacity

    def guarded(nbytes, dtype=torch.uint8):
        raw = torch.full((nbytes + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
        return raw, raw[G:G + nbytes].view(dtype)

    raw_f, d_frames = guarded(nframes * stride)
    for t in range(nframes):
        d_frames[t * stride: t * stride + n] = torch.from_numpy(frames[t]).cuda()
    raw_p, d_pos = guarded(4 * nframes, torch.int32)
    raw_x, d_xs = guarded(4 * nframes * cap, torch.int32)
    raw_d, d_diff = guarded(nframes * cap)
    raw_s, d_show = guarded(nframes * stride)
    s = cvs.Stream(w, h, base, mode=mode)
    s.run_sequence_device(d_frames.data_ptr(), stride, nframes, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(),
                          cap, d_show.data_ptr() if mode else 0, stride,
                          cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s.sequence_status()
    assert d_pos.cpu().tolist() == [n] * nframes
    for raw in (raw_f, raw_p, raw_x, raw_d, raw_s):
        assert bool((raw[:G] == 0xA5).all()) and bool((raw[-G:] == 0xA5).all())
    if not mode:
        assert bool((d_show == 0xA5).all())          # no display buffer requested: untouched
    else:
        for t in range(nframes):                      # the pad between frames of the display buffer is untouched too
            assert bool((d_show[t * stride + n:(t + 1) * stride] == 0xA5).all())
    # the input frames are never modified
    for t in range(nframes):
        assert np.array_equal(d_frames[t * stride: t * stride + n].cpu().numpy(), frames[t])
    s.close()


@pytest.mark.parametrize("density,cap", [(1.0, 1000), (0.5, 4096), (0.05, 256), (1.0, 4)])
def test_truncated_payload_stays_inside_capacity(cvs, oracle, density, cap):
    # a frame with more changed bytes than the payload capacity: the first `cap` entries are delivered, the true count
    # is reported with CVS_ERR_CAPACITY, and nothing is written past the capacity (dense and sparse emission paths)
    import torch
    G = 4096
    w, h, nframes = 250, 130, 3
    n = 3 * w * h
    stride = (n + 15) // 16 * 16
    base, frames = random_sequence(w, h, nframes, density, seed=9)

    def guarded(nbytes, dtype=torch.uint8):
        raw = torch.full((nbytes + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
        return raw, raw[G:G + nbytes].view(dtype)

    d_frames = torch.zeros(nframes * stride, dtype=torch.uint8, device="cuda")
    for t in range(nframes):
        d_frames[t * stride: t * stride + n] = torch.from_numpy(frames[t]).cuda()
    raw_p, d_pos = guarded(4 * nframes, torch.int32)
    raw_x, d_xs = guarded(4 * nframes * cap, torch.int32)
    raw_d, d_diff = guarded(nframes * cap)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    s.run_sequence_device(d_frames.data_ptr(), stride, nframes, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(),
                          cap, 0, stride, cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    with pytest.raises(cvs.CVSError) as e:
        s.sequence_status()
    assert e.value.status == 5  # CVS_ERR_CAPACITY
    for raw in (raw_p, raw_x, raw_d):
        assert bool((raw[:G] == 0xA5).all()) and bool((raw[-G:] == 0xA5).all())
    for t in range(nframes):
        opos, oxs, odiff, _, _ = oc.exec_core(frames[t])
        assert int(d_pos[t]) == opos and opos > cap
        assert np.array_equal(d_xs[t * cap:(t + 1) * cap].cpu().numpy(), oxs[:cap]), f"frame {t}"
        assert np.array_equal(d_diff[t * cap:(t + 1) * cap].cpu().numpy(), odiff[:cap]), f"frame {t}"
    assert np.array_equal(s.reference(), oc.reference())  # the feedback does not depend on the capacity
    s.close()


@pytest.mark.parametrize("levels", [[0], [1], [100], [255], [10, 200], [200, 10], [50, 50, 90], [0, 255, 255]])
def test_threshold_quirks_on_gpu(cvs, oracle, levels):
    # histograms that hit the corners of the two-max loop (server.cpp:108-127): arg-max at bin 0 (isec = -1), ties,
    # records before the maximum, both clamps -- through the real pipeline (average gray, clamp [50,200] and [0,255])
    import torch
    w, h = 64, 48
    p = w * h
    px = np.zeros((p, 3), dtype=np.uint8)
    bounds = np.linspace(0, p, len(levels) + 1).astype(int)
    if len(levels) == 3:
        bounds = np.array([0, p // 4, p // 2, p])  # unequal counts
    for i, g in enumerate(levels):
        px[bounds[i]:bounds[i + 1]] = g
    frame = px.reshape(-1)
    d_in = torch.from_numpy(np.concatenate([frame, np.zeros(64, np.uint8)])).cuda()
    d_out = torch.zeros(3 * p + 64, dtype=torch.uint8, device="cuda")
    d_g = torch.zeros(p + 64, dtype=torch.uint8, device="cuda")
    d_ht = torch.zeros(257, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    g1 = oracle.gray_avg1(frame, w, h)
    hist = oracle.histogram1(g1)
    for lo, hi in ((50, 200), (0, 255), (20, 255)):
        cvs.filters.binarize(d_in.data_ptr(), d_out.data_ptr(), d_g.data_ptr(), d_ht.data_ptr(), w, h, False, lo, hi, st)
        torch.cuda.synchronize()
        thr = oracle.threshold_twomax(hist, lo, hi)
        ht = d_ht.cpu().numpy()
        assert np.array_equal(ht[:256], hist)
        assert ht[256] == thr, f"levels {levels} clamp [{lo},{hi}]: {ht[256]} != {thr}"
        assert np.array_equal(d_out[:3 * p].cpu().numpy(), oracle.binarize(np.repeat(g1, 3), thr))
