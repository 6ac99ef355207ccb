"""Batches: one frame of each of n camera streams in one stream-kernel launch (cvs_run_batch_device,
cvs_submit_io_batch).  Every camera's outputs must be byte for byte those of n separate calls on twin handles and those
of the CPU oracle, references included."""
import ctypes as C
import functools
import re
import shutil
import subprocess

import numpy as np
import pytest

from util import CHARS_STR, glyph_atlas, random_sequence

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
INVALID, ALIGN, CAPACITY = 1, 4, 5


# ---------------------------------------------------------------------------------------------------------------------
# no device needed
# ---------------------------------------------------------------------------------------------------------------------
def test_batch_arguments_refused_without_a_handle(cvs):
    lib = cvs.load_library()
    one = (C.c_void_p * 1)(None)
    frames = (C.c_void_p * 1)(None)
    tk = (C.c_uint64 * 1)()
    for n in (0, -1, cvs.MAX_BATCH + 1):
        assert lib.cvs_run_batch_device(one, n, frames, None, None, None, 16, None, 0, None, None) == INVALID
        assert lib.cvs_submit_io_batch(one, n, frames, frames, None, None, frames, frames, tk) == INVALID
    # a NULL array, a NULL handle
    assert lib.cvs_run_batch_device(None, 1, frames, None, None, None, 16, None, 0, None, None) == INVALID
    assert lib.cvs_run_batch_device(one, 1, frames, None, None, None, 16, None, 0, None, None) == INVALID
    assert lib.cvs_submit_io_batch(None, 1, frames, frames, None, None, frames, frames, tk) == INVALID
    assert lib.cvs_submit_io_batch(one, 1, frames, frames, None, None, frames, frames, tk) == INVALID
    assert b"handle" in lib.cvs_last_error()


@functools.lru_cache(maxsize=1)
def _sass() -> str:
    try:
        return subprocess.run([CUOBJDUMP, "-sass", cvs_library_path()], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError) as e:
        pytest.skip(f"cuobjdump unavailable: {e}")


def cvs_library_path():
    import cudavideostream_b200 as m
    return m.library_path()


@pytest.mark.parametrize("mode", range(8))
@pytest.mark.parametrize("hi", [0, 1])
def test_batch_kernel_sass(mode, hi):
    blocks = re.split(r"(?=\n\s*Function : )", _sass())
    name = r"k_stream_ws_batchILi%dELb%dE" % (mode, hi)
    hit = [b for b in blocks if re.search(r"Function : \S*" + name, b)]
    assert len(hit) == 1, f"k_stream_ws_batch<{mode}, {hi}> missing"
    k = hit[0]
    assert not re.search(r"\b(LDL|STL)\b", k), f"{name} spills to local memory"
    assert "UBLKCP" in k, "the frame ingest must be a TMA bulk copy (cp.async.bulk)"
    assert "SYNCS" in k, "mbarrier (SYNCS.*) expected next to the bulk copy"
    assert k.count("VABSDIFF4") >= 24, "one byte-SIMD absolute difference per word of the 96-byte chunk"


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
def _fast_sequence(w, h, steps, density, seed):
    """random_sequence for full-size frames (vectorised in uint8: changes wrap, drift is 0..2 up)."""
    rng = np.random.default_rng(seed)
    n = 3 * w * h
    base = rng.integers(0, 256, n, dtype=np.uint8)
    frames = np.empty((steps, n), dtype=np.uint8)
    prev = base
    for t in range(steps):
        big = rng.random(n, dtype=np.float32) < density
        cur = np.where(big, prev + rng.integers(21, 236, n, dtype=np.uint8), prev + rng.integers(0, 3, n, dtype=np.uint8))
        frames[t] = cur
        prev = cur
    return base, frames


def _camera(w, h, steps, density, seed, cfg=None, ocfg=None):
    gen = _fast_sequence if 3 * w * h > 1_000_000 else random_sequence
    base, frames = gen(w, h, steps, density, seed)
    return dict(base=base, frames=frames, cfg=cfg or {}, ocfg=ocfg or {})


def _to_device(torch, frame):
    n = frame.size
    buf = np.zeros((n + 15) // 16 * 16 + 16, dtype=np.uint8)
    buf[:n] = frame
    return torch.from_numpy(buf).cuda()


def _status(cvs, s):
    try:
        s.sequence_status()
        return 0
    except cvs.CVSError as e:
        return e.status


def _passes(cam, mode, show, text):
    """launches of a camera's own pre- and post-passes for one frame"""
    return int("noise_filter" in cam["cfg"]) + int(bool(text) and "glyphs" in cam["cfg"]) + 2 * int(mode in (5, 7) and show)


def _run_and_check(cvs, oracle, w, h, cams, steps=1, mode=0, show=False, texts=None, cap=None, threshold=20,
                   orders=None):
    """Runs `steps` consecutive batches of the cameras (batch t in the camera order orders[t]) and the same frames
    through cvs_run_sequence_device(nframes=1) on twin handles and through the oracle; compares everything."""
    import torch
    n_cam, N = len(cams), 3 * w * h
    stride = (N + 15) // 16 * 16
    cap = cap or (N + 3) // 4 * 4
    streams = [cvs.Stream(w, h, c["base"], mode=mode, threshold=threshold, **c["cfg"]) for c in cams]
    twins = [cvs.Stream(w, h, c["base"], mode=mode, threshold=threshold, **c["cfg"]) for c in cams]
    orcs = [oracle.OracleCore(w, h, c["base"], thr=threshold, mode=mode, **c["ocfg"]) for c in cams]
    texts = texts or [None] * n_cam
    cs = torch.cuda.current_stream().cuda_stream
    statuses = []
    for t in range(steps):
        order = orders[t] if orders else list(range(n_cam))
        n = len(order)
        d_frames = [_to_device(torch, cams[i]["frames"][t]) for i in order]
        d_pos = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_xs = torch.full((n * cap,), -7, dtype=torch.int32, device="cuda")
        d_diff = torch.zeros(n * cap, dtype=torch.uint8, device="cuda")
        d_show = torch.zeros(n * stride, dtype=torch.uint8, device="cuda") if show else None
        cvs.run_batch_device([streams[i] for i in order], [f.data_ptr() for f in d_frames], d_pos.data_ptr(),
                             d_xs.data_ptr(), d_diff.data_ptr(), cap, d_show.data_ptr() if show else 0, stride,
                             texts=[texts[i] for i in order], cuda_stream=cs)
        torch.cuda.synchronize()
        st = {i: _status(cvs, streams[i]) for i in order}
        statuses.append(st)
        for k, i in enumerate(order):
            frame = cams[i]["frames"][t]
            # twin: the same frame alone
            t_pos = torch.zeros(1, dtype=torch.int32, device="cuda")
            t_xs = torch.full((cap,), -7, dtype=torch.int32, device="cuda")
            t_diff = torch.zeros(cap, dtype=torch.uint8, device="cuda")
            t_show = torch.zeros(stride, dtype=torch.uint8, device="cuda") if show else None
            twins[i].run_sequence_device(d_frames[k].data_ptr(), stride, 1, t_pos.data_ptr(), t_xs.data_ptr(),
                                         t_diff.data_ptr(), cap, t_show.data_ptr() if show else 0, stride,
                                         text=texts[i] or "", cuda_stream=cs)
            torch.cuda.synchronize()
            assert _status(cvs, twins[i]) == st[i], f"batch {t} camera {i}: status"
            pos = int(d_pos[k])
            got_xs = d_xs[k * cap:(k + 1) * cap].cpu().numpy()
            got_diff = d_diff[k * cap:(k + 1) * cap].cpu().numpy()
            assert pos == int(t_pos[0]), f"batch {t} camera {i}: count"
            m = min(pos, cap)
            assert np.array_equal(got_xs[:m], t_xs[:m].cpu().numpy()), f"batch {t} camera {i}: xs vs separate call"
            assert np.array_equal(got_diff[:m], t_diff[:m].cpu().numpy()), f"batch {t} camera {i}: diff vs separate call"
            opos, oxs, odiff, oshow, _ = orcs[i].exec_core(frame, texts[i] or "")
            assert pos == opos, f"batch {t} camera {i}: count vs oracle"
            assert np.array_equal(got_xs[:m], oxs[:m]) and np.array_equal(got_diff[:m], odiff[:m]), \
                f"batch {t} camera {i}: payload vs oracle"
            assert (got_xs[m:] == -7).all(), f"batch {t} camera {i}: write past the count / capacity"
            if show and mode:  # (mode 0 has no display frame)
                got_show = d_show[k * stride:k * stride + N].cpu().numpy()
                assert np.array_equal(got_show, t_show[:N].cpu().numpy()), f"batch {t} camera {i}: show vs separate call"
                assert np.array_equal(got_show, oshow), f"batch {t} camera {i}: show vs oracle"
            # the caller's frames are never modified
            assert np.array_equal(d_frames[k][:N].cpu().numpy(), frame), f"batch {t} camera {i}: input modified"
    for i in range(n_cam):
        ref = streams[i].reference()
        assert np.array_equal(ref, twins[i].reference()), f"camera {i}: reference vs separate calls"
        assert np.array_equal(ref, orcs[i].reference()), f"camera {i}: reference vs oracle"
    for tw in twins:
        tw.close()
    return streams, statuses


DENS = [0.0, 0.01, 0.1, 0.5, 1.0]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 8, 64])
def test_batch_1080p(cvs, oracle, n):
    """Densities 0 / 1 / 10 / 50 / 100 % alternate from camera to camera, so sparse and dense steps follow each other.
    (A batch of one runs the single-frame path: one launch either way.)"""
    w, h = 1920, 1080
    cams = [_camera(w, h, 1, DENS[i % 5], seed=100 + i) for i in range(n)]
    streams, _ = _run_and_check(cvs, oracle, w, h, cams)
    assert sum(s.launch_count() for s in streams) == 1, "one stream-kernel launch for the whole batch"
    assert streams[0].launch_count() == 1
    for s in streams:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(7, 5), (1919, 1079), (333, 77)])
def test_batch_small_and_odd_sizes(cvs, oracle, w, h):
    # 7x5: N = 105, one block; 1919x1079 and 333x77: 3W % 4 != 0, rows and frames end inside chunks
    cams = [_camera(w, h, 2, DENS[i % 5] + 0.05, seed=7 * i + w) for i in range(3)]
    streams, _ = _run_and_check(cvs, oracle, w, h, cams, steps=2)
    assert sum(s.launch_count() for s in streams) == 2
    for s in streams:
        s.close()


@pytest.mark.gpu
def test_batch_4k_runs_per_handle(cvs, oracle):
    """3840x2160 does not fit one pass: the batch runs the single-frame path of each handle, with the same results."""
    w, h = 3840, 2160
    cams = [_camera(w, h, 1, d, seed=40 + i) for i, d in enumerate((0.02, 0.3))]
    streams, _ = _run_and_check(cvs, oracle, w, h, cams)
    assert [s.launch_count() for s in streams] == [1, 1], "one stream-kernel launch per handle"
    for s in streams:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("show", [False, True])
@pytest.mark.parametrize("mode", range(8))
def test_batch_modes(cvs, oracle, mode, show):
    w, h = 250, 130
    cams = [_camera(w, h, 2, DENS[i % 5], seed=13 * i + mode) for i in range(4)]
    streams, _ = _run_and_check(cvs, oracle, w, h, cams, steps=2, mode=mode, show=show)
    per = sum(_passes(c, mode, show, None) for c in cams)
    assert sum(s.launch_count() for s in streams) == 2 * (1 + per)
    for s in streams:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 5])
def test_batch_noise_filter_and_overlay_per_camera(cvs, oracle, mode):
    """Noise filter on some handles and not on others, different weights, per-camera overlay texts with NULL entries."""
    w, h = 321, 97
    atlas = glyph_atlas(7, 5)
    g = dict(glyphs=atlas, glyph_w=7, glyph_h=5)
    og = dict(glyphs=atlas, gw=7, gh=5, chars=CHARS_STR)
    k3, k5 = oracle.gaussian_kernel(3, 1.5), oracle.mean_kernel(5)
    setups = [({}, {}), (dict(noise_filter=True, ksize=3, kweights=k3), dict(noise_filter=1, K=3, k=k3)),
              (dict(g), dict(og)), (dict(noise_filter=True, ksize=5, kweights=k5, **g), dict(noise_filter=1, K=5, k=k5, **og)),
              (dict(g), dict(og))]
    cams = [_camera(w, h, 3, 0.05 + 0.1 * i, seed=50 + i, cfg=c, ocfg=o) for i, (c, o) in enumerate(setups)]
    texts = [None, "12:34", "FPS 30", None, ""]
    streams, _ = _run_and_check(cvs, oracle, w, h, cams, steps=3, mode=mode, show=mode != 0, texts=texts)
    per = sum(_passes(c, mode, mode != 0, texts[i]) for i, c in enumerate(cams))
    assert sum(s.launch_count() for s in streams) == 3 * (1 + per)
    for s in streams:
        s.close()


@pytest.mark.gpu
def test_twenty_consecutive_batches(cvs, oracle):
    """References carry from batch to batch (drift below the threshold accumulates); the leader changes every batch."""
    w, h, T = 640, 360, 20
    cams = [_camera(w, h, T, (0.002, 0.05, 0.3, 0.0)[i], seed=200 + i) for i in range(4)]
    orders = [[(t + k) % 4 for k in range(4)] for t in range(T)]
    streams, _ = _run_and_check(cvs, oracle, w, h, cams, steps=T, mode=3, show=True, orders=orders)
    for s in streams:
        s.close()


@pytest.mark.gpu
def test_batch_capacity_overflow_is_reported_per_camera(cvs, oracle):
    w, h = 320, 180
    cams = [_camera(w, h, 1, d, seed=300 + i) for i, d in enumerate((0.001, 0.5, 0.001))]
    cap = 4096  # camera 1 has ~86 k entries, the others ~170
    _, statuses = _run_and_check(cvs, oracle, w, h, cams, cap=cap)
    assert statuses[0] == {0: 0, 1: CAPACITY, 2: 0}


@pytest.mark.gpu
def test_batch_refusals_enqueue_nothing(cvs, oracle):
    import torch
    w, h = 200, 120
    N = 3 * w * h
    base, frames = random_sequence(w, h, 1, 0.1, seed=9)
    a, b = cvs.Stream(w, h, base), cvs.Stream(w, h, base)
    wrong = [cvs.Stream(w + 1, h, np.zeros(3 * (w + 1) * h, np.uint8)), cvs.Stream(w, h, base, mode=1),
             cvs.Stream(w, h, base, threshold=21)]
    cap = (N + 3) // 4 * 4
    d_f = _to_device(torch, frames[0])
    d_pos = torch.zeros(2, dtype=torch.int32, device="cuda")
    d_xs = torch.zeros(2 * cap, dtype=torch.int32, device="cuda")
    d_diff = torch.zeros(2 * cap, dtype=torch.uint8, device="cuda")
    cs = torch.cuda.current_stream().cuda_stream
    args = [d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr()]
    hb = cvs.alloc_host(N + 32)
    hx = cvs.alloc_host(4 * N + 32)
    pb = (C.c_uint * 1)()

    def refused(streams, frames_=None, capacity=cap, status=INVALID):
        with pytest.raises(cvs.CVSError) as e:
            cvs.run_batch_device(streams, frames_ or [d_f.data_ptr()] * len(streams), *args, capacity, cuda_stream=cs)
        assert e.value.status == status
        if status == INVALID and frames_ is None and capacity == cap:
            with pytest.raises(cvs.CVSError) as e:
                cvs.submit_io_batch(streams, [hb.ptr] * len(streams), [hb.ptr] * len(streams),
                                    [C.addressof(pb)] * len(streams), [hx.ptr] * len(streams))
            assert e.value.status == INVALID

    for x in wrong:
        refused([a, x])
    refused([a, b, a])
    refused([a, b], frames_=[d_f.data_ptr(), 0])
    refused([a, b], frames_=[d_f.data_ptr(), d_f.data_ptr() + 4], status=ALIGN)
    refused([a, b], capacity=cap - 2)
    launches = a.launch_count() + b.launch_count()
    # nothing was enqueued: a valid batch still starts from the base frame
    cvs.run_batch_device([a, b], [d_f.data_ptr()] * 2, *args, cap, cuda_stream=cs)
    torch.cuda.synchronize()
    assert a.launch_count() + b.launch_count() == launches + 1
    oc = oracle.OracleCore(w, h, base)
    opos, oxs, odiff, _, _ = oc.exec_core(frames[0])
    for k, s in enumerate((a, b)):
        s.sequence_status()
        assert int(d_pos[k]) == opos
        assert np.array_equal(d_xs[k * cap:k * cap + opos].cpu().numpy(), oxs)
        assert np.array_equal(d_diff[k * cap:k * cap + opos].cpu().numpy(), odiff)
        assert np.array_equal(s.reference(), oc.reference())
    for s in [a, b] + wrong:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# cvs_submit_io_batch
# ---------------------------------------------------------------------------------------------------------------------
class _Pageable:
    def __init__(self, nbytes):
        self.buf = np.zeros(nbytes, dtype=np.uint8)
        self.ptr = self.buf.ctypes.data

    def array(self, dtype=np.uint8):
        return self.buf.view(dtype)


def _jumping_frames(n, dens, rng, base):
    frames, cur = [], base.copy()
    for d in dens:
        nxt = cur.copy()
        idx = np.flatnonzero(rng.random(n) < d)
        nxt[idx] = (nxt[idx].astype(np.int64) + rng.integers(40, 200, idx.size)).astype(np.uint8)
        frames.append(nxt)
        cur = nxt
    return frames


class _SubmitRig:
    """Cameras fed through cvs_submit_io_batch and cvs_submit_io, each ticket checked against the camera's oracle in
    completion order."""

    def __init__(self, cvs, oracle, w, h, ncam, nframes, buffers, mode=0, seed=0):
        self.cvs, self.w, self.h, self.N, self.mode = cvs, w, h, 3 * w * h, mode
        rng = np.random.default_rng(seed)
        # densities on both sides of the speculative-copy window [N/64, N/4] (from the previous count), shifted per camera
        dens = [0.001, 0.05, 0.9, 0.0, 0.1, 0.0, 0.3, 1.0, 0.05, 0.06, 0.2, 0.002, 0.6, 0.05, 0.0, 0.45]
        self.base = [rng.integers(0, 256, self.N, dtype=np.uint8) for _ in range(ncam)]
        self.frames = [_jumping_frames(self.N, [dens[(t + 5 * c) % len(dens)] for t in range(nframes)], rng, self.base[c])
                       for c in range(ncam)]
        self.streams = [cvs.Stream(w, h, b, mode=mode) for b in self.base]
        self.orcs = [oracle.OracleCore(w, h, b, mode=mode) for b in self.base]
        self.ring = [cvs.alloc_host(nframes * self.N) for _ in range(ncam)]
        for c in range(ncam):
            for t, f in enumerate(self.frames[c]):
                self.ring[c].array()[t * self.N:(t + 1) * self.N] = f
        alloc = cvs.alloc_host if buffers == "pinned" else _Pageable
        # 5 buffer sets per camera: up to 4 tickets in flight plus the one being submitted
        self.bufs = [[(alloc(self.N + 32), alloc(4 * self.N + 32), (C.c_uint * 1)(), alloc(self.N + 32) if mode else None)
                      for _ in range(5)] for _ in range(ncam)]
        self.next = [0] * ncam          # next frame of each camera
        self.pending = [[] for _ in range(ncam)]  # (ticket, frame index) in submission order

    def args(self, c):
        t = self.next[c]
        db, xb, pb, sb = self.bufs[c][t % 5]
        return self.ring[c].ptr + t * self.N, db.ptr, C.addressof(pb), xb.ptr, (sb.ptr if sb is not None else None)

    def make_room(self, cams, depth=4):
        for c in cams:
            while len(self.pending[c]) >= depth:
                self.complete(c)

    def complete(self, c):
        tk, t = self.pending[c].pop(0)
        self.streams[c].wait(tk)
        db, xb, pb, sb = self.bufs[c][t % 5]
        opos, oxs, odiff, oshow, _ = self.orcs[c].exec_core(self.frames[c][t])
        assert pb[0] == opos, f"camera {c} frame {t}: pos {pb[0]} != {opos}"
        assert np.array_equal(db.array()[:opos], odiff), f"camera {c} frame {t}: diff"
        assert np.array_equal(xb.array(np.int32)[:opos], oxs), f"camera {c} frame {t}: xs"
        if sb is not None:
            assert np.array_equal(sb.array()[:self.N], oshow), f"camera {c} frame {t}: show"

    def batch(self, cams):
        a = [self.args(c) for c in cams]
        tickets = self.cvs.submit_io_batch([self.streams[c] for c in cams], [x[0] for x in a], [x[1] for x in a],
                                           [x[2] for x in a], [x[3] for x in a], show=[x[4] for x in a])
        for c, tk in zip(cams, tickets):
            self.pending[c].append((tk, self.next[c]))
            self.next[c] += 1

    def single(self, c):
        f, d, p, x, sh = self.args(c)
        tk = self.streams[c].submit_io_raw(f, d, sh, "", p, x)
        self.pending[c].append((tk, self.next[c]))
        self.next[c] += 1

    def finish(self):
        for c in range(len(self.streams)):
            while self.pending[c]:
                self.complete(c)
            assert np.array_equal(self.streams[c].reference(), self.orcs[c].reference()), f"camera {c}: reference"
            for t, f in enumerate(self.frames[c][:self.next[c]]):
                assert np.array_equal(self.ring[c].array()[t * self.N:(t + 1) * self.N], f), "captured frame modified"
        for s in self.streams:
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("buffers", ["pinned", "pageable"])
def test_submit_io_batch_interleaved(cvs, oracle, buffers):
    """Batches with a changing leader, single cvs_submit_io tickets on the same handles in between, and up to 4 tickets
    of a handle in flight; pinned buffers get the payload pushed, pageable ones copied in cvs_wait."""
    rig = _SubmitRig(cvs, oracle, 320, 180, 3, 20, buffers, seed=1 if buffers == "pinned" else 2)
    step = 0
    while min(rig.next) < 14:
        order = [(step + k) % 3 for k in range(3)]
        if step % 4 == 3:
            for c in order[:2]:
                rig.make_room([c])
                rig.single(c)
        else:
            rig.make_room(order)
            rig.batch(order if step % 4 != 2 else order[:2])
        step += 1
    rig.finish()


@pytest.mark.gpu
def test_submit_io_batch_show_per_camera(cvs, oracle):
    """Mode 3 with a show buffer for some cameras only: each gets exactly what cvs_submit_io gives it."""
    rig = _SubmitRig(cvs, oracle, 256, 96, 3, 6, "pinned", mode=3, seed=5)
    for c in range(3):
        for k in range(5):
            if (c + k) % 2:
                rig.bufs[c][k] = rig.bufs[c][k][:3] + (None,)
    for t in range(6):
        rig.make_room(range(3), depth=2)
        rig.batch([(t + k) % 3 for k in range(3)])
    rig.finish()


@pytest.mark.gpu
def test_submit_io_batch_fifth_ticket_refused(cvs, oracle):
    rig = _SubmitRig(cvs, oracle, 200, 120, 3, 8, "pinned", seed=3)
    for _ in range(3):
        rig.batch([0, 1, 2])
    rig.single(1)  # camera 1 now has 4 tickets outstanding
    with pytest.raises(cvs.CVSError) as e:
        rig.batch([2, 1, 0])
    assert e.value.status == INVALID
    with pytest.raises(cvs.CVSError):
        rig.batch([1])
    # nothing was enqueued for cameras 0 and 2 either: the same frames as one more batch follow in order
    rig.complete(1)
    rig.batch([2, 1, 0])
    assert [len(p) for p in rig.pending] == [4, 4, 4]
    rig.finish()
