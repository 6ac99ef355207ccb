"""Parity of every configuration bench.py times, at the size and length it is timed (BASELINE.json configs 2-5):

* 1080p x 300 frames x the three bench densities / seeds (config 2)                     -> test_bench_sequences_1080p
* 3840x2160 multi-frame sequences, nseg > 1 with nframes > 1 (config 5), modes 0, 1, 5   -> test_4k_sequences
* 1080p sequences with the noise filter + binarisation (config 3) and heat map / red map (config 4)
* the reference's own camera frames f1.jpg / f2.jpg at full size against the digests recorded in the build
  container (tests/golden/k1_f1_f2.json, REPORT/report.tex:2594)
* what `bench.py --dump-outputs` writes: the last timed step of the headline loop

Every comparison is bit-exact against oracle/cvs_oracle.c on the same frames (generated on the device by the
synthetic camera, whose numpy twin is checked in test_sequence_gpu.py::test_synth_device_twin).
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
BENCH_SEED = 0xC0DA5EED  # bench.py's rank-0 seed


def _device_sequence(cvs, torch, w, h, nframes, density_ppm, seed, stride=None):
    n = 3 * w * h
    stride = stride or (n + 15) // 16 * 16
    st = torch.cuda.current_stream().cuda_stream
    fr = torch.zeros((nframes + 1) * stride + 64, dtype=torch.uint8, device="cuda")
    cvs.synth.base_frame_device(fr.data_ptr(), w, h, seed, st)
    for t in range(nframes):
        cvs.synth.next_frame_device(fr.data_ptr() + t * stride, fr.data_ptr() + (t + 1) * stride, w, h, seed, t,
                                    density_ppm, st)
    torch.cuda.synchronize()
    return fr, stride


def _run(cvs, torch, s, fr, stride, nframes, n, mode):
    cap = (n + 3) // 4 * 4
    d_pos = torch.zeros(nframes, dtype=torch.int32, device="cuda")
    d_xs = torch.empty(nframes * cap, dtype=torch.int32, device="cuda")
    d_diff = torch.empty(nframes * cap, dtype=torch.uint8, device="cuda")
    d_show = torch.zeros(nframes * stride, dtype=torch.uint8, device="cuda") if mode else None
    s.run_sequence_device(fr.data_ptr() + stride, stride, nframes, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(),
                          cap, d_show.data_ptr() if mode else 0, stride,
                          cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s.sequence_status()
    return d_pos.cpu().numpy(), d_xs, d_diff, d_show, cap


@pytest.mark.parametrize("density_ppm", [10000, 100000, 500000])
def test_bench_sequences_1080p(cvs, oracle, density_ppm):
    # exactly what bench.py times for `value`: 300 frames, 1080p, seed 0xC0DA5EED, one launch -- every frame's
    # count, indices and difference bytes and the final reference against orc_diff_compact (test.cu:560-576)
    import torch
    w, h, T = 1920, 1080, 300
    n = 3 * w * h
    fr, stride = _device_sequence(cvs, torch, w, h, T, density_ppm, BENCH_SEED, stride=n)
    base = fr[:n].cpu().numpy()
    s = cvs.Stream(w, h, base, max_sequence=T)
    pos, d_xs, d_diff, _, cap = _run(cvs, torch, s, fr, stride, T, n, 0)
    lib = oracle.lib()
    ref = base.copy()
    xs = np.empty(n, dtype=np.int32)
    u8p, i32p = C.POINTER(C.c_uint8), C.POINTER(C.c_int)
    for t in range(T):
        cur = fr[(t + 1) * stride:(t + 1) * stride + n].cpu().numpy()
        opos = lib.orc_diff_compact(cur.ctypes.data_as(u8p), ref.ctypes.data_as(u8p), xs.ctypes.data_as(i32p), n, 20)
        assert pos[t] == opos, f"frame {t}: pos {pos[t]} != {opos}"
        assert np.array_equal(d_xs[t * cap:t * cap + opos].cpu().numpy(), xs[:opos]), f"frame {t}: xs"
        assert np.array_equal(d_diff[t * cap:t * cap + opos].cpu().numpy(), cur[:opos]), f"frame {t}: diff"
    assert np.array_equal(s.reference(), ref)
    s.close()


@pytest.mark.parametrize("mode,density_ppm", [(0, 10000), (0, 100000), (0, 500000), (1, 100000), (5, 100000)])
def test_4k_sequences(cvs, oracle, mode, density_ppm):
    # config 5: a 3840x2160 frame takes nseg = 4 passes of the grid, and the running total of the earlier segments
    # travels between them; only a multi-frame launch exercises that together with the frame-to-frame state
    import torch
    w, h, T = 3840, 2160, 8
    n = 3 * w * h
    fr, stride = _device_sequence(cvs, torch, w, h, T, density_ppm, BENCH_SEED ^ 5)
    base = fr[:n].cpu().numpy()
    s = cvs.Stream(w, h, base, mode=mode, max_sequence=T)
    pos, d_xs, d_diff, d_show, cap = _run(cvs, torch, s, fr, stride, T, n, mode)
    oc = oracle.OracleCore(w, h, base, mode=mode)
    for t in range(T):
        cur = fr[(t + 1) * stride:(t + 1) * stride + n].cpu().numpy()
        opos, oxs, odiff, oshow, _ = oc.exec_core(cur)
        assert pos[t] == opos, f"frame {t}: pos {pos[t]} != {opos}"
        assert np.array_equal(d_xs[t * cap:t * cap + opos].cpu().numpy(), oxs), f"frame {t}: xs"
        assert np.array_equal(d_diff[t * cap:t * cap + opos].cpu().numpy(), odiff), f"frame {t}: diff"
        if mode:
            assert np.array_equal(d_show[t * stride:t * stride + n].cpu().numpy(), oshow), f"frame {t}: show"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()


@pytest.mark.parametrize("name,mode,noise", [("config3", 5, True), ("config3_nodisplay", 0, True),
                                             ("config4_heat", 1, False), ("config4_red", 2, False)])
def test_1080p_filter_sequences(cvs, oracle, name, mode, noise):
    # config 3: Gaussian K=3 noise filter -> diff, weighted gray -> histogram -> two-max -> binarize;
    # config 4: heat map / heat-map-red against the negative-feedback reference, as 16-frame launches
    import torch
    w, h, T = 1920, 1080, 16
    n = 3 * w * h
    fr, stride = _device_sequence(cvs, torch, w, h, T, 100000, BENCH_SEED ^ 3, stride=n)
    base = fr[:n].cpu().numpy()
    kw, okw = {}, {}
    if noise:
        k = oracle.gaussian_kernel(3, 1.5)
        kw = dict(noise_filter=True, ksize=3, kweights=k)
        okw = dict(noise_filter=1, K=3, k=k)
    s = cvs.Stream(w, h, base, mode=mode, max_sequence=T, **kw)
    pos, d_xs, d_diff, d_show, cap = _run(cvs, torch, s, fr, stride, T, n, mode)
    oc = oracle.OracleCore(w, h, base, mode=mode, **okw)
    for t in range(T):
        cur = fr[(t + 1) * stride:(t + 1) * stride + n].cpu().numpy()
        opos, oxs, odiff, oshow, _ = oc.exec_core(cur)
        assert pos[t] == opos, f"{name} frame {t}: pos {pos[t]} != {opos}"
        assert np.array_equal(d_xs[t * cap:t * cap + opos].cpu().numpy(), oxs), f"{name} frame {t}: xs"
        assert np.array_equal(d_diff[t * cap:t * cap + opos].cpu().numpy(), odiff), f"{name} frame {t}: diff"
        if mode:
            assert np.array_equal(d_show[t * stride:t * stride + n].cpu().numpy(), oshow), f"{name} frame {t}: show"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()


def _same_payloads(a, b):
    return all(x[0] == y[0] and np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2]) for x, y in zip(a, b))


def test_bench_dump_outputs_are_the_last_timed_step(cvs, oracle, tmp_path):
    # bench.py --dump-outputs at the headline frame size, no warmup: every stream runs exactly `steps` passes over the
    # same frames (each pass starts from the reference the previous one left), and the dump is the last of them,
    # against the oracle.  On these frames the pass before and the pass after give other payloads, so a dump of one
    # pass too few or too many, or a --steps that ran another number of passes, does not match.
    import subprocess
    import sys
    import torch
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    w, h, T, steps = 1920, 1080, 4, 2
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--frames", str(T), "--warmup", "0",
                          "--steps", str(steps), "--no-cpu", "--no-side", "--e2e-frames", "4", "--e2e-ring", "4",
                          "--sync-frames", "4", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    files = sorted(os.listdir(tmp_path))
    assert files == sorted("d%d_%s.npy" % (d, k) for d in bench.DENSITIES_PPM for k in ("pos", "xs", "diff", "reference"))
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    n = 3 * w * h
    for d in bench.DENSITIES_PPM:
        got = {k: np.load(tmp_path / ("d%d_%s.npy" % (d, k))) for k in ("pos", "xs", "diff", "reference")}
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        fr, stride = _device_sequence(cvs, torch, w, h, T, d, BENCH_SEED, stride=n)
        frames = fr[:(T + 1) * n].cpu().numpy().reshape(T + 1, n)
        oc = oracle.OracleCore(w, h, frames[0])
        passes, refs = [], []
        for _ in range(steps + 1):
            passes.append([oc.exec_core(f)[:3] for f in frames[1:]])
            refs.append(oc.reference())
        oc.close()
        last = passes[steps - 1]
        assert not _same_payloads(passes[steps - 2], last) and not _same_payloads(passes[steps], last), \
            f"density {d}: neighbouring passes give the same payload, the check would not tell them apart"
        pos = np.array([p for p, _, _ in last])
        assert np.array_equal(got["pos"], pos), f"density {d}: counts"
        slots = bench.dump_slots(pos, got["xs"].shape[1])
        for t, (p, xs, diff) in enumerate(last):
            if p == 0:  # no entries: the dump holds the -1 sentinel
                assert (got["xs"][t] == -1).all() and (got["diff"][t] == -1).all(), f"density {d} frame {t}"
                continue
            assert np.array_equal(got["xs"][t], xs[slots[t]]) and np.array_equal(got["diff"][t], diff[slots[t]]), \
                f"density {d} frame {t}"
        assert np.array_equal(got["reference"], refs[steps - 1][bench.dump_reference_index(n)]), f"density {d}: reference"


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_real_camera_frames_full_size(cvs, oracle):
    # K1 (REPORT/report.tex:2594): the reference's own fixture pair, full 1920x1080 frames through the CUDA path.
    # The digests were recorded from the oracle in the build container (tests/golden/make_golden.py); the JPEGs are
    # the reference's tests/noise_filter_benchmark/f1.jpg and f2.jpg, byte for byte.
    cv2 = pytest.importorskip("cv2")
    with open(os.path.join(GOLDEN, "k1_f1_f2.json")) as f:
        g = json.load(f)
    a = cv2.imread(os.path.join(GOLDEN, "k1_f1.jpg"))
    b = cv2.imread(os.path.join(GOLDEN, "k1_f2.jpg"))
    assert a is not None and b is not None and a.shape == (1080, 1920, 3)
    # the decode must be the one the digests were taken with (same image, same libjpeg-turbo)
    assert _sha(a) == g["sha256_f1"] and _sha(b) == g["sha256_f2"], "JPEG decode differs from the build container's"
    s = cvs.Stream(1920, 1080, a.reshape(-1))
    pos, xs, diff, _ = s.exec(b.reshape(-1))
    assert pos == g["changed_bytes"] == 369350
    assert _sha(xs) == g["sha256_xs"] and _sha(diff) == g["sha256_diff"]
    assert _sha(s.reference()) == g["sha256_new_reference"]
    # and against the oracle run here, entry by entry
    opos, oxs, odiff, oref, _ = oracle.diff_compact(b, a, 20)
    assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff)
    assert np.array_equal(s.reference(), oref)
    s.close()


@pytest.mark.parametrize("w,h,mode", [(2560, 1440, 0), (3001, 1999, 0), (3001, 1999, 2), (2561, 1441, 5)])
def test_banded_sequences_odd_sizes(cvs, oracle, w, h, mode):
    # frames that take more than one pass of the grid are walked band by band when a sequence is long enough (every
    # band = one launch with the reference in registers, counts handed from band to band): sizes whose last band is
    # shorter than the others and whose byte count is not a multiple of the 96-byte chunk
    import torch
    T = 5
    n = 3 * w * h
    fr, stride = _device_sequence(cvs, torch, w, h, T, 60000, BENCH_SEED ^ 7)
    base = fr[:n].cpu().numpy()
    s = cvs.Stream(w, h, base, mode=mode, max_sequence=T)
    pos, d_xs, d_diff, d_show, cap = _run(cvs, torch, s, fr, stride, T, n, mode)
    oc = oracle.OracleCore(w, h, base, mode=mode)
    for t in range(T):
        cur = fr[(t + 1) * stride:(t + 1) * stride + n].cpu().numpy()
        opos, oxs, odiff, oshow, _ = oc.exec_core(cur)
        assert pos[t] == opos, f"frame {t}: pos {pos[t]} != {opos}"
        assert np.array_equal(d_xs[t * cap:t * cap + opos].cpu().numpy(), oxs), f"frame {t}: xs"
        assert np.array_equal(d_diff[t * cap:t * cap + opos].cpu().numpy(), odiff), f"frame {t}: diff"
        if mode:
            assert np.array_equal(d_show[t * stride:t * stride + n].cpu().numpy(), oshow), f"frame {t}: show"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()
