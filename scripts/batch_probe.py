"""Batch probe: n cameras' 1080p frames as n single-frame launches (cvs_run_sequence_device, nframes = 1) against one
cvs_run_batch_device launch, and frames/s end to end through cvs_submit_io against cvs_submit_io_batch (run on the GPU box).

Device leg: per (n, density) the same n handles run alternately (a) n back-to-back single-frame calls and (b) one batch,
each timed with CUDA events around --frames camera-frames and repeated --reps times.  The timed work is queued behind
a spin kernel, so the events measure the device, not the host's enqueue rate (printed beside it).  Every camera walks its own ring of
synthetic frames (forth and back, so consecutive frames differ by the density); the rings of all cameras together hold
more than 160 MB, so the frames and references a pass touches are not in the 126 MB L2 from an earlier pass.
End-to-end leg: 3 and 8 cameras at 1 / 10 / 50 % density (round-robin), each from a pinned host ring of 16 frames with
up to 4 tickets in flight per camera, as bench.py's e2e leg does; (a) cvs_submit_io per camera, (b) one
cvs_submit_io_batch per round."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import cudavideostream_b200 as cvs  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--ns", default="1,2,4,8,16,64")
ap.add_argument("--densities", default="10000,100000,500000", help="ppm")
ap.add_argument("--frames", type=int, default=3000, help="camera-frames per timed run (passes = frames / n)")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--e2e-frames", type=int, default=300, help="frames per camera")
ap.add_argument("--e2e-ns", default="3,8")
ap.add_argument("--skip-e2e", action="store_true")
a = ap.parse_args()

W, H = 1920, 1080
N = 3 * W * H
S = (N + 15) // 16 * 16
CAP = (N + 3) // 4 * 4
st = torch.cuda.current_stream().cuda_stream


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name()} (power limit not readable: {e})"
    return q


def ring(n_frames, seed, density):
    """base frame + n_frames synthetic successors, device-resident, stride S"""
    fr = torch.empty((n_frames + 1) * S, dtype=torch.uint8, device="cuda")
    cvs.synth.base_frame_device(fr.data_ptr(), W, H, seed, st)
    for t in range(n_frames):
        cvs.synth.next_frame_device(fr.data_ptr() + t * S, fr.data_ptr() + (t + 1) * S, W, H, seed, t, density, st)
    return fr


def spread(v):
    v = sorted(v)
    return f"{v[len(v) // 2]:6.2f} [{v[0]:6.2f} .. {v[-1]:6.2f}]"


print(f"card: {card()}")
print(f"1080p, payload capacity N per camera; us per camera-frame, median [min .. max] of {a.reps} alternated runs "
      f"of {a.frames} camera-frames each")
ns = [int(x) for x in a.ns.split(",")]
results = []
for d in [int(x) for x in a.densities.split(",")]:
    for n in ns:
        R = max(4, -(-160_000_000 // (n * N)) + 1)  # frames per camera ring: all rings together > 160 MB
        rings = [ring(R, 1000 + i, d) for i in range(n)]
        torch.cuda.synchronize()
        streams = [cvs.Stream(W, H, rings[i][:N].cpu().numpy()) for i in range(n)]
        order = list(range(1, R + 1)) + list(range(R - 1, 1, -1))  # forth and back over frames 1..R
        pos = torch.zeros(n, dtype=torch.int32, device="cuda")
        xs = torch.empty(n * CAP, dtype=torch.int32, device="cuda")
        df = torch.empty(n * CAP, dtype=torch.uint8, device="cuda")
        k = [0]

        def frames():
            f = [rings[i].data_ptr() + order[(k[0] + i) % len(order)] * S for i in range(n)]
            k[0] += 1
            return f

        def sep(passes):
            for _ in range(passes):
                for i, f in enumerate(frames()):
                    streams[i].run_sequence_device(f, S, 1, pos.data_ptr() + 4 * i, xs.data_ptr() + 4 * i * CAP,
                                                   df.data_ptr() + i * CAP, CAP, cuda_stream=st)

        def bat(passes):
            for _ in range(passes):
                cvs.run_batch_device(streams, frames(), pos.data_ptr(), xs.data_ptr(), df.data_ptr(), CAP, cuda_stream=st)

        passes = max(4, a.frames // n)

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            torch.cuda._sleep(50_000_000)  # ~25 ms: the queue fills behind it
            e0.record()
            h0 = time.perf_counter()
            fn(passes)
            h1 = time.perf_counter()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1000 / (passes * n), (h1 - h0) * 1e6 / (passes * n)

        sep(2)
        bat(2)
        ta, tb, ha, hb = [], [], [], []
        for _ in range(a.reps):
            x, y = timed(sep)
            ta.append(x)
            ha.append(y)
            x, y = timed(bat)
            tb.append(x)
            hb.append(y)
        for s in streams:
            s.sequence_status()
        c = float(pos.to(torch.float64).sum()) / (n * N)
        line = (f"d={d / 1e4:4.0f}% n={n:2d} ring={R:2d} c={c:.3f}  separate {spread(ta)}  batch {spread(tb)}  "
                f"ratio {np.median(tb) / np.median(ta):.3f}  (host enqueue us/frame: {np.median(ha):.1f} / {np.median(hb):.1f})")
        print(line, flush=True)
        results.append((d, n, ta, tb))
        for s in streams:
            s.close()
        del rings, xs, df
        torch.cuda.empty_cache()

if a.skip_e2e:
    sys.exit(0)

print(f"end to end, frames/s (all cameras together), {a.e2e_frames} frames per camera, median [min .. max] of {a.reps} "
      "alternated runs")
RH = 16
for n in [int(x) for x in a.e2e_ns.split(",")]:
    dens = [(10000, 100000, 500000)[i % 3] for i in range(n)]
    hrings, bases = [], []
    for i in range(n):
        fr = ring(RH, 2000 + i, dens[i])
        torch.cuda.synchronize()
        hb_ = cvs.alloc_host(RH * N)
        hb_.array()[:] = np.concatenate([fr[(t + 1) * S:(t + 1) * S + N].cpu().numpy() for t in range(RH)])
        hrings.append(hb_)
        bases.append(fr[:N].cpu().numpy())
        del fr
    streams = [cvs.Stream(W, H, b) for b in bases]
    outs = [[(cvs.alloc_host(N + 32), cvs.alloc_host(4 * N + 32), (C.c_uint * 1)()) for _ in range(5)] for _ in range(n)]
    order = list(range(RH)) + list(range(RH - 2, 0, -1))

    def e2e(frames, batched):
        pend = [[] for _ in range(n)]
        for t in range(frames):
            f = [hrings[i].ptr + order[t % len(order)] * N for i in range(n)]
            for i in range(n):
                if len(pend[i]) == 4:
                    streams[i].wait(pend[i].pop(0))
            bufs = [outs[i][t % 5] for i in range(n)]
            if batched:
                tk = cvs.submit_io_batch(streams, f, [b[0].ptr for b in bufs], [C.addressof(b[2]) for b in bufs],
                                         [b[1].ptr for b in bufs])
            else:
                tk = [streams[i].submit_io_raw(f[i], bufs[i][0].ptr, None, "", C.addressof(bufs[i][2]), bufs[i][1].ptr)
                      for i in range(n)]
            for i in range(n):
                pend[i].append(tk[i])
        for i in range(n):
            for tk_ in pend[i]:
                streams[i].wait(tk_)

    e2e(16, False)
    e2e(16, True)
    fa, fb = [], []
    for _ in range(a.reps):
        for batched, acc in ((False, fa), (True, fb)):
            t0 = time.perf_counter()
            e2e(a.e2e_frames, batched)
            acc.append(n * a.e2e_frames / (time.perf_counter() - t0))
    print(f"cameras={n} (1/10/50 % round-robin)  cvs_submit_io {np.median(fa):8.0f} [{min(fa):.0f} .. {max(fa):.0f}]  "
          f"cvs_submit_io_batch {np.median(fb):8.0f} [{min(fb):.0f} .. {max(fb):.0f}]", flush=True)
    for s in streams:
        s.close()
    del hrings, outs
