"""Raw camera ingest on the GPU (YUV and Bayer): what k_yuv_to_bgr and k_bayer_to_bgr cost and what cvs_submit_yuv and
cvs_submit_bayer buy end to end.

1. Kernel time per frame of cvs_yuv_to_bgr_device for NV12, I420 and YUYV and of cvs_bayer_to_bgr_device (RGGB) at
   1920x1080 and 3840x2160: CUDA events around a CUDA graph of launches that walks a ring of frames larger than the
   126 MB L2 (every frame is read from and written to HBM), against the bytes model (read 1.5 or 2 bytes per pixel for
   YUV, 1 for Bayer; write 3) and the HBM copy peak: the one bench.py uses (MEASURED_PEAKS.json, else its fallback) and
   a device-to-device copy measured here.  Beside them the same graph of launches on a 16x2 (16x3 for Bayer) frame, one
   block: the fixed cost of a launch in a graph, which no frame size goes below.
2. End to end, frames/s of three camera streams per GPU submitted round-robin with four tickets in flight each, as in
   bench.py's e2e leg (1080p, 1 / 10 / 50 % change density, pinned host rings): cvs_submit_yuv with NV12 and with YUYV
   frames and cvs_submit_bayer with RGGB mosaics, each against cvs_submit_io with the very BGR frames they convert to
   ("raw:nv12", "raw:yuyv", "raw:bayer": the pictures, change densities and payloads of a pair are identical; the
   formats keep different colour detail, so the pairs differ from each other in payload), the six forms alternated in
   the same process.
3. The same three streams under CVS_TRACE=1 (a run of its own, 8 warm-up and 40 timed frames per stream and form, the
   warm-up tickets dropped): device time of each ticket's upload and kernels.

Run on the GPU box: python scripts/yuv_probe.py > profiles/bayer_probe.txt (profiles/yuv_probe.txt is the earlier run,
before the Bayer rows)"""
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import cudavideostream_b200 as cvs  # noqa: E402
import bayer_ref as B  # noqa: E402
import yuv_ref as Y  # noqa: E402
from oracle import oracle  # noqa: E402

W, H = 1920, 1080
N = 3 * W * H
DENSITIES_PPM = (10000, 100000, 500000)
L2_BYTES = 126 << 20
FORMS = ("raw:nv12", "nv12", "raw:yuyv", "yuyv", "raw:bayer", "bayer")
BAYER = B.RGGB


def packed(fmt, base, w, h):
    """plane addresses and pitches of a packed frame at device address base"""
    if fmt == Y.YUYV:
        return [base], [2 * w]
    if fmt == Y.NV12:
        return [base, base + w * h], [w, w]
    return [base, base + w * h, base + w * h + w * h // 4], [w, w // 2, w // 2]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    print(f"card: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {q}")


def copy_peak():
    """device-to-device copy of 1 GiB, (read + write) bytes over the time"""
    a = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 20 * 2 * a.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def convert(fmt, src, dst, w, h, stream):
    """one packed frame at device address src -> BGR at dst; fmt: a YUV format, or "bayer" """
    if fmt == "bayer":
        cvs.filters.bayer_to_bgr(BAYER, src, w, dst, w, h, stream)
    else:
        pl, pi = packed(fmt, src, w, h)
        cvs.filters.yuv_to_bgr(fmt, pl, pi, dst, w, h, stream)


def in_bytes(fmt, w, h):
    return w * h if fmt == "bayer" else Y.frame_bytes(fmt, w, h)


def name(fmt):
    return "bayer" if fmt == "bayer" else Y.NAMES[fmt]


def graph_us(fmt, w, h, K):
    """device time per launch of the conversion in a CUDA graph that converts a ring of K packed frames"""
    fin, fout = in_bytes(fmt, w, h), 3 * w * h
    sin, sout = (fin + 15) // 16 * 16, (fout + 15) // 16 * 16
    src = torch.randint(0, 256, (K * sin,), dtype=torch.uint8, device="cuda")
    dst = torch.empty(K * sout, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()

    def launch_ring(stream):
        for i in range(K):
            convert(fmt, src.data_ptr() + i * sin, dst.data_ptr() + i * sout, w, h, stream)

    with torch.cuda.stream(st):
        launch_ring(st.cuda_stream)  # warm-up, outside the graph
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        launch_ring(torch.cuda.current_stream().cuda_stream)
    reps = max(4, -(-3000 // K))
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (reps * K)
    del g, src, dst
    torch.cuda.empty_cache()
    return us


def kernel_times(peak):
    print("\n== k_yuv_to_bgr / k_bayer_to_bgr: device time per frame (CUDA graph of launches over an L2-cold ring, CUDA "
          "events) ==")
    print(f"{'size':>10} {'format':>6} {'ring':>5} {'us/frame':>9} {'model MB':>9} {'GB/s':>7} {'of peak':>8}")
    for w, h in ((1920, 1080), (3840, 2160)):
        for fmt in (Y.NV12, Y.I420, Y.YUYV, "bayer"):
            fin, fout = in_bytes(fmt, w, h), 3 * w * h
            K = max(8, -(-3 * L2_BYTES // (fin + fout + 32)))  # ring of three L2 sizes
            us = graph_us(fmt, w, h, K)
            gbs = (fin + fout) / (us * 1e-6) / 1e9
            print(f"{w}x{h:<5} {name(fmt):>6} {K:5d} {us:9.2f} {(fin + fout) / 1e6:9.2f} {gbs:7.0f} {gbs / peak:8.1%}")
    # one block, and plane pitches that are multiples of 16 as the entries require (16x3: the smallest frame the
    # demosaic computes rather than zeroes)
    for fmt, (w, h) in ((Y.NV12, (16, 2)), (Y.YUYV, (16, 2)), ("bayer", (16, 3))):
        print(f"{f'{w}x{h}':>10} {name(fmt):>6} {64:5d} {graph_us(fmt, w, h, 64):9.2f}   (one block: the fixed cost of a launch)")


def make_rings(R=16):
    """per density: R frames as NV12, as YUYV and as an RGGB mosaic, and as the BGR frames cv2.cvtColor makes of each
    (raw:nv12, raw:yuyv, raw:bayer: what a server uploads today after converting on the host), with the base frame of
    each"""
    rings = []
    for k, d in enumerate(DENSITIES_PPM):
        base, frames = oracle.synth_sequence(W, H, R, d, 0xC0FFEE + k)
        forms, bases = {}, {}
        for name, fmt in (("nv12", Y.NV12), ("yuyv", Y.YUYV)):
            bases[name] = bases["raw:" + name] = Y.yuv_to_bgr(fmt, Y.from_bgr(fmt, base, W, H), W, H).reshape(-1)
            forms[name] = [Y.from_bgr(fmt, f, W, H) for f in frames]
            forms["raw:" + name] = [Y.yuv_to_bgr(fmt, b, W, H).reshape(-1) for b in forms[name]]
        bases["bayer"] = bases["raw:bayer"] = B.bayer_to_bgr(BAYER, B.mosaic(base.reshape(H, W, 3), BAYER)).reshape(-1)
        forms["bayer"] = [B.mosaic(f.reshape(H, W, 3), BAYER).reshape(-1) for f in frames]
        forms["raw:bayer"] = [B.bayer_to_bgr(BAYER, m.reshape(H, W)).reshape(-1) for m in forms["bayer"]]
        host = {}
        for name, lst in forms.items():
            sz = lst[0].size
            hb = cvs.alloc_host(R * sz + 64)
            for t, b in enumerate(lst):
                hb.array()[t * sz:(t + 1) * sz] = b
            host[name] = (hb, sz)
        rings.append({"d": d, "host": host, "bases": bases,
                      "stream": cvs.Stream(W, H, bases["nv12"], threshold=20),
                      "out": [(cvs.alloc_host(N + 32), cvs.alloc_host(4 * N + 32), (C.c_uint * 1)()) for _ in range(4)]})
    return rings


def e2e(rings, form, nframes, R=16):
    order = list(range(R)) + list(range(R - 2, 0, -1))
    for q in rings:
        q["stream"].reset(q["bases"][form])
        q["pending"] = []
    pos_sum = 0

    def run(n):
        nonlocal pos_sum
        for i in range(n):
            for q in rings:
                s, (hb, sz), pending = q["stream"], q["host"][form], q["pending"]
                fb, xb, pb = q["out"][i % 4]
                if len(pending) == 4:
                    tk, pp = pending.pop(0)
                    s.wait(tk)
                    pos_sum += pp[0]
                src = hb.ptr + order[i % len(order)] * sz
                if form.startswith("raw"):
                    tk = s.submit_io_raw(src, fb.ptr, None, "", C.addressof(pb), xb.ptr)
                elif form == "bayer":
                    tk = s.submit_bayer_raw(BAYER, src, fb.ptr, None, "", C.addressof(pb), xb.ptr)
                else:
                    tk = s.submit_yuv_raw(Y.NV12 if form == "nv12" else Y.YUYV, src, fb.ptr, None, "", C.addressof(pb), xb.ptr)
                pending.append((tk, pb))
        for q in rings:
            for tk, pp in q["pending"]:
                q["stream"].wait(tk)
                pos_sum += pp[0]
            q["pending"].clear()

    run(8)
    pos_sum = 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run(nframes)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return nframes * len(rings) / dt, pos_sum / (nframes * len(rings)), rings[0]["host"][form][1]


def e2e_table(nframes=300, rounds=5):
    print(f"\n== end to end: 3 camera streams (1 / 10 / 50 % density), {nframes} frames each per run, round-robin, "
          f"4 tickets in flight per stream; forms alternated, {rounds} rounds ==")
    rings = make_rings()
    res = {f: [] for f in FORMS}
    meta = {}
    for _ in range(rounds):
        for form in res:
            fps, mean_pos, h2d = e2e(rings, form, nframes)
            res[form].append(fps)
            meta[form] = (mean_pos, h2d)
    print(f"{'form':>9} {'H2D B/frame':>12} {'mean pos':>10} {'frames/s median':>16} {'min':>8} {'max':>8}  per round")
    for form, v in res.items():
        print(f"{form:>9} {meta[form][1]:12d} {meta[form][0]:10.0f} {statistics.median(v):16.0f} {min(v):8.0f} {max(v):8.0f}  "
              + " ".join(f"{x:.0f}" for x in v))
    for q in rings:
        q["stream"].close()


def trace():
    """CVS_TRACE=1 timelines (stderr): per form, 8 warm-up and 40 timed frames on each of the three streams"""
    rings = make_rings()
    for form in FORMS:
        print(f"FORM {form}", file=sys.stderr, flush=True)
        e2e(rings, form, 40)


def trace_summary():
    env = dict(os.environ, CVS_TRACE="1")
    r = subprocess.run([sys.executable, __file__, "trace"], env=env, capture_output=True, text=True, timeout=900)
    print("\n== CVS_TRACE=1 (a run of its own; per form 3 streams x (8 warm-up + 40) frames, the 24 warm-up tickets dropped): "
          "mean device time per ticket ==")
    form, rows = None, {}
    pat = re.compile(r"h2d ([\d.]+)-([\d.]+) kern ([\d.]+)-([\d.]+) pos ([\d.]+) done ([\d.]+)")
    for line in r.stderr.splitlines():
        if line.startswith("FORM "):
            form = line.split()[1]
            rows[form] = []
        m = pat.search(line)
        if m and form:
            a = [float(x) for x in m.groups()]
            rows[form].append((a[1] - a[0], a[3] - a[2], a[5] - a[3]))
    for form, v in rows.items():
        v = v[24:]  # past the warm-up frames
        if v:
            print(f"{form:>9}: upload {np.mean([x[0] for x in v]):7.1f} us  kernels {np.mean([x[1] for x in v]):6.1f} us  "
                  f"kernels end -> payload on host {np.mean([x[2] for x in v]):7.1f} us  ({len(v)} tickets)")
    if r.returncode:
        print("trace run failed:", r.stderr[-600:])


if __name__ == "__main__":
    if sys.argv[1:] == ["trace"]:
        trace()
        sys.exit(0)
    card()
    peaks = {}
    pp = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pp):
        with open(pp) as fh:
            peaks = json.load(fh)
    bench_peak = float(peaks.get("hbm_gbs", 6650.0))
    measured = copy_peak()
    print(f"HBM copy peak: bench.py uses {bench_peak:.0f} GB/s ({'MEASURED_PEAKS.json' if peaks else 'its fallback'}); "
          f"a 1 GiB device-to-device copy here: {measured:.0f} GB/s (read + write)")
    kernel_times(bench_peak)
    e2e_table()
    trace_summary()
