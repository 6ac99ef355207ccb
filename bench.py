#!/usr/bin/env python
"""bench.py -- throughput of the CUDAVideoStream hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through libcvs_b200.so)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                    # also writes what the last timed step computed

Headline workload (BASELINE.json configs[1]): 1080p BGR24 synthetic 300-frame sequences at change densities
1 % / 10 % / 50 %, thresholded diff + negative feedback + ordered compaction.  One STEP = one pass over the
three 300-frame sequences (900 frames, 5.6 GB of frames resident in HBM, so every frame is L2-cold).
`value` = frames/s with the frames already in HBM (device-resident sequence API); `e2e` = frames/s through the
pipelined drop-in call (cvs_submit_io/cvs_wait) with frames in pinned HOST memory, H2D and payload D2H inside
the timed region (the three camera streams of a GPU are interleaved, so both PCIe directions stay busy), with the
synchronous drop-in call (cvs_exec, what the unchanged server.cpp:139 does) next to it.

Side workloads, each event-timed with its own algorithmic-byte roofline (config.workloads[]):
  config3   1080p, Gaussian K=3 noise filter -> diff, weighted gray -> histogram -> two-max -> binarize   (3 2/3 + 6c) N
  config4   1080p, diff + heat map (mode 1) and diff + heat-map-red (mode 2)                             (3 + 6c) N
  config5   eight independent 3840x2160 streams, diff + compact, stream s on rank s mod N                (2 + 6c) N

Multi-GPU: one process per GPU, independent camera streams per rank, no collective on the data path (weak
scaling); torch.distributed is used only for the barrier and the max-over-ranks time.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1920, 1080
N = 3 * W * H
DENSITIES_PPM = (10000, 100000, 500000)
SEQ_FRAMES = 300
METRIC = "1080p frames/sec (diff+compact, 300-frame sequences at 1%/10%/50% change density)"
THR = 20
BASE_SEED = 0xC0DA5EED
W4K, H4K = 3840, 2160
N4K = 3 * W4K * H4K
C5_STREAMS, C5_FRAMES, C5_DENSITY = 8, 48, 100000
# --dump-outputs, per density: (xs, diff) entries sampled over the frames of the last step (float64 + float32, 12 bytes
# an entry) and bytes of the final reference frame (float32): three densities x 16 MB, under 64 MB.
DUMP_PAYLOAD_ENTRIES = 1 << 20
DUMP_REFERENCE_BYTES = 1 << 20


def workload_config(frames: int) -> dict:
    """The workload both arms run -- identical in `--impl ours` and `--impl reference` lines."""
    name = "1080p" if (W, H) == (1920, 1080) else "%dx%d" % (W, H)
    return {"workload": "%s_seq%d_d1_10_50" % (name, frames), "width": W, "height": H, "threshold": THR,
            "frames_per_sequence": frames, "sequences_per_step": len(DENSITIES_PPM), "densities_ppm": list(DENSITIES_PPM),
            "seed": "0x%X" % BASE_SEED, "streams_per_gpu": len(DENSITIES_PPM),
            "workloads": ["headline: 1080p diff+compact, 300-frame sequences at 1/10/50 % (BASELINE configs[1]; `value`)",
                          "config3_noiseK3_gray_weighted_binarize (configs[2])", "config4_heat_map, config4_heat_map_red (configs[3])",
                          "config5_8x3840x2160_streams, stream s on rank s mod N (configs[4])"],
            "l2": "inputs larger than L2: 3 x %.2f GB device-resident frame sequences per step" % (frames * N / 1e9)}


def algorithmic_bytes(nframes: int, sum_pos: int, n: int = None, per_frame_n: float = 2.0) -> int:
    """SURVEY.md section 8(d): (k + 6c) N + 4 per frame; k = 2 diff+compact (read cur N + read ref N, + write ref cN +
    payload 5cN + count), 3 with one fused display frame, 3 2/3 for config 3."""
    n = N if n is None else n
    return int(nframes * (per_frame_n * n + 4) + 6 * sum_pos)


def hbm_model_bytes(nframes: int, sum_pos: int) -> int:
    """Bytes that must cross HBM when the reference stays on chip: read cur N + payload 5 pos + count."""
    return nframes * (N + 4) + 5 * sum_pos


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (pynvml)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def result(self):
        self.stop_flag = True
        if self.is_alive():
            self.join(timeout=1)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU loop (oracle restatement of tests/cuda_streaming/test.cu:560-576), one
# independent camera stream per host thread, on the first frames of the very sequences the GPU arm is timed on.
# ------------------------------------------------------------------------------------------------------
CPU_RING = 12  # frames of each density's sequence the CPU legs walk (forth and back)
_RINGS = None


def cpu_rings():
    """(base, ring) per density: frames 1..CPU_RING of the bench sequences (seed 0xC0DA5EED, rank 0), generated by the
    oracle's C twin of the synthetic camera, walked forth and back so consecutive frames stay one step apart."""
    global _RINGS
    if _RINGS is None:
        from oracle import oracle as orc
        _RINGS = []
        for d in DENSITIES_PPM:
            base, fr = orc.synth_sequence(W, H, CPU_RING, d, BASE_SEED)
            _RINGS.append((base, np.ascontiguousarray(np.concatenate([fr, fr[-2:0:-1]]))))
    return _RINGS


def cpu_run(target_seconds: float, threads: int):
    """Times the CPU path on a bounded sample.  Returns dict(value=frames/s, cores, sample, ...)."""
    from oracle import oracle as orc
    orc.build()
    rings = cpu_rings()
    t_cal = sum(orc.bench_diff_compact(r, b, THR, 1, threads)[0] for b, r in rings)  # one frame per thread per density
    iters = max(1, int(target_seconds / max(t_cal, 1e-3)))
    iters = min(iters, 50)
    sec = 0.0
    frames = 0
    sum_pos = 0
    for b, r in rings:
        s, nf, sp = orc.bench_diff_compact(r, b, THR, iters, threads)
        sec += s
        frames += nf
        sum_pos += sp
    return {"value": frames / sec, "seconds": sec, "frames": frames, "cores": threads, "kind": "port",
            "unit": "frames/s", "realised_c": sum_pos / (frames * N),
            "sample": f"{iters} frames x {threads} independent streams x 3 densities (1/10/50 %): the first {CPU_RING} "
                      f"frames of the bench's own 1080p sequences (seed 0x{BASE_SEED:X}) walked forth and back, "
                      f"oracle/cvs_oracle.c orc_diff_compact (test.cu:560-576) -O2, frames in host RAM"}


def cpu_single_thread(frames_per_density: int = 4):
    """SURVEY.md section 8(d): the reference's compute runs on ONE thread (server.cpp:70-146) and its Makefile ships
    -O0 (server/Makefile:13).  A few frames per density of the same workload, one thread, -O2 and -O0 builds."""
    from oracle import oracle as orc
    orc.build()
    out = {}
    for name, o0 in (("O2", False), ("O0", True)):
        sec = 0.0
        for b, r in cpu_rings():
            sec += orc.bench_diff_compact(r, b, THR, frames_per_density, 1, o0=o0)[0]
        out["frames_per_s_1thread_" + name] = 3 * frames_per_density / sec
    return out


def reference_binaries(gpu: bool):
    """The reference's OWN code where it could be compiled (oracle/_ref/, built from the unmodified sources by
    oracle/build_ref.py): ms per 1080p frame between readCap() returning and writeShow() being called in the
    unmodified server.cpp main loop.  cpu = its CPU filter chain (server.cpp:96-135: gray, histogram, two-max,
    binarize -- NOT the diff, which is commented out there); refgpu = its own kernels.cu on this GPU (exec_core incl.
    its synchronous H2D/D2H); dropin = the same server.cpp linked against libcvs_b200.so."""
    try:
        from oracle import oracle as orc, ref_server
        base, fr = orc.synth_sequence(W, H, 10, 100000, BASE_SEED)
        out = {}
        names = ["ref_server_cpu", "ref_server_cpu_O0"] + (["ref_server_refgpu", "ref_server_dropin"] if gpu else [])
        for name in names:
            if ref_server.binary(name) is None:
                continue
            try:
                _, times = ref_server.run(name, W, H, base, fr, want_times=True, timeout=120)
                out[name + "_ms_per_frame"] = float(np.median(times[2:])) / 1e6
            except Exception as e:  # the reference's kernels read/write past their buffers: a fault is theirs
                out[name + "_error"] = str(e)[:200]
        if out:
            out["what"] = ("median ms per 1080p frame (10 % density) inside the reference's unmodified server.cpp loop, "
                           "readCap() -> writeShow(); kind: reference")
        return out or None
    except Exception:
        return None


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    t0 = time.time()
    vals = []
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_run(2.0, threads)
    for _ in range(args.steps):
        vals.append(cpu_run(max(args.ref_seconds / 7.0, args.ref_seconds / args.steps), threads))
    frames = sum(v["frames"] for v in vals)
    sec = sum(v["seconds"] for v in vals)
    value = frames / sec
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sec / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.frames),
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": vals[0]["sample"], "realised_c": vals[0]["realised_c"],
                             "single_thread": cpu_single_thread(),
                             "reference_binaries": reference_binaries(gpu=False)},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.time() - t0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def gaussian_k3():
    """computeGaussianKernel, server/src/server.cpp:20-36 (K = 3, sigma = K*K/6)."""
    K = 3
    sigma = np.float32(K * K / 6.0)
    k = np.empty(K * K, dtype=np.float32)
    total = np.float32(0)
    for i in range(K):
        for j in range(K):
            x = np.float32(i - (K - 1) / 2.0)
            y = np.float32(j - (K - 1) / 2.0)
            v = (1.0 / (2.0 * np.pi * float(sigma) * float(sigma))) * np.exp(-((float(x) * float(x) + float(y) * float(y)) / (2.0 * float(sigma) * float(sigma))))
            k[i * K + j] = np.float32(v)
            total = np.float32(total + k[i * K + j])
    return (k / total).astype(np.float32)


def dump_slots(pos: np.ndarray, per_frame: int) -> np.ndarray:
    """[T, per_frame] payload slots sampled from each frame's count: the same seeded fractions of every count, so two
    builds that agree on `pos` are compared at the same entries."""
    u = np.sort(np.random.default_rng(BASE_SEED).random(per_frame))
    return (u[None, :] * np.asarray(pos, dtype=np.int64)[:, None]).astype(np.int64)


def dump_reference_index(n: int) -> np.ndarray:
    """Sorted, seeded byte positions of a reference frame of n bytes (all of them when n <= DUMP_REFERENCE_BYTES)."""
    if n <= DUMP_REFERENCE_BYTES:
        return np.arange(n)
    return np.sort(np.random.default_rng(BASE_SEED + 1).choice(n, size=DUMP_REFERENCE_BYTES, replace=False))


def dump_outputs(out_dir: str, seqs, T: int, torch) -> None:
    """What the headline's last timed step returned to its caller, per density: DIR/d<ppm>_pos.npy (every frame's
    count), d<ppm>_xs.npy and d<ppm>_diff.npy ([T, S] entries at dump_slots(pos, S); -1 where a frame has none) and
    d<ppm>_reference.npy (the stream's reference frame after the step, at dump_reference_index(N))."""
    os.makedirs(out_dir, exist_ok=True)
    per_frame = max(1, DUMP_PAYLOAD_ENTRIES // T)
    ref_idx = dump_reference_index(N)
    for q in seqs:
        pos = q["pos"].cpu().numpy()
        slots = dump_slots(pos, per_frame) + np.arange(T, dtype=np.int64)[:, None] * q["cap"]
        flat = torch.from_numpy(slots).to(q["xs"].device)
        xs = q["xs"][flat].cpu().numpy().astype(np.float64)
        diff = q["diff"][flat].cpu().numpy().astype(np.float32)
        xs[pos == 0], diff[pos == 0] = -1, -1
        arrays = {"pos": pos.astype(np.float64), "xs": xs, "diff": diff,
                  "reference": q["stream"].reference()[ref_idx].astype(np.float32)}
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, "d%d_%s.npy" % (q["d"], name)), a)


def ours(args):
    import torch
    import torch.distributed as dist
    import cudavideostream_b200 as cvs

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # one host thread + one context per GPU, pinned buffers NUMA-local to it (SURVEY.md section 8e)
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        except Exception:
            pass
        dist.init_process_group("nccl", device_id=dev)
    cvs.load_library()
    st = torch.cuda.current_stream().cuda_stream
    T = args.frames
    seed = BASE_SEED ^ (rank * 0x9E3779B9)
    cap = (N + 3) // 4 * 4  # worst case: every byte of a frame changes

    def device_sequence(w, h, nframes, density, sd):
        n = 3 * w * h
        frames = torch.empty((nframes + 1) * n, dtype=torch.uint8, device=dev)
        cvs.synth.base_frame_device(frames.data_ptr(), w, h, sd, st)
        for t in range(nframes):
            cvs.synth.next_frame_device(frames.data_ptr() + t * n, frames.data_ptr() + (t + 1) * n, w, h, sd, t, density, st)
        return frames

    # ---- headline: device-resident sequences, one Stream (reference state) per density
    seqs = []
    for d in DENSITIES_PPM:
        frames = device_sequence(W, H, T, d, seed)
        torch.cuda.synchronize()
        base = frames[:N].cpu().numpy()
        s = cvs.Stream(W, H, base, threshold=THR, device=local, max_sequence=max(T, 16))
        seqs.append({"d": d, "frames": frames, "stream": s, "cap": cap,
                     "pos": torch.zeros(T, dtype=torch.int32, device=dev),
                     "xs": torch.empty(T * cap, dtype=torch.int32, device=dev),
                     "diff": torch.empty(T * cap, dtype=torch.uint8, device=dev)})

    def run_seq(q):
        q["stream"].run_sequence_device(q["frames"].data_ptr() + N, N, T, q["pos"].data_ptr(), q["xs"].data_ptr(),
                                        q["diff"].data_ptr(), q["cap"], cuda_stream=st)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        for q in seqs:
            run_seq(q)
    torch.cuda.synchronize()
    for q in seqs:
        q["stream"].sequence_status()
    launches0 = sum(q["stream"].launch_count() for q in seqs)

    sampler = ClockSampler(local)
    sampler.start()
    evs = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in seqs]
           for _ in range(args.steps)]
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        for i, q in enumerate(seqs):
            evs[k][i][0].record()
            run_seq(q)
            evs[k][i][1].record()
    e1.record()
    barrier()
    clocks = sampler.result()
    elapsed_ms = e0.elapsed_time(e1)
    for q in seqs:
        q["stream"].sequence_status()
    launches = sum(q["stream"].launch_count() for q in seqs) - launches0
    if args.dump_outputs and rank == 0:  # before the side workloads reuse the payload buffers
        dump_outputs(args.dump_outputs, seqs, T, torch)
    # per-launch durations of the stream kernel and the algorithmic bytes each launch moved
    per_density = []
    tot_alg = tot_hbm = 0
    tot_ms = 0.0
    for i, q in enumerate(seqs):
        ms = [evs[k][i][0].elapsed_time(evs[k][i][1]) for k in range(args.steps)]
        sp = int(q["pos"].to(torch.int64).sum().item())
        alg, hbm = algorithmic_bytes(T, sp), hbm_model_bytes(T, sp)
        mean_ms = float(np.mean(ms))
        per_density.append({"density_ppm": q["d"], "realised_c": sp / (T * N), "ms_per_launch": mean_ms,
                            "us_per_frame": 1e3 * mean_ms / T,
                            "frames_per_s": T / (mean_ms * 1e-3), "algorithmic_GBps": alg / (mean_ms * 1e-3) / 1e9,
                            "hbm_model_GBps": hbm / (mean_ms * 1e-3) / 1e9})
        tot_alg += alg
        tot_hbm += hbm
        tot_ms += mean_ms
    frames_done = args.steps * T * len(seqs)

    # whole-job view: max over ranks of the device time, sum over ranks of the work (no data-path collective)
    elapsed_s, (frames_total, launches_total) = cvs.sharding.reduce_job(elapsed_ms * 1e-3, [frames_done, launches], dev)
    elapsed_ms = elapsed_s * 1e3
    value = frames_total / elapsed_s

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    # ---- end to end through the drop-in call: frames in pinned host memory, pipelined submit/wait
    e2e = e2e_run(cvs, torch, args, seqs, local, barrier)

    # ---- side workloads (BASELINE.json configs 3, 4, 5), event-timed like the headline
    workloads = [] if args.no_side else side_workloads(cvs, torch, args, seqs, dev, local, rank, world, st, peak, barrier,
                                                       device_sequence)

    achieved = tot_alg / (tot_ms * 1e-3) / 1e9
    achieved_hbm = tot_hbm / (tot_ms * 1e-3) / 1e9
    traffic = traffic_src = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            tj = json.load(fh)
            # ncu dram__bytes_read.sum + dram__bytes_write.sum per frame (mean of the three densities) x frames per launch
            traffic = tj["dram_bytes_per_frame_mean"] * T if (W, H) == (1920, 1080) else None
            traffic_src = "static: profiles/traffic.json (one ncu --set full capture, %s), not measured in this run" % tj.get("kernel", "k_stream")
    except Exception:
        pass

    if rank == 0:
        cfg = workload_config(T)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        kname = os.environ.get("CVS_STREAM_KERNEL", "ws")
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": cfg, "per_density": per_density, "workloads": workloads,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0, "traffic": traffic,
                             "traffic_source": traffic_src,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                             "kernel": "cvs::%s<0,false,%s> (one launch = one %d-frame sequence)" % (
                                 "k_stream" if kname == "v1" else "k_stream_ws",
                                 "true" if (N + 95) // 96 <= 512 * sms else "false", T),
                             "achieved_hbm_model": achieved_hbm, "frac_hbm_model": achieved_hbm / peak,
                             "note": "achieved = SURVEY 8(d) algorithmic bytes (2+6c)N+4 per frame / event-timed launch; "
                                     "hbm_model counts only bytes that must cross HBM when the reference stays on chip "
                                     "((1+5c)N+4)"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches_total}
        if world == 1 and not args.no_cpu:
            cb = cpu_run(args.cpu_seconds, os.cpu_count() or 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "realised_c")}
            line["cpu_baseline"]["single_thread"] = cpu_single_thread()
            line["cpu_baseline"]["reference_binaries"] = reference_binaries(gpu=True)
        print(json.dumps(line), flush=True)
    for q in seqs:
        q["stream"].close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def side_workloads(cvs, torch, args, seqs, dev, local, rank, world, st, peak, barrier, device_sequence):
    """BASELINE.json configs 3, 4 and 5 as extra event-timed entries (the headline `value` stays config 2)."""
    T = args.frames
    reps = max(1, min(args.steps, 3))
    out = []
    frames10 = seqs[1]["frames"]   # the 10 % sequence of the headline
    base10 = frames10[:N].cpu().numpy()
    cap = seqs[1]["cap"]
    pos = torch.zeros(T, dtype=torch.int32, device=dev)
    xs = seqs[0]["xs"]             # payload buffers are reused: the workloads run one after the other
    df = seqs[0]["diff"]
    show = torch.empty(T * N, dtype=torch.uint8, device=dev)

    def timed(fn, n_rep):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(n_rep):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return float(np.mean(ms))

    specs = [("config3_noiseK3_gray_weighted_binarize", dict(mode=5, noise_filter=True, ksize=3, kweights=gaussian_k3()), 11.0 / 3.0,
              "(3 2/3 + 6c) N: diff+compact + gray byte written and read + binarised frame written"),
             ("config4_heat_map", dict(mode=1), 3.0, "(3 + 6c) N: diff+compact + one display frame"),
             ("config4_heat_map_red", dict(mode=2), 3.0, "(3 + 6c) N: diff+compact + one display frame")]
    for name, kw, k_n, note in specs:
        s = cvs.Stream(W, H, base10, threshold=THR, device=local, max_sequence=max(T, 16), **kw)
        l0 = s.launch_count()

        def run():
            s.run_sequence_device(frames10.data_ptr() + N, N, T, pos.data_ptr(), xs.data_ptr(), df.data_ptr(), cap,
                                  show.data_ptr(), N, cuda_stream=st)
        ms = timed(run, reps)
        s.sequence_status()
        sp = int(pos.to(torch.int64).sum().item())
        alg = algorithmic_bytes(T, sp, N, k_n)
        gbs = alg / (ms * 1e-3) / 1e9
        out.append({"name": name, "frames": T, "us_per_frame": 1e3 * ms / T, "frames_per_s": T / (ms * 1e-3),
                    "realised_c": sp / (T * N), "algorithmic_GBps": gbs, "frac": gbs / peak, "bytes_model": note,
                    "launches_per_sequence": (s.launch_count() - l0) // (reps + 1)})
        s.close()
    del show

    # ---- config 5: eight independent 3840x2160 streams, stream sid on rank sid mod world
    mine = cvs.sharding.my_streams(C5_STREAMS, rank, world)
    T5 = C5_FRAMES
    cap5 = N4K  # a re-run starts from the reference the previous run left behind: its first frame is dense
    pos5 = torch.zeros(T5, dtype=torch.int32, device=dev)
    xs5 = xs[:T5 * cap5] if xs.numel() >= T5 * cap5 else torch.empty(T5 * cap5, dtype=torch.int32, device=dev)
    df5 = df[:T5 * cap5] if df.numel() >= T5 * cap5 else torch.empty(T5 * cap5, dtype=torch.uint8, device=dev)
    st4 = []
    for sid in mine:
        fr = device_sequence(W4K, H4K, T5, C5_DENSITY, cvs.sharding.stream_seed(BASE_SEED, sid))
        torch.cuda.synchronize()
        st4.append((sid, fr, cvs.Stream(W4K, H4K, fr[:N4K].cpu().numpy(), threshold=THR, device=local, max_sequence=T5)))

    def run5():
        for sid, fr, s in st4:
            s.run_sequence_device(fr.data_ptr() + N4K, N4K, T5, pos5.data_ptr(), xs5.data_ptr(), df5.data_ptr(), cap5,
                                  cuda_stream=st)
    run5()
    torch.cuda.synchronize()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        run5()
    b.record()
    barrier()
    ms5 = a.elapsed_time(b) / reps
    sp5 = 0
    for sid, fr, s in st4:
        s.sequence_status()
    if st4:
        sp5 = int(pos5.to(torch.int64).sum().item()) * len(st4)  # pos5 holds the last stream's counts; same density everywhere
    sec5, (nfr5, sp5) = cvs.sharding.reduce_job(ms5 * 1e-3, [T5 * len(st4), sp5], dev)
    alg5 = algorithmic_bytes(nfr5, sp5, N4K, 2.0)
    per_gpu = alg5 / sec5 / 1e9 / world
    out.append({"name": "config5_8x3840x2160_streams", "streams": C5_STREAMS, "streams_per_gpu": len(mine) if world > 1 else C5_STREAMS,
                "frames_per_stream": T5, "density_ppm": C5_DENSITY, "frames_per_s": nfr5 / sec5,
                "us_per_frame_per_gpu": 1e6 * sec5 / max(1, T5 * len(mine)), "realised_c": sp5 / max(1, nfr5 * N4K),
                "algorithmic_GBps_per_gpu": per_gpu, "frac": per_gpu / peak,
                "bytes_model": "(2 + 6c) N at 3840x2160; whole-job 4K frames/s = frames of all ranks / max-over-ranks device time"})
    for sid, fr, s in st4:
        s.close()
    return out


def e2e_run(cvs, torch, args, seqs, local, barrier):
    """frames/s through cvs_submit_io/cvs_wait with HOST frames: per frame an H2D of N bytes from pinned memory and a
    D2H of the count + payload.  The host ring of each density holds R consecutive frames walked back and forth so
    that consecutive submissions are always one synthetic step apart.  The three camera streams of the GPU are
    submitted round-robin, so the H2D of one overlaps the payload D2H of another."""
    R = args.e2e_ring
    frames_per_density = args.e2e_frames
    rings = []
    for q in seqs:
        hb = cvs.alloc_host(R * N)
        arr = hb.array()
        src = q["frames"]
        for t in range(R):
            arr[t * N:(t + 1) * N] = src[(t + 1) * N:(t + 2) * N].cpu().numpy()
        base = src[:N].cpu().numpy()
        s = cvs.Stream(W, H, base, threshold=THR, device=local)
        out = [(cvs.alloc_host(N + 32), cvs.alloc_host(4 * N + 32), (C.c_uint * 1)()) for _ in range(4)]
        rings.append({"hb": hb, "stream": s, "out": out, "pending": [], "base": base})
    order = list(range(R)) + list(range(R - 2, 0, -1))

    def run(nframes, wire=False):
        """wire: the opt-in compact CVW1 frame (cvs_submit_wire) instead of the reference's (pos, xs, diff)."""
        d2h = 0

        def account(pp, xb):
            if wire:  # the encoded frame lies in xb (the slot's largest pinned buffer); its header holds the size
                return int(cvs.wire.size_of(xb.array()[:16]))
            return 4 + 5 * pp[0]

        for i in range(nframes):
            for q in rings:
                s, hb, out, pending = q["stream"], q["hb"], q["out"], q["pending"]
                fb, xb, pb = out[i % 4]
                if len(pending) == 4:
                    tk, pp, oxb = pending.pop(0)
                    s.wait(tk)
                    d2h += account(pp, oxb)
                # frames stay in the pinned capture ring; the payload bytes go to the slot's own pinned buffer
                src = order[i % len(order)]
                if wire:
                    pending.append((s.submit_wire_raw(hb.ptr + src * N, xb.ptr, None, ""), pb, xb))
                else:
                    pending.append((s.submit_io_raw(hb.ptr + src * N, fb.ptr, None, "", C.addressof(pb), xb.ptr), pb, xb))
        for q in rings:
            for tk, pp, oxb in q["pending"]:
                q["stream"].wait(tk)
                d2h += account(pp, oxb)
            q["pending"].clear()
        return d2h

    run(min(8, frames_per_density))
    launches0 = sum(q["stream"].launch_count() for q in rings)
    barrier()
    t0 = time.perf_counter()
    d2h = run(frames_per_density)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    nfr = frames_per_density * len(rings)
    launches = sum(q["stream"].launch_count() for q in rings) - launches0
    dt, (nfr, d2h, launches) = cvs.sharding.reduce_job(dt, [nfr, d2h, launches], torch.device("cuda", local))
    res = {"value": nfr / dt, "unit": "frames/s", "h2d_bytes_per_step": N * nfr, "d2h_bytes_per_step": d2h,
           "frames": nfr, "seconds": dt, "gpu_launches": launches,
           "note": "one e2e step = %d frames per density x 3 densities per GPU through cvs_submit_io/cvs_wait from a "
                   "pinned host ring, the three streams submitted round-robin" % frames_per_density}

    # ---- the same loop with the opt-in compact wire format (5 -> ~2 bytes per entry over PCIe)
    for q in rings:
        q["stream"].reset(q["base"])
    run(min(8, frames_per_density), wire=True)
    barrier()
    t0 = time.perf_counter()
    d2h_w = run(frames_per_density, wire=True)
    torch.cuda.synchronize()
    dt_w = time.perf_counter() - t0
    dt_w, (nfr_w, d2h_w) = cvs.sharding.reduce_job(dt_w, [frames_per_density * len(rings), d2h_w], torch.device("cuda", local))
    res["wire_cvw1"] = {"value": nfr_w / dt_w, "unit": "frames/s", "d2h_bytes_per_step": d2h_w,
                        "note": "same frames through cvs_submit_wire: per-tile counts + one-byte offsets + values "
                                "(include/cvs_b200.h), opt-in; the default stays the reference's format"}

    # ---- capture-side decode on the GPU: the camera's JPEG bitstream in, payload out (cvs_submit_jpeg).  Real
    #      camera frames (the reference's own fixture pair, 0.43 MB each instead of 6.2 MB raw), alternating
    try:
        res["jpeg_ingest"] = jpeg_leg(cvs, torch, local, min(frames_per_density, 200), barrier=barrier)
    except Exception as e:  # nvJPEG missing on the box, fixtures not shipped ...
        res["jpeg_ingest"] = {"unavailable": str(e)[:160]}

    # ---- the synchronous drop-in call (cvs_exec: what the unchanged server.cpp:139 does), one stream at a time
    nsync = min(args.sync_frames, frames_per_density)
    per = []
    t_all, f_all = 0.0, 0
    for q, sq in zip(rings, seqs):
        s, hb = q["stream"], q["hb"]
        s.reset(q["base"])
        fb, xb, pb = q["out"][0]
        src = hb.array()
        # cvs_exec works in place on the frame buffer (kernels.cu:522): copy the captured frame into it first, as the
        # capture thread does; that host copy is outside the timed call
        times = []
        for i in range(nsync):
            k = order[i % len(order)]
            fb.array()[:N] = src[k * N:(k + 1) * N]
            t1 = time.perf_counter()
            s.exec_raw(fb.ptr, None, "", pb, xb.ptr)
            times.append(time.perf_counter() - t1)
        tm = s.timing()
        tt = float(np.sum(times[2:]))
        t_all += tt
        f_all += len(times) - 2
        per.append({"density_ppm": sq["d"], "frames_per_s": (len(times) - 2) / tt, "last_frame_us": tm})
    res["sync_exec"] = {"value": f_all / t_all, "unit": "frames/s", "per_density": per,
                        "note": "cvs_exec (synchronous H2D + kernels + D2H per call, pinned buffers), host clock around the call"}
    for q in rings:
        q["stream"].close()
    return res


def jpeg_leg(cvs, torch, local, nframes, nstreams=3, barrier=lambda: None):
    """frames/s through cvs_submit_jpeg/cvs_wait: H2D of the JPEG bitstream, GPU decode (the library's own kernels,
    cvs_jpeg.cuh: bit for bit OpenCV's pixels), diff+compact, payload D2H -- `nstreams` camera streams interleaved as in
    the e2e leg, one stream alone, and the same camera frames uploaded raw (cvs_submit_io) for comparison."""
    gold = os.path.join(ROOT, "tests", "golden")
    jpgs = [open(os.path.join(gold, f), "rb").read() for f in ("k1_f1.jpg", "k1_f2.jpg")]
    w, h = 1920, 1080
    n = 3 * w * h
    st = torch.cuda.current_stream().cuda_stream
    streams = [cvs.Stream(w, h, np.zeros(n, dtype=np.uint8), threshold=THR, device=local) for _ in range(nstreams)]
    d = torch.zeros(n + 64, dtype=torch.uint8, device="cuda")
    raw = []
    for j in jpgs:  # the decoded frames, for the raw-upload comparison
        streams[0].decode_jpeg_device(j, d.data_ptr(), st)
        torch.cuda.synchronize()
        streams[0].sequence_status()
        r = cvs.alloc_host(n + 64)
        r.array()[:n] = d[:n].cpu().numpy()
        raw.append(r)
    hb = []
    for j in jpgs:
        b = cvs.alloc_host(len(j) + 64)
        b.array()[:len(j)] = np.frombuffer(j, dtype=np.uint8)
        hb.append((b, len(j)))
    outs = [[(cvs.alloc_host(n + 32), cvs.alloc_host(4 * n + 32), (C.c_uint * 1)()) for _ in range(4)] for _ in range(nstreams)]

    from cudavideostream_b200 import wire as wirefmt
    wouts = [[cvs.alloc_host(wirefmt.bound(w, h) + 64) for _ in range(4)] for _ in range(nstreams)]

    def run(k, ns, jpeg=True, wire=False):
        pend, d2h, h2d = [[] for _ in range(ns)], 0, 0
        for q in range(ns):
            streams[q].reset(raw[0].array()[:n])
        for i in range(k):
            for q in range(ns):
                s = streams[q]
                fb, xb, pb = outs[q][i % 4]
                if len(pend[q]) == 4:
                    tk, pp = pend[q].pop(0)
                    s.wait(tk)
                    d2h += wirefmt.size_of(pp.array()) if wire else 4 + 5 * pp[0]
                if wire:
                    b, nb = hb[(i + 1) % 2]
                    h2d += nb
                    wb = wouts[q][i % 4]
                    pend[q].append((s.submit_jpeg_wire_raw(b.ptr, nb, wb.ptr, None, ""), wb))
                elif jpeg:
                    b, nb = hb[(i + 1) % 2]
                    h2d += nb
                    pend[q].append((s.submit_jpeg_raw(b.ptr, nb, fb.ptr, None, "", C.addressof(pb), xb.ptr), pb))
                else:
                    h2d += n
                    pend[q].append((s.submit_io_raw(raw[(i + 1) % 2].ptr, fb.ptr, None, "", C.addressof(pb), xb.ptr), pb))
        for q in range(ns):
            for tk, pp in pend[q]:
                streams[q].wait(tk)
                d2h += wirefmt.size_of(pp.array()) if wire else 4 + 5 * pp[0]
        return h2d, d2h

    def timed(k, ns, jpeg=True, wire=False):  # whole job: frames of all ranks / max-over-ranks time
        run(8, ns, jpeg, wire)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        h2d, d2h = run(k, ns, jpeg, wire)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt, (nfr, h2d, d2h) = cvs.sharding.reduce_job(dt, [k * ns, h2d, d2h], torch.device("cuda", local))
        return nfr / dt, h2d, d2h

    v, h2d, d2h = timed(nframes, nstreams)
    v1, _, _ = timed(nframes, 1)
    vr, h2dr, _ = timed(nframes, nstreams, jpeg=False)
    vw, h2dw, d2hw = timed(nframes, nstreams, wire=True)
    for s in streams:
        s.close()
    # what the reference does with the same bitstreams: OpenCV (libjpeg-turbo) on one host thread, as its capture
    # thread runs it (server/src/threads.cpp:32-41, :118)
    ref_cpu = None
    try:
        import cv2
        bufs = [np.frombuffer(j, dtype=np.uint8) for j in jpgs]
        cv2.imdecode(bufs[0], cv2.IMREAD_COLOR)
        t0, k = time.perf_counter(), 0
        while time.perf_counter() - t0 < 1.0:
            cv2.imdecode(bufs[k & 1], cv2.IMREAD_COLOR)
            k += 1
        ms = 1e3 * (time.perf_counter() - t0) / k
        ref_cpu = {"opencv_imdecode_ms_per_frame": ms, "frames_per_s_one_thread": 1e3 / ms,
                   "what": "cv2.imdecode of the same two bitstreams on one host thread (the reference's capture-side decode); "
                           "same pixels as the GPU decoder, bit for bit"}
    except Exception as e:  # no OpenCV on the box
        ref_cpu = {"unavailable": str(e)[:120]}
    return {"value": v, "unit": "frames/s", "streams_per_gpu": nstreams, "reference_cpu_decode": ref_cpu, "frames_per_gpu": nframes * nstreams, "h2d_bytes": h2d,
            "d2h_bytes": d2h,
            "one_stream": v1, "same_frames_uploaded_raw": {"value": vr, "h2d_bytes": h2dr},
            "jpeg_in_cvw1_out": {"value": vw, "h2d_bytes": h2dw, "d2h_bytes": d2hw,
                                 "note": "cvs_submit_jpeg_wire: both opt-ins, the fewest bytes across PCIe in either direction"},
            "decoder": os.environ.get("CVS_JPEG_DECODER", "own (cvs_jpeg.cuh), nvJPEG for forms it does not cover"),
            "note": "the reference's camera frames f1.jpg / f2.jpg alternating (about 6 % of the bytes change) on every stream; "
                    "cvs_submit_jpeg decodes the bitstream on the device (hand-written kernels, pixels identical to OpenCV's), "
                    "0.43 MB instead of 6.2 MB cross PCIe per frame"}


def main():
    global W, H, N, METRIC
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=SEQ_FRAMES, help="frames per sequence")
    ap.add_argument("--e2e-frames", type=int, default=300, help="frames per density in the end-to-end leg")
    ap.add_argument("--e2e-ring", type=int, default=16)
    ap.add_argument("--sync-frames", type=int, default=60, help="frames per density through the synchronous cvs_exec")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-side", action="store_true", help="skip the side workloads (configs 3, 4, 5)")
    ap.add_argument("--ref-seconds", type=float, default=20.0, help="--impl reference: CPU seconds over all steps")
    ap.add_argument("--width", type=int, default=W, help="frame width (default: the 1080p headline workload)")
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's last-step payload of the headline (per density: counts, a "
                         "seeded sample of (xs, diff) and of the reference frame) as DIR/*.npy, float32/float64, under "
                         "64 MB, to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if (args.width, args.height) != (W, H):
        # other frame sizes for the headline loop (experiments); the driver runs the 1080p default
        W, H = args.width, args.height
        N = 3 * W * H
        METRIC = "%dx%d frames/sec (diff+compact, %d-frame sequences at 1%%/10%%/50%% change density)" % (W, H, args.frames)
    if args.impl == "reference":
        return reference_arm(args)
    return ours(args)


if __name__ == "__main__":
    sys.exit(main())
