"""End-to-end probe: frames/s through cvs_submit_io/cvs_wait from a pinned host ring, per density."""
import ctypes as C, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import cudavideostream_b200 as cvs
W, H = 1920, 1080
N = 3 * W * H
R, F = 16, int(os.environ.get("FRAMES", "300"))
st = torch.cuda.current_stream().cuda_stream
for d in (10000, 100000, 500000):
    fr = torch.empty((R + 1) * N, dtype=torch.uint8, device="cuda")
    cvs.synth.base_frame_device(fr.data_ptr(), W, H, 1, st)
    for t in range(R):
        cvs.synth.next_frame_device(fr.data_ptr() + t * N, fr.data_ptr() + (t + 1) * N, W, H, 1, t, d, st)
    torch.cuda.synchronize()
    hb = cvs.alloc_host(R * N)
    hb.array()[:] = fr[N:].cpu().numpy()
    s = cvs.Stream(W, H, fr[:N].cpu().numpy())
    out = [(cvs.alloc_host(N + 32), cvs.alloc_host(4 * N + 32), (C.c_uint * 1)()) for _ in range(4)]
    order = list(range(R)) + list(range(R - 2, 0, -1))
    def run(n):
        pend = []; tot = 0
        for i in range(n):
            fb, xb, pb = out[i % 4]
            if len(pend) == 4:
                tk, pp = pend.pop(0); s.wait(tk); tot += pp[0]
            pend.append((s.submit_io_raw(hb.ptr + order[i % len(order)] * N, fb.ptr, None, "", C.addressof(pb), xb.ptr), pb))
        for tk, pp in pend:
            s.wait(tk); tot += pp[0]
        return tot
    run(8)
    t0 = time.perf_counter(); tot = run(F); dt = time.perf_counter() - t0
    print(f"d={d} {F/dt:8.0f} fps  {dt/F*1e6:7.1f} us/frame  payload {5*tot/F/1e6:.2f} MB/frame  last {s.timing()}")
    s.close()
