"""Times the device-resident sequence path for one density (profiling helper; run on the GPU box)."""
import argparse, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cudavideostream_b200 as cvs

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=300)
ap.add_argument("--density", type=int, default=100000)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--mode", type=int, default=0)
ap.add_argument("--noise", type=int, default=0, help="K of the gaussian noise filter (0 = off)")
a = ap.parse_args()
W, H, T = a.width, a.height, a.frames
N = 3 * W * H
S = (N + 15) // 16 * 16
st = torch.cuda.current_stream().cuda_stream
fr = torch.empty((T + 1) * S, dtype=torch.uint8, device="cuda")
cvs.synth.base_frame_device(fr.data_ptr(), W, H, 1, st)
for t in range(T):
    cvs.synth.next_frame_device(fr.data_ptr() + t * S, fr.data_ptr() + (t + 1) * S, W, H, 1, t, a.density, st)
torch.cuda.synchronize()
cap = (N + 3) // 4 * 4
kw = {}
if a.noise:
    K = a.noise
    sig = K * K / 6.0
    x = np.arange(K, dtype=np.float32) - (K - 1) / 2.0
    g = (1.0 / (2.0 * np.pi * sig * sig)) * np.exp(-((x[:, None] ** 2 + x[None, :] ** 2) / (2.0 * sig * sig)))
    g = g.astype(np.float32); g /= g.sum(dtype=np.float32)
    kw = dict(noise_filter=True, ksize=K, kweights=g)
s = cvs.Stream(W, H, fr[:N].cpu().numpy(), mode=a.mode, max_sequence=max(T, 16), **kw)
pos = torch.zeros(T, dtype=torch.int32, device="cuda")
xs = torch.empty(T * cap, dtype=torch.int32, device="cuda")
df = torch.empty(T * cap, dtype=torch.uint8, device="cuda")
show = torch.empty(T * S, dtype=torch.uint8, device="cuda") if a.mode else None
def run():
    s.run_sequence_device(fr.data_ptr() + S, S, T, pos.data_ptr(), xs.data_ptr(), df.data_ptr(), cap,
                          show.data_ptr() if a.mode else 0, S, cuda_stream=st)
run(); torch.cuda.synchronize()
ms = []
for _ in range(a.reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    ms.append(e0.elapsed_time(e1))
try:
    s.sequence_status()
except Exception as e:
    print("status:", e)
sp = int(pos.to(torch.int64).sum())
m = min(ms)
print(f"{W}x{H} T={T} d={a.density} mode={a.mode} noiseK={a.noise} c={sp/(T*N):.4f} "
      f"best {m:.3f} ms  {m*1000/T:.2f} us/frame  hbm_model {(T*(N+4)+5*sp)/m/1e6:.0f} GB/s  alg {(T*(2*N+4)+6*sp)/m/1e6:.0f} GB/s")
