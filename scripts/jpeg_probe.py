"""Decode rate of cvs_decode_jpeg_device on the reference's fixture frames: the library's own decoder (cvs_jpeg.cuh) at
several subsequence lengths, with 1, 2 and 4 streams decoding side by side (rate and distance from OpenCV's pixels).
Run on the GPU box: python scripts/jpeg_probe.py"""
import os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if len(sys.argv) == 1:
    runs = [("own", dict(CVS_JPEG_DECODER="own", CVS_JPEG_SUB_BITS=str(sb))) for sb in (256, 512, 1024, 2048, 4096)]
    for name, extra in runs:
        env = dict(os.environ, **extra)
        r = subprocess.run([sys.executable, __file__, "run"], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=300)
        print(f"{name} {extra}:", r.stdout.decode().strip().splitlines()[-1] if r.stdout.strip() else "no output", flush=True)
    sys.exit(0)
sys.path.insert(0, ROOT)
import numpy as np, torch, cv2
import cudavideostream_b200 as cvs
w, h = 1920, 1080
n = 3 * w * h
gold = os.path.join(ROOT, "tests", "golden")
j = [open(os.path.join(gold, f), "rb").read() for f in ("k1_f1.jpg", "k1_f2.jpg")]
c = [cv2.imread(os.path.join(gold, f)).reshape(-1) for f in ("k1_f1.jpg", "k1_f2.jpg")]
NS = int(os.environ.get("JPEG_PROBE_NS", "4"))  # streams decoding side by side in the last measurement
ss = [cvs.Stream(w, h, np.zeros(n, dtype=np.uint8)) for _ in range(NS)]
ds = [torch.zeros(n + 64, dtype=torch.uint8, device="cuda") for _ in range(NS)]
sts = [torch.cuda.Stream() for _ in range(NS)]
g = []
for k in range(2):
    ss[0].decode_jpeg_device(j[k], ds[0].data_ptr(), sts[0].cuda_stream)
    torch.cuda.synchronize()
    g.append(ds[0][:n].cpu().numpy().copy())
dd = np.abs(g[0].astype(np.int16) - c[0].astype(np.int16))
changed = int((np.abs(g[0].astype(np.int16) - g[1].astype(np.int16)) > 20).sum())
rates = []
for ns in (1, 2, NS):
    K = 60
    for q in range(ns):
        ss[q].decode_jpeg_device(j[0], ds[q].data_ptr(), sts[q].cuda_stream)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        for q in range(ns):
            ss[q].decode_jpeg_device(j[i & 1], ds[q].data_ptr(), sts[q].cuda_stream)
    torch.cuda.synchronize()
    rates.append(K * ns / (time.perf_counter() - t0))
# device time of one decode
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
with torch.cuda.stream(sts[0]):
    e0.record()
    ss[0].decode_jpeg_device(j[0], ds[0].data_ptr(), sts[0].cuda_stream)
    e1.record()
torch.cuda.synchronize()
print(f"decodes/s with 1/2/{NS} streams {rates[0]:7.0f} {rates[1]:7.0f} {rates[2]:7.0f}  one decode {1e3 * e0.elapsed_time(e1):6.0f} us on the device  "
      f"vs OpenCV: max |d| {dd.max()} differing {100*(dd>0).mean():.2f} %  changed bytes f1->f2 {changed} (OpenCV 369350)")
