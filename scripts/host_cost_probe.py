import ctypes as C, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import cudavideostream_b200 as cvs
w,h=1920,1080; n=3*w*h
jpgs=[open(os.path.join(ROOT,"tests","golden",f),"rb").read() for f in ("k1_f1.jpg","k1_f2.jpg")]
hb=[]
for j in jpgs:
    b=cvs.alloc_host(len(j)+64); b.array()[:len(j)]=np.frombuffer(j,dtype=np.uint8); hb.append((b,len(j)))
s=cvs.Stream(w,h,np.zeros(n,dtype=np.uint8))
outs=[(cvs.alloc_host(n+32),cvs.alloc_host(4*n+32),(C.c_uint*1)()) for _ in range(4)]
raw=cvs.alloc_host(n+64)
def burst(jpeg):
    ts=[]
    for rep in range(30):
        tk=[]
        t0=time.perf_counter()
        for i in range(4):
            fb,xb,pb=outs[i]
            if jpeg:
                b,nb=hb[i%2]; tk.append(s.submit_jpeg_raw(b.ptr,nb,fb.ptr,None,"",C.addressof(pb),xb.ptr))
            else:
                tk.append(s.submit_io_raw(raw.ptr,fb.ptr,None,"",C.addressof(pb),xb.ptr))
        t1=time.perf_counter()
        for t in tk: s.wait(t)
        t2=time.perf_counter()
        if rep>=5: ts.append(((t1-t0)/4*1e6,(t2-t1)/4*1e6))
    a=np.array(ts); return a[:,0].mean(), a[:,1].mean()
print("jpeg submit host us / wait us per frame:", burst(True))
print("raw  submit host us / wait us per frame:", burst(False))
