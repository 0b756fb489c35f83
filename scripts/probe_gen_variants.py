import sys, time, os
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0,ROOT); sys.path.insert(0,os.path.join(ROOT,'tests'))
import numpy as np, psd_b200, psd_rng
h=psd_b200.Handle([0])
S=[k%2 for k in range(10)]
A=psd_rng.gen_uniform(1234,64,10,2); psd_b200.gpschur_batched(A,S,"L",handle=h)
def run(A,S,lr):
    h.set_profiling(True); h.kernel_times()
    t0=time.time()
    out=psd_b200.gpschur_batched(A,S,lr,handle=h)
    t1=time.time()-t0
    kt=h.kernel_times()
    return round(kt['iterate_ms']/1e3,3), round(t1,3), int((out[5]!=0).sum())
A5=psd_rng.gen_uniform(1234,512,10,296)
A3=psd_rng.gen_uniform(1234,128,6,592)+1j*psd_rng.gen_uniform(1234,128,6,592,0,1)
cfgs=[({'PSD_DEEP_U':'4'},148),({'PSD_DEEP_U':'2'},148),({'PSD_DEEP_U':'4','PSD_GEN_WIDE':'1'},296),({'PSD_DEEP_U':'2','PSD_GEN_WIDE':'1'},296),({'PSD_DEEP_U':'8','PSD_GEN_WIDE':'1'},296)]
for env,B in cfgs:
    for k in ('PSD_NO_DEEP','PSD_GEN_WIDE','PSD_GEN_THREADS','PSD_DEEP_U'): os.environ.pop(k,None)
    os.environ.update(env)
    r=run(A5[:B],S,"L"); print(env,'C5',B,r,'problems/s %.2f'%(B/r[0]),flush=True)
    r=run(A3,[1,0,1,1,0,1],"R"); print(env,'C3 592',r,'problems/s %.1f'%(592/r[0]),flush=True)
