import sys, os
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0,ROOT); sys.path.insert(0,os.path.join(ROOT,'tests'))
import numpy as np, psd_b200, psd_rng
h=psd_b200.Handle([0])
S=[k%2 for k in range(10)]
A5=psd_rng.gen_uniform(1234,256,10,296)
out=psd_b200.gpschur_batched(A5,S,"L",handle=h)
print(int((out[5]!=0).sum()))
