import sys, os, time
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
import numpy as np
from oracle import pyoracle as O
from tests.synth import synth_frame, warp_frame
O.set_num_threads(8)
t0=time.time()
a = synth_frame(0); b = warp_frame(a, 1000)
print('synth', time.time()-t0)
ks=[];ds=[]
for f in (a,b):
    k,d = O.Akaze(maximum_features=5000).extract(f); ks.append(k); ds.append(d); print('extract', len(d), time.time()-t0)
fi, fd = O.hamming_knn(ds[0], ds[1], 2); ri, rd = O.hamming_knn(ds[1], ds[0], 2)
fwd = np.where(fd[:, 0] + 24 <= fd[:, 1], fi[:, 0].astype(np.int64), -1)
rev = np.where(rd[:, 0] + 24 <= rd[:, 1], ri[:, 0].astype(np.int64), -1)
pairs = np.array([(i, j) for i, j in enumerate(fwd) if j >= 0 and rev[j] == i])
print('pairs', len(pairs), time.time()-t0)
def cal(k):
    x = (k['x'].astype(np.float64) - 960.0)/1000.0; y = (k['y'].astype(np.float64)-540.0)/1000.0
    v = np.stack([x,y,np.ones_like(x)],1); return v/np.linalg.norm(v,axis=1,keepdims=True)
ba = cal(ks[0][pairs[:,0]]); bb = cal(ks[1][pairs[:,1]])
np.savez('' + os.path.join(os.path.dirname(os.path.abspath(__file__)), 'bench_pair0.npz') + '', ba=ba, bb=bb, pairs=pairs)
