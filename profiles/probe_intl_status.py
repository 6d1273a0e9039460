import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0]=[ROOT, ROOT+'/ms-eetc_b200']
import numpy as np, torch
import __graft_entry__ as ge
ge.build()
import bench
from mseetc.ocp import casadiSolver
from mseetc.train import Train
from mseetc.track import Track
train = Train(config={'id': 'NL_Intercity_VIRM6'}); track = Track(config={'id': 'CH_StGallen_Wil'})
opts = dict(bench.OPTS); opts['integrateLosses']=True
solver = casadiSolver(train, track, opts)
tmin = float(np.atleast_1d(solver.minimum_time()[0])[0])
n=4096
T = tmin * (0.8 + 0.4 * np.arange(n) / (n - 1))
for lanes in ('auto', 1):
    solver.sweepLanes = lanes; solver._handle=None; solver._pool=None
    res = solver.solve_batch(T)
    st=np.asarray(res['status']); it=np.asarray(res['iters']); feas = T>=tmin
    bad=np.flatnonzero(feas & ~((st==0)|(st==6)))
    print('lanes',lanes,'hist',{int(k):int((st[feas]==k).sum()) for k in np.unique(st[feas])}, 'bad', len(bad), 'T/Tmin of bad', np.round(T[bad][:10]/tmin,4), 'iters', it[bad][:10], 'kkt', np.asarray(res['kkt'])[bad][:5])
print('--- reversed order of the trip times')
solver.sweepLanes = 'auto'; solver._handle=None; solver._pool=None
Tr = T[::-1].copy()
res = solver.solve_batch(Tr)
st=np.asarray(res['status']); feas = Tr>=tmin
bad=np.flatnonzero(feas & ~((st==0)|(st==6)))
print('hist',{int(k):int((st[feas]==k).sum()) for k in np.unique(st[feas])}, 'bad', len(bad), 'indices', bad[:12], 'T/Tmin', np.round(Tr[bad][:12]/tmin,4))
print('--- only the band, 256 instances')
Tb = tmin*np.linspace(1.07, 1.10, 256)
res = solver.solve_batch(Tb, screen=False)
st=np.asarray(res['status']); bad=np.flatnonzero(~((st==0)|(st==6)))
print('hist',{int(k):int((st==k).sum()) for k in np.unique(st)}, 'bad', len(bad), np.round(Tb[bad][:12]/tmin,4), 'iters', np.asarray(res['iters'])[bad][:12])
