import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ms-eetc_b200'), os.path.join(ROOT, 'profiles')]
import numpy as np
import __graft_entry__ as ge
ge.build()
from mseetc.ocp import casadiSolver
from mseetc.train import Train
from mseetc.track import Track
import bench
n = int(sys.argv[1]); streams = int(sys.argv[2]); screen = bool(int(sys.argv[3]))
rng = np.random.default_rng(20260101)
train = Train(config={'id': 'NL_Intercity_VIRM6'})
solver = casadiSolver(train, Track(config={'id': '00_var_speed_limit_100'}), bench.OPTS)
solver.streams = streams
ov = dict(mass=391000 * rng.uniform(0.85, 1.15, n), r0=train.r0 * rng.uniform(0.8, 1.2, n), etaTraction=rng.uniform(0.80, 0.92, n))
try:
    res = solver.solve_batch(1541.0, overrides=ov, screen=screen)
    print('n', n, 'streams', streams, 'screen', screen, 'ok', int((res['status'] == 0).sum()))
except Exception as e:
    print('n', n, 'streams', streams, 'screen', screen, 'ERR', str(e)[:80])
