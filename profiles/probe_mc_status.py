import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ms-eetc_b200')]
import numpy as np
import __graft_entry__ as ge
ge.build()
import bench
from mseetc.ocp import casadiSolver
from mseetc.train import Train
from mseetc.track import Track
from mseetc.efficiency import totalLossesFunction
train = Train(config={'id': 'NL_Intercity_VIRM6'})
track = Track(config={'id': '00_var_speed_limit_100'})
ov, ov2 = bench.mc_recipe(train)
dtrain = Train(config={'id': 'NL_Intercity_VIRM6'}); dtrain.forceMinPn = 0
dtrain.powerLosses = totalLossesFunction(dtrain, auxiliaries=27000, etaGear=0.96)
for name, tr, o in (('static', train, ov), ('dynamic', dtrain, ov2)):
    out = {}
    for comp in (True, False):
        s = casadiSolver(tr, track, bench.OPTS)
        s._ensure_handle().set_compaction(comp)
        res = s.solve_batch(1541.0, overrides=o, screen=np.zeros(32768, dtype=bool))
        out[comp] = {k: np.array(v) for k, v in res.items() if isinstance(v, np.ndarray)}
        st = res['status']
        print(name, 'compaction', comp, s._ensure_handle().last_compactions(), {int(k): int((st == k).sum()) for k in np.unique(st)}, 'kkt of non-0:', res['kkt'][st != 0][:8], 'iters', res['iters'][st != 0][:8], 'restarted', res.get('restarted'))
    print(name, 'bitwise equal:', all(np.array_equal(out[True][k], out[False][k]) for k in ('z', 'obj', 'kkt', 'iters', 'status')))
