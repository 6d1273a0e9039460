import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'ms-eetc_b200')]
import numpy as np
import __graft_entry__ as ge
ge.build()
from common import config5_instances
from mseetc.ocp import casadiSolver, solve_instances
from mseetc.train import Train
from mseetc.efficiency import totalLossesFunction
train = Train(config={'id': 'NL_Intercity_VIRM6'}); train.forceMinPn = 0
train.powerLosses = totalLossesFunction(train, auxiliaries=27000, etaGear=0.96)
inst = config5_instances(256)
mk = lambda N, track, energy: casadiSolver(train, track, {'numIntervals': N, 'maxIterations': 500, 'integrationMethod': 'RK', 'energyOptimal': energy, 'integrationOptions': {'order': 4, 'numSteps': 1, 'numApproxSteps': 1}})
solvers = [mk(N, tr, True) for N, tr in inst]; tsolvers = [mk(N, tr, False) for N, tr in inst]
lim = [np.minimum(s.points['Speed limit [m/s]'].values[:-1], s._base['velocityMax']) for s in solvers]
horizon = 1.5 * np.array([float(np.sum(s.steps / l)) for s, l in zip(solvers, lim)])
tres = solve_instances(tsolvers, horizon, screen=False)
print('time-optimal: failed', np.flatnonzero(tres['status'] != 0).tolist(), tres['status'][tres['status'] != 0].tolist(), 'restarted', tres.get('restarted'))
nint = np.array([s.numIntervals for s in solvers])
tmin = tres['z'][np.arange(len(inst)), nint * 4]
feasible = tres['status'] == 0
where = np.flatnonzero(feasible)
for stall in (80, 0):
    for s in solvers: s.stallIterations = stall
    res = solve_instances([s for s, f in zip(solvers, feasible) if f], 1.15 * tmin[feasible], screen=False)
    bad = np.flatnonzero((res['status'] != 0))
    print('stall', stall, 'energy: failed', where[bad].tolist(), res['status'][bad].tolist(), 'iters', res['iters'][bad].tolist(), 'kkt', res['kkt'][bad].tolist(), 'restarted', res.get('restarted'))
