#!/usr/bin/env python
"""Benchmark of the hot path: batched OCP solves per second (BASELINE.json metric).

Default workload (BASELINE.json configs[1]): trip-time sweep, 4096 VIRM6 instances PER GPU on tracks/CH_StGallen_Wil.json,
numIntervals 300 (simulations/config.json), terminal times T_k = Tmin*(0.8 + 0.4 k/(n-1)), k = 0..n-1, n = 4096 * gpus.
It is ONE batch: under torchrun its 32-instance tiles are dealt to the ranks (mseetc.sharding.shard_tiles -- a sorted sweep
has all its infeasible instances at one end), every rank solves its share with no collective on the solve path, and the
end-to-end leg gathers the results on rank 0 (mseetc.sharding.solve_batch_sharded).  Instances below the minimum trip
time are infeasible; they are screened / flagged (SURVEY.md 8d) and NOT counted: `value` and `e2e` count the feasible
instances that converged.  The minimum time itself is computed inside every timed step by a time-optimal solve.

  --workload mc65536   BASELINE configs[2]: 65 536-instance parameter Monte Carlo (SURVEY.md 8d recipe, rng 20260101, half
                       constant efficiencies / half spline loss map), ONE batch split contiguously over the ranks
                       (mseetc.sharding.shard_ranges): strong scaling.

One "step" = one pass of the hot path over the whole batch.  `value` is measured with the inputs already in HBM (CUDA events
on the launch stream, profiling off); `roofline` comes from a separate profiled pass; `e2e` goes through the public API with
host arrays, host->device and device->host copies (and the gather) inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload sweep|mc65536] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step computed (z, obj, kkt, iters, status and, for the sweep, the minimum trip
time of every instance) as DIR/<name>.npy in float64, rows in the batch's instance order, `instance` naming each row's index in
the batch (under torchrun every rank writes its share, prefixed rank<r>_).  Rows of instances flagged infeasible (status 4) are
zero but for their status.  The inputs are fixed by the arguments, so two builds can be compared output for output.  The files
stay under 64 MB; a larger batch (mc65536) is represented by a fixed, seeded sample of its instances.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'ms-eetc_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

N_INST = 4096
N_INT = 300
OPTS = {'numIntervals': N_INT, 'maxIterations': 500, 'integrationMethod': 'RK',
        'integrationOptions': {'order': 4, 'numSteps': 1, 'numApproxSteps': 1}}
TMIN_REF = 1035.5536      # restatement-derived (SURVEY appendix E); re-derived on the device in every step
METRIC = 'OCP solves/sec (batched, 1/2/4/8 B200) vs CasADi+IPOPT on host cores'
DUMP_BYTES = (64 << 20) - (1 << 20)      # --dump-outputs stays under 64 MB with room for the .npy headers


def sweep_times(n, tmin=TMIN_REF):
    return tmin * (0.8 + 0.4 * np.arange(n) / (n - 1))


def bench_config(workload, world, per_gpu):
    "The `config` object of the JSON line: identical for the product arm and the reference arm."
    if workload == 'mc65536':
        return {'workload': 'parameter Monte Carlo (BASELINE configs[2]): 65536 VIRM6-class instances on 00_var_speed_limit_100, '
                            'numIntervals 300, T = 1541 s, rng 20260101 (mass, Davis coefficients, efficiencies / loss-map scale, '
                            'auxiliaries), half constant efficiencies, half spline loss map; one batch split contiguously over the GPUs',
                'instances': 65536, 'numIntervals': N_INT, 'counted': 'instances that converged',
                'l2': 'per-tick working set of a rank >> 126 MB L2'}
    return {'workload': 'trip-time sweep (BASELINE configs[1]): %d VIRM6 instances per GPU on CH_StGallen_Wil, numIntervals %d, '
                        'T_k = Tmin*(0.8 + 0.4 k/(n-1)); one batch, tiles dealt to the GPUs' % (per_gpu, N_INT),
            'instances': per_gpu * world, 'numIntervals': N_INT,
            'counted': 'feasible instances (T_k >= Tmin, the upper half of the sweep) that converged; the infeasible half is '
                       'screened / flagged and not counted; the CPU arm times a bounded sample of the feasible half',
            'l2': 'per-tick working set of a rank (1.7 GB) >> 126 MB L2'}


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (numpy/scipy restatement of the reference NLP + IPOPT-style solver) in a process pool
# ----------------------------------------------------------------------------------------------------------
_ORACLE = {}


def _oracle_sweep(T):
    if 'nlp' not in _ORACLE:
        from oracle.problem import load_train, load_track, discretization_points
        from oracle.nlp import ReferenceNLP
        train = load_train(os.path.join(PKG, 'trains', 'NL_Intercity_VIRM6.json'))
        track = load_track(os.path.join(PKG, 'tracks', 'CH_StGallen_Wil.json'))
        pos, g, v, c = discretization_points(track, N_INT)
        _ORACLE['nlp'] = ReferenceNLP(train, pos, g, v, c, track.length,
                                      dict(numSteps=1, numApproxSteps=1, energyOptimal=True, minimumVelocity=1))
    from oracle import ipm
    nlp = _ORACLE['nlp']
    lbz, ubz, lbg, ubg = nlp.bounds(float(T))
    r = ipm.solve(nlp, nlp.x0(float(T)), lbz, ubz, lbg, ubg, max_iter=500)
    return r.success, r.iters


def _oracle_mc(args):
    "One constant-efficiency Monte-Carlo instance of configs[2] (the spline-map half takes 24 s per solve in the torch oracle)."
    mass, f0, f1, f2, etaT, etaR = args
    from oracle.problem import load_train, load_track, discretization_points
    from oracle.nlp import ReferenceNLP
    from oracle import ipm
    train = load_train(os.path.join(PKG, 'trains', 'NL_Intercity_VIRM6.json'))
    train.mass = mass
    train.r0, train.r1, train.r2 = train.r0 * f0, train.r1 * f1, train.r2 * f2
    train.losses = ('static', etaT, etaR)
    if 'mc_grid' not in _ORACLE:
        track = load_track(os.path.join(PKG, 'tracks', '00_var_speed_limit_100.json'))
        _ORACLE['mc_grid'] = (discretization_points(track, N_INT), track.length)
    (pos, g, v, c), length = _ORACLE['mc_grid']
    nlp = ReferenceNLP(train, pos, g, v, c, length, dict(numSteps=1, numApproxSteps=1, energyOptimal=True, minimumVelocity=1))
    lbz, ubz, lbg, ubg = nlp.bounds(1541.0)
    r = ipm.solve(nlp, nlp.x0(1541.0), lbz, ubz, lbg, ubg, max_iter=500)
    return r.success, r.iters


def cpu_sample(workload, n_samples):
    if workload == 'mc65536':
        rng = np.random.default_rng(20260101)
        cols = [391000 * rng.uniform(0.85, 1.15, 32768)] + [rng.uniform(0.8, 1.2, 32768) for _ in range(3)] + \
               [rng.uniform(0.80, 0.92, 32768), rng.uniform(0.55, 0.85, 32768)]
        pick = np.linspace(0, 32767, n_samples).astype(int)
        return _oracle_mc, [tuple(float(c[i]) for c in cols) for i in pick], \
            '%d instances of the constant-efficiency half of the batch (evenly spaced indices)' % n_samples
    Ts = TMIN_REF * np.linspace(1.001, 1.2, n_samples)
    return _oracle_sweep, list(Ts), '%d feasible instances of the sweep (T evenly spaced in Tmin*[1.001, 1.2])' % n_samples


def cpu_pool_rate(workload, n_samples, workers, steps=1, warm=True):
    "Solves/s of the oracle on `workers` processes over a bounded sample of the workload."
    import multiprocessing as mp
    fn, items, what = cpu_sample(workload, n_samples)
    ctx = mp.get_context('spawn')
    with ctx.Pool(workers) as pool:
        if warm:
            pool.map(fn, items[:workers])               # imports + sympy code generation in every worker
        t0 = time.perf_counter()
        for _ in range(steps):
            res = pool.map(fn, items, chunksize=1)
        dt = time.perf_counter() - t0
    ok = sum(1 for s, _ in res if s)
    return ok * steps / dt, ok, dt, what


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 32))
    n_samples = 2 * workers
    value, ok, dt, what = cpu_pool_rate(args.workload, n_samples, workers, steps=args.steps, warm=args.warmup > 0)
    sample = '%s per step on %d worker processes, %d converged' % (what, workers, ok)
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'solves/s', 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True,
            'scaling': 'strong' if args.workload == 'mc65536' else 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': bench_config(args.workload, args.gpus, args.instances),
            'cpu_baseline': {'value': value, 'unit': 'solves/s', 'cores': workers, 'kind': 'port', 'sample': sample,
                             'note': 'oracle port (numpy/scipy restatement of the reference NLP + IPOPT-style filter IP), '
                                     'NOT CasADi+IPOPT: casadi is not installable in this image'},
            'e2e': {'value': value, 'unit': 'solves/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'converged': ok, 'instances_per_step': n_samples}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.QUERY, '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                    if val.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        busy = [x for x in sm if x > 0.5 * max(sm)] if sm else []
        return {'sm_mhz': float(np.median(busy)) if busy else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


class Resident:
    """One rank's share of a batch with its inputs resident in HBM: parameter planes in dealt (stream-pool) order, track
    tables, result buffers; `step()` runs the hot path once (optionally with the concurrent minimum-time presolve)."""

    def __init__(self, solver, dev, streams, lanes, T, overrides=None, lossT=0.0, lossR=0.0, presolve=False, name=''):
        import torch
        from mseetc import _cabi
        self.torch, self.cabi, self.solver, self.dev, self.name = torch, _cabi, solver, dev, name
        n = self.n = len(T)
        zero = np.zeros(n)
        overrides = dict(overrides or {})
        P, self.M = solver._planes(n, T, zero, zero + 1.0, zero + 1.0, overrides, lossT, lossR)
        ds, c0, bmax = solver._tables(solver._base['rho'], solver._base['g'], solver._base['velocityMax'])
        self.perm, self.parts = _cabi.StreamPool.interleave(n, streams) if streams > 1 and n >= 1024 else (np.arange(n), None)
        self.back = np.argsort(self.perm)
        P = np.ascontiguousarray(P[:, self.perm])
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(device=dev, dtype=dt)
        N = solver.numIntervals
        self.d = dict(P=up(P, torch.float64), nint=up(np.full(n, N, np.int32), torch.int32), trk_of=up(np.zeros(n, np.int32), torch.int32),
                      trk_off=up(np.array([0, N], np.int32), torch.int32), ds=up(ds, torch.float64), c0=up(c0, torch.float64),
                      bmax=up(bmax, torch.float64))
        solver.streams = streams
        solver.sweepLanes = lanes
        self.pool = _cabi.StreamPool(solver._make_handle, max(1, streams if self.parts is not None else 1), dev)
        self.handles = list(self.pool.handles)
        h = self.pool.handles[0]
        stp = 3 + h.nu
        self.out = dict(z=torch.zeros((n, N * stp + 2), dtype=torch.float64, device=dev), lam=None,
                        obj=torch.empty(n, dtype=torch.float64, device=dev), kkt=torch.empty(n, dtype=torch.float64, device=dev),
                        iters=torch.empty(n, dtype=torch.int32, device=dev), status=torch.empty(n, dtype=torch.int32, device=dev))
        self.ht = None
        if presolve:
            tsolver = solver._time_sibling()
            tsolver.sweepLanes = lanes
            lim = np.minimum(solver.points['Speed limit [m/s]'].values[:-1], solver._base['velocityMax'])
            horizon = 1.5 * float(np.sum(solver.steps / lim))      # same bound as casadiSolver.minimum_time
            Pt, _ = tsolver._planes(1, np.array([horizon]), np.zeros(1), np.ones(1), np.ones(1), {}, 0.0, 0.0)
            self.d.update(Pt=up(Pt, torch.float64), nint1=up(np.full(1, N, np.int32), torch.int32), trk_of1=up(np.zeros(1, np.int32), torch.int32))
            self.ht = tsolver._ensure_handle()
            self.handles.append(self.ht)
            self.tmin_dev = torch.zeros(n, dtype=torch.float64, device=dev)
            self.side = torch.cuda.Stream(device=dev, priority=-5)
        self.launches = 0
        self.tr = None

    def set_profiling(self, on):
        for hh in self.handles:
            self.cabi.set_profiling(hh, on)

    def step(self):
        torch, d, dev = self.torch, self.d, self.dev
        if self.ht is None:
            out = self.pool.solve(d['P'], d['nint'], d['trk_of'], d['trk_off'], d['ds'], d['c0'], d['bmax'], out=dict(self.out), parts=self.parts)
            self.launches += out['launches']
            return out
        # (1) minimum trip time of the (single) distinct problem of this sweep: time-optimal solve on a side stream, driven by
        #     a second host thread, concurrently with (2); its result lands in tmin_dev while the batch is iterating
        self.tmin_dev.zero_()
        box = {}

        def presolve():
            torch.cuda.set_device(dev)
            self.side.wait_stream(torch.cuda.default_stream(dev))
            with torch.cuda.stream(self.side):
                tr = self.ht.solve_device(d['Pt'], d['nint1'], d['trk_of1'], d['trk_off'], d['ds'], d['c0'], d['bmax'])
                self.tmin_dev.copy_(tr['z'][:, -2].expand(self.n))          # t_N - t_0 with t_0 = 0
                self.side.synchronize()
            box['tr'] = tr

        th = threading.Thread(target=presolve)
        th.start()
        # (2) the sweep; instances below the minimum time are flagged infeasible by the library as soon as it is known
        out = self.pool.solve(d['P'], d['nint'], d['trk_of'], d['trk_off'], d['ds'], d['c0'], d['bmax'], tmin=self.tmin_dev,
                              out=dict(self.out), parts=self.parts)
        th.join()
        self.tr = box['tr']
        self.launches += self.tr['launches'] + out['launches']
        return out

    def profile(self, acc, acc_pre):
        for hh in self.handles:
            tgt = acc_pre if hh is self.ht else acc
            for k, v in self.cabi.last_profile(hh).items():
                t = tgt.setdefault(k, dict(ms=0.0, launches=0, cells=0, bytes_per_cell=0.0))
                t['ms'] += v['ms']; t['launches'] += v['launches']; t['cells'] += v['cells']; t['bytes_per_cell'] = v['bytes_per_cell']


def dump_outputs(dirname, parts, budget, seed=20260101):
    """Writes DIR/<prefix><key>.npy (float64) for parts [(prefix, instance indices, {key: array with one row per instance})].
    If they exceed `budget` bytes, every part keeps the same fixed, seeded fraction of its rows; <prefix>instance.npy holds the
    batch index of every row written."""
    parts = [(p, np.asarray(idx, dtype=np.float64), {k: np.asarray(a, dtype=np.float64) for k, a in arrs.items()}) for p, idx, arrs in parts]
    total = sum(idx.nbytes + sum(a.nbytes for a in arrs.values()) for _, idx, arrs in parts)
    frac = min(1.0, budget / total)
    rng = np.random.default_rng(seed)
    os.makedirs(dirname, exist_ok=True)
    for prefix, idx, arrs in parts:
        n = len(idx)
        rows = np.arange(n) if frac == 1.0 else np.sort(rng.choice(n, max(1, int(n * frac)), replace=False))
        for k, a in dict(arrs, instance=idx).items():
            np.save(os.path.join(dirname, prefix + k + '.npy'), a[rows])


def mc_recipe(train):
    "SURVEY.md 8(d) config 3: per-instance train parameters, first half constant efficiencies, second half spline loss map."
    rng = np.random.default_rng(20260101)
    half = 32768
    ov = dict(mass=391000 * rng.uniform(0.85, 1.15, half), r0=train.r0 * rng.uniform(0.8, 1.2, half), r1=train.r1 * rng.uniform(0.8, 1.2, half),
              r2=train.r2 * rng.uniform(0.8, 1.2, half), etaTraction=rng.uniform(0.80, 0.92, half), etaRgBrake=rng.uniform(0.55, 0.85, half))
    ov2 = dict(mass=391000 * rng.uniform(0.85, 1.15, half), r0=train.r0 * rng.uniform(0.8, 1.2, half), r1=train.r1 * rng.uniform(0.8, 1.2, half),
               r2=train.r2 * rng.uniform(0.8, 1.2, half), auxiliaries=rng.uniform(20e3, 35e3, half), tableScale=rng.uniform(0.9, 1.1, half))
    return ov, ov2


def run_gpu(args):
    import torch
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device (there is no CPU fallback for the product arm)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if dist is not None:
        dist.barrier()
    ge.build()
    from mseetc.ocp import casadiSolver
    from mseetc.train import Train
    from mseetc.track import Track
    from mseetc.efficiency import totalLossesFunction
    from mseetc import _cabi, sharding

    lanes = args.sweep_lanes if args.sweep_lanes == 'auto' else int(args.sweep_lanes)
    mc = args.workload == 'mc65536'
    residents = []          # (Resident, instance indices of the whole batch it holds, api closure)
    if not mc:
        n_total = args.instances * world
        T = sweep_times(n_total)
        idx = sharding.shard_tiles(n_total, world)[rank]
        train = Train(config={'id': 'NL_Intercity_VIRM6'})
        solver = casadiSolver(train, Track(config={'id': 'CH_StGallen_Wil'}), OPTS)
        residents.append((Resident(solver, dev, args.streams, lanes, T[idx], lossT=(1 - train.etaTraction) / train.etaTraction,
                                   lossR=1 - train.etaRgBrake, presolve=True), idx))
        partition = 'tiles'
    else:
        n_total = 65536
        T = np.full(n_total, 1541.0)
        a, b = sharding.shard_ranges(np.full(n_total, N_INT), world)[rank]
        idx = np.arange(a, b)
        train = Train(config={'id': 'NL_Intercity_VIRM6'})
        track = Track(config={'id': '00_var_speed_limit_100'})
        ssolver = casadiSolver(train, track, OPTS)
        dtrain = Train(config={'id': 'NL_Intercity_VIRM6'})
        dtrain.forceMinPn = 0
        dtrain.powerLosses = totalLossesFunction(dtrain, auxiliaries=27000, etaGear=0.96)
        dsolver = casadiSolver(dtrain, track, dict(OPTS, minimumVelocity=1))
        ov, ov2 = mc_recipe(train)
        sel = idx[idx < 32768]
        if len(sel):
            o = {k: v[sel] for k, v in ov.items()}
            etaT, etaR = o.pop('etaTraction'), o.pop('etaRgBrake')
            residents.append((Resident(ssolver, dev, args.streams, lanes, T[sel], overrides=o, lossT=(1 - etaT) / etaT, lossR=1 - etaR,
                                       name='constant_'), sel))
        sel = idx[idx >= 32768]
        if len(sel):
            residents.append((Resident(dsolver, dev, args.streams, lanes, T[sel], overrides={k: v[sel - 32768] for k, v in ov2.items()},
                                       name='lossmap_'), sel))
        partition = 'ranges'

    def step():
        return [r.step() for r, _ in residents]

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, last

    # ---------------- headline: inputs resident in HBM, per-kernel profiling OFF
    for r, _ in residents:
        r.set_profiling(False)
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for r, _ in residents:
        r.launches = 0
    ms, outs = timed(step, args.steps)
    launches = sum(r.launches for r, _ in residents)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # the result buffers are reused by every later pass: copy out what the last timed step left in them
        parts = []
        for (r, sel), out in zip(residents, outs):
            arrs = {k: out[k].cpu().numpy()[r.back] for k in ('z', 'obj', 'kkt', 'iters', 'status')}
            # an instance flagged infeasible stops at whichever iteration the concurrent minimum-time presolve reaches it, which
            # varies from run to run: its rows are blanked (the public API blanks the trajectory of a failed solve as well)
            flagged = arrs['status'] == 4
            for k in ('z', 'obj', 'kkt', 'iters'):
                arrs[k][flagged] = 0
            if r.ht is not None:
                arrs['tmin'] = r.tmin_dev.cpu().numpy()[r.back]
            parts.append(('%s%s' % ('rank%d_' % rank if world > 1 else '', r.name), sel, arrs))
        dump_outputs(args.dump_outputs, parts, DUMP_BYTES // world)

    # what was solved (this rank), then summed over the ranks
    stats = dict(instances=0, feasible=0, converged=0, flagged=0, failed=0, iters_sum=0.0, iters_max=0, ticks=0)
    tmin_s = None
    for (r, sel), out in zip(residents, outs):
        status = out['status'].cpu().numpy()[r.back]
        iters = out['iters'].cpu().numpy()[r.back]
        kkt = out['kkt'].cpu().numpy()[r.back]
        if r.tr is not None:
            tmin_s = float(r.tr['z'][0, -2].item())
            feas = T[sel] >= tmin_s
        else:
            feas = np.ones(len(sel), dtype=bool)
        ok = (status == 0) & feas & (kkt <= 1e-8)
        stats['instances'] += len(sel); stats['feasible'] += int(feas.sum()); stats['converged'] += int(ok.sum())
        stats['flagged'] += int(((status != 0) & ~feas).sum()); stats['failed'] += int((feas & ~ok).sum())
        stats['iters_sum'] += float(iters[ok].sum()); stats['iters_max'] = max(stats['iters_max'], int(iters[ok].max()) if ok.any() else 0)
        stats['ticks'] = max(stats['ticks'], int(out['ticks']))
    per_rank = [stats['instances']]
    if dist is not None:
        t = torch.tensor([stats[k] for k in ('instances', 'feasible', 'converged', 'flagged', 'failed', 'iters_sum')], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        for k, v in zip(('instances', 'feasible', 'converged', 'flagged', 'failed', 'iters_sum'), t.tolist()):
            stats[k] = v if k == 'iters_sum' else int(round(v))
        t = torch.tensor([stats['iters_max'], stats['ticks']], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stats['iters_max'], stats['ticks'] = int(t[0].item()), int(t[1].item())
        g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([float(per_rank[0])], dtype=torch.float64, device=dev))
        per_rank = [int(x.item()) for x in g]

    # ---------------- roofline: a separate pass with per-kernel CUDA events (profiling ON), not part of the headline
    prof, prof_pre = {}, {}
    for r, _ in residents:
        r.set_profiling(True)
    step()
    prof_steps = max(2, min(args.steps, 5))
    for _ in range(prof_steps):
        step()
        for r, _ in residents:
            r.profile(prof, prof_pre)
    for r, _ in residents:
        r.set_profiling(False)

    # ---------------- e2e: public API, host arrays in, host arrays out (gathered on rank 0)
    if not mc:
        api = lambda: sharding.solve_batch_sharded(residents[0][0].solver, T, partition='tiles')
    else:
        full_ov = {k: np.concatenate([ov[k], ov2[k]]) for k in ('mass', 'r0', 'r1', 'r2')}

        def api():
            # two calls: the two halves differ in problem structure (loss family, pneumatic brake).  T = 1541 s is the
            # timetable value of this track with 5 % slack for the nominal train; the mask asserts feasibility per instance
            outs = []
            for solver_, lo, extra in ((ssolver, 0, {k: ov[k] for k in ('etaTraction', 'etaRgBrake')}),
                                       (dsolver, 32768, {k: ov2[k] for k in ('auxiliaries', 'tableScale')})):
                o = {k: v[lo:lo + 32768] for k, v in full_ov.items()}
                o.update(extra)
                outs.append(sharding.solve_batch_sharded(solver_, 1541.0, overrides=o, partition='ranges', screen=np.zeros(32768, dtype=bool)))
            return outs
    for _ in range(min(args.warmup, 3)):
        res = api()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = []
    for _ in range(args.steps):
        ts = time.perf_counter()
        res = api()
        e2e_steps.append(round(1e3 * (time.perf_counter() - ts), 2))
    barrier()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    h2d_local = 0
    for (r, _) in residents:
        h2d_local += int(r.d['P'].numel() * 8 + r.n * 8 + (r.n * 8 if r.ht is not None else 0) + (r.d['ds'].numel() + r.d['c0'].numel() + r.d['bmax'].numel()) * 8)
    if dist is not None:
        t = torch.tensor([float(h2d_local)], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        h2d_total = int(t.item())
    else:
        h2d_total = h2d_local
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    res_list = res if isinstance(res, list) else [res]
    e2e_ok = 0
    d2h = 0
    for rr in res_list:
        st = rr['status']
        if not mc:
            tm = TMIN_REF if tmin_s is None else tmin_s
            e2e_ok += int(((st == 0) & (T >= tm) & (rr['kkt'] <= 1e-8)).sum())
        else:
            e2e_ok += int(((st == 0) & (rr['kkt'] <= 1e-8)).sum())
        d2h += int(sum(v.nbytes for v in rr.values() if isinstance(v, np.ndarray)))

    # ---------------- roofline of the dominant kernel (largest share of the device time of the profiled pass)
    peaks_file = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_file):
        peak, peak_src = float(json.load(open(peaks_file))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    kern = {}
    for k, v in prof.items():
        if v['launches'] == 0 or k == 'misc':
            continue
        gbs = v['cells'] * v['bytes_per_cell'] / (v['ms'] * 1e-3) / 1e9 if v['ms'] > 0 else 0.0
        kern[k] = {'ms_total': v['ms'], 'launches': v['launches'], 'avg_us': 1e3 * v['ms'] / v['launches'],
                   'bytes_per_cell': v['bytes_per_cell'], 'cells': v['cells'], 'achieved_gbs': gbs, 'frac_hbm': gbs / peak}
    if not kern:
        kern = {'inst_step': dict(ms_total=1.0, launches=1, avg_us=0.0, bytes_per_cell=0.0, cells=0, achieved_gbs=0.0, frac_hbm=0.0)}
    top = max(kern, key=lambda k: kern[k]['ms_total'])
    ncu_traffic, capture = None, None
    tfile = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tfile):
        tj = json.load(open(tfile))
        ncu_traffic = tj.get(top)
        capture = (tj.get('captures') or {}).get(top)
    fp64 = None
    ofile = os.path.join(ROOT, 'profiles', 'fp64_ops.json')
    if os.path.exists(ofile):
        ops = json.load(open(ofile))
        peak64 = _cabi.measure_fp64_peak()
        fp64 = {'peak_gflops': peak64, 'peak_source': 'measured here (k_fp64_peak: independent DFMA chains, CUDA events)', 'kernels': {}}
        for k, v in kern.items():
            if k in ops and v['ms_total'] > 0:
                gf = v['cells'] * ops[k]['flop_per_cell'] / (v['ms_total'] * 1e-3) / 1e9
                fp64['kernels'][k] = {'flop_per_cell': ops[k]['flop_per_cell'], 'achieved_gflops': gf, 'frac_fp64': gf / peak64}
    tick_bytes = sum(v['cells'] * v['bytes_per_cell'] for v in kern.values())
    tick_ms = sum(v['ms_total'] for v in kern.values())
    roofline = {'bound': 'hbm', 'kernel': top, 'achieved': kern[top]['achieved_gbs'], 'peak': peak, 'unit': 'GB/s',
                'frac': kern[top]['achieved_gbs'] / peak, 'traffic': ncu_traffic, 'traffic_capture': capture, 'peak_source': peak_src,
                'share_of_device_time': kern[top]['ms_total'] / max(1e-12, tick_ms),
                'bytes_per_launch': kern[top]['cells'] * kern[top]['bytes_per_cell'] / kern[top]['launches'],
                'pass': 'separate profiled pass of %d steps on rank 0 (per-kernel CUDA events on the launch streams); the headline is timed with profiling off' % prof_steps,
                'all_kernels': {'achieved': tick_bytes / max(1e-12, tick_ms * 1e-3) / 1e9, 'frac': tick_bytes / max(1e-12, tick_ms * 1e-3) / 1e9 / peak,
                                'note': 'algorithmic bytes of all solver kernels / sum of their durations'},
                'kernels': kern, 'fp64': fp64,
                'presolve': {'ms_total': sum(v['ms'] for v in prof_pre.values()), 'launches': sum(v['launches'] for v in prof_pre.values()),
                             'note': 'single-instance time-optimal solve on its own stream, concurrent with the sweep (not in `kernels`)'}}

    # ---------------- config-1 latency: one solve through solve(), reference protocol (min of 5, table3.py:33,53-64)
    latency = None
    if world == 1 and not args.no_latency:
        s1 = casadiSolver(Train(config={'id': 'NL_Intercity_VIRM6'}), Track(config={'id': '00_var_speed_limit_100'}), OPTS)
        import contextlib
        import io
        lat, its = [], set()
        with contextlib.redirect_stdout(io.StringIO()):
            for i in range(7):
                df, st = s1.solve(1541)
                if i >= 2:
                    lat.append(st['CPU time [s]']); its.add(st['IP iterations'])
        latency = {'config': 'BASELINE configs[0]: VIRM6 on 00_var_speed_limit_100, simulations/config.json, solve(1541)',
                   'single_solve_ms': 1e3 * min(lat), 'protocol': "min of 5 of stats['CPU time [s]'] after 2 warm-up solves; identical iteration counts",
                   'ip_iterations': sorted(its), 'cost_kwh': float(st['Cost']), 'sweep_lanes': s1._ensure_handle().sweep_lanes()}

    # ---------------- CPU baseline beside it (bounded sample, rank 0, N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        cores = max(1, min(os.cpu_count() or 1, 16))
        rate, ok, dt, what = cpu_pool_rate(args.workload, 3 * cores, cores)          # ~25 s of CPU work
        cpu = {'value': rate, 'unit': 'solves/s', 'cores': cores, 'kind': 'port',
               'sample': '%s on %d worker processes, %.1f s wall, %d converged' % (what, cores, dt, ok),
               'note': 'oracle port (numpy/scipy restatement + IPOPT-style filter IP), not CasADi+IPOPT'}

    counted = stats['converged']
    line = {'metric': METRIC, 'value': counted * args.steps / (ms * 1e-3), 'unit': 'solves/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong' if mc else 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': bench_config(args.workload, world, args.instances),
            'batch': {'instances': stats['instances'], 'instances_per_rank': per_rank, 'partition': 'mseetc.sharding.shard_' + partition,
                      'feasible': stats['feasible'], 'converged_feasible': stats['converged'], 'failed_feasible': stats['failed'],
                      'flagged_infeasible': stats['flagged'], 'tmin_s': tmin_s,
                      'ip_iterations_mean': stats['iters_sum'] / max(1, stats['converged']), 'ip_iterations_max': stats['iters_max'],
                      'ticks': stats['ticks'], 'streams': args.streams, 'sweep_lanes': residents[0][0].pool.handles[0].sweep_lanes()},
            'all_instances_per_s': stats['instances'] * args.steps / (ms * 1e-3),
            'e2e': {'value': e2e_ok * args.steps / e2e_s, 'unit': 'solves/s', 'h2d_bytes_per_step': h2d_total,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': 1e3 * e2e_s / args.steps, 'steps_ms': e2e_steps,
                    'all_instances_per_s': stats['instances'] * args.steps / e2e_s,
                    'path': 'mseetc.sharding.solve_batch_sharded -> casadiSolver.solve_batch per rank; results gathered on rank 0'
                            + (' (NCCL gather of device tensors, one device-to-host copy)' if world > 1 else ''),
                    'instances_per_rank': res_list[0].get('instances_per_rank'),
                    'last_call_breakdown_s': res_list[0].get('timing')},
            'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline}
    if latency is not None:
        line['latency'] = latency
    if cpu is not None:
        line['cpu_baseline'] = cpu
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='sweep', choices=['sweep', 'mc65536'])
    ap.add_argument('--instances', type=int, default=N_INST, help='instances per GPU of the sweep workload')
    ap.add_argument('--no-cpu', action='store_true', help='skip the CPU baseline leg')
    ap.add_argument('--no-latency', action='store_true', help='skip the config-1 single-solve latency leg')
    ap.add_argument('--streams', type=int, default=1, help='concurrent sub-batches (CUDA streams / host threads) per GPU')
    ap.add_argument('--sweep-lanes', default='auto', help="Riccati sweeps: 1 sequential, 8/16/32 parallel in time, 'auto'")
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the results of the last timed step as DIR/<name>.npy (float64, '
                                                          'at most 64 MB: a seeded sample of the instances of a larger batch)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the results of the GPU arm; the reference arm keeps none')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
