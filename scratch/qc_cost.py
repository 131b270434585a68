"""Cost of outlier quality control at BASELINE config 3 (f64, 100 members, 721x1440x3, 1e5 obs): profiles/r05_qc.md.

    python scratch/qc_cost.py [--parent DIR] [--runs 4] [--steps 10] [--out qc_cost.json]

1. With --parent (a built checkout of the parent commit): `bench.py --gpus 1 --no-cpu-baseline --no-e2e --no-api`
   in this tree and in the parent's, alternated run by run; ms_per_step and the obs-solve phase of each run.
2. engine.analysis_device on config 3 with 1 % of the obs moved by 8 to 15 sigma, QC off (outlier_threshold None)
   and on (threshold 3 for every ob), alternated step by step; the state is reset from a device copy of the prior
   before every step, outside the timed window.  Step time (host wall time to a device synchronise), obs-solve time
   (res.ms['obs_solve']), and the number of rejected obs.
The card's name and power limit are read in the same run.
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)


def card():
    import torch
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'torch_name': torch.cuda.get_device_name(0), 'nvidia_smi': q.stdout.strip().splitlines()[:1]}


def stats(v):
    v = np.asarray(v)
    return {'median': float(np.median(v)), 'min': float(v.min()), 'max': float(v.max()), 'n': int(v.size)}


def bench_run(tree):
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--no-cpu-baseline', '--no-e2e', '--no-api']
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('{')]
    if r.returncode != 0 or not lines:
        raise RuntimeError('bench.py failed in %s: %s' % (tree, r.stderr[-2000:]))
    line = json.loads(lines[-1])
    return line['ms_per_step'], line['phases_ms'].get('obs_solve')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--parent', default=None)
    ap.add_argument('--runs', type=int, default=4)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default='qc_cost.json')
    args = ap.parse_args()
    import torch
    info = {'card': card(), 'config': 'config3', 'dtype': 'f64'}
    print(json.dumps(info['card']), flush=True)

    # 1. no QC: this tree against the parent, bench.py runs alternated
    if args.parent:
        runs = {'this': [], 'parent': []}
        for i in range(args.runs):
            for name, tree in (('this', HERE), ('parent', args.parent)):
                runs[name].append(bench_run(tree))
                print('bench %-6s run %d: %.2f ms/step, obs solve %.2f ms' % ((name, i) + runs[name][-1]), flush=True)
        info['bench_no_qc'] = {k: {'ms_per_step': stats([a for a, _ in v]), 'obs_solve_ms': stats([b for _, b in v]),
                                   'runs': v} for k, v in runs.items()}

    # 2. QC off / on on the same inputs
    from efa_xray_b200 import engine
    from efa_xray_b200.synth import CONFIGS, make_case
    dev = torch.device('cuda', 0)
    case = make_case(cutoff_km=2000.0, seed=0, **dict(CONFIGS['config3']))
    rng = np.random.default_rng(5)
    k = rng.choice(case.nobs, case.nobs // 100, replace=False)
    value = case.ob_value.copy()
    value[k] += rng.choice([-1.0, 1.0], k.size) * rng.uniform(8.0, 15.0, k.size) * np.sqrt(case.ob_error[k])
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    nlev = nt * len(case.varnames)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    obs = engine.ObsArrays(value=value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                           halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                           row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                           tw0=wlo, tw1=whi)
    variants = {'qc_off': obs, 'qc_on_t3': dataclasses.replace(obs, threshold=np.full(case.nobs, 3.0))}
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    prior = torch.as_tensor(case.to_vect()).to(dev)
    del case
    X = torch.empty_like(prior)
    steps = {k: [] for k in variants}
    solve = {k: [] for k in variants}
    nrej = {}
    for _ in range(2):
        for name, o in variants.items():
            X.copy_(prior)
            engine.analysis_device(X, nlev, grid, o, engine.LOC_GC)
    for s in range(args.steps):
        for name, o in variants.items():
            X.copy_(prior)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = engine.analysis_device(X, nlev, grid, o, engine.LOC_GC)
            torch.cuda.synchronize()
            steps[name].append(1e3 * (time.perf_counter() - t0))
            solve[name].append(res.ms['obs_solve'])
            nrej[name] = int((o.assimilate.astype(bool) & ~res.assimilated).sum())
    info['qc'] = {name: {'step_ms': stats(steps[name]), 'obs_solve_ms': stats(solve[name]), 'rejected': nrej[name],
                         'gross_errors_added': int(k.size)} for name in variants}
    for name in variants:
        q = info['qc'][name]
        print('%-9s step median %.2f ms [%.2f, %.2f]  obs solve median %.2f ms [%.2f, %.2f]  rejected %d' % (
            name, q['step_ms']['median'], q['step_ms']['min'], q['step_ms']['max'], q['obs_solve_ms']['median'],
            q['obs_solve_ms']['min'], q['obs_solve_ms']['max'], q['rejected']), flush=True)
    os.makedirs(os.path.dirname(args.out) or '.', exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(info, f, indent=1)


if __name__ == '__main__':
    main()
