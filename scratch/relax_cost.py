"""Cost of posterior relaxation at BASELINE config 3 (f64, 100 members, 721x1440x3, 1e5 obs): profiles/r03_relax.md.

    python scratch/relax_cost.py [--steps 10] [--out relax_cost.json]

1. engine.analysis_device with relaxation None / rtps / rtpp, alternated step by step (the state is reset from a
   device copy of the prior before every step, outside the timed window); median and spread of each.
2. CUDA-event times of each relaxation pass on the full state (2.49 GB, far beyond the 126 MB L2), with achieved
   GB/s from the algorithmic bytes (S = state bytes): row spread reads S; the RTPS pass reads S and writes S; the
   RTPP prior copy reads S and writes S; the RTPP pass reads 2 S and writes S.  Against a device-to-device copy of
   the state (torch copy_, reads S and writes S) measured in the same run.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'torch_name': torch.cuda.get_device_name(0), 'nvidia_smi': q.stdout.strip().splitlines()[:1]}


def event_ms(fn, reps):
    import torch
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def stats(v):
    v = np.asarray(v)
    return {'median': float(np.median(v)), 'min': float(v.min()), 'max': float(v.max()),
            'p25': float(np.percentile(v, 25)), 'p75': float(np.percentile(v, 75)), 'n': int(v.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default='relax_cost.json')
    args = ap.parse_args()
    import torch
    from efa_xray_b200 import engine, _lib
    from efa_xray_b200.synth import CONFIGS, make_case
    dev = torch.device('cuda', 0)
    cfg = dict(CONFIGS['config3'])
    case = make_case(cutoff_km=2000.0, seed=0, **cfg)
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    nlev = nt * len(case.varnames)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    obs = engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                           halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                           row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                           tw0=wlo, tw1=whi)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    prior = torch.as_tensor(case.to_vect()).to(dev)
    del case
    X = torch.empty_like(prior)
    nrows, nens = prior.shape
    S = prior.numel() * prior.element_size()
    kinds = {'none': None, 'rtps': ('rtps', np.full(nlev, 0.9)), 'rtpp': ('rtpp', np.full(nlev, 0.5))}
    info = {'card': card(), 'config': 'config3', 'dtype': 'f64', 'state_bytes': S, 'nrows': nrows, 'nens': nens}
    print(json.dumps(info['card']))

    # 1. whole analysis, alternated
    steps = {k: [] for k in kinds}
    relax_ms = {k: [] for k in kinds}
    for warm in range(2):
        for k, r in kinds.items():
            X.copy_(prior)
            engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, relaxation=r)
    for s in range(args.steps):
        for k, r in kinds.items():
            X.copy_(prior)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, relaxation=r)
            torch.cuda.synchronize()
            steps[k].append(1e3 * (time.perf_counter() - t0))
            relax_ms[k].append(res.ms.get('relax', 0.0))
    info['step_ms'] = {k: stats(v) for k, v in steps.items()}
    info['relax_ms_in_step'] = {k: stats(v) for k, v in relax_ms.items() if k != 'none'}
    for k in kinds:
        print('step %-5s median %.2f ms [%.2f, %.2f]  relax %.3f ms' % (k, info['step_ms'][k]['median'],
              info['step_ms'][k]['min'], info['step_ms'][k]['max'], np.median(relax_ms[k])))

    # 2. each pass on the full state.  X is an analysis (the relaxed rows are written on every launch).
    X.copy_(prior)
    engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC)
    Xb = torch.empty_like(prior)
    sigma = torch.empty(nrows, dtype=torch.float64, device=dev)
    alpha = torch.full((nlev,), 0.5, dtype=torch.float64, device=dev)
    npts = nrows // nlev
    sp = _lib.stream_ptr()
    passes = {
        'copy_d2d (torch copy_)': (lambda: Xb.copy_(prior), 2 * S),
        'row_spread_kernel': (lambda: _lib.call('exb_row_spread_f64', _lib.ptr(prior), nlev, npts, 0, npts, nens,
                                                _lib.ptr(sigma), sp), S + 8 * nrows),
        'relax_rtps_kernel': (lambda: _lib.call('exb_relax_rtps_f64', _lib.ptr(X), _lib.ptr(sigma), _lib.ptr(alpha),
                                                nlev, npts, 0, npts, nens, sp), 2 * S + 8 * nrows),
        'rtpp prior copy (torch copy_)': (lambda: Xb.copy_(prior), 2 * S),
        'relax_rtpp_kernel': (lambda: _lib.call('exb_relax_rtpp_f64', _lib.ptr(X), _lib.ptr(Xb), _lib.ptr(alpha),
                                                nlev, npts, 0, npts, nens, sp), 3 * S),
    }
    info['passes'] = {}
    for name, (fn, nbytes) in passes.items():
        for _ in range(3):
            fn()
        t = event_ms(fn, args.reps)
        st = stats(t)
        st['bytes'] = nbytes
        st['GBps_at_median'] = nbytes / (st['median'] * 1e-3) / 1e9
        info['passes'][name] = st
    copy_bw = info['passes']['copy_d2d (torch copy_)']['GBps_at_median']
    for name, st in info['passes'].items():
        st['of_copy_bw'] = st['GBps_at_median'] / copy_bw
        print('%-30s median %.3f ms [%.3f, %.3f]  %.0f GB/s  %.0f %% of copy' % (
            name, st['median'], st['min'], st['max'], st['GBps_at_median'], 100 * st['of_copy_bw']))
    os.makedirs(os.path.dirname(args.out) or '.', exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(info, f, indent=1)


if __name__ == '__main__':
    main()
