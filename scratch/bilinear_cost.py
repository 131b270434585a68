"""Cost of the bilinear forward operator (DESIGN.md section 4.8): profiles/r06_bilinear.md.

    python scratch/bilinear_cost.py [--steps 10] [--reps 200] [--out bilinear_cost.json]

1. BASELINE config 3 (f64, 100 members, 721x1440x3, 1e5 obs): CUDA-event times of exb_stencil_search_rect (the
   reference operator's stencil) and exb_stencil_bilinear_rect over many launches, alternated.
2. engine.analysis_device with forward_operator 'reference' / 'bilinear', alternated step by step (the state is reset
   from a device copy of the prior before every step, outside the timed window); median and spread of each.
3. exb_stencil_bilinear_curv with 1e5 obs on a 1000x1000 Lambert-conformal regional grid and on a 721x1440
   curvilinear grid (the config-3 grid with lat perturbed along x, so that it is not rectilinear).
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
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def lambert_grid(ny, nx, dx_km, lat0=40.0, lon0=-100.0):
    R = 6371.0
    n = np.sin(np.radians(lat0))
    F = np.cos(np.radians(lat0)) * np.tan(np.pi / 4 + np.radians(lat0) / 2) ** n / n
    rho0 = R * F / np.tan(np.pi / 4 + np.radians(lat0) / 2) ** n
    y, x = np.meshgrid((np.arange(ny) - ny / 2) * dx_km, (np.arange(nx) - nx / 2) * dx_km, indexing='ij')
    rho = np.sign(n) * np.hypot(x, rho0 - y)
    lat = np.degrees(2 * np.arctan((R * F / rho) ** (1 / n)) - np.pi / 2)
    lon = lon0 + np.degrees(np.arctan2(x, rho0 - y) / n)
    return np.ascontiguousarray(lat), np.ascontiguousarray(lon)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--reps', type=int, default=200)
    ap.add_argument('--out', default='bilinear_cost.json')
    a = ap.parse_args()
    import torch
    from efa_xray_b200 import engine, _lib
    from efa_xray_b200.synth import make_case, CONFIGS
    dev = torch.device('cuda', 0)
    out = {'card': card()}

    case = make_case(cutoff_km=2000.0, seed=0, **CONFIGS['config3'])
    ny, nx = case.lat2d.shape
    nt, nlev = len(case.times), len(case.varnames) * len(case.times)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    obs_by = {}
    for op in ('reference', 'bilinear'):
        tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time, swapped=op == 'reference')
        obs_by[op] = engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                                      halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                                      row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                                      tw0=wlo, tw1=whi)
    obs = obs_by['reference']
    d_lat, d_lon = engine._dev_f64(obs.lat, dev), engine._dev_f64(obs.lon, dev)
    d_sl, d_cl = engine._dev_f64(np.sin(np.radians(obs.lat)), dev), engine._dev_f64(np.cos(np.radians(obs.lon)), dev)
    engine.stencil_bilinear(grid, d_lat, d_lon)            # builds the tables
    torch.cuda.synchronize()

    # 1. stencil kernels, alternated in blocks
    search = lambda: engine.stencil_search(grid, None, None, dev_tables=(d_lat, d_lon, d_sl, d_cl))
    bil = lambda: engine.stencil_bilinear(grid, d_lat, d_lon)
    for fn in (search, bil):
        event_ms(fn, 10)
    st = {'reference_search_rect': [], 'bilinear_rect': []}
    for _ in range(5):
        st['reference_search_rect'].append(event_ms(search, a.reps))
        st['bilinear_rect'].append(event_ms(bil, a.reps))
    out['stencil_ms_per_call'] = {k: {'median': float(np.median(v)), 'all': v} for k, v in st.items()}
    print(json.dumps(out['stencil_ms_per_call']), flush=True)

    # 2. analysis step per operator, alternated
    prior = torch.as_tensor(case.to_vect()).to(dev)
    X = torch.empty_like(prior)
    steps = {'reference': [], 'bilinear': []}
    setup = {'reference': [], 'bilinear': []}
    for i in range(a.steps + 1):
        for op in ('reference', 'bilinear'):
            X.copy_(prior)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = engine.analysis_device(X, nlev, grid, obs_by[op], engine.LOC_GC, forward_operator=op)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            assert res.n_outside == 0 and res.n_exact == 0
            if i > 0:                                      # the first round is warm-up
                steps[op].append(ms)
                setup[op].append(res.ms.get('setup_ob_priors', float('nan')))
    out['analysis_step_ms'] = {op: {'median': float(np.median(v)), 'min': float(np.min(v)), 'max': float(np.max(v)),
                                    'setup_ob_priors_median': float(np.median(setup[op])), 'all': v}
                               for op, v in steps.items()}
    print(json.dumps(out['analysis_step_ms']), flush=True)
    del prior, X, case

    # 3. curvilinear kernel
    rng = np.random.default_rng(0)
    curv = {}
    lat_l, lon_l = lambert_grid(1000, 1000, 3.0)
    lat_g = np.ascontiguousarray(grid.lat.view(ny, nx).cpu().numpy() + 1e-7 * np.arange(nx)[None, :] / nx)
    lon_g = grid.lon.view(ny, nx).cpu().numpy()
    for name, (la, lo) in (('lambert_1000x1000', (lat_l, lon_l)), ('curvilinear_721x1440', (lat_g, lon_g))):
        g = engine.GridTables(la, lo, dev)
        assert g.bilinear_tables()[0] == 'curv'
        n = 100000
        yy, xx = rng.integers(1, la.shape[0] - 2, n), rng.integers(1, la.shape[1] - 2, n)
        if name.startswith('curvilinear'):
            yy = rng.integers(60, 660, n)                  # away from the pole rows
        olat = la[yy, xx] + rng.uniform(0, 1, n) * (la[yy + 1, xx] - la[yy, xx])
        olon = lo[yy, xx] + rng.uniform(0, 1, n) * (lo[yy, xx + 1] - lo[yy, xx])
        dl, dn = engine._dev_f64(olat, dev), engine._dev_f64(olon, dev)
        fn = lambda: engine.stencil_bilinear(g, dl, dn)
        _, _, nout = fn()
        reps = max(3, a.reps // 40)
        curv[name] = {'ms_per_call': event_ms(fn, reps), 'reps': reps, 'n_outside': int(nout.item()), 'nobs': n,
                      'npts': int(la.size)}
        print(name, json.dumps(curv[name]), flush=True)
    out['curvilinear'] = curv
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
