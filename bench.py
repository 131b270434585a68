#!/usr/bin/env python
"""Benchmark of the serial EnSRF analysis step (BASELINE.json metric: obs assimilated/s and state-element
updates/s, HBM GB/s against the roofline, at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config config3] [--cutoff-km 2000]
    python bench.py --impl reference ...         # the reference's CPU path (numpy oracle) on host cores
    python bench.py ... --dump-outputs DIR       # also write the last timed step's outputs to DIR/*.npy

One step = one complete analysis (all observations of the workload, in serial order) of a synthetic
ensemble.  Three measurements share one JSON line:
  value     the analysis with the prior ensemble already resident in HBM (restored from a device copy at
            the start of every step; the state is far larger than L2, so nothing useful stays cached)
  e2e       the same analysis through the host-buffer API (engine.analysis_host, which the Python
            EnSRF.update() uses): pinned host state -> H2D -> analysis -> D2H, copies inside the timing
  cpu_baseline  the CPU oracle's per-observation loop on a bounded sample, rank 0, N = 1 only
  e2e_api   (N = 1) wall time of the reference-shaped call itself, EnSRF(state, obs, loc='GC').update() on an
            EnsembleState and a list of Observation objects (marshalling of 1e5 Python objects included)
For N > 1 (launched by torchrun, one rank per GPU) the state is sharded in latitude bands; the obs-space solve
is distributed over the ranks through NVLink peer memory (config.obs_solve says what actually ran); NCCL
carries the all-reduce of the ob priors and of the solve's results; after the timed region the sharded
analysis is gathered on rank 0 and compared with an unsharded analysis (sharded_check).  In the e2e measurement the host-resident
state is sharded the same way: every rank uploads and downloads its own band over its own PCIe link
(sharding.scatter_bands / gather_bands remain for callers whose state lives on one rank).  Total work is
fixed as N grows: "scaling": "strong".
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
sys.path.insert(0, ROOT)

from efa_xray_b200 import synth  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='config3', choices=sorted(synth.CONFIGS))
    ap.add_argument('--cutoff-km', type=float, default=2000.0, help='localisation support radius (2 x half-width)')
    ap.add_argument('--nobs', type=int, default=None, help='override the number of observations')
    ap.add_argument('--dtype', default='f64', choices=['f64', 'f32'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-api', action='store_true', help='skip the EnSRF(...).update() wall-time measurement (N = 1)')
    ap.add_argument('--no-check', action='store_true', help='skip the sharded-vs-unsharded comparison (N > 1)')
    ap.add_argument('--cpu-seconds', type=float, default=20.0, help='target CPU time of the baseline sample')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs); '
                         'GPU path only: --impl reference times a partial CPU sample of the analysis, so it has no '
                         'complete output to write')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    return args


def measured_traffic(args, cfg, world, kernel):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/traffic.json), when this
    run is the configuration that capture was taken on; else None."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    if not os.path.exists(path):
        return None
    key = '%s/cutoff%.0f/%s/nobs%d/gpus%d' % (args.config, args.cutoff_km, args.dtype, cfg['nobs'], world)
    with open(path) as f:
        return json.load(f).get(key, {}).get(kernel)


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
                power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': smax,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': sorted(reasons)}


def build_case(args, out=None):
    cfg = dict(synth.CONFIGS[args.config])
    if args.nobs:
        cfg['nobs'] = args.nobs
    case = synth.make_case(cutoff_km=args.cutoff_km, seed=args.seed, out=out, **cfg)
    return case, cfg


def obs_arrays(case):
    from efa_xray_b200 import engine
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    tlo, thi, wlo, whi, outside = engine.time_weights(case.times, case.ob_time)
    assert not outside.any()
    return engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                            halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                            row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                            tw0=wlo, tw1=whi)


DUMP_BYTES = 64 * 10 ** 6


def _fixed_sample(n, cap):
    """All of range(n), or `cap` indices of it drawn with a fixed seed, in increasing order: the same ones in every
    run with the same n."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, cap, replace=False))


def dump_outputs(path, X, res):
    """--dump-outputs: what engine.analysis_device, the timed path, gave back in the last timed step, as
    path/<name>.npy, at most DUMP_BYTES in all.  Inputs depend only on the command line (seeded synthetic case), so
    two builds run with the same arguments can be compared file by file.
      prior_mean, prior_var, post_mean, post_var   per-ob diagnostics, float64 (NaN where an ob was not assimilated)
      assimilated                                  1.0 / 0.0 per ob
      analysis                                     the analysis ensemble [rows, nens] in the storage type of the run
    The diagnostics are kept to a quarter of the budget and the analysis to the rest: past that, a fixed sample of
    obs / state rows (_fixed_sample) is written instead of all of them.  Not available with --impl reference, whose
    timed steps run the CPU loop over a sample of the obs and never produce a complete analysis."""
    os.makedirs(path, exist_ok=True)
    diag = {'prior_mean': res.prior_mean, 'prior_var': res.prior_var, 'post_mean': res.post_mean,
            'post_var': res.post_var, 'assimilated': res.assimilated.astype(np.float64)}
    obs_idx = _fixed_sample(len(res.prior_mean), DUMP_BYTES // 4 // (8 * len(diag)))
    for name, a in diag.items():
        np.save(os.path.join(path, name + '.npy'), np.asarray(a, dtype=np.float64)[obs_idx])
    nrows, nens = X.shape
    room = DUMP_BYTES - 8 * len(diag) * obs_idx.size - 4096          # 4096: the .npy headers
    rows = _fixed_sample(nrows, room // (nens * X.element_size()))
    import torch
    np.save(os.path.join(path, 'analysis.npy'), X[torch.as_tensor(rows, device=X.device)].cpu().numpy())


def workload_name(args, cfg):
    return ('%s: %d-member %dx%d grid x %d vars x %d times, %d obs, serial EnSRF, Gaspari-Cohn cutoff %.0f km'
            % (args.config, cfg['nmem'], cfg['ny'], cfg['nx'], cfg['nvars'], cfg['ntimes'], cfg['nobs'],
               args.cutoff_km))


# ----------------------------------------------------------------------------------------------
# CPU reference arm (oracle)
# ----------------------------------------------------------------------------------------------
class CpuSample:
    """The reference's per-observation loop (oracle.ensrf_loop, a restatement of ensrf.py:50-149 with the
    reference's dense arithmetic) on the FULL state of the workload, carrying only the first `n_carry`
    observations as obs-space rows.  Carrying all 1e5 obs is infeasible for the reference (its ob-prior
    setup alone is hours) -- the sample therefore UNDERSTATES the reference's per-ob cost, which grows with
    the number of carried obs (observation.py:70-74)."""

    def __init__(self, case, n_carry):
        from oracle import ensrf_oracle as O
        self.O = O
        n_carry = min(n_carry, case.nobs)
        self.case = case
        st = O.State.__new__(O.State)
        st.fields = case.fields               # no copy: the loop never writes the state object
        st.varnames = list(case.varnames)
        st.lat, st.lon = case.lat2d, case.lon2d
        st.times = case.times.astype('datetime64[ns]')
        self.state = st
        self.obs = O.obs_from_case(case)[:n_carry]
        ny, nx = case.lat2d.shape
        idx, w = O.stencils_regular(case.lat2d, case.lon2d, case.ob_lat[:n_carry], case.ob_lon[:n_carry])
        ti = np.searchsorted(case.times, case.ob_time[:n_carry])
        ye = np.zeros((n_carry, case.nmem))
        for k in range(n_carry):
            f = case.fields[case.varnames[int(case.ob_var[k])]][ti[k]].reshape(ny * nx, case.nmem)
            ye[k] = (w[k][:, None] * f[idx[k]]).sum(axis=0)
        prior = st.to_vect()
        xbm = prior.mean(axis=1)
        prior -= xbm[:, None]
        self.xam = np.hstack((xbm, ye.mean(axis=1)))
        self.Xap = np.vstack((prior, ye - ye.mean(axis=1, keepdims=True)))
        del prior
        self.done = 0

    def run(self, n):
        """Advance the serial loop by n observations; returns (seconds, number assimilated)."""
        O = self.O
        n = min(n, len(self.obs))
        if n == 0:
            return 0.0, 0
        t0 = time.perf_counter()
        self.xam, self.Xap = O.ensrf_loop(self.state, self.obs, self.xam, self.Xap, loc='GC', max_obs=n)
        dt = time.perf_counter() - t0
        nass = sum(1 for o in self.obs[:n] if o.assimilate_this)
        # the rows of obs already processed are never read again (ensrf.py:61-64): drop them (untimed) so
        # the next call continues the same serial loop with the next ob at row Nstate+0
        ns = self.state.nstate()
        self.xam = np.concatenate([self.xam[:ns], self.xam[ns + n:]])
        self.Xap = np.concatenate([self.Xap[:ns], self.Xap[ns + n:]])
        self.obs = self.obs[n:]
        return dt, nass


def host_mem_ok(need_gb):
    try:
        import psutil
        return psutil.virtual_memory().available / 2 ** 30 > need_gb
    except ImportError:
        return True


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    case, cfg = build_case(args)
    state_gb = cfg['nmem'] * cfg['ny'] * cfg['nx'] * cfg['nvars'] * cfg['ntimes'] * 8 / 2 ** 30
    cores = os.cpu_count()
    if not host_mem_ok(6 * state_gb + 4):
        print(json.dumps({'impl': 'reference', 'unavailable': 'host RAM too small for the oracle at this workload'}))
        return
    n_carry = 256
    cpu = CpuSample(case, n_carry)
    dt1, _ = cpu.run(1)                                    # untimed probe to size the steps
    per_step = max(1, min(8, int(round(args.cpu_seconds / max(dt1, 1e-3) / max(args.steps + args.warmup, 1)))))
    for _ in range(args.warmup):
        cpu.run(per_step)
    tot_t, tot_n = 0.0, 0
    for _ in range(args.steps):
        dt, n = cpu.run(per_step)
        tot_t += dt
        tot_n += n
    value = tot_n / tot_t
    sample = ('%d obs per step of the serial loop on the full %s state, %d of %d obs carried as obs-space rows '
              '(numpy oracle of ensrf.py:50-149; understates the per-ob cost of carrying all obs)'
              % (per_step, args.config, n_carry, cfg['nobs']))
    line = {
        'impl': 'reference', 'metric': 'obs_assimilated_per_s', 'value': value, 'unit': 'obs/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot_t / args.steps,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload_name(args, cfg), 'obs_per_step': per_step},
        'cpu_baseline': {'value': value, 'unit': 'obs/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'obs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from efa_xray_b200 import engine, sharding, _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.gpus > 1 and world == 1:
        # not under torchrun: relaunch ourselves the way the driver does
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(args.gpus),
               '--master-addr', '127.0.0.1', '--master-port', '29531', os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    _lib.require_device()
    tdtype = torch.float64 if args.dtype == 'f64' else torch.float32
    esize = 8 if args.dtype == 'f64' else 4

    # ---- synthetic workload (every rank builds the same case from the same seed) ----------
    cfg = dict(synth.CONFIGS[args.config])
    if args.nobs:
        cfg['nobs'] = args.nobs
    nlev = cfg['nvars'] * cfg['ntimes']
    ny, nx, nens = cfg['ny'], cfg['nx'], cfg['nmem']
    nrows = nlev * ny * nx
    # the host-resident state has the storage type of the run (float32 runs: float32 storage, float64 arithmetic)
    state_gb_host = nrows * nens * esize / 2 ** 30
    if not host_mem_ok(3.0 * state_gb_host + 8):
        raise SystemExit('bench.py: not enough host RAM for a %.1f GB state' % state_gb_host)
    if not args.no_e2e and not host_mem_ok(4.0 * state_gb_host + 8):
        args.no_e2e = True                      # the end-to-end leg needs a second page-locked copy of the state
        print('bench.py: skipping the e2e leg (host RAM)', file=sys.stderr)
    Xh = torch.empty((nrows, nens), dtype=tdtype, pin_memory=True)
    case, _ = build_case(args, out=Xh.numpy().reshape(cfg['nvars'], cfg['ntimes'], ny, nx, nens))
    obs = obs_arrays(case)
    nassim = int(obs.assimilate.sum())
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    loc_mode = engine.LOC_GC

    if world > 1:
        work = sharding.estimate_row_work(case.lat2d, case.lon2d, obs.lat, obs.lon, 2.0 * obs.halfwidth, obs.assimilate)
        bands = sharding.partition_bands(work, world)
        band = bands[rank]
    else:
        bands, band = [(0, ny)], None
    y0, y1 = bands[rank]
    X0 = sharding.band_view(Xh, nlev, ny, nx, y0, y1).contiguous().reshape(-1, nens).to(dev).to(tdtype)
    X = torch.empty_like(X0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        X.copy_(X0)
        return engine.analysis_device(X, nlev, grid, obs, loc_mode, band=band)

    for _ in range(args.warmup):
        res = step()
    peak_tf = peak_dmma = None
    if rank == 0:
        import ctypes as C
        tf = C.c_double(0.0)
        _lib.call('exb_measure_fp64_peak', C.byref(tf), _lib.stream_ptr())
        peak_tf = tf.value
        _lib.call('exb_measure_dmma_peak', C.byref(tf), _lib.stream_ptr())
        peak_dmma = tf.value

    sampler = ClockSampler(local_rank)
    barrier()
    launches0 = _lib.launch_count()
    if rank == 0 and not os.environ.get('EXB_NO_CLOCKS'):
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    e0.record()
    marks[0].record()
    phases = {}
    for i in range(args.steps):
        res = step()
        marks[i + 1].record()
        for k, v in res.ms.items():
            phases[k] = phases.get(k, 0.0) + v / args.steps
    e1.record()
    barrier()
    step_ms = [marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0
    ms_total = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    pairs = torch.tensor([float(res.state_pairs)], dtype=torch.float64, device=dev)
    su_ms = torch.tensor([phases.get('state_update', 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        dist.all_reduce(pairs, op=dist.ReduceOp.SUM)
        su_max = su_ms.clone()
        dist.all_reduce(su_max, op=dist.ReduceOp.MAX)
    else:
        su_max = su_ms
    ms_step = float(ms_total.item()) / args.steps
    state_pairs = float(pairs.item())                      # sum_k |F_s(k)| over the whole grid

    if args.dump_outputs:
        # X holds the analysis of the last timed step; at N > 1 its bands are assembled on rank 0 first
        full = X
        if world > 1:
            full = torch.empty((nrows, nens), dtype=tdtype, device=dev) if rank == 0 else None
            sharding.gather_bands(X, full, bands, nlev, ny, nx, nens, rank)
        if rank == 0:
            dump_outputs(args.dump_outputs, full, res)
        del full

    # ---- e2e: host buffers, copies inside the timed region ------------------------------------
    e2e = None
    if not args.no_e2e:
        # host-resident state: at N = 1 one pinned buffer; at N > 1 sharded by latitude bands, every rank holds,
        # uploads and downloads its own band (pinned) over its own PCIe link
        if world == 1:
            Xh_in, Oh = Xh, torch.empty(Xh.shape, dtype=Xh.dtype, pin_memory=True)
        else:
            Xh_in = sharding.band_view(Xh, nlev, ny, nx, y0, y1).contiguous().reshape(-1, nens).pin_memory()
            Oh = torch.empty(Xh_in.shape, dtype=Xh_in.dtype, pin_memory=True)

        def e2e_step():
            return engine.analysis_host(Xh_in, nlev, case.lat2d, case.lon2d, obs, loc_mode, device=dev, dtype=tdtype,
                                        grid=grid, out=Oh, band=band)

        for _ in range(min(args.warmup, 2)):
            e2e_step()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        n_e2e = max(1, min(args.steps, 3))
        e2e_walls = []
        for _ in range(n_e2e):
            t0 = time.perf_counter()
            r = e2e_step()
            torch.cuda.synchronize()
            e2e_walls.append((round(1e3 * (time.perf_counter() - t0), 1), {k: round(v, 1) for k, v in r.ms.items()}))
        f1.record()
        if os.environ.get('EXB_BENCH_DEBUG'):
            print('e2e steps:', e2e_walls, file=sys.stderr)
        barrier()
        t = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item()) / n_e2e
        ob_bytes = sum(getattr(obs, f).nbytes for f in ('value', 'error', 'lat', 'lon', 'halfwidth', 'assimilate',
                                                        'row0', 'row1', 'tw0', 'tw1')) + 2 * obs.nobs * 8
        e2e = {'value': nassim / (e2e_ms * 1e-3), 'unit': 'obs/s', 'ms_per_step': e2e_ms,
               'h2d_bytes_per_step': int(Xh.numel() * esize + ob_bytes * world),
               'd2h_bytes_per_step': int(Xh.numel() * esize + 8 * obs.nobs * 8 + 24),
               'api': 'efa_xray_b200.engine.analysis_host (pinned host state in, pinned host analysis out%s)'
                      % ('' if world == 1 else '; state sharded over the ranks by latitude band, each rank moves its own band')}

    # ---- N > 1: the sharded analysis against an unsharded one on rank 0 (outside every timed region) ----------
    sharded_check = None
    if world > 1 and not args.no_check:
        X.copy_(X0)
        engine.analysis_device(X, nlev, grid, obs, loc_mode, band=band)
        full = torch.empty((nrows, nens), dtype=tdtype, device=dev) if rank == 0 else None
        sharding.gather_bands(X, full, bands, nlev, ny, nx, nens, rank)
        if rank == 0:
            ref = Xh.to(dev).to(tdtype)
            prior_max_inc = ref.clone()
            engine.analysis_device(ref, nlev, grid, obs, loc_mode)
            inc = float((ref - prior_max_inc).abs().max())
            del prior_max_inc
            diff = float((full - ref).abs().max())
            tol = 1e-9 if args.dtype == 'f64' else 1e-3
            sharded_check = {'max_abs_diff': diff, 'largest_increment': inc, 'rel_to_increment': diff / inc,
                             'tolerance': tol, 'ok': bool(diff <= tol * inc),
                             'what': 'sharded analysis gathered on rank 0 vs an unsharded analysis of the same inputs'}
            del ref, full
        dist.barrier()

    # ---- N = 1: the reference-shaped call itself --------------------------------------------------------------
    e2e_api = None
    if world == 1 and not args.no_api and not args.no_e2e and args.dtype == 'f64':
        from efa_xray_b200.state.ensemble import EnsembleState
        from efa_xray_b200.observation.observation import Observation
        from efa_xray_b200.assimilation.ensrf import EnSRF
        state, oblist = synth.build_objects(case, EnsembleState, Observation)     # adopts the pinned buffer (no copy)
        walls = []
        for i in range(3):
            for o in oblist:
                o.prior_mean = o.post_mean = o.prior_var = o.post_var = None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            post_state, _ = EnSRF(state, oblist, verbose=False, loc='GC').update()
            torch.cuda.synchronize()
            walls.append(1e3 * (time.perf_counter() - t0))
            if i < 2:
                del post_state                    # its page-locked block goes back to the pool for the next call
        api_ms = min(walls[1:])
        pv = np.array([o.post_var for o in oblist], dtype=np.float64)
        e2e_api = {'value': nassim / (api_ms * 1e-3), 'unit': 'obs/s', 'ms_per_call': api_ms, 'wall_ms_all_calls': walls,
                   'api': "efa_xray.assimilation.ensrf.EnSRF(state, obs, loc='GC', verbose=False).update() -- EnsembleState "
                          "(page-locked block) + %d Observation objects in, new EnsembleState + diagnostics on the obs out; "
                          "first call includes the page-locked allocation of the posterior block" % len(oblist),
                   'post_var_matches_device_path': bool(np.allclose(pv, res.post_var, rtol=1e-9, equal_nan=True)),
                   'posterior_checksum': float(np.abs(post_state.to_vect()[::997]).sum())}
        del post_state, state

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (state sweep) -----------------------------------------
    hbm_peak, peak_src = peaks()
    su_s = float(su_max.item()) * 1e-3
    sweep_kernel = ('state_sweep_2p_kernel' if os.environ.get('EXB_SP_IMPL') != 'v3' else 'state_sweep_pipe_kernel') \
        if nens <= 103 else 'state_update_kernel'
    alg_bytes = state_pairs * 2.0 * (nens + 1) * esize          # SURVEY.md 8d: |F_s| * 2 * (Nens+1) * sizeof(T)
    achieved = alg_bytes / su_s / 1e9 / world                   # per GPU
    flops = state_pairs * (4.0 * nens + 3.0)
    line = {
        'metric': 'obs_assimilated_per_s', 'value': nassim / (ms_step * 1e-3), 'unit': 'obs/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
        'config': {'workload': workload_name(args, cfg), 'l2_policy': 'state (%.2f GB) >> L2; restored from a device copy each step'
                   % (nrows * nens * esize / 1e9), 'parallelism': 'lat-bands x%d (work-balanced), obs-space solve %s' % (world, res.obs_solve),
                   'obs_solve': res.obs_solve, 'bands': bands},
        'state_updates_per_s': state_pairs / (ms_step * 1e-3),
        'state_row_updates': state_pairs, 'obs_assimilated': nassim,
        'phases_ms': dict(phases, setup=sum(v for k, v in phases.items() if k.startswith('setup_'))), 'step_ms': step_ms,
        'roofline': {'bound': 'hbm', 'kernel': sweep_kernel, 'achieved': achieved, 'peak': hbm_peak,
                     'unit': 'GB/s', 'frac': achieved / hbm_peak, 'traffic': measured_traffic(args, cfg, world, sweep_kernel),
                     'peak_source': peak_src,
                     'note': 'achieved = ALGORITHMIC bytes of the per-observation formulation (sum_k |F_s(k)| * 2 * '
                             '(Nens+1) * sizeof(T)) / kernel time, per GPU.  The kernel is tile-stationary: the state '
                             'crosses HBM once, so real DRAM traffic (traffic, bytes per launch from ncu) is far below '
                             'the algorithmic bytes and frac > 1 is a traffic reduction; the binding limit is the FP64 '
                             'tensor pipe (roofline_fp64).'},
        'roofline_fp64': {'bound': 'fp64_tensor', 'achieved': flops / su_s / 1e12 / world, 'peak': peak_dmma, 'unit': 'TFLOP/s',
                          'frac': (flops / su_s / 1e12 / world) / peak_dmma if peak_dmma else None,
                          'peak_fma': peak_tf, 'frac_of_fma_peak': (flops / su_s / 1e12 / world) / peak_tf if peak_tf else None,
                          'peak_source': 'exb_measure_dmma_peak (mma.sync m8n8k4 f64, 8 independent tiles per warp) and '
                                         'exb_measure_fp64_peak (DFMA loop), both in this run',
                          'note': 'achieved = algorithmic flop (4 Nens + 3 per (row, ob) pair with non-zero weight) / '
                                  'kernel time'},
        'e2e': e2e, 'e2e_api': e2e_api, 'sharded_check': sharded_check, 'gpu_launches': int(launches), 'clocks': clocks,
    }

    if world == 1 and not args.no_cpu_baseline and args.dtype == 'f64':
        del X, X0
        torch.cuda.empty_cache()
        state_gb = nrows * nens * 8 / 2 ** 30
        if host_mem_ok(6 * state_gb + 4):
            cpu = CpuSample(case, 256)
            dt1, _ = cpu.run(1)
            n = max(2, min(24, int(round(args.cpu_seconds / max(dt1, 1e-3)))))
            dt, nass = cpu.run(n)
            line['cpu_baseline'] = {
                'value': nass / dt, 'unit': 'obs/s', 'cores': os.cpu_count(), 'kind': 'port',
                'sample': '%d obs of the serial loop on the full %s state with 256 of %d obs carried as obs-space rows '
                          '(numpy oracle of ensrf.py:50-149, all BLAS threads; understates the reference\'s per-ob cost)'
                          % (n, args.config, cfg['nobs'])}
        else:
            line['cpu_baseline'] = {'value': None, 'unit': 'obs/s', 'cores': os.cpu_count(), 'kind': 'port',
                                    'sample': 'skipped: not enough host RAM'}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
