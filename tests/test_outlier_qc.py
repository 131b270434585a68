"""Outlier quality control inside the serial loop (DESIGN.md section 4.7).

The reference is the unmodified CPU oracle: the QC analysis is the EnSRF run with flags F' = F and not R, where R is
the set of obs that fail |innov| > t sqrt(varye + R_err) in that run.  R is unique, because the decision for ob k
depends only on obs < k, and qc_reference below finds it with repeated oracle solves.  Cases get gross errors
(5 % of the obs moved by 8 to 15 sigma), and every case asserts that no checked ob lies near its threshold."""
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from efa_xray_b200.synth import make_case, build_objects

F64_RTOL = 1e-10          # as test_gpu_parity._check_post
F64_INC_TOL = 1e-9


def _api():
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    from efa_xray_b200.assimilation.ensrf import EnSRF
    return EnsembleState, Observation, EnSRF


# ---------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------
def qc_reference(ymean, ypert, value, error, halfwidth, lat, lon, assim, threshold, loc='GC', start=None, margin=1e-6):
    """Rejected set R and the oracle's obs-space records of the run with flags assim & ~R.

    Fixed point over oracle.obs_space_solve: each pass runs the solve with the current flags and finds the first ob
    whose decision disagrees with R (a checked ob that fails but is not in R, or an ob in R that passes), and
    flips it.  Obs before it keep their decisions from then on, since those depend only on earlier obs.  `start` is
    an initial guess of R: the result does not depend on it, only the number of solves does.  Asserts that no checked
    ob's |innov| lies within `margin` (relative) of its limit, so a tie fails loudly instead of flaking."""
    from oracle import ensrf_oracle as O
    assim = np.asarray(assim, dtype=bool)
    threshold = np.asarray(threshold, dtype=np.float64)
    checked = assim & np.isfinite(threshold)
    rej = np.zeros(len(value), dtype=bool) if start is None else (np.asarray(start, dtype=bool) & checked)
    for _ in range(int(checked.sum()) + 1):
        rec = O.obs_space_solve(ymean, ypert, value, error, halfwidth, lat, lon, assim & ~rej, loc=loc)
        innov = np.abs(value - rec['prior_mean'])
        with np.errstate(invalid='ignore'):
            limit = threshold * np.sqrt(rec['prior_var'] + error)
            fails = checked & (innov > limit)
        bad = np.flatnonzero(fails != rej)
        if bad.size == 0:
            near = checked & (np.abs(innov - limit) <= margin * limit)
            assert not near.any(), 'obs %s lie within %g of their threshold' % (np.flatnonzero(near)[:10], margin)
            return rej, rec
        rej[bad[0]] = fails[bad[0]]
    raise AssertionError('no fixed point')


def _threshold_per_ob(case, outlier_threshold):
    if isinstance(outlier_threshold, dict):
        per_var = np.array([outlier_threshold.get(v, np.inf) for v in case.varnames], dtype=np.float64)
        return per_var[case.ob_var]
    return np.full(case.nobs, float(outlier_threshold))


def _with_gross_errors(case, frac=0.05, seed=0):
    """A copy of `case` with a fraction of its obs moved by 8 to 15 sigma (sigma = sqrt(error)), either sign."""
    rng = np.random.default_rng(seed)
    k = rng.choice(case.nobs, max(1, int(round(frac * case.nobs))), replace=False)
    value = case.ob_value.copy()
    value[k] += rng.choice([-1.0, 1.0], k.size) * rng.uniform(8.0, 15.0, k.size) * np.sqrt(case.ob_error[k])
    return dataclasses.replace(case, ob_value=value)


def reference_analysis(case, outlier_threshold, loc='GC', margin=1e-6):
    """(R, obs-space records, posterior state vector, reference obs) of the QC analysis of `case`: the oracle's
    ensrf_update with the flags of R cleared."""
    from oracle import ensrf_oracle as O
    state, obs = O.State.from_case(case), O.obs_from_case(case)
    ymean, ypert = O.compute_ob_priors(state, obs)
    rej, rec = qc_reference(ymean, ypert, case.ob_value, case.ob_error, case.ob_halfwidth, case.ob_lat, case.ob_lon,
                            case.ob_assimilate, _threshold_per_ob(case, outlier_threshold),
                            loc=loc if loc else None, margin=margin)
    for o, r in zip(obs, rej):
        o.assimilate_this = o.assimilate_this and not r
    post, obs = O.ensrf_update(O.State.from_case(case), obs, loc=loc)
    return rej, rec, post.to_vect(), obs


# ---------------------------------------------------------------------------------------------------------------
# CPU: the reference has a known answer, and pins the in-loop semantics
# ---------------------------------------------------------------------------------------------------------------
def _pair(value1, error0, threshold):
    """Two obs 0.01 degree apart with identical perturbations (variance 4); ob 0 has no innovation."""
    ypert = np.array([[2.0, -2.0, 2.0, -2.0], [2.0, -2.0, 2.0, -2.0]])
    ymean = np.zeros(2)
    return dict(ymean=ymean, ypert=ypert, value=np.array([0.0, value1]), error=np.array([error0, 1.0]),
                halfwidth=np.full(2, 2000.0), lat=np.array([10.0, 10.01]), lon=np.array([20.0, 20.0]),
                assim=np.ones(2, dtype=bool), threshold=np.full(2, threshold))


def _pre_loop_rejects(p):
    return np.abs(p['value'] - p['ymean']) > p['threshold'] * np.sqrt(p['ypert'].var(axis=1) + p['error'])


def test_reference_rejects_in_loop_what_a_pre_loop_check_keeps():
    """Ob 1 passes against the initial prior (3.5 < 2 sqrt(5)), but ob 0 shrinks its variance from 4 to about 0.28,
    and against the in-loop prior it fails (3.5 > 2 sqrt(1.28))."""
    p = _pair(3.5, 1.0, 2.0)
    assert not _pre_loop_rejects(p).any()
    rej, rec = qc_reference(**p)
    np.testing.assert_array_equal(rej, [False, True])
    assert 0.2 < rec['prior_var'][1] < 0.35
    assert np.isnan(rec['post_mean'][1]) and np.isfinite(rec['post_mean'][0])


def test_reference_keeps_in_loop_what_a_pre_loop_check_rejects():
    """Both obs see an innovation of 4, which fails 1.5 sqrt(4 + 1) for ob 1 against the initial prior.  Ob 0 (error
    9) passes and pulls ob 1's prior mean about 1.6 toward it: against the in-loop prior ob 1 passes."""
    p = _pair(4.0, 9.0, 1.5)
    p['value'][0] = 4.0
    pre = _pre_loop_rejects(p)
    np.testing.assert_array_equal(pre, [False, True])
    rej, rec = qc_reference(**p)
    np.testing.assert_array_equal(rej, [False, False])
    assert abs(p['value'][1] - rec['prior_mean'][1]) < 3.0


def test_reference_does_not_depend_on_the_start():
    from oracle import ensrf_oracle as O
    case = _with_gross_errors(make_case(ny=19, nx=36, nmem=10, nvars=1, nobs=80, cutoff_km=3000.0, seed=7,
                                        frac_skip=0.1), seed=7)
    ymean, ypert = O.compute_ob_priors(O.State.from_case(case), O.obs_from_case(case))
    args = (ymean, ypert, case.ob_value, case.ob_error, case.ob_halfwidth, case.ob_lat, case.ob_lon, case.ob_assimilate,
            np.full(case.nobs, 3.0))
    rej, rec = qc_reference(*args)
    assert 3 <= rej.sum() and not (rej & ~case.ob_assimilate).any()
    for start in (np.ones(case.nobs, dtype=bool), rej, np.random.default_rng(1).uniform(size=case.nobs) < 0.5):
        r2, rec2 = qc_reference(*args, start=start)
        np.testing.assert_array_equal(r2, rej)
        np.testing.assert_array_equal(rec2['prior_var'], rec['prior_var'])


# ---------------------------------------------------------------------------------------------------------------
# CPU: the Python API validates before any device work, and expands the threshold per ob
# ---------------------------------------------------------------------------------------------------------------
def _small_objects(nvars=3):
    EnsembleState, Observation, _ = _api()
    case = make_case(ny=19, nx=36, nmem=6, nvars=nvars, ntimes=2, nobs=9, seed=91)
    return case, build_objects(case, EnsembleState, Observation)


@pytest.mark.parametrize('outlier_threshold', [
    0.0, -1.0, float('nan'), float('inf'), -float('inf'), '3', True, [3.0], (3.0,), {'nope': 3.0}, {'var0': 0.0},
    {'var1': None}, {'var2': float('inf')}, {'var0': '3'}, 0,
])
def test_invalid_outlier_threshold_raises_value_error(outlier_threshold):
    from efa_xray_b200.assimilation.assimilation import update
    _, _, EnSRF = _api()
    _, (state, obs) = _small_objects()
    with pytest.raises(ValueError):
        EnSRF(state, obs, verbose=False, loc='GC', outlier_threshold=outlier_threshold)
    with pytest.raises(ValueError):
        update(state, obs, loc='GC', outlier_threshold=outlier_threshold)


def test_threshold_expands_per_ob():
    from efa_xray_b200 import engine
    _, _, EnSRF = _api()
    case, (state, obs) = _small_objects()
    ens = EnSRF(state, obs, verbose=False)
    assert ens.outlier_threshold is None and not ens._obs_arrays(engine.LOC_GC, None).qc
    for t in (3.0, 2, np.float32(2.5)):
        a = EnSRF(state, obs, verbose=False, outlier_threshold=t)
        np.testing.assert_array_equal(a._obs_arrays(engine.LOC_GC, a.outlier_threshold).threshold,
                                      np.full(case.nobs, float(t)))
    d = {'var2': 4.0, 'var0': 2.5}
    a = EnSRF(state, obs, verbose=False, outlier_threshold=d)
    got = a._obs_arrays(engine.LOC_GC, a.outlier_threshold).threshold
    want = np.array([{0: 2.5, 1: np.inf, 2: 4.0}[v] for v in case.ob_var])
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got, _threshold_per_ob(case, d))
    assert set(case.ob_var.tolist()) == {0, 1, 2}


@pytest.mark.parametrize('threshold', [np.array([3.0]), np.full(8, 3.0), np.full((9, 1), 3.0)])
def test_engine_rejects_thresholds_of_the_wrong_length(threshold):
    """engine.upload_obs (behind analysis_device / analysis_host) refuses a threshold array that is neither empty nor
    one value per ob, before any device work."""
    from efa_xray_b200 import engine
    n = 9
    z = np.zeros(n)
    obs = engine.ObsArrays(value=z, error=z + 1.0, lat=z, lon=z, halfwidth=z + 1000.0, assimilate=np.ones(n, np.uint8),
                           row0=np.zeros(n, np.int64), row1=np.zeros(n, np.int64), tw0=z + 1.0, tw1=z,
                           threshold=threshold)
    with pytest.raises(ValueError, match='one value per ob'):
        engine.upload_obs(obs, 'cpu', engine.LOC_GC)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the public API against the reference
# ---------------------------------------------------------------------------------------------------------------
def _patch(monkeypatch, env):
    """The settings a case runs under: EXB_* environment variables, and attributes of engine (FUSED_MAX_NENS = 0 takes
    the three-call form: split, exb_state_update, recombine)."""
    from efa_xray_b200 import engine
    for name, value in env.items():
        if name.startswith('EXB_'):
            monkeypatch.setenv(name, value)
        else:
            monkeypatch.setattr(engine, name, value)


def _diag(obs, attr):
    return np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr)) for o in obs])


def _check_post(post, ref_post, prior, tol_scale=1.0):
    np.testing.assert_allclose(post, ref_post, rtol=F64_RTOL * tol_scale)
    inc_ref = ref_post - prior
    scale = max(np.abs(inc_ref).max(), 1e-30)
    assert np.abs((post - prior) - inc_ref).max() <= F64_INC_TOL * tol_scale * scale


_C = dict(ny=25, nx=48, nvars=2, ntimes=1, nobs=120, frac_skip=0.05)


@pytest.mark.gpu
@pytest.mark.parametrize('kw,loc,threshold,env', [
    (dict(_C, nmem=50, cutoff_km=2500.0, seed=301), 'GC', 3.0, {}),
    (dict(_C, nmem=50, cutoff_km=2500.0, seed=301), 'GC', 3.0, {'EXB_OBS_IMPL': 'persistent'}),
    (dict(_C, nmem=20, seed=302), False, 3.5, {}),
    (dict(_C, nmem=7, cutoff_km=1500.0, seed=303), 'GC', 2.5, {}),
    (dict(_C, nmem=32, cutoff_km=3000.0, seed=304), 'GC', 3.0, {}),
    (dict(_C, nmem=100, cutoff_km=3000.0, seed=305), 'GC', 3.0, {}),
    (dict(ny=19, nx=36, nvars=1, ntimes=1, nobs=80, nmem=130, cutoff_km=4000.0, seed=306), 'GC', 3.0, {}),
    (dict(_C, nmem=50, cutoff_km=2500.0, seed=307), 'GC', 3.0, {'FUSED_MAX_NENS': 0}),
    (dict(_C, nmem=50, cutoff_km=2500.0, seed=308, frac_skip=0.2), 'GC', {'var1': 2.5}, {}),
    (dict(_C, nmem=50, cutoff_km=2500.0, seed=308, frac_skip=0.2), 'GC', {'var0': 3.0, 'var1': 2.0},
     {'EXB_OBS_IMPL': 'persistent'}),
])
def test_update_with_qc_matches_reference(kw, loc, threshold, env, monkeypatch):
    """EnSRF(..., outlier_threshold=...) against the reference: the rejected set exactly, the state at
    test_gpu_parity's tolerances, the per-ob diagnostics, and the caller's assimilate_this left alone."""
    EnsembleState, Observation, EnSRF = _api()
    case = _with_gross_errors(make_case(**kw), seed=kw['seed'])
    rej, _, ref_post, ref_obs = reference_analysis(case, threshold, loc=loc)
    assert rej.sum() >= 3
    state, obs = build_objects(case, EnsembleState, Observation)
    _patch(monkeypatch, env)
    post, _ = EnSRF(state, obs, verbose=False, loc=loc, outlier_threshold=threshold).update()
    flags = np.array([o.assimilate_this for o in obs])
    np.testing.assert_array_equal(flags, case.ob_assimilate)
    got_rej = flags & ~np.array([o.assimilated for o in obs])
    np.testing.assert_array_equal(got_rej, rej)
    np.testing.assert_array_equal([o.assimilated for o in obs], [o.assimilated for o in ref_obs])
    _check_post(post.to_vect(), ref_post, case.to_vect())
    for attr in ('prior_mean', 'prior_var', 'post_mean', 'post_var'):
        np.testing.assert_allclose(_diag(obs, attr), _diag(ref_obs, attr), rtol=1e-9, equal_nan=True, err_msg=attr)


@pytest.mark.gpu
def test_fp32_with_qc():
    """float32 storage: the rejected set exactly, the state at test_fp32_tolerance's tolerance.  At 130 members the
    state update is the vector kernel, with float32 arithmetic."""
    EnsembleState, Observation, EnSRF = _api()
    for nmem in (50, 130):
        case = _with_gross_errors(make_case(ny=46, nx=90, nmem=nmem, nvars=2, ntimes=1, nobs=300, cutoff_km=2500.0,
                                            seed=23), seed=23)
        rej, _, ref_post, _ = reference_analysis(case, 3.0, margin=1e-3)
        assert rej.sum() >= 5
        state, obs = build_objects(case, EnsembleState, Observation)
        post32, _ = EnSRF(state, obs, verbose=False, loc='GC', dtype='f32', outlier_threshold=3.0).update()
        np.testing.assert_array_equal(~np.array([o.assimilated for o in obs]) & case.ob_assimilate, rej)
        p32 = post32.to_vect()
        m32, mref = p32.mean(axis=1), ref_post.mean(axis=1)
        assert np.abs(m32 - mref).max() <= 1e-5 * np.abs(mref).max(), nmem
        spread = (ref_post - mref[:, None]).std()
        assert np.abs((p32 - m32[:, None]) - (ref_post - mref[:, None])).max() <= 1e-3 * spread, nmem


@pytest.mark.gpu
def test_unreachable_threshold_is_bit_identical(monkeypatch):
    """A threshold no ob reaches gives, bit for bit, the analysis and diagnostics of outlier_threshold=None."""
    EnsembleState, Observation, EnSRF = _api()
    case = _with_gross_errors(make_case(ny=46, nx=90, nmem=50, nvars=2, ntimes=1, nobs=300, cutoff_km=2500.0, seed=311,
                                        frac_skip=0.05), seed=311)
    outs = {}
    for env in ({}, {'EXB_OBS_IMPL': 'persistent'}):
        for t in (None, 1e6, {'var0': 1e6, 'var1': 1e6}):
            state, obs = build_objects(case, EnsembleState, Observation)
            with monkeypatch.context() as m:
                _patch(m, env)
                post, _ = EnSRF(state, obs, verbose=False, loc='GC', outlier_threshold=t).update()
            outs[(str(env), str(t))] = (post.to_vect(), {a: _diag(obs, a) for a in ('prior_mean', 'prior_var', 'post_mean',
                                                                                      'post_var', 'assimilated')})
    for env in ({}, {'EXB_OBS_IMPL': 'persistent'}):
        ref = outs[(str(env), 'None')]
        assert ref[1]['assimilated'].sum() == case.ob_assimilate.sum()
        for t in (1e6, {'var0': 1e6, 'var1': 1e6}):
            got = outs[(str(env), str(t))]
            np.testing.assert_array_equal(got[0], ref[0])
            for a in ref[1]:
                np.testing.assert_array_equal(got[1][a], ref[1][a], err_msg=a)


# ---------------------------------------------------------------------------------------------------------------
# GPU: engine paths
# ---------------------------------------------------------------------------------------------------------------
def _engine_inputs(case, threshold=np.zeros(0)):
    import torch
    from efa_xray_b200 import engine
    dev = torch.device('cuda', 0)
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    obs = engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                           halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                           row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                           tw0=wlo, tw1=whi, threshold=threshold)
    return dev, nt * len(case.varnames), engine.GridTables(case.lat2d, case.lon2d, dev), obs


def _device_analysis(case, obs, **kw):
    import torch
    from efa_xray_b200 import engine
    dev, nlev, grid, _ = _engine_inputs(case)
    X = torch.as_tensor(case.to_vect()).to(dev)
    res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, **kw)
    return X.cpu().numpy(), res


def _rejected(obs, res):
    return obs.assimilate.astype(bool) & ~res.assimilated


@pytest.mark.gpu
@pytest.mark.parametrize('env', [{}, {'EXB_OBS_IMPL': 'persistent'}, {'FUSED_MAX_NENS': 0}])
def test_qc_equals_run_with_rejected_obs_flagged_off(env, monkeypatch):
    """The QC analysis against the analysis without QC and with exactly its rejected obs flagged off: obs-space
    diagnostics bit for bit, the state within the parity tolerance (the sweep batches its obs differently)."""
    case = _with_gross_errors(make_case(ny=46, nx=90, nmem=50, nvars=2, ntimes=1, nobs=600, cutoff_km=2500.0, seed=321,
                                        frac_skip=0.05), seed=321)
    _, _, _, obs = _engine_inputs(case, threshold=np.full(case.nobs, 3.0))
    _patch(monkeypatch, env)
    X, res = _device_analysis(case, obs)
    rej = _rejected(obs, res)
    assert rej.sum() >= 20
    off = dataclasses.replace(obs, assimilate=(obs.assimilate.astype(bool) & ~rej).astype(np.uint8), threshold=np.zeros(0))
    X0, res0 = _device_analysis(case, off)
    for a in ('prior_mean', 'prior_var', 'post_mean', 'post_var', 'assimilated'):
        np.testing.assert_array_equal(getattr(res, a), getattr(res0, a), err_msg=a)
    _check_post(X, X0, case.to_vect())


@pytest.mark.gpu
def test_host_band_pipeline_matches_device_analysis_with_qc():
    """engine.analysis_host with a pinned buffer (several bands) against engine.analysis_device, both with QC."""
    import torch
    from efa_xray_b200 import engine
    case = _with_gross_errors(make_case(ny=361, nx=720, nmem=20, nvars=2, ntimes=1, nobs=800, cutoff_km=2500.0,
                                        seed=331), seed=331)
    dev, nlev, grid, obs = _engine_inputs(case, threshold=np.full(case.nobs, 3.0))
    assert len(engine.sweep_band_schedule(nlev, case.lat2d.shape[0], case.lat2d.shape[1])) >= 3
    ref, rres = _device_analysis(case, obs)
    assert _rejected(obs, rres).sum() >= 20
    prior = case.to_vect()
    host = torch.from_numpy(prior.copy()).pin_memory()
    out = torch.empty_like(host).pin_memory()
    res = engine.analysis_host(host, nlev, None, None, obs, engine.LOC_GC, device=dev, grid=grid, out=out)
    np.testing.assert_array_equal(res.assimilated, rres.assimilated)
    np.testing.assert_array_equal(res.prior_var, rres.prior_var)
    assert np.abs(out.numpy() - ref).max() <= 1e-9 * np.abs(ref - prior).max()
    np.testing.assert_array_equal(host.numpy(), prior)


@pytest.mark.gpu
def test_sharded_logical_ranks_match_unsharded_with_qc():
    """2, 4 and 8 logical latitude-band shards (engine.analysis_device(band=...)) reach the same rejected set and
    the unsharded analysis."""
    import torch
    from efa_xray_b200 import engine, sharding
    case = _with_gross_errors(make_case(ny=61, nx=120, nmem=50, nvars=2, ntimes=2, nobs=3000, cutoff_km=2500.0,
                                        seed=341, offtime=True), seed=341)
    dev, nlev, grid, obs = _engine_inputs(case, threshold=np.full(case.nobs, 3.0))
    ny, nx = case.lat2d.shape
    prior = case.to_vect()
    ref, rres = _device_analysis(case, obs)
    assert _rejected(obs, rres).sum() >= 100
    inc = np.abs(ref - prior).max()
    Xfull = torch.as_tensor(prior).to(dev)
    nens = Xfull.shape[1]
    work = sharding.estimate_row_work(case.lat2d, case.lon2d, obs.lat, obs.lon, 2.0 * obs.halfwidth, obs.assimilate)
    for n in (2, 4, 8):
        bands = sharding.partition_bands(work, n)
        shards = [sharding.band_view(Xfull, nlev, ny, nx, a, b).contiguous().reshape(-1, nens) for a, b in bands]
        parts = [engine.ob_priors(Xs, grid, obs, 'f64', nlev=nlev, band=bd)[0] for Xs, bd in zip(shards, bands)]
        Ysum = torch.stack(parts).sum(dim=0)
        for Xs, bd in zip(shards, bands):
            res = engine.analysis_device(Xs, nlev, grid, obs, engine.LOC_GC, band=bd, Y=Ysum)
            np.testing.assert_array_equal(res.assimilated, rres.assimilated)
        out = torch.empty_like(Xfull)
        for Xs, (a, b) in zip(shards, bands):
            sharding.band_view(out, nlev, ny, nx, a, b).copy_(Xs.view(nlev, b - a, nx, nens))
        assert np.abs(out.cpu().numpy() - ref).max() <= 1e-9 * inc, n


@pytest.mark.gpu
@pytest.mark.parametrize('nobs,nens,cutoff,block', [(3000, 50, 2500.0, 1), (3001, 100, 2500.0, 256)])
def test_distributed_obs_solve_with_qc_is_bit_identical(nobs, nens, cutoff, block):
    """The distributed obs-space solve with thresholds against the replicated one (2 GPUs, torchrun)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs at least 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29573',
           os.path.join(ROOT, 'tests', 'helpers', 'dist_obs_solve_qc_worker.py'), str(nobs), str(nens), str(cutoff),
           str(block)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')]
    assert r.returncode == 0 and lines, r.stderr[-2000:]
    out = json.loads(lines[-1][7:])
    assert out['ok'] and out['block'] == block and out['rejected'][0] == out['rejected'][1] > 0
    assert out['pairs'][0] == out['pairs'][1] and out['nan_pattern_equal']
    assert out['maxdiff_yp'] == 0.0 and out['maxdiff_ym'] == 0.0 and out['maxdiff_rec'] == 0.0


@pytest.mark.gpu
def test_config3_full_size_qc():
    """BASELINE config 3 in full (100 members, 721x1440x3, 1e5 obs) with 1 % gross errors and threshold 3: on the
    first 5 000 obs the rejected set and the obs-space records match the reference (truncating the ob list is exact,
    ob k never depends on later obs), and the analysis is finite."""
    import torch
    from efa_xray_b200 import engine, _lib
    from efa_xray_b200.synth import CONFIGS
    cfg = dict(CONFIGS['config3'])
    case = _with_gross_errors(make_case(cutoff_km=2000.0, seed=0, **cfg), frac=0.01, seed=5)
    dev, nlev, grid, obs = _engine_inputs(case, threshold=np.full(case.nobs, 3.0))
    X = torch.as_tensor(case.to_vect()).to(dev)
    Yp, _ = engine.ob_priors(X, grid, obs, 'f64')
    Ym = torch.empty(obs.nobs, dtype=X.dtype, device=dev)
    _lib.call('exb_split_mean_pert_f64', _lib.ptr(Yp), _lib.ptr(Ym), obs.nobs, X.shape[1], _lib.stream_ptr())
    del case
    res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC)
    rej = _rejected(obs, res)
    assert 500 <= rej.sum() <= 5000 and bool(torch.isfinite(X).all())
    n = 5000
    want_rej, want = qc_reference(Ym[:n].cpu().numpy(), Yp[:n].cpu().numpy(), obs.value[:n], obs.error[:n],
                                  obs.halfwidth[:n], obs.lat[:n], obs.lon[:n], obs.assimilate[:n], obs.threshold[:n],
                                  start=rej[:n])
    np.testing.assert_array_equal(rej[:n], want_rej)
    np.testing.assert_allclose(res.prior_mean[:n], want['prior_mean'], rtol=1e-10)
    np.testing.assert_allclose(res.prior_var[:n], want['prior_var'], rtol=1e-9)
    np.testing.assert_allclose(res.post_mean[:n], want['post_mean'], rtol=1e-10, equal_nan=True)
    np.testing.assert_allclose(res.post_var[:n], want['post_var'], rtol=1e-9, equal_nan=True)
