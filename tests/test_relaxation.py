"""Posterior relaxation (RTPS / RTPP, DESIGN.md section 4.6): the numpy reference's properties, argument checks of
the Python API and of the C entry points (no device needed), and on the GPU the kernels, every analysis path
(fused sweep, three-call path, host-buffer band pipeline, latitude-band shards) and BASELINE config 3 against the
reference (tests/relax_reference.py, built on the CPU oracle)."""

import numpy as np
import pytest

import relax_reference as R
from efa_xray_b200.synth import make_case, make_case_1d, build_objects

F64_RTOL = 1e-10          # as test_gpu_parity._check_post
F64_INC_TOL = 1e-9


def _api():
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    from efa_xray_b200.assimilation.ensrf import EnSRF
    return EnsembleState, Observation, EnSRF


def _ensembles(seed, nrows=40, nens=12):
    """(prior, analysis) rows: the analysis has a shifted mean and a reduced spread."""
    rng = np.random.default_rng(seed)
    xb = 280.0 + rng.normal(0.0, 2.0, (nrows, 1)) + rng.normal(0.0, 1.5, (nrows, nens))
    mb = xb.mean(axis=1, keepdims=True)
    xa = mb + 0.3 * rng.normal(size=(nrows, 1)) + (xb - mb) * rng.uniform(0.2, 0.9, (nrows, 1)) \
        + 0.1 * rng.normal(size=(nrows, nens))
    return xb, xa


# ---------------------------------------------------------------------------------------------------------------
# CPU: the reference
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['rtps', 'rtpp'])
def test_reference_alpha_zero_is_identity(kind):
    xb, xa = _ensembles(1)
    np.testing.assert_array_equal(R.relax(xb, xa, kind, np.zeros(len(xa))), xa)


@pytest.mark.parametrize('kind', ['rtps', 'rtpp'])
def test_reference_preserves_the_analysis_mean(kind):
    xb, xa = _ensembles(2)
    out = R.relax(xb, xa, kind, np.random.default_rng(0).uniform(0, 1, len(xa)))
    np.testing.assert_allclose(out.mean(axis=1), xa.mean(axis=1), rtol=1e-14)
    assert np.abs(out - xa).max() > 0.1


def test_reference_rtps_alpha_one_restores_the_prior_spread():
    xb, xa = _ensembles(3)
    out = R.relax(xb, xa, 'rtps', np.ones(len(xa)))
    np.testing.assert_allclose(out.std(axis=1, ddof=1), xb.std(axis=1, ddof=1), rtol=1e-12)


def test_reference_rtpp_alpha_one_restores_the_prior_perturbations():
    xb, xa = _ensembles(4)
    out = R.relax(xb, xa, 'rtpp', np.ones(len(xa)))
    np.testing.assert_allclose(out - xa.mean(axis=1, keepdims=True), xb - xb.mean(axis=1, keepdims=True),
                               rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('kind', ['rtps', 'rtpp'])
def test_reference_leaves_rows_without_spread_or_change(kind):
    xb, xa = _ensembles(5)
    xa[3] = 281.5                    # no analysis spread
    xa[7] = xb[7]                    # row the analysis did not change
    out = R.relax(xb, xa, kind, np.full(len(xa), 0.7))
    np.testing.assert_array_equal(out[[3, 7]], xa[[3, 7]])
    assert (out[[0, 1, 2]] != xa[[0, 1, 2]]).any()


# ---------------------------------------------------------------------------------------------------------------
# CPU: the Python API validates before any device work, and expands alpha per level
# ---------------------------------------------------------------------------------------------------------------
def _small_objects(nvars=3, ntimes=2):
    EnsembleState, Observation, _ = _api()
    case = make_case(ny=19, nx=36, nmem=6, nvars=nvars, ntimes=ntimes, nobs=5, seed=91)
    return build_objects(case, EnsembleState, Observation)


@pytest.mark.parametrize('relaxation', [
    ('rtpx', 0.5), 'rtps', ('rtps',), ('rtps', 0.5, 1), ('rtps', 1.5), ('rtpp', -0.1), ('rtps', float('nan')),
    ('rtps', '0.5'), ('rtps', True), ('rtpp', {'nope': 0.5}), ('rtpp', {'var0': 2.0}), ('rtps', {'var1': None}),
])
def test_invalid_relaxation_raises_value_error(relaxation):
    from efa_xray_b200.assimilation.assimilation import update
    _, _, EnSRF = _api()
    state, obs = _small_objects()
    with pytest.raises(ValueError):
        EnSRF(state, obs, verbose=False, loc='GC', relaxation=relaxation)
    with pytest.raises(ValueError):
        update(state, obs, loc='GC', relaxation=relaxation)


def test_alpha_expands_per_level():
    _, _, EnSRF = _api()
    state, obs = _small_objects(nvars=3, ntimes=2)
    assert EnSRF(state, obs, verbose=False).relaxation is None
    kind, a = EnSRF(state, obs, verbose=False, relaxation=('rtps', 0.25))._relaxation_levels(('rtps', 0.25))
    assert kind == 'rtps'
    np.testing.assert_array_equal(a, np.full(6, 0.25))
    ens = EnSRF(state, obs, verbose=False, relaxation=('rtpp', {'var2': 0.5, 'var0': 1.0}))
    kind, a = ens._relaxation_levels(ens.relaxation)
    assert kind == 'rtpp'
    np.testing.assert_array_equal(a, [1.0, 1.0, 0.0, 0.0, 0.5, 0.5])     # levels var -> time, as the state rows
    # the same expansion as the reference's per-row alphas
    from oracle import ensrf_oracle as O
    case = make_case(ny=19, nx=36, nmem=6, nvars=3, ntimes=2, nobs=5, seed=91)
    rows = R.alpha_rows(O.State.from_case(case), {'var2': 0.5, 'var0': 1.0})
    np.testing.assert_array_equal(rows, np.repeat(a, 19 * 36))


def test_c_entry_argument_errors_return_status(lib):
    import ctypes as C
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p)
    assert lib.exb_row_spread_f64(None, 1, 4, 0, 4, 4, p, None) == -1
    assert b'exb_row_spread' in lib.exb_last_error()
    assert lib.exb_row_spread_f32(p, 1, 4, 0, 4, 4, None, None) == -1
    assert lib.exb_row_spread_f64(p, 1, 4, 0, 4, 1, p, None) == -1            # nens < 2
    assert b'nens >= 2' in lib.exb_last_error()
    assert lib.exb_row_spread_f64(p, 1, 4, 0, 4, 300, p, None) == -3          # nens > EXB_MAX_NENS
    for args in ((0, 4, 0, 4), (1, 4, 2, 2), (1, 4, 3, 2), (1, 4, -1, 2), (1, 4, 0, 5), (1, 0, 0, 0)):
        assert lib.exb_relax_rtps_f64(p, p, p, *args, 4, None) == -1, args
        assert lib.exb_relax_rtpp_f32(p, p, p, *args, 4, None) == -1, args
    assert lib.exb_relax_rtps_f32(p, None, p, 1, 4, 0, 4, 4, None) == -1
    assert lib.exb_relax_rtps_f64(p, p, None, 1, 4, 0, 4, 4, None) == -1
    assert lib.exb_relax_rtpp_f64(p, None, p, 1, 4, 0, 4, 4, None) == -1
    assert lib.exb_relax_rtpp_f64(None, p, p, 1, 4, 0, 4, 4, None) == -1
    assert b'exb_relax_rtpp' in lib.exb_last_error()


# ---------------------------------------------------------------------------------------------------------------
# GPU: the C entry points against numpy
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('nens', [2, 7, 32, 33, 100, 130])
@pytest.mark.parametrize('sfx', ['f64', 'f32'])
def test_kernels_match_numpy(nens, sfx):
    import torch
    from efa_xray_b200 import _lib
    dev = torch.device('cuda', 0)
    ndt = {'f64': np.float64, 'f32': np.float32}[sfx]
    nlev, npts, pa, pb = 3, 50, 7, 41
    xb, xa = _ensembles(100 + nens, nrows=nlev * npts, nens=nens)
    xb, xa = xb.astype(ndt), xa.astype(ndt)
    xa[[10, 60]] = xa[[10, 60], :1]                      # no analysis spread
    xa[[20, 120]] = xb[[20, 120]]                        # rows the analysis did not change
    alpha = np.array([0.35, 0.0, 1.0])
    rows = np.arange(nlev * npts)
    inside = ((rows % npts) >= pa) & ((rows % npts) < pb)
    a_rows = np.repeat(alpha, npts)
    d_alpha = torch.as_tensor(alpha).to(dev)
    Xb, Xa = torch.as_tensor(xb).to(dev), torch.as_tensor(xa).to(dev)
    # sigma per row, only inside the range
    sig = torch.full((nlev * npts,), float('nan'), dtype=torch.float64, device=dev)
    _lib.call('exb_row_spread_' + sfx, _lib.ptr(Xb), nlev, npts, pa, pb, nens, _lib.ptr(sig), _lib.stream_ptr())
    s = sig.cpu().numpy()
    np.testing.assert_allclose(s[inside], xb[inside].astype(np.float64).std(axis=1, ddof=1), rtol=1e-13)
    assert np.isnan(s[~inside]).all()
    for kind in ('rtps', 'rtpp'):
        X = Xa.clone()
        prior = sig if kind == 'rtps' else Xb
        _lib.call('exb_relax_%s_%s' % (kind, sfx), _lib.ptr(X), _lib.ptr(prior), _lib.ptr(d_alpha), nlev, npts, pa, pb,
                  nens, _lib.stream_ptr())
        got = X.cpu().numpy()
        want = R.relax(xb.astype(np.float64), xa.astype(np.float64), kind, a_rows)
        np.testing.assert_array_equal(got[~inside], xa[~inside])                      # outside the range
        np.testing.assert_array_equal(got[[10, 20, 60, 120]], xa[[10, 20, 60, 120]])   # no spread / unchanged
        np.testing.assert_array_equal(got[a_rows == 0.0], xa[a_rows == 0.0])           # alpha = 0 level
        if sfx == 'f64':
            np.testing.assert_allclose(got[inside], want[inside], rtol=1e-13)
        else:                                            # float64 arithmetic, one rounding on write
            np.testing.assert_allclose(got[inside], want[inside].astype(np.float32), rtol=2e-7)
        assert (got[inside & (a_rows > 0)] != xa[inside & (a_rows > 0)]).any()


@pytest.mark.gpu
def test_kernels_argument_errors_on_device(lib):
    """Range and size checks hold with real device pointers too (nothing is launched)."""
    import torch
    from efa_xray_b200 import _lib
    X = torch.zeros((8, 4), dtype=torch.float64, device='cuda')
    s = torch.zeros(8, dtype=torch.float64, device='cuda')
    assert lib.exb_row_spread_f64(_lib.ptr(X), 2, 4, 0, 5, 4, _lib.ptr(s), _lib.stream_ptr()) == -1
    assert lib.exb_relax_rtps_f64(_lib.ptr(X), _lib.ptr(s), _lib.ptr(s), 2, 4, 0, 4, 1, _lib.stream_ptr()) == -1
    assert lib.exb_relax_rtpp_f64(_lib.ptr(X), _lib.ptr(X), _lib.ptr(s), 2, 4, 0, 4, 257, _lib.stream_ptr()) == -3


# ---------------------------------------------------------------------------------------------------------------
# GPU: the analysis through the public API against the reference
# ---------------------------------------------------------------------------------------------------------------
def _check_post(post, ref_post, prior, tol_scale=1.0):
    np.testing.assert_allclose(post, ref_post, rtol=F64_RTOL * tol_scale)
    inc_ref = ref_post - prior
    scale = max(np.abs(inc_ref).max(), 1e-30)
    assert np.abs((post - prior) - inc_ref).max() <= F64_INC_TOL * tol_scale * scale


_C50 = dict(ny=25, nx=48, nmem=50, nvars=2, ntimes=1, nobs=70, cutoff_km=2500.0, seed=201, frac_skip=0.05)
_INFL_X = ('linspace', 1.0, 1.3, 48)


# env: attributes of engine patched for the case; FUSED_MAX_NENS = 0 takes the three-call form
@pytest.mark.gpu
@pytest.mark.parametrize('kw,loc,relaxation,inflation,env', [
    (_C50, 'GC', ('rtps', 0.6), None, {}),
    (_C50, 'GC', ('rtpp', 0.4), None, {}),
    (_C50, 'GC', ('rtps', {'var1': 0.9}), None, {}),
    (_C50, 'GC', ('rtpp', {'var0': 0.7, 'var1': 0.2}), None, {}),
    (_C50, 'GC', ('rtps', 0.5), 1.15, {}),
    (_C50, 'GC', ('rtpp', 0.5), {'x': _INFL_X}, {}),
    (_C50, 'GC', ('rtps', {'var0': 0.8}), {'var0': 1.1, 'y': ('linspace', 1.2, 1.0, 25)}, {}),
    (dict(ny=25, nx=48, nmem=7, nvars=1, ntimes=1, nobs=60, cutoff_km=1500.0, seed=202), 'GC', ('rtps', 0.9), None, {}),
    (dict(ny=25, nx=48, nmem=100, nvars=2, ntimes=1, nobs=60, cutoff_km=3000.0, seed=203), 'GC', ('rtpp', 0.8), None, {}),
    (dict(ny=19, nx=36, nmem=130, nvars=1, ntimes=1, nobs=40, cutoff_km=4000.0, seed=204), 'GC', ('rtps', 0.7), None, {}),
    (dict(ny=19, nx=36, nmem=130, nvars=1, ntimes=1, nobs=40, cutoff_km=4000.0, seed=204), 'GC', ('rtpp', 0.7), None, {}),
    (_C50, 'GC', ('rtps', 0.6), None, {'FUSED_MAX_NENS': 0}),
    (_C50, 'GC', ('rtpp', 0.4), 1.1, {'FUSED_MAX_NENS': 0}),
    (dict(ny=31, nx=60, nmem=24, nvars=2, ntimes=3, nobs=80, cutoff_km=2000.0, seed=205, offtime=True, frac_skip=0.05),
     'GC', ('rtps', {'var1': 0.5}), None, {}),
    (dict(ny=25, nx=48, nmem=20, nvars=2, ntimes=1, nobs=60, seed=206), False, ('rtps', 0.75), None, {}),
    (dict(ny=25, nx=48, nmem=20, nvars=2, ntimes=1, nobs=60, seed=206), False, ('rtpp', 0.75), None, {}),
    (dict(one_d=True, npts=24, nmem=8, nvars=2, ntimes=1, nobs=30, cutoff_km=4000.0, seed=207), 'GC', ('rtps', 0.8),
     None, {}),
    (dict(one_d=True, npts=24, nmem=8, nvars=2, ntimes=1, nobs=30, cutoff_km=4000.0, seed=207), 'GC', ('rtpp', 0.8),
     None, {}),
])
def test_update_with_relaxation_matches_reference(kw, loc, relaxation, inflation, env, monkeypatch):
    from conftest import decode_inflation
    from oracle import ensrf_oracle as O
    from efa_xray_b200 import engine
    EnsembleState, Observation, EnSRF = _api()
    kw = dict(kw)
    case = make_case_1d(**{k: v for k, v in kw.items() if k != 'one_d'}) if kw.pop('one_d', False) else make_case(**kw)
    inflation = decode_inflation(inflation)
    # the reference runs first: the device path inflates the caller's state, whose arrays are the case's, in place
    ref_post, ref_obs = R.ensrf_update(O.State.from_case(case), O.obs_from_case(case), loc=loc, inflation=inflation,
                                       relaxation=relaxation)
    prior = O.inflate_state(O.State.from_case(case), inflation).to_vect() if inflation is not None else case.to_vect()
    unrelaxed, _ = O.ensrf_update(O.State.from_case(case), O.obs_from_case(case), loc=loc, inflation=inflation)
    assert np.abs(ref_post.to_vect() - unrelaxed.to_vect()).max() > 1e-6       # the relaxation does something
    state, obs = build_objects(case, EnsembleState, Observation)
    for name, value in env.items():
        monkeypatch.setattr(engine, name, value)
    post_state, _ = EnSRF(state, obs, verbose=False, loc=loc, inflation=inflation, relaxation=relaxation).update()
    _check_post(post_state.to_vect(), ref_post.to_vect(), prior)
    # the per-ob diagnostics are those of the serial loop
    for attr in ('prior_mean', 'prior_var', 'post_mean', 'post_var'):
        got = np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr)) for o in obs])
        want = np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr)) for o in ref_obs])
        np.testing.assert_allclose(got, want, rtol=1e-9, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize('relaxation', [('rtps', 0.7), ('rtpp', {'var0': 0.6, 'var1': 0.3})])
def test_fp32_with_relaxation(relaxation):
    """float32 storage at test_fp32_tolerance's tolerance against the float64 reference."""
    from oracle import ensrf_oracle as O
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=46, nx=90, nmem=50, nvars=2, ntimes=1, nobs=300, cutoff_km=2500.0, seed=23)
    state, obs = build_objects(case, EnsembleState, Observation)
    post32, _ = EnSRF(state, obs, verbose=False, loc='GC', dtype='f32', relaxation=relaxation).update()
    ref_post, _ = R.ensrf_update(O.State.from_case(case), O.obs_from_case(case), loc='GC', relaxation=relaxation)
    ref_post = ref_post.to_vect()
    p32 = post32.to_vect()
    m32, mref = p32.mean(axis=1), ref_post.mean(axis=1)
    assert np.abs(m32 - mref).max() <= 1e-5 * np.abs(mref).max()
    spread = (ref_post - mref[:, None]).std()
    assert np.abs((p32 - m32[:, None]) - (ref_post - mref[:, None])).max() <= 1e-3 * spread


# ---------------------------------------------------------------------------------------------------------------
# GPU: engine paths
# ---------------------------------------------------------------------------------------------------------------
def _engine_inputs(case):
    import torch
    from efa_xray_b200 import engine
    dev = torch.device('cuda', 0)
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    obs = engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                           halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                           row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                           tw0=wlo, tw1=whi)
    return dev, nt * len(case.varnames), engine.GridTables(case.lat2d, case.lon2d, dev), obs


def _device_analysis(case, relaxation, **kw):
    import torch
    from efa_xray_b200 import engine
    dev, nlev, grid, obs = _engine_inputs(case)
    X = torch.as_tensor(case.to_vect()).to(dev)
    res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, relaxation=relaxation, **kw)
    return X.cpu().numpy(), res


@pytest.mark.gpu
def test_zero_alpha_and_unreached_rows_are_bit_identical():
    """('rtps', 0) is bit for bit the analysis without relaxation (and launches nothing); with the fused sweep and
    relaxation on, the rows no ob reaches come back bit for bit as the prior."""
    from efa_xray_b200 import _lib
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=46, nx=90, nmem=50, nvars=2, ntimes=1, nobs=25, cutoff_km=1200.0, seed=211)
    prior = case.to_vect()
    outs = {}
    for relaxation in (None, ('rtps', 0.0), ('rtpp', {'var0': 0.0})):
        state, obs = build_objects(case, EnsembleState, Observation)
        n0 = _lib.launch_count()
        post, _ = EnSRF(state, obs, verbose=False, loc='GC', relaxation=relaxation).update()
        outs[str(relaxation)] = (post.to_vect(), _lib.launch_count() - n0)
    ref, nlaunch = outs['None']
    for k, (v, n) in outs.items():
        np.testing.assert_array_equal(v, ref, err_msg=k)
        assert n == nlaunch, k
    nlev = 2
    unreached = (ref == prior).all(axis=1)
    assert 0.2 < unreached.mean() < 0.95
    for relaxation in (('rtps', np.full(nlev, 0.8)), ('rtpp', np.full(nlev, 0.8))):
        X, res = _device_analysis(case, relaxation)
        assert 'relax' in res.ms and res.ms['relax'] > 0
        np.testing.assert_array_equal(X[unreached], prior[unreached])
        assert (X[~unreached] != ref[~unreached]).any()
    X, res = _device_analysis(case, None)
    assert 'relax' not in res.ms


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['rtps', 'rtpp'])
def test_host_band_pipeline_matches_device_analysis(kind):
    """engine.analysis_host with a pinned buffer (several bands, each relaxed between its sweep and its download)
    against engine.analysis_device."""
    import torch
    from efa_xray_b200 import engine
    case = make_case(ny=361, nx=720, nmem=20, nvars=2, ntimes=1, nobs=800, cutoff_km=2500.0, seed=221)
    dev, nlev, grid, obs = _engine_inputs(case)
    ny = case.lat2d.shape[0]
    assert len(engine.sweep_band_schedule(nlev, ny, case.lat2d.shape[1])) >= 3
    relaxation = (kind, np.array([0.8, 0.4]))
    ref, _ = _device_analysis(case, relaxation)
    unrelaxed, _ = _device_analysis(case, None)
    prior = case.to_vect()
    host = torch.from_numpy(prior.copy()).pin_memory()
    out = torch.empty_like(host).pin_memory()
    res = engine.analysis_host(host, nlev, None, None, obs, engine.LOC_GC, device=dev, grid=grid, out=out,
                               relaxation=relaxation)
    got = out.numpy()
    inc = np.abs(ref - prior).max()
    assert np.abs(got - ref).max() <= 1e-9 * inc
    assert np.abs(ref - unrelaxed).max() > 1e-3 * inc
    assert 'relax' in res.ms
    np.testing.assert_array_equal(host.numpy(), prior)


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['rtps', 'rtpp'])
def test_sharded_logical_ranks_match_unsharded_with_relaxation(kind):
    """2, 4 and 8 logical latitude-band shards (engine.analysis_device(band=...)), each relaxing its own rows, against
    the unsharded relaxed analysis."""
    import torch
    from efa_xray_b200 import engine, sharding
    case = make_case(ny=61, nx=120, nmem=50, nvars=2, ntimes=2, nobs=3000, cutoff_km=2500.0, seed=231, offtime=True)
    dev, nlev, grid, obs = _engine_inputs(case)
    ny, nx = case.lat2d.shape
    relaxation = (kind, np.array([0.9, 0.6, 0.3, 0.0]))
    prior = case.to_vect()
    ref, _ = _device_analysis(case, relaxation)
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
            engine.analysis_device(Xs, nlev, grid, obs, engine.LOC_GC, band=bd, Y=Ysum, relaxation=relaxation)
        out = torch.empty_like(Xfull)
        for Xs, (a, b) in zip(shards, bands):
            sharding.band_view(out, nlev, ny, nx, a, b).copy_(Xs.view(nlev, b - a, nx, nens))
        assert np.abs(out.cpu().numpy() - ref).max() <= 1e-9 * inc, n


@pytest.mark.gpu
def test_config3_full_size_relaxation():
    """BASELINE config 3 in full (100 members, 721x1440x3, 1e5 obs): the analysis without relaxation and with each
    kind; on 2000 sampled rows the relaxed analysis is the reference's relaxation of the unrelaxed one, and the
    analysis mean does not move."""
    import torch
    from efa_xray_b200 import engine
    from efa_xray_b200.synth import CONFIGS
    cfg = dict(CONFIGS['config3'])
    case = make_case(cutoff_km=2000.0, seed=0, **cfg)
    dev, nlev, grid, obs = _engine_inputs(case)
    prior_h = case.to_vect()
    prior = torch.as_tensor(prior_h).to(dev)
    del case
    rng = np.random.default_rng(5)
    rows = np.sort(rng.choice(prior.shape[0], 2000, replace=False))
    rows_d = torch.as_tensor(rows, device=dev)
    Xu = prior.clone()
    engine.analysis_device(Xu, nlev, grid, obs, engine.LOC_GC)
    mean_u = Xu.mean(dim=1)
    scale = float(mean_u.abs().max())
    for kind, alpha in (('rtps', np.array([0.9, 0.5, 0.7])), ('rtpp', np.array([0.5, 0.75, 0.25]))):
        X = prior.clone()
        res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, relaxation=(kind, alpha))
        assert res.assimilated.all() and res.ms['relax'] > 0
        want = R.relax(prior_h[rows], Xu[rows_d].cpu().numpy(), kind, np.repeat(alpha, prior.shape[0] // nlev)[rows])
        np.testing.assert_allclose(X[rows_d].cpu().numpy(), want, rtol=1e-12)
        assert float((X.mean(dim=1) - mean_u).abs().max()) <= 1e-12 * scale
        assert float((X[rows_d] - Xu[rows_d]).abs().max()) > 1e-3
        del X
