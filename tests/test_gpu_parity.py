"""GPU parity: the CUDA path, called through the reference-shaped Python API and the C ABI, against
(1) golden vectors from the unmodified reference and (2) the CPU oracle on seeded synthetic cases.

Tolerances: the north star asks for 1e-5 relative in fp64; the asserts below are far tighter (the CUDA
path only differs from numpy in summation order and 1-ulp libm differences).  fp32: analysis mean within
1e-5 of the field magnitude, perturbations within 1e-3 of the ensemble spread.
"""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden, golden_case
from efa_xray_b200.synth import make_case, build_objects

pytestmark = pytest.mark.gpu

F64_RTOL = 1e-10          # on full fields (|x| ~ 288)
F64_INC_TOL = 1e-9        # on the analysis increment, relative to the largest increment


def _api():
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    from efa_xray_b200.assimilation.ensrf import EnSRF
    return EnsembleState, Observation, EnSRF


def _diag(obs, attr):
    return np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr)) for o in obs])


def _check_post(post, ref_post, prior, tol_scale=1.0):
    np.testing.assert_allclose(post, ref_post, rtol=F64_RTOL * tol_scale)
    inc_ref = ref_post - prior
    scale = max(np.abs(inc_ref).max(), 1e-30)
    assert np.abs((post - prior) - inc_ref).max() <= F64_INC_TOL * tol_scale * scale


@pytest.mark.parametrize('name', GOLDEN_CASES)
def test_update_matches_reference_golden(name):
    EnsembleState, Observation, EnSRF = _api()
    g, p = load_golden(name)
    case = golden_case(p)
    state, obs = build_objects(case, EnsembleState, Observation)
    prior = state.to_vect().copy()
    loc = p['loc'] if p['loc'] else False
    post_state, post_obs = EnSRF(state, obs, inflation=p['inflation'], verbose=False, loc=loc).update()
    assert post_obs is obs and post_state is not state
    if p['inflation'] is None:
        np.testing.assert_array_equal(state.to_vect(), prior)          # prior untouched
    # the caller's state after the call, as the reference leaves it: inflated in place by a float / per-variable
    # factors, untouched by per-dimension arrays (assimilation.py:65, :96, :113)
    after = state.to_vect()
    np.testing.assert_allclose([after.sum(), np.abs(after).sum()], g['prior_after_checksum'], rtol=1e-13)
    _check_post(post_state.to_vect(), g['post'], state.to_vect())
    for attr in ('prior_mean', 'prior_var', 'post_mean', 'post_var'):
        np.testing.assert_allclose(_diag(obs, attr), g[attr], rtol=1e-9, equal_nan=True)
    assert np.array_equal([o.assimilated for o in obs], g['assimilated'])


@pytest.mark.parametrize('name', ['gc_small', 'gc_multivar_offtime', 'gc_4deg'])
def test_forward_operator_matches_reference_golden(name):
    EnsembleState, Observation, _ = _api()
    g, p = load_golden(name)
    case = golden_case(p)
    state, obs = build_objects(case, EnsembleState, Observation)
    for k in (0, 1, len(obs) // 2, len(obs) - 1):
        ye = obs[k].estimate(state)
        np.testing.assert_allclose(ye, g['ye'][k], rtol=1e-12)
        cy, cx = state.nearest_points(obs[k].lat, obs[k].lon, npt=4)
        assert set(zip(cy.tolist(), cx.tolist())) == set(map(tuple, g['nearest'][k].T.tolist()))
    from efa_xray_b200.assimilation.assimilation import Assimilation
    means, perts = Assimilation(state, obs).compute_ob_priors()
    np.testing.assert_allclose(means, g['ye'].mean(axis=1), rtol=1e-12)
    np.testing.assert_allclose(perts, g['ye'] - g['ye'].mean(axis=1, keepdims=True), rtol=1e-9, atol=1e-11)
    if p['loc'] == 'GC':
        np.testing.assert_allclose(obs[0].localize(state), g['loc_state0'], rtol=1e-10, atol=1e-13)
        np.testing.assert_allclose(obs[0].localize(obs), g['loc_obs0'], rtol=1e-10, atol=1e-13)


def test_free_functions_match_reference_golden():
    import os
    from conftest import GOLDEN
    from efa_xray_b200.observation.observation import gaspari_cohn, haversine
    f = np.load(os.path.join(GOLDEN, 'functions.npz'))
    np.testing.assert_allclose(gaspari_cohn(f['gc_d'], 1000.0), f['gc_w'], rtol=1e-13, atol=1e-14)   # cancels to ~1e-15 near r=2
    np.testing.assert_allclose(gaspari_cohn(f['gc_d'], -1000.0), f['gc_w_neg'], rtol=1e-13, atol=1e-14)
    hv = np.array([haversine((q[0], q[1]), (q[2], q[3])) for q in f['hv_pairs']])
    np.testing.assert_allclose(hv, f['hv_km'], rtol=1e-13, atol=1e-9)


def test_reference_failure_modes():
    import datetime as dt
    import efa_xray_b200
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=19, nx=36, nmem=4, nobs=2, seed=9)
    state, obs = build_objects(case, EnsembleState, Observation)
    obs[0].lat, obs[0].lon = 10.0, 20.0          # exactly on a grid point: the reference raises IndexError
    with pytest.raises(IndexError):
        obs[0].estimate(state)
    with pytest.raises(IndexError):
        EnSRF(state, obs, verbose=False, loc='GC').update()
    efa_xray_b200.EXACT_MATCH_POLICY = 'nearest'
    try:
        ye = obs[0].estimate(state)
        np.testing.assert_allclose(ye, case.fields['t2m'][0, 10, 2, :], rtol=1e-14)
    finally:
        efa_xray_b200.EXACT_MATCH_POLICY = 'raise'
    obs[0].lat, obs[0].lon = 11.3, 21.7
    obs[0].time = dt.datetime(2031, 1, 1)        # outside the valid times: interpolate returns None
    assert obs[0].estimate(state) is None
    with pytest.raises(AttributeError):
        EnSRF(state, obs, verbose=False, loc='GC').update()
    obs[0].time = obs[1].time
    obs[0].assimilate_this = True
    obs[0].localize_radius = None                # loc='GC' without a radius: TypeError (abs(None))
    with pytest.raises(TypeError):
        EnSRF(state, obs, verbose=False, loc='GC').update()


def _oracle_run(case, loc, inflation=None):
    from oracle import ensrf_oracle as O
    st, obs = O.State.from_case(case), O.obs_from_case(case)
    post, obs = O.ensrf_update(st, obs, loc=loc, inflation=inflation)
    return post.to_vect(), obs


@pytest.mark.parametrize('kw,loc', [
    (dict(ny=37, nx=72, nmem=50, nvars=1, ntimes=1, nobs=150, cutoff_km=2500.0, seed=11, frac_skip=0.05), 'GC'),
    (dict(ny=37, nx=72, nmem=100, nvars=3, ntimes=1, nobs=120, cutoff_km=3000.0, seed=12, mixed_error=True), 'GC'),
    (dict(ny=31, nx=60, nmem=24, nvars=3, ntimes=4, nobs=100, cutoff_km=2000.0, seed=13, offtime=True,
          mixed_radius=True, frac_skip=0.05), 'GC'),
    (dict(ny=25, nx=48, nmem=7, nvars=2, ntimes=1, nobs=70, cutoff_km=1500.0, seed=14), 'GC'),
    (dict(ny=25, nx=48, nmem=33, nvars=1, ntimes=2, nobs=70, cutoff_km=9000.0, seed=15), 'GC'),
    (dict(ny=19, nx=36, nmem=130, nvars=1, ntimes=1, nobs=40, cutoff_km=4000.0, seed=16), 'GC'),
    (dict(ny=19, nx=36, nmem=16, nvars=11, ntimes=1, nobs=40, cutoff_km=4000.0, seed=17), 'GC'),
    (dict(ny=25, nx=48, nmem=20, nvars=2, ntimes=1, nobs=80, seed=18), False),
    (dict(ny=46, nx=90, nmem=50, nvars=1, ntimes=1, nobs=200, cutoff_km=1000.0, seed=19), 'GC'),
    # the largest ensembles of the blocked tensor-core kernel (32 tiles) and of the vector kernel
    (dict(ny=19, nx=36, nmem=255, nvars=1, ntimes=1, nobs=40, cutoff_km=4000.0, seed=20,
         avoid_mirror_ties=True), 'GC'),
    (dict(ny=19, nx=36, nmem=256, nvars=1, ntimes=1, nobs=40, cutoff_km=4000.0, seed=22,
         avoid_mirror_ties=True), 'GC'),
])
def test_update_matches_oracle(kw, loc):
    """Seeded cases against the oracle: ensemble sizes that exercise every kernel variant, many levels,
    off-time obs, mixed radii, no localisation, more obs than one panel (64)."""
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(**kw)
    state, obs = build_objects(case, EnsembleState, Observation)
    prior = state.to_vect().copy()
    post_state, _ = EnSRF(state, obs, verbose=False, loc=loc).update()
    ref_post, ref_obs = _oracle_run(case, loc)
    _check_post(post_state.to_vect(), ref_post, prior)
    for attr in ('prior_mean', 'prior_var', 'post_mean', 'post_var'):
        np.testing.assert_allclose(_diag(obs, attr), _diag(ref_obs, attr), rtol=1e-9, equal_nan=True)
    # perturbation rows keep zero mean (SURVEY.md section 8c)
    pv = post_state.to_vect()
    assert np.abs((pv - pv.mean(axis=1, keepdims=True)).mean(axis=1)).max() < 1e-11


def test_mirror_tie_zone_uses_lowest_flat_index():
    """Next to the 0/180 meridians the reference's pick among exact ties is numpy-sort dependent; this
    package and the oracle both take the lowest flat index."""
    from oracle import ensrf_oracle as O
    EnsembleState, Observation, _ = _api()
    case = make_case(ny=19, nx=36, nmem=4, nobs=1, seed=21)
    state, _ = build_objects(case, EnsembleState, Observation)
    ost = O.State.from_case(case)
    rng = np.random.default_rng(0)
    for lon in list(rng.uniform(-14, 14, 12) % 360) + list(180 + rng.uniform(-14, 14, 12)):
        lat = float(rng.uniform(-70, 70))
        cy, cx = state.nearest_points(lat, float(lon), npt=4)
        oy, ox = O.nearest_points(ost, lat, float(lon), 4)
        assert list(zip(cy.tolist(), cx.tolist())) == list(zip(oy.tolist(), ox.tolist()))


def test_config1_full_size_against_oracle():
    """BASELINE config 1 (181x360, 50 members, 500 obs) in full against the dense oracle."""
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=181, nx=360, nmem=50, nvars=1, ntimes=1, nobs=500, cutoff_km=2000.0, seed=0, frac_skip=0.05)
    state, obs = build_objects(case, EnsembleState, Observation)
    prior = state.to_vect().copy()
    post_state, _ = EnSRF(state, obs, verbose=False, loc='GC').update()
    ref_post, ref_obs = _oracle_run(case, 'GC')
    _check_post(post_state.to_vect(), ref_post, prior)
    np.testing.assert_allclose(_diag(obs, 'post_var'), _diag(ref_obs, 'post_var'), rtol=1e-9, equal_nan=True)


def test_fp32_tolerance():
    """fp32 device arithmetic (scalars stay fp64): mean within 1e-5 of the field magnitude, perturbations
    within 1e-3 of the ensemble spread.  At 50 members the state update is the two-phase sweep (float64 arithmetic
    in registers); at 130 it is the vector kernel, whose row arithmetic is float32 as well."""
    EnsembleState, Observation, EnSRF = _api()
    for nmem in (50, 130):
        case = make_case(ny=46, nx=90, nmem=nmem, nvars=2, ntimes=1, nobs=300, cutoff_km=2500.0, seed=23)
        state, obs = build_objects(case, EnsembleState, Observation)
        post32, _ = EnSRF(state, obs, verbose=False, loc='GC', dtype='f32').update()
        ref_post, _ = _oracle_run(case, 'GC')
        p32 = post32.to_vect()
        m32, mref = p32.mean(axis=1), ref_post.mean(axis=1)
        assert np.abs(m32 - mref).max() <= 1e-5 * np.abs(mref).max(), nmem
        spread = (ref_post - mref[:, None]).std()
        assert np.abs((p32 - m32[:, None]) - (ref_post - mref[:, None])).max() <= 1e-3 * spread, nmem


@pytest.mark.parametrize('pinned', [False, True])
def test_host_buffer_c_abi_entry(pinned):
    """exb_ensrf_host_f64: plain host arrays in, posterior and diagnostics out; pageable and page-locked state
    buffers take different routes through its upload / sweep / download pipeline."""
    import ctypes as C
    import torch
    from efa_xray_b200 import _lib, engine
    g, p = load_golden('gc_multivar_offtime')
    case = golden_case(p)
    X = np.ascontiguousarray(case.to_vect())
    if pinned:
        keep = torch.from_numpy(X).pin_memory()
        X = keep.numpy()
    ny, nx = case.lat2d.shape
    nt, nlev = len(case.times), len(case.varnames) * len(case.times)
    tlo, thi, wlo, whi, outside = engine.time_weights(case.times, case.ob_time)
    assert not outside.any()
    row0 = np.ascontiguousarray((case.ob_var * nt + tlo) * (ny * nx))
    row1 = np.ascontiguousarray((case.ob_var * nt + thi) * (ny * nx))
    diag = np.zeros((4, case.nobs))
    stats = np.zeros(8)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    assim = case.ob_assimilate.astype(np.uint8)
    lat, lon = np.ascontiguousarray(case.lat2d), np.ascontiguousarray(case.lon2d)
    wlo, whi = np.ascontiguousarray(wlo), np.ascontiguousarray(whi)
    _lib.call('exb_ensrf_host_f64', ptr(X), nlev, ny, nx, case.nmem, ptr(lat), ptr(lon), case.nobs,
              ptr(case.ob_value), ptr(case.ob_error), ptr(case.ob_lat), ptr(case.ob_lon), ptr(case.ob_halfwidth),
              ptr(assim), ptr(row0), ptr(row1), ptr(wlo), ptr(whi), 1, 1.0, ptr(diag), ptr(stats))
    _check_post(X, g['post'], case.to_vect())
    np.testing.assert_allclose(diag[0], g['prior_mean'], rtol=1e-9)
    np.testing.assert_allclose(diag[3], g['post_var'], rtol=1e-9, equal_nan=True)
    assert stats[0] > 0 and stats[1] > 0 and stats[2] == 0


def test_rectilinear_search_is_bit_identical_to_brute_force():
    """The separable O(ny+nx) nearest-4 search against the brute-force kernel: same indices in the same
    order and the same weights, including obs next to the 0/180 meridians, the poles and the equator."""
    import torch
    from efa_xray_b200 import engine
    from efa_xray_b200.synth import regular_grid
    rng = np.random.default_rng(5)
    for ny, nx in ((19, 36), (46, 90), (181, 360), (5, 7)):
        lat2d, lon2d = regular_grid(ny, nx)
        grid = engine.GridTables(lat2d, lon2d, torch.device('cuda', 0))
        assert grid.rectilinear
        n = 600
        lat = np.concatenate([np.degrees(np.arcsin(rng.uniform(-1, 1, n))), rng.uniform(-1, 1, 40), rng.uniform(86, 90, 20),
                              rng.uniform(-90, -86, 20)])
        lon = np.concatenate([rng.uniform(0, 360, n), rng.uniform(0, 360, 40), rng.uniform(0, 360, 40)])
        lon[:60] = rng.uniform(-3, 3, 60) % 360
        lon[60:120] = 180 + rng.uniform(-3, 3, 60)
        i_r, w_r, n_r = engine.stencil_search(grid, lat, lon)
        i_g, w_g, n_g = engine.stencil_search(grid, lat, lon, force_general=True)
        assert torch.equal(i_r, i_g)
        assert torch.equal(w_r, w_g)
        assert int(n_r.item()) == int(n_g.item())


def _obs_block(case, dtype='f64'):
    """Device-side inputs of exb_obs_solve_* for a Case: ob priors H.x split into mean + perturbations."""
    import torch
    from efa_xray_b200 import engine
    dev = torch.device('cuda', 0)
    tdt = torch.float64 if dtype == 'f64' else torch.float32
    X = torch.as_tensor(case.to_vect()).to(dev).to(tdt).contiguous()
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    obs = engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                           halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                           row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                           tw0=wlo, tw1=whi)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    Yp, _ = engine.ob_priors(X, grid, obs, dtype)
    Ym = torch.empty(obs.nobs, dtype=tdt, device=dev)
    from efa_xray_b200 import _lib
    _lib.call('exb_split_mean_pert_' + dtype, _lib.ptr(Yp), _lib.ptr(Ym), obs.nobs, X.shape[1], _lib.stream_ptr())
    return obs, Ym, Yp


def _run_obs_solve(obs, Ym, Yp, loc_mode, impl, dtype='f64', budget=None):
    import os
    import torch
    from efa_xray_b200 import engine, _lib
    dev = Yp.device
    obs_dev, geo = engine.upload_obs(obs, dev, loc_mode)
    ym, yp = Ym.clone(), Yp.clone()
    rec = torch.empty((8, obs.nobs), dtype=torch.float64, device=dev)
    counters = torch.zeros(2, dtype=torch.int64, device=dev)
    old = {k: os.environ.get(k) for k in ('EXB_OBS_IMPL', 'EXB_DAG_BUDGET')}
    os.environ['EXB_OBS_IMPL'] = impl
    if budget is not None:
        os.environ['EXB_DAG_BUDGET'] = str(budget)
    try:
        engine.obs_solve(ym, yp, obs_dev, geo, Yp.shape[1], loc_mode, rec, counters, dtype)
        torch.cuda.synchronize()
        _lib.call('exb_obs_solve_async_status')
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return ym.cpu().numpy(), yp.cpu().numpy(), rec.cpu().numpy(), int(counters[0].item())


def _oracle_obs_solve(obs, Ym, Yp, loc_mode):
    """oracle.obs_space_solve (the reference's serial loop on the obs rows, ensrf.py:61-149) on device-side inputs."""
    from oracle import ensrf_oracle as O
    return O.obs_space_solve(Ym.cpu().numpy(), Yp.cpu().numpy(), obs.value, obs.error, obs.halfwidth, obs.lat, obs.lon,
                             obs.assimilate.astype(bool), loc='GC' if loc_mode else None)


def _check_obs_solve(got, want, assim):
    """A device obs-space solve (ym, ye rows, records) against the oracle: ye rows, means and the seven record fields
    at 1e-9 or tighter.  Innovation, c1 and beta only exist for assimilated obs in the oracle."""
    ym, ye, rec = got[:3]
    a = np.asarray(assim, dtype=bool)
    assert np.abs(ye - want['ye']).max() <= 1e-9 * np.abs(want['ye']).max()
    np.testing.assert_allclose(ym, want['prior_mean'], rtol=1e-10)
    np.testing.assert_allclose(rec[0], want['prior_mean'], rtol=1e-10)
    np.testing.assert_allclose(rec[1], want['prior_var'], rtol=1e-9)
    np.testing.assert_allclose(rec[2], want['post_mean'], rtol=1e-10, equal_nan=True)
    np.testing.assert_allclose(rec[3], want['post_var'], rtol=1e-9, equal_nan=True)
    # innovations are differences of O(280 K) numbers: absolute tolerance from the means
    np.testing.assert_allclose(rec[4][a], want['innov'][a], rtol=1e-9, atol=1e-10 * 300.0)
    nens = ye.shape[1]
    np.testing.assert_allclose(rec[5][a], 1.0 / ((nens - 1) * want['kdenom'][a]), rtol=1e-9)
    np.testing.assert_allclose(rec[6][a], want['beta'][a], rtol=1e-9)
    np.testing.assert_array_equal(rec[7], a.astype(np.float64))


@pytest.mark.parametrize('kw,loc_mode', [
    (dict(ny=46, nx=90, nmem=50, nobs=700, cutoff_km=2500.0, seed=31, frac_skip=0.05, mixed_radius=True), 1),
    (dict(ny=46, nx=90, nmem=100, nobs=3000, cutoff_km=800.0, seed=32, mixed_error=True), 1),
    (dict(ny=37, nx=72, nmem=130, nobs=300, cutoff_km=3000.0, seed=33, frac_skip=0.1), 1),
    (dict(ny=37, nx=72, nmem=20, nobs=200, seed=34), 0),
])
def test_obs_solve_variants_match_oracle(kw, loc_mode):
    """The persistent panel kernel and the dependency-driven obs-space solve, the latter also with its predecessor
    lists cut into many row blocks, evolve the closed obs-row subsystem (SURVEY.md section 0) in the reference's
    serial order: records, ye rows and diagnostics match the oracle, and the runs agree with each other, pair counts
    included."""
    import itertools
    case = make_case(**kw)
    obs, Ym, Yp = _obs_block(case)
    want = _oracle_obs_solve(obs, Ym, Yp, loc_mode)
    runs = [_run_obs_solve(obs, Ym, Yp, loc_mode, 'persistent'), _run_obs_solve(obs, Ym, Yp, loc_mode, 'dag'),
            _run_obs_solve(obs, Ym, Yp, loc_mode, 'dag', budget=997)]
    for run in runs:
        _check_obs_solve(run, want, obs.assimilate)
    scale = np.abs(want['ye']).max()
    for (ym, yp, rec, npairs), ref in itertools.combinations(runs, 2):
        assert npairs == ref[3]
        np.testing.assert_allclose(ym, ref[0], rtol=1e-11)
        assert np.abs(yp - ref[1]).max() <= 1e-11 * scale
        np.testing.assert_allclose(rec, ref[2], rtol=1e-9, atol=1e-12, equal_nan=True)


def test_persistent_solve_beyond_256_chunks_per_worker():
    """The persistent solve with more than 256 chunks of 64 obs per trailing worker (nobs = 64 x 260 x SMs; one CTA
    per SM), 8 members, no localisation.  Only the first and the last 512 obs are assimilated.  (1) The pair counter
    counts every later row of every assimilated ob, so every chunk saw every assimilated panel; (2) the assimilated
    obs match the oracle run on them alone, since a skipped ob changes no row; (3) sampled skipped rows, some in chunks
    past slot 256 of their worker, match the oracle on the first 512 obs followed by those rows."""
    import torch
    from oracle import ensrf_oracle as O
    from efa_xray_b200 import engine
    dev = torch.device('cuda', 0)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    nobs, nens, na = 64 * 260 * sms, 8, 512
    rng = np.random.default_rng(91)
    Yp0 = rng.standard_normal((nobs, nens))
    Yp0 -= Yp0.mean(axis=1, keepdims=True)
    Ym0 = 280.0 + rng.standard_normal(nobs)
    assim = np.zeros(nobs, dtype=np.uint8)
    assim[:na] = assim[-na:] = 1
    zeros = np.zeros(nobs, dtype=np.int64)
    obs = engine.ObsArrays(value=Ym0 + rng.standard_normal(nobs), error=rng.uniform(0.5, 2.0, nobs),
                           lat=rng.uniform(-80.0, 80.0, nobs), lon=rng.uniform(0.0, 360.0, nobs),
                           halfwidth=np.full(nobs, 1000.0), assimilate=assim, row0=zeros, row1=zeros,
                           tw0=np.ones(nobs), tw1=np.zeros(nobs))
    ym, ye, rec, npairs = _run_obs_solve(obs, torch.as_tensor(Ym0, device=dev), torch.as_tensor(Yp0, device=dev), 0,
                                         'persistent')
    # (1)
    ks = np.flatnonzero(assim)
    assert npairs == int((nobs - ks).sum())

    def oracle_on(idx):
        return O.obs_space_solve(Ym0[idx], Yp0[idx], obs.value[idx], obs.error[idx], obs.halfwidth[idx], obs.lat[idx],
                                 obs.lon[idx], assim[idx].astype(bool), loc=None)
    # (2)
    _check_obs_solve((ym[ks], ye[ks], rec[:, ks]), oracle_on(ks), assim[ks])
    # (3) chunk p belongs to slot p // (SMs - 1) of its worker
    tail = 64 * 256 * (sms - 1)
    js = np.unique(np.concatenate([rng.integers(na, tail, 31), rng.integers(tail, nobs - na, 31), [na, nobs - na - 1]]))
    want = oracle_on(np.concatenate([np.arange(na), js]))
    scale = np.abs(want['ye'][na:]).max()
    assert np.abs(ye[js] - want['ye'][na:]).max() <= 1e-9 * scale
    np.testing.assert_allclose(rec[0][js], want['prior_mean'][na:], rtol=1e-10)
    np.testing.assert_allclose(rec[1][js], want['prior_var'][na:], rtol=1e-9)


def test_obs_solve_dag_fp32():
    case = make_case(ny=46, nx=90, nmem=50, nobs=500, cutoff_km=2500.0, seed=35)
    obs, Ym, Yp = _obs_block(case, 'f32')
    ref = _run_obs_solve(obs, Ym, Yp, 1, 'persistent', 'f32')
    ym, yp, rec, npairs = _run_obs_solve(obs, Ym, Yp, 1, 'dag', 'f32')
    assert npairs == ref[3]
    np.testing.assert_allclose(ym, ref[0], rtol=1e-5)
    assert np.abs(yp - ref[1]).max() <= 2e-4 * np.abs(ref[1]).max()
    np.testing.assert_allclose(rec[:4], ref[2][:4], rtol=2e-3, equal_nan=True)


def _analysis(case, bands=None):
    """engine.analysis_device on a fresh device copy of the case's state; with `bands` the fused sweep is issued band
    by band (row ranges of the same shard)."""
    import torch
    from efa_xray_b200 import engine
    dev = torch.device('cuda', 0)
    X = torch.as_tensor(case.to_vect()).to(dev).contiguous()
    nlev = len(case.times) * len(case.varnames)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    res = engine.analysis_device(X, nlev, grid, _engine_obs(case), engine.LOC_GC, sweep_bands=bands)
    return X.cpu().numpy(), res


@pytest.mark.parametrize('kw', [
    dict(ny=91, nx=180, nmem=100, nvars=3, ntimes=1, nobs=6000, cutoff_km=1500.0, seed=41, frac_skip=0.05, mixed_radius=True),
    dict(ny=61, nx=120, nmem=50, nvars=2, ntimes=2, nobs=5000, cutoff_km=2500.0, seed=42),
    dict(ny=46, nx=90, nmem=24, nvars=11, ntimes=1, nobs=4500, cutoff_km=3000.0, seed=43),
    dict(ny=46, nx=90, nmem=7, nvars=1, ntimes=1, nobs=300, cutoff_km=3000.0, seed=44),
    # ~2900 candidates per patch: more than one chunk of the two-phase kernel (rows parked between chunks), supports
    # beyond the range of the branch-free weight function
    dict(ny=31, nx=60, nmem=16, nvars=2, ntimes=1, nobs=7000, cutoff_km=9000.0, seed=45, frac_skip=0.02),
])
def test_sweep_variants_agree(kw, monkeypatch):
    """The two-phase sweep, fused with and without a sweep plan, in band-by-band calls and in the three-call form
    (split / exb_state_update / recombine, the same kernel in split mode), applies the same obs in the same order to
    every state row as the fused sweep after the persistent obs-space solve.  A numpy replay of sampled rows from the
    obs-space records checks the default run independently of the sweep kernel."""
    import torch
    from efa_xray_b200 import engine
    case = make_case(**kw)
    prior = case.to_vect()
    with monkeypatch.context() as m:
        m.setenv('EXB_OBS_IMPL', 'persistent')
        ref, res0 = _analysis(case)
    inc = np.abs(ref - prior).max()
    ny, nx = case.lat2d.shape
    runs = {'fused': _analysis(case)}
    with monkeypatch.context() as m:
        m.setattr(engine, 'SweepPlan', lambda *args, **kwargs: None)
        runs['fused_noplan'] = _analysis(case)
    with monkeypatch.context() as m:
        m.setattr(engine, 'FUSED_MAX_NENS', 0)
        runs['split'] = _analysis(case)
    runs['bands'] = _analysis(case, bands=[(0, 7), (7, 30), (30, ny - 1), (ny - 1, ny)])
    for name, (X, res) in runs.items():
        # pairs with a non-zero weight: identical up to the handful of pairs within rounding of the edge of a
        # support (the branch-free weight function and the libm one may round a 1e-16 weight to 0 differently)
        assert abs(res.state_pairs - res0.state_pairs) <= 1e-4 * res0.state_pairs, name
        np.testing.assert_allclose(X, ref, rtol=1e-11, err_msg=name)
        assert np.abs(X - ref).max() <= 1e-9 * inc, name
    obs, Ym, Yp = _obs_block(case)
    _, ye, rec, _ = _run_obs_solve(obs, Ym, Yp, 1, 'dag')
    dev = torch.device('cuda', 0)
    _, geo = engine.upload_obs(obs, dev, 1)
    grid_u = engine.GridTables(case.lat2d, case.lon2d, dev).u.cpu().numpy()
    pts, rows = _sample_rows(np.random.default_rng(4), ny, nx, len(case.times) * len(case.varnames))
    want = _replay_rows(prior[rows], pts, grid_u, ye, rec, geo.cpu().numpy(), 1)
    assert np.abs(runs['fused'][0][rows] - want).max() <= 1e-9 * inc


def test_postprocess_statistics_match_oracle():
    """obs_assimilation_statistics (postprocess/postprocess.py:8-39): batched device H.x of prior and posterior
    against per-ob estimates of the oracle."""
    from oracle import ensrf_oracle as O
    from efa_xray_b200.postprocess.postprocess import obs_assimilation_statistics, COLUMNS
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=37, nx=72, nmem=30, nvars=2, ntimes=3, nobs=60, cutoff_km=3000.0, seed=51, offtime=True, frac_skip=0.1)
    state, obs = build_objects(case, EnsembleState, Observation)
    post, obs = EnSRF(state, obs, verbose=False, loc='GC').update()
    df = obs_assimilation_statistics(state, post, obs)
    assert list(df.columns) == COLUMNS and len(df) == len(obs)
    ost = O.State.from_case(case)
    oobs = O.obs_from_case(case)
    opost, _ = O.ensrf_update(ost, oobs, loc='GC')
    pm = np.array([O.estimate(o, ost).mean() for o in oobs])
    pv = np.array([O.estimate(o, ost).var() for o in oobs])
    qm = np.array([O.estimate(o, opost).mean() for o in oobs])
    qv = np.array([O.estimate(o, opost).var() for o in oobs])
    np.testing.assert_allclose(df['prior mean'].values, pm, rtol=1e-12)
    np.testing.assert_allclose(df['prior variance'].values, pv, rtol=1e-9)
    np.testing.assert_allclose(df['post mean'].values, qm, rtol=1e-10)
    np.testing.assert_allclose(df['post variance'].values, qv, rtol=1e-8)
    assert df['assimilated'].tolist() == [o.assimilated for o in obs]
    assert abs(df['flead'].iloc[0] - (case.ob_time[0] - case.times[0]) / np.timedelta64(3600, 's')) < 1e-9


def _replay_rows(rows_prior, row_pts, grid_u_h, ye, rec, geo, loc_mode):
    """Row-stationary replay in numpy of the state update for a few rows, from the obs-space records the device
    produced: x <- x - beta_k loc_k(row) c1_k (x'.ye_k) ye_k, mean += loc c1 (x'.ye_k) innov_k, k in serial order
    (ensrf.py:95-141).  Independent of the CUDA sweep kernels."""
    R = 6371.0
    out = np.empty_like(rows_prior)
    assim = np.flatnonzero(rec[7] != 0.0)
    ou = geo[0:3, assim]                      # [3, na]
    invhw, amax = geo[3, assim], geo[4, assim]
    for i in range(rows_prior.shape[0]):
        x = rows_prior[i].copy()
        m = x.mean()
        x -= m
        gu = grid_u_h[:, row_pts[i]]
        d = ou - gu[:, None]
        a = 0.25 * (d * d).sum(axis=0)
        if loc_mode == 1:
            cand = np.flatnonzero(a < amax)
            ang = 2.0 * np.arcsin(np.sqrt(np.clip(a[cand], 0.0, 1.0)))
            r = R * ang * invhw[cand]
            w = np.where(r <= 1.0, ((((-0.25 * r + 0.5) * r + 0.625) * r - 5.0 / 3.0) * r * r + 1.0),
                         np.where(r < 2.0, (((((r / 12.0 - 0.5) * r + 0.625) * r + 5.0 / 3.0) * r - 5.0) * r + 4.0
                                             - 2.0 / (3.0 * np.maximum(r, 1e-300))), 0.0))
        else:
            cand = np.arange(assim.size)
            w = np.ones(assim.size)
        for j, k in enumerate(assim[cand]):
            if w[j] == 0.0:
                continue
            dot = x @ ye[k]
            kmat = w[j] * dot * rec[5, k]
            m += kmat * rec[4, k]
            x -= (rec[6, k] * kmat) * ye[k]
        out[i] = x + m
    return out


def _engine_obs(case):
    from efa_xray_b200 import engine
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    return engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                            halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                            row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                            tw0=wlo, tw1=whi)


def _gc_weights(a, invhw, amax):
    """Gaspari-Cohn weights from haversine-a values (numpy restatement of observation.py:117-130)."""
    R = 6371.0
    ang = 2.0 * np.arcsin(np.sqrt(np.clip(a, 0.0, 1.0)))
    r = R * ang * invhw
    w = np.where(r <= 1.0, ((((-0.25 * r + 0.5) * r + 0.625) * r - 5.0 / 3.0) * r * r + 1.0),
                 np.where(r < 2.0, (((((r / 12.0 - 0.5) * r + 0.625) * r + 5.0 / 3.0) * r - 5.0) * r + 4.0
                                     - 2.0 / (3.0 * np.maximum(r, 1e-300))), 0.0))
    return np.where(a < amax, w, 0.0)


def _replay_obs_rows(js, Yp0, ye, rec, geo):
    """Obs-space replay in numpy: row j of the ob-prior perturbations receives the updates of every assimilated
    ob k < j in serial order (ensrf.py:95-141 restricted to the obs rows) and must arrive at ye_j, the row the
    device published for ob j.  Independent of the CUDA solve kernels."""
    out = np.empty((len(js), Yp0.shape[1]))
    for i, j in enumerate(js):
        x = Yp0[j].copy()
        ks = np.flatnonzero(rec[7, :j] != 0.0)
        d = geo[0:3, ks] - geo[0:3, j][:, None]
        w = _gc_weights(0.25 * (d * d).sum(axis=0), geo[3, ks], geo[4, ks])
        for k, wk in zip(ks[w != 0.0], w[w != 0.0]):
            x -= (rec[6, k] * wk * (x @ ye[k]) * rec[5, k]) * ye[k]
        out[i] = x
    return out


def _sample_rows(rng, ny, nx, nlev, n=20):
    pts = np.concatenate([rng.integers(0, ny * nx, n), [0, nx - 1, (ny - 1) * nx, ny * nx - 1, (ny // 2) * nx,
                                                        (ny // 2) * nx + nx - 1, 5 * nx + 7, (ny - 3) * nx + nx // 2]])
    levs = rng.integers(0, nlev, pts.size)
    return pts, levs * (ny * nx) + pts


_CONFIG3 = {}


def _config3():
    """BASELINE config 3 (100 members, 721x1440x3, 1e5 obs, cutoff 2000 km), built once per test session."""
    if not _CONFIG3:
        from efa_xray_b200.synth import CONFIGS
        cfg = dict(CONFIGS['config3'])
        case = make_case(cutoff_km=2000.0, seed=0, **cfg)
        _CONFIG3.update(cfg=cfg, case=case, obs_block=_obs_block(case))
    return _CONFIG3


def test_config3_full_size_properties():
    """BASELINE config 3 in full (100 members, 721x1440x3, 1e5 obs, cutoff 2000 km) through size-independent checks:
    (1) the dependency-driven and the panel obs-space solves agree on all 1e5 records; (2) a numpy replay of the
    serial update from those records reproduces the swept state on sampled rows (poles, equator, date line);
    (3) a numpy replay of sampled obs rows from the records arrives at the ye rows the device published;
    (4) variance can only shrink; (5) rows keep finite values."""
    import torch
    from efa_xray_b200 import engine
    c3 = _config3()
    cfg, case = c3['cfg'], c3['case']
    ny, nx, nens, nlev = cfg['ny'], cfg['nx'], cfg['nmem'], cfg['nvars'] * cfg['ntimes']
    dev = torch.device('cuda', 0)
    prior = case.to_vect()
    X = torch.as_tensor(prior).to(dev)
    obs, Ym, Yp = c3['obs_block']
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC)
    assert res.assimilated.all() and res.state_pairs > 7.0e9 and res.obs_solve == 'single'
    # (1) obs-space solve variants on the full ob set
    a = _run_obs_solve(obs, Ym, Yp, 1, 'dag')
    b = _run_obs_solve(obs, Ym, Yp, 1, 'persistent')
    assert a[3] == b[3] == res.obs_pairs
    assert np.abs(a[1] - b[1]).max() <= 1e-11 * np.abs(b[1]).max()
    np.testing.assert_allclose(a[2], b[2], rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(res.prior_var, a[2][1], rtol=1e-12)
    # (4) every assimilated ob shrinks its own variance; diagnostics are finite
    assert (res.post_var <= res.prior_var * (1 + 1e-12)).all() and np.isfinite(res.post_mean).all()
    # (2) replay sampled state rows from the records
    ym, ye, rec, _ = a
    _, geo = engine.upload_obs(obs, dev, 1)
    geo_h, gu_h = geo.cpu().numpy(), grid.u.cpu().numpy()
    rng = np.random.default_rng(3)
    pts, rows = _sample_rows(rng, ny, nx, nlev)
    got = X[torch.as_tensor(rows, device=dev)].cpu().numpy()
    want = _replay_rows(prior[rows], pts, gu_h, ye, rec, geo_h, 1)
    inc = np.abs(want - prior[rows]).max()
    assert inc > 1e-3
    assert np.abs(got - want).max() <= 1e-9 * inc
    # (3) replay sampled obs rows (late ones have the most predecessors) from the records
    js = np.concatenate([rng.integers(0, obs.nobs, 12), [0, 1, obs.nobs - 1, obs.nobs - 2]])
    want_ye = _replay_obs_rows(js, Yp.cpu().numpy(), ye, rec, geo_h)
    assert np.abs(ye[js] - want_ye).max() <= 1e-9 * np.abs(Yp.cpu().numpy()[js]).max()
    # (5) the whole analysis is finite and its spread did not grow on the sampled rows
    assert bool(torch.isfinite(X).all())
    assert (got.std(axis=1) <= prior[rows].std(axis=1) * (1 + 1e-9)).all()


@pytest.mark.parametrize('nobs,cutoff_km', [(20000, 2000.0), (5000, 5000.0)])
def test_dag_solve_matches_oracle_on_config3_prefix(nobs, cutoff_km):
    """The dependency-driven obs-space solve against the ORACLE (oracle.obs_space_solve, the reference's serial loop
    on the obs rows, ensrf.py:61-149) on the first `nobs` observations of BASELINE config 3: truncating the ob
    list is exact because ob k never depends on later obs.  Records, ye rows and diagnostics at 1e-9.  20 000 obs
    at 2000 km: dependency chain ~1e3; 5 000 obs at 5000 km: every ob sees ~15 % of the earlier ones."""
    c3 = _config3()
    case = c3['case']
    obs_all, Ym, Yp = c3['obs_block']
    import dataclasses
    obs = dataclasses.replace(obs_all, **{f.name: getattr(obs_all, f.name)[:nobs] for f in dataclasses.fields(obs_all)})
    if cutoff_km != 2000.0:
        obs = dataclasses.replace(obs, halfwidth=np.full(nobs, 0.5 * cutoff_km))
    ym, yp = Ym[:nobs].contiguous(), Yp[:nobs].contiguous()
    got = _run_obs_solve(obs, ym, yp, 1, 'dag')
    assert obs.assimilate.all()
    _check_obs_solve(got, _oracle_obs_solve(obs, ym, yp, 1), obs.assimilate)
    assert got[3] > nobs


def _sharded_analysis(case, nshards, Yfull=None):
    """N LOGICAL latitude-band shards run one after the other on one device through engine.analysis_device(band=...),
    exactly as N ranks would (work-balanced bands, offset shard, shard-local stencils, replicated obs-space solve;
    without a process group the partial ob priors are summed here instead of all-reduced)."""
    import torch
    from efa_xray_b200 import engine, sharding
    dev = torch.device('cuda', 0)
    ny, nx = case.lat2d.shape
    nlev = len(case.times) * len(case.varnames)
    obs = _engine_obs(case)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    Xfull = torch.as_tensor(case.to_vect()).to(dev)
    nens = Xfull.shape[1]
    work = sharding.estimate_row_work(case.lat2d, case.lon2d, obs.lat, obs.lon, 2.0 * obs.halfwidth, obs.assimilate)
    bands = sharding.partition_bands(work, nshards)
    shards = [sharding.band_view(Xfull, nlev, ny, nx, a, b).contiguous().reshape(-1, nens) for a, b in bands]
    # H.x as the ranks compute it: every shard sums the stencil points it owns, the partial sums add up
    parts = [engine.ob_priors(Xs, grid, obs, 'f64', nlev=nlev, band=bd)[0] for Xs, bd in zip(shards, bands)]
    Ysum = torch.stack(parts).sum(dim=0)
    results = [engine.analysis_device(Xs, nlev, grid, obs, engine.LOC_GC, band=bd, Y=Ysum) for Xs, bd in zip(shards, bands)]
    out = torch.empty_like(Xfull)
    for Xs, (a, b) in zip(shards, bands):
        sharding.band_view(out, nlev, ny, nx, a, b).copy_(Xs.view(nlev, b - a, nx, nens))
    return out, Ysum, results, bands


@pytest.mark.parametrize('kw', [
    dict(ny=91, nx=180, nmem=100, nvars=3, ntimes=1, nobs=6000, cutoff_km=1500.0, seed=71, frac_skip=0.05, mixed_radius=True),
    dict(ny=61, nx=120, nmem=50, nvars=2, ntimes=2, nobs=3000, cutoff_km=2500.0, seed=72, offtime=True),
])
def test_sharded_logical_ranks_match_unsharded(kw):
    """The latitude-band path (engine.analysis_device(band=...), SURVEY 8e; the reference's intended split is
    assimilation.py:186-202) as 2, 4 and 8 logical shards on one device against the unsharded analysis.
    The obs-space results are band-independent and must be IDENTICAL on every shard; the state agrees to rounding
    (a shard's patches start at its own first row, so a row meets the same obs in the same order but grouped into
    different batches of 8, which changes the last bits only)."""
    import torch
    from efa_xray_b200 import engine
    case = make_case(**kw)
    dev = torch.device('cuda', 0)
    nlev = len(case.times) * len(case.varnames)
    obs = _engine_obs(case)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    prior = case.to_vect()
    Xref = torch.as_tensor(prior).to(dev)
    Yref, _ = engine.ob_priors(Xref, grid, obs, 'f64')
    ref = engine.analysis_device(Xref, nlev, grid, obs, engine.LOC_GC)
    inc = float((Xref - torch.as_tensor(prior).to(dev)).abs().max())
    for n in (2, 4, 8):
        out, Ysum, results, bands = _sharded_analysis(case, n)
        assert len(bands) == n and bands[0][0] == 0 and bands[-1][1] == case.lat2d.shape[0]
        assert float((Ysum - Yref).abs().max()) <= 1e-12 * float(Yref.abs().max())
        for r in results:
            assert r.obs_solve == 'replicated'
            for f in ('prior_mean', 'prior_var', 'post_mean', 'post_var', 'assimilated'):
                np.testing.assert_array_equal(getattr(r, f), getattr(results[0], f))
            np.testing.assert_allclose(r.prior_var, ref.prior_var, rtol=1e-10)
            np.testing.assert_allclose(r.post_mean, ref.post_mean, rtol=1e-10, equal_nan=True)
        assert sum(r.state_pairs for r in results) == pytest.approx(ref.state_pairs, rel=1e-4)
        assert float((out - Xref).abs().max()) <= 1e-9 * inc
        assert bool(torch.isfinite(out).all())


def test_sharded_logical_ranks_config3():
    """Same check at BASELINE config 3 (the configuration the multi-GPU numbers are quoted on), 8 logical shards."""
    import torch
    from efa_xray_b200 import engine
    c3 = _config3()
    case, cfg = c3['case'], c3['cfg']
    dev = torch.device('cuda', 0)
    nlev = cfg['nvars'] * cfg['ntimes']
    obs = _engine_obs(case)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    out, Ysum, results, bands = _sharded_analysis(case, 8)
    prior = torch.as_tensor(case.to_vect()).to(dev)
    Xref = prior.clone()
    ref = engine.analysis_device(Xref, nlev, grid, obs, engine.LOC_GC)
    inc = float((Xref - prior).abs().max())
    del prior
    assert sum(r.state_pairs for r in results) == pytest.approx(ref.state_pairs, rel=1e-5)
    np.testing.assert_allclose(results[3].post_var, ref.post_var, rtol=1e-9)
    diff = float((out - Xref).abs().max())
    assert diff <= 1e-9 * inc, (diff, inc)


def _full_size_replay(cfg, cutoff_km, seed, dtypes=('f64',), n_rows=12):
    """A BASELINE configuration in full through engine.analysis_device, checked by the numpy row replay from the
    device's obs-space records on sampled rows.  Returns {dtype: (sampled analysis rows, result)} + the replay."""
    import torch
    from efa_xray_b200 import engine
    ny, nx, nlev = cfg['ny'], cfg['nx'], cfg['nvars'] * cfg['ntimes']
    case = make_case(cutoff_km=cutoff_km, seed=seed, **cfg)
    dev = torch.device('cuda', 0)
    obs = _engine_obs(case)
    grid = engine.GridTables(case.lat2d, case.lon2d, dev)
    prior = case.to_vect()
    rng = np.random.default_rng(5)
    pts, rows = _sample_rows(rng, ny, nx, nlev, n=n_rows)
    out = {}
    for dt in dtypes:
        X = torch.as_tensor(prior).to(dev)
        if dt == 'f32':
            X = X.to(torch.float32)
        res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC)
        assert bool(torch.isfinite(X).all())
        out[dt] = (X[torch.as_tensor(rows, device=dev)].cpu().numpy().astype(np.float64), res)
        del X
    # records of the float64 obs-space solve for the replay
    X = torch.as_tensor(prior).to(dev)
    Yp, _ = engine.ob_priors(X, grid, obs, 'f64')
    del X
    Ym = torch.empty(obs.nobs, dtype=torch.float64, device=dev)
    from efa_xray_b200 import _lib
    _lib.call('exb_split_mean_pert_f64', _lib.ptr(Yp), _lib.ptr(Ym), obs.nobs, Yp.shape[1], _lib.stream_ptr())
    _, ye, rec, _ = _run_obs_solve(obs, Ym, Yp, 1, 'dag')
    _, geo = engine.upload_obs(obs, dev, 1)
    want = _replay_rows(prior[rows], pts, grid.u.cpu().numpy(), ye, rec, geo.cpu().numpy(), 1)
    return out, want, prior[rows]


def test_config2_full_size_replay():
    """BASELINE config 2 in full: 50 members, 361x720, 3 variables x 4 times (12 levels per patch), 5000 obs."""
    from efa_xray_b200.synth import CONFIGS
    out, want, prior_rows = _full_size_replay(dict(CONFIGS['config2']), 2000.0, seed=1)
    got, res = out['f64']
    inc = np.abs(want - prior_rows).max()
    assert inc > 1e-3 and res.assimilated.all()
    assert np.abs(got - want).max() <= 1e-9 * inc


def test_config4_full_size_replay_f64_and_fp32_tolerance():
    """BASELINE config 4 in full (100 members, 721x1440 x 10 levels, 1e5 obs): the float64 analysis against the
    numpy replay at 1e-9 of the increment, and the float32 instantiation against it at the stated float32
    tolerance: analysis within 1e-5 of the field magnitude, perturbations within 1e-3 of the ensemble spread."""
    from efa_xray_b200.synth import CONFIGS
    out, want, prior_rows = _full_size_replay(dict(CONFIGS['config4']), 2000.0, seed=2, dtypes=('f64', 'f32'), n_rows=6)
    got, res = out['f64']
    inc = np.abs(want - prior_rows).max()
    assert inc > 1e-3 and res.assimilated.all()
    assert np.abs(got - want).max() <= 1e-9 * inc
    got32, res32 = out['f32']
    assert np.abs(got32 - want).max() <= 1e-5 * np.abs(want).max()
    pert = want - want.mean(axis=1, keepdims=True)
    pert32 = got32 - got32.mean(axis=1, keepdims=True)
    assert np.abs(pert32 - pert).max() <= 1e-3 * pert.std()
    np.testing.assert_allclose(res32.post_var, res.post_var, rtol=2e-3)


def test_edge_cases_skipped_single_and_polar_obs():
    """Reference edge cases (ensrf.py:66-76): when every ob is skipped the state comes back unchanged and the prior
    diagnostics are still recorded; a single ob; obs next to the poles and on the date line (largest footprints,
    SURVEY 7.2) against the oracle."""
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=37, nx=72, nmem=20, nvars=2, ntimes=1, nobs=30, cutoff_km=2500.0, seed=61)
    # (1) nothing assimilated
    state, obs = build_objects(case, EnsembleState, Observation)
    for o in obs:
        o.assimilate_this = False
    prior = state.to_vect().copy()
    post, obs = EnSRF(state, obs, verbose=False, loc='GC').update()
    np.testing.assert_array_equal(post.to_vect(), prior)
    assert all(o.assimilated is False and o.prior_mean is not None and o.prior_var > 0 for o in obs)
    # (2) a single ob
    case1 = make_case(ny=37, nx=72, nmem=20, nvars=1, ntimes=1, nobs=1, cutoff_km=2500.0, seed=62)
    state, obs = build_objects(case1, EnsembleState, Observation)
    post, obs = EnSRF(state, obs, verbose=False, loc='GC').update()
    ref_post, ref_obs = _oracle_run(case1, 'GC')
    _check_post(post.to_vect(), ref_post, state.to_vect())
    # (3) polar and date-line obs
    case.ob_lat[:6] = [88.7, -88.9, 86.2, -87.4, 0.3, -0.7]
    case.ob_lon[:6] = [12.3, 200.1, 359.2, 0.4, 359.6, 0.6]
    state, obs = build_objects(case, EnsembleState, Observation)
    post, obs = EnSRF(state, obs, verbose=False, loc='GC').update()
    ref_post, ref_obs = _oracle_run(case, 'GC')
    _check_post(post.to_vect(), ref_post, state.to_vect())
    np.testing.assert_allclose(_diag(obs, 'post_var'), _diag(ref_obs, 'post_var'), rtol=1e-9, equal_nan=True)


@pytest.mark.parametrize('obs_range,ob_error,inflation', [((1, 5), 1.0, 1.0), ((2, 4), 0.25, 2.0), ((1, 1), 2.0, 1.5)])
def test_single_point_efa_demo_matches_notebook_arithmetic(obs_range, ob_error, inflation):
    """efa_demo.ipynb cell 11 (`enkf`): one-point forecast trajectory, obs of its first valid times in shuffled order,
    no localisation, optional inflation -- the library path against the notebook's numpy statements."""
    from efa_xray_b200.demo import enkf, synthetic_point_ensemble
    from oracle.demo_oracle import enkf_numpy
    _, prior = synthetic_point_ensemble(ntimes=13, nmems=21, seed=4)
    obs = [275.0, 275.0, 275.0, 275.0, 276.0]
    n = obs_range[1] - obs_range[0] + 1
    order = np.random.default_rng(8).permutation(n)
    got = enkf(obs, prior, obs_range=obs_range, ob_error=ob_error, inflation=inflation, order=order)
    want = enkf_numpy(obs, prior, obs_range=obs_range, ob_error=ob_error, inflation=inflation, order=order)
    np.testing.assert_allclose(got, want, rtol=1e-11)
    assert np.abs(want - prior).max() > 0.1
    # the notebook shuffles the obs on every call; its variance (ddof 0) and covariance (ddof 1) normalisations differ
    # (cell 11, lines 64 and 75), so the result depends on the order even without localisation: check a second order
    order2 = order[::-1].copy()
    np.testing.assert_allclose(enkf(obs, prior, obs_range=obs_range, ob_error=ob_error, inflation=inflation, order=order2),
                               enkf_numpy(obs, prior, obs_range=obs_range, ob_error=ob_error, inflation=inflation, order=order2),
                               rtol=1e-11)


def test_one_dimensional_latlon_state_matches_reference_golden():
    """States with 1-D lat(x)/lon(x) (state/ensemble.py:185-192, ensrf.py:110-111): nearest points, the forward
    operator (leading axis of length 1, state read at (y, x) = (n, n)) and the x-only localisation against the
    unmodified reference; the full update is covered by test_update_matches_reference_golden[gc_1d_points]."""
    EnsembleState, Observation, _ = _api()
    g, p = load_golden('gc_1d_points')
    case = golden_case(p)
    state, obs = build_objects(case, EnsembleState, Observation)
    assert state['lat'].shape == (24,) and state.shape() == (2, 1, 24, 24, 8)
    for k in (0, 7, len(obs) - 1):
        near = state.nearest_points(obs[k].lat, obs[k].lon, npt=4)
        assert len(near) == 1 and set(near[0].tolist()) == set(g['nearest'][k][0].tolist())
        ye = obs[k].estimate(state)
        assert ye.shape == (1, 8)
        np.testing.assert_allclose(ye, g['ye'][k], rtol=1e-12)
    w = obs[0].localize(state)
    assert w.shape == (24,)
    np.testing.assert_allclose(w, g['loc_state0'], rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(obs[0].localize(obs), g['loc_obs0'], rtol=1e-10, atol=1e-13)
    # any npt (ensemble.py:165 takes the first npt of a full argsort): the first four of nine are the four
    near4 = state.nearest_points(obs[0].lat, obs[0].lon, npt=4)
    near9 = state.nearest_points(obs[0].lat, obs[0].lon, npt=9)
    assert len(near9) == 1 and near9[0].shape == (9,) and near9[0][:4].tolist() == near4[0].tolist()
    assert len(set(near9[0].tolist())) == 9


def test_empty_observation_list_returns_the_prior():
    """A window without observations: the reference's loop body never runs (ensrf.py:50) and the posterior is the
    prior -- inflated first if inflation was requested (assimilation.py:132-134)."""
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=19, nx=36, nmem=6, nvars=2, ntimes=1, nobs=3, seed=81)
    state, _ = build_objects(case, EnsembleState, Observation)
    prior = state.to_vect().copy()
    post, obs = EnSRF(state, [], verbose=False, loc='GC').update()
    assert obs == [] and post is not state
    np.testing.assert_array_equal(post.to_vect(), prior)
    np.testing.assert_array_equal(state.to_vect(), prior)
    post, _ = EnSRF(state, [], inflation=1.5, verbose=False, loc='GC').update()
    m = prior.mean(axis=1, keepdims=True)
    np.testing.assert_allclose(post.to_vect(), (prior - m) * 1.5 + m, rtol=1e-14)
    np.testing.assert_allclose(state.to_vect(), (prior - m) * 1.5 + m, rtol=1e-14)     # inflated in place, as the reference
