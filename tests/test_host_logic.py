"""Host-side logic that needs no GPU: band schedules, ob-order helper, time weights, sharding helpers."""
import numpy as np
import pytest


def test_sweep_band_schedule_covers_rows_on_patch_boundaries(lib):
    from efa_xray_b200 import engine
    for nlev, ny, nx in ((3, 721, 1440), (1, 181, 360), (12, 361, 720), (10, 721, 1440), (3, 90, 1440), (2, 7, 9)):
        g = lib.exb_state_sweep_row_granularity(nlev, ny, nx)
        assert 1 <= g <= 12
        bands = engine.sweep_band_schedule(nlev, ny, nx)
        assert bands[0][0] == 0 and bands[-1][1] == ny
        for (a, b), (c, d) in zip(bands[:-1], bands[1:]):
            assert b == c and a < b
        for a, b in bands[:-1]:
            assert b % g == 0          # a patch is never split between two calls
        assert len(bands) <= 7
    # the last band is the short one (its download is what stays exposed)
    bands = engine.sweep_band_schedule(3, 721, 1440)
    assert bands[-1][1] - bands[-1][0] <= (bands[0][1] - bands[0][0])


def test_patch_shape_of_the_sweep_kernel(lib):
    """128 rows per patch with one CTA of 16 warps per SM: the band schedule follows the kernel's patch rows."""
    from efa_xray_b200 import engine
    assert lib.exb_state_sweep_row_granularity(3, 721, 1440) == 6       # 42 points x 3 levels: 6 x 7 points
    g = lib.exb_state_sweep_row_granularity(10, 721, 1440)              # 12 points x 10 levels: 3 x 4
    assert g == 3
    for a, b in engine.sweep_band_schedule(10, 721, 1440)[:-1]:
        assert b % g == 0


def test_randomize_obs_order_is_a_seeded_permutation():
    from efa_xray.assimilation.assimilation import randomize_obs_order
    obs = list(range(50))
    a = randomize_obs_order(list(obs), seed=3)
    b = randomize_obs_order(list(obs), seed=3)
    c = randomize_obs_order(list(obs), seed=4)
    assert a == b and a != c and sorted(a) == obs and a != obs
    same = list(obs)
    assert randomize_obs_order(same, seed=1) is same          # in place


def test_time_weights_follow_the_reference_including_its_swap():
    """state/ensemble.py:202-224: an ob exactly on a valid time gets weight 1 there; between two times the
    reference attaches the LARGER weight to the FARTHER time (its weights are swapped); outside -> flagged."""
    from efa_xray_b200 import engine
    valid = np.array(['2020-01-01T00', '2020-01-01T06', '2020-01-01T12'], dtype='datetime64[s]')
    t = np.array(['2020-01-01T06', '2020-01-01T07:30', '2020-01-01T00', '2019-12-31T23', '2020-01-01T13'], dtype='datetime64[s]')
    lo, hi, wlo, whi, outside = engine.time_weights(valid, t)
    assert outside.tolist() == [False, False, False, True, True]
    assert (hi[0], whi[0], wlo[0]) == (1, 1.0, 0.0)
    assert (lo[1], hi[1]) == (1, 2)
    np.testing.assert_allclose([wlo[1], whi[1]], [0.25, 0.75])   # 1.5 h after 06: upper level (4.5 h away) gets 0.75
    assert (hi[2], whi[2]) == (0, 1.0)


def test_postprocess_module_is_reexported():
    import efa_xray.postprocess.postprocess as p
    from efa_xray_b200.postprocess.postprocess import COLUMNS
    assert callable(p.obs_assimilation_statistics)
    assert COLUMNS[:4] == ['validtime', 'flead', 'lat', 'lon'] and COLUMNS[-1] == 'post variance'


def test_localize_stencil_keeps_only_band_rows():
    from efa_xray_b200.sharding import localize_stencil, partition_bands, equal_bands
    nlev, ny, nx = 2, 10, 4
    idx = np.array([[0, 5 * nx + 1, ny * nx + 9 * nx + 3, 3 * nx]])
    w = np.array([[0.1, 0.2, 0.3, 0.4]])
    li, lw = localize_stencil(idx, w, nlev, ny, nx, 3, 6)
    assert lw.tolist() == [[0.0, 0.2, 0.0, 0.4]]
    assert li[0, 1] == (0 * 3 + 2) * nx + 1 and li[0, 3] == 0 * nx + 0
    assert equal_bands(10, 3) == [(0, 3), (3, 7), (7, 10)]
    assert partition_bands(np.ones(10), 2) == [(0, 5), (5, 10)]


def _small_state(**kw):
    from efa_xray_b200.synth import make_case, build_objects
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    case = make_case(**dict(dict(ny=7, nx=9, nmem=5, nvars=2, ntimes=2, nobs=6, seed=11), **kw))
    state, obs = build_objects(case, EnsembleState, Observation)
    return case, state, obs


def test_state_block_layout_is_the_state_vector():
    """The variables of an EnsembleState are views of one [nvar, nt, ny, nx, nmem] block, which is the reference's
    to_vect layout (state/ensemble.py:110-121): to_vect is a read-only view, from_vect writes through, a deep copy
    is independent, and replacing a variable's array falls back to stacking."""
    from copy import deepcopy
    case, state, _ = _small_state()
    want = case.to_vect()
    v = state.to_vect()
    assert v.shape == (state.nstate(), state.nmems()) == want.shape
    np.testing.assert_array_equal(v, want)
    assert not v.flags.writeable and np.shares_memory(v, state.variables['var0'].values)
    assert state.shape() == (2, 2, 7, 9, 5)
    state.variables['var1'][:] = state.variables['var1'].values * 2.0          # in place through a view
    np.testing.assert_array_equal(state.to_vect()[state.nstate() // 2:], 2.0 * want[state.nstate() // 2:])
    cp = deepcopy(state)
    cp.from_vect(np.zeros_like(want))
    assert np.abs(cp.to_vect()).max() == 0.0 and np.abs(state.to_vect()).max() > 0.0
    assert np.shares_memory(cp.to_vect(), cp.variables['var0'].values)
    # a variable whose array was replaced no longer aliases the block: to_vect stacks, as the reference does
    state['var0'].values = np.ones_like(state['var0'].values)
    w = state.to_vect()
    assert w.flags.writeable and (w[:state.nstate() // 2] == 1.0).all()
    np.testing.assert_array_equal(w[state.nstate() // 2:], 2.0 * want[state.nstate() // 2:])


def test_state_adopts_a_callers_contiguous_buffer():
    from efa_xray_b200.synth import make_case, build_objects
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    out = np.empty((3, 1, 5, 6, 4))
    case = make_case(ny=5, nx=6, nmem=4, nvars=3, ntimes=1, nobs=2, seed=12, out=out)
    state, _ = build_objects(case, EnsembleState, Observation)
    assert np.shares_memory(state.to_vect(), out)          # no copy at construction
    np.testing.assert_array_equal(state.to_vect(), out.reshape(-1, 4))


def test_save_to_disk_round_trip_and_hostile_file(tmp_path):
    """state/ensemble.py:269-273 (netCDF needs xarray; the archive carries the same variables, coordinates, dims)."""
    from efa_xray_b200.state.ensemble import EnsembleState
    _, state, _ = _small_state()
    fn = str(tmp_path / 'ens_state.nc')
    state.save_to_disk(fn)
    back = EnsembleState.load_from_disk(fn)
    np.testing.assert_array_equal(back.to_vect(), state.to_vect())
    assert back.vars() == state.vars() and back.shape() == state.shape()
    for k in ('lat', 'lon', 'validtime', 'mem', 'y', 'x'):
        np.testing.assert_array_equal(back.coords[k].values, state.coords[k].values)
        assert back.coords[k].dims == state.coords[k].dims
    # the dims record is data, never code
    bad = str(tmp_path / 'bad.npz')
    np.savez(bad, __dims__=np.array("__import__('os').system('true')"), var__a=np.zeros(1))
    with pytest.raises(ValueError):
        EnsembleState.load_from_disk(bad)


@pytest.mark.parametrize('inflation', [1.5, {'var1': 1.25, 'nosuch': 3.0},
                                       {'validtime': np.array([1.1, 1.4]), 'y': np.linspace(1, 1.5, 7), 'var0': 1.2,
                                        'x': np.linspace(1.3, 0.9, 9)}])
def test_inflation_factor_tables_match_the_oracle(inflation, capsys):
    """Assimilation._inflation_factors (one factor per level, or per state row for per-dimension arrays) applied as
    (x - mean) * f + mean reproduces the oracle's restatement of assimilation.py:52-118."""
    from efa_xray_b200.assimilation.assimilation import Assimilation
    from oracle import ensrf_oracle as O
    case, state, obs = _small_state()
    fac = Assimilation(state, obs, inflation=inflation)._inflation_factors()
    X = case.to_vect()
    f = np.repeat(fac, X.shape[0] // fac.shape[0])
    m = X.mean(axis=1, keepdims=True)
    got = (X - m) * f[:, None] + m
    want = O.inflate_state(O.State.from_case(case), inflation).to_vect()
    np.testing.assert_allclose(got, want, rtol=1e-13)
    with pytest.raises(ValueError):                      # 2-D lat cannot carry a per-dimension array (nor in the reference)
        Assimilation(state, obs, inflation={'lat': np.ones(7)})._inflation_factors()


def test_obs_marshalling_is_vectorised_and_keeps_reference_errors():
    from efa_xray_b200.assimilation.assimilation import Assimilation
    from efa_xray_b200 import engine
    case, state, obs = _small_state(offtime=True, frac_skip=0.3, mixed_radius=True)
    a = Assimilation(state, obs)._obs_arrays(engine.LOC_GC)
    np.testing.assert_array_equal(a.value, case.ob_value)
    np.testing.assert_array_equal(a.lat, case.ob_lat)
    np.testing.assert_array_equal(a.assimilate, case.ob_assimilate.astype(np.uint8))
    np.testing.assert_array_equal(a.halfwidth[case.ob_assimilate], case.ob_halfwidth[case.ob_assimilate])
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time)
    np.testing.assert_array_equal(a.row0, (case.ob_var * 2 + tlo) * 63)
    np.testing.assert_array_equal(a.tw1, whi)
    assert Assimilation(state, [])._obs_arrays(engine.LOC_GC).nobs == 0          # an empty window is not an error
    k = int(np.flatnonzero(case.ob_assimilate)[0])
    obs[k].localize_radius = None
    with pytest.raises(TypeError):                       # abs(None), observation.py:120
        Assimilation(state, obs)._obs_arrays(engine.LOC_GC)
    obs[k].localize_radius = 100.0
    obs[k].obtype = 'nosuchvar'
    with pytest.raises(KeyError):
        Assimilation(state, obs)._obs_arrays(engine.LOC_GC)


def test_block_dealing_of_obs_rows_is_a_partition_in_increasing_order():
    """The distributed obs-space solve deals blocks of consecutive obs to the ranks (exb_obs_plan_create_dist): the
    v-th row of rank r is ((v // b) * world + r) * b + v % b.  The engine's ownership mask ((j // b) % world == r) and
    the library's row count formula must describe the same partition, each rank's rows in increasing order."""
    for nobs, world, b in ((10, 2, 1), (3001, 2, 256), (2501, 4, 7), (100000, 8, 256), (5, 8, 3)):
        owner = (np.arange(nobs) // b) % world
        seen = np.zeros(nobs, dtype=int)
        for r in range(world):
            cyc = b * world
            rem = nobs % cyc - r * b
            nrows = (nobs // cyc) * b + min(max(rem, 0), b)
            v = np.arange(nrows)
            rows = ((v // b) * world + r) * b + v % b
            assert np.array_equal(rows, np.flatnonzero(owner == r))
            assert (np.diff(rows) > 0).all()
            seen[rows] += 1
        assert (seen == 1).all()
