"""The bilinear forward operator (forward_operator='bilinear', DESIGN.md section 4.8): axis classification, time
weights, the numpy reference's known answers and the argument checks of the API and of the C entries (no device
needed); on the GPU both stencil kernels against the reference (tests/bilinear_reference.py), and every analysis path
against the reference analysis built on the unchanged CPU oracle."""
import dataclasses

import numpy as np
import pytest

import bilinear_reference as B
from efa_xray_b200 import engine
from efa_xray_b200.synth import make_case, make_case_1d, build_objects

F64_RTOL = 1e-10          # as test_gpu_parity._check_post
F64_INC_TOL = 1e-9


def _api():
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    from efa_xray_b200.assimilation.ensrf import EnSRF
    return EnsembleState, Observation, EnSRF


def _mesh(lat_y, lon_x):
    lon2d, lat2d = np.meshgrid(np.asarray(lon_x, dtype=np.float64), np.asarray(lat_y, dtype=np.float64))
    return np.ascontiguousarray(lat2d), np.ascontiguousarray(lon2d)


def _gaussian_lats(n):
    return np.degrees(np.arcsin(np.polynomial.legendre.leggauss(n)[0]))


# rectilinear grids: name -> (lat_y, lon_x, periodic)
RECT_GRIDS = {
    'global_asc_0360': (np.linspace(-90.0, 90.0, 19), np.arange(36) * 10.0, True),
    'global_desc_pm180': (np.linspace(90.0, -90.0, 19), -180.0 + np.arange(36) * 10.0, True),
    'cell_centred': (np.arange(-85.0, 86.0, 10.0), 5.0 + np.arange(36) * 10.0, True),
    'regional': (np.linspace(20.0, 60.0, 21), np.linspace(-130.0, -60.0, 36), False),
    'regional_desc_dateline': (np.linspace(60.0, 20.0, 17), (160.0 + np.arange(30) * 2.5 + 180.0) % 360.0 - 180.0,
                               False),
    'gaussian': (_gaussian_lats(32), np.arange(64) * 5.625, True),
}


# ---------------------------------------------------------------------------------------------------------------
# CPU: axis classification, time weights, the reference
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', sorted(RECT_GRIDS))
def test_rectilinear_axes_are_classified(name):
    lat_y, lon_x, periodic = RECT_GRIDS[name]
    kind, ly, lon_u, per = engine.bilinear_axes(*_mesh(lat_y, lon_x))
    assert kind == 'rect' and per == periodic
    np.testing.assert_array_equal(ly, lat_y)
    assert (np.diff(lon_u) > 0).all() and lon_u[0] == lon_x[0]
    np.testing.assert_allclose(np.mod(lon_u, 360.0), np.mod(lon_x, 360.0), atol=1e-12)
    assert B.classify(*_mesh(lat_y, lon_x))[0] == 'rect' and B.classify(*_mesh(lat_y, lon_x))[3] == periodic


def test_non_monotone_or_non_rectilinear_axes_go_to_the_curvilinear_path():
    lat = np.linspace(-60.0, 60.0, 9)
    lon = np.arange(12) * 10.0
    for lat_y, lon_x in ((lat[[0, 1, 3, 2, 4, 5, 6, 7, 8]], lon),           # non-monotone lat
                         (np.concatenate([lat[:4], lat[3:8]]), lon),          # repeated lat
                         (lat, lon[[0, 1, 2, 4, 3, 5, 6, 7, 8, 9, 10, 11]]),  # lon not increasing after unwrapping
                         (lat, np.arange(12) * 40.0)):                        # lon spans more than 360
        assert engine.bilinear_axes(*_mesh(lat_y, lon_x))[0] == 'curv'
        assert B.classify(*_mesh(lat_y, lon_x))[0] == 'curv'
    lat2d, lon2d = _mesh(lat, lon)
    lat2d[3, 4] += 0.01                                                       # not rectilinear
    assert engine.bilinear_axes(lat2d, lon2d)[0] == 'curv'


def test_axes_that_are_not_2d_are_rejected():
    with pytest.raises(ValueError):
        engine.bilinear_axes(np.linspace(0, 10, 5), np.linspace(0, 10, 5))
    with pytest.raises(ValueError):
        engine.bilinear_axes(*_mesh([10.0], np.arange(5.0)))


def test_time_weights_correctly_oriented():
    valid = np.array(['2020-01-01T00', '2020-01-01T06', '2020-01-01T12'], dtype='datetime64[ns]')
    t = np.array(['2020-01-01T00', '2020-01-01T01:30', '2020-01-01T06', '2020-01-01T10:30', '2020-01-01T12'],
                 dtype='datetime64[ns]')
    lo, hi, wlo, whi, outside = engine.time_weights(valid, t, swapped=False)
    assert not outside.any()
    np.testing.assert_array_equal(hi, [0, 1, 1, 2, 2])
    np.testing.assert_array_equal(lo, [0, 0, 0, 1, 1])
    np.testing.assert_allclose(whi, [1.0, 0.25, 1.0, 0.75, 1.0], rtol=1e-15)
    np.testing.assert_allclose(wlo, [0.0, 0.75, 0.0, 0.25, 0.0], rtol=1e-15)
    # the default keeps the reference's swapped weights
    _, _, swlo, swhi, _ = engine.time_weights(valid, t)
    np.testing.assert_allclose(swhi, [1.0, 0.75, 1.0, 0.25, 1.0], rtol=1e-15)
    # the reference's levels give the same field
    rlo, rhi, rwlo, rwhi = B.time_levels(valid, t)
    for k in range(len(t)):
        a, b = np.zeros(3), np.zeros(3)
        a[lo[k]] += wlo[k]; a[hi[k]] += whi[k]
        b[rlo[k]] += rwlo[k]; b[rhi[k]] += rwhi[k]
        np.testing.assert_allclose(a, b, atol=1e-15)


@pytest.mark.parametrize('name', sorted(RECT_GRIDS))
def test_reference_reproduces_a_linear_field(name):
    """A field linear in (lat, unwrapped lon) inside a cell is reproduced exactly, on either path of the reference."""
    lat_y, lon_x, periodic = RECT_GRIDS[name]
    lat2d, lon2d = _mesh(lat_y, lon_x)
    rng = np.random.default_rng(1)
    ny, nx = lat2d.shape
    # cells without a pole corner: the curvilinear path does not support those
    j = rng.choice(np.flatnonzero(np.maximum(np.abs(lat_y[:-1]), np.abs(lat_y[1:])) < 89.0), 200)
    i = rng.integers(0, nx - 1, 200)
    s, t = rng.uniform(0, 1, 200), rng.uniform(0, 1, 200)
    lon_u = engine.bilinear_axes(lat2d, lon2d)[2]
    ob_lat = lat_y[j] + t * (lat_y[j + 1] - lat_y[j])
    ob_lon = lon_u[i] + s * (lon_u[i + 1] - lon_u[i])
    field = 3.0 * lat2d + 0.5 * (lon_u[None, :] + 0 * lat2d)
    for fn in (B.stencil, lambda la, lo, a, b: B.stencil_curv(la, lo, a, b)):
        idx4, w4, out = fn(lat2d, lon2d, ob_lat, (ob_lon + 180.0) % 360.0 - 180.0)
        assert not out.any()
        est = (w4 * field.ravel()[idx4]).sum(axis=1)
        np.testing.assert_allclose(est, 3.0 * ob_lat + 0.5 * ob_lon, rtol=1e-12)


def test_reference_ob_on_a_grid_point_gets_weight_one():
    lat_y, lon_x, _ = RECT_GRIDS['global_asc_0360']
    lat2d, lon2d = _mesh(lat_y, lon_x)
    ob_lat = np.array([10.0, -30.0, 50.0])
    ob_lon = np.array([20.0, 350.0, -10.0])
    for fn in (B.stencil, B.stencil_curv):
        idx4, w4, out = fn(lat2d, lon2d, ob_lat, ob_lon)
        assert not out.any()
        for k in range(3):
            p = int(np.argmax(w4[k]))
            if fn is B.stencil:                                # exact on the rectilinear path
                assert w4[k, p] == 1.0 and (np.delete(w4[k], p) == 0.0).all()
            else:                                              # to the Newton solve's accuracy
                assert w4[k, p] >= 1.0 - 1e-12
            y, x = divmod(int(idx4[k, p]), lon2d.shape[1])
            assert lat2d[y, x] == ob_lat[k] and lon2d[y, x] == ob_lon[k] % 360.0


def test_reference_seam_cell():
    lat_y, lon_x, _ = RECT_GRIDS['global_asc_0360']        # columns 0, 10, ..., 350
    lat2d, lon2d = _mesh(lat_y, lon_x)
    idx4, w4, out = B.stencil(lat2d, lon2d, np.array([5.0, 5.0, 5.0]), np.array([352.5, -2.5, 357.5]))
    assert not out.any()
    nx = 36
    j = 9                                                      # lat_y[9] = 0, lat_y[10] = 10: t = 0.5
    for k, s in enumerate((0.25, 0.75, 0.75)):
        np.testing.assert_array_equal(idx4[k], [j * nx + 35, j * nx + 0, (j + 1) * nx + 35, (j + 1) * nx + 0])
        np.testing.assert_allclose(w4[k], [(1 - s) / 2, s / 2, (1 - s) / 2, s / 2], atol=1e-15)
    # not periodic: past the last column is outside
    lat_y, lon_x, _ = RECT_GRIDS['regional']
    _, _, out = B.stencil(*_mesh(lat_y, lon_x), np.array([40.0, 40.0]), np.array([-59.0, -131.0]))
    assert out.all()


def test_reference_descending_axis_equals_ascending():
    rng = np.random.default_rng(2)
    lat_a, lon_x = np.linspace(-90.0, 90.0, 19), np.arange(36) * 10.0
    ob_lat = np.concatenate([rng.uniform(-90, 90, 300), lat_a])
    ob_lon = np.concatenate([rng.uniform(-180, 360, 300), rng.uniform(0, 360, 19)])
    field = rng.normal(size=(19, 36))
    ia, wa, oa = B.stencil(*_mesh(lat_a, lon_x), ob_lat, ob_lon)
    idd, wd, od = B.stencil(*_mesh(lat_a[::-1], lon_x), ob_lat, ob_lon)
    assert not oa.any() and not od.any()
    ea = (wa * field.ravel()[ia]).sum(axis=1)
    ed = (wd * field[::-1].ravel()[idd]).sum(axis=1)
    np.testing.assert_allclose(ed, ea, rtol=1e-13, atol=1e-13)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the API validates before any device work; the C entries validate their arguments
# ---------------------------------------------------------------------------------------------------------------
def _small_objects(one_d=False):
    EnsembleState, Observation, _ = _api()
    case = make_case_1d(npts=12, nmem=6, nobs=5, seed=3) if one_d else make_case(ny=19, nx=36, nmem=6, nobs=5, seed=91)
    return build_objects(case, EnsembleState, Observation)


@pytest.mark.parametrize('op,one_d', [('nope', False), ('Bilinear', False), (None, False), ('bilinear', True)])
def test_invalid_forward_operator_raises_value_error(op, one_d):
    from efa_xray_b200.assimilation.assimilation import Assimilation, update
    from efa_xray_b200.postprocess.postprocess import ob_estimates
    _, _, EnSRF = _api()
    state, obs = _small_objects(one_d)
    for fn in (lambda: EnSRF(state, obs, verbose=False, loc='GC', forward_operator=op),
               lambda: update(state, obs, loc='GC', forward_operator=op),
               lambda: Assimilation(state, obs, forward_operator=op),
               lambda: ob_estimates(state, obs, forward_operator=op),
               lambda: state.interpolate(obs[0].obtype, obs[0].time, obs[0].lat, obs[0].lon, forward_operator=op),
               lambda: obs[0].estimate(state, forward_operator=op)):
        with pytest.raises(ValueError):
            fn()
    assert EnSRF(state, obs, verbose=False).forward_operator == 'reference'


def test_obs_arrays_take_the_time_orientation_of_the_operator():
    from efa_xray_b200.assimilation.assimilation import Assimilation
    EnsembleState, Observation, _ = _api()
    case = make_case(ny=19, nx=36, nmem=6, ntimes=3, nobs=40, seed=5, offtime=True)
    state, obs = build_objects(case, EnsembleState, Observation)
    a_ref = Assimilation(state, obs)._obs_arrays(engine.LOC_NONE)
    a_bil = Assimilation(state, obs, forward_operator='bilinear')._obs_arrays(engine.LOC_NONE)
    off = (a_ref.tw1 != 1.0) & (a_ref.tw1 != 0.0)
    assert off.sum() > 10
    np.testing.assert_allclose(a_bil.tw1[off], a_ref.tw0[off], rtol=1e-12)
    np.testing.assert_array_equal(a_bil.row0, a_ref.row0)


def test_c_entry_argument_errors_return_status(lib):
    import ctypes as C
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p)
    assert lib.exb_stencil_bilinear_rect(None, p, 4, 4, 1, p, p, 2, p, p, p, None) == -1
    assert b'exb_stencil_bilinear_rect' in lib.exb_last_error()
    assert lib.exb_stencil_bilinear_rect(p, p, 4, 4, 1, p, p, 2, p, p, None, None) == -1
    assert lib.exb_stencil_bilinear_rect(p, p, 1, 4, 1, p, p, 2, p, p, p, None) == -1
    assert lib.exb_stencil_bilinear_rect(p, p, 4, 4, 2, p, p, 2, p, p, p, None) == -1
    assert lib.exb_stencil_bilinear_rect(p, p, 4, 4, 0, p, p, 0, p, p, p, None) == -1
    assert lib.exb_stencil_bilinear_curv(None, p, p, 4, 4, p, p, 2, p, p, p, None) == -1
    assert b'exb_stencil_bilinear_curv' in lib.exb_last_error()
    assert lib.exb_stencil_bilinear_curv(p, p, p, 4, 4, p, None, 2, p, p, p, None) == -1
    assert lib.exb_stencil_bilinear_curv(p, p, p, 4, 1, p, p, 2, p, p, p, None) == -1


# ---------------------------------------------------------------------------------------------------------------
# GPU: the stencil kernels against the reference
# ---------------------------------------------------------------------------------------------------------------
def _gpu_stencil(lat2d, lon2d, ob_lat, ob_lon, force_curvilinear=False):
    import torch
    dev = torch.device('cuda', 0)
    grid = engine.GridTables(lat2d, lon2d, dev)
    d_lat = torch.as_tensor(np.ascontiguousarray(ob_lat, dtype=np.float64)).to(dev)
    d_lon = torch.as_tensor(np.ascontiguousarray(ob_lon, dtype=np.float64)).to(dev)
    idx4, w4, nout = engine.stencil_bilinear(grid, d_lat, d_lon, force_curvilinear=force_curvilinear)
    return idx4.cpu().numpy(), w4.cpu().numpy(), int(nout.item())


def _rect_obs(lat_y, lon_x, seed, seam=True):
    """Random obs plus obs on grid points, on grid lines, on and around the seam (seam=True), at +-90 and outside the
    grid, with longitudes in several conventions."""
    rng = np.random.default_rng(seed)
    ny, nx = len(lat_y), len(lon_x)
    lo, hi = min(lat_y[0], lat_y[-1]), max(lat_y[0], lat_y[-1])
    lon_u = engine.bilinear_axes(*_mesh(lat_y, lon_x))[2]
    lat = [rng.uniform(lo, hi, 400)]
    lon = [rng.uniform(lon_u[0], lon_u[-1], 400) + 360.0 * rng.integers(-1, 2, 400)]
    gy, gx = rng.integers(0, ny, 60), rng.integers(0, nx, 60)
    lat.append(lat_y[gy]); lon.append(lon_x[gx])                                       # grid points
    lat.append(lat_y[rng.integers(0, ny, 40)]); lon.append(rng.uniform(lon_u[0], lon_u[-1], 40))   # grid rows
    lat.append(rng.uniform(lo, hi, 40)); lon.append(lon_x[rng.integers(0, nx, 40)] - 360.0)       # grid columns
    seam = None if not seam else np.array([lon_u[-1], lon_u[0] + 360.0, 0.5 * (lon_u[-1] + lon_u[0] + 360.0), lon_u[0] - 1e-9,
                     lon_u[-1] + 1e-9, lon_u[0] + 360.0 - 1e-13])
    if seam is not None:
        lat.append(rng.uniform(lo, hi, len(seam))); lon.append(seam)
    lat.append(np.array([90.0, -90.0, 90.0, -90.0])); lon.append(np.array([0.0, 123.0, lon_u[0], lon_u[-1]]))
    lat.append(np.array([lo - 1.0, hi + 1.0, 95.0, -91.0, np.nan, 0.5 * (lo + hi)]))            # outside / NaN
    lon.append(np.array([lon_u[0], lon_u[0], lon_u[0], lon_u[0], lon_u[0], np.nan]))
    return np.concatenate(lat), np.concatenate(lon)


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(RECT_GRIDS))
def test_rect_kernel_matches_reference(name):
    lat_y, lon_x, periodic = RECT_GRIDS[name]
    lat2d, lon2d = _mesh(lat_y, lon_x)
    assert engine.bilinear_axes(lat2d, lon2d)[0] == 'rect'
    ob_lat, ob_lon = _rect_obs(lat_y, lon_x, seed=sorted(RECT_GRIDS).index(name))
    idx, w, nout = _gpu_stencil(lat2d, lon2d, ob_lat, ob_lon)
    ridx, rw, rout = B.stencil_rect(lat_y, lon_x, periodic, ob_lat, ob_lon)
    assert nout == int(rout.sum()) and nout >= 3
    np.testing.assert_allclose(w, rw, rtol=0, atol=1e-14)
    pos = rw > 0
    np.testing.assert_array_equal(idx[pos], ridx[pos])
    assert (w[rout] == 0).all() and (idx[rout] == 0).all()
    np.testing.assert_allclose(w[~rout].sum(axis=1), 1.0, rtol=1e-14)


def _rotated_pole_grid(ny=40, nx=56):
    """A rotated-pole regional grid: regular in rotated (lat, lon), turned to geographic coordinates."""
    rlat, rlon = np.meshgrid(np.linspace(-15.0, 15.0, ny), np.linspace(-20.0, 20.0, nx), indexing='ij')
    v = B._unit(rlat, rlon)
    b, a = np.radians(-35.0), np.radians(250.0)
    ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    rz = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
    g = v @ (rz @ ry).T
    lat = np.degrees(np.arcsin(np.clip(g[..., 2], -1, 1)))
    lon = np.degrees(np.arctan2(g[..., 1], g[..., 0])) % 360.0
    return np.ascontiguousarray(lat), np.ascontiguousarray(lon)


def _lambert_grid(ny=45, nx=60, dx_km=40.0, lat0=40.0, lon0=-100.0):
    """A Lambert-conformal (tangent cone at lat0) regional grid, WRF style, regular in projected x / y."""
    R = 6371.0
    n = np.sin(np.radians(lat0))
    F = np.cos(np.radians(lat0)) * np.tan(np.pi / 4 + np.radians(lat0) / 2) ** n / n
    rho0 = R * F / np.tan(np.pi / 4 + np.radians(lat0) / 2) ** n
    y, x = np.meshgrid((np.arange(ny) - ny / 2) * dx_km, (np.arange(nx) - nx / 2) * dx_km, indexing='ij')
    rho = np.sign(n) * np.hypot(x, rho0 - y)
    theta = np.arctan2(x, rho0 - y)
    lat = np.degrees(2 * np.arctan((R * F / rho) ** (1 / n)) - np.pi / 2)
    lon = lon0 + np.degrees(theta / n)
    return np.ascontiguousarray(lat), np.ascontiguousarray(lon)


def _obs_in_cells(lat2d, lon2d, n, seed, margin=0):
    """n points inside random cells (the bilinear image of random (s, t) in the (lat, unwrapped lon) plane)."""
    rng = np.random.default_rng(seed)
    ny, nx = lat2d.shape
    y = rng.integers(margin, ny - 1 - margin, n)
    x = rng.integers(margin, nx - 1 - margin, n)
    s, t = rng.uniform(0, 1, n), rng.uniform(0, 1, n)
    ref = lon2d[y, x]
    c = [(lat2d[y + a, x + b], ref + B._wrap180(lon2d[y + a, x + b] - ref)) for a, b in ((0, 0), (0, 1), (1, 0), (1, 1))]
    w = [(1 - s) * (1 - t), s * (1 - t), (1 - s) * t, s * t]
    return sum(wi * ci[0] for wi, ci in zip(w, c)), sum(wi * ci[1] for wi, ci in zip(w, c))


def _sparse(idx4, w4, npts):
    from scipy.sparse import csr_matrix
    n = idx4.shape[0]
    return csr_matrix((w4.ravel(), (np.repeat(np.arange(n), 4), idx4.ravel())), shape=(n, npts))


@pytest.mark.gpu
@pytest.mark.parametrize('grid', ['rotated_pole', 'lambert'])
def test_curv_kernel_matches_reference(grid):
    lat2d, lon2d = _rotated_pole_grid() if grid == 'rotated_pole' else _lambert_grid()
    assert engine.bilinear_axes(lat2d, lon2d)[0] == 'curv'
    ob_lat, ob_lon = _obs_in_cells(lat2d, lon2d, 2000, seed=7)
    ny, nx = lat2d.shape
    ob_lat = np.concatenate([ob_lat, lat2d[::7, ::5].ravel(), [-60.0, -10.0, 0.0]])
    ob_lon = np.concatenate([ob_lon, lon2d[::7, ::5].ravel() - 360.0, [0.0, 30.0, 0.0]])
    idx, w, nout = _gpu_stencil(lat2d, lon2d, ob_lat, ob_lon)
    ridx, rw, rout = B.stencil_curv(lat2d, lon2d, ob_lat, ob_lon)
    assert nout == int(rout.sum()) == 3
    out = (w == 0).all(axis=1)
    np.testing.assert_array_equal(out, rout)
    diff = _sparse(idx, w, ny * nx) - _sparse(ridx, rw, ny * nx)
    assert abs(diff).max() <= 1e-12


@pytest.mark.gpu
def test_curv_kernel_reproduces_rect_kernel_on_a_rectilinear_grid():
    lat_y, lon_x, _ = RECT_GRIDS['regional']
    lat2d, lon2d = _mesh(lat_y, lon_x)
    # no seam obs: within 1e-10 of the grid's edge the curvilinear path's containment tolerance accepts an ob
    ob_lat, ob_lon = _rect_obs(lat_y, lon_x, seed=11, seam=False)
    idx, w, nout = _gpu_stencil(lat2d, lon2d, ob_lat, ob_lon)
    cidx, cw, cout = _gpu_stencil(lat2d, lon2d, ob_lat, ob_lon, force_curvilinear=True)
    assert nout == cout and nout >= 3
    diff = _sparse(idx, w, lat2d.size) - _sparse(cidx, cw, lat2d.size)
    assert abs(diff).max() <= 1e-12


# ---------------------------------------------------------------------------------------------------------------
# GPU: the analysis through the public API against the reference analysis
# ---------------------------------------------------------------------------------------------------------------
def _check_post(post, ref_post, prior, tol_scale=1.0):
    np.testing.assert_allclose(post, ref_post, rtol=F64_RTOL * tol_scale)
    inc_ref = ref_post - prior
    scale = max(np.abs(inc_ref).max(), 1e-30)
    assert np.abs((post - prior) - inc_ref).max() <= F64_INC_TOL * tol_scale * scale


def _check_diag(obs, ref_obs):
    for attr in ('prior_mean', 'prior_var', 'post_mean', 'post_var'):
        got = np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr)) for o in obs])
        want = np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr)) for o in ref_obs])
        np.testing.assert_allclose(got, want, rtol=1e-9, equal_nan=True)
    assert [o.assimilated for o in obs] == [o.assimilated for o in ref_obs]


def _regrid(case, lat2d, lon2d, seed):
    """The case on another grid of the same shape, with its obs moved into random cells of that grid."""
    ob_lat, ob_lon = _obs_in_cells(lat2d, lon2d, case.nobs, seed)
    return dataclasses.replace(case, lat2d=lat2d, lon2d=lon2d, ob_lat=ob_lat, ob_lon=ob_lon)


def _curv_case():
    lat2d, lon2d = _lambert_grid(ny=30, nx=40, dx_km=60.0)
    case = make_case(ny=30, nx=40, nmem=30, nvars=2, ntimes=2, nobs=80, cutoff_km=600.0, seed=301, offtime=True,
                     frac_skip=0.05)
    return _regrid(case, lat2d, lon2d, seed=302)


_MULTI = dict(ny=31, nx=60, nmem=24, nvars=2, ntimes=3, nobs=90, cutoff_km=2000.0, seed=305, offtime=True,
              frac_skip=0.08)
_C50 = dict(ny=25, nx=48, nmem=50, nvars=2, ntimes=2, nobs=70, cutoff_km=2500.0, seed=306, offtime=True,
            frac_skip=0.05)


# env: attributes of engine patched for the case; FUSED_MAX_NENS = 0 takes the three-call form
@pytest.mark.gpu
@pytest.mark.parametrize('kw,loc,inflation,env', [
    (_MULTI, 'GC', None, {}),
    (_C50, 'GC', None, {}),
    (_C50, 'GC', None, {'FUSED_MAX_NENS': 0}),
    (_C50, False, None, {}),
    (_C50, 'GC', 1.15, {}),
    (dict(ny=25, nx=48, nmem=7, nvars=1, ntimes=2, nobs=60, cutoff_km=1500.0, seed=307, offtime=True), 'GC', None, {}),
    (dict(ny=25, nx=48, nmem=100, nvars=2, ntimes=1, nobs=60, cutoff_km=3000.0, seed=308), 'GC', None, {}),
    (dict(ny=19, nx=36, nmem=130, nvars=1, ntimes=2, nobs=40, cutoff_km=4000.0, seed=309, offtime=True), 'GC', None,
     {}),
    ('curv', 'GC', None, {}),
])
def test_update_bilinear_matches_reference(kw, loc, inflation, env, monkeypatch):
    EnsembleState, Observation, EnSRF = _api()
    case = _curv_case() if kw == 'curv' else make_case(**kw)
    ref_post, ref_obs, prior = B.ensrf_update(case, loc=loc, inflation=inflation)
    state, obs = build_objects(case, EnsembleState, Observation)
    for name, value in env.items():
        monkeypatch.setattr(engine, name, value)
    post, _ = EnSRF(state, obs, verbose=False, loc=loc, inflation=inflation, forward_operator='bilinear').update()
    _check_post(post.to_vect(), ref_post, prior)
    _check_diag(obs, ref_obs)
    assert sum(o.assimilated for o in obs) > 0.8 * len(obs)


@pytest.mark.gpu
def test_update_bilinear_with_relaxation_and_qc_matches_reference():
    import relax_reference as RR
    from test_outlier_qc import qc_reference, _with_gross_errors
    from oracle import ensrf_oracle as O
    EnsembleState, Observation, EnSRF = _api()
    case = _with_gross_errors(make_case(**_C50), seed=3)
    thr, relaxation = 4.0, ('rtps', 0.6)
    prior = case.to_vect()
    ye = B.ob_priors(prior, case.lat2d, case.lon2d, case.times, case.ob_var, case.ob_time, case.ob_lat, case.ob_lon)
    ym = ye.mean(axis=1)
    rej, _ = qc_reference(ym, ye - ym[:, None], case.ob_value, case.ob_error, case.ob_halfwidth, case.ob_lat,
                          case.ob_lon, case.ob_assimilate, np.full(case.nobs, thr))
    assert rej.sum() >= 2
    ref_obs = O.obs_from_case(case)
    for o, r in zip(ref_obs, rej):
        o.assimilate_this = o.assimilate_this and not r
    post, ref_obs, _ = B.ensrf_update(case, loc='GC', obs=ref_obs)
    ref_post = RR.relax(prior, post, relaxation[0], RR.alpha_rows(O.State.from_case(case), relaxation[1]))
    state, obs = build_objects(case, EnsembleState, Observation)
    got, _ = EnSRF(state, obs, verbose=False, loc='GC', outlier_threshold=thr, relaxation=relaxation,
                   forward_operator='bilinear').update()
    _check_post(got.to_vect(), ref_post, prior)
    _check_diag(obs, ref_obs)


@pytest.mark.gpu
def test_fp32_bilinear():
    """float32 storage at test_fp32_tolerance's tolerance against the float64 reference."""
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=46, nx=90, nmem=50, nvars=2, ntimes=2, nobs=300, cutoff_km=2500.0, seed=311, offtime=True)
    ref_post, _, _ = B.ensrf_update(case, loc='GC')
    state, obs = build_objects(case, EnsembleState, Observation)
    post32, _ = EnSRF(state, obs, verbose=False, loc='GC', dtype='f32', forward_operator='bilinear').update()
    p32 = post32.to_vect()
    m32, mref = p32.mean(axis=1), ref_post.mean(axis=1)
    assert np.abs(m32 - mref).max() <= 1e-5 * np.abs(mref).max()
    spread = (ref_post - mref[:, None]).std()
    assert np.abs((p32 - m32[:, None]) - (ref_post - mref[:, None])).max() <= 1e-3 * spread


@pytest.mark.gpu
def test_obs_near_grid_points_assimilate_under_raise_policy():
    import efa_xray_b200 as pkg
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(**_C50)
    rng = np.random.default_rng(4)
    k = rng.choice(case.nobs, 20, replace=False)
    ny, nx = case.lat2d.shape
    gy, gx = rng.integers(1, ny - 1, 20), rng.integers(0, nx, 20)
    lat, lon = case.ob_lat.copy(), case.ob_lon.copy()
    lat[k] = case.lat2d[gy, gx] + rng.uniform(-0.004, 0.004, 20)          # within 1 km
    lon[k] = case.lon2d[gy, gx] + rng.uniform(-0.004, 0.004, 20)
    case = dataclasses.replace(case, ob_lat=lat, ob_lon=lon)
    assert pkg.EXACT_MATCH_POLICY == 'raise'
    state, obs = build_objects(case, EnsembleState, Observation)
    with pytest.raises(IndexError):
        EnSRF(state, obs, verbose=False, loc='GC').update()
    ref_post, ref_obs, prior = B.ensrf_update(case, loc='GC')
    state, obs = build_objects(case, EnsembleState, Observation)
    post, _ = EnSRF(state, obs, verbose=False, loc='GC', forward_operator='bilinear').update()
    _check_post(post.to_vect(), ref_post, prior)
    _check_diag(obs, ref_obs)


@pytest.mark.gpu
def test_outside_ob_raises_and_leaves_obs_and_prior_alone():
    EnsembleState, Observation, EnSRF = _api()
    from efa_xray_b200.assimilation.assimilation import update
    lat2d, lon2d = _mesh(np.linspace(20.0, 60.0, 25), np.linspace(-130.0, -60.0, 48))
    case = _regrid(make_case(**_C50), lat2d, lon2d, seed=5)
    lat, lon = case.ob_lat.copy(), case.ob_lon.copy()
    lat[[3, 40]] = [10.0, 45.0]
    lon[[3, 40]] = [-100.0, -40.0]
    case = dataclasses.replace(case, ob_lat=lat, ob_lon=lon)
    state, obs = build_objects(case, EnsembleState, Observation)
    prior = state.to_vect().copy()
    for run in (lambda: EnSRF(state, obs, verbose=False, loc='GC', forward_operator='bilinear').update(),
                lambda: update(state, obs, loc='GC', forward_operator='bilinear')):
        with pytest.raises(ValueError, match='2 observation'):
            run()
        assert all(o.prior_mean is None and o.post_mean is None and not o.assimilated for o in obs)
        np.testing.assert_array_equal(state.to_vect(), prior)


def _engine_inputs(case):
    import torch
    dev = torch.device('cuda', 0)
    ny, nx = case.lat2d.shape
    nt = len(case.times)
    tlo, thi, wlo, whi, _ = engine.time_weights(case.times, case.ob_time, swapped=False)
    obs = engine.ObsArrays(value=case.ob_value, error=case.ob_error, lat=case.ob_lat, lon=case.ob_lon,
                           halfwidth=case.ob_halfwidth, assimilate=case.ob_assimilate.astype(np.uint8),
                           row0=(case.ob_var * nt + tlo) * (ny * nx), row1=(case.ob_var * nt + thi) * (ny * nx),
                           tw0=wlo, tw1=whi)
    return dev, nt * len(case.varnames), engine.GridTables(case.lat2d, case.lon2d, dev), obs


@pytest.mark.gpu
def test_host_band_pipeline_and_shards_match_device_analysis():
    """engine.analysis_host (pinned buffer, several bands) and 2, 4 and 8 logical latitude-band shards
    (engine.analysis_device(band=...)) against the unsharded device analysis, all with the bilinear operator."""
    import torch
    from efa_xray_b200 import sharding
    case = make_case(ny=181, nx=360, nmem=40, nvars=2, ntimes=2, nobs=2000, cutoff_km=2500.0, seed=321, offtime=True)
    dev, nlev, grid, obs = _engine_inputs(case)
    ny, nx = case.lat2d.shape
    prior = case.to_vect()
    X = torch.as_tensor(prior).to(dev)
    engine.ob_priors(X, grid, obs, 'f64')
    assert grid._bilinear is None                             # the reference operator builds no bilinear tables
    Y, nout = engine.ob_priors(X, grid, obs, 'f64', forward_operator='bilinear')
    ye = B.ob_priors(prior, case.lat2d, case.lon2d, case.times, case.ob_var, case.ob_time, case.ob_lat, case.ob_lon)
    assert int(nout.item()) == 0
    np.testing.assert_allclose(Y.cpu().numpy(), ye, rtol=1e-12)
    res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, forward_operator='bilinear')
    ref = X.cpu().numpy()
    assert res.n_outside == 0 and res.assimilated.all()
    assert grid._bilinear is not None
    inc = np.abs(ref - prior).max()
    host = torch.from_numpy(prior.copy()).pin_memory()
    out = torch.empty_like(host).pin_memory()
    hres = engine.analysis_host(host, nlev, None, None, obs, engine.LOC_GC, device=dev, grid=grid, out=out,
                                forward_operator='bilinear')
    assert hres.n_outside == 0
    assert np.abs(out.numpy() - ref).max() <= 1e-9 * inc
    np.testing.assert_array_equal(host.numpy(), prior)
    Xfull = torch.as_tensor(prior).to(dev)
    nens = Xfull.shape[1]
    work = sharding.estimate_row_work(case.lat2d, case.lon2d, obs.lat, obs.lon, 2.0 * obs.halfwidth, obs.assimilate)
    for n in (2, 4, 8):
        bands = sharding.partition_bands(work, n)
        shards = [sharding.band_view(Xfull, nlev, ny, nx, a, b).contiguous().reshape(-1, nens) for a, b in bands]
        parts = [engine.ob_priors(Xs, grid, obs, 'f64', nlev=nlev, band=bd, forward_operator='bilinear')[0]
                 for Xs, bd in zip(shards, bands)]
        Ysum = torch.stack(parts).sum(dim=0)
        for Xs, bd in zip(shards, bands):
            engine.analysis_device(Xs, nlev, grid, obs, engine.LOC_GC, band=bd, Y=Ysum, forward_operator='bilinear')
        got = torch.empty_like(Xfull)
        for Xs, (a, b) in zip(shards, bands):
            sharding.band_view(got, nlev, ny, nx, a, b).copy_(Xs.view(nlev, b - a, nx, nens))
        assert np.abs(got.cpu().numpy() - ref).max() <= 1e-9 * inc, n


@pytest.mark.gpu
def test_diagnostics_interpolate_and_estimate():
    from efa_xray_b200.postprocess.postprocess import obs_assimilation_statistics, ob_estimates
    EnsembleState, Observation, EnSRF = _api()
    case = make_case(ny=25, nx=48, nmem=20, nvars=2, ntimes=3, nobs=30, cutoff_km=2500.0, seed=331, offtime=True)
    state, obs = build_objects(case, EnsembleState, Observation)
    post, _ = EnSRF(state, obs, verbose=False, loc='GC', forward_operator='bilinear').update()
    args = (case.lat2d, case.lon2d, case.times, case.ob_var, case.ob_time, case.ob_lat, case.ob_lon)
    ye_prior, ye_post = B.ob_priors(case.to_vect(), *args), B.ob_priors(post.to_vect(), *args)
    df = obs_assimilation_statistics(state, post, obs, forward_operator='bilinear')
    np.testing.assert_allclose(df['prior mean'], ye_prior.mean(axis=1), rtol=1e-12)
    np.testing.assert_allclose(df['prior variance'], ye_prior.var(axis=1), rtol=1e-10)
    np.testing.assert_allclose(df['post mean'], ye_post.mean(axis=1), rtol=1e-12)
    np.testing.assert_allclose(df['post variance'], ye_post.var(axis=1), rtol=1e-10)
    for k in (0, 7, 19):
        o = obs[k]
        np.testing.assert_allclose(state.interpolate(o.obtype, o.time, o.lat, o.lon, forward_operator='bilinear'),
                                   ye_prior[k], rtol=1e-12)
        np.testing.assert_allclose(o.estimate(state, forward_operator='bilinear'), ye_prior[k], rtol=1e-12)
        np.testing.assert_array_equal(o.estimate(state, forward_operator='reference'), o.estimate(state))
        np.testing.assert_array_equal(state.interpolate(o.obtype, o.time, o.lat, o.lon, forward_operator='reference'),
                                      state.interpolate(o.obtype, o.time, o.lat, o.lon))
    np.testing.assert_array_equal(ob_estimates(state, obs, forward_operator='reference'), ob_estimates(state, obs))
    a = obs_assimilation_statistics(state, post, obs, forward_operator='reference')
    b = obs_assimilation_statistics(state, post, obs)
    assert a.equals(b)
    with pytest.raises(ValueError):
        state.interpolate(obs[0].obtype, obs[0].time, 95.0, 10.0, forward_operator='bilinear')


@pytest.mark.gpu
def test_config3_full_size_bilinear():
    """BASELINE config 3 in full (100 members, 721x1440x3, 1e5 obs): every ob prior against the vectorised reference,
    and one analysis with no ob outside the grid and a finite result."""
    import torch
    from efa_xray_b200.synth import CONFIGS
    case = make_case(cutoff_km=2000.0, seed=0, **CONFIGS['config3'])
    dev, nlev, grid, obs = _engine_inputs(case)
    prior_h = case.to_vect()
    X = torch.as_tensor(prior_h).to(dev)
    Y, nout = engine.ob_priors(X, grid, obs, 'f64', forward_operator='bilinear')
    assert int(nout.item()) == 0
    ridx, rw, rout = B.stencil(case.lat2d, case.lon2d, case.ob_lat, case.ob_lon)
    assert not rout.any()
    want = np.concatenate([B.ob_priors(prior_h, case.lat2d, case.lon2d, case.times, case.ob_var[a:a + 10000],
                                       case.ob_time[a:a + 10000], case.ob_lat[a:a + 10000], case.ob_lon[a:a + 10000],
                                       idx4=ridx[a:a + 10000], w4=rw[a:a + 10000])
                           for a in range(0, case.nobs, 10000)])
    got = Y.cpu().numpy()
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    del case, Y
    res = engine.analysis_device(X, nlev, grid, obs, engine.LOC_GC, forward_operator='bilinear')
    assert res.n_outside == 0 and res.assimilated.all()
    assert bool(torch.isfinite(X).all())
