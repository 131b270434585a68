"""Numpy reference of the bilinear forward operator (DESIGN.md section 4.8), written independently of the product:
np.searchsorted on the axes of rectilinear grids, a brute-force great-circle search and Newton's method for the
inverse bilinear map on curvilinear grids, and time weights from np.interp.  The reference analysis puts these ob
priors into the xbm / Xbp of format_prior_state and runs the unchanged CPU oracle's serial loop
(oracle/ensrf_oracle.py, which is not modified).

TEST INFRASTRUCTURE, NOT PRODUCT: the GPU operator is checked against this module."""
import numpy as np

from oracle import ensrf_oracle as O

IN_TOL = 1e-10


def classify(lat2d, lon2d):
    """('rect', lat_y, lon_x, periodic) or ('curv', None, None, False), as DESIGN.md section 4.8 states the rule."""
    lat2d, lon2d = np.asarray(lat2d, dtype=np.float64), np.asarray(lon2d, dtype=np.float64)
    rows_equal = all(np.array_equal(lat2d[:, x], lat2d[:, 0]) for x in range(lat2d.shape[1]))
    cols_equal = all(np.array_equal(lon2d[y], lon2d[0]) for y in range(lon2d.shape[0]))
    if not (rows_equal and cols_equal):
        return 'curv', None, None, False
    lat_y, lon_x = lat2d[:, 0], lon2d[0]
    if not (np.all(lat_y[1:] > lat_y[:-1]) or np.all(lat_y[1:] < lat_y[:-1])):
        return 'curv', None, None, False
    steps = (lon_x[1:] - lon_x[:-1]) % 360.0
    if steps.min() <= 0.0 or steps.max() >= 360.0 or steps.sum() >= 360.0:
        return 'curv', None, None, False
    return 'rect', lat_y, lon_x, bool(360.0 - steps.sum() <= steps.max() * (1.0 + 1e-9))


def stencil_rect(lat_y, lon_x, periodic, ob_lat, ob_lon):
    """(idx4 [nobs, 4], w4 [nobs, 4], outside [nobs]) on a rectilinear grid."""
    lat_y, lon_x = np.asarray(lat_y, dtype=np.float64), np.asarray(lon_x, dtype=np.float64)
    ob_lat, ob_lon = np.asarray(ob_lat, dtype=np.float64), np.asarray(ob_lon, dtype=np.float64)
    ny, nx = len(lat_y), len(lon_x)
    L = lon_x[0] + np.concatenate(([0.0], np.cumsum((lon_x[1:] - lon_x[:-1]) % 360.0)))
    lam = L[0] + np.mod(ob_lon - L[0], 360.0)
    # columns: closing cell (nx-1 -> 0) past the last column of a periodic grid
    i = np.clip(np.searchsorted(L[:nx - 1], lam, side='right') - 1, 0, nx - 2)
    seam = lam > L[-1]
    i = np.where(seam, nx - 1, i)
    i1 = np.where(seam, 0, i + 1)
    xl = L[i]
    xr = np.where(seam, L[0] + 360.0, L[np.minimum(i + 1, nx - 1)])
    # rows on the ascending axis; a descending axis is the ascending one read backwards
    desc = lat_y[-1] < lat_y[0]
    la = lat_y[::-1] if desc else lat_y
    ja = np.clip(np.searchsorted(la, ob_lat, side='left') - 1, 0, ny - 2)   # lowest cell with la[j] <= phi <= la[j+1]
    if desc:
        # ascending cell ja is descending cell ny-2-ja; the lowest descending j wins a tie, i.e. the highest ja
        ja = np.clip(np.searchsorted(la, ob_lat, side='right') - 1, 0, ny - 2)
        j = ny - 2 - ja
    else:
        j = ja
    outside = ~((ob_lat >= la[0]) & (ob_lat <= la[-1])) | np.isnan(lam)
    if not periodic:
        outside |= seam
    s = (lam - xl) / (xr - xl)
    t = (ob_lat - lat_y[j]) / (lat_y[j + 1] - lat_y[j])
    idx4 = np.stack([j * nx + i, j * nx + i1, (j + 1) * nx + i, (j + 1) * nx + i1], axis=1).astype(np.int64)
    w4 = np.stack([(1 - s) * (1 - t), s * (1 - t), (1 - s) * t, s * t], axis=1)
    idx4[outside] = 0
    w4[outside] = 0.0
    return idx4, w4, outside


def _unit(lat, lon):
    p, l = np.radians(lat), np.radians(lon)
    return np.stack([np.cos(p) * np.cos(l), np.cos(p) * np.sin(l), np.sin(p)], axis=-1)


def _wrap180(d):
    d = np.fmod(d, 360.0)
    return np.where(d > 180.0, d - 360.0, np.where(d < -180.0, d + 360.0, d))


def _newton_cell(lat2d, lon2d, y, x, ob_lat, ob_lon):
    """Inverse bilinear (s, t) of every ob in cell (y, x) (arrays) by Newton's method, and whether it converged."""
    cx = [_wrap180(lon2d[y + a, x + b] - ob_lon) for a, b in ((0, 0), (0, 1), (1, 0), (1, 1))]
    cy = [lat2d[y + a, x + b] - ob_lat for a, b in ((0, 0), (0, 1), (1, 0), (1, 1))]
    s = np.full(len(ob_lat), 0.5)
    t = np.full(len(ob_lat), 0.5)
    for _ in range(40):
        w = [(1 - s) * (1 - t), s * (1 - t), (1 - s) * t, s * t]
        fx = sum(wi * c for wi, c in zip(w, cx))
        fy = sum(wi * c for wi, c in zip(w, cy))
        # Jacobian d(fx, fy) / d(s, t)
        xs = (1 - t) * (cx[1] - cx[0]) + t * (cx[3] - cx[2])
        ys = (1 - t) * (cy[1] - cy[0]) + t * (cy[3] - cy[2])
        xt = (1 - s) * (cx[2] - cx[0]) + s * (cx[3] - cx[1])
        yt = (1 - s) * (cy[2] - cy[0]) + s * (cy[3] - cy[1])
        det = xs * yt - xt * ys
        with np.errstate(divide='ignore', invalid='ignore'):
            ds = (fx * yt - fy * xt) / det
            dt = (xs * fy - ys * fx) / det
        s, t = s - ds, t - dt
    w = [(1 - s) * (1 - t), s * (1 - t), (1 - s) * t, s * t]
    res = np.hypot(sum(wi * c for wi, c in zip(w, cx)), sum(wi * c for wi, c in zip(w, cy)))
    size = np.hypot(cx[3] - cx[0], cy[3] - cy[0])
    ok = np.isfinite(s) & np.isfinite(t) & (res <= 1e-9 * size)
    return s, t, ok


def stencil_curv(lat2d, lon2d, ob_lat, ob_lon, chunk=2048):
    """(idx4, w4, outside) on any 2-D grid, by the curvilinear rule: nearest point by great-circle distance, the cells
    with it as a corner, then the rest of the 4x4-cell block around it."""
    lat2d, lon2d = np.asarray(lat2d, dtype=np.float64), np.asarray(lon2d, dtype=np.float64)
    ob_lat, ob_lon = np.asarray(ob_lat, dtype=np.float64), np.asarray(ob_lon, dtype=np.float64)
    ny, nx = lat2d.shape
    ug = _unit(lat2d.ravel(), lon2d.ravel())
    uo = _unit(ob_lat, ob_lon)
    best = np.concatenate([np.argmax(uo[a:a + chunk] @ ug.T, axis=1) for a in range(0, len(ob_lat), chunk)])
    py, px = best // nx, best % nx
    nobs = len(ob_lat)
    idx4 = np.zeros((nobs, 4), dtype=np.int64)
    w4 = np.zeros((nobs, 4))
    found = np.zeros(nobs, dtype=bool)
    inner = [(dy, dx) for dy in (-1, 0) for dx in (-1, 0)]
    outer = [(dy, dx) for dy in range(-2, 2) for dx in range(-2, 2) if (dy, dx) not in inner]
    for dy, dx in inner + outer:
        y, x = py + dy, px + dx
        todo = ~found & (y >= 0) & (y <= ny - 2) & (x >= 0) & (x <= nx - 2)
        if not todo.any():
            continue
        k = np.flatnonzero(todo)
        s, t, ok = _newton_cell(lat2d, lon2d, y[k], x[k], ob_lat[k], ob_lon[k])
        hit = ok & (s >= -IN_TOL) & (s <= 1 + IN_TOL) & (t >= -IN_TOL) & (t <= 1 + IN_TOL)
        k, s, t = k[hit], np.clip(s[hit], 0, 1), np.clip(t[hit], 0, 1)
        yy, xx = y[k], x[k]
        idx4[k] = np.stack([yy * nx + xx, yy * nx + xx + 1, (yy + 1) * nx + xx, (yy + 1) * nx + xx + 1], axis=1)
        w4[k] = np.stack([(1 - s) * (1 - t), s * (1 - t), (1 - s) * t, s * t], axis=1)
        found[k] = True
    return idx4, w4, ~found


def stencil(lat2d, lon2d, ob_lat, ob_lon):
    kind, lat_y, lon_x, periodic = classify(lat2d, lon2d)
    if kind == 'rect':
        return stencil_rect(lat_y, lon_x, periodic, ob_lat, ob_lon)
    return stencil_curv(lat2d, lon2d, ob_lat, ob_lon)


def time_levels(valid_times, ob_times):
    """(lo, hi, w_lo, w_hi) of the correctly oriented linear time weights, from np.interp."""
    v = (np.asarray(valid_times).astype('datetime64[ns]') - np.datetime64(0, 'ns')) / np.timedelta64(1, 's')
    t = (np.asarray(ob_times).astype('datetime64[ns]') - np.datetime64(0, 'ns')) / np.timedelta64(1, 's')
    assert ((t >= v[0]) & (t <= v[-1])).all()
    f = np.interp(t, v, np.arange(len(v), dtype=np.float64))
    lo = np.floor(f).astype(np.int64)
    w_hi = f - lo
    hi = np.minimum(lo + 1, len(v) - 1)
    return lo, hi, 1.0 - w_hi, w_hi


def ob_priors(vect, lat2d, lon2d, times, ob_var, ob_time, ob_lat, ob_lon, idx4=None, w4=None):
    """H x [nobs, nens] of the state vector vect [nvar * nt * ny * nx, nens] (rows var -> time -> y -> x)."""
    ny, nx = np.shape(lat2d)
    nt = len(times)
    if idx4 is None:
        idx4, w4, outside = stencil(lat2d, lon2d, ob_lat, ob_lon)
        assert not outside.any()
    lo, hi, wlo, whi = time_levels(times, ob_time)
    out = np.zeros((len(ob_lat), vect.shape[1]))
    for lev, tw in ((lo, wlo), (hi, whi)):
        base = (np.asarray(ob_var) * nt + lev) * (ny * nx)
        for p in range(4):
            out += (tw * w4[:, p])[:, None] * vect[base + idx4[:, p]]
    return out


def ensrf_update(case, loc='GC', inflation=None, obs=None):
    """(posterior state vector, obs) of the EnSRF with the bilinear operator: the oracle's format_prior_state with
    these ob priors, then its unchanged serial loop.  `obs` (oracle obs) defaults to those of the case."""
    state = O.State.from_case(case)
    obs = O.obs_from_case(case) if obs is None else obs
    if inflation is not None:
        state = O.inflate_state(state, inflation)
    prior = state.to_vect()
    ye = ob_priors(prior, case.lat2d, case.lon2d, case.times, case.ob_var, case.ob_time, case.ob_lat, case.ob_lon)
    xbm = prior.mean(axis=1)
    ym = ye.mean(axis=1)
    xam = np.hstack((xbm, ym))
    Xap = np.vstack((prior - xbm[:, None], ye - ym[:, None]))
    xam, Xap = O.ensrf_loop(state, obs, xam, Xap, loc=loc)
    return (xam[:, None] + Xap)[:state.nstate()], obs, prior
