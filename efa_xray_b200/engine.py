"""Array-level driver of the serial EnSRF analysis on B200.

This is the host side between the reference-shaped Python API (efa_xray_b200.assimilation) and the C ABI
(include/efa_xray_b200.h).  torch is used for device memory, streams, events and (multi-GPU)
torch.distributed only; every arithmetic step is a kernel of libefa_xray_b200.

Sequence (reference: assimilation/ensrf.py:33-151, assimilation/assimilation.py:120-171):
    upload  ->  [inflate]  ->  ob priors H.x  ->  mean/perturbation split  ->  obs-space serial solve
            ->  state sweep (per latitude band)  ->  recombine  ->  [relax]  ->  download
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from . import _lib

LOC_NONE, LOC_GC = 0, 1


@dataclass
class ObsArrays:
    """Structure-of-arrays view of a list of Observation objects (observation/observation.py:18-36)."""
    value: np.ndarray
    error: np.ndarray            # variance
    lat: np.ndarray
    lon: np.ndarray
    halfwidth: np.ndarray        # km; ignored when loc_mode == LOC_NONE
    assimilate: np.ndarray       # uint8
    row0: np.ndarray             # first state row of (variable, lower time level)
    row1: np.ndarray             # first state row of (variable, upper time level)
    tw0: np.ndarray              # time weights of the two levels (state/ensemble.py:202-224)
    tw1: np.ndarray
    # outlier threshold per ob (inf: not checked); empty, the default: no check at all (DESIGN.md 4.7).  Every field
    # is a per-ob array, so a slice of every field is the ObsArrays of those obs.
    threshold: np.ndarray = field(default_factory=lambda: np.zeros(0))

    @property
    def qc(self):
        return len(self.threshold) > 0

    @property
    def nobs(self):
        return int(self.value.shape[0])


@dataclass
class AnalysisResult:
    prior_mean: np.ndarray
    prior_var: np.ndarray
    post_mean: np.ndarray        # NaN where the ob was not assimilated
    post_var: np.ndarray
    assimilated: np.ndarray      # bool
    n_exact: int = 0             # obs within 1 km of a selected grid point
    n_outside: int = 0           # obs outside the grid (forward_operator='bilinear')
    state_pairs: int = 0         # sum_k |F_s(k)|   (state rows with non-zero weight, all levels)
    obs_pairs: int = 0           # sum_k |F_o(k)|
    obs_solve: str = ''          # which obs-space solve ran: 'replicated' | 'distributed(block=b)' | 'single'
    ms: dict = field(default_factory=dict)


def time_weights(valid_times, ob_times, swapped=True):
    """Vectorised restatement of the time-weight logic of EnsembleState.interpolate
    (state/ensemble.py:202-224), including its swapped linear weights.  Returns
    (tlo, thi, wlo, whi, outside) with weights attached to time indices tlo = lastdex-1, thi = lastdex.
    swapped=False gives the correctly oriented linear weights of forward_operator='bilinear':
    whi = (t - t_lo) / (t_hi - t_lo)."""
    valids = np.asarray(valid_times).astype('datetime64[ns]')
    t = np.asarray(ob_times).astype('datetime64[ns]')
    outside = (t < valids[0]) | (t > valids[-1])
    lastdex = np.searchsorted(valids, t, side='left')            # first index with valids >= t
    lastdex = np.clip(lastdex, 0, len(valids) - 1)
    exact = valids[lastdex] == t
    lo = np.maximum(lastdex - 1, 0)
    totsec = np.abs((valids[lastdex] - valids[lo]) / np.timedelta64(1, 's'))
    if swapped:
        thissec = np.abs((t - valids[lastdex]) / np.timedelta64(1, 's'))
    else:
        thissec = np.abs((t - valids[lo]) / np.timedelta64(1, 's'))
    with np.errstate(divide='ignore', invalid='ignore'):
        frac = thissec.astype(np.float64) / totsec
    whi = np.where(exact, 1.0, frac)                              # timeweights[lastdex]
    wlo = np.where(exact, 0.0, 1.0 - frac)                        # timeweights[lastdex-1]
    return lo.astype(np.int64), lastdex.astype(np.int64), wlo, whi, outside


FORWARD_OPERATORS = ('reference', 'bilinear')


def check_forward_operator(forward_operator, lat_ndim):
    """Raise ValueError unless forward_operator is one of FORWARD_OPERATORS and usable on a state whose lat/lon
    coordinates have `lat_ndim` dimensions ('bilinear' needs 2-D lat/lon)."""
    if not isinstance(forward_operator, str) or forward_operator not in FORWARD_OPERATORS:
        raise ValueError('forward_operator must be one of %r, got %r' % (FORWARD_OPERATORS, forward_operator))
    if forward_operator == 'bilinear' and lat_ndim != 2:
        raise ValueError("forward_operator='bilinear' needs 2-D lat(y, x) / lon(y, x) coordinates; this state's "
                         "lat/lon are %d-D" % lat_ndim)


def bilinear_axes(lat2d, lon2d):
    """Which path of the bilinear forward operator serves a 2-D grid (DESIGN.md section 4.8), pure numpy:
    ('rect', lat_y, lon_unwrapped, periodic) when lat depends on y only and is strictly monotone, and lon depends on x
    only and is strictly increasing after unwrapping (steps d_i = (lon_x[i+1] - lon_x[i]) mod 360 in (0, 360), span
    S = sum d_i below 360); periodic when the wrap gap 360 - S is at most max d_i (1 + 1e-9).  Otherwise
    ('curv', None, None, False)."""
    lat2d = np.asarray(lat2d, dtype=np.float64)
    lon2d = np.asarray(lon2d, dtype=np.float64)
    if lat2d.ndim != 2 or lat2d.shape != lon2d.shape:
        raise ValueError('the bilinear forward operator needs 2-D lat(y, x) / lon(y, x) of one shape, got %r and %r'
                         % (lat2d.shape, lon2d.shape))
    if lat2d.shape[0] < 2 or lat2d.shape[1] < 2:
        raise ValueError('the bilinear forward operator needs at least 2 x 2 grid points, got %r' % (lat2d.shape,))
    curv = ('curv', None, None, False)
    if not ((lat2d == lat2d[:, :1]).all() and (lon2d == lon2d[:1, :]).all()):
        return curv
    lat_y, lon_x = lat2d[:, 0], lon2d[0, :]
    dlat = np.diff(lat_y)
    if not ((dlat > 0).all() or (dlat < 0).all()):
        return curv
    d = np.mod(np.diff(lon_x), 360.0)
    span = float(np.sum(d))
    if not ((d > 0).all() and (d < 360.0).all() and span < 360.0):
        return curv
    lon_u = lon_x[0] + np.concatenate(([0.0], np.cumsum(d)))
    periodic = bool(360.0 - span <= d.max() * (1.0 + 1e-9))
    return 'rect', np.ascontiguousarray(lat_y), lon_u, periodic


def _torch():
    import torch
    return torch


def _dev_f64(a, device):
    torch = _torch()
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(device)


class GridTables:
    """Device-resident geometry of the (ny, nx) grid: lat/lon, the pseudo-metric tables of
    nearest_points (state/ensemble.py:160-163, computed with numpy so that ties fall where they do on the
    host) and unit vectors for great-circle distances."""

    def __init__(self, lat2d, lon2d, device, ny=None):
        """lat2d / lon2d: 2-D (y, x) coordinates, or 1-D arrays of nx points with `ny` given: the reference's 1-D
        lat/lon branch (state/ensemble.py:185-192, assimilation/ensrf.py:110-111), where localisation depends on x
        only and the forward operator reads the state at (y, x) = (n, n) for a point index n."""
        torch = _torch()
        lat2d = np.ascontiguousarray(lat2d, dtype=np.float64)
        lon2d = np.ascontiguousarray(lon2d, dtype=np.float64)
        self.diag = lat2d.ndim == 1
        if self.diag:
            assert ny is not None and lat2d.shape == lon2d.shape
            if ny < lat2d.shape[0]:
                raise IndexError('1-D lat/lon state: the forward operator indexes y with the point index '
                                 '(state/ensemble.py:226), which needs ny >= nx (ny=%d, nx=%d)' % (ny, lat2d.shape[0]))
            self.lat1 = _dev_f64(lat2d, device)
            self.lon1 = _dev_f64(lon2d, device)
            self.sinlat1 = _dev_f64(np.sin(np.radians(lat2d)), device)
            self.coslon1 = _dev_f64(np.cos(np.radians(lon2d)), device)
            self.u1 = torch.empty((3, lat2d.shape[0]), dtype=torch.float64, device=device)
            _lib.call('exb_grid_unitvec', _lib.ptr(self.lat1), _lib.ptr(self.lon1), lat2d.shape[0], _lib.ptr(self.u1),
                      _lib.stream_ptr())
            lat2d = np.ascontiguousarray(np.broadcast_to(lat2d[None, :], (ny, lat2d.shape[0])))
            lon2d = np.ascontiguousarray(np.broadcast_to(lon2d[None, :], (ny, lon2d.shape[0])))
        assert lat2d.ndim == 2 and lat2d.shape == lon2d.shape, '2-D lat(y,x)/lon(y,x) or 1-D lat(x)/lon(x) required'
        self.ny, self.nx = lat2d.shape
        self.npts = self.ny * self.nx
        self.device = device
        self.lat = _dev_f64(lat2d.ravel(), device)
        self.lon = _dev_f64(lon2d.ravel(), device)
        self.sinlat = _dev_f64(np.sin(np.radians(lat2d)).ravel(), device)
        self.coslon = _dev_f64(np.cos(np.radians(lon2d)).ravel(), device)
        # rectilinear grid (lat = f(y), lon = f(x)): the nearest-point search separates (O(ny+nx) per ob)
        self.rectilinear = bool((lat2d == lat2d[:, :1]).all() and (lon2d == lon2d[:1, :]).all()) and not self.diag
        if self.rectilinear:
            self.lat_y = _dev_f64(lat2d[:, 0], device)
            self.lon_x = _dev_f64(lon2d[0, :], device)
            self.sinlat_y = _dev_f64(np.sin(np.radians(lat2d[:, 0])), device)
            self.coslon_x = _dev_f64(np.cos(np.radians(lon2d[0, :])), device)
        self.u = torch.empty((3, self.npts), dtype=torch.float64, device=device)
        _lib.call('exb_grid_unitvec', _lib.ptr(self.lat), _lib.ptr(self.lon), self.npts, _lib.ptr(self.u),
                  _lib.stream_ptr())
        self._host_latlon = None if self.diag else (lat2d, lon2d)
        self._bilinear = None

    def bilinear_tables(self):
        """(path, device tables) of the bilinear forward operator, built on first use: ('rect', (lat_y,
        unwrapped lon_x, periodic)) or ('curv', None), from bilinear_axes."""
        if self._bilinear is None:
            if self.diag:
                raise ValueError("forward_operator='bilinear' needs 2-D lat(y, x) / lon(y, x) coordinates")
            kind, lat_y, lon_u, periodic = bilinear_axes(*self._host_latlon)
            tables = (_dev_f64(lat_y, self.device), _dev_f64(lon_u, self.device), int(periodic)) \
                if kind == 'rect' else None
            self._bilinear = (kind, tables)
        return self._bilinear


def stencil_bilinear(grid: GridTables, d_lat, d_lon, force_curvilinear=False):
    """Bilinear stencils (DESIGN.md section 4.8) of the obs at device coordinates d_lat / d_lon -> device tensors
    idx4 [nobs,4] int64, w4 [nobs,4] float64 and the int32 count of obs outside the grid (idx 0 / w 0 there).
    force_curvilinear runs the curvilinear path on any 2-D grid."""
    torch = _torch()
    dev = grid.device
    kind, tables = grid.bilinear_tables()
    nobs = d_lat.shape[0]
    idx4 = torch.empty((nobs, 4), dtype=torch.int64, device=dev)
    w4 = torch.empty((nobs, 4), dtype=torch.float64, device=dev)
    nout = torch.empty(1, dtype=torch.int32, device=dev)
    if kind == 'rect' and not force_curvilinear:
        lat_y, lon_u, periodic = tables
        _lib.call('exb_stencil_bilinear_rect', _lib.ptr(lat_y), _lib.ptr(lon_u), grid.ny, grid.nx, periodic,
                  _lib.ptr(d_lat), _lib.ptr(d_lon), nobs, _lib.ptr(idx4), _lib.ptr(w4), _lib.ptr(nout),
                  _lib.stream_ptr())
    else:
        _lib.call('exb_stencil_bilinear_curv', _lib.ptr(grid.u), _lib.ptr(grid.lat), _lib.ptr(grid.lon), grid.ny,
                  grid.nx, _lib.ptr(d_lat), _lib.ptr(d_lon), nobs, _lib.ptr(idx4), _lib.ptr(w4), _lib.ptr(nout),
                  _lib.stream_ptr())
    return idx4, w4, nout


def stencil_search(grid: GridTables, ob_lat, ob_lon, force_general=False, dev_tables=None):
    """4 nearest points (pseudo-metric) and inverse-distance weights for every ob -> device tensors
    idx4 [nobs,4] int64, w4 [nobs,4] float64, and the number of obs within 1 km of a selected point.
    dev_tables = (lat, lon, sin(lat), cos(lon)) already on the device (upload_obs) saves four small uploads."""
    torch = _torch()
    dev = grid.device
    if dev_tables is None:
        ob_lat = np.ascontiguousarray(ob_lat, dtype=np.float64)
        ob_lon = np.ascontiguousarray(ob_lon, dtype=np.float64)
        d_lat, d_lon = _dev_f64(ob_lat, dev), _dev_f64(ob_lon, dev)
        d_sl = _dev_f64(np.sin(np.radians(ob_lat)), dev)
        d_cl = _dev_f64(np.cos(np.radians(ob_lon)), dev)
    else:
        d_lat, d_lon, d_sl, d_cl = dev_tables
    nobs = d_lat.shape[0]
    idx4 = torch.empty((nobs, 4), dtype=torch.int64, device=dev)
    w4 = torch.empty((nobs, 4), dtype=torch.float64, device=dev)
    nex = torch.zeros(1, dtype=torch.int32, device=dev)
    if grid.diag:                    # 1-D point list: the search runs over the nx points, idx4 are point indices
        _lib.call('exb_stencil_search', _lib.ptr(grid.sinlat1), _lib.ptr(grid.coslon1), _lib.ptr(grid.lat1),
                  _lib.ptr(grid.lon1), grid.nx, _lib.ptr(d_sl), _lib.ptr(d_cl), _lib.ptr(d_lat), _lib.ptr(d_lon),
                  nobs, _lib.ptr(idx4), _lib.ptr(w4), _lib.ptr(nex), _lib.stream_ptr())
    elif grid.rectilinear and not force_general:
        _lib.call('exb_stencil_search_rect', _lib.ptr(grid.sinlat_y), _lib.ptr(grid.coslon_x), _lib.ptr(grid.lat_y),
                  _lib.ptr(grid.lon_x), grid.ny, grid.nx, _lib.ptr(d_sl), _lib.ptr(d_cl), _lib.ptr(d_lat),
                  _lib.ptr(d_lon), nobs, _lib.ptr(idx4), _lib.ptr(w4), _lib.ptr(nex), _lib.stream_ptr())
    else:
        _lib.call('exb_stencil_search', _lib.ptr(grid.sinlat), _lib.ptr(grid.coslon), _lib.ptr(grid.lat),
                  _lib.ptr(grid.lon), grid.npts, _lib.ptr(d_sl), _lib.ptr(d_cl), _lib.ptr(d_lat), _lib.ptr(d_lon),
                  nobs, _lib.ptr(idx4), _lib.ptr(w4), _lib.ptr(nex), _lib.stream_ptr())
    return idx4, w4, nex


def pseudo_distance_order(grid: GridTables, lat, lon, npt):
    """Flat indices of the npt grid points with the smallest pseudo-distance to (lat, lon), ordered by (distance,
    flat index): nearest_points for any npt (state/ensemble.py:152-168)."""
    torch = _torch()
    n = grid.nx if grid.diag else grid.npts
    d2 = torch.empty(n, dtype=torch.float64, device=grid.device)
    _lib.call('exb_pseudo_distance', _lib.ptr(grid.sinlat1 if grid.diag else grid.sinlat),
              _lib.ptr(grid.coslon1 if grid.diag else grid.coslon), n,
              float(np.sin(np.radians(lat))), float(np.cos(np.radians(lon))), _lib.ptr(d2), _lib.stream_ptr())
    order = torch.sort(d2, stable=True).indices[:npt]
    return order.cpu().numpy()


def ob_priors(X, grid: GridTables, obs: ObsArrays, sfx, nlev=None, band=None, group=None, obs_dev=None,
              forward_operator='reference'):
    """(Y[nobs, nens] = H X for all obs, device int32 counter) (compute_ob_priors, assimilation/assimilation.py:36-49).
    The counter is the number of obs within 1 km of a selected grid point for forward_operator='reference', and the
    number of obs outside the grid for 'bilinear' (DESIGN.md section 4.8; their rows of Y are 0).  The caller picks
    the time weights (obs.tw0 / tw1) that go with the operator.

    X may also be a PINNED host tensor: the gather kernel then reads the <= 8 stencil rows per ob straight from
    host memory over PCIe (unified addressing), which lets the obs-space solve start while the state is still
    being uploaded.

    With band=(y0, y1), X holds only that latitude band of the state: each rank sums the stencil points it
    owns and the partial sums are all-reduced, so every rank ends with the same full Y.
    obs_dev: the device copies of the per-ob tables made by upload_obs (saves re-uploading them)."""
    torch = _torch()
    dev = grid.device
    check_forward_operator(forward_operator, 1 if grid.diag else 2)
    if obs_dev is None or 'row0' not in obs_dev:
        obs_dev = {'lat': _dev_f64(obs.lat, dev), 'lon': _dev_f64(obs.lon, dev),
                   'sinlat': _dev_f64(np.sin(np.radians(obs.lat)), dev), 'coslon': _dev_f64(np.cos(np.radians(obs.lon)), dev),
                   'row0': torch.as_tensor(np.ascontiguousarray(obs.row0, dtype=np.int64)).to(dev),
                   'row1': torch.as_tensor(np.ascontiguousarray(obs.row1, dtype=np.int64)).to(dev),
                   'tw0': _dev_f64(obs.tw0, dev), 'tw1': _dev_f64(obs.tw1, dev)}
    if forward_operator == 'bilinear':
        idx4, w4, nex = stencil_bilinear(grid, obs_dev['lat'], obs_dev['lon'])
    else:
        tables = (obs_dev['lat'], obs_dev['lon'], obs_dev['sinlat'], obs_dev['coslon'])
        idx4, w4, nex = stencil_search(grid, None, None, dev_tables=tables)
    # 8-point stencil = 4 space points x 2 time levels, re-based to the band's shard (index/weight bookkeeping only)
    y0, y1 = band if band is not None else (0, grid.ny)
    idx8 = torch.empty((obs.nobs, 8), dtype=torch.int64, device=dev)
    w8 = torch.empty((obs.nobs, 8), dtype=torch.float64, device=dev)
    _lib.call('exb_stencil_combine', _lib.ptr(idx4), _lib.ptr(w4), _lib.ptr(obs_dev['row0']), _lib.ptr(obs_dev['row1']),
              _lib.ptr(obs_dev['tw0']), _lib.ptr(obs_dev['tw1']), obs.nobs, grid.ny, grid.nx, y0, y1, int(grid.diag), _lib.ptr(idx8),
              _lib.ptr(w8), _lib.stream_ptr())
    Y = torch.empty((obs.nobs, X.shape[1]), dtype=X.dtype, device=dev)
    _lib.call('exb_gather_' + sfx, _lib.ptr(X), X.shape[0], X.shape[1], _lib.ptr(idx8), _lib.ptr(w8), 8,
              obs.nobs, _lib.ptr(Y), _lib.stream_ptr())
    if band is not None:
        import torch.distributed as dist
        if dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(Y, group=group)
    return Y, nex


def _sfx(dtype):
    torch = _torch()
    if dtype == torch.float64:
        return 'f64'
    if dtype == torch.float32:
        return 'f32'
    raise TypeError('efa_xray_b200 supports float64 and float32 states, got %r' % (dtype,))


class _Timer:
    def __init__(self, enabled=True):
        self.torch = _torch()
        self.enabled = enabled
        self.marks = []

    def mark(self, name):
        if self.enabled:
            e = self.torch.cuda.Event(enable_timing=True)
            e.record()
            self.marks.append((name, e))

    def result(self):
        if not self.enabled or not self.marks:
            return {}
        self.torch.cuda.synchronize()
        out = {}
        for (n0, e0), (n1, e1) in zip(self.marks[:-1], self.marks[1:]):
            out[n1] = out.get(n1, 0.0) + e0.elapsed_time(e1)
        return out


def _qc_args(obs_dev):
    """('qc_', (threshold pointer,)) for the _qc entries of the obs-space solve when upload_obs staged outlier
    thresholds, else ('', ())."""
    thr = obs_dev.get('threshold')
    return ('qc_', (_lib.ptr(thr),)) if thr is not None else ('', ())


def obs_solve(Ym, Yp, obs_dev, geo, nens, loc_mode, rec, counters, sfx, plan=None):
    qc, thr = _qc_args(obs_dev)
    if plan is not None:
        _lib.call('exb_obs_solve_planned_' + qc + sfx, plan.handle, _lib.ptr(Ym), _lib.ptr(Yp), _lib.ptr(obs_dev['value']),
                  _lib.ptr(obs_dev['error']), _lib.ptr(obs_dev['assimilate']), *thr, _lib.ptr(geo), Ym.shape[0], nens,
                  loc_mode, _lib.ptr(rec), _lib.ptr(counters), _lib.stream_ptr())
        return
    _lib.call('exb_obs_solve_' + qc + sfx, _lib.ptr(Ym), _lib.ptr(Yp), _lib.ptr(obs_dev['value']),
              _lib.ptr(obs_dev['error']), _lib.ptr(obs_dev['assimilate']), *thr, _lib.ptr(geo), Ym.shape[0], nens,
              loc_mode, _lib.ptr(rec), _lib.ptr(counters), _lib.stream_ptr())


class ObsPlan:
    """The geometry-only part of the obs-space solve (predecessor lists), built on a side stream while the host and
    the current stream compute the ob priors: the constructor only enqueues the counting pass (exb_obs_plan_create),
    finish() sizes the lists and enqueues the fill pass (exb_obs_plan_finish)."""

    def __init__(self, obs_dev, geo, nobs, loc_mode, rank=0, world=1, block=1):
        torch = _torch()
        self.handle = C.c_void_p()
        self.rank, self.world, self.block = rank, world, block
        self.stream = torch.cuda.Stream(device=geo.device)
        ready = obs_dev.get('_ready')
        if ready is not None:
            self.stream.wait_event(ready)
        else:
            self.stream.wait_stream(torch.cuda.current_stream())
        if world > 1:           # lists of this rank's rows only (distributed solve)
            _lib.call('exb_obs_plan_create_dist', _lib.ptr(geo), _lib.ptr(obs_dev['assimilate']), nobs, loc_mode, rank,
                      world, block, C.c_void_p(self.stream.cuda_stream), C.byref(self.handle))
        else:
            _lib.call('exb_obs_plan_create', _lib.ptr(geo), _lib.ptr(obs_dev['assimilate']), nobs, loc_mode,
                      C.c_void_p(self.stream.cuda_stream), C.byref(self.handle))

    def finish(self):
        _lib.call('exb_obs_plan_finish', self.handle)

    def destroy(self):
        if self.handle:
            _lib.call('exb_obs_plan_destroy', self.handle)
            self.handle = C.c_void_p()


class SweepPlan:
    """The geometry-only part of the fused state sweep (scan records of the obs, candidate lists per coarse tile),
    built on a side stream while the ob priors and the obs-space solve are computed (exb_sweep_plan_create).  Creating
    the plan blocks its caller until the counting pass is done (the list is sized on the host)."""

    def __init__(self, grid_u, nlev, ny, nx, obs_dev, geo, nobs, loc_mode, y_begin=0, y_end=None):
        torch = _torch()
        self.handle = C.c_void_p()
        self.grid_u, self.geo = grid_u, geo          # keep the inputs alive and identical to what the sweep is given
        self.stream = torch.cuda.Stream(device=geo.device)
        ready = obs_dev.get('_ready')
        if ready is not None:
            self.stream.wait_event(ready)
        self.stream.wait_stream(torch.cuda.current_stream())
        _lib.call('exb_sweep_plan_create', _lib.ptr(grid_u), nlev, ny, nx, _lib.ptr(geo), _lib.ptr(obs_dev['assimilate']),
                  nobs, 0, nobs, y_begin, ny if y_end is None else y_end, loc_mode, C.c_void_p(self.stream.cuda_stream),
                  C.byref(self.handle))

    def destroy(self):
        if self.handle:
            _lib.call('exb_sweep_plan_destroy', self.handle)
            self.handle = C.c_void_p()


_DIST_BUFFERS = {}


def _dist_buffers(nobs, nens, dtype, device, group):
    """Symmetric (peer-mapped) record buffers of the distributed obs-space solve, cached per shape: the tensors, the
    rendezvous handles and ctypes arrays of the peers' pointers."""
    torch = _torch()
    import torch.distributed as dist
    import torch.distributed._symmetric_memory as symm_mem
    mc = 4 if nens <= 128 else 8
    key = (nobs, mc, dtype, str(device), id(group))
    if key not in _DIST_BUFFERS:
        g = group if group is not None else dist.group.WORLD
        P = symm_mem.empty(nobs * 32 * mc, dtype=dtype, device=device)
        S = symm_mem.empty(nobs * 2, dtype=torch.float64, device=device)
        hP, hS = symm_mem.rendezvous(P, g), symm_mem.rendezvous(S, g)
        world = dist.get_world_size(g)
        pp = (C.c_void_p * 8)(*[C.c_void_p(int(hP.buffer_ptrs[q])) if q < world else None for q in range(8)])
        sp = (C.c_void_p * 8)(*[C.c_void_p(int(hS.buffer_ptrs[q])) if q < world else None for q in range(8)])
        _DIST_BUFFERS[key] = (P, S, hP, hS, pp, sp)
    return _DIST_BUFFERS[key]


def obs_solve_distributed(Ym, Yp, obs_dev, geo, nens, loc_mode, rec, counters, sfx, plan, group=None):
    """Obs-space solve with the rows dealt to the ranks of `group` (one process per GPU of an NVLink domain) in blocks
    of plan.block consecutive obs: every rank solves nobs/world rows and publishes their records into all ranks'
    record buffers over peer memory (exb_obs_solve_dist_*); afterwards ye rows, means, records and the pair counter
    are summed over the group so that every rank holds the complete result, as after the replicated solve.  Returns
    False (nothing done) when the plan is dense / multi-block or symmetric memory is unavailable."""
    torch = _torch()
    import torch.distributed as dist
    g = group if group is not None else dist.group.WORLD
    world, rank = dist.get_world_size(g), dist.get_rank(g)
    nobs = Ym.shape[0]
    try:
        P, S, hP, hS, pp, sp = _dist_buffers(nobs, nens, Yp.dtype, Yp.device, group)
    except Exception as e:             # no peer access / symmetric memory in this build
        import warnings
        warnings.warn('distributed obs-space solve unavailable (%s); using the replicated one' % (e,))
        return False
    P.view(torch.uint8).fill_(255)
    S.view(torch.uint8).fill_(255)
    flag = torch.zeros(1, dtype=torch.int32, device=Yp.device)
    dist.all_reduce(flag, group=g)     # stream-ordered barrier: every rank's sentinel fill precedes every kernel
    rec.zero_()
    c0 = counters[0:1].clone()
    counters[0:1].zero_()
    lib = _lib.load()
    qc, thr = _qc_args(obs_dev)
    rc = getattr(lib, 'exb_obs_solve_dist_' + qc + sfx)(
        plan.handle, _lib.ptr(Ym), _lib.ptr(Yp), _lib.ptr(obs_dev['value']), _lib.ptr(obs_dev['error']),
        _lib.ptr(obs_dev['assimilate']), *thr, _lib.ptr(geo), nobs, nens, loc_mode, _lib.ptr(rec), _lib.ptr(counters), rank,
        world, pp, sp, _lib.stream_ptr())
    if rc == -3:                       # EXB_ERR_UNSUPPORTED: identical decision on every rank (same plan)
        counters[0:1].copy_(c0)
        return False
    if rc != 0:
        raise _lib.ExbError('exb_obs_solve_dist_%s%s failed (%d): %s' % (qc, sfx, rc,
                                                                       lib.exb_last_error().decode('utf-8', 'replace')))
    merge_distributed_records(Ym, rec, counters[0:1], plan.block, rank, world, g)
    counters[0:1].add_(c0)
    # every rank's record buffer holds the published ye row of EVERY ob once all ranks are done (the all-reduces above
    # are behind every rank's kernel): the 80 MB of ye rows need no collective, only a local copy out of the padded
    # records
    mc = P.numel() // (nobs * 32)
    Yp.copy_(P.view(nobs, 32 * mc)[:, :nens])
    return True


def merge_distributed_records(Ym, rec, pair_counter, block, rank, world, group):
    """After a distributed obs-space solve every rank holds means / records / pair count of ITS rows only (rank r owns
    ob j when (j // block) % world == r): zero the others and sum over the group, so that every rank ends up with the
    complete, identical result.  NaN marks "not assimilated" in the records (post mean / variance) and must survive the
    sum.  Pure torch (works on any backend; tests/test_sharding_gloo.py runs it over gloo)."""
    torch = _torch()
    import torch.distributed as dist
    nobs = Ym.shape[0]
    mine = (torch.arange(nobs, device=Ym.device) // block) % world == rank
    Ym.mul_(mine.to(Ym.dtype))
    rec.mul_(mine.to(rec.dtype)[None, :])           # (NaN * 0 = NaN: rows of other ranks are zero-filled by the caller)
    nanmask = torch.isnan(rec)
    rec.masked_fill_(nanmask, 0.0)
    skipped = (nanmask & mine[None, :]).to(rec.dtype)
    for t in (Ym, rec, skipped, pair_counter):
        dist.all_reduce(t, group=group)
    rec.masked_fill_(skipped > 0, float('nan'))


def obs_dist_wanted(group):
    """Multi-GPU runs over NCCL distribute the obs-space solve over the ranks (EXB_OBS_DIST=0: replicate it)."""
    import os
    import torch.distributed as dist
    if os.environ.get('EXB_OBS_DIST', '1') != '1' or not dist.is_initialized():
        return False
    return dist.get_world_size(group) > 1 and dist.get_backend(group) == 'nccl'


def obs_dist_block():
    """Block size of the distributed obs-space solve's dealing (EXB_OBS_DIST_BLOCK; 1 = round-robin).  Default 256:
    consecutive obs of a dependency chain are a few tens of indices apart, so most hops of the chain then stay on one
    GPU (measured at N = 2, config 3: 17.5 ms against 22.8 ms round-robin and 20.2 ms replicated)."""
    import os
    return max(1, int(os.environ.get('EXB_OBS_DIST_BLOCK', '256')))


def obs_plan_wanted(loc_mode):
    import os
    return loc_mode == LOC_GC and os.environ.get('EXB_OBS_IMPL', 'dag') == 'dag'


def state_update(xm, Xp, nlev, ny, nx, grid_u, Yp, rec, geo, nobs, loc_mode, counters, sfx, ob_begin=0, ob_end=None):
    _lib.call('exb_state_update_' + sfx, _lib.ptr(xm), _lib.ptr(Xp), nlev, ny, nx, Xp.shape[-1], _lib.ptr(grid_u),
              _lib.ptr(Yp), _lib.ptr(rec), _lib.ptr(geo), nobs, ob_begin, nobs if ob_end is None else ob_end,
              loc_mode, _lib.ptr(counters), _lib.stream_ptr())


def state_sweep_fused(X, nlev, ny, nx, grid_u, Yp, rec, geo, nobs, loc_mode, counters, y_begin=0, y_end=None,
                      ob_begin=0, ob_end=None, plan=None):
    """Fused split + sweep + recombine of grid rows [y_begin, y_end) of a shard holding full ensemble values
    (exb_state_sweep_f64 / _f32; with a SweepPlan the geometry-only part was built ahead)."""
    if plan is not None:
        _lib.call('exb_state_sweep_planned_' + _sfx(X.dtype), plan.handle, _lib.ptr(X), nlev, ny, nx, X.shape[-1],
                  _lib.ptr(grid_u), _lib.ptr(Yp), _lib.ptr(rec), _lib.ptr(geo), nobs, ob_begin, nobs if ob_end is None else ob_end,
                  y_begin, ny if y_end is None else y_end, loc_mode, _lib.ptr(counters), _lib.stream_ptr())
        return
    _lib.call('exb_state_sweep_' + _sfx(X.dtype), _lib.ptr(X), nlev, ny, nx, X.shape[-1], _lib.ptr(grid_u), _lib.ptr(Yp),
              _lib.ptr(rec), _lib.ptr(geo), nobs, ob_begin, nobs if ob_end is None else ob_end, y_begin,
              ny if y_end is None else y_end, loc_mode, _lib.ptr(counters), _lib.stream_ptr())


# Largest ensemble of the fused sweep: 13 tiles of 8 columns, the last of which also carries the ensemble mean as a
# pseudo-member (state_sweep_2p.cu), so 8 * 13 - 1 members.
FUSED_MAX_NENS = 103


def fused_sweep_available(nens):
    """The fused sweep (exb_state_sweep_*) serves float64 and float32 (storage) ensembles of up to FUSED_MAX_NENS
    members; larger ones take the three-call form (split, exb_state_update_*, recombine)."""
    return nens <= FUSED_MAX_NENS


RELAX_KINDS = ('rtps', 'rtpp')


def relaxation_device(relaxation, nlev, device):
    """(kind, alpha per level) -> (kind, the alphas as a float64 tensor on `device`), or None when there is nothing to
    relax (relaxation None, or every alpha 0).  The alphas go up in one copy from page-locked memory, so the call does
    not wait for the host: callers that stream the state in on another stream call this first (analysis_host), or the
    copy would queue behind the state.  A pair whose alphas are already a device tensor is returned as it is."""
    if relaxation is None:
        return None
    torch = _torch()
    kind, alpha = relaxation
    if kind not in RELAX_KINDS:
        raise ValueError('relaxation kind must be one of %r, got %r' % (RELAX_KINDS, kind))
    if isinstance(alpha, torch.Tensor) and alpha.device.type == 'cuda':
        return relaxation
    a = np.ascontiguousarray(alpha, dtype=np.float64).ravel()
    if a.shape != (nlev,):
        raise ValueError('relaxation needs one alpha per level (%d), got shape %r' % (nlev, a.shape))
    if not ((a >= 0.0) & (a <= 1.0)).all():
        raise ValueError('relaxation alphas must lie in [0, 1], got %r' % (a,))
    if not a.any():
        return None
    return kind, torch.from_numpy(a).pin_memory().to(device, non_blocking=True)


class _Relaxation:
    """RTPS / RTPP of the state rows after the serial loop (DESIGN.md section 4.6), applied row range by row range:
    before(pa, pb) records what the prior rows [pa, pb) of every level look like (sigma_b per row for RTPS, a copy of
    the rows for RTPP) and must run before the sweep changes them; after(pa, pb) relaxes them once the analysis is
    there.  Both run on the current stream.  ms() is the device time of the passes."""

    def __init__(self, relaxation, X, nlev, timing):
        torch = _torch()
        self.kind, self.alpha = relaxation
        self.X, self.nlev = X, nlev
        self.npts = X.shape[0] // nlev
        self.nens = X.shape[1]
        self.sfx = _sfx(X.dtype)
        if self.kind == 'rtps':
            self.sigma_b = torch.empty(X.shape[0], dtype=torch.float64, device=X.device)
        else:
            self.Xb = torch.empty_like(X)
        self.events = [] if timing else None

    def _timed(self, fn):
        if self.events is None:
            return fn()
        torch = _torch()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        self.events.append((e0, e1))

    def before(self, pa, pb):
        def run():
            if self.kind == 'rtps':
                _lib.call('exb_row_spread_' + self.sfx, _lib.ptr(self.X), self.nlev, self.npts, pa, pb, self.nens,
                          _lib.ptr(self.sigma_b), _lib.stream_ptr())
            else:
                shape = (self.nlev, self.npts, self.nens)
                self.Xb.view(shape)[:, pa:pb].copy_(self.X.view(shape)[:, pa:pb])
        self._timed(run)

    def after(self, pa, pb):
        prior = self.sigma_b if self.kind == 'rtps' else self.Xb
        self._timed(lambda: _lib.call('exb_relax_%s_%s' % (self.kind, self.sfx), _lib.ptr(self.X), _lib.ptr(prior),
                                      _lib.ptr(self.alpha), self.nlev, self.npts, pa, pb, self.nens, _lib.stream_ptr()))

    def ms(self):
        return sum(e0.elapsed_time(e1) for e0, e1 in self.events)


_OBS_FIELDS = ('value', 'error', 'lat', 'lon', 'halfwidth', 'tw0', 'tw1', 'row0', 'row1')
_STAGING = {}


def upload_obs(obs: ObsArrays, device, loc_mode):
    """Per-ob tables on the device + the obgeo block of exb_obs_prepare.  Everything goes up in ONE copy from a cached
    page-locked staging buffer (nine 8-byte fields + the assimilate flags per ob): small pageable copies cost a
    host synchronisation each and may not queue behind bulk state copies.  With outlier thresholds (obs.qc) they are
    a tenth 8-byte field, d['threshold']; without, d has no such entry and the layout is the nine fields."""
    torch = _torch()
    n = obs.nobs
    if obs.qc and np.shape(obs.threshold) != (n,):
        raise ValueError('ObsArrays.threshold needs one value per ob (%d) or none, got shape %r'
                         % (n, np.shape(obs.threshold)))
    fields = _OBS_FIELDS + ('threshold',) if obs.qc else _OBS_FIELDS
    nf = len(fields)
    key = (n, nf, str(device))
    ent = _STAGING.get(key)
    if ent is None:
        if len(_STAGING) > 8:
            _STAGING.clear()
        ent = {'host': torch.empty(nf * n * 8 + n, dtype=torch.uint8).pin_memory(), 'event': None}
        _STAGING[key] = ent
    if ent['event'] is not None:
        ent['event'].synchronize()               # the previous upload from this buffer has left the host
    hb = ent['host'].numpy()
    f64 = hb[:nf * n * 8].view(np.float64).reshape(nf, n)
    i64 = hb[:nf * n * 8].view(np.int64).reshape(nf, n)
    f64[0], f64[1], f64[2], f64[3] = obs.value, obs.error, obs.lat, obs.lon
    f64[4] = obs.halfwidth if loc_mode == LOC_GC else 1.0
    f64[5], f64[6] = obs.tw0, obs.tw1
    i64[7], i64[8] = obs.row0, obs.row1
    if obs.qc:
        f64[9] = obs.threshold
    hb[nf * n * 8:] = obs.assimilate
    db = torch.empty(nf * n * 8 + n, dtype=torch.uint8, device=device)
    db.copy_(ent['host'], non_blocking=True)
    ent['event'] = torch.cuda.Event()
    ent['event'].record()
    df = db[:nf * n * 8].view(torch.float64).view(nf, n)
    di = db[:nf * n * 8].view(torch.int64).view(nf, n)
    d = {name: (di[i] if name in ('row0', 'row1') else df[i]) for i, name in enumerate(fields)}
    d['assimilate'] = db[nf * n * 8:]
    d['_buffer'] = db
    if loc_mode != LOC_GC:
        d['halfwidth'] = None
    # ob-side tables of the nearest-point search, on the device (5 ms of host trigonometry for 1e5 obs otherwise)
    trig = torch.empty((2, n), dtype=torch.float64, device=device)
    _lib.call('exb_obs_trig', _lib.ptr(d['lat']), _lib.ptr(d['lon']), n, _lib.ptr(trig[0]), _lib.ptr(trig[1]), _lib.stream_ptr())
    d['sinlat'], d['coslon'] = trig[0], trig[1]
    geo = torch.empty((8, n), dtype=torch.float64, device=device)
    _lib.call('exb_obs_prepare', _lib.ptr(d['lat']), _lib.ptr(d['lon']), _lib.ptr(d['halfwidth']), n,
              loc_mode, _lib.ptr(geo), _lib.stream_ptr())
    d['_ready'] = torch.cuda.Event()
    d['_ready'].record()
    return d, geo


def analysis_device(X, nlev, grid: GridTables, obs: ObsArrays, loc_mode, inflation=None, timing=True,
                    band=None, group=None, Y=None, sweep_bands=None, on_band_done=None, before_band=None,
                    obs_device=None, relaxation=None, forward_operator='reference'):
    """Serial EnSRF analysis of a device-resident ensemble, in place.

    X        torch tensor [nlev*ny*nx, nens] (float64 or float32) on a CUDA device, to_vect layout
             (state/ensemble.py:110-114); overwritten with the analysis ensemble.  With band=(y0, y1) X is
             only that latitude band, [nlev*(y1-y0)*nx, nens], of a state sharded over the ranks of `group`;
             `grid` always describes the full grid.
    inflation  None, or a numpy array of per-level multiplicative factors (length nlev).
    relaxation  None, or (kind, alpha per level): posterior relaxation of the state rows after the serial loop,
             kind 'rtps' (relaxation to prior spread) or 'rtpp' (relaxation to prior perturbations), relative to the
             prior as the sweep receives it (after inflation); DESIGN.md section 4.6.  Every alpha 0 launches nothing.
             The per-ob diagnostics stay those of the serial loop.  res.ms gains 'relax' when it ran.
    obs.threshold  empty (no check), or outlier thresholds per ob: the obs-space solve rejects an ob whose innovation exceeds
             its threshold times sqrt(prior variance + error) inside the serial loop (DESIGN.md section 4.7);
             rejected obs come back with assimilated False, and the state sweep applies a zero update for them.
    forward_operator  'reference' (the reference's 4-point inverse-distance operator) or 'bilinear' (DESIGN.md
             section 4.8; obs.tw0 / tw1 must then be the weights of time_weights(swapped=False)).  With 'bilinear',
             res.n_outside counts the obs outside the grid: their priors are 0, so callers reject such a result.
    sweep_bands  optional list of (ya, yb) row ranges of the shard: the fused sweep is issued range by range and
             on_band_done(ya, yb) is called after each launch has been enqueued (e.g. to start its download),
             before_band(ya, yb) before it (e.g. to wait for its upload).
    Returns an AnalysisResult with the per-ob diagnostics of ensrf.py:66-70,144-149 (identical on all ranks).
    """
    torch = _torch()
    _lib.require_device()
    sfx = _sfx(X.dtype)
    dev = X.device
    nrows, nens = X.shape
    nx = grid.nx
    y0, y1 = band if band is not None else (0, grid.ny)
    ny = y1 - y0
    assert nrows == nlev * ny * nx, (nrows, nlev, ny, nx)
    assert X.is_contiguous()
    tm = _Timer(timing)
    tm.mark('start')
    plan = None
    splan = None
    with torch.cuda.device(dev):
        if inflation is not None:
            fac = np.ascontiguousarray(inflation, dtype=np.float64).ravel()
            # one factor per level (float / per-variable dict) or one per state row (per-dimension arrays)
            assert fac.shape[0] in (nlev, nrows), (fac.shape, nlev, nrows)
            _lib.call('exb_inflate_' + sfx, _lib.ptr(X), nrows, nens, fac.ctypes.data_as(C.c_void_p), fac.shape[0],
                      nrows // fac.shape[0], _lib.stream_ptr())
        if obs.nobs == 0:
            # an assimilation window without observations: the reference's loop body never runs (ensrf.py:50) and
            # the (inflated) prior comes back as the posterior
            z = np.zeros(0)
            return AnalysisResult(prior_mean=z, prior_var=z, post_mean=z, post_var=z, assimilated=np.zeros(0, dtype=bool),
                                  ms=tm.result(), obs_solve='none')
        # (small host-to-device copies: callers that stream the state in on another stream do them first and pass
        # the result, or they would queue behind the state in the copy engine)
        obs_dev, geo = obs_device if obs_device is not None else upload_obs(obs, dev, loc_mode)
        relaxation = relaxation_device(relaxation, nlev, dev)
        relax = _Relaxation(relaxation, X, nlev, timing) if relaxation is not None else None
        tm.mark('setup_upload')
        try:
            # predecessor lists of the obs-space solve: geometry only, started on a side stream now so that they are
            # built while the host and this stream work on the ob priors
            dist_solve = band is not None and obs_plan_wanted(loc_mode) and obs_dist_wanted(group)
            if dist_solve:
                import torch.distributed as dist
                plan = ObsPlan(obs_dev, geo, obs.nobs, loc_mode, dist.get_rank(group), dist.get_world_size(group),
                               obs_dist_block())
            elif obs_plan_wanted(loc_mode):
                plan = ObsPlan(obs_dev, geo, obs.nobs, loc_mode)
            fused = fused_sweep_available(nens)
            grid_u = grid.u if band is None else grid.u[:, y0 * nx:y1 * nx].contiguous()
            if Y is None:
                Yp, nex = ob_priors(X, grid, obs, sfx, nlev=nlev, band=band, group=group, obs_dev=obs_dev,
                                    forward_operator=forward_operator)
            elif isinstance(Y, tuple):   # (H.x, counter) from ob_priors, owned by this call
                Yp, nex = Y
            else:       # ob priors H.x computed by the caller (e.g. before the state was scattered)
                Yp, nex = Y.clone(), torch.zeros(1, dtype=torch.int32, device=dev)
            Ym = torch.empty(obs.nobs, dtype=X.dtype, device=dev)
            _lib.call('exb_split_mean_pert_' + sfx, _lib.ptr(Yp), _lib.ptr(Ym), obs.nobs, nens, _lib.stream_ptr())
            tm.mark('setup_ob_priors')
            if plan is not None:
                # the solve is next on the critical path: its lists are filled before the sweep's plan is started
                plan.finish()
            if fused:
                # candidate lists of the sweep: geometry only as well, built on another side stream.  Creating the plan
                # blocks its caller until the counting pass is done, so it comes after the ob priors have been enqueued
                # (the device computes them meanwhile)
                splan = SweepPlan(grid_u, nlev, ny, nx, obs_dev, geo, obs.nobs, loc_mode)
            if not fused:
                if relax is not None:
                    relax.before(0, ny * nx)
                xm = torch.empty(nrows, dtype=X.dtype, device=dev)
                _lib.call('exb_split_mean_pert_' + sfx, _lib.ptr(X), _lib.ptr(xm), nrows, nens, _lib.stream_ptr())
            tm.mark('setup_plans')
            rec = torch.empty((8, obs.nobs), dtype=torch.float64, device=dev)
            counters = torch.zeros(2, dtype=torch.int64, device=dev)
            done = False
            which = 'replicated' if band is not None else 'single'
            if dist_solve:
                done = obs_solve_distributed(Ym, Yp, obs_dev, geo, nens, loc_mode, rec, counters, sfx, plan, group=group)
                if done:
                    which = 'distributed(block=%d)' % plan.block
                else:                   # dense graph or no peer memory: replicated solve with a full plan
                    plan.destroy()
                    plan = ObsPlan(obs_dev, geo, obs.nobs, loc_mode)
                    plan.finish()
            if not done:
                obs_solve(Ym, Yp, obs_dev, geo, nens, loc_mode, rec, counters, sfx, plan=plan)
            tm.mark('obs_solve')
            if fused:
                for ya, yb in (sweep_bands or [(0, ny)]):
                    if before_band is not None:
                        before_band(ya, yb)
                    if relax is not None:
                        relax.before(ya * nx, yb * nx)
                    state_sweep_fused(X, nlev, ny, nx, grid_u, Yp, rec, geo, obs.nobs, loc_mode, counters, ya, yb, plan=splan)
                    if relax is not None:
                        relax.after(ya * nx, yb * nx)
                    if on_band_done is not None:
                        on_band_done(ya, yb)
                tm.mark('state_update')
            else:
                state_update(xm, X, nlev, ny, nx, grid_u, Yp, rec, geo, obs.nobs, loc_mode, counters, sfx)
                tm.mark('state_update')
                _lib.call('exb_recombine_' + sfx, _lib.ptr(X), _lib.ptr(xm), nrows, nens, _lib.stream_ptr())
                if relax is not None:
                    relax.after(0, ny * nx)
            tm.mark('recombine')
            rec_h = rec.cpu().numpy()
            _lib.call('exb_obs_solve_async_status')
            cnt = counters.cpu().numpy()
            nex_h = int(nex.item())
        finally:
            if plan is not None:
                plan.destroy()
            if splan is not None:
                splan.destroy()
    ms = tm.result()
    if relax is not None and timing:
        ms['relax'] = relax.ms()
    bilinear = forward_operator == 'bilinear'
    return AnalysisResult(prior_mean=rec_h[0], prior_var=rec_h[1], post_mean=rec_h[2], post_var=rec_h[3],
                          assimilated=rec_h[7] != 0.0, n_exact=0 if bilinear else nex_h,
                          n_outside=nex_h if bilinear else 0, state_pairs=int(cnt[1]) * nlev,
                          obs_pairs=int(cnt[0]), ms=ms, obs_solve=which)


def sweep_band_schedule(nlev, ny, nx, nbands=None):
    """Row ranges for a band-by-band sweep whose bands are uploaded / downloaded while other bands are swept:
    equal row counts (on a lat-lon grid every row has the same number of points, and with obs spread over the
    sphere every point sees about the same number of obs), edges on patch-row boundaries, the last band halved
    so that the download left exposed at the end is short.  The schedule only affects how well copies and
    kernels overlap."""
    g = max(1, int(_lib.load().exb_state_sweep_row_granularity(nlev, ny, nx)))
    if nbands is None:
        # every launch costs a tail and a small pre-pass: about 180 grid rows per band, at most 6 bands
        nbands = max(1, min(6, ny // 180))
    nbands = max(1, min(nbands, ny // g if ny >= g else 1))
    edges = sorted(set([0, ny] + [int(round(ny * i / nbands / g)) * g for i in range(1, nbands)]))
    edges = [e for e in edges if 0 <= e <= ny]
    ya, yb = edges[-2], edges[-1]
    mid = ((ya + yb) // 2 // g) * g
    if ya < mid < yb:
        edges.insert(-1, mid)
    return [(edges[i], edges[i + 1]) for i in range(len(edges) - 1)]


def analysis_host(X_host, nlev, lat2d, lon2d, obs: ObsArrays, loc_mode, inflation=None, device='cuda:0',
                  dtype=None, grid=None, out=None, pipeline=True, band=None, group=None, relaxation=None,
                  forward_operator='reference'):
    """Host-buffer entry: X_host is a numpy array or CPU torch tensor [nlev*ny*nx, nens]; it is uploaded,
    analysed on `device`, and the analysis is written to `out` (default: back into X_host).  Pinned host
    memory makes the copies asynchronous.  With the fused sweep (up to FUSED_MAX_NENS members, pipeline=True and
    localisation) the state is swept in latitude bands and each finished band is downloaded on a second stream while the next one is swept, so
    only the last band's download is exposed; the upload is overlapped with the obs-space solve when X_host is
    pinned (see ob_priors).  res.ms gains 'upload' (duration of the host-to-device copies) and 'download' (what is
    left of the device-to-host copies after the last sweep).

    With band=(y0, y1) X_host / out hold only that latitude band of a host-resident state sharded over the ranks of
    `group` (one process per GPU): every rank moves its own band over its own PCIe link, the partial ob priors are
    all-reduced (NCCL), the obs-space solve is distributed over the ranks through NVLink peer memory (or replicated, see
    res.obs_solve) and no other data crosses between ranks.

    relaxation: as for analysis_device; with the band pipeline each band is relaxed between its sweep and its
    download.  forward_operator: as for analysis_device."""
    torch = _torch()
    _lib.require_device()
    Xh = X_host if isinstance(X_host, torch.Tensor) else torch.from_numpy(X_host)
    Oh = Xh if out is None else (out if isinstance(out, torch.Tensor) else torch.from_numpy(out))
    assert Xh.is_contiguous() and Oh.is_contiguous() and Oh.shape == Xh.shape
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    with torch.cuda.device(device):
        main = torch.cuda.current_stream()
        if grid is None:
            grid = GridTables(lat2d, lon2d, torch.device(device))
        nens = Xh.shape[1]
        xdtype = Xh.dtype if dtype is None else dtype
        y0, y1 = band if band is not None else (0, grid.ny)
        ny_loc = y1 - y0
        banded = (pipeline and fused_sweep_available(nens) and Oh.dtype == xdtype and Xh.dtype == xdtype
                  and loc_mode == LOC_GC and obs.nobs > 0)
        if banded:
            # Three streams: uploads (band by band, in sweep order), compute, downloads.  With a pinned source and
            # no inflation step the ob priors are gathered straight from host memory, so the obs-space solve runs
            # while the state is still arriving; a band is swept as soon as it is on the device and downloaded
            # while the next ones are swept.
            copy_in, copy_out = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)
            npts = ny_loc * grid.nx
            X = torch.empty((nlev * npts, nens), dtype=xdtype, device=device)
            X3, H3, O3 = X.view(nlev, npts, nens), Xh.view(nlev, npts, nens), Oh.view(nlev, npts, nens)
            bands = sweep_band_schedule(nlev, ny_loc, grid.nx)
            ev[0].record()
            obs_device = upload_obs(obs, torch.device(device), loc_mode)
            relaxation = relaxation_device(relaxation, nlev, torch.device(device))
            Y = None
            if inflation is None and Xh.is_pinned():
                # PCIe is used by one thing at a time: first the gather (25 % of the state in 800-byte pieces),
                # then the band uploads, which overlap the obs-space solve and the sweep of earlier bands
                Y = ob_priors(Xh, grid, obs, _sfx(xdtype), nlev=nlev, band=band, group=group, obs_dev=obs_device[0],
                              forward_operator=forward_operator)
            arrived = {}
            copy_in.wait_stream(main)
            with torch.cuda.stream(copy_in):
                for ya, yb in bands:
                    for lev in range(nlev):
                        X3[lev, ya * grid.nx:yb * grid.nx].copy_(H3[lev, ya * grid.nx:yb * grid.nx], non_blocking=True)
                    arrived[(ya, yb)] = torch.cuda.Event()
                    arrived[(ya, yb)].record(copy_in)
                up_done = torch.cuda.Event(enable_timing=True)
                up_done.record(copy_in)
            if Y is None:
                main.wait_stream(copy_in)
            ev[1].record()

            def wait_upload(ya, yb):
                main.wait_event(arrived[(ya, yb)])

            def download(ya, yb):
                done = torch.cuda.Event()
                done.record(main)
                copy_out.wait_event(done)
                with torch.cuda.stream(copy_out):
                    for lev in range(nlev):
                        O3[lev, ya * grid.nx:yb * grid.nx].copy_(X3[lev, ya * grid.nx:yb * grid.nx], non_blocking=True)

            res = analysis_device(X, nlev, grid, obs, loc_mode, inflation, Y=Y, sweep_bands=bands, band=band, group=group,
                                  before_band=wait_upload, on_band_done=download, obs_device=obs_device,
                                  relaxation=relaxation, forward_operator=forward_operator)
            ev[2].record()
            main.wait_stream(copy_out)
            ev[3].record()
            torch.cuda.synchronize()
            res.ms['upload'] = ev[0].elapsed_time(up_done)
        else:
            ev[0].record()
            X = Xh.to(device, non_blocking=True)
            if dtype is not None and X.dtype != dtype:
                X = X.to(dtype)
            ev[1].record()
            res = analysis_device(X, nlev, grid, obs, loc_mode, inflation, band=band, group=group, relaxation=relaxation,
                                  forward_operator=forward_operator)
            ev[2].record()
            Oh.copy_(X.to(Oh.dtype) if X.dtype != Oh.dtype else X, non_blocking=True)
            ev[3].record()
            torch.cuda.synchronize()
            res.ms['upload'] = ev[0].elapsed_time(ev[1])
        res.ms['download'] = ev[2].elapsed_time(ev[3])
    return res
