"""Observation objects (efa_xray/observation/observation.py:17-146)."""
from __future__ import print_function

import math

import numpy as np

from .. import _lib
from ..state.ensemble import EnsembleState


class Observation:
    """Attribute record of one point observation (observation.py:17-37).  `error` is a VARIANCE;
    `localize_radius` is the Gaspari-Cohn half-width in km (the weight reaches zero at twice that);
    `assimilate_this` defaults to False, as in the reference."""

    def __init__(self, value=None, obtype=None, time=None, error=None, lat=None,
                 lon=None, vert=None,
                 prior_mean=None, post_mean=None, prior_var=None, post_var=None,
                 assimilate_this=False, description=None, localize_radius=None):
        self.value = value
        self.obtype = obtype
        self.time = time
        self.error = error
        self.lat = lat
        self.lon = lon
        self.vert = vert
        self.prior_mean = prior_mean
        self.post_mean = post_mean
        self.prior_var = prior_var
        self.post_var = post_var
        self.assimilate_this = assimilate_this
        self.assimilated = False
        self.description = description
        self.localize_radius = localize_radius

    def estimate(self, state, forward_operator='reference'):
        """Ensemble estimate of this observation: the state interpolated to the ob (observation.py:40-50), with the
        forward operator of EnsembleState.interpolate."""
        return state.interpolate(self.obtype, self.time, self.lat, self.lon, forward_operator=forward_operator)

    def distance_to_state(self, state):
        """Distance in km from this ob to every grid point (observation.py:53-56)."""
        return state.distance_to_point(self.lat, self.lon)

    def localize(self, state, type='GC', full_state=False):
        """Localisation weights of this ob for a state (-> [ny, nx]) or a list of obs (-> [nobs])
        (observation.py:59-87)."""
        import torch
        halfwidth = self.localize_radius
        _lib.require_device()
        if isinstance(state, EnsembleState):
            grid = state._grid_tables()
            u, n = (grid.u1, grid.nx) if grid.diag else (grid.u, grid.npts)      # 1-D lat/lon: one weight per point
            shape, dev = state['lat'].shape, grid.device
        else:
            dev = torch.device('cuda', torch.cuda.current_device())
            lat = torch.as_tensor(np.array([ob.lat for ob in state], dtype=np.float64)).to(dev)
            lon = torch.as_tensor(np.array([ob.lon for ob in state], dtype=np.float64)).to(dev)
            n, shape = lat.shape[0], (lat.shape[0],)
            u = torch.empty((3, n), dtype=torch.float64, device=dev)
            _lib.call('exb_grid_unitvec', _lib.ptr(lat), _lib.ptr(lon), n, _lib.ptr(u), _lib.stream_ptr())
        if type == 'GC':
            if halfwidth is None:
                abs(halfwidth)          # TypeError, as gaspari_cohn(distances, None) in the reference
            mode, hw = 1, float(halfwidth)
        elif halfwidth is None:
            mode, hw = 0, 1.0           # "return an array of ones", observation.py:77-79
        else:
            raise UnboundLocalError("localization type %r is not implemented (only 'GC')" % (type,))
        w = torch.empty(n, dtype=torch.float64, device=dev)
        _lib.call('exb_localization_weights', _lib.ptr(u), n, float(self.lat), float(self.lon), hw, mode, None,
                  _lib.ptr(w), _lib.stream_ptr())
        return w.cpu().numpy().reshape(shape)


def gaspari_cohn(distances, halfwidth):
    """Gaspari-Cohn weights of a distance array for a half-width (observation.py:117-130)."""
    import torch
    _lib.require_device()
    d = np.ascontiguousarray(distances, dtype=np.float64)
    dev = torch.device('cuda', torch.cuda.current_device())
    dd = torch.as_tensor(d.ravel()).to(dev)
    w = torch.empty_like(dd)
    _lib.call('exb_gaspari_cohn', _lib.ptr(dd), dd.shape[0], float(abs(halfwidth)), _lib.ptr(w), _lib.stream_ptr())
    return w.cpu().numpy().reshape(d.shape)


def haversine(loc1, loc2):
    """Great-circle distance in km between two (lat, lon) pairs, R = 6371 km (observation.py:135-146)."""
    R = 6371.
    lat1 = math.radians(loc1[0])
    lat2 = math.radians(loc2[0])
    dlat = lat2 - lat1
    dlon = math.radians(loc2[1] - loc1[1])
    a = math.sin(dlat / 2) ** 2 + math.cos(lat1) * math.cos(lat2) * math.sin(dlon / 2) ** 2
    c = 2 * math.atan2(math.sqrt(a), math.sqrt(1 - a))
    return R * c
