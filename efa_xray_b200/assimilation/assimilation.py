"""Assimilation base class and the module-level update() entry point
(efa_xray/assimilation/assimilation.py:10-230)."""
from __future__ import print_function

from copy import deepcopy

import numpy as np

import efa_xray_b200 as _pkg
from .. import _lib
from .. import engine


class ObTimeOutsideState(AttributeError, ValueError):
    """An observation's time is outside the state's valid times.  The reference's interpolate returns None
    there (state/ensemble.py:206-208) and compute_ob_priors then dies with AttributeError on `.mean()`
    (assimilation/assimilation.py:47); this is that failure with a message."""


class Assimilation():
    """Computes obs priors and formats the state for the update (assimilation.py:10-171)."""

    def __init__(self, state, obs, nproc=1, inflation=None, verbose=False, forward_operator='reference'):
        """inflation: None, a float (all variables), or a dict of {variable name: float} and/or
        {'validtime' | 'y' | 'x' (| 'lat' | 'lon' when 1-D): array along that dimension}
        (assimilation.py:19-26; the netCDF file-name form needs xarray and is not ported).
        nproc is accepted and ignored, as in the reference (assimilation.py:31).
        forward_operator (not in the reference): 'reference' (default), the reference's 4-point inverse-distance
        operator with its time weights, or 'bilinear', bilinear in space on the grid cell that contains the ob and
        linear in time with correctly oriented weights (DESIGN.md section 4.8; needs 2-D lat/lon).  An unknown name,
        or 'bilinear' on a state with 1-D lat/lon, raises ValueError here, before any device work."""
        engine.check_forward_operator(forward_operator, np.ndim(state['lat'].values))
        self.forward_operator = forward_operator
        self.prior = state
        self.obs = obs
        self.verbose = verbose
        self.nproc = nproc
        self.inflation = inflation
        self.is_inflated = False
        # the reference also deep-copies the state into self.post and never uses it (assimilation.py:29)

    # ---- marshalling ------------------------------------------------------------------
    def _loc_mode(self, loc):
        if loc in [None, False]:
            return engine.LOC_NONE
        if loc == 'GC':
            return engine.LOC_GC
        raise ValueError("loc must be None, False or 'GC' (got %r); other localisation types are not "
                         "defined by the reference (observation/observation.py:82)" % (loc,))

    def _obs_arrays(self, loc_mode, outlier_threshold=None):
        """Structure-of-arrays view of self.obs with the forward-operator bookkeeping per ob.  One pass over the list
        (operator.attrgetter pulls the eight attributes of an ob in C); everything after that is vectorised.
        outlier_threshold (validated by _validate_outlier_threshold) becomes the per-ob threshold array: the float for
        every ob, or a dict's value for the obs of that variable and inf (not checked) for the others."""
        from operator import attrgetter
        st = self.prior
        obs = self.obs
        varnames = st.vars()
        nt, ny, nx = st.ntimes(), st.ny(), st.nx()
        n = len(obs)
        if n:
            cols = list(zip(*map(attrgetter('value', 'error', 'lat', 'lon', 'obtype', 'time', 'assimilate_this',
                                            'localize_radius'), obs)))
        else:
            cols = [()] * 8
        value, error, lat, lon, obtype, obtime, flag, radius = cols
        vidx = {v: i for i, v in enumerate(varnames)}
        try:
            var = np.fromiter(map(vidx.__getitem__, obtype), dtype=np.int64, count=n)
        except KeyError as e:
            raise KeyError('observation type %s is not a state variable %r' % (e, varnames))
        # ob times: converting 1e5 datetime objects one by one is slow, and obs usually share a handful of distinct
        # times -- convert the distinct ones and index
        uniq = {}
        codes = np.fromiter((uniq.setdefault(t, len(uniq)) for t in obtime), dtype=np.int64, count=n)
        utimes = np.array([np.datetime64(t) for t in uniq], dtype='datetime64[ns]') if uniq else \
            np.zeros(0, dtype='datetime64[ns]')
        times = utimes[codes] if n else np.zeros(0, dtype='datetime64[ns]')
        tlo, thi, wlo, whi, outside = engine.time_weights(st['validtime'].values, times,
                                                          swapped=self.forward_operator == 'reference')
        if outside.any():
            print("Interpolation is outside of time range in state!")
            raise ObTimeOutsideState("observation %d (time %s) is outside the state's valid times"
                                     % (int(np.argmax(outside)), obs[int(np.argmax(outside))].time))
        assim = np.fromiter(map(bool, flag), dtype=np.bool_, count=n).astype(np.uint8)
        hw = np.ones(n)
        if loc_mode == engine.LOC_GC:
            # abs(localize_radius) of the obs that will be assimilated: TypeError on None, as observation.py:120
            radii = [r if f else 1.0 for r, f in zip(radius, flag)]
            if any(r is None for r in radii):
                abs(None)                                # numpy would turn None into NaN silently
            hw = np.abs(np.array(radii, dtype=np.float64))
        thr = np.zeros(0)                                             # no check
        if isinstance(outlier_threshold, dict):
            per_var = np.full(len(varnames), np.inf)
            for k, t in outlier_threshold.items():
                per_var[varnames.index(k)] = float(t)
            thr = per_var[var]
        elif outlier_threshold is not None:
            thr = np.full(n, float(outlier_threshold))
        return engine.ObsArrays(
            value=np.array(value, dtype=np.float64), error=np.array(error, dtype=np.float64),
            lat=np.array(lat, dtype=np.float64), lon=np.array(lon, dtype=np.float64),
            halfwidth=hw, assimilate=assim,
            row0=(var * nt + tlo) * (ny * nx), row1=(var * nt + thi) * (ny * nx), tw0=wlo, tw1=whi, threshold=thr)

    _DIM_KEYS = ['validtime', 'lat', 'lon', 'x', 'y']

    def _inflation_factors(self, inflation=None):
        """Multiplicative inflation factors, or None: shape (nvars*ntimes,) -- one per level, for a float or a
        per-variable dict (assimilation.py:62-69, :101-114) -- or (nvars, ntimes, ny, nx) flattened to one factor per
        state row when the dict has per-dimension arrays (assimilation.py:83-100: validtime / y / x, and lat / lon
        when those are 1-D coordinates; the reference multiplies the perturbations by each array in turn, broadcast
        along its dimension, so the factors multiply)."""
        inflation = self.inflation if inflation is None else inflation
        if inflation is None:
            return None
        st = self.prior
        varnames = st.vars()
        nt = st.ntimes()
        fac = np.ones((len(varnames), nt))
        field = None                                                   # [nt, ny, nx] per-dimension product
        if isinstance(inflation, float):
            fac[:] = inflation                                        # assimilation.py:62-69
        elif isinstance(inflation, dict):
            for k, v in inflation.items():                            # assimilation.py:82-114, in dict order
                if k in self._DIM_KEYS:
                    v = np.asarray(v, dtype=np.float64)
                    coord = st.coords[k]
                    assert v.ndim == 1 and v.shape[0] == len(coord)   # assimilation.py:87-88
                    if len(coord.dims) != 1:
                        # DataArray(v, [(k, 2-D coordinate values)]) cannot be built in the reference either
                        raise ValueError('inflation along %r needs a 1-D %r coordinate (it has dims %r)'
                                         % (k, k, coord.dims))
                    if field is None:
                        field = np.ones((nt, st.ny(), st.nx()))
                    ax = ('validtime', 'y', 'x').index(coord.dims[0])
                    shape = [1, 1, 1]
                    shape[ax] = v.shape[0]
                    field = field * v.reshape(shape)
                    continue
                assert isinstance(v, float)
                if k not in varnames:
                    print("Unable to find variable {:s} to inflate.  Skipping...".format(k))
                    continue
                fac[varnames.index(k), :] = fac[varnames.index(k), :] * v
        else:
            raise NotImplementedError('inflation from a netCDF file name needs xarray (assimilation.py:71-79)')
        if field is not None:
            return (fac[:, :, None, None] * field[None]).ravel()
        return fac.ravel()

    @staticmethod
    def _check_alpha(a, what):
        if isinstance(a, bool) or not isinstance(a, (int, float, np.integer, np.floating)):
            raise ValueError('relaxation alpha %s must be a float, got %r' % (what, a))
        if not 0.0 <= float(a) <= 1.0:                            # NaN fails here too
            raise ValueError('relaxation alpha %s must lie in [0, 1], got %r' % (what, a))

    def _validate_relaxation(self, relaxation):
        """None, ('rtps', a) or ('rtpp', a) with a a float in [0, 1] or a dict {variable name: float}; raises
        ValueError otherwise.  Only reads the state's variable names (no device work)."""
        if relaxation is None:
            return
        if not isinstance(relaxation, (tuple, list)) or len(relaxation) != 2:
            raise ValueError("relaxation must be None, ('rtps', alpha) or ('rtpp', alpha), got %r" % (relaxation,))
        kind, alpha = relaxation
        if kind not in engine.RELAX_KINDS:
            raise ValueError('relaxation kind must be one of %r, got %r' % (engine.RELAX_KINDS, kind))
        if isinstance(alpha, dict):
            varnames = self.prior.vars()
            for k, v in alpha.items():
                if k not in varnames:
                    raise ValueError('relaxation names %r, which is not a state variable %r' % (k, varnames))
                self._check_alpha(v, 'of %r' % (k,))
        else:
            self._check_alpha(alpha, '')

    @staticmethod
    def _check_threshold(t, what):
        if isinstance(t, bool) or not isinstance(t, (int, float, np.integer, np.floating)):
            raise ValueError('outlier threshold %s must be a float, got %r' % (what, t))
        if not 0.0 < float(t) < np.inf:                           # NaN fails here too
            raise ValueError('outlier threshold %s must be positive and finite, got %r' % (what, t))

    def _validate_outlier_threshold(self, outlier_threshold):
        """None, a positive finite float, or a dict {variable name: positive finite float}; raises ValueError
        otherwise.  Only reads the state's variable names (no device work)."""
        if outlier_threshold is None:
            return
        if isinstance(outlier_threshold, dict):
            varnames = self.prior.vars()
            for k, t in outlier_threshold.items():
                if k not in varnames:
                    raise ValueError('outlier_threshold names %r, which is not a state variable %r' % (k, varnames))
                self._check_threshold(t, 'of %r' % (k,))
        else:
            self._check_threshold(outlier_threshold, '')

    def _relaxation_levels(self, relaxation):
        """(kind, alpha per level) for engine.analysis_*, or None: one alpha per (variable, time) level, in the
        order of the state rows (as _inflation_factors orders inflation factors); variables a dict does not name get
        0."""
        if relaxation is None:
            return None
        kind, alpha = relaxation
        st = self.prior
        varnames = st.vars()
        a = np.zeros((len(varnames), st.ntimes()))
        if isinstance(alpha, dict):
            for k, v in alpha.items():
                a[varnames.index(k), :] = float(v)
        else:
            a[:] = float(alpha)
        return kind, a.ravel()

    def _host_matrix(self):
        """[Nstate, Nens] host matrix of the prior in to_vect layout: the state's own block when it has one (no
        copy; callers only read it or hand it to the device), else a stacked copy."""
        st = self.prior
        if hasattr(st, '_consolidate'):
            st._consolidate()
            blk = st._block_view()
            if blk is not None:
                return blk.reshape(st.nstate(), st.nmems())
        return np.ascontiguousarray(st.to_vect())

    def _device(self):
        import torch
        _lib.require_device()
        return torch.device('cuda', torch.cuda.current_device())

    # ---- reference methods --------------------------------------------------------------
    def compute_ob_priors(self):
        """Prior means [nobs] and perturbations [nobs, nmems] of every ob (assimilation.py:36-49)."""
        import torch
        dev = self._device()
        obs = self._obs_arrays(engine.LOC_NONE)
        X = torch.from_numpy(self._host_matrix()).to(dev)
        grid = self.prior._grid_tables()
        Y, nex = engine.ob_priors(X, grid, obs, engine._sfx(X.dtype), forward_operator=self.forward_operator)
        if self.forward_operator == 'bilinear':
            self._check_outside(int(nex.item()))
        else:
            self._check_exact(int(nex.item()))
        Ym = torch.empty(obs.nobs, dtype=X.dtype, device=dev)
        sfx = engine._sfx(X.dtype)
        _lib.call('exb_split_mean_pert_' + sfx, _lib.ptr(Y), _lib.ptr(Ym), obs.nobs, X.shape[1], _lib.stream_ptr())
        return Ym.cpu().numpy().astype(np.float64), Y.cpu().numpy().astype(np.float64)

    @staticmethod
    def _check_exact(n_exact):
        if n_exact > 0 and _pkg.EXACT_MATCH_POLICY == 'raise':
            raise IndexError('%d observation(s) lie within 1 km of a grid point: the reference raises here '
                             '(state/ensemble.py:195-196); set efa_xray_b200.EXACT_MATCH_POLICY = "nearest" '
                             'to use the nearest point instead' % n_exact)

    @staticmethod
    def _check_outside(n_outside):
        if n_outside > 0:
            raise ValueError("%d observation(s) lie outside the grid, where forward_operator='bilinear' has no cell "
                             "to interpolate from (DESIGN.md section 4.8)" % n_outside)

    def _apply_inflation(self, fac):
        import ctypes as C
        import torch
        dev = self._device()
        X = torch.from_numpy(self._host_matrix()).to(dev)
        sfx = engine._sfx(X.dtype)
        _lib.call('exb_inflate_' + sfx, _lib.ptr(X), X.shape[0], X.shape[1], fac.ctypes.data_as(C.c_void_p), fac.shape[0],
                  X.shape[0] // fac.shape[0], _lib.stream_ptr())
        self.prior.from_vect(X.cpu().numpy())

    def inflate_state(self):
        """Inflate self.prior about its ensemble mean (assimilation.py:52-118).

        As in the reference, a float and per-variable entries change the caller's state IN PLACE
        (`variables[v][:] = ...`, :65, :113), while the first per-dimension entry REBINDS self.prior to a new state
        (`self.prior = perts * infl + mean`, :96): the caller's object keeps what had been applied before it, and
        everything from there on acts on the new one."""
        if self.is_inflated:
            print("State already inflated.  Skipping additional inflation.")
            return
        if isinstance(self.inflation, dict):
            items = list(self.inflation.items())
            first_dim = next((i for i, (k, _) in enumerate(items) if k in self._DIM_KEYS), len(items))
            pre, post = dict(items[:first_dim]), dict(items[first_dim:])
            if pre:
                self._apply_inflation(self._inflation_factors(pre))
            if post:
                self.prior = deepcopy(self.prior)
                self._apply_inflation(self._inflation_factors(post))
        else:
            self._apply_inflation(self._inflation_factors())
        self.is_inflated = True

    def format_prior_state(self):
        """(xbm [Nstate+Nobs], Xbp [Nstate+Nobs, Nens]): ensemble mean and perturbations of the state with
        the ob priors appended as extra rows (assimilation.py:120-154)."""
        import torch
        if self.inflation is not None:
            if self.verbose: print("Inflating Prior State")
            self.inflate_state()
        if self.verbose: print("Computing observation priors")
        obmeans, obperts = self.compute_ob_priors()
        if self.verbose: print("Converting state to vector")
        dev = self._device()
        X = torch.from_numpy(self._host_matrix()).to(dev)
        xm = torch.empty(X.shape[0], dtype=X.dtype, device=dev)
        _lib.call('exb_split_mean_pert_' + engine._sfx(X.dtype), _lib.ptr(X), _lib.ptr(xm), X.shape[0], X.shape[1],
                  _lib.stream_ptr())
        xbm = np.hstack((xm.cpu().numpy(), obmeans))
        Xbp = np.vstack((X.cpu().numpy(), obperts))
        return xbm, Xbp

    def format_posterior_state(self, xam, Xap):
        """Posterior state object from analysis mean and perturbations (assimilation.py:157-171)."""
        if self.verbose: print("Formatting posterior")
        post_state = deepcopy(self.prior)
        Nstate = self.prior.nstate()
        post = (xam[:, None] + Xap)[:Nstate]
        post_state.from_vect(post)
        return post_state, self.obs


def update(prior_state, obs, inflate=None, loc=False, nproc=1, verbose=False, relaxation=None, outlier_threshold=None,
           forward_operator='reference'):
    """Module-level entry point (assimilation.py:176-222).  In the reference this calls an undefined
    enkf_update; here it runs the EnSRF.  nproc is accepted for signature compatibility: the GPU path does
    not fork worker processes.  relaxation: posterior relaxation, outlier_threshold: outlier quality control,
    forward_operator: the forward operator H, all as for EnSRF."""
    from .ensrf import EnSRF
    return EnSRF(prior_state, obs, nproc=nproc, inflation=inflate, verbose=verbose, loc=loc,
                 relaxation=relaxation, outlier_threshold=outlier_threshold, forward_operator=forward_operator).update()


def randomize_obs_order(obs, seed=None):
    """Shuffle a list of observations in place and return it: the demo notebook assimilates in random order
    (efa_demo.ipynb cell 11, lines 44-46).  With localisation the analysis depends on the serial order, so the
    order used is part of the experiment; pass a seed to make it reproducible."""
    rng = np.random.default_rng(seed)
    perm = rng.permutation(len(obs))
    obs[:] = [obs[i] for i in perm]
    return obs
