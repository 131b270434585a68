#!/usr/bin/env python
"""Generate golden vectors by running the UNMODIFIED reference package.

Run in the build container only (it reads /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference (lmadaus/efa_xray) needs xarray/netCDF4/matplotlib/pytz and a Python-2 module
(cPickle); none are installable here.  tests/golden/refshim/ provides a minimal stand-in for
the xarray surface the reference touches plus empty stubs for the unused imports, so that the
reference's own arithmetic -- EnSRF.update (assimilation/ensrf.py:33-151),
Assimilation.format_prior_state / compute_ob_priors (assimilation/assimilation.py:36-49,120-171),
EnsembleState.interpolate / nearest_points / distance_to_point (state/ensemble.py:152-267),
Observation.localize / gaspari_cohn / haversine (observation/observation.py:59-146) -- runs
unchanged.  Inputs come from efa_xray_b200.synth.make_case(seed, ...) and are NOT stored; only the
case parameters and the reference's outputs are written to tests/golden/*.npz.
"""
import os
import sys
import json
from copy import deepcopy

import numpy as np
import pandas  # noqa: F401  imported BEFORE the stubs go on sys.path (pandas probes for a real pytz)

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(HERE, 'refshim'))
sys.path.insert(1, '/root/reference')
sys.path.append(REPO)

from efa_xray.state.ensemble import EnsembleState            # noqa: E402  (the reference)
from efa_xray.observation.observation import Observation, gaspari_cohn, haversine  # noqa: E402
from efa_xray.assimilation.ensrf import EnSRF                 # noqa: E402
import efa_xray                                               # noqa: E402
assert efa_xray.__file__.startswith('/root/reference'), efa_xray.__file__

from efa_xray_b200.synth import make_case, make_case_1d, build_objects      # noqa: E402

# name -> (make_case kwargs, loc, inflation)
CASES = {
    'gc_small': (dict(ny=19, nx=36, nmem=8, nvars=1, ntimes=1, nobs=40, cutoff_km=4000.0, seed=0,
                      frac_skip=0.1), 'GC', None),
    'gc_multivar_offtime': (dict(ny=25, nx=48, nmem=10, nvars=2, ntimes=2, nobs=60, cutoff_km=3000.0,
                                 seed=1, frac_skip=0.05, mixed_error=True, offtime=True,
                                 mixed_radius=True), 'GC', None),
    'noloc_small': (dict(ny=19, nx=36, nmem=6, nvars=1, ntimes=1, nobs=20, cutoff_km=4000.0, seed=2),
                    False, None),
    'gc_4deg': (dict(ny=46, nx=90, nmem=20, nvars=1, ntimes=2, nobs=100, cutoff_km=2000.0, seed=3,
                     frac_skip=0.05), 'GC', None),
    'gc_inflate': (dict(ny=19, nx=36, nmem=8, nvars=2, ntimes=1, nobs=30, cutoff_km=5000.0, seed=4),
                   'GC', 1.5),
    # more obs than one panel / batch, many overlapping supports, mixed radii and errors, skipped obs
    'gc_dense300': (dict(ny=37, nx=72, nmem=12, nvars=2, ntimes=1, nobs=300, cutoff_km=1500.0, seed=5,
                         frac_skip=0.05, mixed_error=True, mixed_radius=True), 'GC', None),
    # inflation as a per-variable dict (assimilation.py:101-114), incl. a name that is not a state variable
    'gc_inflate_vardict': (dict(ny=19, nx=36, nmem=8, nvars=3, ntimes=2, nobs=30, cutoff_km=5000.0, seed=6),
                           'GC', {'var0': 1.3, 'var2': 1.7, 'nosuchvar': 2.0}),
    # inflation per dimension (assimilation.py:83-100): arrays along validtime, y and x, plus one variable factor
    'gc_inflate_dims': (dict(ny=19, nx=36, nmem=8, nvars=2, ntimes=2, nobs=30, cutoff_km=5000.0, seed=7),
                        'GC', {'validtime': [1.1, 1.4], 'y': ('linspace', 1.0, 1.5, 19), 'var1': 1.2,
                               'x': ('linspace', 1.3, 0.9, 36)}),
    # 1-D lat(x)/lon(x) coordinates: the reference's second branch (state/ensemble.py:185-192, ensrf.py:110-111)
    'gc_1d_points': (dict(one_d=True, npts=24, nmem=8, nvars=2, ntimes=1, nobs=30, cutoff_km=4000.0, seed=8,
                          frac_skip=0.1), 'GC', None),
}


def decode_inflation(infl):
    """JSON-able inflation spec -> what EnSRF takes: lists / ('linspace', a, b, n) become float arrays."""
    if not isinstance(infl, dict):
        return infl
    out = {}
    for k, v in infl.items():
        if isinstance(v, (list, tuple)) and len(v) == 4 and v[0] == 'linspace':
            out[k] = np.linspace(float(v[1]), float(v[2]), int(v[3]))
        elif isinstance(v, (list, tuple)):
            out[k] = np.array(v, dtype=np.float64)
        else:
            out[k] = v
    return out


def run_case(name, kw, loc, inflation):
    if kw.get('one_d'):
        case = make_case_1d(**{k: v for k, v in kw.items() if k != 'one_d'})
    else:
        kw = dict(kw, avoid_mirror_ties=True)
        case = make_case(**kw)
    state, obs = build_objects(case, EnsembleState, Observation)
    prior_vect = state.to_vect().copy()

    # forward operator outputs for every ob, before anything is modified
    ye = np.array([ob.estimate(state) for ob in obs])
    near = np.array([np.array(state.nearest_points(ob.lat, ob.lon, npt=4)) for ob in obs])   # [nobs,2,4] (1-D: [nobs,1,4])
    loc_state0 = obs[0].localize(state, type='GC') if loc == 'GC' else np.zeros((1, 1))
    loc_obs0 = obs[0].localize(obs, type='GC') if loc == 'GC' else np.zeros(1)

    import io
    import contextlib
    with contextlib.redirect_stdout(io.StringIO()):     # "Unable to find variable ... Skipping"
        post_state, post_obs = EnSRF(state, obs, inflation=decode_inflation(inflation), verbose=False, loc=loc).update()
    post_vect = post_state.to_vect()
    # stored as post - prior, which keeps the files small (tests/conftest.py:load_golden adds back the prior
    # regenerated from the seed); the round trip must be exact
    post_minus_prior = post_vect - prior_vect
    assert np.array_equal(prior_vect + post_minus_prior, post_vect), name
    f = lambda attr: np.array([np.nan if getattr(o, attr) is None else float(getattr(o, attr))
                               for o in post_obs])
    out = dict(
        params=json.dumps(dict(kw=kw, loc=loc, inflation=inflation)),
        prior_checksum=np.array([prior_vect.sum(), np.abs(prior_vect).sum()]),
        # the caller's state after the call (inflated in place by the float / per-variable forms only)
        prior_after_checksum=np.array([state.to_vect().sum(), np.abs(state.to_vect()).sum()]),
        ye=ye, nearest=near, loc_state0=loc_state0, loc_obs0=loc_obs0,
        post_minus_prior=post_minus_prior,
        prior_mean=f('prior_mean'), prior_var=f('prior_var'),
        post_mean=f('post_mean'), post_var=f('post_var'),
        assimilated=np.array([bool(o.assimilated) for o in post_obs]),
    )
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print('%-22s Nstate=%d Nens=%d Nobs=%d  assimilated=%d  |post-prior|max=%.3e'
          % (name, post_vect.shape[0], post_vect.shape[1], len(obs), out['assimilated'].sum(),
             np.abs(post_vect - (prior_vect if inflation is None else post_vect)).max()))


def function_vectors():
    """Known-answer vectors for the free functions."""
    rng = np.random.default_rng(123)
    d = np.concatenate([np.array([0.0, 1e-9, 250.0, 999.999, 1000.0, 1000.001, 1999.999, 2000.0, 2000.001, 5e4]),
                        rng.uniform(0, 2500, 200)])
    gc = gaspari_cohn(d, 1000.0)
    gc_neg = gaspari_cohn(d, -1000.0)
    pairs = np.column_stack([rng.uniform(-90, 90, 300), rng.uniform(-180, 360, 300),
                             rng.uniform(-90, 90, 300), rng.uniform(-180, 360, 300)])
    pairs[0] = (0, 0, 0, 90)
    pairs[1] = (10, 20, 10, 20)
    pairs[2] = (90, 0, -90, 0)
    pairs[3] = (0, 0, 0, 180)
    hv = np.array([haversine((p[0], p[1]), (p[2], p[3])) for p in pairs])
    # the 1-km branch of interpolate raises in the reference (state/ensemble.py:195-196)
    case = make_case(ny=19, nx=36, nmem=4, nobs=1, seed=9)
    state, obs = build_objects(case, EnsembleState, Observation)
    obs[0].lat, obs[0].lon = 10.0, 20.0     # exactly on a grid point
    try:
        obs[0].estimate(state)
        raised = ''
    except Exception as e:                  # noqa: BLE001
        raised = type(e).__name__
    # ob outside the state's time range returns None (state/ensemble.py:206-208)
    import datetime as dt
    obs[0].lat, obs[0].lon = 11.3, 21.7
    obs[0].time = dt.datetime(2031, 1, 1)
    import io
    import contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        outside = obs[0].estimate(state)
    np.savez_compressed(os.path.join(HERE, 'functions.npz'), gc_d=d, gc_w=gc, gc_w_neg=gc_neg,
                        hv_pairs=pairs, hv_km=hv, exact_point_raises=np.array(raised),
                        outside_time_is_none=np.array(outside is None))
    print('functions: GC(0)=%.17g GC(c)=%.17g GC(2c)=%.3g  hav(0,0->0,90)=%.6f  exact-point raises %r  outside-time None=%s'
          % (gc[0], gc[4], gc[7], hv[0], raised, outside is None))


if __name__ == '__main__':
    only = sys.argv[1:]
    if not only:
        function_vectors()
    for name, (kw, loc, infl) in CASES.items():
        if not only or name in only:
            run_case(name, kw, loc, infl)
