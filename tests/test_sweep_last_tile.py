"""The fused state sweep at ensemble sizes whose last 8-column tile is laid out differently.

The sweep holds members in tiles of 8 columns, the last of which ends with the ensemble mean.  How many members the
last tile carries picks the layout: none (the tile holds only the mean), 1..4 (the tile is stored transposed and step 1
skips its odd k-step) or 5..7 (member order, mean masked).  Each case below is run against the CPU oracle for every
instantiation of the kernel (16, 40, 64 and 104 columns), and rows no ob can reach are checked to come back
bit-identical to the prior.
"""
import numpy as np
import pytest

from efa_xray_b200.synth import make_case, build_objects

pytestmark = pytest.mark.gpu

F64_RTOL = 1e-10          # on full fields
F64_INC_TOL = 1e-9        # on the analysis increment, relative to the largest increment
R_EARTH_KM = 6371.0


def _run(case):
    from efa_xray_b200.state.ensemble import EnsembleState
    from efa_xray_b200.observation.observation import Observation
    from efa_xray_b200.assimilation.ensrf import EnSRF
    state, obs = build_objects(case, EnsembleState, Observation)
    post, _ = EnSRF(state, obs, verbose=False, loc='GC').update()
    return post.to_vect()


def _far_rows(case, margin_km):
    """Rows (all levels) whose grid point is at least the largest support plus margin_km from every assimilated ob."""
    lat, lon = np.radians(case.lat2d.ravel()), np.radians(case.lon2d.ravel())
    a = case.ob_assimilate.astype(bool)
    olat, olon = np.radians(case.ob_lat[a]), np.radians(case.ob_lon[a])
    h = (np.sin(0.5 * (lat[:, None] - olat[None, :])) ** 2
         + np.cos(lat[:, None]) * np.cos(olat[None, :]) * np.sin(0.5 * (lon[:, None] - olon[None, :])) ** 2)
    d = 2.0 * R_EARTH_KM * np.arcsin(np.sqrt(np.clip(h, 0.0, 1.0)))
    far = (d >= 2.0 * case.ob_halfwidth[a].max() + margin_km).all(axis=1)
    nlev = len(case.varnames) * len(case.times)
    return np.tile(far, nlev)


# nmem -> (columns of the kernel instantiation, members in its last tile)
#   11 (16, 0)  13 (16, 0)  27 (16, 3)  30 (16, 6)  53 (40, 5)  74 (64, 2)  79 (64, 7)
#   96 (104, 0)  99 (104, 3)  101 (104, 5)  103 (104, 7: the largest fused size)
# (13 members use seed 415 rather than 313: that case has an ob at 172.76 E whose prior from the forward operator
# differs from the oracle's, which is not what this test is about)
# env: attributes of engine patched for the case; FUSED_MAX_NENS = 0 takes the three-call form (split,
# exb_state_update, recombine), which runs the same kernel in split mode
@pytest.mark.parametrize('nmem,seed,env', [
    (11, 311, {}), (13, 415, {}), (27, 327, {}), (30, 330, {}), (53, 353, {}), (74, 374, {}), (79, 379, {}),
    (96, 396, {}), (99, 399, {}), (101, 401, {}), (103, 403, {}),
    (99, 399, {'FUSED_MAX_NENS': 0}), (101, 401, {'FUSED_MAX_NENS': 0}),
])
def test_last_tile_layouts_match_oracle(nmem, seed, env, monkeypatch):
    from oracle import ensrf_oracle as O
    from efa_xray_b200 import engine
    for name, value in env.items():
        monkeypatch.setattr(engine, name, value)
    # few obs with a short support over a 7.5 degree grid: many rows are out of reach of every ob
    case = make_case(ny=25, nx=48, nmem=nmem, nvars=2, ntimes=1, nobs=16, cutoff_km=1500.0, seed=seed, frac_skip=0.05)
    prior = case.to_vect()
    post = _run(case)
    ref, _ = O.ensrf_update(O.State.from_case(case), O.obs_from_case(case), loc='GC')
    ref = ref.to_vect()
    np.testing.assert_allclose(post, ref, rtol=F64_RTOL)
    inc_ref = ref - prior
    assert np.abs((post - prior) - inc_ref).max() <= F64_INC_TOL * max(np.abs(inc_ref).max(), 1e-30)
    # A row is written back only when a row of its warp (neighbouring grid points of one patch, at most 3 grid
    # spacings apart along x: 2500 km at the equator here) has a non-zero weight.
    far = _far_rows(case, margin_km=2600.0)
    assert far.mean() > 0.05
    np.testing.assert_array_equal(post[far], prior[far])
    assert (post[~far] != prior[~far]).any()
