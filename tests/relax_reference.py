"""Numpy reference of posterior relaxation (RTPS / RTPP, DESIGN.md section 4.6), composed with the CPU oracle's
serial EnSRF (oracle/ensrf_oracle.py, which stays the restatement of the unmodified reference and is not changed).

TEST INFRASTRUCTURE, NOT PRODUCT: the GPU relaxation is checked against this module."""
import numpy as np

from oracle import ensrf_oracle as O


def relax(prior_vect, post_vect, kind, alpha_rows):
    """Relaxed copy of the analysis rows post_vect [nrows, nens] toward the prior rows prior_vect, one alpha per row.

    RTPS: x = m_a + x'_a (1 + alpha (sigma_b - sigma_a) / sigma_a);  RTPP: x = m_a + (1 - alpha) x'_a + alpha x'_b,
    with sigma the ensemble standard deviation (ddof = 1; exactly 0 when every member is equal).  A row is left as it is when alpha = 0, sigma_a = 0, or
    nothing changed it (RTPS: sigma_a == sigma_b; RTPP: every member equals the prior's)."""
    xb = np.asarray(prior_vect, dtype=np.float64)
    xa = np.asarray(post_vect, dtype=np.float64)
    a = np.broadcast_to(np.asarray(alpha_rows, dtype=np.float64).ravel(), (xa.shape[0],))
    ma, mb = xa.mean(axis=1), xb.mean(axis=1)
    # sigma is exactly 0 for a row of equal members (its rounded mean may differ from them)
    sa = np.where((xa == xa[:, :1]).all(axis=1), 0.0, xa.std(axis=1, ddof=1))
    sb = np.where((xb == xb[:, :1]).all(axis=1), 0.0, xb.std(axis=1, ddof=1))
    pa, pb = xa - ma[:, None], xb - mb[:, None]
    if kind == 'rtps':
        with np.errstate(divide='ignore', invalid='ignore'):      # sigma_a = 0 rows are kept below
            f = 1.0 + a * (sb - sa) / sa
            new = ma[:, None] + pa * f[:, None]
        keep = (sa == sb)
    elif kind == 'rtpp':
        new = ma[:, None] + (1.0 - a)[:, None] * pa + a[:, None] * pb
        keep = (xa == xb).all(axis=1)
    else:
        raise ValueError(kind)
    keep = keep | (a == 0.0) | (sa == 0.0)
    return np.where(keep[:, None], xa, new)


def alpha_rows(state, alpha):
    """Per-row alphas of a float or {variable name: float} alpha for an oracle State (rows var -> time -> y -> x)."""
    nv, nt, ny, nx, _ = state.shape()
    if isinstance(alpha, dict):
        per_var = np.array([float(alpha.get(v, 0.0)) for v in state.varnames])
    else:
        per_var = np.full(nv, float(alpha))
    return np.repeat(per_var, nt * ny * nx)


def ensrf_update(state, obs, loc='GC', inflation=None, relaxation=None):
    """O.ensrf_update with posterior relaxation: relaxation None, ('rtps', alpha) or ('rtpp', alpha).  The prior of
    the relaxation is the state format_prior_state returns, i.e. after prior inflation."""
    xam, Xap, state = O.format_prior_state(state, obs, inflation)
    prior = state.to_vect().copy()
    xam, Xap = O.ensrf_loop(state, obs, xam, Xap, loc=loc)
    post_state = state.copy()
    post = (xam[:, None] + Xap)[:state.nstate()]
    if relaxation is not None:
        kind, alpha = relaxation
        post = relax(prior, post, kind, alpha_rows(state, alpha))
    post_state.from_vect(post)
    return post_state, obs
