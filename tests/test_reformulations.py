"""CPU checks of the algebraic reformulations the CUDA path rests on, against the oracle's serial loop
(oracle.obs_space_solve restates the obs rows of ensrf.py:50-149):

* the obs-space solve as a dependency-driven (sparse triangular) solve: a row needs only the published records of the
  EARLIER obs whose support reaches it, applied in index order; rows can then be processed in any order compatible
  with those dependencies, by any number of workers (obs_solve_dag.cu, its distributed variant);
* the blocked 8-ob form of the state update (Gram recurrence) used on the FP64 tensor cores (state_sweep_2p.cu);
* the constants of the branch-free localisation weight (common.cuh) are the series of asin(sqrt a)/sqrt a.
"""
import os
import re
from fractions import Fraction
from math import factorial

import numpy as np

from conftest import ROOT
from efa_xray_b200.synth import make_case
from oracle import ensrf_oracle as O


def _obs_block(case):
    st, obs = O.State.from_case(case), O.obs_from_case(case)
    means, perts = O.compute_ob_priors(st, obs)
    return np.asarray(means), np.asarray(perts)


def _weight(case, k, j):
    d = O.haversine((case.ob_lat[k], case.ob_lon[k]), (case.ob_lat[j], case.ob_lon[j]))
    return float(O.gaspari_cohn(np.array([d]), case.ob_halfwidth[k])[0])


def test_dependency_driven_obs_solve_equals_serial_loop_in_any_compatible_order():
    case = make_case(ny=37, nx=72, nmem=24, nvars=1, ntimes=1, nobs=220, cutoff_km=1800.0, seed=71, frac_skip=0.07,
                     mixed_radius=True, mixed_error=True)
    ym, yp = _obs_block(case)
    ref = O.obs_space_solve(ym, yp, case.ob_value, case.ob_error, case.ob_halfwidth, case.ob_lat, case.ob_lon,
                            case.ob_assimilate, loc='GC')
    nobs, nens = yp.shape
    W = np.array([[_weight(case, k, j) if (k < j and case.ob_assimilate[k]) else 0.0 for j in range(nobs)] for k in range(nobs)])
    preds = [np.flatnonzero(W[:, j]) for j in range(nobs)]
    # a processing order that is NOT the index order: repeatedly take, in random order, rows whose predecessors are done
    rng = np.random.default_rng(5)
    done = np.zeros(nobs, bool)
    order = []
    while len(order) < nobs:
        ready = [j for j in rng.permutation(nobs) if not done[j] and done[preds[j]].all()]
        assert ready
        take = ready[:max(1, len(ready) // 3)]          # a few "workers" at a time
        order.extend(take)
        done[take] = True
    assert order != sorted(order)
    pub_ye = np.zeros((nobs, nens)); pub = {}
    out = dict(prior_mean=np.zeros(nobs), prior_var=np.zeros(nobs), post_mean=np.full(nobs, np.nan), post_var=np.full(nobs, np.nan))
    for j in order:
        x, m = yp[j].copy(), float(ym[j])
        for k in preds[j]:                               # ascending = the serial order of the reference
            innov, c1, beta = pub[k]
            kmat = W[k, j] * (x @ pub_ye[k]) * c1
            m += kmat * innov
            x -= beta * kmat * pub_ye[k]
        varye = np.var(x)
        out['prior_mean'][j], out['prior_var'][j] = m, varye
        if case.ob_assimilate[j]:
            kdenom = varye + case.ob_error[j]
            innov, c1 = case.ob_value[j] - m, 1.0 / ((nens - 1) * kdenom)
            beta = 1.0 / (1.0 + np.sqrt(case.ob_error[j] / kdenom))
            pub[j], pub_ye[j] = (innov, c1, beta), x
            kself = _weight(case, j, j) * (x @ x) * c1
            out['post_mean'][j] = m + kself * innov
            out['post_var'][j] = np.var(x - beta * kself * x)
    for key in out:
        np.testing.assert_allclose(out[key], ref[key], rtol=1e-10, atol=1e-12, equal_nan=True)
    a = case.ob_assimilate
    np.testing.assert_allclose(pub_ye[a], ref['ye'][a], rtol=1e-10, atol=1e-12)
    # the dependency graph is sparse here, so its longest path is far shorter than the ob count
    depth = np.zeros(nobs, int)
    for j in range(nobs):
        depth[j] = 1 + (depth[preds[j]].max() if len(preds[j]) else 0)
    assert depth.max() < nobs // 2


def test_blocked_gram_recurrence_equals_sequential_rank1_updates():
    """8 obs at a time:  g = Y x0,  e_q = omega_q (g_q - sum_{p<q} G_qp e_p),  x = x0 - sum_q e_q y_q  with G = Y Y^T
    is the same as applying  x -= omega_q (y_q . x) y_q  for q = 0..7 in order (ensrf.py:95-141 with the localisation
    weight, 1/((N-1) kdenom) and beta folded into omega); the mean rides along as a pseudo-member."""
    rng = np.random.default_rng(9)
    nens = 100
    Y = rng.standard_normal((8, nens))
    x0 = rng.standard_normal(nens)
    mean0 = 287.3
    omega = rng.uniform(0.0, 0.02, 8)
    omega[[2, 5]] = 0.0                                  # obs that do not reach this row
    innov_over_beta = rng.standard_normal(8)
    # sequential
    x, mean = x0.copy(), mean0
    for q in range(8):
        e = omega[q] * (Y[q] @ x)
        x -= e * Y[q]
        mean += e * innov_over_beta[q]                   # kmat*innov = (beta*kmat) * innov/beta
    # blocked, with the pseudo-member column -innov/beta masked out of the dot products
    Yext = np.hstack([Y, -innov_over_beta[:, None]])
    xext = np.append(x0, mean0)
    g = Y @ x0
    G = Y @ Y.T
    e = np.zeros(8)
    for q in range(8):
        e[q] = omega[q] * (g[q] - G[q, :q] @ e[:q])
    xb = xext - e @ Yext
    np.testing.assert_allclose(xb[:-1], x, rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(xb[-1], mean, rtol=1e-14)


def test_fast_localisation_weight_constants_and_accuracy():
    src = open(os.path.join(ROOT, 'efa_xray_b200', 'csrc', 'common.cuh')).read()
    body = src[src.index('exb_asin_sqrt_over_sqrt'):src.index('EXB_SHORT_AMAX')]
    consts = {int(n): float(v) for v, n in re.findall(r'([0-9.]+(?:e-?[0-9]+)?)\s*[;,)][^\n]*?//\s*c(\d+)', body)}
    found = dict(re.findall(r'//\s*(c\d+), (c\d+)', body))
    coef = [float(x) for x in re.findall(r'fma\(p[eo], a2, ([0-9.e-]+)\)', body)] + \
           [float(x) for x in re.findall(r'double pe = ([0-9.e-]+), po = ([0-9.e-]+);', body)[0]]
    exact = [float(Fraction(factorial(2 * n), 4 ** n * factorial(n) ** 2 * (2 * n + 1))) for n in range(20)]
    assert sorted(coef) == sorted(exact)                 # every series coefficient c0..c19, bit for bit
    # the same evaluation order in numpy against arcsin, over the range the kernel uses it on (a <= 0.15)
    a = np.concatenate([np.logspace(-14, -2, 60), np.linspace(0.01, 0.15, 200)])
    a2 = a * a
    pe, po = exact[18], exact[19]
    for k in range(8, -1, -1):
        pe, po = pe * a2 + exact[2 * k], po * a2 + exact[2 * k + 1]
    q = po * a + pe
    np.testing.assert_allclose(np.sqrt(a) * q, np.arcsin(np.sqrt(a)), rtol=4e-16)
    # the same coefficients again in the parameter-block table of the lean weight function (exb_loc_const)
    tab = src[src.index('const double c[20] = {'):]
    tab = [float(x) for x in re.findall(r'[0-9.]+(?:e-?[0-9]+)?', tab[tab.index('{') + 1:tab.index('}')])]
    assert tab == exact
    # the 10-term series of exb_asin_sqrt_over_sqrt_short: same coefficients c0..c9, valid up to EXB_SHORT_AMAX = 0.03
    sbody = src[src.index('double exb_asin_sqrt_over_sqrt_short'):src.index('template <bool SHORT>')]
    scoef = [float(x) for x in re.findall(r'fma\(p[eo], a2, ([0-9.e-]+)\)', sbody)] + \
            [float(x) for x in re.findall(r'double pe = ([0-9.e-]+), po = ([0-9.e-]+);', sbody)[0]]
    assert sorted(scoef) == sorted(exact[:10])
    assert float(re.search(r'#define EXB_SHORT_AMAX ([0-9.]+)', src).group(1)) == 0.03
    s_a = np.concatenate([np.logspace(-14, -3, 40), np.linspace(0.001, 0.03, 200)])
    s_a2 = s_a * s_a
    pe, po = exact[8], exact[9]
    for k in range(3, -1, -1):
        pe, po = pe * s_a2 + exact[2 * k], po * s_a2 + exact[2 * k + 1]
    np.testing.assert_allclose(np.sqrt(s_a) * (po * s_a + pe), np.arcsin(np.sqrt(s_a)), rtol=4e-16)
    # Gaspari-Cohn through that path against the oracle's (reference) formulation, 2000 km support
    hw = 1000.0
    r = 2.0 * 6371.0 * np.sqrt(a) * q / hw
    p1 = (((-0.25 * r + 0.5) * r + 0.625) * r - 5.0 / 3.0) * r * r + 1.0
    p2 = ((((r / 12.0 - 0.5) * r + 0.625) * r + 5.0 / 3.0) * r - 5.0) * r + 4.0 - (2.0 / 3.0) / np.clip(r, 1.0, 2.0)
    w = np.where(r <= 1.0, p1, np.where(r < 2.0, p2, 0.0))
    d = 6371.0 * 2.0 * np.arcsin(np.sqrt(a))
    np.testing.assert_allclose(w, O.gaspari_cohn(d, hw), rtol=0, atol=2e-15)
