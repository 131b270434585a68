"""EnSRF -- serial ensemble square-root filter update (efa_xray/assimilation/ensrf.py:8-151)."""
from __future__ import print_function

from copy import deepcopy

import numpy as np

from .assimilation import Assimilation
from .. import engine


class EnSRF(Assimilation):
    """EnSRF(state, obs, nproc=1, inflation=None, verbose=True, loc=False, relaxation=None,
    outlier_threshold=None, forward_operator='reference').update() -> (post_state, obs).

    Same contract as the reference (ensrf.py:28-33, assimilation.py:171): `obs` is the caller's list,
    mutated in place with prior_mean / prior_var / post_mean / post_var / assimilated (ensrf.py:66-70,
    :144-149); `post_state` is a new EnsembleState; the prior is only modified by inflation.
    Observations are assimilated strictly in list order.  `dtype` ('f64' or 'f32') selects the device
    arithmetic; results are returned in the state's own dtype.

    `relaxation` (not in the reference) relaxes the analysis back toward the prior after the serial loop, to
    counter the loss of spread of repeated analyses:
      None                 no relaxation (default)
      ('rtps', alpha)      relaxation to prior spread (Whitaker & Hamill 2012):
                           x = m_a + x'_a * (1 + alpha * (sigma_b - sigma_a) / sigma_a)
      ('rtpp', alpha)      relaxation to prior perturbations (Zhang et al. 2004):
                           x = m_a + (1 - alpha) * x'_a + alpha * x'_b
    alpha is a float in [0, 1] or a dict {variable name: float}; variables the dict does not name get 0.  The prior
    (m_b, x'_b, sigma_b) is the state as the serial loop receives it, i.e. after prior inflation.  The analysis mean
    is unchanged, and rows without spread or that the analysis did not change are left as they are.  The per-ob
    diagnostics (prior_mean, prior_var, post_mean, post_var) are those of the serial loop: they are not re-evaluated
    after relaxation.  Invalid values raise ValueError here, before any device work.

    `outlier_threshold` (not in the reference) keeps gross observation errors out of the analysis, as DART's
    outlier threshold does, but checked inside the serial loop:
      None                 no check (default)
      t                    a positive finite float: the threshold of every ob
      {variable: t}        a threshold per variable; obs of variables the dict does not name are not checked
    An ob k with assimilate_this is rejected when |value - prior_mean| > t * sqrt(prior_var + error), with the prior
    of ob k as the serial loop sees it, i.e. after obs 0..k-1 have been assimilated.  A rejected ob is treated as if
    assimilate_this were False: prior_mean and prior_var are set, post_mean and post_var are not, assimilated is
    False, and neither the state nor any later ob's prior feels it.  assimilate_this itself is left alone.  Invalid
    values raise ValueError here, before any device work.  (A check against the priors before the loop needs no
    library support: compute_ob_priors and assimilate_this.)

    `forward_operator` (not in the reference) selects the forward operator H (DESIGN.md section 4.8):
      'reference'          the reference's operator: inverse-distance weights on 4 points under its pseudo-metric,
                           with its time weights (default; EXACT_MATCH_POLICY applies)
      'bilinear'           bilinear in space on the grid cell that contains the ob, linear in time with correctly
                           oriented weights; needs 2-D lat/lon.  An ob outside the grid raises ValueError in
                           update(), before any ob attribute is written and before the posterior is built.
    An unknown name, or 'bilinear' on a state with 1-D lat/lon, raises ValueError here, before any device work.
    """

    def __init__(self, state, obs, nproc=1, inflation=None, verbose=True, loc=False, dtype='f64', relaxation=None,
                 outlier_threshold=None, forward_operator='reference'):
        Assimilation.__init__(self, state, obs, nproc, inflation, verbose, forward_operator=forward_operator)
        self.loc = loc
        self.dtype = dtype
        self._validate_relaxation(relaxation)
        self.relaxation = relaxation
        self._validate_outlier_threshold(outlier_threshold)
        self.outlier_threshold = outlier_threshold
        self.last_result = None

    def update(self):
        import torch
        if self.verbose: print("Beginning update sequence")
        loc_mode = self._loc_mode(self.loc)
        dev = self._device()

        if self.inflation is not None and not self.is_inflated:
            # the reference inflates the prior before anything else (assimilation.py:132-134): the caller's state in
            # place, except that per-dimension arrays rebind self.prior to a new state (inflate_state)
            if self.verbose: print("Inflating Prior State")
            self.inflate_state()
        st = self.prior
        nlev = st.nvars() * st.ntimes()

        if self.verbose: print("Computing observation priors")
        obs = self._obs_arrays(loc_mode, self.outlier_threshold)
        tdtype = {'f64': torch.float64, 'f32': torch.float32}[self.dtype]
        if self.verbose: print("Beginning observation loop")
        # The prior is read where it lies (the state's contiguous, page-locked block: no to_vect copy, and the prior
        # itself stays untouched, assimilation.py:165) and the analysis is written into a fresh block that the
        # posterior state adopts (no deepcopy of the data, no from_vect copy).  Upload, sweep and download overlap
        # band by band inside engine.analysis_host.
        st._consolidate()
        prior_blk = st._block_view()
        if prior_blk is not None:
            from ..state.ensemble import BLOCK_POOL
            host = prior_blk.reshape(st.nstate(), st.nmems())
            out_blk, owner = BLOCK_POOL.alloc(prior_blk.shape, prior_blk.dtype)
            out = out_blk.reshape(host.shape)
        else:                                    # variables on different dims / dtypes: stacked copy
            host = np.array(st.to_vect(), order='C', copy=True)
            out_blk, owner, out = None, None, host
        res = engine.analysis_host(host, nlev, None, None, obs, loc_mode, device=dev, dtype=tdtype,
                                   grid=st._grid_tables(), out=out, relaxation=self._relaxation_levels(self.relaxation),
                                   forward_operator=self.forward_operator)
        self._check_exact(res.n_exact)
        self._check_outside(res.n_outside)
        self.last_result = res

        # per-ob diagnostics back onto the caller's objects (ensrf.py:66-76, :144-149)
        pm, pv = res.prior_mean.tolist(), res.prior_var.tolist()
        qm, qv = res.post_mean.tolist(), res.post_var.tolist()
        done = res.assimilated.tolist()
        for ob, a, b, c, d, f in zip(self.obs, pm, pv, qm, qv, done):
            ob.prior_mean = a
            ob.prior_var = b
            if f:
                ob.post_mean = c
                ob.post_var = d
                ob.assimilated = True
            else:
                ob.assimilated = False

        if self.verbose: print("Formatting posterior")
        if out_blk is not None:
            post_state = st._new_with_block(out_blk, owner)
        else:
            post_state = deepcopy(self.prior)
            post_state.from_vect(host)
        return post_state, self.obs
