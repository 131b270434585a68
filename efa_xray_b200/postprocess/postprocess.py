"""Post-analysis observation statistics (reference: efa_xray/postprocess/postprocess.py:8-39).

The reference loops over the observations and calls ob.estimate() twice per ob (a full-grid argsort each time).
Here the two sets of ob estimates are two batched H.x gathers on the device (exb_stencil_search_* once, exb_gather_*
twice, exb_split_mean_pert_* for the means) followed by a row variance; the result is the same pandas DataFrame,
one row per observation, same columns.
"""
import numpy as np

from .. import engine, _lib
from ..assimilation.assimilation import Assimilation
from ..state.ensemble import EnsembleState

COLUMNS = ['validtime', 'flead', 'lat', 'lon', 'obtype', 'description', 'ob error', 'value', 'assimilated',
           'prior mean', 'post mean', 'prior variance', 'post variance']


def ob_estimates(state, obs, forward_operator='reference'):
    """[Nobs, Nens] ensemble estimates of every ob (Observation.estimate, observation.py:40-50, for all obs at once)
    computed on the device, with the forward operator of Assimilation (DESIGN.md section 4.8)."""
    a = Assimilation(state, obs, verbose=False, forward_operator=forward_operator)
    means, perts = a.compute_ob_priors()
    return perts + means[:, None]


def obs_assimilation_statistics(prior, post, obs, forward_operator='reference'):
    """Builds a pandas dataframe with statistical info about the observations (postprocess.py:8-39):
    prior/post mean and variance (numpy .var(), ddof 0) of the ensemble estimate of every ob, plus its metadata.
    Pass the analysis's forward_operator so that the estimates use its H."""
    import pandas as pd
    assert isinstance(prior, EnsembleState)
    assert isinstance(post, EnsembleState)
    prior_ye = ob_estimates(prior, obs, forward_operator)
    post_ye = ob_estimates(post, obs, forward_operator)
    t0 = pd.to_datetime(prior['validtime'].values[0])
    oblist = []
    for k, ob in enumerate(obs):
        oblist.append({
            'validtime': ob.time,
            'flead': (pd.to_datetime(ob.time) - t0).total_seconds() / 3600,
            'lat': ob.lat, 'lon': ob.lon, 'obtype': ob.obtype, 'description': ob.description,
            'ob error': ob.error, 'value': ob.value, 'assimilated': ob.assimilated,
            'prior mean': prior_ye[k].mean(), 'post mean': post_ye[k].mean(),
            'prior variance': prior_ye[k].var(), 'post variance': post_ye[k].var(),
        })
    return pd.DataFrame(oblist, columns=COLUMNS)
