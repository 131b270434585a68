import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
GOLDEN_CASES = ['gc_small', 'gc_multivar_offtime', 'noloc_small', 'gc_4deg', 'gc_inflate', 'gc_dense300',
                'gc_inflate_vardict', 'gc_inflate_dims', 'gc_1d_points']


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA (B200) device; run with -m gpu on the GPU box')


def decode_inflation(infl):
    """JSON-able inflation spec of a golden case -> what EnSRF takes (same decoding as tests/golden/make_golden.py)."""
    import numpy as np
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


def load_golden(name):
    """(arrays, parameters) of a golden case.  The file holds the reference's posterior as post - prior (it compresses
    better), with the prior regenerated from the case's seed; make_golden.py checked when writing it that adding the
    prior back rebuilds 'post' bit for bit."""
    import json
    import numpy as np
    g = dict(np.load(os.path.join(GOLDEN, name + '.npz')))
    p = json.loads(str(g['params']))
    p['inflation'] = decode_inflation(p['inflation'])
    g['post'] = golden_case(p).to_vect() + g.pop('post_minus_prior')
    return g, p


def golden_case(p):
    """The synthetic Case a golden file was generated from (its make_case / make_case_1d parameters)."""
    from efa_xray_b200.synth import make_case, make_case_1d
    kw = dict(p['kw'])
    if kw.pop('one_d', False):
        return make_case_1d(**kw)
    return make_case(**kw)


@pytest.fixture(scope='session')
def lib():
    from efa_xray_b200 import _lib
    return _lib.load()
