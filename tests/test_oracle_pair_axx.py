"""The Axx statistic at two distinct inputs (the pair blocks of the joint predictive covariance of f): the closed form
tests.pair_oracle.psi_axx_pairs against the reference's own integrand integrated at distinct t1, t2
(tests.pair_oracle.psi_axx_pairs_generic), for the causal, acausal and causal_id models, at pairs inside and outside the
window of the inducing inputs; on the diagonal t1 = t2 both reproduce psi_Axx."""
import numpy as np
import pytest

torch = pytest.importorskip('torch')
from oracle import model as om
from tests import pair_oracle as po

HYP = (5., 30., 40.)
TX = np.linspace(0., 1., 6)
# inside the window, past both ends, and far enough apart that most of the envelope underflows
T1 = np.array([-.35, .05, .3, .62, 1.2])
T2 = np.array([-.1, .3, .55, .97, 1.45, 2.1])

MODELS = [dict(causal=True, causal_id=False), dict(causal=False, causal_id=False), dict(causal=True, causal_id=True)]
IDS = ['causal', 'acausal', 'causal_id']


@pytest.mark.parametrize('model', MODELS, ids=IDS)
def test_closed_form_matches_the_reference_integrand(model):
    g = po.psi_axx_pairs_generic(T1, T2, TX, *HYP, **model).numpy()
    c = po.psi_axx_pairs(T1, T2, TX, *HYP, **model).numpy()
    assert g.shape == c.shape == (T1.size, T2.size, TX.size, TX.size)
    assert np.all(np.isfinite(g)) and np.abs(g).max() > 0
    assert np.abs(g - c).max() <= 1e-13 * np.abs(g).max(), np.abs(g - c).max() / np.abs(g).max()
    # the two inputs are not interchangeable: Axx(t1, t2)[k, l] = Axx(t2, t1)[l, k], not Axx(t2, t1)[k, l]
    back = po.psi_axx_pairs(T2, T1, TX, *HYP, **model).numpy()
    np.testing.assert_allclose(c, back.transpose(1, 0, 3, 2), rtol=1e-13, atol=1e-300)
    off = np.abs(c - back.transpose(1, 0, 2, 3)).max()
    assert off > 1e-6 * np.abs(c).max()


@pytest.mark.parametrize('model', MODELS, ids=IDS)
def test_equal_inputs_reproduce_psi_axx(model):
    t = np.array([-.2, .1, .45, .8, 1.3])
    ref = om.psi_Axx(t, TX, *[om.T(v) for v in HYP], **model).numpy()
    c = po.psi_axx_pairs(t, t, TX, *HYP, **model).numpy()
    g = po.psi_axx_pairs_generic(t, t, TX, *HYP, **model).numpy()
    diag_c = c[np.arange(t.size), np.arange(t.size)]
    diag_g = g[np.arange(t.size), np.arange(t.size)]
    assert np.array_equal(diag_c, ref)
    assert np.abs(diag_g - ref).max() <= 1e-13 * np.abs(ref).max()
