"""CPU tests of the element-wise reference the ragged GPU tests rely on (oracle/analytic.py, magnitudes=True):
on the ragged batches of tests/ragged.py the analytic restatement agrees with autograd, its magnitudes bound
the values they stand for, and the data-term magnitudes behave as sums over rows do."""
import numpy as np
import pytest
import torch

from oracle.analytic import analytic_loss_and_grads
from oracle.spmf_oracle import draw_noise
from tests.ragged import POISSON_CASES, make_case, worst_ratio
from tests.util import make_oracle, perturbed_params, rel_err

K, S = 8, 2


def _setup(name, scale_rows=True):
    case = make_case(name)
    N, D = case.x.shape
    oracle = make_oracle(D, K, N, case.x, scale_rows=scale_rows)
    params = perturbed_params(oracle, 0.3, seed=7)
    noise = draw_noise(oracle, params, S, seed=8)
    return case, oracle, params, noise


@pytest.mark.parametrize("name", POISSON_CASES + ["rows_650"])
def test_analytic_matches_autograd_and_magnitudes_bound_values(name):
    case, oracle, params, noise = _setup(name)
    xb = case.batch
    xt = torch.tensor(xb, dtype=torch.float64)
    l1, g1, p1 = oracle.loss_and_grads(params, noise, {'counts': xt})
    l2, g2, p2, mags, rows = analytic_loss_and_grads(oracle, params, noise, xb, magnitudes=True)
    assert abs(l1 - l2) < 1e-10 * abs(l1)
    for k in g1:
        # the InverseGamma family sums cancelling terms over all of D and K: float64 rounding reaches ~1e-9 there
        assert rel_err(g2[k], g1[k].numpy()) < (1e-9 if k.split('/')[0] in 'vwus' else 1e-8), k
    for k in p1:
        assert rel_err(p2[k], p1[k].numpy()) < 1e-10, k
    assert {k for k in mags if not k.startswith('data/')} == {f'{v}/{p}' for v in 'vwus' for p in ('loc', 'scale_raw')}
    for k, M in mags.items():
        if k in g2:
            assert M.shape == g2[k].shape
            assert (M >= np.abs(g2[k])).all(), k
            assert worst_ratio(g2[k], g1[k].numpy(), M) < 1e-9, k          # the two oracles, element-wise
    theta, _ = oracle.sample(params, noise)
    z, Mz = rows['z']
    np.testing.assert_allclose(z, oracle.encode(xt, theta['u'], theta['s']).detach().numpy(), rtol=1e-12, atol=1e-300)
    assert (Mz >= np.abs(z)).all()
    ll, Mll = rows['row_ll']
    ref_ll = oracle.log_likelihood_components(data={'counts': xt}, **{k: theta[k] for k in 'suvw'})
    ref_ll = ref_ll['log_likelihood'].sum(-1).detach().numpy()
    assert ll.shape == (S, case.B) and worst_ratio(ll, ref_ll, Mll) < 1e-12
    assert (Mll >= np.abs(ll)).all()
    empty = xb.sum(1) == 0                          # row scaling: r = 0, so z = 0 on empty rows
    assert (z[:, empty] == 0).all()


@pytest.mark.parametrize("name", ["empty_rows", "large_counts"])
@pytest.mark.parametrize("scale_rows", [True, False])
def test_data_term_magnitudes_are_row_sums(name, scale_rows):
    """M of the data term is a sum over rows: a row permutation leaves it unchanged and duplicating the batch
    doubles it."""
    case, oracle, params, noise = _setup(name, scale_rows)
    xb = case.batch
    run = lambda x: analytic_loss_and_grads(oracle, params, noise, x, c_gamma=True, magnitudes=True)
    _, _, _, m0, r0 = run(xb)
    perm = np.random.default_rng(0).permutation(case.B)
    _, _, _, m1, r1 = run(xb[perm])
    _, _, _, m2, _ = run(np.concatenate([xb, xb]))
    for k in m0:
        np.testing.assert_allclose(m1[k], m0[k], rtol=1e-12, err_msg=k)
    for k in ('data/GAp', 'data/GEV', 'data/Gphi'):
        np.testing.assert_allclose(m2[k], 2 * m0[k], rtol=1e-12, err_msg=k)
    np.testing.assert_allclose(r1['row_ll'][1], r0['row_ll'][1][:, perm], rtol=1e-12)
