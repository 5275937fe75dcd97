"""CPU tests of PSIS leave-one-out: the numpy reference oracle/psis.py against exact leave-one-out of a conjugate
model and against generalised Pareto samples of known shape; its edge cases; the scalar pieces of
csrc/spmf_loo.cuh (run on the host through tests/loo_math.cpp) against the reference; loo_compare; and the
argument checks of spmf_psis_loo."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
import scipy.stats as st
import torch

from oracle import psis

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "loo_math.cpp")


@pytest.fixture(scope="module")
def hc():
    """g++ build of tests/loo_math.cpp into a temporary directory (nothing is written into the tree)."""
    so = os.path.join(tempfile.mkdtemp(prefix="spmf_loo_math_"), "libloo_math.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", so, "-lm"])
    lib = C.CDLL(so)
    d, i = C.c_double, C.c_int
    for name, res, args in (("hc_tail_len", i, [i]), ("hc_grid_size", i, [i]), ("hc_quartile_index", i, [i]),
                            ("hc_grid_b", d, [i, i, d, d]), ("hc_profile", d, [i, d, d]),
                            ("hc_gpd_quantile", d, [d, d, d]), ("hc_log_dbl_min", d, []), ("hc_max_tail", i, []),
                            ("hc_max_grid", i, [])):
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


@pytest.fixture(scope="module")
def conjugate():
    """y_i ~ N(theta, 1), theta ~ N(0, 1): 4,000 exact posterior draws and the closed-form leave-one-out
    predictive density of every point."""
    rng = np.random.default_rng(0)
    N = 20
    y = rng.normal(0.5, 1.0, N)
    prec = 1.0 + N
    theta = rng.normal(y.sum() / prec, 1.0 / np.sqrt(prec), 4000)
    exact = np.array([st.norm.logpdf(y[i], (y.sum() - y[i]) / N, np.sqrt(1.0 + 1.0 / N)) for i in range(N)])
    ll = st.norm.logpdf(y[:, None], theta[None, :], 1.0)        # (N, S)
    return ll, exact


def test_psis_matches_exact_loo_of_a_conjugate_model(conjugate):
    ll, exact = conjugate
    elpd, lppd, khat = psis.psis_loo(ll)
    assert np.abs(elpd - exact).max() < 0.02
    assert khat.max() < 0.5
    assert np.all(lppd >= elpd)               # leaving a point out never predicts it better


@pytest.mark.parametrize("k", [0.1, 0.5, 0.9])
def test_gpd_fit_recovers_the_shape(k):
    y = np.sort(st.genpareto.rvs(k, size=5000, random_state=1))
    khat, sigma = psis.gpdfit(y)
    assert abs(khat - k) < 0.08
    assert sigma > 0


@pytest.mark.parametrize("S", [1, 2, 7, 1000])
def test_constant_row(S):
    elpd, lppd, khat = psis.psis_loo_row(np.full(S, -3.25))
    assert elpd == pytest.approx(-3.25, abs=1e-14) and lppd == pytest.approx(-3.25, abs=1e-14)
    assert lppd - elpd == pytest.approx(0.0, abs=1e-14)
    assert khat == np.inf


def test_nonfinite_rows():
    rng = np.random.default_rng(3)
    ll = rng.normal(-2.0, 1.0, 100)
    a = ll.copy()
    a[17] = -np.inf
    elpd, lppd, khat = psis.psis_loo_row(a)
    assert elpd == -np.inf and khat == np.inf
    assert lppd == pytest.approx(np.log(np.exp(ll).sum() - np.exp(ll[17])) - np.log(100), rel=1e-12)
    assert psis.psis_loo_row(np.full(5, -np.inf))[:2] == (-np.inf, -np.inf)
    for bad in (np.nan, np.inf):
        b = ll.copy()
        b[3], b[4] = -np.inf, bad
        assert all(np.isnan(v) for v in psis.psis_loo_row(b))


def test_short_rows_are_not_smoothed():
    # S <= 20 keeps at most 4 values in the tail: k-hat = inf, raw importance weights
    rng = np.random.default_rng(4)
    for S in (2, 5, 13, 20):
        ll = rng.normal(0, 2, S)
        elpd, lppd, khat = psis.psis_loo_row(ll)
        assert khat == np.inf
        r = -ll - (-ll).max()
        lw = r - np.log(np.exp(r).sum())
        assert elpd == pytest.approx(np.log(np.exp(lw + ll).sum()), rel=1e-12)      # = -log mean exp(-ll)
        assert elpd == pytest.approx(-np.log(np.mean(np.exp(-ll))), rel=1e-12)


def test_header_pieces_agree_with_the_reference(hc):
    assert hc.hc_log_dbl_min() == psis.LOG_DBL_MIN
    tails = [hc.hc_tail_len(S) for S in range(1, 8193)]
    assert tails == [psis.tail_length(S) for S in range(1, 8193)]
    assert max(tails) == hc.hc_max_tail() == tails[-1]
    assert hc.hc_grid_size(hc.hc_max_tail()) == hc.hc_max_grid()
    for n in range(5, hc.hc_max_tail() + 1):
        assert hc.hc_grid_size(n) == psis.grid_size(n)
        assert hc.hc_quartile_index(n) == psis.quartile_index(n)
    rng = np.random.default_rng(5)
    for n in (5, 17, 100, 272):
        y = np.sort(np.exp(rng.normal(0, 2, n)))
        m = psis.grid_size(n)
        q = psis.quartile_index(n)
        for j in range(1, m + 1):
            b = psis.grid_b(j, m, y[-1], y[q])
            assert hc.hc_grid_b(j, m, y[-1], y[q]) == pytest.approx(b, rel=1e-12, abs=0)
            k = float(np.log1p(-b * y).mean())
            assert hc.hc_profile(n, b, k) == pytest.approx(float(psis.profile(n, b, k)), rel=1e-12, abs=0)
    for k in (-0.5, -1e-17, 0.0, 1e-17, 1e-6, 0.3, 0.7, 1.5):
        for p in (1e-4, 0.01, 0.5, 0.99, 1 - 1e-4):
            assert hc.hc_gpd_quantile(p, k, 2.5) == pytest.approx(float(psis.gpd_quantile(p, k, 2.5)), rel=1e-12)


def test_loo_compare():
    from spmf_b200.poisson import loo_compare
    a = {'pointwise': {'elpd_loo': torch.tensor([-1.0, -2.0, -3.5, -0.5], dtype=torch.float64)}}
    b = {'pointwise': {'elpd_loo': torch.tensor([-1.5, -2.0, -3.0, -1.5], dtype=torch.float64)}}
    d = np.array([0.5, 0.0, -0.5, 1.0])
    got = loo_compare(a, b)
    assert got['elpd_diff'] == pytest.approx(1.0, rel=1e-15)
    assert got['se_diff'] == pytest.approx(math.sqrt(4 * d.var(ddof=1)), rel=1e-14)
    assert loo_compare(a, a) == {'elpd_diff': 0.0, 'se_diff': 0.0}
    with pytest.raises(ValueError):
        loo_compare(a, {'pointwise': {'elpd_loo': torch.zeros(3, dtype=torch.float64)}})


def test_psis_loo_rejects_bad_arguments():
    from spmf_b200 import _abi
    assert _abi.LOO_MAX_S == 8192
    fake = 0x1000                                       # never dereferenced: the checks come first
    for args in ((None, 4, 2, 4, fake, fake, fake), (fake, 4, 2, 4, None, fake, fake),
                 (fake, 3, 2, 4, fake, fake, fake),       # ld < S
                 (fake, 4, 0, 4, fake, fake, fake), (fake, 0, 2, 0, fake, fake, fake),
                 (fake, 9000, 2, 8193, fake, fake, fake)):
        with pytest.raises(_abi.SpmfError):
            _abi.call("spmf_psis_loo", *args, None)
