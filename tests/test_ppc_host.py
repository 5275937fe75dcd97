"""CPU tests of the posterior predictive check: the replicate samplers of csrc/spmf_math.cuh (poisson_draw /
bernoulli_draw, run on the host through tests/ppc_samplers.cpp) against scipy's distributions, and the p-value
assembly of spmf_b200.poisson.ppc_p_values on hand-built statistics with ties."""
import ctypes as C
import os
import subprocess
import tempfile
import types

import numpy as np
import pytest
import scipy.stats as st
import torch

N = 200_000
KEY = (0x1234567, 0x89ABCDE)
_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ppc_samplers.cpp")


def _load_samplers():
    """g++ build of tests/ppc_samplers.cpp into a temporary directory (nothing is written into the tree)."""
    so = os.path.join(tempfile.mkdtemp(prefix="spmf_ppc_samplers_"), "libppc_samplers.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", so, "-lm"])
    lib = C.CDLL(so)
    f = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
    i = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
    for fn in (lib.hc_poisson, lib.hc_bernoulli):
        fn.argtypes = [f, i, C.c_longlong, C.c_uint, C.c_uint, C.c_uint]

    def draw(fn, x, key=(0, 0), stream=0):
        """fn of every parameter in `x`: draw i uses key `key` and counter (i, 0, stream, 0)."""
        x = np.ascontiguousarray(x, np.float32).ravel()
        out = np.empty(x.size, np.int32)
        fn(x, out, x.size, int(key[0]), int(key[1]), int(stream))
        return out

    return types.SimpleNamespace(poisson=lambda x, key=(0, 0), stream=0: draw(lib.hc_poisson, x, key, stream),
                                 bernoulli=lambda x, key=(0, 0), stream=0: draw(lib.hc_bernoulli, x, key, stream))


hc = _load_samplers()


def _merged_chi2(draws, dist):
    """Chi-square goodness of fit with the bins merged (left to right) until each expects >= 5 draws."""
    n = draws.size
    lo, hi = int(dist.ppf(1e-12)), int(dist.isf(1e-12)) + 1
    ks = np.arange(lo, hi + 1)
    exp = n * dist.pmf(ks)
    exp[0] = n * dist.cdf(lo)                       # tails folded into the end bins
    exp[-1] = n * dist.sf(hi - 1)
    obs = np.bincount(np.clip(draws, lo, hi) - lo, minlength=ks.size).astype(np.float64)
    o_bins, e_bins, o_acc, e_acc = [], [], 0.0, 0.0
    for o, e in zip(obs, exp):
        o_acc, e_acc = o_acc + o, e_acc + e
        if e_acc >= 5:
            o_bins.append(o_acc), e_bins.append(e_acc)
            o_acc = e_acc = 0.0
    if e_acc > 0:                                   # remainder joins the last bin
        o_bins[-1] += o_acc
        e_bins[-1] += e_acc
    o_bins, e_bins = np.array(o_bins), np.array(e_bins)
    if o_bins.size < 2:
        return 1.0
    return st.chisquare(o_bins, e_bins * o_bins.sum() / e_bins.sum()).pvalue


# 9.99 / 10.01: either side of the switch from inversion to PTRS (kPoissonInvMax = 10)
@pytest.mark.parametrize("lam", [1e-3, 0.3, 2.5, 9.99, 10.01, 37.0, 1e3, 1e5])
def test_poisson_draws_follow_the_poisson_law(lam):
    x = hc.poisson(np.full(N, lam, np.float32), key=KEY, stream=7)
    assert x.min() >= 0
    p = _merged_chi2(x, st.poisson(lam))
    assert p > 1e-6, p
    se_mean = np.sqrt(lam / N)
    se_var = np.sqrt((lam + 2 * lam * lam) / N)
    assert abs(x.mean() - lam) < 6 * se_mean
    assert abs(x.var(ddof=1) - lam) < 6 * se_var


@pytest.mark.parametrize("p", [1e-3, 0.1, 0.5, 0.9, 0.999])
def test_bernoulli_draws_follow_the_bernoulli_law(p):
    x = hc.bernoulli(np.full(N, p, np.float32), key=KEY, stream=3)
    assert set(np.unique(x)) <= {0, 1}
    se = np.sqrt(p * (1 - p) / N)
    assert abs(x.mean() - p) < 6 * se
    ones = int(x.sum())
    assert st.chisquare([N - ones, ones], [N * (1 - p), N * p]).pvalue > 1e-6


def test_draws_are_pure_functions_of_key_and_counter():
    lam = np.geomspace(1e-3, 1e5, 4096).astype(np.float32)
    a, b = hc.poisson(lam, key=KEY, stream=1), hc.poisson(lam, key=KEY, stream=1)
    assert np.array_equal(a, b)
    assert not np.array_equal(a, hc.poisson(lam, key=KEY, stream=2))
    assert not np.array_equal(a, hc.poisson(lam, key=(KEY[0] + 1, KEY[1]), stream=1))
    p = np.linspace(0.05, 0.95, 4096).astype(np.float32)
    assert np.array_equal(hc.bernoulli(p, key=KEY, stream=1), hc.bernoulli(p, key=KEY, stream=1))
    assert not np.array_equal(hc.bernoulli(p, key=KEY, stream=1), hc.bernoulli(p, key=KEY, stream=2))


def test_edge_rates():
    # rate 0 gives 0; invalid rates (negative, NaN, inf, above 2^24) give 0 as well (the kernel counts them)
    x = hc.poisson(np.array([0.0, -1.0, np.nan, np.inf, 2.0 ** 25], np.float32), key=KEY)
    assert np.array_equal(x, np.zeros(5, np.int32))
    assert np.array_equal(hc.bernoulli(np.array([0.0, 1.0] * 512, np.float32), key=KEY), np.tile([0, 1], 512))


def test_p_values_mid_p_with_ties():
    from spmf_b200.poisson import ppc_p_values
    S, N, D = 4, 3, 2
    obs = dict(row_total=torch.tensor([2., 5., 0.], dtype=torch.float64), row_nnz=torch.tensor([1, 2, 0]),
               col_total=torch.tensor([4., 3.], dtype=torch.float64), col_sumsq=torch.tensor([10., 5.], dtype=torch.float64),
               col_nnz=torch.tensor([2, 1]), total=torch.tensor(7., dtype=torch.float64), nnz=torch.tensor(3),
               max=torch.tensor(4., dtype=torch.float64), discrepancy=torch.tensor([1.0, 2.0, 3.0, 4.0], dtype=torch.float64))
    rep = dict(row_total=torch.tensor([[2, 5, 0], [3, 4, 0], [1, 5, 1], [2, 6, 0]]),
               row_nnz=torch.tensor([[1, 2, 0]] * 4),
               col_total=torch.tensor([[4, 3], [5, 2], [4, 4], [3, 3]]),
               col_sumsq=torch.tensor([[10, 5], [13, 4], [8, 10], [5, 5]]),
               col_nnz=torch.tensor([[2, 1], [2, 1], [2, 1], [2, 1]]),
               total=torch.tensor([7, 7, 8, 8]), nnz=torch.tensor([3, 2, 3, 4]), max=torch.tensor([4, 4, 3, 5]),
               discrepancy=torch.tensor([2.0, 2.0, 1.0, 4.0], dtype=torch.float64))
    p = ppc_p_values(obs, rep)
    # row 0: reps (2, 3, 1, 2) vs 2 -> 1 above, 2 ties -> (1 + 1) / 4
    assert p['row_total'].tolist() == [0.5, 0.5, 0.625]
    assert p['row_nnz'].tolist() == [0.5, 0.5, 0.5]                  # all ties
    assert p['col_total'].tolist() == [(1 + 0.5 * 2) / 4, (1 + 0.5 * 2) / 4]
    assert float(p['total']) == (2 + 0.5 * 2) / 4
    assert float(p['nnz']) == (1 + 0.5 * 2) / 4
    assert float(p['max']) == (1 + 0.5 * 2) / 4
    # paired per draw: (2 > 1), (2 == 2), (1 < 3), (4 == 4) -> (1 + 0.5 * 2) / 4
    assert float(p['discrepancy']) == 0.5
    # column variances from the integer sums, (sumsq - total^2 / N) / (N - 1)
    var = lambda t, q: (q - t * t / N) / (N - 1)
    ov = [var(4., 10.), var(3., 5.)]
    rv = [[var(4, 10), var(3, 5)], [var(5, 13), var(2, 4)], [var(4, 8), var(4, 10)], [var(3, 5), var(3, 5)]]
    want = [(sum(r[j] > ov[j] for r in rv) + 0.5 * sum(r[j] == ov[j] for r in rv)) / S for j in range(D)]
    assert p['col_var'].tolist() == want
    assert all(v.dtype == torch.float64 for v in p.values())


def test_check_entry_points_reject_null_pointers():
    from spmf_b200 import _abi
    with pytest.raises(_abi.SpmfError):
        _abi.call("spmf_ppc_rows", None, 4, 5, 3, 2, 0, *([None] * 3), 1, 0, *([None] * 12))
    with pytest.raises(_abi.SpmfError):
        _abi.call("spmf_ppc_observed", *([None] * 3), 4, 5, *([None] * 6))
