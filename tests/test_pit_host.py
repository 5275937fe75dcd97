"""CPU tests of LOO-PIT: the predictive CDFs and the Czado binning of csrc/spmf_pit.cuh (run on the host through
tests/pit_math.cpp) against scipy / mpmath and the numpy reference oracle/pit.py; the reference against the exact
leave-one-out predictive of a conjugate Gamma-Poisson model; miscalibration made visible; and the argument checks
of the new entry points."""
import ctypes as C
import os
import subprocess
import tempfile
import types

import numpy as np
import pytest
import scipy.special as sp
import scipy.stats as st

from oracle import pit

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pit_math.cpp")
MAX_ITER = 40000                 # kPitMaxIter (csrc/spmf_pit.cuh)


def _load():
    """g++ build of tests/pit_math.cpp into a temporary directory (nothing is written into the tree)."""
    so = os.path.join(tempfile.mkdtemp(prefix="spmf_pit_math_"), "libpit_math.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", so, "-lm"])
    lib = C.CDLL(so)
    d = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    i = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
    lib.hc_poisson_cdf.argtypes = [d, d, d, C.c_longlong]
    lib.hc_poisson_cdf_pair.argtypes = [d, d, d, d, i, C.c_longlong]
    lib.hc_bernoulli_cdf.argtypes = [d, d, d, C.c_longlong]
    lib.hc_czado_bins.argtypes = [d, d, C.c_longlong, C.c_int, d]
    lib.hc_count_ok.argtypes = [C.c_float, C.c_int]

    def arr(*xs):
        return [np.ascontiguousarray(np.broadcast_arrays(*xs)[k], np.float64).ravel() for k in range(len(xs))]

    def cdf(x, lam):
        x, lam = arr(x, lam)
        out = np.empty_like(x)
        lib.hc_poisson_cdf(x, lam, out, x.size)
        return out

    def pair(x, lam):
        x, lam = arr(x, lam)
        fm, fp, it = np.empty_like(x), np.empty_like(x), np.empty(x.size, np.int32)
        lib.hc_poisson_cdf_pair(x, lam, fm, fp, it, x.size)
        return fm, fp, it

    def bern(x, logit):
        x, logit = arr(x, logit)
        out = np.empty_like(x)
        lib.hc_bernoulli_cdf(x, logit, out, x.size)
        return out

    def bins(pm, pp, J):
        pm, pp = arr(pm, pp)
        out = np.empty((pm.size, J))
        lib.hc_czado_bins(pm, pp, pm.size, J, out)
        return out

    return types.SimpleNamespace(cdf=cdf, pair=pair, bern=bern, bins=bins, count_ok=lib.hc_count_ok)


hc = _load()
LAMBDAS = [0.0, 1e-8, 0.5, 9.99, 10.0, 1e2, 1e4, 1e6, 2.0 ** 24]


def _xs(lam):
    """x from 0 to 50, across lam +- 10 sqrt(lam), and at 2^24."""
    s = np.sqrt(lam)
    xs = set(range(51)) | {2 ** 24 - 1, 2 ** 24}
    xs |= {int(max(0.0, np.floor(lam + k * s))) for k in np.linspace(-10, 10, 161)}
    return np.array(sorted(xs), np.float64)


@pytest.mark.parametrize("lam", LAMBDAS)
def test_poisson_cdf_matches_scipy(lam):
    x = _xs(lam)
    fm, fp, it = hc.pair(x, lam)
    assert np.array_equal(fp, hc.cdf(x, lam))
    assert it.max() < MAX_ITER                   # the stated bound holds with room to spare
    for got, xx in ((fp, x), (fm, x - 1)):
        ref = st.poisson.cdf(xx, lam)
        err = np.abs(got - ref)
        bad = err > 1e-12
        if bad.any():
            # scipy's pdtr loses digits in a band around x = lam + 4.6 sqrt(lam) at lam = 1e6 (2e-11 there):
            # those points are settled by mpmath at 40 digits
            mp = pytest.importorskip("mpmath")
            mp.mp.dps = 40
            for k in np.flatnonzero(bad):
                exact = float(mp.gammainc(xx[k] + 1, lam, mp.inf, regularized=True)) if xx[k] >= 0 else 0.0
                assert abs(got[k] - exact) <= 1e-12, (xx[k], lam, got[k], exact, ref[k])
    assert hc.cdf(-1.0, lam)[0] == 0.0


def test_poisson_cdf_edges():
    assert np.array_equal(hc.cdf([0, 1, 5], 0.0), [1.0, 1.0, 1.0])
    fm, fp, _ = hc.pair(np.arange(0, 30.0), 3.0)
    np.testing.assert_allclose(fp - fm, st.poisson.pmf(np.arange(0, 30), 3.0), rtol=1e-12, atol=1e-15)
    assert np.all(fm <= fp) and fm[0] == 0.0


def test_bernoulli_cdf_matches_expit():
    logit = np.array([-800.0, -40.0, -3.0, -1e-9, 0.0, 1e-9, 2.5, 40.0, 800.0])
    np.testing.assert_allclose(hc.bern(0.0, logit), sp.expit(-logit), rtol=1e-15, atol=1e-300)
    assert np.array_equal(hc.bern(1.0, logit), np.ones_like(logit))
    assert np.array_equal(hc.bern(-1.0, logit), np.zeros_like(logit))


def test_count_support():
    ok = lambda x, b=0: bool(hc.count_ok(x, b))
    assert ok(0.0) and ok(7.0) and ok(2.0 ** 24)
    assert not ok(-1.0) and not ok(0.5) and not ok(float("nan")) and not ok(2.0 ** 25) and not ok(float("inf"))
    assert ok(0.0, 1) and ok(1.0, 1) and not ok(2.0, 1) and not ok(0.5, 1)


def test_czado_binning_hand_built():
    J = 4
    pm = np.array([0.0, 0.2, 0.5, 1.0, 0.0, 0.25, 0.0, 0.3, -0.1, 0.6])
    pp = np.array([0.3, 0.2, 0.9, 1.0, 0.0, 0.25, 1.0, 0.1, 1.2, 0.6])
    want = np.array([
        [5 / 6, 1 / 6, 0, 0],          # uniform on [0, 0.3]
        [1, 0, 0, 0],                  # P- = P+ = 0.2: unit mass in bin floor(0.8) = 0
        [0, 0, 0.625, 0.375],          # uniform on [0.5, 0.9]
        [0, 0, 0, 1],                  # P- = P+ = 1: bin min(J - 1, 4) = 3
        [1, 0, 0, 0],                  # P- = P+ = 0: bin 0
        [0, 1, 0, 0],                  # P- = P+ = 0.25: bin floor(1.0) = 1
        [0.25, 0.25, 0.25, 0.25],      # uniform on [0, 1]
        [1, 0, 0, 0],                  # P+ < P-: unit mass in bin floor(0.4) = 0
        [0.25, 0.25, 0.25, 0.25],      # clamped to [0, 1]
        [0, 0, 1, 0],                  # 0.6: bin floor(2.4) = 2
    ])
    np.testing.assert_allclose(hc.bins(pm, pp, J), want, rtol=0, atol=1e-15)
    np.testing.assert_allclose(pit.czado_bins(pm, pp, J), want, rtol=0, atol=1e-15)
    rng = np.random.default_rng(0)
    a, b = rng.uniform(-0.1, 1.1, 500), rng.uniform(-0.1, 1.1, 500)
    for J in (1, 7, 20, 1000):
        k = hc.bins(np.minimum(a, b), np.maximum(a, b), J)
        np.testing.assert_allclose(k, pit.czado_bins(np.minimum(a, b), np.maximum(a, b), J), rtol=0, atol=1e-12)
        np.testing.assert_allclose(k.sum(1), 1.0, rtol=0, atol=1e-12)


def _gamma_poisson(B, D, S, seed, alpha=2.0, beta=1.0, nb_size=None):
    """Counts x (B, D): Poisson(lam_d) with lam_d ~ Gamma(alpha, beta), or -- nb_size -- negative binomial of the
    same means (over-dispersed).  Exact posterior draws lam (S, D) of the conjugate Poisson model, their per-row
    log-likelihoods ll (B, S) and rates (S, B, D)."""
    rng = np.random.default_rng(seed)
    lam_true = rng.gamma(alpha, 1.0 / beta, D) + 1.0
    if nb_size is None:
        x = rng.poisson(lam_true, (B, D)).astype(np.float64)
    else:
        x = rng.negative_binomial(nb_size, nb_size / (nb_size + lam_true), (B, D)).astype(np.float64)
    a, c = alpha + x.sum(0), beta + B
    lam = rng.gamma(a, 1.0 / c, (S, D))
    ll = st.poisson.logpmf(x[None], lam[:, None, :]).sum(2).T
    return x, np.broadcast_to(lam[:, None, :], (S, B, D)), ll, (a, c)


def test_reference_matches_the_exact_loo_predictive():
    """Gamma-Poisson: without row b, lam_d ~ Gamma(a - x_bd, c - 1), so the exact leave-one-out predictive of x_bd
    is negative binomial (n = a - x_bd, p = (c - 1)/c).  PSIS over 4000 exact posterior draws recovers its CDFs
    at x - 1 and x: mean error below 0.005, worst below 0.03 (Monte Carlo error of the weighted sums)."""
    B, D, S = 60, 6, 4000
    x, rate, ll, (a, c) = _gamma_poisson(B, D, S, seed=1)
    r = pit.loo_pit(x, rate, ll, J=10)
    assert np.all(r['khat'] < 0.5)
    n = a[None, :] - x
    p = (c - 1.0) / c
    exact = np.stack([st.nbinom.cdf(x - 1, n, p), st.nbinom.cdf(x, n, p)], -1)
    err = np.abs(r['P'] - exact)
    assert err.mean() < 5e-3 and err.max() < 3e-2, (err.mean(), err.max())
    assert np.all(r['valid']) and int(r['n']) == B * D
    np.testing.assert_allclose(np.exp(r['lw']).sum(1), 1.0, rtol=0, atol=1e-12)


def test_miscalibration_is_visible():
    """Negative-binomial counts (size 1.5) scored with the Poisson model's leave-one-out predictive pile their PIT
    values at both ends (a U) and move the PIT ECDF much further from uniform than Poisson counts do."""
    B, D, S, J = 200, 8, 1000, 10
    good = pit.loo_pit(*_gamma_poisson(B, D, S, seed=2)[:3], J=J)
    bad = pit.loo_pit(*_gamma_poisson(B, D, S, seed=2, nb_size=1.5)[:3], J=J)
    h = bad['hist'] / bad['n']
    assert h[0] > 1.5 / J and h[-1] > 1.5 / J and h[J // 2] < 0.7 / J, h
    assert bad['ecdf_dev'] > 3 * good['ecdf_dev'], (bad['ecdf_dev'], good['ecdf_dev'])
    assert good['ecdf_dev'] < 0.05
    assert np.all(bad['col_ecdf_dev'] > good['col_ecdf_dev'].max())


def test_new_entry_points_reject_bad_arguments():
    from spmf_b200 import _abi
    lib, BAD = _abi._lib, -1
    fake = C.c_void_p(16)                      # never dereferenced: the checks come first
    # spmf_psis_loo_lw: lw NULL, ldw < S
    assert lib.spmf_psis_loo_lw(fake, 8, 4, 8, fake, fake, fake, None, 8, None) == BAD
    assert lib.spmf_psis_loo_lw(fake, 8, 4, 8, fake, fake, fake, fake, 7, None) == BAD
    assert lib.spmf_psis_loo_lw(fake, 8, 4, 8, None, fake, fake, fake, 8, None) == BAD
    # spmf_loo_pit_accum(xd, nrows, D, K, S, link, EV, PH, z, lw, ldw, acc, inv, rate_out, stream)
    ok = [fake, 4, 5, 3, 2, 0, fake, fake, fake, fake, 2, fake, fake, None, None]
    for i in (0, 6, 7, 8, 9, 11, 12):
        args = list(ok)
        args[i] = None
        assert lib.spmf_loo_pit_accum(*args) == BAD, i
    for i, v in ((1, 0), (2, 0), (3, 0), (3, 513), (4, 0), (4, 65), (5, -1), (5, 4), (10, 1)):
        args = list(ok)
        args[i] = v
        assert lib.spmf_loo_pit_accum(*args) == BAD, (i, v)
    # spmf_loo_pit_hist(acc, inv, nrows, D, J, col_hist, col_n, col_pit_sum, scratch, stream)
    ok = [fake, fake, 4, 5, 20, fake, fake, fake, fake, None]
    for i in (0, 1, 5, 6, 7, 8):
        args = list(ok)
        args[i] = None
        assert lib.spmf_loo_pit_hist(*args) == BAD, i
    for i, v in ((2, 0), (3, 0), (4, 0), (4, 1001)):
        args = list(ok)
        args[i] = v
        assert lib.spmf_loo_pit_hist(*args) == BAD, (i, v)
    assert lib.spmf_loo_pit_hist_scratch_doubles(4, 5, 0) < 0
    assert lib.spmf_loo_pit_hist_scratch_doubles(3000, 5, 20) == 3 * 5 * 22
