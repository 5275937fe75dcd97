"""GPU tests of PSIS leave-one-out: the spmf_psis_loo kernel (csrc/spmf_loo.cu) against the numpy reference
oracle/psis.py, and PoissonFactorization / BernoulliFactorization .loo() against the reference applied to
row_log_likelihood with the same draws, for every link and for custom callables; determinism, batch-size
invariance, training left untouched, the draw limit, and a C4-shaped run."""
import math

import numpy as np
import pytest
import torch

from oracle import psis
from tests.util import make_counts

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
SEED = 12345


def _kernel(ll, S=None, ld_pad=3):
    """spmf_psis_loo on the rows of `ll` (N, S) through the ABI, with a padded leading dimension."""
    from spmf_b200 import _abi
    N, S0 = ll.shape
    S = S0 if S is None else S
    buf = torch.full((N, S0 + ld_pad), 123.0, dtype=torch.float64, device=DEV)     # padding is never read
    buf[:, :S0] = torch.as_tensor(ll, dtype=torch.float64, device=DEV)
    elpd = torch.empty(N, dtype=torch.float64, device=DEV)
    lppd = torch.empty(N, dtype=torch.float64, device=DEV)
    khat = torch.empty(N, dtype=torch.float32, device=DEV)
    _abi.call("spmf_psis_loo", buf.data_ptr(), S0 + ld_pad, N, S, elpd.data_ptr(), lppd.data_ptr(), khat.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return elpd.cpu().numpy(), lppd.cpu().numpy(), khat.cpu().numpy()


def _rows(S, seed):
    """Rows of every kind: Gaussian log-likelihoods (sd 0.1, 1, 5), heavy right tails of the log-ratio (log-t),
    constant rows, rows with many ties (at the cutoff too), and rows holding -inf, NaN or +inf."""
    rng = np.random.default_rng(seed)
    rows = []
    for sd in (0.1, 1.0, 5.0):
        for _ in range(3):
            rows.append(rng.normal(-4.0, sd, S))
    for df in (1.0, 2.0, 4.0):
        rows.append(-3.0 - np.abs(rng.standard_t(df, S)))
    rows.append(np.full(S, -2.5))
    rows.append(-3.0 - 0.5 * rng.integers(0, 4, S))                    # four distinct values: ties everywhere
    t = rng.normal(-4.0, 1.0, S)                                      # ties straddling the cutoff
    M = psis.tail_length(S)
    srt = np.sort(t)
    t[(t >= srt[max(M - 2, 0)]) & (t <= srt[min(M + 2, S - 1)])] = srt[M]
    rows.append(t)
    a = rng.normal(-4.0, 1.0, S)
    a[rng.integers(0, S)] = -np.inf
    rows.append(a)
    rows.append(np.full(S, -np.inf))
    for bad in (np.nan, np.inf):
        b = rng.normal(-4.0, 1.0, S)
        b[rng.integers(0, S)] = bad
        rows.append(b)
    return np.array(rows)


def _assert_like_oracle(got, ref, rtol=1e-10, k_tol=1e-9):
    (e, l, k), (re, rl, rk) = got, ref
    for a, b in ((e, re), (l, rl)):
        assert np.array_equal(np.isnan(a), np.isnan(b))
        assert np.array_equal(np.isposinf(a), np.isposinf(b)) and np.array_equal(np.isneginf(a), np.isneginf(b))
        f = np.isfinite(b)
        np.testing.assert_allclose(a[f], b[f], rtol=rtol, atol=1e-12)
    assert np.array_equal(np.isnan(k), np.isnan(rk)) and np.array_equal(np.isposinf(k), np.isposinf(rk))
    f = np.isfinite(rk)
    # k-hat is returned in fp32: within k_tol of the reference, plus the rounding to fp32
    ulp = np.spacing(np.abs(rk[f]).astype(np.float32)).astype(np.float64)
    assert np.all(np.abs(k[f].astype(np.float64) - rk[f]) <= k_tol + 0.5 * ulp), np.abs(k[f] - rk[f]).max()


@pytest.mark.parametrize("S", [1, 4, 5, 20, 64, 1000, 4095, 8192])
def test_kernel_matches_the_reference(S):
    from spmf_b200.poisson import waic_terms
    ll = _rows(S, seed=S)
    got = _kernel(ll)
    _assert_like_oracle(got, psis.psis_loo(ll))
    fin = np.isfinite(ll).all(1)
    lppd_w, _ = waic_terms(torch.tensor(ll[fin].T))
    np.testing.assert_allclose(got[1][fin], lppd_w.numpy(), rtol=1e-12, atol=1e-12)
    if S >= 1000:
        assert np.isfinite(got[2]).sum() >= 10                     # the smoothed rows are exercised


def test_kernel_is_deterministic_and_rows_are_independent():
    ll = np.concatenate([_rows(1000, seed=s) for s in range(4)])
    a, b = _kernel(ll), _kernel(ll)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    part = _kernel(ll[5:23])
    for x, y in zip(a, part):
        assert np.array_equal(x[5:23].view(np.uint8), y.view(np.uint8))


def _model(link, D, K, custom=False):
    import spmf_b200
    kw = dict(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / math.sqrt(400 * D), device=DEV, seed=3)
    if custom:
        return spmf_b200.PoissonFactorization(encoder_function=lambda x: torch.log1p(x),
                                              decoder_function=lambda y: torch.nn.functional.softplus(y), **kw)
    cls = spmf_b200.BernoulliFactorization if link >= 2 else spmf_b200.PoissonFactorization
    return cls(log_transform=bool(link & 1), **kw)


def _data(link, B, D, seed=1):
    x = make_counts(B, D, seed=seed, kind="noise", rate=1.2)
    return (x > 0).astype(np.float32) if link >= 2 else x


def _chunked_draws(m, S):
    """The draws loo() takes: chunk c = sample(n_c, seed + c), n_c <= LOO_DRAW_CHUNK."""
    from spmf_b200.poisson import LOO_DRAW_CHUNK
    return [m.surrogate_distribution.sample(min(LOO_DRAW_CHUNK, S - c0), seed=SEED + c)
            for c, c0 in enumerate(range(0, S, LOO_DRAW_CHUNK))]


@pytest.mark.parametrize("S", [100, 129])
@pytest.mark.parametrize("link", [0, 1, 2, 3, "custom"])
def test_loo_matches_the_reference_on_row_log_likelihood(link, S):
    D, K, B = 40, 4, 120
    custom = link == "custom"
    link = 0 if custom else link
    m = _model(link, D, K, custom)
    x = _data(link, B, D)
    m.compute_scales(lambda: [{'counts': x}])
    chunks = _chunked_draws(m, S)
    draws = {k: torch.cat([c[k] for c in chunks]) for k in 'suvw'}
    # the reference on the per-chunk row passes (the engines loo() uses, so the same log-likelihoods)
    ll = torch.cat([m.row_log_likelihood({'counts': x}, **c) for c in chunks]).t().cpu().numpy()
    ref = psis.psis_loo(ll)
    res = m.loo({'counts': x}, **draws)
    pw = res['pointwise']
    got = (pw['elpd_loo'].cpu().numpy(), (pw['elpd_loo'] + pw['p_loo']).cpu().numpy(), pw['khat'].cpu().numpy())
    _assert_like_oracle(got, ref, rtol=1e-10)
    assert pw['elpd_loo'].shape == pw['p_loo'].shape == pw['khat'].shape == (B,)
    e, l, k = ref
    thr = min(1 - 1 / math.log10(S), 0.7)
    assert res['khat_threshold'] == thr
    assert res['n_khat_above'] == int((k > thr).sum()) and res['n_nonfinite'] == int((~np.isfinite(e)).sum())
    assert res['elpd_loo'] == pytest.approx(e.sum(), rel=1e-12)
    assert res['lppd'] == pytest.approx(l.sum(), rel=1e-12)
    assert res['p_loo'] == pytest.approx((l - e).sum(), rel=1e-9)
    assert res['looic'] == -2 * res['elpd_loo']
    assert res['se'] == pytest.approx(math.sqrt(B * e.var(ddof=1)), rel=1e-8)
    # The sampled call regenerates the same draws but forms its operands directly (spmf_draw_operands), not through
    # sample()'s fp32 values and _operands_from_theta: its log-likelihoods agree with the explicit ones to fp32
    # operand accuracy, and its results are the reference's on its own log-likelihoods.  (k-hat of a 20-value tail
    # moves by ~100x a relative change of the log-likelihoods, so k-hat is not compared across the two paths.)
    smp = m.loo({'counts': x}, sample_size=S)
    ll_s = m._loo_row_ll(m._csr_batch({'counts': x}, "test"), S, SEED, None).cpu().numpy()
    np.testing.assert_allclose(ll_s, ll, rtol=1e-4, atol=1e-4)
    sp = smp['pointwise']
    got_s = (sp['elpd_loo'].cpu().numpy(), (sp['elpd_loo'] + sp['p_loo']).cpu().numpy(), sp['khat'].cpu().numpy())
    _assert_like_oracle(got_s, psis.psis_loo(ll_s), rtol=1e-10)
    np.testing.assert_allclose(got_s[0], e, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("link", [0, 2])
def test_loo_is_deterministic_and_batch_size_invariant(link):
    from spmf_b200.data import CsrShard
    D, K, B, S = 50, 6, 300, 70
    m = _model(link, D, K)
    x = _data(link, B, D, seed=2)
    shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
    m.compute_scales(shard)
    runs = [m.loo(shard, sample_size=S, batch_size=bs) for bs in (300, 300, 64, 77)]
    totals = ('elpd_loo', 'se', 'p_loo', 'looic', 'lppd', 'n_khat_above', 'n_nonfinite')
    assert all(runs[1][key] == runs[0][key] for key in totals)        # the same call: the same bits
    for r in runs[1:]:
        for key in ('elpd_loo', 'p_loo', 'khat'):
            assert torch.equal(r['pointwise'][key], runs[0]['pointwise'][key]), key
        for key in totals:
            assert r[key] == pytest.approx(runs[0][key], rel=1e-12), key


def test_loo_between_fits_leaves_training_untouched():
    """fit -> loo (its first chunk runs on the training engine, S = 64, on batches larger than the training batch)
    -> fit, against the same two fits without it: the bars of the predictive check's test of the same kind."""
    import spmf_b200
    from spmf_b200.data import CsrShard
    D, K, S, LR = 120, 8, 64, 0.03
    x = make_counts(256, D, seed=6, kind="sparse")
    kw = dict(num_steps=3, sample_size=S, learning_rate=LR, rel_tol=None, verbose=False)

    def run(loo):
        m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=DEV, seed=11)
        shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
        m.compute_scales(shard)
        factory = lambda: shard.iter_batches(64)
        losses = m.fit(factory, **kw)
        eng = m._engine_for(S)
        if loo:
            counters = {s: (e.rng_step, e.opt_step) for s, e in m._engines.items()}
            r = m.loo(shard, sample_size=100, batch_size=256)
            assert np.isfinite(r['lppd'])
            assert {s: (e.rng_step, e.opt_step) for s, e in m._engines.items() if s in counters} == counters
        losses += m.fit(factory, **kw)
        torch.cuda.synchronize()
        return torch.tensor(losses, dtype=torch.float64), eng

    la, ea = run(False)
    lb, eb = run(True)
    assert torch.allclose(la, lb, rtol=1e-7, atol=0), (la - lb).abs().max()
    assert float((ea.params - eb.params).abs().max()) <= 1e-4 * LR * 24
    assert torch.allclose(ea.adam_v, eb.adam_v, rtol=1e-3, atol=1e-12)
    assert (ea.rng_step, ea.opt_step) == (eb.rng_step, eb.opt_step)


def test_loo_rejects_too_many_draws():
    from spmf_b200 import _abi
    m = _model(0, 20, 3)
    x = _data(0, 10, 20)
    with pytest.raises(ValueError):
        m.loo({'counts': x}, sample_size=_abi.LOO_MAX_S + 1)
    with pytest.raises(ValueError):
        m.loo({'counts': x}, sample_size=0)


def test_loo_c4_batch():
    """One C4-shaped batch (8,192 x 20,000, K = 32, S = 1000): finite lppd; the share of rows above the k-hat
    threshold is reported, not asserted -- on rows this wide many high k-hat are the diagnostic doing its job."""
    import spmf_b200
    from spmf_b200.data import synth_scrna_csr_device
    B, D, K = 8192, 20000, 32
    shard = synth_scrna_csr_device(B, D, 0.05, seed=1, device=DEV, gene_seed=1237)
    m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=DEV, u_tau_scale=1e-3)
    m.compute_scales(shard)
    r = m.loo(shard, sample_size=1000, batch_size=B)
    assert math.isfinite(r['lppd'])
    assert r['pointwise']['khat'].shape == (B,)
    print(f"C4 loo: elpd_loo {r['elpd_loo']:.1f}, p_loo {r['p_loo']:.1f}, rows above k-hat "
          f"{r['khat_threshold']:.3f}: {r['n_khat_above'] / B:.3f}")
