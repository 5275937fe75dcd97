"""GPU tests of the posterior predictive check (csrc/spmf_ppc.cu): PoissonFactorization / BernoulliFactorization
.posterior_predictive_check and .posterior_predictive_sample.

The fused statistics are checked against torch reductions of the materialised replicates (the same kernel, draws
and Philox streams, so integer statistics agree exactly), the discrepancies against torch / the float64 oracle
from the rates, the samplers' laws through the public API, invariance to the batch split, run-to-run
determinism, and that a check between two fits leaves training where it was."""
import numpy as np
import pytest
import torch

from tests.util import make_counts, make_oracle

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
INT_KEYS = ('row_total', 'row_nnz', 'col_total', 'col_sumsq', 'col_nnz', 'total', 'nnz', 'max')


def _model(link, D, K, **kw):
    import spmf_b200
    cls = spmf_b200.BernoulliFactorization if link >= 2 else spmf_b200.PoissonFactorization
    return cls(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=DEV, seed=5, log_transform=bool(link & 1), **kw)


def _data(link, B, D, seed):
    x = make_counts(B, D, seed=seed, kind="noise", rate=1.5)
    return (x > 0).astype(np.float32) if link >= 2 else x


def _draws(link, D, K, S, seed, invalid=True):
    """Explicit draws (leading sample axis).  Poisson links: rates that cover both samplers (intercepts up to ~60
    on every third feature) and, with `invalid`, features of negative rate; Bernoulli: logits of either sign."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(S, D, K, generator=g) * (2.0 / D)
    v = torch.rand(S, K, D, generator=g) * (2.0 / K)
    w = torch.rand(S, 1, D, generator=g) * 3.0
    s = torch.rand(S, 2, D, generator=g) + 0.5
    if link >= 2:
        v, w = v - 1.0 / K, 3.0 * w - 4.5
    else:
        w[:, :, ::3] *= 20.0
        if invalid:
            w[:, :, 1::7] = -50.0
    return dict(s=s, u=u, v=v, w=w)


def _torch_discrepancy(link, rate, y):
    """D(y, theta) per draw over the valid entries, float64."""
    rate = rate.double()
    if link < 2:
        valid = torch.isfinite(rate) & (rate >= 0) & (rate <= 2.0 ** 24)
        mean, var = rate, rate
    else:
        valid = torch.isfinite(rate)
        mean = torch.sigmoid(rate)
        var = mean * torch.sigmoid(-rate)
    term = (y.double() - mean) ** 2 / torch.where(valid, var, torch.ones_like(var))
    return torch.where(valid, term, torch.zeros_like(term)).sum((1, 2)), (~valid).sum((1, 2))


@pytest.mark.parametrize("link", [0, 1, 2, 3])
@pytest.mark.parametrize("K,S", [(3, 1), (32, 4), (200, 6)])
def test_fused_statistics_equal_reductions_of_the_replicates(link, K, S):
    D, B, seed, half = 70, 50, 77, 25
    x = _data(link, B, D, seed=1)
    m = _model(link, D, K)
    m.compute_scales(lambda: [{'counts': x}])
    dr = _draws(link, D, K, S, seed=2)
    xt = torch.from_numpy(x).to(DEV).double()
    obs, rep, p, inv = m.posterior_predictive_check(x, seed=seed, **dr)
    y = m.posterior_predictive_sample(x, seed=seed, row_offset=0, **dr).long()
    assert y.shape == (S, B, D) and int(y.min()) >= 0
    # rows are keyed by their global index: the second half alone, numbered from `half`, draws the same replicates
    y2 = m.posterior_predictive_sample(x[half:], seed=seed, row_offset=half, **dr).long()
    assert torch.equal(y2, y[:, half:])
    assert torch.equal(obs['row_total'], xt.sum(1)) and torch.equal(obs['row_nnz'].long(), (xt != 0).sum(1))
    assert torch.equal(rep['row_total'], y.sum(2))
    assert torch.equal(rep['row_nnz'].long(), (y != 0).sum(2))
    assert torch.equal(rep['col_total'], y.sum(1))
    assert torch.equal(rep['col_sumsq'], (y * y).sum(1))
    assert torch.equal(rep['col_nnz'].long(), (y != 0).sum(1))
    assert torch.equal(rep['max'].long(), y.amax((1, 2)))
    assert torch.equal(rep['total'], y.sum((1, 2)))
    assert torch.equal(rep['nnz'], (y != 0).sum((1, 2)))
    assert torch.equal(obs['col_total'], xt.sum(0)) and torch.equal(obs['col_sumsq'], (xt * xt).sum(0))
    assert torch.equal(obs['col_nnz'].long(), (xt != 0).sum(0))
    assert float(obs['total']) == float(xt.sum()) and int(obs['nnz']) == int((xt != 0).sum())
    assert float(obs['max']) == float(xt.max())
    rate = m.log_likelihood_components(data=x, **dr)['rate']
    d_rep, n_bad = _torch_discrepancy(link, rate, y)
    d_obs, _ = _torch_discrepancy(link, rate, xt[None].expand_as(y))
    assert torch.equal(inv, n_bad)
    if link < 2:
        assert int(inv.sum()) > 0                   # the negative-rate features
    assert torch.allclose(rep['discrepancy'], d_rep, rtol=1e-4, atol=0), (rep['discrepancy'], d_rep)
    assert torch.allclose(obs['discrepancy'], d_obs, rtol=1e-4, atol=0), (obs['discrepancy'], d_obs)
    for k, v in p.items():
        assert v.dtype == torch.float64 and bool(((v >= 0) & (v <= 1)).all()), k


def test_observed_discrepancy_matches_the_float64_oracle():
    D, K, B, S = 60, 8, 40, 4
    x = make_counts(B, D, seed=4)
    m = _model(0, D, K)
    m.compute_scales(lambda: [{'counts': x}])
    dr = _draws(0, D, K, S, seed=5, invalid=False)
    oracle = make_oracle(D, K, B, x)
    rate = oracle.log_likelihood_components(data={'counts': torch.tensor(x, dtype=torch.float64)},
                                            **{k: v.double() for k, v in dr.items()})['rate']
    want = ((torch.tensor(x, dtype=torch.float64)[None] - rate) ** 2 / rate).sum((1, 2))
    obs, rep, p, inv = m.posterior_predictive_check(x, seed=3, **dr)
    assert int(inv.sum()) == 0
    got = obs['discrepancy'].cpu()
    assert torch.allclose(got, want, rtol=1e-4, atol=0), (got, want)


@pytest.mark.parametrize("link", [0, 3])
def test_statistics_do_not_depend_on_the_batch_size(link):
    from spmf_b200.data import CsrShard
    D, K, N, S = 90, 16, 150, 4
    x = _data(link, N, D, seed=8)
    m = _model(link, D, K)
    shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
    m.compute_scales(shard)
    a = m.posterior_predictive_check(shard, sample_size=S, batch_size=N, seed=21)
    b = m.posterior_predictive_check(shard, sample_size=S, batch_size=37, seed=21)
    for part in (0, 1):
        for k in INT_KEYS:
            assert torch.equal(a[part][k], b[part][k]), (part, k)
        assert torch.allclose(a[part]['discrepancy'], b[part]['discrepancy'], rtol=1e-12, atol=0)
    assert torch.equal(a[3], b[3])


def test_two_calls_are_bit_identical_and_the_seed_matters():
    from spmf_b200.data import CsrShard
    D, K, N, S = 80, 8, 120, 4
    x = make_counts(N, D, seed=9, kind="sparse")
    m = _model(0, D, K)
    shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
    m.compute_scales(shard)
    a = m.posterior_predictive_check(shard, sample_size=S, batch_size=50, seed=1)
    b = m.posterior_predictive_check(shard, sample_size=S, batch_size=50, seed=1)
    c = m.posterior_predictive_check(shard, sample_size=S, batch_size=50, seed=2)
    for part in (0, 1, 2):
        for k in a[part]:
            assert torch.equal(a[part][k], b[part][k]), (part, k)
    assert torch.equal(a[3], b[3])
    assert not torch.equal(a[1]['row_total'], c[1]['row_total'])
    assert not torch.equal(a[1]['discrepancy'], c[1]['discrepancy'])


@pytest.mark.parametrize("link", [0, 1])
def test_poisson_replicates_have_the_poisson_law_on_the_device(link):
    """u = 0 makes every rate the intercept: lambda_bd = phi_d = eta_d * s1/(s0+s1) * w_d = w_d / 2 (eta = 1,
    s = 1).  phi spans 1e-3 .. 1e4 (both samplers); the per-column mean and variance over N rows must match."""
    D, K, N, S = 24, 4, 10_000, 2
    x = make_counts(N, D, seed=10)
    m = _model(link, D, K)
    phi = torch.tensor(np.geomspace(1e-3, 1e4, D), dtype=torch.float64)
    dr = dict(u=torch.zeros(S, D, K), v=torch.rand(S, K, D), s=torch.ones(S, 2, D),
              w=(2 * phi).float().expand(S, 1, D).clone())
    obs, rep, p, inv = m.posterior_predictive_check(x, seed=31, **dr)
    lam = phi.float().double().to(DEV)              # the fp32 rate the kernel sees
    tot, sq = rep['col_total'].double(), rep['col_sumsq'].double()
    mean = tot / N
    var = (sq - tot * tot / N) / (N - 1)
    assert bool((mean - lam).abs().le(6 * (lam / N).sqrt()).all()), (mean, lam)
    assert bool((var - lam).abs().le(6 * ((lam + 2 * lam * lam) / N).sqrt()).all()), (var, lam)
    assert int(inv.sum()) == 0


def test_bernoulli_replicates_have_the_bernoulli_law_on_the_device():
    D, K, N, S = 16, 4, 10_000, 2
    x = (make_counts(N, D, seed=11) > 0).astype(np.float32)
    m = _model(2, D, K)
    logit = torch.linspace(-6.0, 6.0, D)
    dr = dict(u=torch.zeros(S, D, K), v=torch.rand(S, K, D), s=torch.ones(S, 2, D),
              w=(2 * logit).expand(S, 1, D).clone())
    obs, rep, p, inv = m.posterior_predictive_check(x, seed=32, **dr)
    pr = torch.sigmoid(logit.double()).to(DEV)
    freq = rep['col_total'].double() / N
    assert torch.equal(rep['col_total'], rep['col_sumsq'])       # 0 / 1 replicates
    assert bool((freq - pr).abs().le(6 * (pr * (1 - pr) / N).sqrt()).all()), (freq, pr)
    assert int(rep['max'].max()) == 1 and int(inv.sum()) == 0


def test_check_between_fits_leaves_training_untouched():
    """fit (resident shard, CUDA graphs) -> check on batches 4x the training batch -> fit, against the same two fits
    without the check: the same losses and parameters (to the bars of tests/test_gpu_graphs.py: fp32 atomics
    re-associate between runs), the same counters; the check grew the workspace and moved its generation."""
    import spmf_b200
    from spmf_b200.data import CsrShard
    D, K, S, LR = 120, 8, 4, 0.03
    x = make_counts(256, D, seed=6, kind="sparse")
    kw = dict(num_steps=3, sample_size=S, learning_rate=LR, rel_tol=None, verbose=False)

    def run(check):
        m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=DEV, seed=11)
        shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
        m.compute_scales(shard)
        factory = lambda: shard.iter_batches(64)
        losses = m.fit(factory, **kw)
        eng = m._engine_for(S)
        assert eng.use_graphs and eng.graph_launches > 0
        if check:
            gen, rows, counters = eng._ws_gen, eng.ws.max_rows, (eng.rng_step, eng.opt_step)
            m.posterior_predictive_check(shard, sample_size=S, batch_size=256, seed=4)
            assert eng.ws.max_rows == 256 > rows and eng._ws_gen > gen
            assert (eng.rng_step, eng.opt_step) == counters
        launches = eng.graph_launches
        losses += m.fit(factory, **kw)
        assert eng.graph_launches > launches
        torch.cuda.synchronize()
        return torch.tensor(losses, dtype=torch.float64), eng

    la, ea = run(False)
    lb, eb = run(True)
    assert torch.allclose(la, lb, rtol=1e-7, atol=0), (la - lb).abs().max()
    assert float((ea.params - eb.params).abs().max()) <= 1e-4 * LR * 24
    assert torch.allclose(ea.adam_v, eb.adam_v, rtol=1e-3, atol=1e-12)
    assert (ea.rng_step, ea.opt_step) == (eb.rng_step, eb.opt_step)


def test_errors():
    import spmf_b200
    from spmf_b200.data import DeviceBatch, as_device_batch
    D, K = 30, 4
    x = make_counts(20, D, seed=12)
    custom = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=DEV, encoder_function=lambda t: t)
    with pytest.raises(spmf_b200.SpmfError):
        custom.posterior_predictive_check(x, sample_size=2)
    with pytest.raises(spmf_b200.SpmfError):
        custom.posterior_predictive_sample(x, sample_size=2)
    m = _model(0, D, K)
    b = as_device_batch(x, DEV, D)
    hybrid_only = DeviceBatch(rowptr=b.rowptr, cols=None, vals=None, rowsum=b.rowsum, lgam=b.lgam, nrows=b.nrows,
                              nnz=b.nnz, D=D)
    with pytest.raises(ValueError):
        m.posterior_predictive_check(hybrid_only, sample_size=2)
    with pytest.raises(ValueError):
        m.posterior_predictive_sample(hybrid_only, sample_size=2)
    big = np.ones((512, 600), np.float32)
    with pytest.raises(ValueError):                 # 4096 x 512 x 600 > 2^30 replicates
        _model(0, 600, K).posterior_predictive_sample(big, sample_size=4096)
