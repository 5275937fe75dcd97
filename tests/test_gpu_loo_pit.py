"""GPU tests of LOO-PIT: spmf_psis_loo_lw (csrc/spmf_loo.cu) against spmf_psis_loo and oracle/pit.py, spmf_loo_pit_accum
and spmf_loo_pit_hist (csrc/spmf_pit.cu) against the reference fed the kernels' own fp32 rates and weights, and
PoissonFactorization / BernoulliFactorization .loo_pit / .loo_pit_values end to end against the float64 reference;
determinism and batch-size invariance, training left untouched, a calibration contrast, a C4-shaped run, errors."""
import math

import numpy as np
import pytest
import torch

from oracle import pit
from tests.ragged import make_case
from tests.test_gpu_loo import _rows
from tests.util import make_counts, make_oracle

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
SEED = 12345


def _loo_lw(ll):
    """(elpd, lppd, khat, lw) of spmf_psis_loo_lw and (elpd, lppd, khat) of spmf_psis_loo on the rows of ll."""
    from spmf_b200 import _abi
    N, S = ll.shape
    t = torch.as_tensor(ll, dtype=torch.float64, device=DEV).contiguous()
    out = [torch.empty(N, dtype=torch.float64, device=DEV) for _ in range(4)]
    kh = [torch.empty(N, dtype=torch.float32, device=DEV) for _ in range(2)]
    lw = torch.full((N, S + 2), 7.0, dtype=torch.float64, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    _abi.call("spmf_psis_loo_lw", t.data_ptr(), S, N, S, out[0].data_ptr(), out[1].data_ptr(), kh[0].data_ptr(),
              lw.data_ptr(), S + 2, st)
    _abi.call("spmf_psis_loo", t.data_ptr(), S, N, S, out[2].data_ptr(), out[3].data_ptr(), kh[1].data_ptr(), st)
    torch.cuda.synchronize()
    assert bool((lw[:, S:] == 7.0).all())                      # the row padding is never written
    return (out[0], out[1], kh[0], lw[:, :S]), (out[2], out[3], kh[1])


@pytest.mark.parametrize("S", [1, 5, 64, 1000, 8192])
def test_log_weights_match_the_reference_and_leave_loo_unchanged(S):
    ll = _rows(S, seed=S)
    (e, l, k, lw), (e0, l0, k0) = _loo_lw(ll)
    for a, b in ((e, e0), (l, l0), (k, k0)):                   # bit for bit
        assert torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(), b.nan_to_num())
    ref, elpd, _ = pit.loo_weights(ll)
    lw = lw.cpu().numpy()
    fin = np.isfinite(elpd)
    assert np.array_equal(np.isfinite(e.cpu().numpy()), fin)
    assert np.isnan(lw[~fin]).all()
    np.testing.assert_allclose(lw[fin], ref[fin], rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(np.exp(lw[fin]).sum(1), 1.0, rtol=0, atol=1e-12)


def _model(link, D, K, **kw):
    import spmf_b200
    cls = spmf_b200.BernoulliFactorization if link >= 2 else spmf_b200.PoissonFactorization
    return cls(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / math.sqrt(400 * D), device=DEV, seed=3,
               log_transform=bool(link & 1), **kw)


def _data(link, B, D, seed=1):
    """Counts with a few large ones (up to 1e5) and one non-integer (Poisson); 0/1 with one 2 (Bernoulli)."""
    x = make_counts(B, D, seed=seed, kind="noise", rate=1.2)
    if link >= 2:
        x = (x > 0).astype(np.float32)
        x[1, 2] = 2.0                                # not in the Bernoulli support: invalid
        return x
    x[0, :3] = [1e5, 3e4, 999.0]
    x[2, 1] = 2.5                                    # not an integer: invalid
    return x


def _draws(link, D, K, S, seed=2):
    """Explicit draws; Poisson links get features of negative rate (invalid entries) on every 7th feature."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(S, D, K, generator=g) * (2.0 / D)
    v = torch.rand(S, K, D, generator=g) * (2.0 / K)
    w = torch.rand(S, 1, D, generator=g) * 3.0
    s = torch.rand(S, 2, D, generator=g) + 0.5
    if link >= 2:
        v, w = v - 1.0 / K, 3.0 * w - 4.5
    else:
        w[:, :, 3::7] = -50.0
    return dict(s=s, u=u, v=v, w=w)


def _accum_against_reference(m, x, S, draws=None, bernoulli=False):
    """The kernels' (P-, P+) and invalid counts of batch x against oracle/pit.py on the kernel's own fp32 rates and
    log weights; returns the kernel's P."""
    b = m._csr_batch({'counts': x}, "test")
    theta = None if draws is None else {k: torch.as_tensor(draws[k]) for k in 'suvw'}
    rates = []
    acc, inv, elpd, _ = m._loo_pit_batch(b, S, SEED, theta, rates=rates)
    ll = m._loo_row_ll(b, S, SEED, theta)
    (_, _, _, lw), _ = _loo_lw(ll)
    rate = torch.cat(rates).cpu().numpy()
    assert rate.shape == (S,) + x.shape
    P, n_inv = pit.pit_values(np.abs(x), rate, lw.cpu().numpy(), bernoulli)
    fin = torch.isfinite(elpd).cpu().numpy()
    got = acc.cpu().numpy()
    assert np.array_equal(inv.cpu().numpy(), n_inv)
    np.testing.assert_allclose(got[fin], P[fin], rtol=0, atol=1e-10)
    return got, n_inv


@pytest.mark.parametrize("K", [3, 32, 200, 512])
@pytest.mark.parametrize("link", [0, 1, 2, 3])
def test_accum_matches_the_reference_on_the_kernels_rates(link, K):
    D, B, S = 45, 37, 5
    m = _model(link, D, K)
    x = _data(link, B, D)
    m.compute_scales(lambda: [{'counts': x}])
    _, n_inv = _accum_against_reference(m, x, S, _draws(link, D, K, S), bernoulli=link >= 2)
    assert n_inv.sum() > 0                          # the invalid entries are exercised


@pytest.mark.parametrize("S", [1, 64, 129])
@pytest.mark.parametrize("link", [0, 3])
def test_accum_over_several_chunks(link, S):
    D, B, K = 40, 30, 32
    m = _model(link, D, K)
    x = _data(link, B, D, seed=4)
    m.compute_scales(lambda: [{'counts': x}])
    _accum_against_reference(m, x, S, bernoulli=link >= 2)             # sampled draws, chunks of 64
    _accum_against_reference(m, x, S, _draws(link, D, K, S), bernoulli=link >= 2)


@pytest.mark.parametrize("case", ["empty_rows", "empty_cols", "long_rows", "large_counts", "rows_1", "rows_129"])
def test_accum_on_ragged_batches(case):
    c = make_case(case)
    m = _model(0, c.D, 8)
    m.compute_scales(lambda: [{'counts': c.x}])
    _accum_against_reference(m, c.batch, 5)


@pytest.mark.parametrize("link", [0, 1])
def test_end_to_end_against_the_float64_reference(link):
    D, K, B, S = 30, 4, 40, 70
    m = _model(link, D, K)
    x = make_counts(B, D, seed=5, kind="noise", rate=1.2)
    m.compute_scales(lambda: [{'counts': x}])
    dr = _draws(link, D, K, S, seed=6)
    for k in dr:
        dr[k] = dr[k].abs()                         # every rate valid
    oracle = make_oracle(D, K, B, x, log_transform=bool(link & 1))
    comp = oracle.log_likelihood_components(data={'counts': torch.tensor(x, dtype=torch.float64)},
                                            **{k: v.double() for k, v in dr.items()})
    rate = comp['rate'].cpu().numpy()
    ll = comp['log_likelihood'].sum(-1).T.cpu().numpy()
    ref = pit.loo_pit(x, rate, ll, J=10)
    got = m.loo_pit_values({'counts': x}, **dr).cpu().numpy()
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, ref['P'], rtol=0, atol=1e-4)


@pytest.mark.parametrize("J", [1, 20, 1000])
@pytest.mark.parametrize("link", [0, 2])
def test_histograms_match_the_reference_on_the_kernels_values(link, J):
    D, K, B, S = 50, 6, 60, 20
    m = _model(link, D, K)
    x = _data(link, B, D, seed=7)
    m.compute_scales(lambda: [{'counts': x}])
    dr = _draws(link, D, K, S, seed=8)
    r = m.loo_pit({'counts': x}, bins=J, **dr)
    P = m.loo_pit_values({'counts': x}, **dr).cpu().numpy()
    valid = ~np.isnan(P).any(-1)
    col_hist, col_n, col_pit = pit.histograms(np.nan_to_num(P), valid, J)
    hist, n, dev, col_dev = pit.summary(col_hist, col_n)
    np.testing.assert_allclose(r['col_hist'].cpu().numpy(), col_hist, rtol=1e-12, atol=1e-13)
    assert np.array_equal(r['col_n'].cpu().numpy(), col_n) and r['n'] == n
    np.testing.assert_allclose(r['col_mean_pit'].cpu().numpy(), col_pit / col_n, rtol=1e-12)
    np.testing.assert_allclose(r['hist'].cpu().numpy(), hist, rtol=1e-12, atol=1e-13)
    assert r['ecdf_dev'] == pytest.approx(dev, rel=1e-10, abs=1e-13)
    np.testing.assert_allclose(r['col_ecdf_dev'].cpu().numpy(), col_dev, rtol=1e-10, atol=1e-13)
    assert r['n_invalid'] + r['n_rows_excluded'] * D == int((~valid).sum()) and r['n_invalid'] > 0
    assert r['n'] + r['n_invalid'] + r['n_rows_excluded'] * D == B * D
    thr = min(1 - 1 / math.log10(S), 0.7)
    assert r['khat_threshold'] == thr


def test_results_are_bit_identical_across_calls_and_batch_sizes():
    from spmf_b200.data import CsrShard
    D, K, N, S = 60, 8, 30, 70
    m = _model(0, D, K)
    x = make_counts(N, D, seed=9, kind="noise", rate=1.0)
    shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
    m.compute_scales(shard)
    full = m.loo_pit_values({'counts': x}, sample_size=S)
    assert torch.equal(full, m.loo_pit_values({'counts': x}, sample_size=S))
    # batches cut from one shard (the row pass that encodes z sums a row the same way wherever the row starts in
    # the same CSR arrays; fresh arrays may start it at another alignment, which moves z by an fp32 rounding)
    for lo, hi in ((0, 1), (3, 10), (29, 30)):
        assert torch.equal(m.loo_pit_values(shard.batch(lo, hi - lo), sample_size=S), full[lo:hi]), (lo, hi)
    runs = {bs: m.loo_pit(shard, sample_size=S, batch_size=bs, bins=12) for bs in (N, N, 7, 1)}
    again = m.loo_pit(shard, sample_size=S, batch_size=N, bins=12)
    for k in ('hist', 'col_hist', 'col_n', 'col_mean_pit', 'col_ecdf_dev'):
        assert torch.equal(again[k], runs[N][k]), k
        for bs in (7, 1):
            assert torch.allclose(runs[bs][k].double(), runs[N][k].double(), rtol=1e-12, atol=1e-14), (bs, k)
    for bs in (7, 1):
        for k in ('n', 'n_invalid', 'n_rows_excluded', 'n_khat_above'):
            assert runs[bs][k] == runs[N][k], (bs, k)
        assert torch.equal(runs[bs]['col_n'], runs[N]['col_n'])


def test_loo_pit_between_fits_leaves_training_untouched():
    import spmf_b200
    from spmf_b200.data import CsrShard
    D, K, S, LR = 120, 8, 64, 0.03
    x = make_counts(256, D, seed=6, kind="sparse")
    kw = dict(num_steps=3, sample_size=S, learning_rate=LR, rel_tol=None, verbose=False)

    def run(check):
        m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=DEV, seed=11)
        shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
        m.compute_scales(shard)
        factory = lambda: shard.iter_batches(64)
        losses = m.fit(factory, **kw)
        eng = m._engine_for(S)
        if check:
            counters = {s: (e.rng_step, e.opt_step) for s, e in m._engines.items()}
            r = m.loo_pit(shard, sample_size=100, batch_size=256)
            assert r['n'] > 0
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


def test_calibration_contrast_on_the_device():
    """u = 0 makes every rate the intercept phi_d, whatever the counts: counts replicated from the model by
    posterior_predictive_sample are calibrated, negative-binomial counts of the same means (size 1) are not."""
    D, K, N, S = 16, 4, 4000, 8
    m = _model(0, D, K)
    phi = torch.tensor(np.geomspace(0.3, 30.0, D), dtype=torch.float32)
    dr = dict(u=torch.zeros(S, D, K), v=torch.rand(S, K, D), s=torch.ones(S, 2, D),
              w=(2 * phi).expand(S, 1, D).clone())
    seed_x = make_counts(N, D, seed=12)
    y = m.posterior_predictive_sample(seed_x, seed=5, **{k: v[:1] for k, v in dr.items()})[0].float()
    g = torch.Generator(device=DEV).manual_seed(3)
    lam = phi.to(DEV)[None].expand(N, D) * torch._standard_gamma(torch.ones(N, D, device=DEV), generator=g)
    over = torch.poisson(lam, generator=g)
    good = m.loo_pit({'counts': y.cpu().numpy()}, bins=10, **dr)
    bad = m.loo_pit({'counts': over.cpu().numpy()}, bins=10, **dr)
    assert good['n'] == bad['n'] == N * D
    assert float(bad['col_ecdf_dev'].min()) > float(good['col_ecdf_dev'].max())
    assert bad['ecdf_dev'] > 3 * good['ecdf_dev']
    h = (bad['hist'] / bad['n']).cpu().numpy()
    assert h[0] > 0.15 and h[-1] > 0.15                      # the U of over-dispersed data


def test_loo_pit_c4_batch():
    """A C4-shaped batch (8,192 x 20,000, K = 32) at S = 64: finite results of the right shapes."""
    import spmf_b200
    from spmf_b200.data import synth_scrna_csr_device
    B, D, K, J = 8192, 20000, 32, 20
    shard = synth_scrna_csr_device(B, D, 0.05, seed=1, device=DEV, gene_seed=1237)
    m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=DEV, u_tau_scale=1e-3)
    m.compute_scales(shard)
    r = m.loo_pit(shard, sample_size=64, bins=J)
    assert r['hist'].shape == (J,) and r['col_hist'].shape == (D, J) and r['col_n'].shape == (D,)
    assert r['n'] + r['n_invalid'] + r['n_rows_excluded'] * D == B * D
    assert math.isfinite(r['ecdf_dev']) and bool(torch.isfinite(r['hist']).all())
    assert float(r['hist'].sum()) == pytest.approx(r['n'], rel=1e-9)
    print(f"C4 loo_pit (S = 64): ecdf_dev {r['ecdf_dev']:.4f}, invalid {r['n_invalid']}, "
          f"rows excluded {r['n_rows_excluded']}, rows above k-hat {r['n_khat_above']}")


def test_errors():
    import spmf_b200
    D, K = 30, 4
    x = make_counts(20, D, seed=12)
    custom = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=DEV, encoder_function=lambda t: t)
    with pytest.raises(spmf_b200.SpmfError):
        custom.loo_pit({'counts': x}, sample_size=2)
    with pytest.raises(spmf_b200.SpmfError):
        custom.loo_pit_values({'counts': x}, sample_size=2)
    m = _model(0, D, K)
    for bins in (0, 1001):
        with pytest.raises(ValueError):
            m.loo_pit({'counts': x}, sample_size=2, bins=bins)
    with pytest.raises(ValueError):
        m.loo_pit({'counts': x}, sample_size=0)
    import scipy.sparse
    big = _model(0, 1 << 14, K)
    with pytest.raises(ValueError):                 # (2^13 + 1) x 2^14 > 2^27 entries
        n = (1 << 13) + 1
        one = scipy.sparse.csr_matrix((np.ones(n, np.float32), (np.arange(n), np.zeros(n, int))), shape=(n, 1 << 14))
        big.loo_pit_values({'counts': one}, sample_size=2)
