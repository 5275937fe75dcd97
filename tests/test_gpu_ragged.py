"""Data-term kernels on ragged batches, checked per element and per row against the float64 oracles.

The parity suite compares whole tensors with a max-norm, which cannot see an error confined to a weakly
expressed feature or to one row.  Here every gradient element of v, w, u and s is held to
|got - ref| <= rtol * M, where M (oracle/analytic.py, magnitudes=True) is the same sum with every summand in
absolute value: the bound an fp32 kernel can be held to whatever the element's size.  The batches
(tests/ragged.py) carry the structure the sparse kernels branch on: empty rows and columns, every row length
against every alignment, columns spanning or ending on the column pass's slices, rows longer than the hot
split's stash, counts either side of the lgamma table and of the upload formats, batches one past a row tile.

Every batch is cut from a larger matrix at a nonzero row offset, and the scales come from that whole matrix.
The Poisson-linear step runs on the gather kernels (K = 4, 32, 256) and the tile-hybrid step (K = 32, 128),
resident and through each host upload format; the log-transform and Bernoulli links (dense kernels) are held
per feature and per row against the autograd oracle.  The InverseGamma-family gradients are reductions over
all of D and K and keep the parity suite's max-norm.

Each tolerance is at most 10x the worst value measured on a B200 (listed below); a run with -s prints the worst
value of every path and tensor at the end of the module.
"""
import functools

import numpy as np
import pytest
import torch
from scipy.special import gammaln

from oracle.analytic import analytic_loss_and_grads
from tests.ragged import (DENSE_LINK_CASES, FEATURE_AXIS, POISSON_CASES, make_case, per_slice_rel_err,
                          worst_ratio)
from tests.util import make_oracle, perturbed_params, rel_err

pytestmark = pytest.mark.gpu

TOL, TOL_IG = 1e-4, 5e-4
# Worst values measured on one NVIDIA B200 (1,000 W power limit): |got - ref| / M 1.0e-6 on the gather path
# (u/loc), 1.1e-5 on the tile path (v/loc: the bf16 three-term split of the tensor-core products), 1.0e-6 for
# encode and 2.1e-7 for the row log-likelihood; per-feature / per-row error 6.4e-5 with the log link (s/scale_raw)
# and 2.7e-5 with the Bernoulli link (w/loc).
RTOL = {"gather": 1e-5, "tile": 1e-4}         # element-wise |got - ref| <= RTOL * M
RTOL_ROWS = 1e-5                               # encode and the per-row log-likelihood, element-wise
TOL_DENSE = {"log_transform": 5e-4, "bernoulli": 2e-4}     # dense links: per-feature / per-row max-norm
RTOL_LGAM = 2e-6                               # row constants: |lgam - ref| <= RTOL_LGAM * sum |lgamma(x + 1)|

# name -> (K, hot_density, S)
PATHS = {"gather4": (4, 0.0, 4), "gather32": (32, 0.0, 4), "gather256": (256, 0.0, 2),
         "tile32": (32, 0.05, 4), "tile128": (128, 0.05, 4)}
UPLOAD_PATHS = ("gather32", "tile32")         # paths that also take every host upload format

WORST = {}


def _record(key, value):
    WORST[key] = max(WORST.get(key, 0.0), value)


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    for key in sorted(WORST):
        print(f"worst {'/'.join(key)}: {WORST[key]:.3e}")


def _load(eng, params):
    views = eng.layout.views(eng.params)
    for k, v in params.items():
        views[k].copy_(v.to(device=eng.device, dtype=torch.float32))


def _uploads(case, sh, model, eng, all_formats):
    """(label, DeviceBatch) of the case's batch: the resident shard's rows and, if asked, each host upload."""
    from spmf_b200.data import BatchUploader, HostCsr, HostDense
    out = [("resident", sh.batch(case.start, case.B))]
    if all_formats:
        hosts = (("int32", HostCsr.from_shard(sh, compact=False)), ("uint16", HostCsr.from_shard(sh)),
                 ("u8", HostCsr.from_shard(sh, compact="u8")), ("dense", HostDense(case.x)))
        for label, host in hosts:
            up = BatchUploader(sh.rowptr.device, case.D, hot=model._hot_spec(eng))
            out.append((label, up.upload(host.batch(case.start, case.B))))
    return out


def _check_row_consts(db, xb, label):
    torch.cuda.synchronize()
    np.testing.assert_allclose(db.rowsum[:xb.shape[0]].cpu().numpy(), xb.astype(np.float64).sum(1), rtol=1e-6,
                               err_msg=label)
    lg = gammaln(xb.astype(np.float64) + 1.0)
    got = db.lgam[:xb.shape[0]].cpu().numpy().astype(np.float64)
    assert (np.abs(got - lg.sum(1)) <= RTOL_LGAM * np.abs(lg).sum(1) + 1e-6).all(), (label, got, lg.sum(1))


@functools.lru_cache(maxsize=2)
def _reference(name, K, S):
    """Oracle, parameters, noise and the analytic step with magnitudes (shared by the paths of one K)."""
    from oracle.spmf_oracle import draw_noise
    case = make_case(name)
    N, D = case.x.shape
    oracle = make_oracle(D, K, N, case.x)
    params = perturbed_params(oracle, 0.3, seed=7)
    noise = draw_noise(oracle, params, S, seed=8)
    return oracle, params, noise, analytic_loss_and_grads(oracle, params, noise, case.batch, c_gamma=True,
                                                          magnitudes=True)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("name", POISSON_CASES)
def test_poisson_step_per_element(name, path):
    import spmf_b200
    K, hd, S = PATHS[path]
    family = "tile" if hd > 0 else "gather"
    case = make_case(name)
    N, D = case.x.shape
    dev = torch.device("cuda:0")
    xb = case.batch
    oracle, params, noise, ref = _reference(name, K, S)
    ref_loss, ref_grads, ref_parts, mags, rows = ref

    model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(N * D),
                                           device=dev, hot_density=hd, seed=1)
    sh = spmf_b200.CsrShard.from_dense(case.x, dev)
    model.compute_scales(sh)
    assert rel_err(model.eta_i.numpy(), oracle.eta_i.numpy()) < 1e-12
    eng = model._engine_for(S)
    if family == "tile":
        assert eng.hybrid_ok and eng.hot_cols >= 64, (eng.hybrid_ok, eng.hot_cols)
    else:
        assert eng.hot_cols == 0
    for label, db in _uploads(case, sh, model, eng, path in UPLOAD_PATHS):
        _check_row_consts(db, xb, label)
        _load(eng, params)
        eng.set_noise_from(noise)
        p = eng.loss_and_grad(db, fresh_noise=False)
        torch.cuda.synchronize()
        if family == "tile":
            assert db.hot is not None and db.hot.H == eng.hot_cols, label
        loss = float(eng.loss_value(p).item())
        assert abs(loss - ref_loss) <= TOL * abs(ref_loss), (label, loss, ref_loss)
        pd = eng.parts_dict()
        for pn, ref in ref_parts.items():
            assert np.abs(pd[pn].numpy() - ref).max() <= TOL * max(np.abs(ref).max(), 1.0), (label, pn)
        grads = eng.layout.views(eng.grads)
        for k, g in ref_grads.items():
            got = grads[k].cpu().numpy()
            if k in mags:
                r = worst_ratio(got, g, mags[k])
                _record((family, k), r)
                assert r <= RTOL[family], (label, k, r)
            else:
                assert rel_err(got, g) <= TOL_IG, (label, k)

    # row-side outputs, row by row, with the same draws
    theta, _ = oracle.sample(params, noise)
    th = {k: theta[k].detach().to(dev, torch.float32) for k in ("s", "u", "v", "w")}
    db = sh.batch(case.start, case.B)
    z = model.encode(db, th["u"], th["s"]).cpu().numpy()
    r = worst_ratio(z, *rows["z"])
    _record(("rows", "z"), r)
    assert r <= RTOL_ROWS, ("z", r)
    ll = model.row_log_likelihood(db, **th).cpu().numpy()
    r = worst_ratio(ll, *rows["row_ll"])
    _record(("rows", "row_ll"), r)
    assert r <= RTOL_ROWS, ("row_ll", r)


@pytest.mark.parametrize("name", POISSON_CASES + ["rows_650"])
def test_ppc_observed_statistics_exact(name):
    """The check's statistics of the data itself on the ragged batches, against numpy."""
    import spmf_b200
    case = make_case(name)
    N, D = case.x.shape
    dev = torch.device("cuda:0")
    model = spmf_b200.PoissonFactorization(latent_dim=4, feature_dim=D, device=dev, seed=2)
    sh = spmf_b200.CsrShard.from_dense(case.x, dev)
    model.compute_scales(sh)
    th = model.sample(2, seed=3)
    obs, _, _, _ = model.posterior_predictive_check(sh.batch(case.start, case.B),
                                                    **{k: th[k] for k in ("s", "u", "v", "w")})
    x = case.batch.astype(np.float64)
    exp = dict(row_total=x.sum(1), row_nnz=(x != 0).sum(1), col_total=x.sum(0), col_nnz=(x != 0).sum(0),
               total=x.sum(), nnz=(x != 0).sum(), max=x.max())
    for k, v in exp.items():
        np.testing.assert_array_equal(obs[k].cpu().numpy(), v, err_msg=k)
    sq = (x * x).sum(0)
    if (x == np.round(x)).all():
        np.testing.assert_array_equal(obs["col_sumsq"].cpu().numpy(), sq)
    else:          # squares of non-integer fp32 counts carry more bits than a double sum keeps in every order
        np.testing.assert_allclose(obs["col_sumsq"].cpu().numpy(), sq, rtol=1e-15)


@pytest.mark.parametrize("link", ["log_transform", "bernoulli"])
@pytest.mark.parametrize("name", DENSE_LINK_CASES)
def test_dense_link_step_per_feature_and_row(name, link):
    import spmf_b200
    from oracle.spmf_oracle import OracleBernoulliFactorization, draw_noise
    K, S = 8, 2
    case = make_case(name)
    N, D = case.x.shape
    dev = torch.device("cuda:0")
    full = case.x if link == "log_transform" else (case.x > 0).astype(np.float32)
    xb = full[case.start:case.start + case.B]
    data = {'counts': torch.tensor(xb, dtype=torch.float64)}
    kw = dict(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(N * D), device=dev)
    if link == "log_transform":
        oracle = make_oracle(D, K, N, full, log_transform=True)
        params = perturbed_params(oracle, 0.3, seed=2)
        model = spmf_b200.PoissonFactorization(log_transform=True, **kw)
        model.compute_scales(spmf_b200.CsrShard.from_dense(full, dev))
        assert rel_err(model.eta_i.numpy(), oracle.eta_i.numpy()) < 1e-12
    else:
        oracle = OracleBernoulliFactorization(K, D, u_tau_scale=1.0 / np.sqrt(N * D))
        params = perturbed_params(oracle, 0.3, seed=4)
        g = torch.Generator().manual_seed(9)        # logits of both signs (v, w are unconstrained here)
        params['v/loc'] = (0.3 * torch.randn(params['v/loc'].shape, generator=g, dtype=torch.float64)).float().double()
        params['w/loc'] = (0.5 * torch.randn(params['w/loc'].shape, generator=g, dtype=torch.float64)).float().double()
        params['u/loc'] = params['u/loc'] + 4.0
        model = spmf_b200.BernoulliFactorization(**kw)
    noise = draw_noise(oracle, params, S, seed=3)
    ref_loss, ref_grads, ref_parts = oracle.loss_and_grads(params, noise, data)
    eng = model._engine_for(S)
    assert eng.link != 0
    sh = spmf_b200.CsrShard.from_dense(full, dev)
    db = sh.batch(case.start, case.B)
    _load(eng, params)
    eng.set_noise_from(noise)
    p = eng.loss_and_grad(db, fresh_noise=False)
    torch.cuda.synchronize()
    loss = float(eng.loss_value(p).item())
    assert abs(loss - ref_loss) <= TOL * abs(ref_loss), (loss, ref_loss)
    pd = eng.parts_dict()
    for pn, ref in ref_parts.items():
        ref = ref.numpy()
        assert np.abs(pd[pn].numpy() - ref).max() <= TOL * max(np.abs(ref).max(), 1.0), pn
    grads = eng.layout.views(eng.grads)
    for k, g in ref_grads.items():
        got, g = grads[k].cpu().numpy(), g.numpy()
        var = k.split('/')[0]
        if var in FEATURE_AXIS:
            e = per_slice_rel_err(got, g, FEATURE_AXIS[var])
            _record((link, k), e)
            assert e <= TOL_DENSE[link], (k, e)
        else:
            assert rel_err(got, g) <= TOL_IG, k
    theta, _ = oracle.sample(params, noise)
    th64 = {k: theta[k].detach() for k in ("s", "u", "v", "w")}
    th = {k: v.to(dev, torch.float32) for k, v in th64.items()}
    z = model.encode(db, th["u"], th["s"]).cpu().numpy()
    e = per_slice_rel_err(z, oracle.encode(data['counts'], th64["u"], th64["s"]).numpy(), axis=1)
    _record((link, "z"), e)
    assert e <= TOL_DENSE[link], ("z", e)
    ll = model.row_log_likelihood(db, **th).cpu().numpy()
    ref_ll = oracle.log_likelihood_components(data=data, **th64)['log_likelihood'].sum(-1).numpy()
    e = per_slice_rel_err(ll, ref_ll, axis=1)
    _record((link, "row_ll"), e)
    assert e <= TOL_DENSE[link], ("row_ll", e)
