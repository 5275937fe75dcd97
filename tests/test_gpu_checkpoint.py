"""Checkpoints (save_checkpoint / load / fit(checkpoint_path=..., resume=True)): a model loaded from a checkpoint
continues exactly like the live model it was taken from.  Two runs of the same computation are compared with the
bars of tests/test_gpu_graphs.py: losses to rtol 1e-7 per step, parameters within a fraction of one Adam step,
adam_v to rtol 1e-3 (fp32 atomics re-associate between runs), counters equal."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.util import make_counts

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda:0")
LR, CLIP = 0.03, 2.0


def _read(path):
    import dill
    with open(path, "rb") as f:
        return dill.load(f)


def _data(D, kind, bernoulli):
    x = make_counts(256, D, seed=3, kind=kind)
    return (x > 0).astype(np.float32) if bernoulli else x


def _model(bernoulli, D, K, log_transform=False, **kw):
    import spmf_b200
    cls = spmf_b200.BernoulliFactorization if bernoulli else spmf_b200.PoissonFactorization
    return cls(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=DEV, seed=11, log_transform=log_transform, **kw)


def _steps(m, shard, S, first, n):
    batches = list(shard.iter_batches(64))
    out = []
    for i in range(first, first + n):
        cur = LR * (0.5 if i >= 12 else 1.0)         # a learning-rate change after the resume
        out.append(m.elbo_step({'counts': batches[i % len(batches)]}, S, learning_rate=cur, clip_value=CLIP))
    return out


def _assert_same_run(ea, eb, steps):
    assert float((ea.params - eb.params).abs().max()) <= 1e-4 * LR * steps
    assert torch.allclose(ea.adam_v, eb.adam_v, rtol=1e-3, atol=1e-12)
    assert ea.opt_step == eb.opt_step and ea.rng_step == eb.rng_step


@pytest.mark.parametrize("D,K,S,kind,log_transform,bernoulli", [
    (192, 16, 4, "linear", False, False),      # tcgen05 tile-hybrid step
    (40, 4, 4, "noise", False, False),         # gather step
    (300, 32, 4, "sparse", False, False),      # hot + cold columns
    (48, 8, 2, "noise", True, False),          # dense link
    (64, 8, 4, "noise", False, True),          # Bernoulli
])
def test_resume_from_checkpoint_matches_uninterrupted_steps(tmp_path, D, K, S, kind, log_transform, bernoulli):
    from spmf_b200.data import CsrShard
    x = _data(D, kind, bernoulli)
    shard_a, shard_b = CsrShard.from_dense(torch.from_numpy(x), DEV), CsrShard.from_dense(torch.from_numpy(x), DEV)
    a = _model(bernoulli, D, K, log_transform)
    a.compute_scales(shard_a)
    la = _steps(a, shard_a, S, 0, 16)
    b = _model(bernoulli, D, K, log_transform)
    b.compute_scales(shard_b)
    lb = _steps(b, shard_b, S, 0, 8)
    path = tmp_path / "run.ckpt"
    b.save_checkpoint(str(path))
    assert not os.path.exists(str(path) + ".tmp")
    c = type(b).load(str(path), device=DEV)                   # no compute_scales: the checkpoint carries the ranking
    lc = _steps(c, shard_b, S, 8, 8)
    torch.cuda.synchronize()
    la, lbc = torch.stack(la).cpu(), torch.stack(lb + lc).cpu()
    assert torch.allclose(la, lbc, rtol=1e-7, atol=0), (la - lbc).abs().max()
    assert bool(torch.isfinite(lbc).all())
    ea, ec = a._engine_for(S), c._engine_for(S)
    _assert_same_run(ea, ec, 16)
    assert ea.opt_step == 16
    assert torch.equal(a.eta_i, c.eta_i) and a.xi_u_global == c.xi_u_global
    # the same step form: hot columns and the tile-hybrid path
    batch = next(iter(shard_b.iter_batches(64)))
    assert (ec.hot_cols, ec.hybrid_ok, ec._runs_hybrid(batch)) == (ea.hot_cols, ea.hybrid_ok, ea._runs_hybrid(batch))
    if kind == "linear":
        assert ec._runs_hybrid(batch)
    # every engine's counters travel (engines for different S keep their own)
    for s_, e in a._engines.items():
        got = (c._engines[s_].opt_step, c._engines[s_].rng_step) if s_ in c._engines else c._pending_counters[s_]
        assert got == (e.opt_step, e.rng_step), s_


def _fit_kwargs():
    return dict(num_steps=6, learning_rate=0.05, sample_size=4, clip_value=2.0, rel_tol=None, patience=1,
                lr_decay_factor=0.5, verbose=False)


def test_fit_resumes_after_preemption(tmp_path):
    from spmf_b200.data import CsrShard
    D, K = 300, 32
    x = make_counts(256, D, seed=5, kind="sparse")
    shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
    keep = []                                                # (models stay alive: no buffer is reused meanwhile)

    def make():
        m = _model(False, D, K)
        m.compute_scales(shard)
        keep.append(m)
        return m

    def factory():
        return ({'counts': b} for b in shard.iter_batches(64))

    p_full, p_cut = str(tmp_path / "full.ckpt"), str(tmp_path / "cut.ckpt")
    full = make().fit(factory, checkpoint_path=p_full, **_fit_kwargs())
    calls = [0]

    def flaky():
        calls[0] += 1
        if calls[0] == 4:
            raise RuntimeError("preempted")
        return factory()

    with pytest.raises(RuntimeError, match="preempted"):
        make().fit(flaky, checkpoint_path=p_cut, **_fit_kwargs())
    assert _read(p_cut)['training']['fit']['epoch'] == 3
    resumed = make().fit(factory, checkpoint_path=p_cut, resume=True, **_fit_kwargs())
    assert len(resumed) == len(full) == 6
    np.testing.assert_allclose(resumed, full, rtol=1e-6)
    fa, fb = _read(p_full)['training']['fit'], _read(p_cut)['training']['fit']
    assert fa['epoch'] == fb['epoch'] == 6 and fa['decays'] == fb['decays'] and fa['lr'] == fb['lr']
    e_full, e_resumed = keep[0]._engine_for(4), keep[2]._engine_for(4)
    assert (e_full.opt_step, e_full.rng_step) == (e_resumed.opt_step, e_resumed.rng_step)
    # a finished run resumes to nothing more
    again = make().fit(factory, checkpoint_path=p_cut, resume=True, **_fit_kwargs())
    assert again == resumed


def test_streamed_resume_builds_the_hybrid_form_from_the_stored_ranking(tmp_path):
    from spmf_b200.data import CsrShard, HostCsr
    D, K, S = 192, 16, 4
    x = make_counts(256, D, seed=3, kind="linear")
    shard = CsrShard.from_dense(torch.from_numpy(x), DEV)
    host = HostCsr.from_shard(shard)

    def factory():
        return ({'counts': b} for b in host.iter_batches(64))

    kw = dict(learning_rate=0.03, sample_size=S, clip_value=2.0, rel_tol=None, verbose=False)
    a = _model(False, D, K)
    a.compute_scales(shard)
    la = a.fit(factory, num_steps=4, **kw)
    b = _model(False, D, K)
    b.compute_scales(shard)
    path = str(tmp_path / "stream.ckpt")
    b.fit(factory, num_steps=2, checkpoint_path=path, **kw)
    c = _model(False, D, K)                                  # no compute_scales
    lc = c.fit(factory, num_steps=4, checkpoint_path=path, resume=True, **kw)
    np.testing.assert_allclose(lc, la, rtol=1e-6)
    eng = c._engine_for(S)
    assert c.hot_cols == a.hot_cols > 0 and torch.equal(c.col_rank, a.col_rank)
    assert c._hot_spec(eng) is not None
    db = next(iter(c._device_batches(factory(), eng)))
    assert db.hot is not None and db.hot.H == a.hot_cols and eng._runs_hybrid(db)
    _assert_same_run(a._engine_for(S), eng, 16)


def test_custom_encoder_round_trips_through_a_checkpoint(tmp_path):
    import spmf_b200
    D, K, S = 24, 3, 2
    x = make_counts(64, D, seed=4)
    m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1e-2, device=DEV, seed=5,
                                       encoder_function=lambda t: torch.log1p(t) * 0.5)
    m.compute_scales(lambda: [{'counts': x}])
    for _ in range(3):
        m.elbo_step({'counts': x}, S, learning_rate=0.02)
    path = str(tmp_path / "custom.ckpt")
    m.save_checkpoint(path)
    again = spmf_b200.PoissonFactorization.load(path, device=DEV)
    probe = torch.rand(5, D, device=DEV)
    assert torch.equal(again.encoder_function(probe), m.encoder_function(probe))
    l1 = m.elbo_step({'counts': x}, S, learning_rate=0.02)
    l2 = again.elbo_step({'counts': x}, S, learning_rate=0.02)
    torch.cuda.synchronize()
    assert abs(float(l1) - float(l2)) <= 1e-6 * abs(float(l1))
    _assert_same_run(m._engine_for(S), again._engine_for(S), 4)


def test_save_file_loads_as_before_and_mismatches_raise(tmp_path):
    import spmf_b200
    D, K, S = 40, 4, 4
    x = make_counts(64, D, seed=6)
    m = _model(False, D, K)
    m.compute_scales(lambda: [{'counts': x}])
    for _ in range(3):
        m.elbo_step({'counts': x}, S, learning_rate=0.02)
    plain = str(tmp_path / "model.pkl")
    m.save(plain)
    st = _read(plain)
    assert 'training' not in st and set(st) == {'surrogate_vars', 'eta_i', 'xi_u_global', 'hyper'}
    old = spmf_b200.PoissonFactorization.load(plain, device=DEV)
    eng = old._engine_for(S)
    assert eng.opt_step == 0 and eng.rng_step == 0
    assert float(eng.adam_m.abs().max()) == 0.0 and float(eng.adam_v.abs().max()) == 0.0
    for got, want in zip(old.surrogate_vars, m.surrogate_vars):
        assert torch.equal(got, want)
    ck = str(tmp_path / "model.ckpt")
    m.save_checkpoint(ck)
    full = _read(ck)
    assert torch.equal(full['eta_i'], st['eta_i'])
    assert full['xi_u_global'] == st['xi_u_global'] and pickle.dumps(full['hyper']) == pickle.dumps(st['hyper'])
    assert all(torch.equal(a, b) for a, b in zip(full['surrogate_vars'], st['surrogate_vars']))
    with pytest.raises(spmf_b200.SpmfError):
        spmf_b200.BernoulliFactorization.load(ck, device=DEV)
    with pytest.raises(spmf_b200.SpmfError):
        _model(False, D, K + 1).fit(lambda: [{'counts': x}], num_steps=1, checkpoint_path=ck, resume=True)
    with pytest.raises(spmf_b200.SpmfError):
        _model(False, D, K).fit(lambda: [{'counts': x}], num_steps=1, checkpoint_path=plain, resume=True)


def _cli_run(tmp_path, csv_path, epochs, ckpt):
    import importlib.util
    spec = importlib.util.spec_from_file_location("factorize_csv", os.path.join(ROOT, "bin", "factorize_csv.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    cli.main(["-f", csv_path, "-e", str(epochs), "-d", "2", "-b", "32", "-rn", "--sample-size", "4",
              "--checkpoint", ckpt])
    return _read(ckpt)['training']['fit']['losses']


def test_cli_resumes_from_its_checkpoint(tmp_path):
    import csv
    rng = np.random.default_rng(0)
    x = rng.poisson(1.5, size=(64, 12))
    x[:, 0] = np.maximum(x[:, 0], 1)
    x[0, :] = np.maximum(x[0, :], 1)
    p = str(tmp_path / "counts.csv")
    with open(p, "w") as f:
        csv.writer(f).writerows(x.tolist())
    one = _cli_run(tmp_path, p, 4, str(tmp_path / "one.ckpt"))
    _cli_run(tmp_path, p, 2, str(tmp_path / "two.ckpt"))
    two = _cli_run(tmp_path, p, 4, str(tmp_path / "two.ckpt"))
    assert len(one) == len(two)
    np.testing.assert_allclose(two, one, rtol=1e-6)


def _torchrun(port, extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                           "--master-addr", "127.0.0.1", "--master-port", str(port),
                           os.path.join(ROOT, "tests", "dp_checkpoint_check.py")],
                          capture_output=True, text=True, timeout=600, env=env)


def test_data_parallel_checkpoint_two_gpus(tmp_path):
    """2-rank checkpoint with the peer-memory exchange and with the NCCL fallback; one GPU resumes it (skipped
    with < 2 GPUs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    p2p, nccl = str(tmp_path / "p2p.ckpt"), str(tmp_path / "nccl.ckpt")
    out = _torchrun(29523, {"DP_CKPT_PATH": p2p})
    assert "DP_CKPT_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    out = _torchrun(29524, {"DP_CKPT_PATH": nccl, "SPMF_P2P": "0"})
    assert "DP_CKPT_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    a, b = _read(p2p)['training'], _read(nccl)['training']
    assert a['counters'] == b['counters']
    for k in ('adam_m', 'adam_v'):                  # (entries whose gradient sums to ~0 get a small absolute floor)
        assert torch.allclose(a[k], b[k], rtol=1e-3, atol=1e-5 * float(b[k].abs().max())), k
    # one GPU takes over the 2-rank run
    import spmf_b200
    m = spmf_b200.PoissonFactorization.load(p2p, device=DEV)
    sys.path.insert(0, ROOT)
    from tests.dp_checkpoint_check import problem
    D, K, S, x = problem()
    loss = m.elbo_step({'counts': spmf_b200.CsrShard.from_dense(torch.from_numpy(x), DEV).batch(0, x.shape[0])}, S,
                       learning_rate=0.02)
    assert np.isfinite(float(loss)) and m._engine_for(S).opt_step == 4
