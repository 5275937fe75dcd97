"""Latent dimensions above 128 on the GPU: the gather kernels with 256- and 512-wide records, the
parameter-side kernels that walk the latent space in 128-wide chunks, the dense links and the exact guard.
Same oracle, harnesses and tolerances as the K <= 128 tests (1e-4; 5e-4 for the InverseGamma family).
The tensor-core hybrid path stops at K = 128: a wider model runs the gather step whatever hot_density says."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.test_gpu_graphs import test_graph_replay_is_bit_identical_to_eager as _graph_case
from tests.test_gpu_links import test_bernoulli_step_matches_oracle as _bernoulli_case
from tests.test_gpu_links import test_guard_training_step_matches_guarded_autograd as _guard_case
from tests.test_gpu_links import test_log_transform_step_matches_oracle as _log_case
from tests.test_gpu_parity import _run_case
from tests.test_gpu_scale import test_adam_trajectory_matches_oracle as _adam_case
from tests.util import make_counts, make_oracle, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.mark.parametrize("D,K,B,S,kind", [
    (60, 129, 40, 2, "noise"),      # just above the old limit: KP = 256, SV = 2
    (80, 256, 48, 4, "sparse"),     # SV = 2: two draw groups
    (50, 256, 33, 1, "noise"),
    (40, 300, 24, 3, "noise"),      # KP = 512, padded latent dims
    (64, 512, 32, 2, "sparse"),     # KP = 512, SV = 1
])
def test_step_matches_oracle(D, K, B, S, kind):
    eng = _run_case(D, K, B, S, kind)
    assert eng.hot_cols == 0 and eng.ws.KP * eng.ws.SV <= 512


def test_surface_matches_oracle_at_k256():
    import spmf_b200
    dev = torch.device("cuda:0")
    D, K, B, S = 70, 256, 48, 4
    x = make_counts(B, D, seed=6)
    oracle = make_oracle(D, K, 400, x)
    model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(400 * D), device=dev)
    model.compute_scales(lambda: [{'counts': x[:24]}, {'counts': x[24:]}])
    data = {'counts': torch.tensor(x, dtype=torch.float64)}
    th = model.surrogate_distribution.sample(S, seed=12345)
    th64 = {k: v.cpu().double() for k, v in th.items()}
    z = model.encode(x, th['u'], th['s']).cpu().double().numpy()
    assert z.shape == (S, B, K) and rel_err(z, oracle.encode(data['counts'], th64['u'], th64['s']).numpy()) < 1e-5
    got = model.unormalized_log_prob_parts({'counts': x}, **th)
    ref = oracle.unormalized_log_prob_parts(data, **th64)
    assert set(got) == set(ref)
    for k in ref:
        r = ref[k].numpy()
        assert np.abs(got[k].cpu().numpy() - r).max() <= TOL * max(np.abs(r).max(), 1.0), k
    ll = oracle.log_likelihood_components(data=data, **{k: th64[k] for k in 'suvw'})['log_likelihood'].sum(-1).numpy()
    np.testing.assert_allclose(model.row_log_likelihood({'counts': x}, **th).cpu().numpy(), ll, rtol=1e-5, atol=1e-3)


def test_log_transform_step_at_k256():
    _log_case(48, 256, 40, 4, "noise")


def test_bernoulli_step_at_k256():
    _bernoulli_case(40, 256, 48, 2, False)


def test_exact_guard_at_k256():
    _guard_case(48, 256, 40, 4, "noise", False)


def test_hot_columns_are_ignored_above_the_tile_limit():
    """hot_density > 0 at K = 256 gives the very same launches as hot_density = 0: identical loss parts; the
    gradients agree up to the run-to-run re-association of the column pass's fp32 atomics."""
    import spmf_b200
    dev = torch.device("cuda:0")
    D, K, B, S = 160, 256, 192, 4
    x = make_counts(B, D, seed=4, kind="noise", rate=2.0)        # every column populated in most rows
    out = []
    for hd in (0.05, 0.0):
        m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=dev, seed=7,
                                           hot_density=hd)
        m.compute_scales(lambda: [{'counts': x}])
        assert m.hot_cols == 0 and m.col_rank is None
        eng = m._engine_for(S)
        assert eng.hot_cols == 0 and not eng.hybrid_ok
        eng.fill_noise(step=0)
        p = eng.loss_and_grad(spmf_b200.as_device_batch(x, dev), fresh_noise=False)
        torch.cuda.synchronize()
        out.append((p.clone(), eng.grads.clone()))
    assert torch.equal(out[0][0], out[1][0])
    assert rel_err(out[0][1].cpu().numpy(), out[1][1].cpu().numpy()) < 1e-6


def test_graph_replay_at_k256():
    _graph_case(96, 256, 4, "sparse", False)


def test_u8_host_stream_matches_resident_at_k256():
    """Training steps fed from a HostCsr(compact="u8") stream follow the resident shard step for step."""
    import spmf_b200
    from spmf_b200.data import CsrShard, HostCsr, prefetch_to_device
    dev = torch.device("cuda:0")
    D, K, S, B = 120, 256, 4, 64
    x = make_counts(4 * B, D, seed=12, kind="sparse")
    x[5, 7] = 300.0                                   # through the overflow list of the 2-byte format
    sh = CsrShard.from_dense(x, dev)
    host = HostCsr.from_shard(sh, compact="u8")
    runs = []
    for stream in (False, True):
        m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1e-3, device=dev, seed=5)
        m.compute_scales(sh)
        batches = prefetch_to_device(host.iter_batches(B), dev) if stream else sh.iter_batches(B)
        losses = [m.elbo_step({'counts': b}, S, learning_rate=0.02) for b in batches]
        torch.cuda.synchronize()
        runs.append((torch.stack(losses).cpu(), m._engine_for(S).params.clone()))
    assert len(runs[0][0]) == 4
    assert rel_err(runs[1][0].numpy(), runs[0][0].numpy()) < 1e-6
    assert float((runs[1][1] - runs[0][1]).abs().max()) <= 1e-4 * 0.02 * 4


def test_adam_trajectory_at_k256():
    _adam_case(80, 256, 400, "noise", False)


def test_latent_dim_above_max_raises():
    import spmf_b200
    from spmf_b200._abi import SpmfError
    with pytest.raises(SpmfError):
        m = spmf_b200.PoissonFactorization(latent_dim=513, feature_dim=20, device=torch.device("cuda:0"))
        m._engine_for(4)


def test_data_parallel_two_gpus_at_k256():
    """Row-sharded step on 2 GPUs == single-GPU step at K = 256 (skipped with < 2 GPUs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29519",
                          os.path.join(root, "tests", "dp_wide_check.py")], capture_output=True, text=True, timeout=600)
    assert "DP_WIDE_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
