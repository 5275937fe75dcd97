"""Data-parallel parity at a wide latent space (K = 256): run under torchrun with N >= 2 ranks.

Every rank evaluates one ADVI step on its row shard (identical Philox noise) and the exchange sums the
gradients; rank 0 compares them with a single-rank step on the whole batch.  Prints DP_WIDE_OK on success.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
      --master-port 29519 tests/dp_wide_check.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import spmf_b200
    from spmf_b200.engine import AdviEngine
    from spmf_b200.parallel import shard_rows
    from tests.util import make_counts

    D, K, S, B = 300, 256, 4, 512
    x = make_counts(B, D, seed=21, kind="sparse")            # same matrix on every rank
    lo, hi = shard_rows(B, rank, world)
    model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(B * D),
                                           device=dev, seed=99)
    shard = spmf_b200.CsrShard.from_dense(x[lo:hi], dev)
    model.compute_scales(shard)
    eng = model._engine_for(S)
    assert eng.world_size == world and eng.hot_cols == 0
    p_before = eng.params.clone()
    loss = model.elbo_step({'counts': shard.batch(0, hi - lo)}, S, learning_rate=None)
    grads = eng.grads.clone()
    torch.cuda.synchronize()
    ref = grads.clone()
    dist.broadcast(ref, src=0)
    ok = bool(torch.equal(ref, grads))                       # replicas hold identical gradients
    if rank == 0:
        single = AdviEngine(D, K, S, dev, model.u_tau_scale, model.s_tau_scale, model.symmetry_breaking_decay,
                            True, 1.0, 1.0, world_size=1, seed=99)
        single.params.copy_(p_before)
        single.eta.copy_(eng.eta)
        single.inv_xi = eng.inv_xi
        single.rng_step = 0
        parts = single.loss_and_grad(spmf_b200.CsrShard.from_dense(x, dev).batch(0, B))
        single.clear_comm_slack()
        torch.cuda.synchronize()
        l1, l2 = float(single.loss_value(parts).item()), float(loss.item())
        e_loss = abs(l1 - l2) / abs(l1)
        g1, g2 = single.grads.cpu().double().numpy(), grads.cpu().double().numpy()
        L = eng.layout
        e_grad = 0.0
        for name, v in L.views(torch.arange(L.n_params)).items():
            idx = v.reshape(-1).numpy()
            e_grad = max(e_grad, np.abs(g1[idx] - g2[idx]).max() / (np.abs(g1[idx]).max() + 1e-300))
        print(f"dp_wide_check world={world} K={K}: loss single={l1:.6f} dp={l2:.6f} rel={e_loss:.2e}; "
              f"worst grad rel={e_grad:.2e}")
        ok = ok and e_loss < 1e-6 and e_grad < 5e-5
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if not bool(flag.item()):
        sys.exit(1)
    if rank == 0:
        print("DP_WIDE_OK")


if __name__ == "__main__":
    main()
