"""Data-parallel checkpoint on real GPUs: run under torchrun with N >= 2 ranks; DP_CKPT_PATH names the file.

Every rank takes 3 Adam steps on its row shard and calls save_checkpoint (rank 0 writes).  With the peer-memory
exchange a rank holds the Adam moments of its own slice of the data block only: the file must carry each rank's
slice bit for bit.  Fresh models on every rank then load the file and take 3 more steps: replicas stay
bit-identical, and the parameters match an uninterrupted 6-step run within the Adam bars of dp_check.py.
Prints DP_CKPT_OK on success.

  DP_CKPT_PATH=/tmp/dp.ckpt python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 \
      --master-addr 127.0.0.1 --master-port 29523 tests/dp_checkpoint_check.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LR, CLIP = 0.02, 2.5


def problem():
    """(D, K, S, counts): the same matrix on every rank."""
    from tests.util import make_counts
    D, K, S, B = 400, 32, 4, 1024
    return D, K, S, make_counts(B, D, seed=21, kind="sparse")


def main():
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import dill
    import spmf_b200
    from spmf_b200 import _abi
    from spmf_b200.parallel import exchange_kind, shard_rows

    path = os.environ["DP_CKPT_PATH"]
    D, K, S, x = problem()
    B = x.shape[0]
    lo, hi = shard_rows(B, rank, world)
    shard = spmf_b200.CsrShard.from_dense(torch.from_numpy(x[lo:hi]), dev)
    batch = {'counts': shard.batch(0, hi - lo)}

    def make():
        m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(B * D),
                                           device=dev, seed=99)
        m.compute_scales(shard)                              # all-reduces the column statistics
        return m

    def steps(m, n):
        for _ in range(n):
            m.elbo_step(batch, S, learning_rate=LR, clip_value=CLIP)
        torch.cuda.synchronize()

    ref = make()                                             # the uninterrupted run (all models stay alive)
    p0 = ref._engine_for(S).params.clone()
    steps(ref, 6)
    a = make()
    steps(a, 3)
    a.save_checkpoint(path)
    with open(path, "rb") as f:
        tr = dill.load(f)['training']
    eng = a._engine_for(S)
    L = eng.layout
    kind = exchange_kind(eng)
    own = _abi.p2p_owned_range(L.comm_off, world, rank) if kind == "p2p-kernel" else (0, L.n_params)
    ok = True
    for name in ("adam_m", "adam_v"):
        mine = getattr(eng, name).cpu()
        ok = ok and torch.equal(tr[name][own[0]:own[1]], mine[own[0]:own[1]])       # this rank's slice, bit for bit
        ok = ok and torch.equal(tr[name][L.n_data_block:], mine[L.n_data_block:])  # the replicated tail
    ok = ok and torch.equal(tr['params'], eng.params.cpu()) and tr['counters'][S] == (3, 3)
    if rank == 0:
        print(f"dp_ckpt world={world}: exchange = {kind}, owned slice of rank 0 = {own}, file moments ok = {ok}")

    b = spmf_b200.PoissonFactorization.load(path, device=dev)
    steps(b, 3)
    eb = b._engine_for(S)
    p_b = eb.params.clone()
    r = p_b.clone()
    dist.broadcast(r, src=0)
    ok = ok and torch.equal(r, p_b) and (eb.opt_step, eb.rng_step) == (6, 6)
    upd_ref = (ref._engine_for(S).params - p0).double()
    upd_b = (p_b - p0).double()
    mask = torch.ones(L.n_params, dtype=torch.bool, device=dev)
    mask[L.comm_off:L.comm_off + L.comm_slack] = False      # scalar slack is not a parameter
    diff = (upd_ref - upd_b)[mask].abs()
    frac_off = float((diff > 1e-2 * LR).double().mean())
    e_adam = float(diff.median() / upd_ref[mask].abs().median())
    if rank == 0:
        print(f"dp_ckpt world={world}: 3 + 3 steps through the checkpoint vs 6 uninterrupted: median update "
              f"rel={e_adam:.2e}, entries off by >1% of a step: {frac_off:.2e}")
    ok = ok and e_adam < 1e-4 and frac_off < 1e-3
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if not bool(flag.item()):
        sys.exit(1)
    if rank == 0:
        print("DP_CKPT_OK")


if __name__ == "__main__":
    main()
