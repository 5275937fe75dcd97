"""Time the posterior predictive check at the C4 shape with CUDA events.

    python scripts/ppc_time.py [--rows 8192] [--D 20000] [--K 32] [--S 4 32] [--iters 10] [--out FILE]

Data: one batch of scRNA-shaped CSR counts (rows x D, ~5 % density, the C4 generator of bench.py).  Draws: S
explicit draws of the "null" model whose rate is the column mean, lambda_bd = mean_b x_bd (u = 0, so the latent
contraction is still evaluated but adds 0): the rates then span the genes' range of means.  For each S, after two
warm-up calls:
  * pass: the per-batch device work of the check (densify, encode, the fused spmf_ppc_rows kernel and its
    fixed-order reduction, the observed statistics), median over `iters` CUDA-event windows;
  * call: the whole public posterior_predictive_check on the batch (host clock around a device synchronise),
    which adds the operand packing, the assembly of the result and the p-values.
Prints the GPU name and power limit, then one JSON line per S with the times and entries/s = S*rows*D / time.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                      text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        out = torch.cuda.get_device_name(0) + ", power limit unknown"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--D", type=int, default=20000)
    ap.add_argument("--K", type=int, default=32)
    ap.add_argument("--S", type=int, nargs="+", default=[4, 32])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppc_time.py measures on a CUDA device; none is visible")
    import spmf_b200
    from spmf_b200.data import synth_scrna_csr_device

    dev = torch.device("cuda:0")
    print("gpu:", gpu_info(), flush=True)
    B, D, K = args.rows, args.D, args.K
    shard = synth_scrna_csr_device(B, D, 0.05, seed=1, device=dev, gene_seed=1237)
    m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=dev, u_tau_scale=1e-3)
    m.compute_scales(shard)
    colsum, _ = shard.column_stats()
    colmean = (colsum / B).float().cpu()
    batch = shard.batch(0, B)
    lines = []
    for S in args.S:
        eta = m.eta_i.reshape(-1).float()
        # phi = eta * s1/(s0+s1) * w with s = 1: w = 2 * colmean / eta gives rate = colmean
        draws = dict(u=torch.zeros(S, D, K), v=torch.rand(S, K, D), s=torch.ones(S, 2, D),
                     w=(2 * colmean / eta).expand(S, 1, D).clone())
        eng = m._ppc_engine(draws, S, 0)
        acc = m._ppc_acc(S)
        obs_col = [torch.zeros(D, dtype=torch.float64, device=dev), torch.zeros(D, dtype=torch.float64, device=dev),
                   torch.zeros(D, dtype=torch.int32, device=dev)]
        ot = torch.empty(B, dtype=torch.float64, device=dev)
        on = torch.empty(B, dtype=torch.int32, device=dev)

        def one_pass():
            m._ppc_pass(eng, batch, 12345, 0, acc)
            spmf_b200._abi.call("spmf_ppc_observed", batch.rowptr.data_ptr(), batch.cols.data_ptr(),
                                batch.vals.data_ptr(), B, D, ot.data_ptr(), on.data_ptr(),
                                *(t.data_ptr() for t in obs_col), torch.cuda.current_stream().cuda_stream)

        for _ in range(2):
            one_pass()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            one_pass()
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        ms.sort()
        for _ in range(2):
            m.posterior_predictive_check(shard, batch_size=B, **draws)
        torch.cuda.synchronize()
        call_ms = []
        for _ in range(max(3, args.iters // 3)):
            t0 = time.perf_counter()
            res = m.posterior_predictive_check(shard, batch_size=B, **draws)
            torch.cuda.synchronize()
            call_ms.append((time.perf_counter() - t0) * 1e3)
        call_ms.sort()
        entries = S * B * D
        rec = dict(shape=f"{B}x{D}", K=K, S=S, nnz=int(batch.nnz), pass_ms_median=round(ms[len(ms) // 2], 3),
                   pass_ms_min=round(ms[0], 3), pass_ms_max=round(ms[-1], 3),
                   call_ms_median=round(call_ms[len(call_ms) // 2], 3),
                   entries_per_s=float(f"{entries / (ms[len(ms) // 2] * 1e-3):.4g}"),
                   invalid=int(res[3].sum()), max_replicate=int(res[1]['max'].max()), gpu=gpu_info())
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
