"""Time PSIS leave-one-out (PoissonFactorization.loo) at the C4 shape with CUDA events.

    python scripts/loo_time.py [--rows 8192] [--D 20000] [--K 32] [--S 1000 4096] [--iters 10] [--out FILE]

Data: one batch of scRNA-shaped CSR counts (rows x D, ~5 % density, the C4 generator of bench.py); the model's
surrogate at its initial values after compute_scales.  For each S, after a warm-up call:
  * regen: the per-chunk draw regeneration (Normal noise + operand tables, LOO_DRAW_CHUNK draws at a time), summed
    over the chunks of one batch;
  * rows: the row passes of those chunks (spmf_csr_rows and the copy into the [B][S] fp64 buffer), summed;
  * kernel: spmf_psis_loo alone on that buffer, median over `iters` CUDA-event windows;
  * call: the whole public loo() on the batch (host clock around a device synchronise), median of 3.
Prints the GPU name and power limit, then one JSON line per S.
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
    ap.add_argument("--S", type=int, nargs="+", default=[1000, 4096])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("loo_time.py measures on a CUDA device; none is visible")
    import spmf_b200
    from spmf_b200 import _abi
    from spmf_b200.data import synth_scrna_csr_device
    from spmf_b200.engine import AdviEngine
    from spmf_b200.poisson import LOO_DRAW_CHUNK

    dev = torch.device("cuda:0")
    print("gpu:", gpu_info(), flush=True)
    B, D, K, seed = args.rows, args.D, args.K, 12345
    shard = synth_scrna_csr_device(B, D, 0.05, seed=1, device=dev, gene_seed=1237)
    m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=dev, u_tau_scale=1e-3)
    m.compute_scales(shard)
    batch = shard.batch(0, B)
    st = lambda: torch.cuda.current_stream().cuda_stream
    ev = lambda: torch.cuda.Event(enable_timing=True)
    lines = []
    for S in args.S:
        m.loo(shard, sample_size=S, batch_size=B)                   # warm-up: engines, workspaces, modules
        torch.cuda.synchronize()
        chunks = [(c0, min(LOO_DRAW_CHUNK, S - c0)) for c0 in range(0, S, LOO_DRAW_CHUNK)]
        ll = torch.empty(B, S, dtype=torch.float64, device=dev)
        marks = []
        for c, (c0, nc) in enumerate(chunks):
            eng = m._engine_for(nc)
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            eng.fill_noise(step=seed + c, which=AdviEngine.NOISE_NORMAL, advance=False)
            eng.draw_operands()
            e1.record()
            ll[:, c0:c0 + nc].copy_(m._row_ll(eng, batch).t())
            e2.record()
            marks.append((e0, e1, e2))
        torch.cuda.synchronize()
        regen_ms = sum(a.elapsed_time(b) for a, b, _ in marks)
        rows_ms = sum(b.elapsed_time(c) for _, b, c in marks)
        elpd = torch.empty(B, dtype=torch.float64, device=dev)
        lppd = torch.empty(B, dtype=torch.float64, device=dev)
        khat = torch.empty(B, dtype=torch.float32, device=dev)
        run = lambda: _abi.call("spmf_psis_loo", ll.data_ptr(), S, B, S, elpd.data_ptr(), lppd.data_ptr(),
                                khat.data_ptr(), st())
        run()
        kms = []
        for _ in range(args.iters):
            a, b = ev(), ev()
            a.record()
            run()
            b.record()
            b.synchronize()
            kms.append(a.elapsed_time(b))
        kms.sort()
        call_ms = []
        for _ in range(3):
            t0 = time.perf_counter()
            res = m.loo(shard, sample_size=S, batch_size=B)
            torch.cuda.synchronize()
            call_ms.append((time.perf_counter() - t0) * 1e3)
        call_ms.sort()
        rec = dict(shape=f"{B}x{D}", K=K, S=S, nnz=int(batch.nnz), chunks=len(chunks),
                   regen_ms=round(regen_ms, 3), rows_ms=round(rows_ms, 3),
                   kernel_ms_median=round(kms[len(kms) // 2], 3), kernel_ms_min=round(kms[0], 3),
                   kernel_ms_max=round(kms[-1], 3), call_ms_median=round(call_ms[1], 1),
                   khat_threshold=round(res['khat_threshold'], 4), frac_khat_above=round(res['n_khat_above'] / B, 4),
                   n_nonfinite=res['n_nonfinite'], gpu=gpu_info())
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
