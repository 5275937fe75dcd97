"""Time LOO-PIT (PoissonFactorization.loo_pit) at the C4 shape with CUDA events.

    python scripts/loo_pit_time.py [--rows 8192] [--D 20000] [--K 32] [--S 1000] [--bins 20] [--iters 5] [--out FILE]

Data: scRNA-shaped CSR counts (rows x D, ~5 % density, the C4 generator of bench.py); the model's surrogate at its
initial values after compute_scales.  One batch of loo_pit's default size (the (B, D, 2) fp64 accumulator within
1 GiB: 3,355 rows at D = 20,000) is timed piece by piece, after a warm-up call:
  * weights: the per-row log-likelihoods of every draw chunk (_loo_row_ll) and spmf_psis_loo_lw;
  * accum: one spmf_loo_pit_accum chunk of LOO_DRAW_CHUNK draws alone (operands already in place), median over
    `iters` CUDA-event windows; entries/s = B * D * draws / time;
  * hist: spmf_loo_pit_hist alone, median over `iters`;
  * call: the whole public loo_pit() over all rows (host clock around a device synchronise).
Prints the GPU name and power limit, then one JSON line.
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
    ap.add_argument("--S", type=int, default=1000)
    ap.add_argument("--bins", type=int, default=20)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("loo_pit_time.py measures on a CUDA device; none is visible")
    import spmf_b200
    from spmf_b200 import _abi
    from spmf_b200.data import _ptr, synth_scrna_csr_device
    from spmf_b200.poisson import LOO_DRAW_CHUNK, LOO_PIT_ACC_BYTES

    dev = torch.device("cuda:0")
    print("gpu:", gpu_info(), flush=True)
    N, D, K, S, J, seed = args.rows, args.D, args.K, args.S, args.bins, 12345
    shard = synth_scrna_csr_device(N, D, 0.05, seed=1, device=dev, gene_seed=1237)
    m = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, device=dev, u_tau_scale=1e-3)
    m.compute_scales(shard)
    B = min(N, LOO_PIT_ACC_BYTES // (16 * D))
    b = shard.batch(0, B)
    st = lambda: torch.cuda.current_stream().cuda_stream
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(fn, iters):
        out = []
        for _ in range(iters):
            a, z = ev(), ev()
            a.record()
            fn()
            z.record()
            z.synchronize()
            out.append(a.elapsed_time(z))
        return sorted(out)[len(out) // 2]

    m._loo_pit_batch(b, S, seed, None)                           # warm-up: engines, workspaces, modules
    torch.cuda.synchronize()
    lw = torch.empty(B, S, dtype=torch.float64, device=dev)
    elpd, lppd = (torch.empty(B, dtype=torch.float64, device=dev) for _ in range(2))
    khat = torch.empty(B, dtype=torch.float32, device=dev)

    def weights():
        ll = m._loo_row_ll(b, S, seed, None)
        _abi.call("spmf_psis_loo_lw", _ptr(ll), S, B, S, _ptr(elpd), _ptr(lppd), _ptr(khat), _ptr(lw), S, st())
    weights_ms = timed(weights, 1)
    # one chunk of the accumulation: the first chunk's operands, batch densified and encoded (as _loo_pit_batch)
    nc = min(LOO_DRAW_CHUNK, S)
    eng = m._engine_for(nc)
    from spmf_b200.engine import AdviEngine
    eng.fill_noise(step=seed, which=AdviEngine.NOISE_NORMAL, advance=False)
    eng.draw_operands()
    eng.ensure_rows(B)
    xd = eng.dense_scratch(B)
    ws = eng.ws
    eng.dense_scatter(b, xd)
    _abi.call("spmf_csr_encode", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum), eng.inv_xi,
              int(m.scale_rows), B, D, K, nc, _ptr(ws.Ap), _ptr(ws.z), st())
    acc = torch.zeros(B, D, 2, dtype=torch.float64, device=dev)
    inv = torch.zeros(B, D, dtype=torch.int32, device=dev)
    accum = lambda: _abi.call("spmf_loo_pit_accum", _ptr(xd), B, D, K, nc, m.link, _ptr(ws.EV), _ptr(ws.PH),
                              _ptr(ws.z), _ptr(lw), S, _ptr(acc), _ptr(inv), None, st())
    accum_ms = timed(accum, args.iters)
    acc, inv, _, _ = m._loo_pit_batch(b, S, seed, None)
    col_hist = torch.zeros(D, J, dtype=torch.float64, device=dev)
    col_n = torch.zeros(D, dtype=torch.int64, device=dev)
    col_pit = torch.zeros(D, dtype=torch.float64, device=dev)
    scratch = torch.empty(_abi._lib.spmf_loo_pit_hist_scratch_doubles(B, D, J), dtype=torch.float64, device=dev)
    hist = lambda: _abi.call("spmf_loo_pit_hist", _ptr(acc), _ptr(inv), B, D, J, _ptr(col_hist), _ptr(col_n),
                             _ptr(col_pit), _ptr(scratch), st())
    hist_ms = timed(hist, args.iters)
    t0 = time.perf_counter()
    res = m.loo_pit(shard, sample_size=S, bins=J)
    torch.cuda.synchronize()
    call_s = time.perf_counter() - t0
    rec = dict(shape=f"{N}x{D}", batch_rows=B, K=K, S=S, bins=J, nnz_batch=int(b.nnz),
               weights_ms=round(weights_ms, 1), accum_chunk_ms=round(accum_ms, 2), accum_chunk_draws=nc,
               accum_entries_per_s=float(f"{B * D * nc / (accum_ms * 1e-3):.3g}"), hist_ms=round(hist_ms, 2),
               call_s=round(call_s, 2), ecdf_dev=round(res['ecdf_dev'], 5), n_invalid=res['n_invalid'],
               n_rows_excluded=res['n_rows_excluded'], gpu=gpu_info())
    print(json.dumps(rec), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
