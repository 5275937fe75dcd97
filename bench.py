#!/usr/bin/env python
"""Benchmark of the ADVI step (ELBO + gradient + all-reduce + Adam) -- BASELINE.json's metric:
nonzeros*K per second, whole job over N GPUs, plus roofline and CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c3|c1] [--impl ours|reference]
                  [--dump-outputs DIR]

Workload at the default (`c4`, BASELINE.json configs[3], the configuration the north-star target is
quoted on): scRNA-seq shaped CSR counts, D=20,000 genes, ~5 % density, K=32, S=4 draws, 8,192
rows per GPU per step, each GPU holding a 131,072-row shard (16 batches; ~2 GB of CSR+CSC, far
larger than L2, cycled so no step sees a cache-warm batch).  Weak scaling: per-GPU work is fixed.

A "step" = fresh Philox noise -> reparameterised draws -> row pass -> column pass -> backward to
the 24 variational tensors -> one NCCL all-reduce (N>1) -> Adam.  `value` has inputs resident in
HBM; `e2e` streams every step's CSR minibatch from pinned host memory through the public API
(`PoissonFactorization.elbo_step`), builds its row constants and CSC copy on the device, and reads
the loss back.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: D, K, S, rows/GPU/step, batches/GPU, kind
    "c4": dict(D=20000, K=32, S=4, rows=8192, nbatch=16, kind="scrna", density=0.05,
               desc="C4 scRNA-shaped CSR N=1e6xD=20000 ~5% density, K=32, S=4, 8192 rows/GPU/step; weak scaling: each "
                    "GPU holds a 131,072-row shard (16 resident batches) of the 1M-row matrix"),
    "c3": dict(D=2000, K=16, S=4, rows=6250, nbatch=20, kind="linear",
               desc="C3 dense-origin counts N=1e6xD=2000, K=16, S=4, 6250 rows/GPU/step (50000/8)"),
    "c2": dict(D=1000, K=8, S=4, rows=5000, nbatch=20, kind="linear",
               desc="C2 linear-structure counts N=1e5xD=1000, K=8, S=4, 5000 rows/step"),
    "c1": dict(D=100, K=2, S=4, rows=1000, nbatch=10, kind="noise",
               desc="C1 Poisson(1) noise N=1e4xD=100, K=2, S=4, 1000 rows/step"),
}
# rows of the workload the float64 CPU port is timed on (C4: the reference formulation materialises ~20
# (S,B,D) float64 tensors, 1 GB each at 1,536 rows; 8,192 rows would need ~100 GB)
CPU_SAMPLE_ROWS = {"c4": 1536, "c3": 2000, "c2": 5000, "c1": 1000}
DUMP_BYTES = 64 * 10 ** 6           # --dump-outputs: all files together stay below this


def step_outputs(eng, loss):
    """What a caller of `elbo_step` holds after a step, as host float32 / float64 arrays: the returned loss,
    the (S,16) energy terms per draw, and the 24 variational tensors with the gradient the step applied to
    them (reference shapes, '/' in a name becomes '.')."""
    out = {"loss": loss.detach().double().cpu().numpy(), "parts": eng.ws.parts.view(eng.S, -1).cpu().numpy()}
    for prefix, flat in (("param", eng.params), ("grad", eng.grads)):
        for k, v in eng.layout.views(flat).items():
            out[prefix + "." + k.replace("/", ".")] = v.detach().float().cpu().numpy()
    return out


def dump_outputs(out_dir, arrays, seed=0):
    """Writes every array as <out_dir>/<name>.npy.  If together they exceed DUMP_BYTES, every array keeps the
    same share of its elements, flattened, at positions drawn by a generator seeded with `seed` (same shapes:
    same positions, so two runs compare element for element)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    share = min(1.0, 0.99 * (DUMP_BYTES - 256 * len(arrays)) / max(total, 1))
    for name, a in arrays.items():
        if share < 1.0:
            idx = np.sort(np.random.default_rng(seed).choice(a.size, max(1, int(a.size * share)), replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region.  Uses NVML in-process (a few
    microseconds per query); falls back to spawning nvidia-smi, which is heavy enough to perturb a
    50 ms timed region, only if NVML is unavailable."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mx, self.reasons = index, [], 0.0, set()
        self._stop_evt = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        self.mx = max(self.mx, float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for name, bit in self.BITS.items():
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                              "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
        r = [c.strip() for c in out.strip().split(",")]
        self.sm.append(float(r[0]))
        self.mx = max(self.mx, float(r[1]))
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[2:6]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self._stop_evt.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.02 if self.nvml else 0.25)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx or None,
                "reasons": sorted(self.reasons), "samples": len(sm),
                "source": "nvml" if self.nvml else "nvidia-smi"}


def make_shard(wl, device, seed):
    import torch
    from spmf_b200.data import CsrShard, synth_linear_dense, synth_noise_dense, synth_scrna_csr_device
    n = wl["rows"] * wl["nbatch"]
    if wl["kind"] == "scrna":
        # one dataset, row-sharded: the gene profile is shared by all ranks, the cells are per rank
        return synth_scrna_csr_device(n, wl["D"], wl["density"], seed=seed, device=device, gene_seed=1234 + 3)
    x = synth_linear_dense(n, wl["D"], seed=seed) if wl["kind"] == "linear" else synth_noise_dense(n, wl["D"], seed=seed)
    x[0, :] = x[0, :].clip(min=1)
    sh = CsrShard.from_dense(torch.from_numpy(x), device)
    sh._dense_host = x                      # dense-origin workload: the e2e leg streams the dense slabs themselves
    return sh


def oracle_step_time(wl, rows, steps, warmup, seed=0):
    """Float64 torch-CPU oracle (reference formulation: dense (S,B,D) rate, autograd backward) on a
    bounded sample of the workload.  Returns (seconds per step, nnz in the sample, cores)."""
    import numpy as np
    import torch
    import oracle.spmf_oracle as _o
    from oracle.spmf_oracle import OraclePoissonFactorization, draw_noise
    _o.FAST_GAMMA_GRAD = True       # native implicit-gradient op, as TF's would be (see oracle header)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    D, K, S = wl["D"], wl["K"], wl["S"]
    rng = np.random.default_rng(seed)
    if wl["kind"] == "scrna":
        g = np.exp(1.5 * rng.standard_normal(D)); c = np.exp(0.5 * rng.standard_normal(rows))
        lo, hi = -30.0, 10.0
        for _ in range(50):
            mid = 0.5 * (lo + hi)
            lo, hi = (mid, hi) if (1 - np.exp(-c[:, None] * g[None, :] * np.exp(mid))).mean() < wl["density"] else (lo, mid)
        x = rng.poisson(c[:, None] * g[None, :] * np.exp(lo)).astype(np.float64)
    elif wl["kind"] == "linear":
        from spmf_b200.data import synth_linear_dense
        x = synth_linear_dense(rows, D, seed=seed).astype(np.float64)
    else:
        x = rng.poisson(1.0, size=(rows, D)).astype(np.float64)
    x[0, :] = np.maximum(x[0, :], 1); x[:, 0] = np.maximum(x[:, 0], 1)
    nnz = int((x > 0).sum())
    m = OraclePoissonFactorization(K, D, u_tau_scale=1.0 / np.sqrt(1e6 * D))
    data = {"counts": torch.tensor(x)}
    m.compute_scales([data])
    params = m.init_params()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        noise = draw_noise(m, params, S, seed=i)
        m.loss_and_grads(params, noise, data)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    times.sort()
    return times[len(times) // 2], nnz, cores


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = CPU_SAMPLE_ROWS[args.workload]
    sec, nnz, cores = oracle_step_time(wl, rows, args.steps, args.warmup)
    val = nnz * wl["K"] / sec
    sample = f"{rows} rows x D={wl['D']} densified ({nnz} nonzeros), S={wl['S']}, float64 torch-CPU oracle port of poisson.py"
    print(json.dumps({
        "impl": "reference", "metric": "advi_elbo_grad_nnzK_per_s", "value": val, "unit": "nonzeros*K/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": wl["desc"], "sample": sample},
        "cpu_baseline": {"value": val, "unit": "nonzeros*K/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "nonzeros*K/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--K", type=int, default=None, help="override the workload's latent dim (C5 sweep)")
    ap.add_argument("--S", type=int, default=None, help="override the number of Monte-Carlo draws")
    ap.add_argument("--hot-density", type=float, default=None,
                    help="column population threshold of the tensor-core hot block (0 = gather kernels only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, energy terms, parameters, gradients; "
                         "last e2e loss) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    wl = dict(WORKLOADS[args.workload])
    if args.K:
        wl["K"] = args.K
        wl["desc"] += f" [K overridden to {args.K}]"
    if args.S:
        wl["S"] = args.S
        wl["desc"] += f" [S overridden to {args.S}]"
    if args.impl == "reference":
        run_reference(args, wl)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import spmf_b200
    from spmf_b200.data import HostCsr

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    D, K, S, B = wl["D"], wl["K"], wl["S"], wl["rows"]
    shard = make_shard(wl, dev, seed=1234 + 3 + 1000 * rank)
    n_total = shard.nrows * world
    model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(n_total * D),
                                           device=dev, seed=1234, hot_density=args.hot_density)
    model.compute_scales(shard)
    batches = list(shard.iter_batches(B))
    eng = model._engine_for(S)
    hybrid = eng.hot_cols > 0 and eng.hybrid_ok
    prep_ms = None
    for bi, b in enumerate(batches):
        if hybrid:
            if bi == 2:                                # time one build of the hybrid form (after warm-up)
                torch.cuda.synchronize()
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
            eng.prepare_batch(b)                       # ranked CSR/CSC + dense bf16 hot block
            if bi == 2:
                p1.record()
                torch.cuda.synchronize()
                prep_ms = p0.elapsed_time(p1)
        else:
            b.ensure_csc()
    eng.ws.ensure_rows(B)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(n, get_batch, lr):
        loss = None
        for i in range(n):
            loss = model.elbo_step({"counts": get_batch(i)}, S, learning_rate=lr, variant=args.variant)
        return loss

    # ------------------------------------------------ device-resident: `value`
    run_steps(args.warmup, lambda i: batches[i % len(batches)], args.lr)
    # every resident batch replays its step as one CUDA graph: capture them all before the timed region
    # (training does this once per batch in its first epoch)
    primed = sum(bool(eng.prime_graph(b, lr=args.lr)) for b in batches)
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    launches0, graphs0 = eng.launches, eng.graph_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("spmf_timed")
    e0.record()
    last_loss = run_steps(args.steps, lambda i: batches[(args.warmup + i) % len(batches)], args.lr)
    e1.record()
    torch.cuda.nvtx.range_pop()
    barrier()
    ms = e0.elapsed_time(e1)
    # copied before the instrumented pass below steps the model further
    outputs = step_outputs(eng, last_loss) if args.dump_outputs and rank == 0 else None
    launches = eng.launches - launches0
    graph_replays = eng.graph_launches - graphs0
    # per-kernel timings for the roofline: a short instrumented pass AFTER the timed region (CUDA events
    # around the dominant kernels on their launching streams; instrumented steps are launched eagerly,
    # the timed region above replays each resident batch's step as one CUDA graph)
    eng.kernel_events = {}
    run_steps(min(args.steps, 8), lambda i: batches[i % len(batches)], args.lr)
    barrier()
    kev, eng.kernel_events = eng.kernel_events, None
    nnz_done = sum(batches[(args.warmup + i) % len(batches)].nnz for i in range(args.steps))
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(nnz_done)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_max, nnz_all = float(t.item()), float(tot.item())
    value = nnz_all * K / (ms_max * 1e-3)
    final_loss = float(eng.loss_value().item())

    # ------------------------------------------------ host-resident: `e2e`
    # Every step's minibatch starts in pinned host memory (compact CSR: uint16 column ids and
    # counts where they fit), is copied H2D, widened, gets its row constants and CSC copy built on
    # the device (prefetched one batch ahead on a copy stream), runs the step through the public
    # API, and its loss is read back D2H -- all inside the timed region.
    from spmf_b200.data import prefetch_to_device
    fmt = os.environ.get("BENCH_HOST_FORMAT", "auto")
    x_host = getattr(shard, "_dense_host", None)
    if fmt in ("auto", "dense") and x_host is not None and hybrid and eng.hot_mode == 2:
        # dense-origin counts (C2 / C3): the uint8 slab itself travels and goes straight to the hybrid form
        from spmf_b200.data import HostDense
        host, fmt = HostDense(x_host), "dense-" + str(HostDense(x_host[:1]).x.dtype).replace("torch.", "")
    else:
        fmt = "u8" if fmt in ("auto", "dense") else fmt
        host = HostCsr.from_shard(shard, compact=fmt if fmt != "u16" else True)
    hbatches = [host.batch(i * B, B) for i in range(len(batches))]

    LOOKAHEAD = 2            # the host blocks on the loss of step i-2: two steps are always enqueued behind it
    loss_bufs = [torch.empty(1, dtype=torch.float64).pin_memory() for _ in range(LOOKAHEAD + 1)]
    losses_read = []

    def run_e2e(n, start):
        # each step's loss is copied D2H asynchronously right behind the step and read by the host LOOKAHEAD
        # steps later, so launches for the next steps are issued while this one runs; every loss is read
        # inside the timed region
        src = (hbatches[(start + i) % len(hbatches)] for i in range(n))
        pending = []
        tlast = time.perf_counter()
        for i, db in enumerate(prefetch_to_device(src, dev, depth=LOOKAHEAD + 1,
                                                  hot=model._hot_spec(eng) if hybrid else None)):
            if os.environ.get("BENCH_DEBUG"):
                tnow = time.perf_counter()
                print(f"e2e iter {i} host dt {1e3 * (tnow - tlast):.2f} ms", file=sys.stderr)
                tlast = tnow
            loss = model.elbo_step({"counts": db}, S, learning_rate=args.lr, variant=args.variant)
            buf = loss_bufs[i % (LOOKAHEAD + 1)]
            buf.copy_(loss.reshape(1), non_blocking=True)             # D2H read of this step's result
            ev = torch.cuda.Event()
            ev.record()
            pending.append((ev, buf))
            if len(pending) > LOOKAHEAD:
                e0, b0 = pending.pop(0)
                e0.synchronize()
                losses_read.append(float(b0[0]))
        for e0, b0 in pending:
            e0.synchronize()
            losses_read.append(float(b0[0]))

    run_e2e(args.warmup, 0)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("spmf_e2e")
    e2.record()
    run_e2e(args.steps, args.warmup)
    e3.record()
    torch.cuda.nvtx.range_pop()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    t2 = torch.tensor([ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = nnz_all * K / (float(t2.item()) * 1e-3)
    h2d = sum(hbatches[(args.warmup + i) % len(hbatches)].nbytes() for i in range(args.steps)) / args.steps
    clk = clocks.stop() if clocks else None
    exchange = None
    if world > 1:
        from spmf_b200.parallel import check_exchange, exchange_kind
        check_exchange(eng)                 # raises if a rank ever gave up waiting for a peer
        exchange = exchange_kind(eng)

    # ------------------------------------------------ roofline of the dominant kernel
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    KP, SV = eng.ws.KP, eng.ws.SV
    C = KP * S                                        # channels per row/column: KP * SV * NQ
    kern = {}
    for name, evs in ((n, e) for n, e in kev.items() if n in ("csr_rows", "csc_cols")):
        dur = [a.elapsed_time(b) for a, b, _, _ in evs]
        nz = [n for _, _, n, _ in evs]
        if name == "csr_rows":      # CSR stream + both operand tables + z, dzr out (fp32)
            byts = [8.0 * n + 8 * (B + 1) + 2 * D * C * 4 + D * S * 4 + 2 * B * C * 4 + B * 16 * S for n in nz]
        else:                       # CSC stream + z, dzr in + EV in + GAp, GEV, Gphi out
            byts = [8.0 * n + 4 * (D + 1) + 2 * B * C * 4 + D * C * 4 + D * S * 4 + 2 * D * C * 4 + D * S * 4 for n in nz]
        kern[name] = {"ms": sum(dur) / len(dur), "bytes": sum(byts) / len(byts),
                      "flop": sum(nz) / len(nz) * (6 if name == "csr_rows" else 6) * K * S}
    if hybrid and "umma_gemm_gradA" in kev:
        # tensor-core side of the column pass: split + tcgen05 GEMM GA'[0:H] += X_hot^T . dzr (3 bf16 terms)
        dur = [a.elapsed_time(b) for a, b, _, _ in kev["umma_gemm_gradA"]]
        Hp, Bp = (eng.hot_cols + 63) // 64 * 64, (B + 63) // 64 * 64
        gemm_ms = sum(dur) / len(dur)
        gemm_info = {"ms": gemm_ms, "bf16_TFLOPs": 2.0 * eng.hot_cols * Bp * C * 3 / (gemm_ms * 1e-3) / 1e12,
                     "shape": f"M={eng.hot_cols} N={C} K={Bp} x3 bf16 terms", "Hp": Hp}
    else:
        gemm_info = None
    step_ms = ms_max / args.steps
    bf16_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1800.0)))   # inside a long step
    # per-launch DRAM traffic of the dominant kernels from the committed `ncu --set full` capture
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        pass
    tile = None
    if hybrid and eng.hot_mode == 2 and "hot_tile" in kev:
        # fused tcgen05 tile kernel over the dense hot block: per (row, hot column, draw) three
        # K-long contractions (rate, dz, GEV) = 6*K flop; each runs as 3 bf16 MMAs on K padded to KK
        dur = [a.elapsed_time(b) for a, b, _, _ in kev["hot_tile"]]
        tms = sum(dur) / len(dur)
        H = int(eng.hot_cols)
        KK = max(KP, 16)
        alg_flop = 6.0 * K * S * B * H
        mma_flop = 2.0 * S * (128 * ((B + 127) // 128)) * (64 * ((H + 63) // 64)) * (3 * KK + 3 * KK + 3 * (KK + 8))
        tile = {"ms": tms, "alg_TFLOPs": alg_flop / (tms * 1e-3) / 1e12, "mma_bf16_TFLOPs": mma_flop / (tms * 1e-3) / 1e12,
                "alg_flop": alg_flop, "elements": float(S) * B * H,
                "alg_bytes": 2.0 * B * H + 4.0 * S * H * (2 * K + 1) + 3 * 4.0 * S * B * K}
    hot_cover = 0.0
    if hybrid:        # share of the nonzeros that the dense hot block covers (the rest runs on the gather kernels)
        cov = sum(int(b.hot.rowmid.sum().item()) for b in batches if b.hot is not None)
        hot_cover = cov / max(sum(b.nnz for b in batches if b.hot is not None), 1)
    dom = max(kern, key=lambda k: kern[k]["ms"])
    if tile is not None and tile["ms"] >= 0.3 * kern["csr_rows"]["ms"]:
        # the tile kernel is the largest single launch of the step; its binding resource is the SM's
        # shared-memory data pipe (MMA operand fetch + element-wise traffic) and MUFU, not DRAM --
        # reported against the tensor roofline the contract names, with the useful (un-split) flops
        nnz_step = nnz_all / world / args.steps
        roofline = {"bound": "tensor", "binding_pipe_ncu": "shared-memory data pipe (MMA operand fetch + LSU), see "
                                                           "profiles/: tensor pipe 26 %, smem/LSU wavefronts 65 %",
                    "kernel": "hot_tile", "achieved": tile["alg_TFLOPs"], "peak": bf16_peak,
                    "unit": "TFLOP/s", "frac": tile["alg_TFLOPs"] / bf16_peak,
                    # the same kernel time charged with the flops of the NONZEROS it covers only (the block is
                    # mostly zeros): SURVEY 8(d)'s per-nonzero unit
                    "frac_nonzero": 6.0 * K * S * nnz_step * hot_cover / (tile["ms"] * 1e-3) / 1e12 / bf16_peak,
                    "hot_block_nonzero_share": hot_cover,
                    "traffic": traffic.get("hot_tile"),
                    "peak_source": peak_src + " (sustained bf16)", "kernel_ms": tile["ms"],
                    "kernel_share_of_step": tile["ms"] / step_ms,
                    "executed_mma_bf16_TFLOPs": tile["mma_bf16_TFLOPs"],
                    "alg_flop_per_launch": tile["alg_flop"], "alg_bytes_per_launch": tile["alg_bytes"],
                    "hbm_GBps": tile["alg_bytes"] / (tile["ms"] * 1e-3) / 1e9, "hbm_peak": hbm_peak}
    else:
        achieved = kern[dom]["bytes"] / (kern[dom]["ms"] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": traffic.get(dom), "peak_source": peak_src,
                    "kernel_ms": kern[dom]["ms"], "kernel_share_of_step": kern[dom]["ms"] / step_ms}
    roofline.update({
        "kernels": {k: {"ms": v["ms"], "alg_GBps": v["bytes"] / (v["ms"] * 1e-3) / 1e9,
                        "fp32_TFLOPs": v["flop"] / (v["ms"] * 1e-3) / 1e12} for k, v in kern.items()},
        "hot_cols": int(eng.hot_cols) if hybrid else 0, "umma_gemm_gradA": None,
        "hot_prepare_ms_per_batch": prep_ms, "hot_mode": int(eng.hot_mode) if hybrid else 0,
        "note": "csr_rows / csc_cols time the whole row / column side of the step (hybrid: GEMMs, tile kernel and "
                "gather kernels together).  Gather kernels: per nonzero 8 B of HBM vs ~2 KB of L2/L1 record "
                "gathers and 12*K*S flop (fp32 FMA peak 74.4 TFLOP/s); tile kernel: 6*K flop per (row, hot "
                "column, draw) executed as 3 bf16 MMA terms, bound by the shared-memory data pipe"})

    roofline["umma_gemm_gradA"] = gemm_info

    # ------------------------------------------------ CPU baseline (rank 0, bounded sample)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        rows = CPU_SAMPLE_ROWS[args.workload]
        sec, nnz_s, cores = oracle_step_time(wl, rows, 3, 1)
        # the CPU step has a fixed O(D*K*S) parameter-side cost that a small sample cannot amortise the way
        # the GPU arm's full batch does: time a second, smaller sample and report the split
        rows2 = max(rows // 4, 16)
        sec2, nnz2, _ = oracle_step_time(wl, rows2, 2, 1)
        per_row = max((sec - sec2) / (rows - rows2), 0.0)
        fixed = max(sec - per_row * rows, 0.0)
        full_rows = B
        proj = (nnz_s / rows) * full_rows * K / (fixed + per_row * full_rows) if (fixed + per_row) > 0 else None
        cpu = {"value": nnz_s * K / sec, "unit": "nonzeros*K/s", "cores": cores, "kind": "port",
               "sample": f"{rows} rows x D={D} densified ({nnz_s} nonzeros), S={S}, float64 torch-CPU oracle, "
                         f"{sec:.2f} s/step, median of 3 after 1 warm-up",
               "fixed_s_per_step": fixed, "s_per_row": per_row, "second_sample_rows": rows2,
               "projected_value_at_gpu_batch_rows": proj,
               "note": f"projected = the same port extrapolated to the GPU arm's {full_rows} rows/step "
                       "(fixed parameter-side cost amortised identically); the port cannot run that batch "
                       "(it would materialise ~100 GB of (S,B,D) float64 tensors)"}

    if rank == 0:
        print(json.dumps({
            "metric": "advi_elbo_grad_nnzK_per_s", "value": value, "unit": "nonzeros*K/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": wl["desc"], "rows_per_gpu_per_step": B, "shard_rows_per_gpu": shard.nrows,
                       "nnz_per_gpu_per_step": nnz_all / world / args.steps, "D": D, "K": K, "S": S,
                       "parallelism": (f"dp{world} row-sharded, 1 exchange/step ({exchange})" if world > 1
                                       else "dp1 (single GPU: no exchange)"),
                       "l2": "inputs larger than L2 (16 distinct batches cycled; ~130 MB of CSR+CSC each, "
                             "plus ~260 MB of bf16 hot block in hybrid mode)",
                       "variant": args.variant, "final_loss": final_loss,
                       # SURVEY 8(d): work/t and work*S/t -- `value` counts each nonzero once per step;
                       # every one is evaluated for all S draws
                       "nnzK_times_draws_per_s": value * S},
            "e2e": {"value": e2e_value, "unit": "nonzeros*K/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 8, "ms_per_step": float(t2.item()) / args.steps, "host_format": fmt},
            "gpu_launches": launches, "graph_replays": graph_replays, "graphs_primed": primed,
            "clocks": clk, "roofline": roofline, "cpu_baseline": cpu,
        }))
    if outputs is not None:
        outputs["e2e_loss"] = np.array(losses_read[-1], dtype=np.float64)
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
