"""Time the parameter-side entry points of one step in isolation with CUDA events.

    python scripts/param_side_time.py [--D 20000] [--S 4] [--K 32 128] [--iters 200] [--tag NAME]

For each K: the Gamma draws + implicit gradients (spmf_gamma_draw_grad_dev), the data-independent half of
the backward (spmf_backward_pre_m) and its data half (spmf_backward_post_m), each launched `iters` times
back to back on one stream, five windows each; prints one JSON line per (K, entry point) with the median
and the spread of the per-launch time in microseconds.  The inputs are seeded random tensors of the step's
shapes (C4: D = 20,000, S = 4); every buffer stays resident in L2 between launches (the working set at
K = 32 is ~100 MB), so these are warm-cache kernel times.
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from spmf_b200 import _abi  # noqa: E402

SEED = 0x5EED1234ABCD


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def time_calls(fn, iters, windows=5):
    fn()
    torch.cuda.synchronize()
    per = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        per.append(a.elapsed_time(b) * 1e3 / iters)
    per.sort()
    return per[len(per) // 2], per[0], per[-1]


def run(D, K, S, iters, tag):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(0)
    toff, noff = _abi.layout(D, K, S)
    KP, SV = _abi.kpad(K), _abi.draw_vec_k(K, S)
    NQ = S // SV
    params = (0.5 * torch.randn(toff[-1], generator=g)).to(dev)
    noise = torch.zeros(noff[-1], device=dev)
    dgda = torch.zeros(noff[-1], device=dev)
    eta = (0.5 + torch.rand(2 * D, generator=g)).to(dev)
    rank = torch.randperm(D, generator=g).to(torch.int32).to(dev)
    GAp = (0.1 * torch.randn(NQ * D * SV * KP, generator=g)).to(dev)
    GEV = (0.1 * torch.randn(NQ * D * SV * KP, generator=g)).to(dev)
    Gph = torch.rand(NQ * D * SV, generator=g).to(dev)
    zcol = torch.randn(NQ * SV * KP, generator=g, dtype=torch.float64).to(dev)
    datasums = torch.randn(NQ * 4 * SV, generator=g, dtype=torch.float64).to(dev)
    phisum = torch.rand(NQ * SV, generator=g, dtype=torch.float64).to(dev)
    nf, nd = _abi.backward_scratch(D, K, S)
    scr_f = torch.zeros(nf, device=dev)
    scr_d = torch.zeros(nd, dtype=torch.float64, device=dev)
    grads = torch.zeros(toff[-1], device=dev)
    parts = torch.zeros(S * 16, dtype=torch.float64, device=dev)
    hyper = (8192.0, 0.01, 1.0, 0.9, 1.0, 1.0, 1)
    _abi.call("spmf_fill_noise_dev", _p(noise), _p(params), D, K, S, SEED, 0, 1, None, None)

    def gamma():
        _abi.call("spmf_gamma_draw_grad_dev", _p(params), _p(noise), _p(dgda), D, K, S, SEED, 0, None, None)

    def pre():
        _abi.call("spmf_backward_pre_m", _p(params), _p(noise), _p(dgda), _p(eta), D, K, S, *hyper, _p(grads),
                  _p(scr_f), _p(scr_d), _abi.MODEL_POISSON, None)

    def post():
        _abi.call("spmf_backward_post_m", _p(params), _p(noise), _p(eta), _p(rank), D, K, S, _p(GAp), _p(GEV),
                  _p(Gph), _p(zcol), _p(datasums), _p(phisum), *hyper, _p(grads), _p(parts), _p(scr_f),
                  _p(scr_d), None, _abi.MODEL_POISSON, None)

    gamma()
    pre()
    for name, fn in (("spmf_gamma_draw_grad_dev", gamma), ("spmf_backward_pre_m", pre),
                     ("spmf_backward_post_m", post)):
        med, lo, hi = time_calls(fn, iters)
        print(json.dumps({"tag": tag, "D": D, "K": K, "S": S, "entry": name, "us_median": round(med, 2),
                          "us_min": round(lo, 2), "us_max": round(hi, 2),
                          "gpu": torch.cuda.get_device_name(0)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--D", type=int, default=20000)
    ap.add_argument("--S", type=int, default=4)
    ap.add_argument("--K", type=int, nargs="+", default=[32, 128])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--tag", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("param_side_time.py needs a CUDA device")
    for K in a.K:
        run(a.D, K, a.S, a.iters, a.tag)


if __name__ == "__main__":
    main()
