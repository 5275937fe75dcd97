"""Parameter-side kernels of one step: the split backward (data-independent half on the side stream, data
half after the data term) against the one-pass backward, and the Gamma draws and their implicit gradients
against the CPU host check of the same spmf_math.cuh bodies."""
import ctypes as C

import numpy as np
import pytest
import torch

from spmf_b200 import _abi
from tests.util import rel_err

pytestmark = pytest.mark.gpu

VAR_UETA, NUM_VARS = 4, 12
SEED = 0x5EED1234ABCD


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _setup(D, K, S, seed=0):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(seed)
    toff, noff = _abi.layout(D, K, S)
    # Gamma concentrations around softplus(0.5) ~ 1: no draw so close to 0 that beta / g overflows
    params = (0.5 + 0.3 * torch.randn(toff[-1], generator=g)).to(dev)
    noise = torch.zeros(noff[-1], device=dev)
    dgda = torch.zeros(noff[-1], device=dev)
    _abi.call("spmf_fill_noise_dev", _p(noise), _p(params), D, K, S, SEED, 0, 1, None, None)
    _abi.call("spmf_gamma_draw_grad_dev", _p(params), _p(noise), _p(dgda), D, K, S, SEED, 0, None, None)
    return dev, g, toff, noff, params, noise, dgda


def _backward(D, K, S, split, seed=0):
    dev, g, toff, noff, params, noise, dgda = _setup(D, K, S, seed)
    KP, SV = _abi.kpad(K), _abi.draw_vec_k(K, S)
    NQ = S // SV
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
    hyper = (64.0, 0.01, 1.0, 0.9, 1.0, 1.0, 1)   # batch rows, u_tau / s_tau scale, decay, entropy / prior weight, world
    if split:
        _abi.call("spmf_backward_pre_m", _p(params), _p(noise), _p(dgda), _p(eta), D, K, S, *hyper, _p(grads),
                  _p(scr_f), _p(scr_d), _abi.MODEL_POISSON, None)
        _abi.call("spmf_backward_post_m", _p(params), _p(noise), _p(eta), _p(rank), D, K, S, _p(GAp), _p(GEV),
                  _p(Gph), _p(zcol), _p(datasums), _p(phisum), *hyper, _p(grads), _p(parts), _p(scr_f),
                  _p(scr_d), None, _abi.MODEL_POISSON, None)
    else:
        _abi.call("spmf_backward_params_ranked_m", _p(params), _p(noise), _p(dgda), _p(eta), _p(rank), D, K, S,
                  _p(GAp), _p(GEV), _p(Gph), _p(zcol), _p(datasums), _p(phisum), *hyper, _p(grads), _p(parts),
                  _p(scr_f), _p(scr_d), None, _abi.MODEL_POISSON, None)
    torch.cuda.synchronize()
    return toff, grads.cpu().numpy(), parts.cpu().numpy().reshape(S, 16)


@pytest.mark.parametrize("S", [1, 3, 4])
@pytest.mark.parametrize("K", [2, 8, 32, 128, 256])
def test_split_backward_matches_one_pass(K, S):
    D = 300
    toff, g1, p1 = _backward(D, K, S, split=False)
    _, g2, p2 = _backward(D, K, S, split=True)
    assert np.isfinite(g1).all() and np.isfinite(p1).all()
    for t in range(len(toff) - 1):
        a, b = g1[toff[t]:toff[t + 1]], g2[toff[t]:toff[t + 1]]
        assert rel_err(b, a) < 1e-6, (t, rel_err(b, a))
    for s in range(S):
        assert rel_err(p2[s], p1[s]) < 1e-6, (s, p1[s], p2[s])


def test_gamma_draws_and_gradients_match_host_check():
    import tests.hostcheck as hc
    D, K, S = 257, 32, 4
    _, _, toff, noff, params, noise, dgda = _setup(D, K, S, seed=1)
    P, N, G = params.cpu().numpy(), noise.cpu().numpy(), dgda.cpu().numpy()
    rng = np.random.default_rng(0)
    nelems = {4: D * K, 5: K, 6: 2 * D, 7: D, 8: D * K, 9: K, 10: 2 * D, 11: D}
    for v in range(VAR_UETA, NUM_VARS):
        nelem = nelems[v]
        for e in rng.choice(min(nelem, 96), size=6, replace=False):
            alpha, sg = np.empty(1, np.float32), np.empty(1, np.float32)
            hc.lib.hc_softplus(np.array([P[toff[2 * v] + e]], np.float32), alpha, sg, 1)
            alpha = float(alpha[0])
            idx = np.array([s * nelem + e for s in range(S)])
            # the draw of element i uses the Philox stream of (variable, step 0) at counter i
            host = hc.gammas(int(idx[-1]) + 1, alpha, stream=v, seed=SEED)[idx]
            got = N[noff[v] + idx]
            # the device evaluates log / cos with single-MUFU intrinsics, the host with libm
            np.testing.assert_allclose(got, host, rtol=2e-5, atol=1e-30)
            ref = hc.gamma_grad4(np.full(4, alpha, np.float32), got.astype(np.float32))
            np.testing.assert_allclose(G[noff[v] + idx], ref, rtol=2e-4, atol=1e-6 * np.abs(ref).max())
