"""GPU tests of the hybrid step: tcgen05 GEMMs on the dense hot-column block + gather kernels.

* the tensor-core GEMM (bf16 counts x 3-way bf16 split of an fp32 operand) against float64;
* the hot split (ranked, partitioned CSR + dense bf16 block) against a numpy restatement;
* the full ADVI step in hybrid mode against the float64 oracle, same tolerances as the gather path
  (1e-4 relative; 5e-4 for the InverseGamma-family tensors), and against the gather path itself."""
import numpy as np
import pytest
import torch

from tests.util import make_counts, make_oracle, perturbed_params, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-4
TOL_IG = 5e-4


def _ptr(t):
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("M,N,Kd,NQ,splits", [
    (128, 128, 64, 1, 1),        # one tile, one stage
    (300, 128, 192, 1, 1),       # ragged M, three chunks (pipeline wraps once)
    (257, 64, 640, 2, 3),        # split-K with atomics, two draw groups, N=64
    (96, 32, 448, 1, 0),         # M < tile, N=32, automatic split
    (1024, 128, 1024, 1, 2),     # many chunks per CTA: every stage / phase parity reused
])
def test_umma_gemm3_matches_float64(M, N, Kd, NQ, splits):
    from spmf_b200 import _abi
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N)
    A = torch.randint(0, 40, (M, Kd), generator=g).to(torch.float32)
    A[torch.rand(M, Kd, generator=g) < 0.6] = 0
    Bsrc = torch.randn(NQ, Kd, N, generator=g) * torch.exp(2 * torch.randn(NQ, Kd, N, generator=g))
    Arow = A.to(dev).to(torch.bfloat16).contiguous()
    Ad = torch.empty(_abi._lib.spmf_umma_tiled_a_elems(M, Kd), dtype=torch.bfloat16, device=dev)
    _abi.call("spmf_umma_tile_a", _ptr(Arow), Kd, M, Kd, _ptr(Ad), _stream())
    # the tiling helper agrees with the index function the producers use
    probe = [(0, 0), (M - 1, Kd - 1), (M // 2, 17), (min(M - 1, 129), 64 % Kd)]
    for r, k in probe:
        assert float(Ad[_abi._lib.spmf_umma_tiled_a_index(r, k, Kd)]) == float(Arow[r, k])
    Bd = Bsrc.to(dev).contiguous()
    qs = _abi._lib.spmf_umma_tiled_b_elems(N, Kd)
    B3 = torch.zeros(NQ * qs, dtype=torch.bfloat16, device=dev)
    _abi.call("spmf_split3_transpose", _ptr(Bd), N, Kd * N, Kd, Kd, N, _ptr(B3), qs, NQ, _stream())
    torch.cuda.synchronize()
    # the three terms reproduce the fp32 operand to 24 bits: tiles [k/64][term] of N x 64, core matrices 8 x 8
    t = B3.view(NQ, Kd // 64, 3, N // 8, 8, 8, 8).to(torch.float64).sum(2)      # q, kc, n8, k8, n, k
    rec = t.permute(0, 1, 3, 5, 2, 4).reshape(NQ, Kd, N).cpu()                  # q, (kc,k8,k), (n8,n)
    assert rel_err(rec.numpy(), Bsrc.double().numpy()) < 2e-7
    C0 = torch.randn(NQ, M, N, generator=g)
    C = C0.to(dev).contiguous()
    _abi.call("spmf_umma_gemm3", _ptr(Ad), 0, M, _ptr(B3), qs, _ptr(C), N, M * N, N, Kd, NQ, splits, _stream())
    torch.cuda.synchronize()
    ref = C0.double() + torch.einsum("mk,qkn->qmn", A.double(), Bsrc.double())
    err = (C.cpu().double() - ref).abs().max() / ref.abs().max()
    assert float(err) < 2e-6, float(err)

    # the transposed product straight from the same tiles (MN-major operand): Ct[q][Kd'][N] += A^T . Bt^T
    # with k = the rows of A (padded to whole 128-row tiles)
    Mp = (M + 127) // 128 * 128
    Msel = min(Kd, 100)                                    # first Msel columns of A
    Bt_src = torch.randn(NQ, M, N, generator=g)
    qs2 = _abi._lib.spmf_umma_tiled_b_elems(N, Mp)
    Bt3 = torch.zeros(NQ * qs2, dtype=torch.bfloat16, device=dev)
    _abi.call("spmf_split3_transpose", _ptr(Bt_src.to(dev).contiguous()), N, M * N, M, Mp, N, _ptr(Bt3), qs2, NQ,
              _stream())
    Ct = torch.zeros(NQ, Msel, N, device=dev)
    _abi.call("spmf_umma_gemm3_at", _ptr(Ad), Kd, M, Msel, _ptr(Bt3), qs2, _ptr(Ct), N, Msel * N, N, NQ, splits,
              _stream())
    torch.cuda.synchronize()
    reft = torch.einsum("mk,qmn->qkn", A.double()[:, :Msel], Bt_src.double())
    errt = (Ct.cpu().double() - reft).abs().max() / reft.abs().max()
    assert float(errt) < 2e-6, float(errt)


def test_hot_split_wide_block_fallback():
    """The direct-scatter variant of the split (hot blocks too wide for shared-memory staging), forced
    on a small input in a fresh process: same hybrid form as the staged kernel."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SPMF_SPLIT_UNSTAGED="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", os.path.join(root, "tests", "test_gpu_hybrid.py"),
                        "-k", "partitions_and_fills or fit_reduces or u8_format_fused_into_the_split"],
                       env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_hot_split_partitions_and_fills_dense_block():
    from spmf_b200 import _abi
    from spmf_b200.data import CsrShard
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(3)
    B, D, H = 70, 90, 33
    x = rng.poisson(0.8, size=(B, D)).astype(np.float32)
    x[rng.random((B, D)) < 0.02] = 300.0          # not exact in bf16 -> stays on the gather path
    x[5, :] = 0
    x[5, 7] = 2.5                                  # exact in bf16, non-integer
    x[6, 3] = 257.0                                # not exact
    rank = rng.permutation(D).astype(np.int32)
    sh = CsrShard.from_dense(torch.from_numpy(x), dev)
    b = sh.batch(0, B)
    junk = torch.full((1 << 22,), 1.5, dtype=torch.bfloat16, device=dev)   # dirty the allocator's free blocks:
    del junk                                                              # the split must write every chunk of xhot
    h = b.ensure_hot(torch.from_numpy(rank).to(dev), H)
    torch.cuda.synchronize()
    rp = h.rowptr.cpu().numpy()
    cols, vals, mid = h.cols.cpu().numpy(), h.vals.cpu().numpy(), h.rowmid.cpu().numpy()
    Hp = (H + 63) // 64 * 64

    def untile(t, rows, kd):     # UMMA-tiled [rows/128][kd/64] tiles of (16 x 8) core matrices of 8 x 8
        rp_ = (rows + 127) // 128 * 128
        v = t[:rp_ * kd].view(rp_ // 128, kd // 64, 16, 8, 8, 8).float()      # mt, kc, r8, k8, r, k
        return v.permute(0, 2, 4, 1, 3, 5).reshape(rp_, kd).cpu().numpy()
    xh = untile(h.xhot, B, Hp)
    assert (xh[B:] == 0).all()                                    # padding rows of the last 128-row tile
    xh = xh[:B]
    assert rp[0] == 0 and rp[-1] == int((x != 0).sum())
    dense = np.zeros((B, D), np.float32)
    exp_hot = np.zeros((B, Hp), np.float32)
    for r in range(B):
        seg = slice(rp[r], rp[r + 1])
        c, v = cols[seg], vals[seg]
        assert (v[:mid[r]] < 0).all() and (v[mid[r]:] > 0).all()
        assert (c[:mid[r]] < H).all()
        dense[r, c] = np.abs(v)
        exp_hot[r, c[:mid[r]]] = -v[:mid[r]]
    inv = np.empty(D, np.int64)
    inv[rank] = np.arange(D)
    assert np.array_equal(dense[:, rank], x)                      # ranked ids, values intact
    # coverage rule: rank < H and exactly representable in bf16
    xr = x[:, inv]                                                # columns in rank order
    exact = torch.from_numpy(xr).to(torch.bfloat16).float().numpy() == xr
    cov = (xr > 0) & exact & (np.arange(D)[None, :] < H)
    assert not cov[:, H:].any() and np.array_equal(exp_hot[:, :H] != 0, cov[:, :H])
    assert np.array_equal(xh, exp_hot)
    assert (xh[:, H:] == 0).all()
    # the CSC copy of the uncovered entries
    want = np.where(cov, 0, xr)
    cp = h.colptr.cpu().numpy()
    cr, cv = h.crows.cpu().numpy(), h.cvals.cpu().numpy()
    assert cp[0] == 0 and cp[-1] == int((want != 0).sum())
    back = np.zeros((B, D), np.float32)
    for d in range(D):
        back[cr[cp[d]:cp[d + 1]], d] = cv[cp[d]:cp[d + 1]]
    assert np.array_equal(back, want)


def _step(model, eng, params, noise, batch):
    views = eng.layout.views(eng.params)
    for k, v in params.items():
        views[k].copy_(v.to(device=eng.device, dtype=torch.float32))
    eng.set_noise_from(noise)
    parts = eng.loss_and_grad(batch, fresh_noise=False)
    torch.cuda.synchronize()
    return float(eng.loss_value(parts).item())


@pytest.mark.parametrize("D,K,B,S,kind,big", [
    (128, 32, 200, 4, "noise", False),     # REC=128, every column hot, ragged row tile
    (300, 32, 96, 4, "sparse", True),      # hot + cold columns, counts > 256 mixed in
    (200, 16, 150, 4, "linear", False),    # REC=64
    (96, 8, 130, 4, "linear", False),      # REC=32
    (160, 32, 70, 2, "noise", True),       # SV=2 -> REC=64
    (130, 20, 300, 8, "sparse", False),    # K padded to 32, two draw groups
    (150, 128, 140, 2, "sparse", True),    # K=128 (C5): REC=256 -> GEMMs in two blocks of 128 channels; wide tile kernel
    (320, 128, 200, 4, "sparse", False),   # K=128, S=4 (REC=512): 5 column chunks over 2 input stages, ragged row tiles
    (100, 64, 96, 4, "noise", False),      # K=64, REC=256: fused tile kernel with 64 latent dims
    (300, 64, 200, 4, "sparse", True),     # K=64: hot + cold columns, ragged row tiles, 5 column chunks
    (140, 50, 130, 2, "linear", False),    # K padded to 64, SV=2 -> REC=128
    (90, 100, 70, 4, "linear", False),     # K padded to 128, REC=512 (four blocks)
])
def test_hybrid_step_matches_oracle_and_gather_path(D, K, B, S, kind, big):
    import spmf_b200
    from oracle.spmf_oracle import draw_noise
    dev = torch.device("cuda:0")
    x = make_counts(B, D, seed=11, kind=kind)
    if big:
        rng = np.random.default_rng(5)
        m = (rng.random(x.shape) < 0.01) & (x > 0)
        x[m] = 300.0 + x[m]
    N = 10 * B
    oracle = make_oracle(D, K, N, x)
    params = perturbed_params(oracle, 0.3, 11)
    noise = draw_noise(oracle, params, S, seed=12)
    ref_loss, ref_grads, ref_parts = oracle.loss_and_grads(params, noise, {'counts': torch.tensor(x, dtype=torch.float64)})

    out = {}
    # tile: count products and the per-nonzero terms of the hot block on the tensor cores;
    # gather: CUDA-core kernels only
    for name, dens in (("tile", 0.03), ("gather", 0.0)):
        model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(N * D),
                                               device=dev, hot_density=dens)
        model.compute_scales(lambda: [{'counts': x}])
        eng = model._engine_for(S)
        if name != "gather":
            assert eng.hot_cols >= 64 and eng.hybrid_ok, (eng.hot_cols, eng.hybrid_ok)
        else:
            assert eng.hot_cols == 0
        batch = spmf_b200.as_device_batch(x, dev)
        loss = _step(model, eng, params, noise, batch)
        if name != "gather":
            assert batch.hot is not None and batch.hot.H == eng.hot_cols
        assert abs(loss - ref_loss) <= TOL * abs(ref_loss), (name, loss, ref_loss)
        pd = eng.parts_dict()
        for pn in list(ref_parts):
            ref = ref_parts[pn].numpy()
            assert np.abs(pd[pn].numpy() - ref).max() <= TOL * max(np.abs(ref).max(), 1.0), (name, pn)
        grads = {k: v.cpu().numpy().copy() for k, v in eng.layout.views(eng.grads).items()}
        for k, g in ref_grads.items():
            tol = TOL if k.split('/')[0] in ('v', 'w', 'u', 's') else TOL_IG
            e = rel_err(grads[k], g.numpy())
            assert e <= tol, (name, k, e)
        out[name] = (loss, grads)
    # the CUDA paths agree with each other far inside the oracle tolerance
    assert abs(out["tile"][0] - out["gather"][0]) <= 2e-6 * abs(out["gather"][0])
    for k in out["gather"][1]:
        assert rel_err(out["tile"][1][k], out["gather"][1][k]) <= 3e-5, k


def test_hybrid_fit_reduces_loss_and_streams():
    """Training through the public API in hybrid mode: resident batches and host-streamed batches
    give the same losses; the loss goes down."""
    import spmf_b200
    from spmf_b200.data import CsrShard, HostCsr
    dev = torch.device("cuda:0")
    B, D, K = 256, 192, 16
    x = make_counts(4 * B, D, seed=2, kind="linear")
    sh = CsrShard.from_dense(torch.from_numpy(x), dev)

    def run(stream):
        model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(x.size),
                                               device=dev, seed=3, hot_density=0.03)
        model.compute_scales(sh)
        assert model.hot_cols >= 64
        if stream:
            host = HostCsr.from_shard(sh)
            fac = lambda: ({'counts': hb} for hb in host.iter_batches(B))
        else:
            fac = lambda: ({'counts': b} for b in sh.iter_batches(B))
        return model.fit(fac, num_steps=4, learning_rate=0.05, sample_size=4, verbose=False, rel_tol=None)

    a, b = run(False), run(True)
    assert a[-1] < a[0]
    assert np.allclose(a, b, rtol=1e-5), (a, b)


@pytest.mark.parametrize("D,K,B,S,kind,big", [
    (160, 16, 192, 4, "noise", False),     # dense-origin counts: every column hot, nothing uncovered
    (300, 32, 200, 4, "sparse", False),    # hot + cold columns: the cold nonzeros go to the ranked CSR
    (192, 32, 130, 4, "linear", True),     # counts that bf16 cannot hold (uint16 transfer) stay out of the block
])
def test_dense_ingest_matches_csr_path(D, K, B, S, kind, big):
    """HostDense -> one H2D of the slab -> spmf_dense_hot_split: the same hybrid form and the same step as the
    CSR upload of the same rows (bit-identical arrays, step equal up to fp32 atomics)."""
    import spmf_b200
    from spmf_b200.data import CsrShard, HostDense, HostDenseBatch, prefetch_to_device
    dev = torch.device("cuda:0")
    x = make_counts(3 * B, D, seed=8, kind=kind)
    if big:
        x[3, 5], x[B + 7, 11], x[2 * B + 1, 0] = 1001.0, 257.0, 40000.0
    sh = CsrShard.from_dense(x, dev)
    model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(x.size),
                                           device=dev, seed=3)
    model.compute_scales(sh)
    eng = model._engine_for(S)
    assert eng.hot_mode == 2 and eng.hot_cols > 0
    host = HostDense(x)
    assert host.x.dtype == (torch.uint16 if big else torch.uint8)
    assert isinstance(host.batch(0, B), HostDenseBatch) and host.batch(0, B).nnz == int((x[:B] != 0).sum())
    eng.fill_noise(step=0)
    hot = model._hot_spec(eng)
    got = []
    for i, db in enumerate(prefetch_to_device(host.iter_batches(B), dev, hot=hot)):
        assert db.dense_raw is not None and db.cols is None
        ref_b = sh.batch(i * B, B, cache=False)
        h_ref = ref_b.ensure_hot(eng.rank, eng.hot_cols, version=getattr(eng, "rank_version", 0))
        h = db.hot
        torch.cuda.synchronize()
        n_unc = int(h.rowptr[B].item())
        assert torch.equal(h.xhot[:h_ref.xhot.numel()].view(torch.int16), h_ref.xhot.view(torch.int16))
        assert torch.equal(db.rowsum, ref_b.rowsum) and torch.allclose(db.lgam, ref_b.lgam, rtol=1e-6)
        assert torch.equal(h.colptr, h_ref.colptr)            # CSC of the uncovered entries: same column counts
        nu = int(h.colptr[-1].item())
        assert nu == n_unc
        # (the order inside a column follows the atomic cursor of the CSC build: compare as sorted (col, row, value))
        def entries(hh):
            col = torch.repeat_interleave(torch.arange(D, device=dev), (hh.colptr[1:] - hh.colptr[:-1]).long())
            key = col * B + hh.crows[:nu].long()
            o = torch.argsort(key)
            return key[o], hh.cvals[:nu][o]
        (k1, v1), (k2, v2) = entries(h), entries(h_ref)
        assert torch.equal(k1, k2) and torch.equal(v1, v2)
        p = eng.loss_and_grad(db, fresh_noise=False).clone()
        g = eng.grads.clone()
        p0 = eng.loss_and_grad(ref_b, fresh_noise=False).clone()
        assert rel_err(p.cpu().numpy(), p0.cpu().numpy()) < 1e-6
        assert rel_err(g.cpu().numpy(), eng.grads.cpu().numpy()) < 2e-5
        got.append(p)
    assert len(got) == 3


def test_dense_ingest_fit_and_gather_fallback():
    """fit() over HostDense batches == fit() over the resident shard, for a tile-hybrid engine (direct ingest)
    and for a gather-only one (K = 4: the uploader compacts the slab to CSR on the device)."""
    import spmf_b200
    from spmf_b200.data import CsrShard, HostDense
    dev = torch.device("cuda:0")
    B, D = 256, 192
    x = make_counts(4 * B, D, seed=2, kind="linear")
    sh = CsrShard.from_dense(x, dev)
    host = HostDense(x)
    for K in (16, 4):
        def run(stream):
            model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(x.size),
                                                   device=dev, seed=3)
            model.compute_scales(sh)
            fac = (lambda: ({'counts': hb} for hb in host.iter_batches(B))) if stream else \
                  (lambda: ({'counts': b} for b in sh.iter_batches(B)))
            return model.fit(fac, num_steps=4, learning_rate=0.05, sample_size=4, verbose=False, rel_tol=None)
        a, b = run(False), run(True)
        assert a[-1] < a[0]
        assert np.allclose(a, b, rtol=1e-5), (K, a, b)


@pytest.mark.parametrize("D,K,B", [(300, 32, 200), (2600, 16, 130)])
def test_u8_format_fused_into_the_split(D, K, B):
    """2-byte transfer format read by the hot split itself (spmf_hot_split_u8): same hybrid form and step as the
    CSR upload.  Covers counts above 254 (overflow list), zero-valued bridge entries (gaps > 256 columns) and a
    row longer than the split's shared-memory stash (its columns are re-scanned in the second pass)."""
    import spmf_b200
    from spmf_b200.data import CsrShard, HostCsr, prefetch_to_device
    dev = torch.device("cuda:0")
    S = 4
    x = make_counts(2 * B, D, seed=9, kind="sparse")
    x[0, :] = np.maximum(x[0, :], 1.0)              # a full row (D = 2600: longer than the 2048-entry stash)
    x[0, D - 3], x[5, 1], x[B + 2, D // 2] = 700.0, 255.0, 3000.0
    x[7, :] = 0
    x[7, 0], x[7, D - 1] = 2.0, 1.0                 # D = 2600: a gap of 2598 columns -> bridge entries
    sh = CsrShard.from_dense(x, dev)
    model = spmf_b200.PoissonFactorization(latent_dim=K, feature_dim=D, u_tau_scale=1.0 / np.sqrt(x.size),
                                           device=dev, seed=3)
    model.compute_scales(sh)
    eng = model._engine_for(S)
    assert eng.hot_mode == 2 and 0 < eng.hot_cols
    host = HostCsr.from_shard(sh, compact="u8")
    eng.fill_noise(step=0)
    for i, db in enumerate(prefetch_to_device(host.iter_batches(B), dev, hot=model._hot_spec(eng))):
        assert db.cols is None and db.hot is not None           # never widened to int32 / fp32 feature-order arrays
        ref_b = sh.batch(i * B, B, cache=False)
        h_ref = ref_b.ensure_hot(eng.rank, eng.hot_cols, version=getattr(eng, "rank_version", 0))
        h = db.hot
        assert torch.equal(h.xhot[:h_ref.xhot.numel()].view(torch.int16), h_ref.xhot.view(torch.int16))
        assert torch.equal(db.rowsum, ref_b.rowsum) and torch.allclose(db.lgam, ref_b.lgam, rtol=1e-6)
        assert torch.equal(h.rowmid[:B], h_ref.rowmid[:B])
        p = eng.loss_and_grad(db, fresh_noise=False).clone()
        g = eng.grads.clone()
        p0 = eng.loss_and_grad(ref_b, fresh_noise=False).clone()
        assert rel_err(p.cpu().numpy(), p0.cpu().numpy()) < 1e-6
        assert rel_err(g.cpu().numpy(), eng.grads.cpu().numpy()) < 2e-5
