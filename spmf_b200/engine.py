"""Launch sequence of one ADVI step on one GPU: owns the device workspace and calls the C ABI.

Replaces, for `PoissonFactorization`, what bayesianquilts' `minibatch_fit_surrogate_posterior`
does per batch in the reference stack [EXT L3/L4] (call site tests/spmf_test.py:35-43):
draw S reparameterised samples, evaluate `log q - unormalized_log_prob` (poisson.py:575-621) and
back-propagate to the 24 variational tensors -- as one native call (`spmf_advi_step`, ~25 kernel
launches over five streams in hybrid mode) instead of a TensorFlow graph, never materialising the
(S,B,D) rate tensor of poisson.py:174-184.
"""
from __future__ import annotations

import itertools
import os
from typing import Optional

import torch

from . import _abi
from .data import DeviceBatch, StepGraphs as _StepGraphs, _ptr, _stream
from .variables import VariableLayout, PART_NAMES

# engine serial numbers: the key of an engine's cached step graphs (an id() may be reused by a later engine, e.g.
# one loaded from a checkpoint in the same process, whose graphs would then replay the freed engine's buffers)
_ENGINE_SERIAL = itertools.count()


class StepWorkspace:
    """All per-step device buffers for fixed (D, K, S) and a maximum batch size."""

    def __init__(self, D, K, S, max_rows, device):
        self.D, self.K, self.S = D, K, S
        self.KP, self.SV = _abi.kpad(K), _abi.draw_vec_k(K, S)
        self.NQ = S // self.SV
        self.max_rows = 0
        self.device = device
        f32, f64 = torch.float32, torch.float64
        C = self.KP * self.SV
        n_op = self.NQ * D * C
        self.Ap = torch.empty(n_op, dtype=f32, device=device)
        self.EV = torch.empty(n_op, dtype=f32, device=device)
        self.PH = torch.empty(self.NQ * D * self.SV, dtype=f32, device=device)
        self.GAp = torch.empty(n_op, dtype=f32, device=device)
        self.GEV = torch.empty(n_op, dtype=f32, device=device)
        self.Gph = torch.empty(self.NQ * D * self.SV, dtype=f32, device=device)
        self.vsum = torch.empty(self.NQ * C, dtype=f64, device=device)
        self.phisum = torch.empty(self.NQ * self.SV, dtype=f64, device=device)
        self.zcolsum = torch.empty(self.NQ * C, dtype=f64, device=device)
        self.datasums = torch.empty(self.NQ * 4 * self.SV, dtype=f64, device=device)
        nf, nd = _abi.backward_scratch(D, K, S)
        self.scr_f = torch.empty(nf, dtype=f32, device=device)
        self.scr_d = torch.empty(nd, dtype=f64, device=device)
        self.scr_dpre = torch.empty(nd, dtype=f64, device=device)    # split backward: side-stream half
        self.parts = torch.zeros(S * _abi.NUM_PARTS, dtype=f64, device=device)
        self.ensure_rows(max_rows)

    def ensure_hybrid(self, H, nrows):
        """bf16 three-term operands of the tcgen05 GEMMs (UMMA-tiled B3): ApT3 over the hot columns,
        dzrT3 over the batch rows; one block of `t3_qstride` elements per draw group."""
        kd = max((int(H) + 63) // 64 * 64, (int(nrows) + 127) // 128 * 128)
        changed = False
        if getattr(self, "t3_kd", 0) < kd:
            self.t3_kd = kd
            self.t3_qstride = int(_abi._lib.spmf_umma_tiled_b_elems(self.KP * self.SV, kd))
            self.ApT3 = torch.zeros(self.NQ * self.t3_qstride, dtype=torch.bfloat16, device=self.device)
            self.dzrT3 = torch.zeros(self.NQ * self.t3_qstride, dtype=torch.bfloat16, device=self.device)
            changed = True
        # the EV / phi tile workspace is sized by H alone (not by kd): track it separately
        evt_bytes = max(int(_abi._lib.spmf_hot_tile_scratch_bytes(int(H), self.K, self.S)), 16)
        if getattr(self, "evt_bytes", 0) < evt_bytes:
            self.evt_bytes = evt_bytes
            self.EVt = torch.zeros(evt_bytes, dtype=torch.uint8, device=self.device)
            changed = True
        return changed

    def ensure_dense(self, nrows):
        """fp32 [nrows][D] scratch of the dense evaluation (spmf_dense.cu): every step for the links without
        a closed-form sum(rate), only when the non-finite guard fires for the default link."""
        need = int(nrows) * self.D
        if getattr(self, "xdense", None) is None or self.xdense.numel() < need:
            self.xdense = torch.empty(max(need, 1), dtype=torch.float32, device=self.device)
            return True
        return False

    def ensure_rows(self, nrows):
        """Grow the per-row buffers to `nrows` rows; True if they moved.  Callers outside __init__ go through
        AdviEngine.ensure_rows, which also invalidates what points into the old buffers."""
        if nrows <= self.max_rows:
            return False
        C = self.KP * self.SV
        self.max_rows = int(nrows)
        self.z = torch.empty(self.NQ * nrows * C, dtype=torch.float32, device=self.device)
        self.dzr = torch.empty(self.NQ * nrows * C, dtype=torch.float32, device=self.device)
        self.rowacc = torch.empty(self.NQ * nrows * 4 * self.SV, dtype=torch.float32, device=self.device)
        return True


class AdviEngine:
    """ELBO + gradient of one minibatch; optimiser state; everything stays on the device."""

    # exact guard scratch is nrows*D floats; above this many bytes the guard degrades to drop-and-count
    GUARD_SCRATCH_LIMIT = 16 << 30

    def __init__(self, D, K, S, device, u_tau_scale, s_tau_scale, decay, scale_rows=True,
                 entropy_weight=1.0, prior_weight=1.0, world_size=1, seed=0, max_rows=0, link=0,
                 exact_guard=True, model=0):
        if K > _abi.MAX_K:
            raise _abi.SpmfError(f"latent_dim {K} > {_abi.MAX_K} is not supported by the CUDA path")
        self.D, self.K, self.S = int(D), int(K), int(S)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _abi.SpmfError("spmf_b200 computes on CUDA devices only (no CPU fallback)")
        self.layout = VariableLayout(D, K, S)
        self.u_tau_scale, self.s_tau_scale, self.decay = float(u_tau_scale), float(s_tau_scale), float(decay)
        self.scale_rows = bool(scale_rows)
        self.entropy_weight, self.prior_weight = float(entropy_weight), float(prior_weight)
        self.world_size = int(world_size)
        self.seed = int(seed)
        L = self.layout
        from . import p2p
        if self.world_size > 1 and p2p.enabled():
            # data-parallel: parameters / gradients live in memory the peer GPUs can map (csrc/spmf_p2p.cu)
            self.params, self.grads = p2p.peer_zeros(L.n_params, self.device), p2p.peer_zeros(L.n_params, self.device)
        else:
            self.params = torch.zeros(L.n_params, dtype=torch.float32, device=self.device)
            self.grads = torch.zeros(L.n_params, dtype=torch.float32, device=self.device)
        L.fill_initial(self.params, self.u_tau_scale, self.s_tau_scale)
        self.adam_m = torch.zeros(L.n_params, dtype=torch.float32, device=self.device)
        self.adam_v = torch.zeros(L.n_params, dtype=torch.float32, device=self.device)
        self.noise = torch.empty(L.n_noise, dtype=torch.float32, device=self.device)
        self.dgda = torch.zeros(L.n_noise, dtype=torch.float32, device=self.device)
        # [2][D]: decoder scale eta_i | encoder divisor (eta_i, or 1 under log_transform) -- spmf_model.cuh
        self.eta = torch.ones(2 * D, dtype=torch.float32, device=self.device)
        # link function (SPMF_LINK_*): 0 = linear Poisson (sparse / tensor-core path with closed-form sum(rate));
        # log_transform / Bernoulli run the dense CUDA-core path of spmf_dense.cu
        self.link = int(link)
        self.model = int(model)           # SPMF_MODEL_*: Bernoulli = Identity bijector + Normal priors on v, w
        self.exact_guard = bool(exact_guard)
        self.custom_link = None           # (encoder, decoder) torch callables: data term in torch (see custom_forward)
        # device guard state (poisson.py:606-616): flag | nbad | (min finite log-likelihood, entry)
        self.gs = torch.zeros(int(_abi._lib.spmf_guard_state_bytes()), dtype=torch.uint8, device=self.device)
        self.reset_guard()
        # per-step scalars on the device (Philox step, Adam step / rates): what a replayed graph reads
        self.step_state = torch.zeros(max(int(_abi._lib.spmf_step_state_bytes()), 64), dtype=torch.uint8,
                                      device=self.device)
        # Resident batches (cut from a CsrShard) replay their step as ONE CUDA graph launch (SPMF_GRAPHS=0:
        # always launch eagerly).  Measured on B200 with captures outside the timed region
        # (profiles/r2_graph_replay.txt): C1 0.137 -> 0.114, C2 0.202 -> 0.170, C3 0.282 -> 0.250,
        # C4 1.104 -> 1.096 ms/step.  A capture + instantiation costs ~2 ms per (batch, configuration).
        self.use_graphs = os.environ.get("SPMF_GRAPHS", "1") != "0"
        self._ws_gen = 0                  # bumped whenever a workspace buffer moves: invalidates graphs
        self._warm_cfgs = set()
        self.graph_launches = 0
        self._serial = next(_ENGINE_SERIAL)
        self.rank = None          # int32 [D]: table row of each feature (hot-column ordering), or None
        self.hot_cols = 0         # H > 0 enables the hybrid (tensor-core hot block + gather) step
        # tile-hybrid step: GEMMs for the count products + fused tile kernel for the per-nonzero terms
        self.hybrid_ok = self.link == 0 and _abi._lib.spmf_hybrid_supported(self.K, self.S) != 0
        self.hot_mode = 2 if self.hybrid_ok else 0    # spmf_hybrid_supported's code for the tile-hybrid step
        self.inv_xi = 1.0
        self._ws = None
        self._side = None
        self._args = None
        self.stream_mode = os.environ.get("SPMF_STREAMS", "prio")
        # Adam of the data-free tensors under the data term (spmf_step_args.adam_tail_early): needs the split
        # backward on its side stream
        self.adam_early = (os.environ.get("SPMF_ADAM_EARLY", "1") != "0" and self.stream_mode == "prio"
                           and os.environ.get("SPMF_SPLIT_BACKWARD", "1") != "0")
        self._max_rows = max_rows
        self.opt_step = 0
        self.tail_stepped = False
        self.rng_step = 0
        self.launches = 0     # CUDA kernel launches issued through the ABI (bench's gpu_launches)
        self.kernel_events = None   # when a dict: name -> [(start,end) CUDA events] around the hot kernels

    @property
    def ws(self) -> StepWorkspace:
        if self._ws is None:     # lazily: sampling-only uses (surrogate.sample) never need it
            self._ws = StepWorkspace(self.D, self.K, self.S, self._max_rows, self.device)
        return self._ws

    # ------------------------------------------------------------------ pieces
    NOISE_NORMAL, NOISE_GAMMA = 1, 2

    def reset_guard(self):
        """Re-arm the guard state (the training step's last kernel does this itself; the API paths that
        stop after the data term call it explicitly)."""
        _abi.call("spmf_guard_reset", _ptr(self.gs), 2 if self.link != 0 else 0, _stream())

    def guard_report(self):
        """(flag, nbad, replacement value min(finite) - 10) of the last data-term evaluation (host sync)."""
        import ctypes as C
        raw = bytes(self.gs.cpu().numpy().tobytes())
        buf = C.create_string_buffer(raw, len(raw))
        flag, nbad, mv = C.c_int(), C.c_int(), C.c_float()
        _abi.call("spmf_guard_decode", C.cast(buf, C.c_void_p), C.byref(flag), C.byref(nbad), C.byref(mv))
        return flag.value, nbad.value, mv.value

    def _workspace_moved(self):
        """A workspace buffer was reallocated: the cached step arguments and every captured step graph point into
        the old one (the generation is part of the graph cache key)."""
        self._args = None
        self._ws_gen += 1

    def ensure_rows(self, nrows):
        """Per-row workspace (z, dzr, rowacc) for batches of `nrows` rows.  Every user of the workspace grows
        it here -- the step, and the evaluation paths (encode, data_term, row_log_likelihood, the predictive
        check) -- so that a later graph replay never reads freed buffers."""
        if self.ws.ensure_rows(nrows):
            self._workspace_moved()

    def dense_scratch(self, nrows):
        """fp32 [nrows][D] scratch of the dense kernels (grown like ensure_rows)."""
        w = self.ws
        if w.ensure_dense(max(int(nrows), w.max_rows)):
            self._workspace_moved()
        return w.xdense

    def _guard_scratch(self, nrows):
        """Dense scratch pointer for the exact guard / dense links, or None (guard degrades to drop-and-count)."""
        if self.link == 0 and (not self.exact_guard or 4 * int(nrows) * self.D > self.GUARD_SCRATCH_LIMIT):
            return None
        return self.dense_scratch(nrows)

    def fill_noise(self, step=None, which=3, advance=True):
        """Philox draws for `step`: N(0,1) for v,w,u,s (which&1), Gamma(alpha,1) for the rest (which&2)."""
        step = self.rng_step if step is None else step
        _abi.call("spmf_fill_noise", _ptr(self.noise), _ptr(self.params), self.D, self.K, self.S,
                  self.seed, step, which, _stream())
        if advance:
            self.rng_step = step + 1
        self.launches += (which & 1) + ((which >> 1) & 1)

    def draw_operands(self):
        w = self.ws
        _abi.call("spmf_draw_operands_ranked_m", _ptr(self.params), _ptr(self.noise), _ptr(self.eta), None, self.D,
                  self.K, self.S, _ptr(w.Ap), _ptr(w.EV), _ptr(w.PH), _ptr(w.vsum), _ptr(w.phisum),
                  _ptr(w.scr_d), self.model, _stream())
        self.launches += 5

    def data_term(self, b: DeviceBatch, variant=0):
        """Row pass + batch sums + column pass of `b` for the operands currently in the workspace (API
        path: unormalized_log_prob_parts; the training step issues the same sequence natively), including
        the exact non-finite guard / the dense links."""
        w = self.ws
        self.ensure_rows(b.nrows)
        st = _stream()
        self.reset_guard()
        xd = self._guard_scratch(b.nrows)
        if self.custom_link is not None:
            self.custom_data_term(b, xd, forward_only=True)
            return
        if self.link != 0:
            self.dense_data_term(b, xd)
            return
        b.ensure_csc()
        ev = self.kernel_events
        if ev is not None:
            e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
            e0.record()
        _abi.call("spmf_csr_rows", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum),
                  _ptr(b.lgam), self.inv_xi, int(self.scale_rows), b.nrows, self.D, self.K, self.S,
                  _ptr(w.Ap), _ptr(w.EV), _ptr(w.PH), _ptr(w.vsum), _ptr(w.z), _ptr(w.dzr),
                  _ptr(w.rowacc), variant, _ptr(self.gs), st)
        if xd is not None and self.world_size > 1 and torch.distributed.is_initialized():
            # rows are sharded: if ANY rank met a non-finite entry, every rank needs its dense statistics
            # (the replacement value is the minimum over the whole batch, poisson.py:609)
            mine = self.guard_report()[0] & 1
            t = torch.tensor([float(mine)], device=self.device)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX, group=getattr(self, "process_group", None))
            if t.item() > 0 and not mine:
                _abi.call("spmf_guard_reset", _ptr(self.gs), 1, st)
        if xd is not None:
            _abi.call("spmf_guard_rows_fix", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum), _ptr(b.lgam),
                      self.inv_xi, int(self.scale_rows), b.nrows, self.D, self.K, self.S, _ptr(w.EV), _ptr(w.PH),
                      _ptr(w.z), _ptr(w.dzr), _ptr(w.rowacc), _ptr(xd), _ptr(self.gs), st)
        if ev is not None:
            e1.record()
        _abi.call("spmf_batch_sums", _ptr(w.z), _ptr(w.rowacc), b.nrows, self.K, self.S,
                  _ptr(w.zcolsum), _ptr(w.datasums), _ptr(w.scr_d), st)
        if ev is not None:
            e2.record()
        _abi.call("spmf_csc_cols", _ptr(b.colptr), _ptr(b.crows), _ptr(b.cvals), b.nnz, b.nrows,
                  self.D, self.K, self.S, _ptr(w.z), _ptr(w.dzr), _ptr(w.EV), _ptr(w.PH), _ptr(w.GAp),
                  _ptr(w.GEV), _ptr(w.Gph), variant, st)
        if xd is not None:
            _abi.call("spmf_guard_cols_fix", b.nrows, self.D, self.K, self.S, _ptr(w.EV), _ptr(w.PH), _ptr(w.z),
                      _ptr(w.GEV), _ptr(w.Gph), _ptr(xd), _ptr(self.gs), st)
        if ev is not None:
            e3.record()
            ev.setdefault("csr_rows", []).append((e0, e1, b.nnz, b.nrows))
            ev.setdefault("csc_cols", []).append((e2, e3, b.nnz, b.nrows))
        self.launches += 1 + 4 + 1 + 3 + (2 if xd is not None else 0)   # rows, 4 reduce launches, cols (+3 memsets), guard

    def dense_scatter(self, b: DeviceBatch, xd):
        if b.cols is None:
            raise _abi.SpmfError("the dense links need the batch's CSR arrays (not a hybrid-only upload)")
        _abi.call("spmf_dense_scatter", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), b.nrows, self.D, _ptr(xd), _stream())

    def dense_encode(self, b: DeviceBatch, xd):
        w = self.ws
        _abi.call("spmf_dense_encode", _ptr(xd), _ptr(self.eta), _ptr(b.rowsum), self.inv_xi, int(self.scale_rows),
                  b.nrows, self.D, self.K, self.S, self.link, _ptr(w.Ap), _ptr(w.z), _stream())

    def dense_data_term(self, b: DeviceBatch, xd, forward_only=False):
        """Data term of the links without a closed-form sum(rate) (log_transform / Bernoulli), spmf_dense.cu."""
        w, st = self.ws, _stream()
        self.dense_scatter(b, xd)
        self.dense_encode(b, xd)
        for mode, cond in ((_abi.DENSE_OPTIMISTIC, 0), (_abi.DENSE_STATS, 1), (_abi.DENSE_GUARDED, 1)):
            _abi.call("spmf_dense_rows", _ptr(xd), _ptr(b.rowsum), _ptr(b.lgam), self.inv_xi, int(self.scale_rows),
                      b.nrows, self.D, self.K, self.S, self.link, mode, cond, _ptr(w.EV), _ptr(w.PH), _ptr(w.z),
                      _ptr(w.dzr), _ptr(w.rowacc), _ptr(self.gs), st)
        _abi.call("spmf_batch_sums", _ptr(w.z), _ptr(w.rowacc), b.nrows, self.K, self.S,
                  _ptr(w.zcolsum), _ptr(w.datasums), _ptr(w.scr_d), st)
        self.launches += 2 + 2 + 3 + 2
        if forward_only:
            return
        _abi.call("spmf_zero_col_grads", _ptr(w.GAp), _ptr(w.GEV), _ptr(w.Gph), self.D, self.K, self.S, st)
        _abi.call("spmf_dense_cols", _ptr(xd), _ptr(self.eta), b.nrows, self.D, self.K, self.S, self.link, 1,
                  _ptr(w.z), _ptr(w.dzr), _ptr(w.EV), _ptr(w.PH), _ptr(w.GAp), _ptr(w.GEV), _ptr(w.Gph),
                  _ptr(self.gs), st)
        self.launches += 4

    # ---- user-supplied encoder / decoder callables (poisson.py:94-97) ------------------------------------
    # An arbitrary Python link cannot run inside a CUDA kernel: for those models the DATA TERM (and only it) is
    # evaluated with torch ops on the device, dense over every entry like the reference's own formulation, and
    # differentiated by autograd down to the operand tables (A', EV, phi); sampling, the 12 prior terms, the
    # entropy, the chain rule to the 24 variational tensors and Adam stay in the native kernels.
    def _table_to_sdk(self, tab):
        """[NQ][D][REC] gather-record table -> (S, D, K)."""
        w = self.ws
        perm = torch.tensor(_abi.rec_perm(w.KP, w.SV), device=self.device)
        t = tab[:w.NQ * self.D * w.SV * w.KP].view(w.NQ, self.D, w.SV * w.KP)[:, :, perm]
        return t.view(w.NQ, self.D, w.SV, w.KP).permute(0, 2, 1, 3).reshape(self.S, self.D, w.KP)[..., :self.K]

    def _sdk_to_table(self, t, tab):
        w = self.ws
        perm = torch.tensor(_abi.rec_perm(w.KP, w.SV), device=self.device)
        o = torch.zeros(w.NQ, self.D, w.SV, w.KP, dtype=torch.float32, device=self.device)
        o[:, :, :, :self.K] = t.reshape(w.NQ, w.SV, self.D, self.K).permute(0, 2, 1, 3)
        rec = torch.empty(w.NQ, self.D, w.SV * w.KP, dtype=torch.float32, device=self.device)
        rec[:, :, perm] = o.reshape(w.NQ, self.D, w.SV * w.KP)
        tab[:rec.numel()].copy_(rec.reshape(-1))

    def custom_forward(self, b: DeviceBatch, xd, need_grad):
        """(z, rate, log-likelihood (S,B,D) with the guard of poisson.py:606-616 applied, leaves) for the operands
        in the workspace; leaves = (A', v, phi) as autograd leaves when need_grad."""
        enc, dec = self.custom_link
        w, S, D = self.ws, self.S, self.D
        self.dense_scatter(b, xd)
        x = xd[:b.nrows * D].view(b.nrows, D)
        eta = self.eta[:D]
        A = self._table_to_sdk(w.Ap).contiguous()                                  # a u  (encoder divisor = 1)
        v = (self._table_to_sdk(w.EV) / eta[None, :, None]).transpose(1, 2).contiguous()      # (S,K,D)
        phi = w.PH[:w.NQ * D * w.SV].view(w.NQ, D, w.SV).permute(0, 2, 1).reshape(S, 1, D).contiguous()
        if need_grad:
            A, v, phi = (t.detach().requires_grad_(True) for t in (A, v, phi))
        z = torch.matmul(enc(x), A)                                                # poisson.py:640-643
        if self.scale_rows:
            z = z * (b.rowsum * self.inv_xi)[None, :, None]                        # :644-649
        rate = dec(torch.matmul(z, v)) + phi                                       # :173-177
        lg = torch.lgamma(x + 1.0)
        with torch.no_grad():
            bad = ~torch.isfinite(torch.xlogy(x, rate) - rate - lg)
        one = torch.ones((), dtype=rate.dtype, device=rate.device)
        # log(rate) is only formed where it is used (finite entries with x > 0), so that masked branches do not
        # inject 0 * inf into the gradient
        ll = x * torch.log(torch.where(bad | (x == 0), one, rate)) - torch.where(bad, torch.zeros_like(rate), rate) - lg
        mn = torch.where(bad, torch.zeros_like(ll), ll).min()                      # :606-609 min of the finite portion
        ll = torch.where(bad, mn - 10.0, ll)                                       # :610-616
        return z, rate, ll, (A, v, phi), bad

    def custom_data_term(self, b: DeviceBatch, xd, forward_only=False):
        w, S, D = self.ws, self.S, self.D
        with torch.enable_grad():
            z, rate, ll, leaves, bad = self.custom_forward(b, xd, need_grad=not forward_only)
            if not forward_only:
                gA, gv, gphi = torch.autograd.grad(ll.sum() - 0.5 * (z * z).sum(), leaves)
        with torch.no_grad():
            ll, z = ll.detach(), z.detach()
            ds = torch.zeros(S, 4, dtype=torch.float64, device=self.device)
            ds[:, 0] = ll.sum((1, 2), dtype=torch.float64)      # sum of the log-likelihood, replacement applied
            ds[:, 2] = (z * z).sum((1, 2), dtype=torch.float64)  # -> the HalfNormal(1) prior of z (poisson.py:597-604)
            w.datasums[:w.NQ * 4 * w.SV].copy_(ds.view(w.NQ, w.SV, 4).permute(0, 2, 1).reshape(-1))
            self.last_row_ll = ll.sum(-1, dtype=torch.float64)   # (S,B): WAIC / row_log_likelihood
            self.last_nbad = bad.sum()
            if forward_only:
                return
            self._sdk_to_table(gA, w.GAp)
            self._sdk_to_table(gv.transpose(1, 2) / self.eta[:D][None, :, None], w.GEV)     # d/dEV, EV = eta v
            w.Gph[:w.NQ * D * w.SV].copy_(gphi.reshape(w.NQ, w.SV, D).permute(0, 2, 1).reshape(-1))

    def custom_encode(self, b: DeviceBatch, xd):
        """z (S,B,K) for the operands in the workspace (inference)."""
        self.dense_scatter(b, xd)
        with torch.no_grad():
            x = xd[:b.nrows * self.D].view(b.nrows, self.D)
            z = torch.matmul(self.custom_link[0](x), self._table_to_sdk(self.ws.Ap))
            if self.scale_rows:
                z = z * (b.rowsum * self.inv_xi)[None, :, None]
        return z

    def _step_custom(self, batch, fresh_noise, lr, clip_value, beta1, beta2, eps):
        """The step with a torch data term: native sampling -> operands -> [torch: rate, log-likelihood, autograd]
        -> native backward to the 24 tensors -> Adam."""
        if self.world_size > 1:
            raise _abi.SpmfError("custom encoder / decoder callables are single-GPU only")
        w = self.ws
        self.ensure_rows(batch.nrows)
        xd = self._guard_scratch(batch.nrows)
        if fresh_noise:
            self.fill_noise()
        self.gamma_grad()
        self.draw_operands()
        self.reset_guard()
        self.custom_data_term(batch, xd)
        self.backward_params(batch.nrows)
        if lr is not None:
            self.clear_comm_slack()
            self.adam_step(lr, beta1, beta2, eps, clip_value)
        return w.parts.view(self.S, _abi.NUM_PARTS)

    def gamma_grad(self):
        _abi.call("spmf_gamma_grad", _ptr(self.params), _ptr(self.noise), self.D, self.K, self.S,
                  _ptr(self.dgda), _stream())
        self.launches += 1

    def backward_params(self, batch_rows):
        w = self.ws
        _abi.call("spmf_backward_params_ranked_m", _ptr(self.params), _ptr(self.noise), _ptr(self.dgda),
                  _ptr(self.eta), None, self.D, self.K, self.S, _ptr(w.GAp), _ptr(w.GEV), _ptr(w.Gph), _ptr(w.zcolsum),
                  _ptr(w.datasums), _ptr(w.phisum), float(batch_rows), self.u_tau_scale,
                  self.s_tau_scale, self.decay, self.entropy_weight, self.prior_weight,
                  self.world_size, _ptr(self.grads), _ptr(w.parts), _ptr(w.scr_f), _ptr(w.scr_d),
                  _ptr(self.gs), self.model, _stream())
        self.launches += 9

    def _mark(self, name, start):
        """Phase timing hook (bench): CUDA events on the launching stream around a phase."""
        ev = self.kernel_events
        if ev is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        if start is not None:
            ev.setdefault(name, []).append((start, e, 0, 0))
        return e

    # ------------------------------------------------------------------ one step
    def _step_args(self):
        """The (cached) argument block of spmf_advi_step: everything that does not change per batch."""
        if self._args is None:
            a, w, L = _abi.StepArgs(), self.ws, self.layout
            a.D, a.K, a.S, a.world_size = self.D, self.K, self.S, self.world_size
            a.u_tau_scale, a.s_tau_scale, a.decay = self.u_tau_scale, self.s_tau_scale, self.decay
            a.w_entropy, a.w_prior, a.seed = self.entropy_weight, self.prior_weight, self.seed
            for name in ("params", "grads", "adam_m", "adam_v", "noise", "dgda", "eta"):
                setattr(a, name, _ptr(getattr(self, name)))
            a.n_params, a.comm_off, a.comm_slack = L.n_params, L.comm_off, L.comm_slack
            for name in ("Ap", "EV", "PH", "GAp", "GEV", "Gph", "scr_f", "vsum", "phisum", "zcolsum",
                         "datasums", "parts", "scr_d"):
                setattr(a, name, _ptr(getattr(w, name)))
            if os.environ.get("SPMF_SPLIT_BACKWARD", "1") != "0":
                a.scr_dpre = _ptr(w.scr_dpre)
            if self.stream_mode == "prio":
                self._hot = torch.cuda.Stream(device=self.device, priority=-1)
                self._side = torch.cuda.Stream(device=self.device, priority=0)
                self._sync_events = [torch.cuda.Event() for _ in range(3)]
                for e in self._sync_events:
                    e.record()                       # materialise the cudaEvent_t handles
                a.hot_stream, a.side_stream = self._hot.cuda_stream, self._side.cuda_stream
                a.ev_fork, a.ev_join, a.ev_done = (e.cuda_event for e in self._sync_events)
                self._ev_noise = torch.cuda.Event()
                self._ev_noise.record()
                a.ev_noise = self._ev_noise.cuda_event
                # hybrid step: the GA' GEMM and the cold column pass run next to the hot column pass
                self._aux = [torch.cuda.Stream(device=self.device, priority=-1) for _ in range(2)]
                self._aux_events = [torch.cuda.Event() for _ in range(3)]
                for e in self._aux_events:
                    e.record()
                if os.environ.get("SPMF_AUX_STREAMS", "1") != "0":
                    a.aux_stream1, a.aux_stream2 = (st.cuda_stream for st in self._aux)
                    a.ev_aux_fork, a.ev_aux_join1, a.ev_aux_join2 = (e.cuda_event for e in self._aux_events)
            self._args = a
        return self._args

    def prepare_batch(self, batch: DeviceBatch):
        """Build (once) the form of `batch` this engine's step reads: the hybrid form (ranked CSR/CSC + dense
        bf16 hot block) or the plain CSC copy.  step() does it on first use; resident training loops call
        this up front so that no step pays for it."""
        hybrid = self._runs_hybrid(batch)
        if hybrid:
            batch.ensure_hot(self.rank, self.hot_cols, version=getattr(self, "rank_version", 0))
        elif self.link == 0:
            batch.ensure_csc()
        return hybrid

    def _runs_hybrid(self, batch: DeviceBatch):
        """Whether this engine steps `batch` in the hybrid form."""
        return self.hybrid_ok and self.hot_cols > 0 and self.rank is not None and batch.nnz > 0

    def prime_graph(self, batch: DeviceBatch, fresh_noise=True, lr=None, clip_value=0.0):
        """Capture (without running it) the CUDA graph of this batch's step for the given configuration, so
        that no later step pays the ~ms capture + instantiation.  Needs one eager step of the same
        configuration before (any batch); returns True if a graph is now cached."""
        if not (self.use_graphs and getattr(batch, "_resident", False)):
            return False
        return bool(self.step(batch, fresh_noise=fresh_noise, lr=lr, clip_value=clip_value, _capture_only=True))

    def step(self, batch: DeviceBatch, fresh_noise=True, lr=None, clip_value=0.0, beta1=0.9, beta2=0.999,
             eps=1e-7, _capture_only=False):
        """ONE native call: noise -> operands -> row pass -> column pass -> backward (-> Adam when `lr`
        is given and world_size == 1).  Gamma draws / implicit gradients run on a low-priority side
        stream underneath the gather-bound data-term kernels (stream_mode "prio")."""
        if self.custom_link is not None:
            return self._step_custom(batch, fresh_noise, lr, clip_value, beta1, beta2, eps)
        w = self.ws
        self.ensure_rows(batch.nrows)
        hybrid = self._runs_hybrid(batch)
        if hybrid:
            h = batch.ensure_hot(self.rank, self.hot_cols, version=getattr(self, "rank_version", 0))
            if w.ensure_hybrid(self.hot_cols, batch.nrows):
                self._workspace_moved()
        else:
            if batch.dense_raw is not None:
                raise _abi.SpmfError("this batch was ingested dense for the tile-hybrid step, but the engine for "
                                     f"S={self.S} does not run it; upload it through an uploader made for this engine")
            if batch.cols is None or batch.vals is None:
                raise _abi.SpmfError("this batch was uploaded in hybrid-only form (no CSR arrays) but the engine "
                                     f"for S={self.S} runs the gather step; upload it without a hot split")
            if self.link == 0:
                batch.ensure_csc()
        xd = self._guard_scratch(batch.nrows)
        a = self._step_args()
        a.step_state = _ptr(self.step_state)
        a.link, a.gs, a.xdense, a.xdense_in = self.link, _ptr(self.gs), _ptr(xd), None
        a.model = self.model
        a.dense_raw, a.dense_raw_dtype = _ptr(batch.dense_raw), int(batch.dense_dtype)
        a.z, a.dzr, a.rowacc = _ptr(w.z), _ptr(w.dzr), _ptr(w.rowacc)
        a.inv_xi, a.scale_rows = self.inv_xi, int(self.scale_rows)
        a.fresh_noise, a.rng_step = int(fresh_noise), self.rng_step
        a.rowsum, a.lgam = _ptr(batch.rowsum), _ptr(batch.lgam)
        # (a streamed batch lives in persistent staging: its kernels are sized by the staging capacity so that
        # the captured graph of one slot serves every batch that passes through it; counts are device-side)
        a.nrows, a.nnz = batch.nrows, int(getattr(batch, "_nnz_bound", batch.nnz))
        if hybrid:
            a.rowptr, a.cols, a.vals = _ptr(h.rowptr), _ptr(h.cols), _ptr(h.vals)
            a.colptr, a.crows, a.cvals = _ptr(h.colptr), _ptr(h.crows), _ptr(h.cvals)
            a.rank, a.hot_cols, a.gemm_splits = _ptr(self.rank), int(self.hot_cols), 0
            a.rowmid, a.xhot = _ptr(h.rowmid), _ptr(h.xhot)
            a.t3_qstride = w.t3_qstride
            a.ApT3, a.dzrT3 = _ptr(w.ApT3), _ptr(w.dzrT3)
            a.EVt = _ptr(w.EVt)
        else:
            a.rowptr, a.cols, a.vals = _ptr(batch.rowptr), _ptr(batch.cols), _ptr(batch.vals)
            a.colptr, a.crows, a.cvals = _ptr(batch.colptr), _ptr(batch.crows), _ptr(batch.cvals)
            a.rank, a.hot_cols = None, 0
        # one rank: Adam ends the native step; several ranks: it follows the all-reduce (parallel.allreduce_step)
        do_adam = lr is not None
        # the tensors that never see a data term are stepped under the data term (side stream); with several
        # ranks that is the only Adam inside the native step -- the data-touched block belongs to the exchange
        early = do_adam and self.adam_early and bool(a.scr_dpre)
        a.adam_tail_early = int(early)
        a.adam_lr = float(lr) if (do_adam and (self.world_size == 1 or early)) else 0.0
        a.adam_beta1, a.adam_beta2, a.adam_eps, a.clip_value = beta1, beta2, eps, float(clip_value)
        a.adam_t = self.opt_step + 1
        a.caller_stream = _stream()
        ev = self.kernel_events
        if ev is not None:
            tev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
            for e in tev:
                e.record()
            a.ev_rows0, a.ev_rows1, a.ev_cols0, a.ev_cols1 = (e.cuda_event for e in tev[:4])
            ev.setdefault("csr_rows", []).append((tev[0], tev[1], batch.nnz, batch.nrows))
            ev.setdefault("csc_cols", []).append((tev[2], tev[3], batch.nnz, batch.nrows))
            if hybrid:
                a.ev_gemm0, a.ev_gemm1 = tev[4].cuda_event, tev[5].cuda_event
                ev.setdefault("umma_gemm_gradA", []).append((tev[4], tev[5], batch.nnz, batch.nrows))
                a.ev_tile0, a.ev_tile1 = tev[6].cuda_event, tev[7].cuda_event
                ev.setdefault("hot_tile", []).append((tev[6], tev[7], batch.nnz, batch.nrows))
            else:
                a.ev_gemm0 = a.ev_gemm1 = a.ev_tile0 = a.ev_tile1 = None
        else:
            a.ev_rows0 = a.ev_rows1 = a.ev_cols0 = a.ev_cols1 = a.ev_gemm0 = a.ev_gemm1 = None
            a.ev_tile0 = a.ev_tile1 = None
        if _capture_only:
            return self._launch_step(a, batch, ev is None, hybrid, fresh_noise, capture_only=True)
        self._launch_step(a, batch, ev is None, hybrid, fresh_noise)
        if fresh_noise:
            self.rng_step += 1
        if do_adam:
            self.opt_step += 1
        # kernels issued by spmf_advi_step (counted against the ncu launch lists under profiles/):
        # 17 in gather mode with the split backward (16 with the one-pass backward), +7 tile-hybrid
        # (2 splits, 2 GEMMs, EV tiles, tile kernel, row finalisation); +1 Adam
        self._last_adam = (float(lr), beta1, beta2, eps, float(clip_value)) if do_adam else None
        self.tail_stepped = bool(a.adam_tail_early)     # (multi-GPU tail: the exchange skips those tensors)
        base = 17 if a.scr_dpre else 16
        if self.link != 0:
            base += 6              # scatter (2), encode, two conditional row passes, zeroing -- minus nothing
        elif xd is not None:
            base += 2              # the two conditional guard launches
        n_adam = (1 if (a.adam_lr > 0 and self.world_size == 1) else 0) + (1 if a.adam_tail_early else 0)
        self.launches += base + n_adam + (7 if hybrid else 0)
        return w.parts.view(self.S, _abi.NUM_PARTS)

    def _launch_step(self, a, batch, graphable, hybrid, fresh_noise, capture_only=False):
        """Eager native step, or -- for a RESIDENT batch (cut from a CsrShard: same object, same device
        arrays every epoch) -- one CUDA graph launch (spmf_step_graph_launch).  The first step of every
        configuration runs eagerly: it performs the kernels' lazy one-time initialisation, which must
        not happen under stream capture."""
        cfg = (int(fresh_noise), a.adam_lr > 0, bool(hybrid), int(self.link), int(a.adam_tail_early))
        warm = cfg in self._warm_cfgs
        if not (self.use_graphs and graphable and warm and getattr(batch, "_resident", False)):
            if capture_only:
                return False
            _abi.call("spmf_advi_step", a)
            self._warm_cfgs.add(cfg)
            return
        import ctypes as C
        cache = batch.__dict__.get("_step_graphs")
        if cache is None:
            cache = batch.__dict__["_step_graphs"] = _StepGraphs()
        key = (self._serial, self._ws_gen) + cfg + (batch.nrows, int(a.nnz), getattr(self, "rank_version", 0),
                                                  a.inv_xi, a.scale_rows, a.rowptr, a.xhot)
        h = cache.handles.get(key)
        if h is None:
            cache.drop(self._ws_gen)
            hp = C.c_void_p()
            rc = _abi._lib.spmf_step_graph_create(C.byref(a), C.byref(hp))
            if rc != 0:                      # not capturable in this configuration: stay eager for good
                self.use_graphs = False
                self.graph_error = rc
                if capture_only:
                    return False
                _abi.call("spmf_advi_step", a)
                return
            h = cache.handles[key] = hp.value
        if capture_only:
            return True
        _abi.call("spmf_step_graph_launch", h, a.rng_step, a.adam_t, a.adam_lr, a.adam_beta1, a.adam_beta2,
                  a.adam_eps, a.clip_value, a.caller_stream)
        self.graph_launches += 1

    def loss_and_grad(self, batch: DeviceBatch, fresh_noise=True, variant=0):
        """Fills self.grads and self.ws.parts for `batch`; returns the (S,16) parts tensor (device,
        float64): 12 prior terms in var_list order, logq, z, x, per-draw loss."""
        return self.step(batch, fresh_noise=fresh_noise, lr=None)

    def loss_value(self, parts=None):
        """mean_s [ w_e log q - w_p prior - z - x ]  as a 0-d device tensor."""
        parts = self.ws.parts.view(self.S, _abi.NUM_PARTS) if parts is None else parts
        return parts[:, 15].mean()

    def adam_args(self, n_step=None):
        """spmf_adam_args of the optimiser step the last `step(lr=...)` call took (multi-GPU tail)."""
        lr, b1, b2, eps, clip = self._last_adam
        a = _abi.AdamArgs()
        a.lr, a.beta1, a.beta2, a.eps, a.clip_value, a.grad_scale = lr, b1, b2, eps, clip, 1.0
        a.step = int(self.opt_step if n_step is None else n_step)
        a.params, a.m, a.v = _ptr(self.params), _ptr(self.adam_m), _ptr(self.adam_v)
        return a

    def adam_step(self, lr, beta1=0.9, beta2=0.999, eps=1e-7, clip_value=0.0, grad_scale=1.0):
        self.opt_step += 1
        t = self._mark(None, None)
        _abi.call("spmf_adam_step", _ptr(self.params), _ptr(self.grads), _ptr(self.adam_m),
                  _ptr(self.adam_v), self.layout.n_params, float(lr), beta1, beta2, eps,
                  self.opt_step, float(clip_value), float(grad_scale), _stream())
        self._mark("adam", t)
        self.launches += 1

    def clear_comm_slack(self):
        L = self.layout
        self.grads[L.comm_off: L.comm_off + L.comm_slack].zero_()

    # ------------------------------------------------------------------ helpers
    def set_noise_from(self, noise_dict):
        """Parity hook: load host-provided base noise {var: (S,*shape)} instead of Philox draws."""
        for name, t in noise_dict.items():
            self.layout.noise_view(self.noise, name).copy_(
                torch.as_tensor(t).to(device=self.device, dtype=torch.float32))

    def noise_dict(self):
        return {name: self.layout.noise_view(self.noise, name).clone() for name in self.layout.shapes}

    def parts_dict(self):
        p = self.ws.parts.view(self.S, _abi.NUM_PARTS).cpu()
        return {n: p[:, i] for i, n in enumerate(PART_NAMES)}

    def samples(self):
        out = torch.empty_like(self.noise)
        _abi.call("spmf_sample_m", _ptr(self.params), _ptr(self.noise), self.D, self.K, self.S,
                  _ptr(out), self.model, _stream())
        return {name: self.layout.noise_view(out, name) for name in self.layout.shapes}
