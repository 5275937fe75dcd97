"""`PoissonFactorization` -- host-side mirror of the reference's model surface.

Same names, argument meaning and dict keys as mederrata_spmf/poisson.py::PoissonFactorization
(class at poisson.py:25-717; constructor :56-64), backed by the sm_100a kernels behind the C ABI
(include/spmf_b200.h) instead of a TensorFlow-Probability graph.  The training loop the reference
inherits from bayesianquilts (`fit`, call site tests/spmf_test.py:35-43; legacy `calibrate_advi`,
bin/factorize_csv.py:121-124) is re-created here as thin host code around `AdviEngine`.

Differences that are deliberate:
  * arithmetic is fp32 on the GPU (the reference defaults to float64 on the CPU); parity with the
    float64 oracle is checked at 1e-4 relative;
  * batches may be dense arrays (compacted to CSR by a kernel), scipy.sparse matrices, or
    device-resident `DeviceBatch`es cut from a `CsrShard`;
  * `log_transform=True` (poisson.py:41-42, 52-53) has no closed-form sum(rate): it runs the dense
    CUDA-core kernels of csrc/spmf_dense.cu over every (draw, row, feature) entry;
  * the non-finite guard of poisson.py:606-616 is exact: a step that meets a non-finite
    log-likelihood is re-evaluated densely with the reference's min(finite) - 10 replacement;
  * `horshoe_plus=False` (the reference's own branch fails at construction: misplaced kwarg at
    poisson.py:388) raises -- no silent fallback;
  * custom `encoder_function` / `decoder_function` (poisson.py:94-97) are torch callables; a Python callable
    cannot run inside a CUDA kernel, so such a model evaluates its data term with torch ops + autograd on the
    device (engine.custom_forward) between the native sampling and the native backward / Adam.
"""
from __future__ import annotations

import math
import os
import pickle
from typing import Callable, Dict, Iterable, Optional

import numpy as np
import torch

from . import _abi
from .data import CsrShard, DeviceBatch, as_device_batch, _ptr, _stream
from .engine import AdviEngine
from .variables import VAR_LIST, NORMAL_VARS, var_shapes

LINK_CUSTOM = 64      # host-side only: user-supplied encoder / decoder callables (data term in torch, engine.custom_forward)
CHECKPOINT_VERSION = 1   # layout of the 'training' entry that save_checkpoint adds to state()


def _pickle_module():
    try:
        import dill as _pk          # (custom encoder / decoder callables are dill pickles)
    except ImportError:             # pragma: no cover - dill ships with the image
        _pk = pickle
    return _pk


def _read_state(filename):
    with open(filename, 'rb') as f:
        return _pickle_module().load(f)


def waic_terms(ll):
    """(lppd_i, pwaic_i) from per-observation log-likelihoods ll (S, n): log-mean-exp and the sample
    variance over the S draws."""
    ll = ll.to(torch.float64)
    S = ll.shape[0]
    lppd = torch.logsumexp(ll, 0) - math.log(S)
    pwaic = ll.var(0, unbiased=True) if S > 1 else torch.zeros_like(lppd)
    return lppd, pwaic


LOO_DRAW_CHUNK = 64     # surrogate draws loo() regenerates at a time (bounds its engine memory whatever S is)
LOO_PIT_ACC_BYTES = 1 << 30      # loo_pit()'s default batch keeps its (B, D, 2) fp64 accumulator within 1 GiB
LOO_PIT_VALUES_LIMIT = 1 << 27   # entries loo_pit_values() returns at most (2 GiB of (P-, P+) pairs)


def loo_compare(a, b):
    """Difference of two loo() results over the same rows (e.g. two latent dimensions or links):
    'elpd_diff' = sum_i (a_i - b_i) and 'se_diff' = sqrt(n var(a_i - b_i)) of the pointwise elpd_loo."""
    ea, eb = a['pointwise']['elpd_loo'], b['pointwise']['elpd_loo']
    if ea.numel() != eb.numel():
        raise ValueError(f"loo_compare: the results cover {ea.numel()} and {eb.numel()} rows; they must be the same rows")
    d = ea.to(torch.float64) - eb.to(device=ea.device, dtype=torch.float64)
    n = d.numel()
    var = float(d.var(unbiased=True)) if n > 1 else 0.0
    return {'elpd_diff': float(d.sum()), 'se_diff': math.sqrt(n * var)}


PPC_SAMPLE_LIMIT = 1 << 30      # replicates posterior_predictive_sample materialises at most (4 GiB of int32)
PPC_INTEGER_STATS = ('row_total', 'row_nnz', 'col_total', 'col_sumsq', 'col_nnz', 'total', 'nnz', 'max')


def ppc_p_values(observed, replicated):
    """Posterior predictive p-values from the statistics of posterior_predictive_check.

    Every statistic T uses the mid-p  (#{s: T_rep_s > T_obs} + 0.5 #{s: T_rep_s == T_obs}) / S,  elementwise over
    rows / columns.  The discrepancy is paired per draw: D(x_rep_s, theta_s) against D(x, theta_s).  'col_var' is
    the per-column sample variance over the N rows, (sumsq - total^2 / N) / (N - 1), computed in fp64 from the
    exact integer sums on both sides."""
    S = replicated['discrepancy'].shape[0]

    def mid_p(rep, obs):
        rep, obs = rep.to(torch.float64), obs.to(torch.float64)
        return ((rep > obs).sum(0, dtype=torch.float64) + 0.5 * (rep == obs).sum(0, dtype=torch.float64)) / S

    def col_var(t):
        n = float(observed['row_total'].shape[-1])
        tot, sq = t['col_total'].to(torch.float64), t['col_sumsq'].to(torch.float64)
        return (sq - tot * tot / n) / max(n - 1.0, 1.0)

    out = {k: mid_p(replicated[k], observed[k]) for k in PPC_INTEGER_STATS + ('discrepancy',)}
    out['col_var'] = mid_p(col_var(replicated), col_var(observed))
    return out


class _SurrogateDistribution:
    """Stand-in for `self.surrogate_distribution` (a tfd.JointDistributionNamed in the reference,
    poisson.py:567-569): `.sample(n)` returns a dict of reference-shaped draws."""

    def __init__(self, model):
        self._m = model

    def sample(self, n=None, seed=None):
        m = self._m
        S = 1 if n is None else int(n)
        eng = m._engine_for(S)
        # a sampling call must not move the training stream's Philox counter (fit continues where it was)
        eng.fill_noise(step=(seed if seed is not None else eng.rng_step), advance=seed is None)
        out = {k: v.clone() for k, v in eng.samples().items()}
        if n is None:
            out = {k: v[0] for k, v in out.items()}
        return out

    @property
    def trainable_variables(self):
        return self._m.surrogate_vars

    @property
    def variables(self):
        return self._m.surrogate_vars


class _PriorDistribution:
    """Stand-in for `self.prior_distribution` (tfd.JointDistributionNamed, poisson.py:400-401): the
    horseshoe+ hierarchy of poisson.py:228-377.  `log_prob_parts` is what the energy calls
    (poisson.py:590); `sample` draws ancestrally (diagnostics only -- the training step never samples
    the prior)."""

    def __init__(self, model):
        self._m = model

    def log_prob_parts(self, params):
        return self._m._prior_parts_torch(params)

    def log_prob(self, params=None, **kw):
        return sum(self.log_prob_parts(params if params is not None else kw).values())

    def sample(self, n=None, seed=None):
        m = self._m
        D, K = m.feature_dim, m.latent_dim
        shp = () if n is None else (int(n),)
        gen = torch.Generator(device=m.device)
        gen.manual_seed(int(seed) if seed is not None else 0)
        f64 = dict(device=m.device, dtype=torch.float64)

        def half_normal(scale, shape):
            shape = tuple(scale.shape) if torch.is_tensor(scale) else shp + tuple(shape)
            return (torch.randn(*shape, generator=gen, **f64) * scale).abs()

        def inv_gamma(conc, scale, shape):            # 1 / Gamma(conc, rate=scale)
            g = torch._standard_gamma(torch.full(shp + shape, conc, **f64), generator=gen)
            return scale / g

        ck = m.symmetry_breaking_decay ** torch.arange(K, **f64)[None, :]
        out = {}
        out['u_eta_a'] = inv_gamma(0.5, 1.0, (D, K))
        out['u_tau_a'] = inv_gamma(0.5, 1.0 / m.u_tau_scale ** 2, (1, K))
        out['s_eta_a'] = inv_gamma(0.5, 1.0, (2, D))
        out['s_tau_a'] = inv_gamma(0.5, 1.0 / m.s_tau_scale ** 2, (1, D))
        for name, a in (('u_eta', 'u_eta_a'), ('u_tau', 'u_tau_a'), ('s_eta', 's_eta_a'), ('s_tau', 's_tau_a')):
            out[name] = inv_gamma(0.5, 1.0 / out[a], tuple(out[a].shape[len(shp):])).sqrt()   # SqrtInverseGamma
        out['u'] = half_normal(out['u_eta'] * out['u_tau'] * ck, ())
        out['s'] = half_normal(out['s_eta'] * out['s_tau'], ())
        out['v'] = half_normal(0.1, (K, D))
        out['w'] = half_normal(1.0, (1, D))
        if m._model_id == _abi.MODEL_BERNOULLI:       # Normal, not HalfNormal (bernoulli.py:200-215)
            for k in ('v', 'w'):
                out[k] = out[k] * (torch.randint(0, 2, out[k].shape, generator=gen, device=m.device) * 2 - 1)
        return out


class PoissonFactorization:
    """Sparse (horseshoe) Poisson matrix factorisation, ADVI on B200."""

    bijectors = None
    var_list = []
    s_tau_scale = 1
    _model_id = _abi.MODEL_POISSON

    def __init__(self, latent_dim=None, feature_dim=None, u_tau_scale=0.01, s_tau_scale=1.,
                 symmetry_breaking_decay=0.99, strategy=None, encoder_function=None,
                 decoder_function=None, scale_columns=True, scale_rows=True, log_transform=False,
                 horshoe_plus=True, column_norms=None, count_key='counts',
                 initialize_distributions=True, dtype=torch.float32, device=None,
                 entropy_weight=1.0, prior_weight=1.0, seed=0, process_group=None, hot_density=None,
                 exact_guard=None, **kwargs):
        if not horshoe_plus:
            raise _abi.SpmfError("horshoe_plus=False (AbsHorseshoe priors) has no CUDA path")
        self.link = self._link_id(bool(log_transform))
        # poisson.py:94-97: user-supplied encoder g(x) / decoder f(y) -- torch callables on device tensors
        # ((B,D) -> (B,D) and (S,B,D) -> (S,B,D), differentiable).  A Python callable cannot run inside a CUDA
        # kernel: such a model evaluates its DATA TERM with torch ops + autograd (engine.custom_forward); the
        # other half of the pair defaults to the reference's own function of eta_i (poisson.py:34-54).
        self._custom_link = None
        if encoder_function is not None or decoder_function is not None:
            self._custom_link = (encoder_function or self._default_encoder, decoder_function or self._default_decoder)
            self.link = LINK_CUSTOM
        if exact_guard is None:
            exact_guard = os.environ.get("SPMF_EXACT_GUARD", "1") != "0"
        self.exact_guard = bool(exact_guard)
        if feature_dim is None:
            raise ValueError("feature_dim is required")
        self.scale_rows = scale_rows                      # poisson.py:85-92
        self.scale_columns = scale_columns
        self.horseshoe_plus = horshoe_plus
        self.count_key = count_key
        self.dtype = dtype
        self.symmetry_breaking_decay = symmetry_breaking_decay
        self.log_transform = log_transform
        self.feature_dim = int(feature_dim)
        self.latent_dim = self.feature_dim if latent_dim is None else int(latent_dim)
        self.u_tau_scale = float(u_tau_scale)
        self.s_tau_scale = float(s_tau_scale)
        self.strategy = strategy
        self.process_group = process_group
        self.entropy_weight, self.prior_weight = float(entropy_weight), float(prior_weight)
        self.seed = int(seed)
        self.device = torch.device(device) if device is not None else torch.device("cuda")
        self.eta_i = torch.ones(1, self.feature_dim, dtype=torch.float64)
        self.xi_u_global = 1.
        if column_norms is not None:
            self.eta_i = torch.as_tensor(column_norms, dtype=torch.float64).reshape(1, -1).cpu()
        # columns populated in at least this fraction of the rows form the dense "hot block" whose
        # count products and per-nonzero terms run on the tcgen05 tensor cores (0 = gather kernels only)
        if hot_density is None:
            hot_density = float(os.environ.get("SPMF_HOT_DENSITY", "0.05"))
        self.hot_density = float(hot_density)
        self.col_rank = None        # int32 [D] device tensor: rank of each feature by population
        self.hot_cols = 0
        self.calibrated_expectations = {}
        self._last_data_factory = None
        self._engines: Dict[int, AdviEngine] = {}
        self._pending_counters = {}     # S -> (opt_step, rng_step) of a loaded checkpoint, for engines not created yet
        self._params = None
        if initialize_distributions:
            self.create_distributions()
        print(f"Feature dim: {self.feature_dim} -> Latent dim {self.latent_dim}")   # poisson.py:110-111

    def _default_encoder(self, x):
        """poisson.py:34-43 as a torch callable (used when only a decoder is supplied)."""
        eta = self.eta_i.reshape(-1).to(device=x.device, dtype=x.dtype)
        return torch.log(x / eta + 1.0) if self.log_transform else x / eta

    def _default_decoder(self, y):
        """poisson.py:45-54 as a torch callable (used when only an encoder is supplied)."""
        eta = self.eta_i.reshape(-1).to(device=y.device, dtype=y.dtype)
        return torch.expm1(y * eta) if self.log_transform else y * eta

    @property
    def encoder_function(self):
        return self._custom_link[0] if self._custom_link else self._default_encoder

    @property
    def decoder_function(self):
        return self._custom_link[1] if self._custom_link else self._default_decoder

    @staticmethod
    def _link_id(log_transform):
        """SPMF_LINK_* of this model class (poisson.py:34-54, 177-183)."""
        return _abi.LINK_POISSON_LOG if log_transform else _abi.LINK_POISSON

    # ------------------------------------------------------------------ distributions
    def create_distributions(self):
        """poisson.py:212-573: (re)initialise the 24 variational tensors; priors are implicit in
        the kernels (spmf_model.cuh)."""
        self.bijectors = {k: 'softplus' for k in VAR_LIST}          # all Softplus, poisson.py:215-224,297-301
        self.var_list = list(VAR_LIST)                               # poisson.py:572
        self._engines = {}
        self._pending_counters = {}
        self._params = None
        eng = self._engine_for(1)
        self._params = eng.params
        self.surrogate_distribution = _SurrogateDistribution(self)
        self.prior_distribution = _PriorDistribution(self)
        self.set_calibration_expectations()

    def _engine_for(self, S) -> AdviEngine:
        S = int(S)
        if S not in self._engines:
            world = 1
            if self.process_group is not None or (torch.distributed.is_available()
                                                  and torch.distributed.is_initialized()):
                world = torch.distributed.get_world_size(self.process_group)
            eng = AdviEngine(self.feature_dim, self.latent_dim, S, self.device, self.u_tau_scale,
                             self.s_tau_scale, self.symmetry_breaking_decay, self.scale_rows,
                             self.entropy_weight, self.prior_weight, world, self.seed, link=self.link,
                             exact_guard=self.exact_guard, model=self._model_id)
            eng.process_group = self.process_group
            eng.custom_link = self._custom_link
            if self._params is not None:                # engines share parameters / optimiser state
                first = next(iter(self._engines.values()))
                if eng.params.data_ptr() != first.params.data_ptr():
                    from . import p2p
                    p2p.release(eng.params)
                    p2p.release(eng.grads)
                eng.params, eng.grads = first.params, first.grads
                eng.adam_m, eng.adam_v = first.adam_m, first.adam_v
            self._engines[S] = eng
            self._push_scales(eng)
            if S in self._pending_counters:
                eng.opt_step, eng.rng_step = self._pending_counters.pop(S)
        return self._engines[S]

    def _push_scales(self, eng):
        D = self.feature_dim
        eta = self.eta_i.reshape(-1).to(torch.float32)
        eng.eta[:D].copy_(eta)                                  # decoder scale (poisson.py:52-54)
        if self.log_transform or self._custom_link:
            eng.eta[D:].fill_(1.0)                              # encoder log(x/eta + 1) / g(x) acts on the counts
        else:
            eng.eta[D:].copy_(eta)                              # encoder x/eta folded into A'
        xi = float(self.xi_u_global)
        eng.inv_xi = 1.0 / xi if self.scale_rows else 1.0
        eng.scale_rows = bool(self.scale_rows)
        eng.rank, eng.hot_cols = self.col_rank, int(self.hot_cols)
        eng.rank_version = getattr(self, "_rank_version", 0)

    @property
    def surrogate_vars(self):
        """24 tensors, reference order (2 per var_list entry), views into the flat device buffer."""
        eng = self._engine_for(1)
        return list(eng.layout.views(eng.params).values())

    def surrogate_parameters(self):
        eng = self._engine_for(1)
        return eng.layout.views(eng.params)

    # ------------------------------------------------------------------ compute_scales
    def compute_scales(self, data_factory, compute_normalization=True, n=None):
        """poisson.py:113-154.  `data_factory()` yields batches (dicts keyed by count_key); a
        `CsrShard` may be passed directly."""
        self._last_data_factory = data_factory
        if not (self.scale_columns and compute_normalization):
            return
        print("Looping through the entire dataset once to get some stats")          # poisson.py:116
        colsum = torch.zeros(self.feature_dim, dtype=torch.float64, device=self.device)
        colnnz = torch.zeros(self.feature_dim, dtype=torch.float32, device=self.device)
        nrows_seen = 0
        if isinstance(data_factory, CsrShard):
            shards = [data_factory]
        else:
            shards = []
            for batch in iter(data_factory()):
                c = batch[self.count_key] if isinstance(batch, dict) else batch
                if isinstance(c, DeviceBatch):
                    nrows_seen += c.nrows
                    n0 = int(c.rowptr[0].item())
                    cols, vals = c.cols[n0:n0 + c.nnz], c.vals[n0:n0 + c.nnz]
                    _abi.call("spmf_csr_colstats", _ptr(cols), _ptr(vals), c.nnz, self.feature_dim,
                              _ptr(colsum), _ptr(colnnz), _stream())
                else:
                    shards.append(c if isinstance(c, CsrShard) else
                                  (CsrShard.from_scipy(c, self.device) if hasattr(c, "tocsr")
                                   else CsrShard.from_dense(c, self.device)))
        for sh in shards:
            cs, cn = sh.column_stats()
            colsum += cs
            colnnz += cn
            nrows_seen += sh.nrows
        nrows_all = torch.tensor([float(nrows_seen)], dtype=torch.float64, device=self.device)
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            torch.distributed.all_reduce(colsum, group=self.process_group)
            torch.distributed.all_reduce(colnnz, group=self.process_group)
            torch.distributed.all_reduce(nrows_all, group=self.process_group)
        self._choose_hot_columns(colnnz, float(nrows_all.item()))
        self._set_scales_from_stats(colsum.cpu(), colnnz.cpu())

    def _hot_spec(self, eng):
        """(rank, H, version) for the streaming uploader, decided by the engine that will consume
        the batches: the hybrid form is only built when THAT engine (its S decides KP*SV) runs the
        hybrid step; otherwise batches keep their plain CSR + CSC form."""
        if eng.hybrid_ok and eng.hot_cols > 0 and eng.rank is not None:
            return (eng.rank, int(eng.hot_cols), getattr(eng, "rank_version", 0))
        return None

    def _choose_hot_columns(self, colnnz, nrows):
        """Column ordering for the hybrid step: features ranked by how many rows populate them; the
        H columns populated in >= hot_density of the rows form the tensor-core block.  Identical on
        every rank (computed from the all-reduced counts)."""
        self.col_rank, self.hot_cols = None, 0
        if self.link != _abi.LINK_POISSON:
            return                      # dense links: no closed form, no hot / cold split
        self._rank_version = getattr(self, "_rank_version", 0) + 1     # invalidates cached hybrid forms
        # (whether a given engine uses the hot block is its own decision: hybrid_ok depends on S)
        if self.hot_density <= 0 or nrows <= 0 or self.latent_dim > _abi.MAX_TILE_K:
            return
        order = torch.argsort(colnnz.to(torch.float64), descending=True, stable=True)
        H = int((colnnz.to(torch.float64) >= self.hot_density * nrows).sum().item())
        if H < 64:                      # not worth a GEMM
            return
        rank = torch.empty(self.feature_dim, dtype=torch.int32, device=self.device)
        rank[order] = torch.arange(self.feature_dim, dtype=torch.int32, device=self.device)
        self.col_rank, self.hot_cols = rank, H

    def _set_scales_from_stats(self, colsum, colnnz):
        colmeans_nonzero = colsum.to(torch.float64) / colnnz.to(torch.float64)      # :136-138
        rowmean_nonzero = colmeans_nonzero.sum()                                     # :139-140
        self.eta_i = torch.where(colmeans_nonzero > 1, colmeans_nonzero,
                                 torch.ones_like(colmeans_nonzero)).reshape(1, -1)   # :142-149
        self.xi_u_global = float(rowmean_nonzero) if self.scale_rows else 1.          # :151-154
        for eng in self._engines.values():
            self._push_scales(eng)

    # ------------------------------------------------------------------ encoder / decoder surface
    def set_calibration_expectations(self, samples=24, seed=12345):
        """[EXT] BayesianModel.set_calibration_expectations (called at poisson.py:573): posterior
        means of every variable, estimated from surrogate draws."""
        draws = self.surrogate_distribution.sample(samples, seed=seed)
        self.calibrated_expectations = {k: v.mean(0) for k, v in draws.items()}

    def encoding_matrix(self, u=None, s=None):
        """A = (s0/(s0+s1)) u, shape (...,D,K)   (poisson.py:652-666)."""
        u = self.calibrated_expectations['u'] if u is None else u
        s = self.calibrated_expectations['s'] if s is None else s
        weights = s / s.sum(-2, keepdim=True)
        return weights[..., 0, :].unsqueeze(-1) * u

    def decoding_matrix(self, v=None):
        """poisson.py:668-678."""
        return self.calibrated_expectations['v'] if v is None else v

    def intercept_matrix(self, w=None, s=None):
        """phi = eta (s1/(s0+s1)) w, shape (...,1,D)   (poisson.py:680-701)."""
        w = self.calibrated_expectations['w'] if w is None else w
        s = self.calibrated_expectations['s'] if s is None else s
        weights = s / s.sum(-2, keepdim=True)
        eta = self.eta_i.to(device=w.device, dtype=w.dtype)
        return eta * weights[..., 1, :].unsqueeze(-2) * w

    def _operands_from_theta(self, eng, u, v, w, s):
        """Pack explicit draws (S leading axis) into the kernels' gather layout."""
        S, D, K = eng.S, self.feature_dim, self.latent_dim
        ws = eng.ws
        f32 = dict(device=self.device, dtype=torch.float32)
        eta = self.eta_i.reshape(-1).to(**f32)
        u, v, w, s = (torch.as_tensor(t).to(**f32) for t in (u, v, w, s))
        if u.dim() == 2:
            u, v, w, s = u[None], v[None], w[None], s[None]
        a = s[:, 0, :] / (s[:, 0, :] + s[:, 1, :])
        b = 1.0 - a
        eta_enc = torch.ones_like(eta) if (self.log_transform or self._custom_link) else eta
        Ap = a[:, :, None] * u / eta_enc[None, :, None]              # (S,D,K)
        EV = eta[None, :, None] * v.transpose(-1, -2)                # (S,D,K)
        PH = eta[None, :] * b * w[:, 0, :]                           # (S,D)

        perm = torch.tensor(_abi.rec_perm(ws.KP, ws.SV), device=self.device)

        def pack(t):   # (S,D,K) -> [NQ][D][REC] in the kernels' record order
            o = torch.zeros(ws.NQ, D, ws.SV, ws.KP, **f32)
            o[:, :, :, :K] = t.view(ws.NQ, ws.SV, D, K).permute(0, 2, 1, 3)
            rec = torch.empty(ws.NQ, D, ws.SV * ws.KP, **f32)
            rec[:, :, perm] = o.reshape(ws.NQ, D, ws.SV * ws.KP)
            return rec.reshape(-1)
        ws.Ap.copy_(pack(Ap))
        ws.EV.copy_(pack(EV))
        ws.PH.copy_(PH.view(ws.NQ, ws.SV, D).permute(0, 2, 1).reshape(-1))
        ws.vsum.copy_(ws.EV.view(ws.NQ, D, ws.KP * ws.SV).to(torch.float64).sum(1).reshape(-1))
        ws.phisum.copy_(ws.PH.view(ws.NQ, D, ws.SV).to(torch.float64).sum(1).reshape(-1))

    def _unpack_rows(self, eng, flat, nrows):
        ws = eng.ws
        perm = torch.tensor(_abi.rec_perm(ws.KP, ws.SV), device=flat.device)
        t = flat[:ws.NQ * nrows * ws.KP * ws.SV].view(ws.NQ, nrows, ws.SV * ws.KP)[:, :, perm]
        t = t.view(ws.NQ, nrows, ws.SV, ws.KP)
        return t.permute(0, 2, 1, 3).reshape(eng.S, nrows, ws.KP)[..., :self.latent_dim]

    def encode(self, x, u=None, s=None):
        """z = (x/eta) A * rowsum(x)/xi, shape (...,B,K)   (poisson.py:623-650)."""
        u = self.calibrated_expectations['u'] if u is None else u
        s = self.calibrated_expectations['s'] if s is None else s
        batched = torch.as_tensor(u).dim() == 3
        S = u.shape[0] if batched else 1
        eng = self._engine_for(S)
        b = as_device_batch(x, self.device, self.feature_dim)
        eng.ensure_rows(b.nrows)
        D, K = self.feature_dim, self.latent_dim
        zeros_v = torch.zeros((S, K, D) if batched else (K, D), device=self.device)
        zeros_w = torch.zeros((S, 1, D) if batched else (1, D), device=self.device)
        self._operands_from_theta(eng, u, zeros_v, zeros_w, s)
        ws = eng.ws
        if self._custom_link:
            z = eng.custom_encode(b, eng._guard_scratch(b.nrows))
            return z if batched else z[0]
        if self.link & 1:              # log(x/eta + 1) encoder: dense kernel (spmf_dense.cu)
            xd = eng._guard_scratch(b.nrows)
            eng.dense_scatter(b, xd)
            eng.dense_encode(b, xd)
        else:
            _abi.call("spmf_csr_encode", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum),
                      eng.inv_xi, int(self.scale_rows), b.nrows, D, K, S, _ptr(ws.Ap), _ptr(ws.z), _stream())
        z = self._unpack_rows(eng, ws.z, b.nrows).clone()
        return z if batched else z[0]

    # ------------------------------------------------------------------ energy
    def unormalized_log_prob_parts(self, data, prior_weight=1., **params):
        """poisson.py:582-621: dict of 14 (S,) terms -- 12 priors, 'z', 'x' -- evaluated by the
        CUDA data-term kernels for explicit draws `params` (each with a leading sample axis)."""
        S = params['u'].shape[0] if params['u'].dim() == 3 else 1
        eng = self._engine_for(S)
        b = as_device_batch(data[self.count_key] if isinstance(data, dict) else data, self.device)
        self._operands_from_theta(eng, params['u'], params['v'], params['w'], params['s'])
        eng.data_term(b)
        x_part, z_part = self._data_parts(eng, b.nrows)
        parts = {k: v * prior_weight for k, v in self._prior_parts_torch(params).items()}
        parts['z'] = z_part
        parts['x'] = x_part
        return parts

    def _data_parts(self, eng, nrows):
        """('x', 'z') parts of the last eng.data_term(): closed-form assembly, or -- if the exact guard
        fired or the link is dense -- sum over the finite entries + (#non-finite) * (min(finite) - 10)
        (poisson.py:606-619).  Multi-rank: rows are sharded, so sums / counts are all-reduced and the
        minimum is the GLOBAL one, as the reference's single (S,B,D) tensor would give."""
        ws, S = eng.ws, eng.S
        ds = ws.datasums.view(ws.NQ, 4, ws.SV).permute(0, 2, 1).reshape(S, 4).contiguous().clone()
        flag, nbad, min_val = eng.guard_report()
        dist_on = torch.distributed.is_available() and torch.distributed.is_initialized() and eng.world_size > 1
        rows = torch.tensor([float(nrows)], dtype=torch.float64, device=self.device)
        if dist_on:
            t = torch.tensor([float(flag != 0), -float(min_val)], dtype=torch.float64, device=self.device)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX, group=self.process_group)
            min_val = -float(t[1].item())        # (eng.data_term made the flag collective already)
            torch.distributed.all_reduce(ds, group=self.process_group)
            torch.distributed.all_reduce(rows, group=self.process_group)
        n = float(rows.item())
        if flag:
            x_part = ds[:, 0] + ds[:, 3] * min_val
        else:
            x_part = ds[:, 0] - ds[:, 1] - n * ws.phisum.view(S)
        z_part = n * self.latent_dim * 0.5 * math.log(2.0 / math.pi) - 0.5 * ds[:, 2]
        return x_part, z_part

    def unormalized_log_prob(self, data=None, prior_weight=1., **params):
        # poisson.py:575-580 -- the caller's prior_weight is discarded there; kept for parity.
        parts = self.unormalized_log_prob_parts(data, prior_weight=1., **params)
        return sum(parts.values())

    def _prior_parts_torch(self, th):
        """Prior terms for explicit draws (API path only; the training step uses the fused kernel).
        Small O(S*D*K) torch expressions on the device -- poisson.py:225-377."""
        f64 = dict(device=self.device, dtype=torch.float64)
        th = {k: torch.as_tensor(v).to(**f64) for k, v in th.items()}
        th = {k: (v[None] if v.dim() == 2 else v) for k, v in th.items()}
        c0, lgh = 0.5 * math.log(2.0 / math.pi), math.lgamma(0.5)
        ck = self.symmetry_breaking_decay ** torch.arange(self.latent_dim, **f64)[None, :]
        red = lambda t: t.sum((-1, -2))
        hn = lambda y, sc: c0 - torch.log(sc) - 0.5 * (y / sc) ** 2
        ig = lambda y, c, b: c * torch.log(b) - math.lgamma(c) - (c + 1) * torch.log(y) - b / y
        sig = lambda y, c, b: ig(y * y, c, b) + torch.log(2 * y)
        one = torch.ones((), **f64)
        return {
            'v': red(self._vw_prior(th['v'], 0.1 * one)), 'w': red(self._vw_prior(th['w'], one)),
            'u': red(hn(th['u'], th['u_eta'] * th['u_tau'] * ck)),
            'u_eta': red(sig(th['u_eta'], 0.5, 1.0 / th['u_eta_a'])),
            'u_tau': red(sig(th['u_tau'], 0.5, 1.0 / th['u_tau_a'])),
            's_eta': red(sig(th['s_eta'], 0.5, 1.0 / th['s_eta_a'])),
            's_tau': red(sig(th['s_tau'], 0.5, 1.0 / th['s_tau_a'])),
            's': red(hn(th['s'], th['s_eta'] * th['s_tau'])),
            'u_eta_a': red(ig(th['u_eta_a'], 0.5, one)),
            'u_tau_a': red(ig(th['u_tau_a'], 0.5, one / self.u_tau_scale ** 2)),
            's_eta_a': red(ig(th['s_eta_a'], 0.5, one)),
            's_tau_a': red(ig(th['s_tau_a'], 0.5, one / self.s_tau_scale ** 2)),
        }

    @staticmethod
    def _vw_prior(y, sc):
        """HalfNormal(scale) log-density of v and w (poisson.py:229-242)."""
        return 0.5 * math.log(2.0 / math.pi) - torch.log(sc) - 0.5 * (y / sc) ** 2

    def log_likelihood_components(self, s, u, v, w, data, *args, **kwargs):
        """poisson.py:156-184: {'log_likelihood','rate'}, both (S,B,D) -- dense by definition, so
        this diagnostic surface materialises them with torch ops on the device; the training step
        never calls it."""
        c = data[self.count_key] if isinstance(data, dict) else data
        x = torch.as_tensor(c.toarray() if hasattr(c, "toarray") else c).to(self.device, torch.float32)
        f32 = dict(device=self.device, dtype=torch.float32)
        s, u, v, w = (torch.as_tensor(t).to(**f32) for t in (s, u, v, w))
        z = self.encode(x, u, s)
        if self._custom_link:
            rate = self._custom_link[1](torch.matmul(z, v)) + self.intercept_matrix(w, s)
            return {'log_likelihood': self._log_prob(x, rate), 'rate': rate}
        lin = torch.matmul(z, v) * self.eta_i.to(**f32)
        rate = (torch.expm1(lin) if self.log_transform else lin) + self.intercept_matrix(w, s)   # :52-54, :177
        return {'log_likelihood': self._log_prob(x, rate), 'rate': rate}

    @staticmethod
    def _log_prob(x, rate):
        """tfd.Poisson(rate).log_prob(x)  (poisson.py:178-183)."""
        return torch.xlogy(x, rate) - rate - torch.lgamma(x + 1.0)

    def predictive_distribution(self, s, u, v, w, data, *args, **kwargs):
        """poisson.py:187-210 (the reference reduces a key 'll' that does not exist; here 'll' is
        the log-likelihood summed over the trailing (B,D) axes when draws carry a sample axis)."""
        out = self.log_likelihood_components(s=s, u=u, v=v, w=w, data=data)
        if torch.as_tensor(u).dim() > 2:
            out['ll'] = out['log_likelihood'].sum((-1, -2))
        return out

    def row_log_likelihood(self, data, sample_size=32, seed=None, **params):
        """Per-row Poisson log-likelihood of every draw, shape (S, B): sum_d log Poisson(x_bd | lambda_sbd),
        i.e. poisson.py:156-184's 'log_likelihood' summed over the feature axis, evaluated by the CUDA
        row pass (sum x log lambda - lgamma(x+1) gathered over the nonzeros; sum_d lambda in closed
        form) without materialising (S,B,D).  `params`: explicit draws of s, u, v, w with a leading
        sample axis; default: `sample_size` draws of the surrogate posterior."""
        if not params:
            params = self.surrogate_distribution.sample(int(sample_size), seed=seed)
        u = torch.as_tensor(params['u'])
        S = u.shape[0] if u.dim() == 3 else 1
        eng = self._engine_for(S)
        b = self._csr_batch(data, "row_log_likelihood")
        self._operands_from_theta(eng, params['u'], params['v'], params['w'], params['s'])
        return self._row_ll(eng, b)

    def _csr_batch(self, data, who):
        c = data[self.count_key] if isinstance(data, dict) else data
        b = c if isinstance(c, DeviceBatch) else as_device_batch(c, self.device, self.feature_dim)
        if b.cols is None:
            raise ValueError(f"{who} needs a batch with its CSR arrays (not a hybrid-only upload)")
        return b

    def _row_ll(self, eng, b):
        """(S, B) float64 per-row log-likelihoods of batch `b` for the operand tables currently in `eng`'s
        workspace: the CUDA row pass (sparse link), the dense row pass (other links) or the torch data term of
        custom callables."""
        S = eng.S
        eng.ensure_rows(b.nrows)
        ws = eng.ws
        if self._custom_link:
            eng.reset_guard()
            eng.custom_data_term(b, eng._guard_scratch(b.nrows), forward_only=True)
            return eng.last_row_ll
        if self.link != _abi.LINK_POISSON:        # dense links: per-row sums over every entry (spmf_dense.cu)
            eng.reset_guard()
            eng.dense_data_term(b, eng._guard_scratch(b.nrows), forward_only=True)
            ra = ws.rowacc[:ws.NQ * b.nrows * 4 * ws.SV].view(ws.NQ, b.nrows, 4, ws.SV).to(torch.float64)
            return ra[:, :, 0, :].permute(0, 2, 1).reshape(S, b.nrows)
        _abi.call("spmf_csr_rows", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum), _ptr(b.lgam),
                  eng.inv_xi, int(self.scale_rows), b.nrows, self.feature_dim, self.latent_dim, S,
                  _ptr(ws.Ap), _ptr(ws.EV), _ptr(ws.PH), _ptr(ws.vsum), _ptr(ws.z), _ptr(ws.dzr),
                  _ptr(ws.rowacc), 0, None, _stream())
        ra = ws.rowacc[:ws.NQ * b.nrows * 4 * ws.SV].view(ws.NQ, b.nrows, 4, ws.SV).to(torch.float64)
        ll = (ra[:, :, 0, :] - ra[:, :, 1, :]).permute(0, 2, 1).reshape(S, b.nrows)
        return ll - ws.phisum.view(S, 1)

    def waic(self, data=None, sample_size=32, batch_size=None, seed=12345):
        """[EXT] BayesianModel.waic() (notebooks/factorizing_random_noise.ipynb:447-453): widely applicable
        information criterion over the ROWS of `data` with `sample_size` surrogate draws (the same draws
        for every batch): lppd_i = log mean_s exp(ll_si), pwaic_i = var_s(ll_si), waic = -2 sum_i
        (lppd_i - pwaic_i), se = 2 sqrt(n var_i(lppd_i - pwaic_i)).  Returns the reference's dict
        {'waic', 'se', 'lppd', 'pwaic'}.  `data`: a batch factory as for fit(), a CsrShard, or one
        batch / array; default: the factory last given to fit() / compute_scales()."""
        batches = self._batches_of(data, batch_size, "waic()")
        draws = self.surrogate_distribution.sample(int(sample_size), seed=seed)
        acc = torch.zeros(4, dtype=torch.float64, device=self.device)     # lppd, pwaic, elpd, elpd^2
        n = 0
        for batch in batches:
            ll = self.row_log_likelihood(batch, **draws)
            stats = waic_terms(ll)
            elpd = stats[0] - stats[1]
            acc += torch.stack([stats[0].sum(), stats[1].sum(), elpd.sum(), (elpd * elpd).sum()])
            n += ll.shape[1]
        lppd, pwaic, e1, e2 = (float(t) for t in acc.cpu())
        var = max(e2 / n - (e1 / n) ** 2, 0.0) * (n / (n - 1.0) if n > 1 else 1.0)
        return {'waic': -2.0 * e1, 'se': 2.0 * math.sqrt(n * var), 'lppd': lppd, 'pwaic': pwaic}

    def loo(self, data=None, sample_size=1000, batch_size=None, seed=12345, **params):
        """Pareto-smoothed importance-sampling leave-one-out cross-validation (PSIS-LOO, Vehtari, Gelman & Gabry
        2017) over the ROWS of `data`, with the Pareto k-hat diagnostic of every row: where k-hat is above
        `khat_threshold`, that row's estimate is not to be trusted.

        `data` is taken as by waic().  Draws: explicit s, u, v, w with a leading sample axis, else `sample_size`
        surrogate draws; the same draws serve every batch.  Surrogate draws are taken in chunks of LOO_DRAW_CHUNK:
        chunk c holds exactly the draws surrogate_distribution.sample(n_c, seed=seed + c) returns.  Draws are
        regenerated per batch and chunk, so memory stays at one chunk's engine and one batch's [B][S] fp64
        log-likelihoods whatever S is (at most LOO_MAX_S).  The per-row log-likelihoods come from the row pass of
        row_log_likelihood; the smoothing runs in one CUDA kernel per batch (spmf_psis_loo, csrc/spmf_loo.cu).
        Neither rng_step nor opt_step moves.  Under torch.distributed each rank evaluates its own shard.

        Returns a dict: 'elpd_loo' = sum_i elpd_i, 'se' = sqrt(n var(elpd_i)), 'p_loo' = sum_i (lppd_i - elpd_i),
        'looic' = -2 elpd_loo, 'lppd' = sum_i lppd_i, 'khat_threshold' = min(1 - 1/log10(S), 0.7),
        'n_khat_above' (rows above it, k-hat = inf included), 'n_nonfinite' (rows whose elpd is not finite: a
        draw of zero likelihood gives -inf, a NaN or +inf log-likelihood gives NaN), and 'pointwise': device
        tensors 'elpd_loo', 'p_loo' (float64) and 'khat' (float32) of shape (N,), in row order.  Sums over rows
        run in batch order."""
        batches = self._batches_of(data, batch_size, "loo()")
        theta, S = self._loo_draws(sample_size, params, "loo()")
        dev, f64 = self.device, torch.float64
        acc = torch.zeros(4, dtype=f64, device=dev)     # elpd, elpd^2, lppd, p_loo
        elpd_all, ploo_all, khat_all = [], [], []
        for batch in batches:
            b = self._csr_batch(batch, "loo()")
            if b.nrows == 0:
                continue
            ll = self._loo_row_ll(b, S, seed, theta)
            elpd = torch.empty(b.nrows, dtype=f64, device=dev)
            lppd = torch.empty(b.nrows, dtype=f64, device=dev)
            khat = torch.empty(b.nrows, dtype=torch.float32, device=dev)
            _abi.call("spmf_psis_loo", _ptr(ll), S, b.nrows, S, _ptr(elpd), _ptr(lppd), _ptr(khat), _stream())
            ploo = lppd - elpd
            acc += torch.stack([elpd.sum(), (elpd * elpd).sum(), lppd.sum(), ploo.sum()])
            elpd_all.append(elpd)
            ploo_all.append(ploo)
            khat_all.append(khat)
        if not elpd_all:
            raise ValueError("loo(): the data holds no rows")
        elpd, ploo, khat = torch.cat(elpd_all), torch.cat(ploo_all), torch.cat(khat_all)
        n = elpd.numel()
        e1, e2, lppd, p_loo = (float(t) for t in acc.cpu())
        var = max(e2 / n - (e1 / n) ** 2, 0.0) * (n / (n - 1.0) if n > 1 else 1.0)
        threshold = min(1.0 - 1.0 / math.log10(S), 0.7) if S > 1 else -math.inf
        return {'elpd_loo': e1, 'se': math.sqrt(n * var), 'p_loo': p_loo, 'looic': -2.0 * e1, 'lppd': lppd,
                'khat_threshold': threshold, 'n_khat_above': int((khat > threshold).sum()),
                'n_nonfinite': int((~torch.isfinite(elpd)).sum()),
                'pointwise': {'elpd_loo': elpd, 'p_loo': ploo, 'khat': khat}}

    def _loo_row_ll(self, b, S, seed, theta):
        """[B][S] fp64 per-row log-likelihoods of batch `b` for loo(): draws in chunks of LOO_DRAW_CHUNK, chunk c
        either the Normal draws sample(n_c, seed + c) makes (theta None, regenerated here without moving rng_step)
        or the slice of the explicit draws `theta` (dict of s, u, v, w with a leading sample axis)."""
        ll = torch.empty(b.nrows, S, dtype=torch.float64, device=self.device)
        for c, c0 in enumerate(range(0, S, LOO_DRAW_CHUNK)):
            nc = min(LOO_DRAW_CHUNK, S - c0)
            eng = self._engine_for(nc)
            if theta is None:
                eng.fill_noise(step=int(seed) + c, which=AdviEngine.NOISE_NORMAL, advance=False)
                eng.draw_operands()
            else:
                self._operands_from_theta(eng, *(theta[k][c0:c0 + nc] for k in ('u', 'v', 'w', 's')))
            ll[:, c0:c0 + nc].copy_(self._row_ll(eng, b).t())
        return ll

    # ------------------------------------------------------------------ LOO-PIT
    def _loo_draws(self, sample_size, params, who):
        """(theta, S) of loo() and loo_pit(): explicit draws (leading sample axis) or `sample_size` surrogate draws."""
        if params:
            theta = {k: torch.as_tensor(params[k]) for k in ('s', 'u', 'v', 'w')}
            if theta['u'].dim() == 2:
                theta = {k: t[None] for k, t in theta.items()}
            S = theta['u'].shape[0]
        else:
            theta, S = None, int(sample_size)
        if not 1 <= S <= _abi.LOO_MAX_S:
            raise ValueError(f"{who} takes 1 to {_abi.LOO_MAX_S} draws, got {S}")
        return theta, S

    def _loo_pit_batch(self, b, S, seed, theta, rates=None):
        """(P-, P+) of every entry of batch `b` in an fp64 (B, D, 2) tensor, the per-entry invalid draw counts
        (B, D) and the batch's (elpd, khat): _loo_row_ll, spmf_psis_loo_lw, then a second pass over the same draw
        chunks that regenerates the operands, densifies and encodes the batch as _ppc_pass does and calls
        spmf_loo_pit_accum (csrc/spmf_pit.cu).  `rates` (a list, for checking): receives every chunk's (n_c, B, D)
        fp32 rates as the kernel formed them."""
        if self._custom_link:
            raise _abi.SpmfError("LOO-PIT has no CUDA path for custom encoder / decoder callables")
        dev, f64, B, D = self.device, torch.float64, b.nrows, self.feature_dim
        ll = self._loo_row_ll(b, S, seed, theta)
        lw = torch.empty(B, S, dtype=f64, device=dev)
        elpd = torch.empty(B, dtype=f64, device=dev)
        lppd = torch.empty(B, dtype=f64, device=dev)
        khat = torch.empty(B, dtype=torch.float32, device=dev)
        st = _stream()
        _abi.call("spmf_psis_loo_lw", _ptr(ll), S, B, S, _ptr(elpd), _ptr(lppd), _ptr(khat), _ptr(lw), S, st)
        del ll
        acc = torch.zeros(B, D, 2, dtype=f64, device=dev)
        inv = torch.zeros(B, D, dtype=torch.int32, device=dev)
        for c, c0 in enumerate(range(0, S, LOO_DRAW_CHUNK)):
            nc = min(LOO_DRAW_CHUNK, S - c0)
            eng = self._engine_for(nc)
            if theta is None:
                eng.fill_noise(step=int(seed) + c, which=AdviEngine.NOISE_NORMAL, advance=False)
                eng.draw_operands()
            else:
                self._operands_from_theta(eng, *(theta[k][c0:c0 + nc] for k in ('u', 'v', 'w', 's')))
            eng.ensure_rows(B)
            xd = eng.dense_scratch(B)
            ws = eng.ws
            eng.dense_scatter(b, xd)
            if self.link & 1:              # log(x/eta + 1) encoder: dense kernel, as encode()
                eng.dense_encode(b, xd)
            else:
                _abi.call("spmf_csr_encode", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum),
                          eng.inv_xi, int(self.scale_rows), B, D, self.latent_dim, nc, _ptr(ws.Ap), _ptr(ws.z), st)
            rate = None if rates is None else torch.empty(nc, B, D, dtype=torch.float32, device=dev)
            _abi.call("spmf_loo_pit_accum", _ptr(xd), B, D, self.latent_dim, nc, self.link, _ptr(ws.EV), _ptr(ws.PH),
                      _ptr(ws.z), _ptr(lw) + 8 * c0, S, _ptr(acc), _ptr(inv), _ptr(rate), st)
            if rates is not None:
                rates.append(rate)
        return acc, inv, elpd, khat

    def loo_pit(self, data=None, sample_size=1000, batch_size=None, seed=12345, bins=20, **params):
        """LOO-PIT calibration check (Gabry et al. 2019): the probability integral transform of every entry
        (row, feature) under the leave-one-ROW-out predictive, which PSIS-LOO approximates by weighting the posterior
        draws with the row's Pareto-smoothed importance weights.  For counts the PIT is non-randomised (Czado,
        Gneiting & Held 2009): entry (b, d) has P- = sum_s w_bs F(x_bd - 1 | theta_s) and P+ = sum_s w_bs
        F(x_bd | theta_s), and its PIT is uniform on [P-, P+].  Under a calibrated model the PIT values are uniform:
        a U-shaped histogram means the data are over-dispersed against the predictive, a hump under-dispersed, a
        tilt biased.  Zeros are included.  The (S, B, D) rates are never materialised: a fused CUDA pass
        (csrc/spmf_pit.cu) weights each entry's CDFs as it forms them.

        `data`, the draws, their chunking and seeds are exactly loo()'s, so the weights are those loo() reports k-hat
        for.  `batch_size` cuts a CsrShard; by default it keeps the (B, D, 2) fp64 accumulator at or below 1 GiB.
        `bins` = J, 1 to LOO_PIT_MAX_BINS.  Neither rng_step nor opt_step moves.  Under torch.distributed each rank
        checks its own shard.  Custom encoder / decoder callables raise SpmfError.

        Returns a dict:
          'hist' (J,), 'col_hist' (D, J): summed PIT distributions of the valid entries (bin j covers (j/J, (j+1)/J]);
          'n', 'col_n' (D,): valid entries;  'col_mean_pit' (D,): their mean PIT (P- + P+)/2;
          'ecdf_dev', 'col_ecdf_dev' (D,): max_j |cumulative histogram_j / n - (j+1)/J|, overall and per feature;
          'n_invalid': entries left out because a draw gave an invalid rate / logit or the count is not in the
                       support (see posterior_predictive_check), in the rows not excluded;
          'n_rows_excluded': rows whose elpd is not finite (their weights are undefined: all their entries);
          'khat_threshold', 'n_khat_above': as loo() defines them -- these rows' weights are used, and counted.
        Device tensors are float64 (col_n int64).  Sums over the rows run in batch order."""
        if self._custom_link:
            raise _abi.SpmfError("LOO-PIT has no CUDA path for custom encoder / decoder callables")
        J = int(bins)
        if not 1 <= J <= _abi.LOO_PIT_MAX_BINS:
            raise ValueError(f"loo_pit() takes 1 to {_abi.LOO_PIT_MAX_BINS} bins, got {bins}")
        D, dev, f64 = self.feature_dim, self.device, torch.float64
        if batch_size is None:
            batch_size = max(1, LOO_PIT_ACC_BYTES // (16 * D))
        batches = self._batches_of(data, batch_size, "loo_pit()")
        theta, S = self._loo_draws(sample_size, params, "loo_pit()")
        col_hist = torch.zeros(D, J, dtype=f64, device=dev)
        col_n = torch.zeros(D, dtype=torch.int64, device=dev)
        col_pit = torch.zeros(D, dtype=f64, device=dev)
        threshold = min(1.0 - 1.0 / math.log10(S), 0.7) if S > 1 else -math.inf
        n_invalid = n_excl = n_khat = rows = 0
        for batch in batches:
            b = self._csr_batch(batch, "loo_pit()")
            if b.nrows == 0:
                continue
            acc, inv, elpd, khat = self._loo_pit_batch(b, S, seed, theta)
            scratch = torch.empty(_abi._lib.spmf_loo_pit_hist_scratch_doubles(b.nrows, D, J), dtype=f64, device=dev)
            _abi.call("spmf_loo_pit_hist", _ptr(acc), _ptr(inv), b.nrows, D, J, _ptr(col_hist), _ptr(col_n),
                      _ptr(col_pit), _ptr(scratch), _stream())
            ok = torch.isfinite(elpd)
            n_invalid += int(((inv != 0) & ok[:, None]).sum())
            n_excl += int((~ok).sum())
            n_khat += int((khat > threshold).sum())
            rows += b.nrows
        if rows == 0:
            raise ValueError("loo_pit(): the data holds no rows")
        hist = col_hist.sum(0)
        n = int(col_n.sum())
        edges = torch.arange(1, J + 1, dtype=f64, device=dev) / J

        def ecdf_dev(h, cnt):
            return (h.cumsum(-1) / cnt.unsqueeze(-1) - edges).abs().amax(-1)
        cn = col_n.to(f64)
        return {'hist': hist, 'col_hist': col_hist, 'n': n, 'col_n': col_n,
                'col_mean_pit': col_pit / cn,
                'ecdf_dev': float(ecdf_dev(hist, torch.tensor(float(n), dtype=f64, device=dev))),
                'col_ecdf_dev': ecdf_dev(col_hist, cn),
                'n_invalid': n_invalid, 'n_rows_excluded': n_excl,
                'khat_threshold': threshold, 'n_khat_above': n_khat}

    def loo_pit_values(self, batch, sample_size=1000, seed=12345, **params):
        """The (B, D, 2) fp64 device tensor of (P-, P+) of every entry of one batch, from the kernels of loo_pit()
        with the same draws and weights.  Entries left out by loo_pit() hold NaN: an invalid draw or count, or a
        row whose elpd is not finite.  Raises ValueError above LOO_PIT_VALUES_LIMIT (2^27) entries."""
        b = self._csr_batch(batch, "loo_pit_values()")
        if b.nrows * self.feature_dim > LOO_PIT_VALUES_LIMIT:
            raise ValueError(f"{b.nrows} x {self.feature_dim} entries exceed the limit of {LOO_PIT_VALUES_LIMIT}: "
                             "use loo_pit(), or fewer rows")
        theta, S = self._loo_draws(sample_size, params, "loo_pit_values()")
        acc, inv, elpd, khat = self._loo_pit_batch(b, S, seed, theta)
        bad = (inv != 0) | ~torch.isfinite(elpd)[:, None]
        return acc.masked_fill_(bad[..., None], math.nan)

    def _batches_of(self, data, batch_size, who):
        """The batches of `data` for the evaluation passes: a CsrShard cut into `batch_size` rows (default
        min(N, 8192)), a batch factory as for fit(), or one batch / array; default: the factory last given to
        fit() / compute_scales()."""
        data = self._last_data_factory if data is None else data
        if data is None:
            raise ValueError(f"{who} needs data (none was seen by fit / compute_scales yet)")
        if isinstance(data, CsrShard):
            return data.iter_batches(batch_size or min(data.nrows, 8192))
        if callable(data):
            return iter(data())
        return [data]

    # ------------------------------------------------------------------ posterior predictive check
    def _ppc_engine(self, params, sample_size, seed):
        """Engine holding the operands of the check's draws: explicit `params` (leading sample axis) or
        `sample_size` surrogate draws from `seed`.  Neither moves rng_step or opt_step."""
        if self._custom_link:
            raise _abi.SpmfError("the posterior predictive check has no CUDA path for custom encoder / decoder "
                                 "callables")
        if not params:
            params = self.surrogate_distribution.sample(int(sample_size), seed=seed)
        u = torch.as_tensor(params['u'])
        S = u.shape[0] if u.dim() == 3 else 1
        if S > _abi.PPC_MAX_S:
            raise ValueError(f"the check takes at most {_abi.PPC_MAX_S} draws, got {S}")
        eng = self._engine_for(S)
        self._operands_from_theta(eng, params['u'], params['v'], params['w'], params['s'])
        return eng

    def _ppc_device_batch(self, batch):
        c = batch[self.count_key] if isinstance(batch, dict) else batch
        b = c if isinstance(c, DeviceBatch) else as_device_batch(c, self.device, self.feature_dim)
        if b.cols is None:
            raise ValueError("the posterior predictive check needs a batch with its CSR arrays "
                             "(not a hybrid-only upload)")
        return b

    def _ppc_pass(self, eng, b, seed, row_offset, acc, out=None):
        """Replicates of batch `b` and their statistics (spmf_ppc_rows): per-row results are returned,
        per-column / per-draw ones accumulate into `acc`."""
        S, D, B = eng.S, self.feature_dim, b.nrows
        eng.ensure_rows(B)
        xd = eng.dense_scratch(B)
        ws, st = eng.ws, _stream()
        eng.dense_scatter(b, xd)
        if self.link & 1:                  # log(x/eta + 1) encoder: dense kernel, as encode()
            eng.dense_encode(b, xd)
        else:
            _abi.call("spmf_csr_encode", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), _ptr(b.rowsum),
                      eng.inv_xi, int(self.scale_rows), B, D, self.latent_dim, S, _ptr(ws.Ap), _ptr(ws.z), st)
        dev = self.device
        row_total = torch.empty(S, B, dtype=torch.int64, device=dev)
        row_nnz = torch.empty(S, B, dtype=torch.int32, device=dev)
        row_disc = torch.empty(S, B, 2, dtype=torch.float64, device=dev)
        disc = torch.empty(S, 2, dtype=torch.float64, device=dev)
        _abi.call("spmf_ppc_rows", _ptr(xd), B, D, self.latent_dim, S, self.link, _ptr(ws.EV), _ptr(ws.PH),
                  _ptr(ws.z), int(seed) & 0xFFFFFFFFFFFFFFFF, int(row_offset), _ptr(row_total), _ptr(row_nnz),
                  _ptr(row_disc), _ptr(acc['col_total']), _ptr(acc['col_sumsq']), _ptr(acc['col_nnz']),
                  _ptr(acc['max']), _ptr(acc['invalid']), _ptr(out), _ptr(disc), _ptr(acc['scratch']), st)
        return row_total, row_nnz, disc

    def _ppc_acc(self, S):
        z = lambda *shape, dt=torch.int64: torch.zeros(*shape, dtype=dt, device=self.device)
        return dict(col_total=z(S, self.feature_dim), col_sumsq=z(S, self.feature_dim),
                    col_nnz=z(S, self.feature_dim, dt=torch.int32), max=z(S, dt=torch.int32), invalid=z(S),
                    scratch=torch.empty(128 * S, dtype=torch.float64, device=self.device))

    def posterior_predictive_check(self, data=None, sample_size=32, batch_size=None, seed=12345, **params):
        """Posterior predictive check over the rows of `data`: for every draw theta_s a replicated count matrix
        x_rep ~ p(x | theta_s) (Poisson(rate), or Bernoulli(sigmoid(logit)) for BernoulliFactorization) is drawn
        by a fused CUDA pass over every entry (csrc/spmf_ppc.cu) and reduced to check statistics on the fly; the
        (S,B,D) rate and replicate tensors never exist.

        `data` is taken as by waic(): a batch factory, a CsrShard (cut into `batch_size` rows), one batch or an
        array; default: the factory last given to fit() / compute_scales().  Draws: explicit s, u, v, w with a
        leading sample axis (as for row_log_likelihood), else `sample_size` surrogate draws from `seed`; the same
        draws serve every batch.  The replicate of entry (s, row, d) comes from a Philox stream keyed by (seed, s,
        global row, d) -- rows are numbered across the batches in order -- so the result does not depend on the
        batch size, and two calls with the same arguments give bit-identical results.  Neither rng_step nor
        opt_step moves.  Under torch.distributed each rank checks its own shard (no aggregation across ranks).

        Returns (observed, replicated, p_value, invalid):
          observed:   'row_total', 'row_nnz' (N,); 'col_total', 'col_sumsq', 'col_nnz' (D,); 'total', 'nnz',
                      'max' (scalars); 'discrepancy' (S,) = D(x, theta_s)
          replicated: the same keys with a leading S axis (integers, exact); 'discrepancy' (S,) = D(x_rep_s, theta_s)
          p_value:    ppc_p_values(observed, replicated): the mid-p (#{T_rep > T_obs} + 0.5 #{T_rep == T_obs}) / S of
                      every statistic, the discrepancy paired per draw, plus 'col_var'
          invalid:    (S,) entries whose rate is negative, not finite or above 2^24 (Poisson) or whose logit is
                      not finite (Bernoulli): their replicate is 0 and they are left out of both discrepancies.
        The discrepancy is D(y, theta) = sum (y - rate)^2 / rate (Poisson) or sum (y - p)^2 / (p (1 - p))
        (Bernoulli) over the valid entries, summed in fp64 in a fixed order; an entry with rate (or p (1 - p))
        0 adds 0 where y equals it and +inf elsewhere."""
        batches = self._batches_of(data, batch_size, "posterior_predictive_check()")
        eng = self._ppc_engine(params, sample_size, seed)
        S, D, dev = eng.S, self.feature_dim, self.device
        acc = self._ppc_acc(S)
        obs_col = dict(col_total=torch.zeros(D, dtype=torch.float64, device=dev),
                       col_sumsq=torch.zeros(D, dtype=torch.float64, device=dev),
                       col_nnz=torch.zeros(D, dtype=torch.int32, device=dev))
        rep_rows, rep_nnz, obs_rows, obs_nnz = [], [], [], []
        disc = torch.zeros(S, 2, dtype=torch.float64, device=dev)
        obs_max = torch.zeros((), dtype=torch.float32, device=dev)
        row_offset = 0
        for batch in batches:
            b = self._ppc_device_batch(batch)
            rt, rn, d = self._ppc_pass(eng, b, seed, row_offset, acc)
            rep_rows.append(rt)
            rep_nnz.append(rn)
            disc += d                                       # batch order: a fixed summation order
            ot = torch.empty(b.nrows, dtype=torch.float64, device=dev)
            on = torch.empty(b.nrows, dtype=torch.int32, device=dev)
            _abi.call("spmf_ppc_observed", _ptr(b.rowptr), _ptr(b.cols), _ptr(b.vals), b.nrows, D, _ptr(ot),
                      _ptr(on), _ptr(obs_col['col_total']), _ptr(obs_col['col_sumsq']), _ptr(obs_col['col_nnz']),
                      _stream())
            obs_rows.append(ot)
            obs_nnz.append(on)
            obs_max = torch.maximum(obs_max, eng.ws.xdense[:b.nrows * D].max())
            row_offset += b.nrows
        if row_offset == 0:
            raise ValueError("posterior_predictive_check(): the data holds no rows")
        rep_rows, rep_nnz = torch.cat(rep_rows, 1), torch.cat(rep_nnz, 1)
        obs_rows, obs_nnz = torch.cat(obs_rows), torch.cat(obs_nnz)
        observed = dict(row_total=obs_rows, row_nnz=obs_nnz, **obs_col, total=obs_rows.sum(),
                        nnz=obs_nnz.sum(dtype=torch.int64), max=obs_max.to(torch.float64), discrepancy=disc[:, 1])
        replicated = dict(row_total=rep_rows, row_nnz=rep_nnz, col_total=acc['col_total'],
                          col_sumsq=acc['col_sumsq'], col_nnz=acc['col_nnz'], total=rep_rows.sum(1),
                          nnz=rep_nnz.sum(1, dtype=torch.int64), max=acc['max'], discrepancy=disc[:, 0])
        return observed, replicated, ppc_p_values(observed, replicated), acc['invalid']

    def posterior_predictive_sample(self, data, sample_size=8, seed=12345, row_offset=0, **params):
        """The replicates x_rep of one batch as an int32 (S, B, D) device tensor: the same kernel, draws and
        Philox streams as posterior_predictive_check (rows numbered from `row_offset`), so the statistics of these
        replicates are the check's statistics.  Draws as for the check.  Raises ValueError above PPC_SAMPLE_LIMIT
        (2^30) entries."""
        b = self._ppc_device_batch(data)
        u = torch.as_tensor(params['u']) if params else None
        S = int(sample_size) if u is None else (u.shape[0] if u.dim() == 3 else 1)
        if S * b.nrows * self.feature_dim > PPC_SAMPLE_LIMIT:
            raise ValueError(f"{S} x {b.nrows} x {self.feature_dim} replicates exceed the limit of {PPC_SAMPLE_LIMIT} "
                             "entries: use posterior_predictive_check, or fewer rows / draws")
        eng = self._ppc_engine(params, sample_size, seed)
        out = torch.empty(eng.S, b.nrows, self.feature_dim, dtype=torch.int32, device=self.device)
        self._ppc_pass(eng, b, seed, row_offset, self._ppc_acc(eng.S), out=out)
        return out

    def sample(self, n=None, seed=None):
        """[EXT] BayesianModel.sample: draws of every latent variable from the surrogate posterior."""
        return self.surrogate_distribution.sample(n, seed=seed)

    def unormalized_log_prob_list(self, *x):
        """poisson.py:703-709 (positional wrapper; needs `data` bound by the caller)."""
        return self.unormalized_log_prob(**{v: t for v, t in zip(self.var_list, x)})

    # ------------------------------------------------------------------ training loop [EXT L4]
    def elbo_step(self, batch, sample_size, learning_rate=None, clip_value=0.0, variant=0):
        """One ADVI step on one minibatch: loss + gradients (+ all-reduce + Adam if learning_rate)."""
        eng = self._engine_for(sample_size)
        c = batch[self.count_key] if isinstance(batch, dict) else batch
        b = as_device_batch(c, self.device)
        if eng.world_size > 1:
            from .parallel import allreduce_step
            parts = eng.step(b, lr=learning_rate, clip_value=clip_value)
            loss = allreduce_step(eng, parts, self.process_group, adam=learning_rate is not None)
        else:
            parts = eng.step(b, lr=learning_rate, clip_value=clip_value)   # one native call, Adam included
            loss = eng.loss_value(parts)
            if learning_rate is None:
                eng.clear_comm_slack()
        return loss

    def fit(self, batched_data_factory, batch_size=None, dataset_size=None, num_steps=100,
            learning_rate=0.01, rel_tol=1e-4, abs_tol=None, clip_value=0.0, sample_size=8,
            sample_batches=1, max_decay_steps=25, lr_decay_factor=0.99, patience=5, verbose=True,
            checkpoint_path=None, checkpoint_every=1, resume=False, **kwargs):
        """Minibatch ADVI (call site tests/spmf_test.py:35-43).  [EXT] behaviour restated from the
        reference's notebook logs (SURVEY.md section 5): an epoch is one pass over
        `batched_data_factory()`; the mean batch loss is tracked; on improvement the parameters are
        snapshotted, on a plateau the learning rate decays by `lr_decay_factor` and the best
        snapshot is restored; stops on rel_tol / abs_tol / max_decay_steps / num_steps.
        Returns the list of epoch losses.

        `checkpoint_path`: write a checkpoint (save_checkpoint, plus the state of this loop) after every
        `checkpoint_every` epochs, after the last epoch and when the loop stops early.  `resume=True` with an
        existing `checkpoint_path`: continue the run stored there (parameters, optimiser, counters, column
        ranking, epoch, losses, learning rate, best snapshot); `num_steps` counts the epochs of the whole run and
        the returned list includes the epochs before the resume."""
        self._last_data_factory = batched_data_factory
        S = int(sample_size) * int(sample_batches)
        eng = self._engine_for(S)
        losses, best, best_state = [], float('inf'), None
        lr, decays, since_best = float(learning_rate), 0, 0
        if checkpoint_path is not None and int(checkpoint_every) < 1:
            raise ValueError("checkpoint_every must be >= 1")
        start, stopped = 0, False
        if resume and checkpoint_path is not None and os.path.exists(checkpoint_path):
            loop = self._apply_checkpoint(_read_state(checkpoint_path))
            if loop is not None:
                start, stopped, losses = int(loop['epoch']), bool(loop['stopped']), list(loop['losses'])
                lr, decays, since_best, best = float(loop['lr']), int(loop['decays']), int(loop['since_best']), float(loop['best'])
                bs = loop['best_state']
                if bs is not None:
                    best_state = tuple(t.to(self.device) for t in bs[:3]) + (int(bs[3]),)
                if verbose:
                    print(f"Resuming from {checkpoint_path} at epoch {start}")
        if stopped:                    # the stored run had already met its stopping rule
            self.set_calibration_expectations()
            return losses
        for epoch in range(start, int(num_steps)):
            acc = torch.zeros((), dtype=torch.float64, device=self.device)
            nb, last = 0, None
            batches = batched_data_factory()
            limit = self._common_batch_count(batches) if eng.world_size > 1 else None
            for batch in self._device_batches(batches, eng):
                if limit is not None and nb >= limit:
                    break              # ranks must issue the same number of all-reduces per epoch
                last = self.elbo_step(batch, S, learning_rate=lr, clip_value=clip_value)
                acc += last
                nb += 1
            if nb == 0:
                raise ValueError("batched_data_factory() yielded no batches")
            mean_loss = float(acc.item()) / nb                 # one host sync per epoch
            if eng.world_size > 1:
                from .parallel import check_exchange
                check_exchange(eng)
            losses.append(mean_loss)
            if verbose:
                print(f"Epoch {epoch}: average-batch loss: {mean_loss} last batch loss: {float(last.item())}")
            stop = False
            if not math.isfinite(mean_loss):
                if best_state is not None:
                    if verbose:
                        print("Got NaN, restoring a checkpoint")
                    self._restore(eng, best_state)
                lr *= lr_decay_factor
                decays += 1
            elif mean_loss < best:
                improved = best - mean_loss
                prev_best = best
                best, since_best = mean_loss, 0
                best_state = self._snapshot(eng)
                if math.isfinite(prev_best):
                    if abs_tol is not None and improved < abs_tol:
                        stop = True
                    elif rel_tol is not None and improved < rel_tol * abs(prev_best):
                        stop = True
            else:
                since_best += 1
                if since_best >= patience:
                    lr *= lr_decay_factor
                    decays += 1
                    since_best = 0
                    if verbose:
                        print(f"New learning rate: {lr}")
                    self._restore(eng, best_state)
            if decays >= max_decay_steps:
                stop = True
            if checkpoint_path is not None and (stop or epoch + 1 == int(num_steps)
                                                or (epoch + 1) % int(checkpoint_every) == 0):
                self._write_checkpoint(checkpoint_path, dict(
                    epoch=epoch + 1, stopped=stop, losses=list(losses), lr=lr, decays=decays,
                    since_best=since_best, best=best, best_state=best_state))
            if stop:
                break
        else:
            if verbose:
                print("Terminating because we are out of iterations")
        self.set_calibration_expectations()
        return losses

    calibrate_advi = fit     # legacy name used by bin/factorize_csv.py:121-124

    def _common_batch_count(self, batches):
        """Multi-GPU: every rank must run the same number of steps per epoch (one all-reduce each).  When
        the per-rank batch count is known (`len()`), agree on the minimum across ranks and truncate;
        iterables without a length must be balanced by the caller (e.g. drop_remainder sharding)."""
        try:
            n = len(batches)
        except TypeError:
            return None
        t = torch.tensor([n, -n], dtype=torch.int64, device=self.device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN, group=self.process_group)
        lo, hi = int(t[0].item()), -int(t[1].item())
        if lo != hi:
            print(f"[spmf_b200] ranks hold {lo}..{hi} batches per epoch; truncating every rank to {lo}")
        return lo

    def _device_batches(self, batches, eng):
        """Host-resident CSR batches are uploaded one ahead on a copy stream; anything else passes through."""
        from .data import HostCsrBatch, HostDenseBatch, prefetch_to_device
        it = iter(batches)
        try:
            first = next(it)
        except StopIteration:
            return iter(())
        import itertools
        chained = itertools.chain([first], it)
        c = first[self.count_key] if isinstance(first, dict) else first
        if isinstance(c, (HostCsrBatch, HostDenseBatch)):
            return prefetch_to_device((b[self.count_key] if isinstance(b, dict) else b for b in chained),
                                      self.device, hot=self._hot_spec(eng))
        return chained

    @staticmethod
    def _snapshot(eng):
        return (eng.params.clone(), eng.adam_m.clone(), eng.adam_v.clone(), eng.opt_step)

    @staticmethod
    def _restore(eng, st):
        eng.params.copy_(st[0]); eng.adam_m.copy_(st[1]); eng.adam_v.copy_(st[2]); eng.opt_step = st[3]

    # ------------------------------------------------------------------ persistence
    def state(self):
        return {
            'surrogate_vars': [t.detach().cpu().clone() for t in self.surrogate_vars],
            'eta_i': self.eta_i.clone(), 'xi_u_global': float(self.xi_u_global),
            'hyper': dict(latent_dim=self.latent_dim, feature_dim=self.feature_dim,
                          u_tau_scale=self.u_tau_scale, s_tau_scale=self.s_tau_scale,
                          symmetry_breaking_decay=self.symmetry_breaking_decay,
                          scale_columns=self.scale_columns, scale_rows=self.scale_rows,
                          log_transform=self.log_transform, count_key=self.count_key, seed=self.seed,
                          entropy_weight=self.entropy_weight, prior_weight=self.prior_weight,
                          **({'encoder_function': self._custom_link[0] if self._custom_link[0] != self._default_encoder else None,
                              'decoder_function': self._custom_link[1] if self._custom_link[1] != self._default_decoder else None}
                             if self._custom_link else {})),
        }

    def save(self, filename):
        """[EXT] BayesianModel.save (a dill pickle in the reference; bin/factorize_csv.py:136-139).  The
        state is plain tensors / floats, so the file loads with either dill or pickle."""
        with open(filename, 'wb') as f:
            _pickle_module().dump(self.state(), f)

    def save_checkpoint(self, path):
        """Write what training needs to continue exactly where it stands: state() plus a 'training' entry with
        the flat parameters, the Adam moments, the optimiser and Philox counters of every engine, and the
        hot-column ranking (see _training_state).  `load` restores all of it.  The file is written to
        `path + '.tmp'` and renamed, so an interrupted write leaves the previous checkpoint intact.  Under
        torch.distributed the call is collective: every rank calls it, rank 0 writes."""
        self._write_checkpoint(path, None)

    def _moment_gatherer(self, eng):
        """t -> full copy of a moment buffer.  With the peer-memory exchange a rank keeps the moments of its own
        slice of the data block only (csrc/spmf_p2p.cu): the slices are gathered from all ranks (collective)."""
        if eng.world_size > 1:
            from .parallel import exchange_kind, gather_owned
            if exchange_kind(eng) == "p2p-kernel":
                return lambda t: gather_owned(eng, t, self.process_group)
        return lambda t: t

    def _training_state(self, loop=None):
        """The 'training' entry of a checkpoint (CPU tensors and plain values).  `loop`: the state of fit()."""
        eng = self._engine_for(1)
        full = self._moment_gatherer(eng)
        counters = dict(self._pending_counters)
        counters.update({S: (int(e.opt_step), int(e.rng_step)) for S, e in self._engines.items()})
        tr = {
            'version': CHECKPOINT_VERSION, 'model': int(self._model_id), 'link': int(self.link),
            'params': eng.params.detach().to('cpu', copy=True),
            'adam_m': full(eng.adam_m).to('cpu', copy=True), 'adam_v': full(eng.adam_v).to('cpu', copy=True),
            'counters': counters,
            'col_rank': None if self.col_rank is None else self.col_rank.to('cpu', torch.int32, copy=True),
            'hot_cols': int(self.hot_cols), 'hot_density': float(self.hot_density),
            'exact_guard': bool(self.exact_guard), 'rank_version': int(getattr(self, '_rank_version', 0)),
        }
        if loop is not None:
            loop = dict(loop)
            bs = loop['best_state']
            if bs is not None:
                loop['best_state'] = (bs[0].to('cpu', copy=True), full(bs[1]).to('cpu', copy=True),
                                      full(bs[2]).to('cpu', copy=True), int(bs[3]))
            tr['fit'] = loop
        return tr

    def _write_checkpoint(self, path, loop):
        path = os.fspath(path)
        ck = self.state()
        ck['training'] = self._training_state(loop)
        dist_on = torch.distributed.is_available() and torch.distributed.is_initialized()
        err = None
        if not dist_on or torch.distributed.get_rank(self.process_group) == 0:
            try:
                tmp = path + ".tmp"
                with open(tmp, 'wb') as f:
                    _pickle_module().dump(ck, f)
                    f.flush()
                    os.fsync(f.fileno())
                os.replace(tmp, path)
            except Exception as e:     # noqa: BLE001 -- re-raised below, after the other ranks learn of it
                err = e
        if dist_on:                    # every rank returns once the file is in place, or raises with rank 0
            ok = torch.tensor([0.0 if err else 1.0], device=self.device)
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN, group=self.process_group)
            if err is None and float(ok.item()) == 0.0:
                raise _abi.SpmfError(f"rank 0 could not write the checkpoint {path}")
        if err is not None:
            raise err

    def _restore_training(self, tr):
        """Take over the 'training' entry of a checkpoint: parameters, moments (full on every rank: only a rank's
        owned slice is read under the peer-memory exchange), ranking, and the counters of every engine -- those
        of engines not created yet are applied when _engine_for creates them."""
        if tr.get('version') != CHECKPOINT_VERSION:
            raise _abi.SpmfError(f"checkpoint format {tr.get('version')} is not {CHECKPOINT_VERSION}")
        if int(tr['model']) != self._model_id or int(tr['link']) != self.link:
            raise _abi.SpmfError(f"checkpoint of model {tr['model']} / link {tr['link']} cannot resume "
                                 f"{type(self).__name__} (model {self._model_id} / link {self.link})")
        eng = self._engine_for(1)
        n = eng.layout.n_params
        if any(tuple(tr[k].shape) != (n,) for k in ('params', 'adam_m', 'adam_v')):
            raise _abi.SpmfError(f"checkpoint holds {tuple(tr['params'].shape)} parameters, this model {n}")
        eng.params.copy_(tr['params'])
        eng.adam_m.copy_(tr['adam_m'])
        eng.adam_v.copy_(tr['adam_v'])
        self.hot_density, self.exact_guard = float(tr['hot_density']), bool(tr['exact_guard'])
        rank = tr['col_rank']
        self.col_rank = None if rank is None else rank.to(device=self.device, dtype=torch.int32)
        self.hot_cols, self._rank_version = int(tr['hot_cols']), int(tr['rank_version'])
        counters = {int(S): (int(a), int(b)) for S, (a, b) in tr['counters'].items()}
        for S, e in self._engines.items():
            self._push_scales(e)
            e.exact_guard = self.exact_guard
            e.opt_step, e.rng_step = counters.pop(S, (0, 0))
        self._pending_counters = counters

    def _apply_checkpoint(self, state):
        """fit(resume=True): take over the scales and training state of a checkpoint; returns fit's loop state
        (None when the checkpoint was written by save_checkpoint)."""
        tr = state.get('training')
        if tr is None:
            raise _abi.SpmfError("the file has no training state (written by save(), not save_checkpoint())")
        hy = state['hyper']
        if (int(hy['feature_dim']), int(hy['latent_dim'])) != (self.feature_dim, self.latent_dim):
            raise _abi.SpmfError(f"checkpoint of D={hy['feature_dim']}, K={hy['latent_dim']} cannot resume a model "
                                 f"of D={self.feature_dim}, K={self.latent_dim}")
        self.eta_i = torch.as_tensor(state['eta_i'], dtype=torch.float64).reshape(1, -1)
        self.xi_u_global = float(state.get('xi_u_global', 1.0))
        self._restore_training(tr)
        return tr.get('fit')

    def reconstitute(self, state):
        """poisson.py:711-717: re-create distributions, then assign the saved tensors in order."""
        self.create_distributions()
        for dst, value in zip(self.surrogate_vars, state['surrogate_vars']):
            dst.copy_(torch.as_tensor(value).to(device=self.device, dtype=torch.float32))
        if 'eta_i' in state:
            self.eta_i = torch.as_tensor(state['eta_i'], dtype=torch.float64).reshape(1, -1)
            self.xi_u_global = float(state.get('xi_u_global', 1.0))
            for eng in self._engines.values():
                self._push_scales(eng)

    @classmethod
    def load(cls, filename, device=None):
        """A model from a save() file, or -- from a save_checkpoint() file -- one that continues training exactly
        where the saved model stood (parameters, Adam moments and step, Philox counters, column ranking)."""
        state = _read_state(filename)
        tr = state.get('training')
        extra = {}
        if tr is not None:
            if int(tr['model']) != cls._model_id:
                raise _abi.SpmfError(f"checkpoint of model {tr['model']} cannot be loaded as {cls.__name__}")
            extra = dict(hot_density=tr['hot_density'], exact_guard=tr['exact_guard'])
        m = cls(device=device, **state['hyper'], **extra)
        m.reconstitute(state)
        if tr is not None:
            m._restore_training(tr)
        m.set_calibration_expectations()
        return m
