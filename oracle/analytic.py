"""Analytic (hand-derived) forward+backward of the SPMF ADVI step in numpy float64.

TEST INFRASTRUCTURE.  Second, independent restatement used to cross-check
``oracle/spmf_oracle.py`` (autograd) and to document, on the CPU, exactly the
decomposition the CUDA kernels implement:

  draw  ->  derived operands (A' = a*u/eta, EV = eta*v, phi)  ->  data term with the
  sparse closed form (only nonzeros need log / div; -sum(rate) is O(BK+KD))  ->
  backward to the 24 variational tensors.

Formulas: SURVEY.md section 3.4 (restating mederrata_spmf/poisson.py:34-54,156-184,
575-701).  PARITY UNPINNED (see spmf_oracle.py header).
"""
from __future__ import annotations

import math

import numpy as np
from scipy.special import digamma, gammaln

from .spmf_oracle import (VAR_LIST, NORMAL_VARS, HALF_LOG_2_OVER_PI, HALF_LOG_2PI,
                          gamma_sample_der_alpha)


def softplus(x):
    return np.logaddexp(0.0, x)


def sigmoid(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def log_sigmoid(x):
    return -np.logaddexp(0.0, -x)


def _as_csr(x):
    """Dense array or scipy.sparse matrix -> (scipy CSR float64 with explicit zeros removed)."""
    import scipy.sparse as sp
    if sp.issparse(x):
        m = x.tocsr().astype(np.float64)
    else:
        m = sp.csr_matrix(np.asarray(x, dtype=np.float64))
    m.eliminate_zeros()
    m.sort_indices()
    return m


def analytic_loss_and_grads(model, params, noise, x, c_gamma=False, magnitudes=False):
    """Returns (loss, grads dict, parts dict of (S,) arrays).  `model` is an
    OraclePoissonFactorization (only its hyper-parameters / eta / xi are read).  `x`: the (B,D)
    counts, dense or scipy.sparse -- only the nonzeros are visited (the same sparse closed form
    the kernels use), so a bench-sized batch (8192 x 20000, ~8e6 nonzeros) is evaluated in float64
    on the CPU without the (S,B,D) rate tensor.  c_gamma: use the C helper (oracle/gamma_der.c) for
    the implicit Gamma gradient instead of the vectorised python series (same expansions).

    magnitudes=True returns (loss, grads, parts, mags, rows) for an element-wise check of an fp32 kernel:
      mags: for every gradient of v, w, u, s ('<var>/loc', '<var>/scale_raw'), a float64 array M of the same
            shape: the same formulas evaluated with every summand of every signed sum replaced by its absolute
            value, data term, chain and prior terms alike.  M bounds the cancellation at each element, so
            |got - ref| <= rtol * M is a test whose strength does not depend on the element's size.  Also the
            data-term sums alone, summed over the draws: 'data/GAp' (D,K), 'data/GEV' (D,K), 'data/Gphi' (D,).
      rows: {'z': (z, Mz) of shape (S,B,K), 'row_ll': (ll, Mll) of shape (S,B)} -- the encoding and the
            per-row Poisson log-likelihood with their magnitudes.  Mll counts x (|log lambda| + 1) per
            nonzero: an error relative to lambda is an absolute error in log lambda."""
    import scipy.sparse as sp
    import torch
    P = {k: v.detach().numpy().astype(np.float64) for k, v in params.items()}
    Nz = {k: v.detach().numpy().astype(np.float64) for k, v in noise.items()}
    X = _as_csr(x)
    B, D = X.shape
    K = model.latent_dim
    S = Nz['u'].shape[0]
    eta = model.eta_i.numpy().reshape(D)
    xi = float(model.xi_u_global)
    assert not model.log_transform

    # ---------------- draws, log q, d(logq)/d(theta-path) ----------------
    th, t_pre, sg = {}, {}, {}
    logq = np.zeros(S)
    aux = {}
    for k in VAR_LIST:
        if k in NORMAL_VARS:
            rho = P[k + '/scale_raw']
            sig = softplus(rho)
            t = P[k + '/loc'] + sig * Nz[k]
            base = -0.5 * Nz[k] ** 2 - np.log(sig) - HALF_LOG_2PI
            aux[k] = (sig,)
        else:
            al = softplus(P[k + '/conc_raw'])
            be = softplus(P[k + '/scale_raw'])
            g = Nz[k]
            t = be / g
            base = al * np.log(be) - gammaln(al) - (al + 1.0) * np.log(t) - be / t
            aux[k] = (al, be, g)
        t_pre[k] = t
        sg[k] = sigmoid(t)
        th[k] = softplus(t)
        logq += (base - log_sigmoid(t)).sum((-1, -2))

    # ---------------- prior terms and d(target)/d(theta) ----------------
    c_k = model.symmetry_breaking_decay ** np.arange(K)[None, :]
    parts = {}
    dth = {k: np.zeros_like(th[k]) for k in VAR_LIST}      # d(target_s)/d(theta_s)
    red = lambda a: a.sum((-1, -2))
    c0 = HALF_LOG_2_OVER_PI
    lg_half = gammaln(0.5)

    parts['v'] = red(c0 - math.log(0.1) - 0.5 * (th['v'] / 0.1) ** 2)
    dth['v'] += -th['v'] / 0.01
    parts['w'] = red(c0 - 0.5 * th['w'] ** 2)
    dth['w'] += -th['w']

    def halfnormal_scaled(yname, scale_terms):
        """HalfNormal(y; sigma = prod(scale_terms)) value + grads wrt y and every factor."""
        sigma = np.ones_like(th[yname])
        for n, f in scale_terms:
            sigma = sigma * (th[n] if n else f)
        y = th[yname]
        val = c0 - np.log(sigma) - 0.5 * (y / sigma) ** 2
        dth[yname] += -y / sigma ** 2
        dsig = -1.0 / sigma + y ** 2 / sigma ** 3
        for n, f in scale_terms:
            if n:
                contrib = dsig * sigma / th[n]
                # reduce broadcast axes
                for ax, (a, b) in enumerate(zip(contrib.shape, th[n].shape)):
                    if a != b:
                        contrib = contrib.sum(ax, keepdims=True)
                dth[n] += contrib
        return red(val)

    parts['u'] = halfnormal_scaled('u', [('u_eta', None), ('u_tau', None), (None, c_k)])
    parts['s'] = halfnormal_scaled('s', [('s_eta', None), ('s_tau', None)])

    def sqrt_ig(yname, aname):
        y, a = th[yname], th[aname]
        beta = 1.0 / a
        val = 0.5 * np.log(beta) - lg_half - 2.0 * np.log(y) - beta / y ** 2 + math.log(2.0)
        dth[yname] += -2.0 / y + 2.0 * beta / y ** 3
        dbeta = 0.5 / beta - 1.0 / y ** 2
        dth[aname] += dbeta * (-1.0 / a ** 2)
        return red(val)

    def ig_half(aname, b):
        a = th[aname]
        val = 0.5 * math.log(b) - lg_half - 1.5 * np.log(a) - b / a
        dth[aname] += -1.5 / a + b / a ** 2
        return red(val)

    parts['u_eta'] = sqrt_ig('u_eta', 'u_eta_a')
    parts['u_eta_a'] = ig_half('u_eta_a', 1.0)
    parts['u_tau'] = sqrt_ig('u_tau', 'u_tau_a')
    parts['u_tau_a'] = ig_half('u_tau_a', 1.0 / model.u_tau_scale ** 2)
    parts['s_eta'] = sqrt_ig('s_eta', 's_eta_a')
    parts['s_eta_a'] = ig_half('s_eta_a', 1.0)
    parts['s_tau'] = sqrt_ig('s_tau', 's_tau_a')
    parts['s_tau_a'] = ig_half('s_tau_a', 1.0 / model.s_tau_scale ** 2)

    # ---------------- derived operands ----------------
    s0, s1 = th['s'][:, 0, :], th['s'][:, 1, :]                   # (S,D)
    a_d = s0 / (s0 + s1)
    b_d = s1 / (s0 + s1)
    Ap = a_d[:, :, None] * th['u'] / eta[None, :, None]           # (S,D,K)  A' = A/eta
    EV = eta[None, :, None] * np.swapaxes(th['v'], -1, -2)        # (S,D,K)  eta*v
    phi = eta[None, :] * b_d * th['w'][:, 0, :]                   # (S,D)
    rowsum = np.asarray(X.sum(1)).reshape(B)
    r = rowsum / xi if model.scale_rows else np.ones(B)           # (B,)

    # ---------------- data term, sparse closed form ----------------
    indptr, di, xv = X.indptr, X.indices, X.data
    bi = np.repeat(np.arange(B), np.diff(indptr))
    lgam_total = gammaln(xv + 1.0).sum()
    Xr = sp.diags(r) @ X                                          # rows scaled by r_b
    Lx = np.zeros(S); Lz = np.zeros(S)
    GAp = np.zeros_like(Ap); GEV = np.zeros_like(EV); Gphi = np.zeros_like(phi)
    # magnitudes: every operand is >= 0 here (x, r, A', eta*v, phi, z, lambda), so only the signed
    # sums (dz, GEV, Gphi) and what they feed need the absolute-value restatement
    MGAp = np.zeros_like(Ap); MGEV = np.zeros_like(EV); MGphi = np.zeros_like(phi)
    Z = np.zeros((S, B, K)); ROW_LL = np.zeros((S, B)); MROW_LL = np.zeros((S, B))
    lgam_row = np.asarray(sp.csr_matrix((gammaln(xv + 1.0), di, indptr), shape=(B, D)).sum(1)).reshape(B)
    CH = 1 << 20                                                  # nonzeros per chunk (bounds temporaries)
    for s in range(S):
        z = Xr @ Ap[s]                                            # (B,K) = r_b * (x @ A')
        vsum = EV[s].sum(0)                                       # (K,)
        lam = np.empty(xv.shape[0])
        for j0 in range(0, xv.shape[0], CH):
            sl = slice(j0, j0 + CH)
            lam[sl] = np.einsum('nk,nk->n', z[bi[sl]], EV[s][di[sl]]) + phi[s][di[sl]]
        gq = xv / lam                                             # x/lambda at nonzeros
        Lx[s] = (xv * np.log(lam)).sum() - lgam_total - (z @ vsum).sum() - B * phi[s].sum()
        Lz[s] = (c0 - 0.5 * z ** 2).sum()
        W = sp.csr_matrix((gq, di, indptr), shape=(B, D))         # x/lambda on the sparsity pattern
        dz = W @ EV[s] - vsum[None, :] - z
        GEV[s] = W.T @ z - z.sum(0)[None, :]
        Gphi[s] = np.asarray(W.sum(0)).reshape(D) - B
        GAp[s] = Xr.T @ dz
        if magnitudes:
            Mdz = W @ EV[s] + vsum[None, :] + z
            MGEV[s] = W.T @ z + z.sum(0)[None, :]
            MGphi[s] = np.asarray(W.sum(0)).reshape(D) + B
            MGAp[s] = Xr.T @ Mdz
            Z[s] = z
            xl = sp.csr_matrix((xv * np.log(lam), di, indptr), shape=(B, D))
            xm = sp.csr_matrix((xv * (np.abs(np.log(lam)) + 1.0), di, indptr), shape=(B, D))
            rate_sum = z @ vsum + phi[s].sum()
            ROW_LL[s] = np.asarray(xl.sum(1)).reshape(B) - lgam_row - rate_sum
            MROW_LL[s] = np.asarray(xm.sum(1)).reshape(B) + lgam_row + rate_sum
    parts['z'] = Lz
    parts['x'] = Lx

    # ---------------- chain to u, v, w, s ----------------
    dth['u'] += GAp * a_d[:, :, None] / eta[None, :, None]
    da = (GAp * th['u']).sum(-1) / eta[None, :]
    dth['v'] += np.swapaxes(GEV * eta[None, :, None], -1, -2)
    dth['w'] += (eta[None, :] * b_d * Gphi)[:, None, :]
    db = eta[None, :] * th['w'][:, 0, :] * Gphi
    den = (s0 + s1) ** 2
    dth['s'][:, 0, :] += (da - db) * s1 / den
    dth['s'][:, 1, :] += (db - da) * s0 / den
    if magnitudes:
        # prior terms of v, w, u, s in absolute value (the InverseGamma family is not checked element-wise)
        sig_u = th['u_eta'] * th['u_tau'] * c_k
        sig_s = th['s_eta'] * th['s_tau']
        mth = {'v': th['v'] / 0.01, 'w': th['w'].copy(), 'u': th['u'] / sig_u ** 2, 's': th['s'] / sig_s ** 2}
        mth['u'] += MGAp * a_d[:, :, None] / eta[None, :, None]
        Mda = (MGAp * th['u']).sum(-1) / eta[None, :]
        mth['v'] += np.swapaxes(MGEV * eta[None, :, None], -1, -2)
        mth['w'] += (eta[None, :] * b_d * MGphi)[:, None, :]
        Mdb = eta[None, :] * th['w'][:, 0, :] * MGphi
        mth['s'][:, 0, :] += (Mda + Mdb) * s1 / den
        mth['s'][:, 1, :] += (Mda + Mdb) * s0 / den

    # ---------------- loss and grads of the 24 variational tensors ----------------
    target = sum(parts.values())
    loss = float((logq - target).mean())
    grads = {}
    mags = {}
    for k in VAR_LIST:
        # d loss_s / d t  with loss_s = logq_s - target_s ;  y = softplus(t)
        Gy = -dth[k]
        if k in NORMAL_VARS:
            (sig,) = aux[k]
            dt = Gy * sg[k] - (1.0 - sg[k])
            grads[k + '/loc'] = dt.mean(0)
            srho = sigmoid(P[k + '/scale_raw'])
            grads[k + '/scale_raw'] = (dt * Nz[k]).mean(0) * srho - srho / sig
            if magnitudes:
                Mdt = mth[k] * sg[k] + (1.0 - sg[k])
                mags[k + '/loc'] = Mdt.mean(0)
                mags[k + '/scale_raw'] = (Mdt * np.abs(Nz[k])).mean(0) * srho + srho / sig
        else:
            al, be, g = aux[k]
            t = t_pre[k]
            dlogq_dt = -(al + 1.0) / t + be / t ** 2 - (1.0 - sg[k])
            dt = Gy * sg[k] + dlogq_dt
            if c_gamma:
                from .cbuild import gamma_sample_der_alpha_c
                dg_da = gamma_sample_der_alpha_c(np.broadcast_to(al, g.shape), g)
            else:
                dg_da = gamma_sample_der_alpha(torch.as_tensor(np.broadcast_to(al, g.shape).copy()),
                                               torch.as_tensor(g)).numpy()
            dt_da = -be / g ** 2 * dg_da
            dt_db = 1.0 / g
            dal = (np.log(be) - digamma(al) - np.log(t)) + dt * dt_da
            dbe = (al / be - 1.0 / t) + dt * dt_db
            grads[k + '/conc_raw'] = dal.mean(0) * sigmoid(P[k + '/conc_raw'])
            grads[k + '/scale_raw'] = dbe.mean(0) * sigmoid(P[k + '/scale_raw'])
    parts['logq'] = logq
    if not magnitudes:
        return loss, grads, parts
    mags['data/GAp'] = MGAp.sum(0)
    mags['data/GEV'] = MGEV.sum(0)
    mags['data/Gphi'] = MGphi.sum(0)
    return loss, grads, parts, mags, {'z': (Z, Z.copy()), 'row_ll': (ROW_LL, MROW_LL)}
