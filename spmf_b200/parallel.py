"""Row-sharded data parallelism: one process per GPU, one all-reduce per step.

The reference only carries a `strategy` hook (tf.distribute, poisson.py:60,72,82-83) that every
driver leaves at None; this is the net-new multi-GPU path (SURVEY.md 8e).  Every rank holds the
same variational parameters and draws the same Philox noise, evaluates the data term on its own
rows, and adds its 1/world share of the prior + entropy gradient of the data-touched tensors
(v, w, u, s).  ONE `all_reduce(sum)` over the contiguous block
    [ grads of v,w,u,s (loc|scale_raw) | per-draw 'z','x' parts as (hi,lo) float pairs ]
then yields the exact full-batch gradient and loss on every rank.  The other 16 tensors only see
prior/entropy terms, are computed redundantly (deterministic kernels => bit-identical replicas)
and are not communicated.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _abi


def shard_rows(n_rows, rank, world):
    """Contiguous row block [lo, hi) of this rank (SURVEY.md 8e partition)."""
    base, rem = divmod(n_rows, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def comm_block(eng):
    """The all-reduced view: data-touched gradients followed by the scalar slack."""
    return eng.grads[: eng.layout.n_data_block]


def unpack_data_parts(eng, parts):
    """Write the all-reduced ('z','x') sums back into parts[:,13:15] and recompute the per-draw loss."""
    L = eng.layout
    S = eng.S
    sl = eng.grads[L.comm_off: L.comm_off + 4 * S].to(torch.float64).view(S, 4)
    parts[:, 13] = sl[:, 0] + sl[:, 1]
    parts[:, 14] = sl[:, 2] + sl[:, 3]
    prior = parts[:, :12].sum(1)
    parts[:, 15] = eng.entropy_weight * parts[:, 12] - eng.prior_weight * prior - parts[:, 13] - parts[:, 14]
    eng.grads[L.comm_off: L.comm_off + L.comm_slack].zero_()
    return parts


_LINKS = {}


def peer_link(eng, group=None):
    """The PeerLink of this engine's (shared) parameter buffer, set up on first use -- a collective call: every
    rank reaches it at its first optimiser step.  None when the buffers cannot be peer-mapped on this node
    (decided collectively; the NCCL all-reduce path is used instead) or SPMF_P2P=0."""
    from . import p2p
    if not p2p.enabled():
        return None
    key = (eng.params.data_ptr(), eng.grads.data_ptr())
    if key not in _LINKS:
        _LINKS[key] = p2p.PeerLink(eng.params, eng.grads, eng.device, group)
    link = _LINKS[key]
    return link if link.ok else None


def check_exchange(eng):
    """Raise if a peer-memory exchange of this engine gave up waiting for a rank (host sync; fit calls it once
    per epoch next to its loss read-back)."""
    link = _LINKS.get((eng.params.data_ptr(), eng.grads.data_ptr()))
    if link is not None and link.ok:
        link.check()


def exchange_kind(eng):
    link = _LINKS.get((eng.params.data_ptr(), eng.grads.data_ptr()))
    return "p2p-kernel" if (link is not None and link.ok) else "nccl-allreduce"


def gather_owned(eng, t, group=None):
    """Full copy of a per-parameter buffer (adam_m / adam_v or a snapshot of them) of which, under the peer-memory
    exchange, each rank holds only its owned slice of the reduced block current (spmf_p2p_owned_range); the
    replicated tail [n_data_block, n_params) is the same on every rank and is taken from this one.  Collective."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    spans = [_abi.p2p_owned_range(eng.layout.comm_off, world, q) for q in range(world)]
    width = max(hi - lo for lo, hi in spans)
    lo, hi = spans[rank]
    mine = torch.zeros(width, dtype=t.dtype, device=t.device)
    mine[:hi - lo] = t[lo:hi]
    pieces = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(pieces, mine, group=group)
    full = t.clone()
    for (a, b), piece in zip(spans, pieces):
        full[a:b] = piece[:b - a]
    return full


def allreduce_step(eng, parts, group=None, adam=False):
    """All-reduce gradients + data parts in one collective; returns the global loss (0-d tensor).
    adam=True: the optimiser step (all 24 tensors; the 16 replicated ones are bit-identical on every rank)
    rides in the same launch as the post-collective bookkeeping."""
    dev = getattr(eng, "device", None)
    if adam and dev is not None and dev.type == "cuda" and eng.S <= 64:
        link = peer_link(eng, group)
        if getattr(eng, "_loss_buf", None) is None:
            eng._loss_buf = torch.zeros(1, dtype=torch.float64, device=eng.device)
        if link is not None:
            # ONE kernel per rank over NVLink peer memory: reduce-scatter -> Adam -> all-gather (no NCCL call)
            link.reduce_adam(eng, parts, eng.adam_args(), eng._loss_buf, skip_tail=eng.tail_stepped)
            eng.launches += 1
            return eng._loss_buf[0]
    dist.all_reduce(comm_block(eng), op=dist.ReduceOp.SUM, group=group)
    if adam and dev is not None and dev.type == "cuda" and eng.S <= 64:
        import ctypes as C
        L = eng.layout
        slack = eng.grads[L.comm_off: L.comm_off + L.comm_slack]
        a = eng.adam_args()
        _abi.call("spmf_unpack_adam", slack.data_ptr(), L.comm_slack, eng.S, eng.entropy_weight, eng.prior_weight,
                  parts.data_ptr(), eng._loss_buf.data_ptr(), eng.grads.data_ptr(),
                  L.n_data_block if eng.tail_stepped else L.n_params, C.byref(a),
                  torch.cuda.current_stream().cuda_stream)
        eng.launches += 1
        return eng._loss_buf[0]
    if dev is not None and dev.type == "cuda" and eng.S <= 64:
        # one launch instead of a handful of tiny tensor ops on the critical path between the
        # collective and Adam
        L = eng.layout
        if getattr(eng, "_loss_buf", None) is None:
            eng._loss_buf = torch.zeros(1, dtype=torch.float64, device=eng.device)
        slack = eng.grads[L.comm_off: L.comm_off + L.comm_slack]
        _abi.call("spmf_unpack_parts", slack.data_ptr(), L.comm_slack, eng.S, eng.entropy_weight, eng.prior_weight,
                  parts.data_ptr(), eng._loss_buf.data_ptr(), torch.cuda.current_stream().cuda_stream)
        eng.launches += 1
        return eng._loss_buf[0]
    unpack_data_parts(eng, parts)
    return parts[:, 15].mean()
