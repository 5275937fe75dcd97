"""CPU tests of the checkpoint plumbing: the owned-range helper of the peer-memory exchange
(spmf_p2p_owned_range), the gather of per-rank moment slices (gloo, world 2 and 3) and the CLI flags."""
import importlib.util
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_owned_ranges_cover_the_block_once_in_rank_order():
    from spmf_b200 import _abi
    for comm_off in (0, 4, 12, 32, 1020, 4096, 10004, 2_702_336, 10_725_376):
        nvec = comm_off // 4
        for world in range(1, _abi.P2P_MAX_WORLD + 1):
            spans = [_abi.p2p_owned_range(comm_off, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == comm_off, (comm_off, world, spans)
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:])), (comm_off, world, spans)
            assert all(lo <= hi and lo % 4 == 0 and hi % 4 == 0 for lo, hi in spans)
            per = (nvec + world - 1) // world              # the exchange kernel's split: ceil(nvec / world) vectors
            assert all(hi - lo == 4 * min(per, max(nvec - per * r, 0)) for r, (lo, hi) in enumerate(spans))


def test_owned_range_rejects_bad_arguments():
    from spmf_b200 import _abi
    for args in ((6, 2, 0), (-4, 2, 0), (16, 0, 0), (16, _abi.P2P_MAX_WORLD + 1, 0), (16, 2, 2), (16, 2, -1)):
        with pytest.raises(_abi.SpmfError):
            _abi.p2p_owned_range(*args)


class _FakeEngine:
    def __init__(self, D, K, S):
        from spmf_b200.variables import VariableLayout
        self.layout = VariableLayout(D, K, S)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from spmf_b200 import _abi
    from spmf_b200.parallel import gather_owned
    eng = _FakeEngine(37, 5, 2)
    L = eng.layout
    truth = torch.arange(L.n_params, dtype=torch.float32) * 0.5
    local = torch.full((L.n_params,), -1.0 - rank)             # stale everywhere ...
    lo, hi = _abi.p2p_owned_range(L.comm_off, world, rank)
    local[lo:hi] = truth[lo:hi]                                 # ... except the owned slice
    local[L.comm_off:] = truth[L.comm_off:]                     # slack and replicated tail: the same on every rank
    full = gather_owned(eng, local)
    out[rank] = (full, truth, local)
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gather_owned_assembles_the_full_moments(world):
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gather_worker, args=(world, port, out), nprocs=world, join=True)
    for r in range(world):
        full, truth, local = out[r]
        assert torch.equal(full, truth), r
        assert not torch.equal(local, truth)                    # the input was not complete on its own


def test_cli_checkpoint_flags():
    spec = importlib.util.spec_from_file_location("factorize_csv", os.path.join(ROOT, "bin", "factorize_csv.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    a = m.build_parser().parse_args([])
    assert a.checkpoint is None and a.checkpoint_every == 1
    a = m.build_parser().parse_args(["-f", "x.csv", "--checkpoint", "run.ckpt", "--checkpoint-every", "5"])
    assert a.checkpoint == "run.ckpt" and a.checkpoint_every == 5
