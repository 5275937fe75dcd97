"""Latent dimensions above 128 (up to SPMF_MAX_K = 512) without a GPU: the flat layouts, the gather
record permutations of the wide records and the draws-per-record rule spmf_draw_vec_k."""
import pytest

from spmf_b200 import _abi


@pytest.mark.parametrize("K", [129, 256, 300, 512])
def test_layout_matches_host_check(K):
    import tests.hostcheck as hc
    for D, S in ((10, 1), (37, 4), (64, 3)):
        t, n = _abi.layout(D, K, S)
        ht, hn = hc.layout(D, K, S)
        assert list(t) == list(ht) and list(n) == list(hn)
        assert all(o % 32 == 0 for o in t) and all(o % 32 == 0 for o in n)


@pytest.mark.parametrize("KP,SV", [(256, 1), (256, 2), (512, 1)])
def test_wide_record_permutation(KP, SV):
    perm = _abi.rec_perm(KP, SV)
    assert sorted(perm) == list(range(KP * SV))


def test_draw_vec_k_rule():
    assert _abi.MAX_K == 512 and _abi.MAX_TILE_K == 128
    for S in range(1, 17):
        for K in range(1, _abi.MAX_TILE_K + 1):
            assert _abi.draw_vec_k(K, S) == _abi.draw_vec(S), (K, S)
        for K in range(1, _abi.MAX_K + 1):
            sv = _abi.draw_vec_k(K, S)
            assert sv in (1, 2, 4) and S % sv == 0 and _abi.kpad(K) * sv <= 512, (K, S, sv)
    assert [_abi.draw_vec_k(256, S) for S in (1, 2, 3, 4, 8)] == [1, 2, 1, 2, 2]
    assert [_abi.draw_vec_k(512, S) for S in (1, 2, 4)] == [1, 1, 1]


def test_layout_above_max_k_raises():
    with pytest.raises(_abi.SpmfError):
        _abi.layout(10, 513, 1)


def test_hybrid_path_stops_at_tile_limit():
    assert _abi._lib.spmf_hybrid_supported(128, 4) == 2
    for K, S in ((129, 4), (256, 2), (512, 1)):
        assert _abi._lib.spmf_hybrid_supported(K, S) == 0
