"""ctypes binding of the C ABI declared in include/spmf_b200.h.

The shared library is the product: if it is missing or a call fails, we raise -- there is no
CPU / PyTorch fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libspmf_b200.so")

NUM_TENSORS = 24
NUM_VARS = 12
NUM_PARTS = 16
MAX_K = 512        # latent dimensions of the gather / dense kernels (SPMF_MAX_K)
MAX_TILE_K = 128   # latent dimensions of the tensor-core hybrid path (SPMF_MAX_TILE_K)


class SpmfError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python spmf_b200/build.py` "
            "(nvcc, sm_100a).  spmf_b200 has no CPU fallback.")
    return C.CDLL(LIB_PATH)


_lib = _load()

p = C.c_void_p
i32 = C.c_int
i64 = C.c_longlong
f32 = C.c_float
u64 = C.c_ulonglong
u32 = C.c_uint

_SIGS = {
    "spmf_kpad": (i32, [i32]),
    "spmf_draw_vec": (i32, [i32]),
    "spmf_draw_vec_k": (i32, [i32, i32]),
    "spmf_rec_pos": (i32, [i32, i32, i32, i32]),
    "spmf_layout": (i32, [i32, i32, i32, C.POINTER(i64), C.POINTER(i64)]),
    "spmf_backward_scratch_floats": (i64, [i32, i32, i32]),
    "spmf_backward_scratch_doubles": (i64, [i32, i32, i32]),
    "spmf_fill_noise": (i32, [p, p, i32, i32, i32, u64, u32, i32, p]),
    "spmf_sample": (i32, [p, p, i32, i32, i32, p, p]),
    "spmf_draw_operands": (i32, [p, p, p, i32, i32, i32, p, p, p, p, p, p, p]),
    "spmf_csr_row_consts": (i32, [p, p, i64, p, p, p]),
    "spmf_csr_rows": (i32, [p, p, p, p, p, f32, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, i32, p, p]),
    "spmf_csr_encode": (i32, [p, p, p, p, f32, i32, i32, i32, i32, i32, p, p, p]),
    "spmf_csc_cols": (i32, [p, p, p, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, i32, p]),
    "spmf_batch_sums": (i32, [p, p, i32, i32, i32, p, p, p, p]),
    "spmf_gamma_grad": (i32, [p, p, i32, i32, i32, p, p]),
    "spmf_gamma_draw_grad": (i32, [p, p, p, i32, i32, i32, u64, u32, p]),
    "spmf_backward_params": (i32, [p, p, p, p, i32, i32, i32, p, p, p, p, p, p, f32, f32, f32, f32, f32,
                                   f32, i32, p, p, p, p, p, p]),
    "spmf_backward_pre": (i32, [p, p, p, p, i32, i32, i32, f32, f32, f32, f32, f32, f32, i32, p, p, p, p]),
    "spmf_backward_post": (i32, [p, p, p, p, i32, i32, i32, p, p, p, p, p, p, f32, f32, f32, f32, f32, f32, i32,
                                 p, p, p, p, p, p]),
    "spmf_unpack_adam": (i32, [p, i32, i32, f32, f32, p, p, p, i64, p, p]),
    "spmf_adam_step": (i32, [p, p, p, p, i64, f32, f32, f32, f32, i32, f32, f32, p]),
    "spmf_unpack_parts": (i32, [p, i32, i32, f32, f32, p, p, p]),
    "spmf_sumsq": (i32, [p, i64, p, p, p, p]),
    "spmf_colsum": (i32, [p, i64, i32, i32, p, p, p]),
    "spmf_csr_colstats": (i32, [p, p, i64, i32, p, p, p]),
    "spmf_csc_scratch_ints": (i64, [i32]),
    "spmf_csr_to_csc": (i32, [p, p, p, i32, i32, p, p, p, p, p]),
    "spmf_csr_unpack16": (i32, [p, p, i64, p, p, p]),
    "spmf_csr_unpack8": (i32, [p, p, p, i32, p, p, i32, p, p, p]),
    "spmf_dense_count": (i32, [p, i32, i32, p, p]),
    "spmf_dense_fill": (i32, [p, i32, i32, p, p, p, p]),
    "spmf_version": (C.c_char_p, []),
    # hybrid path (tcgen05 hot block)
    "spmf_hybrid_supported": (i32, [i32, i32]),
    "spmf_draw_operands_ranked": (i32, [p, p, p, p, i32, i32, i32, p, p, p, p, p, p, p]),
    "spmf_operand_sums": (i32, [p, p, i32, i32, i32, p, p, p, p]),
    "spmf_backward_params_ranked": (i32, [p, p, p, p, p, i32, i32, i32, p, p, p, p, p, p, f32, f32, f32, f32,
                                          f32, f32, i32, p, p, p, p, p, p]),
    "spmf_umma_tiled_a_elems": (i64, [i64, i64]),
    "spmf_umma_tiled_b_elems": (i64, [i32, i64]),
    "spmf_umma_tiled_a_index": (i64, [i64, i64, i64]),
    "spmf_umma_tile_a": (i32, [p, i64, i32, i32, p, p]),
    "spmf_umma_gemm3_at": (i32, [p, i32, i32, i32, p, i64, p, i64, i64, i32, i32, i32, p]),
    "spmf_umma_probe": (i32, [p, i32, p, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, p, p]),
    "spmf_hot_split": (i32, [p, p, p, i32, i64, p, i32, p, p, p, p, p, p, p, p]),
    "spmf_hot_split_u8": (i32, [p, p, p, p, p, i32, i32, p, i32, p, p, p, p, p, p, p, p]),
    "spmf_hot_split_packed": (i32, [p, p, p, p, p, i32, i64, p, i32, p, p, p, p, p, p, p, p]),
    "spmf_split3_transpose": (i32, [p, i64, i64, i32, i32, i32, p, i64, i32, p]),
    "spmf_umma_gemm3": (i32, [p, i64, i32, p, i64, p, i64, i64, i32, i32, i32, i32, p]),
    "spmf_hot_tile_scratch_bytes": (i64, [i32, i32, i32]),
    "spmf_hot_ev_tiles": (i32, [p, p, i32, i32, i32, i32, p, p]),
    "spmf_csr_rows_cold": (i32, [p, p, p, p, p, f32, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, p]),
    "spmf_hot_tile": (i32, [p, p, p, i32, i32, i32, i32, i32, p, p, p, p, p, p]),
    "spmf_rows_finish": (i32, [p, p, f32, i32, i32, i32, i32, p, p, p, p, p, p]),
    # dense evaluation of the data term: log / Bernoulli links, exact non-finite guard (spmf_dense.cu)
    "spmf_guard_state_bytes": (i32, []),
    "spmf_guard_reset": (i32, [p, i32, p]),
    "spmf_guard_decode": (i32, [p, C.POINTER(i32), C.POINTER(i32), C.POINTER(f32)]),
    "spmf_dense_scatter": (i32, [p, p, p, i32, i32, p, p]),
    "spmf_dense_encode": (i32, [p, p, p, f32, i32, i32, i32, i32, i32, i32, p, p, p]),
    "spmf_dense_rows": (i32, [p, p, p, f32, i32, i32, i32, i32, i32, i32, i32, i32, p, p, p, p, p, p, p]),
    "spmf_dense_cols": (i32, [p, p, i32, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, p, p]),
    "spmf_guard_rows_fix": (i32, [p, p, p, p, p, f32, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, p]),
    "spmf_guard_cols_fix": (i32, [i32, i32, i32, i32, p, p, p, p, p, p, p, p]),
    "spmf_guard_rows_fix_dense": (i32, [p, i32, p, p, p, f32, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, p]),
    "spmf_dense_hot_split": (i32, [p, i32, i32, i32, p, i32, p, p, p, p, p, p, p, p]),
    "spmf_zero_col_grads": (i32, [p, p, p, i32, i32, i32, p]),
    "spmf_csc_cols_accum": (i32, [p, p, p, i32, i32, i32, i32, i32, p, p, p, p, p, p, p, p]),
    "spmf_csr_to_csc_part": (i32, [p, p, i32, p, p, i32, i32, p, p, p, p, p]),
}



class AdamArgs(C.Structure):
    """Mirror of `spmf_adam_args` (include/spmf_b200.h)."""
    _fields_ = ([(n, f32) for n in ("lr", "beta1", "beta2", "eps", "clip_value", "grad_scale")]
                + [("step", i32), ("reserved", i32), ("params", p), ("m", p), ("v", p)])


P2P_MAX_WORLD, P2P_HANDLE_BYTES = 8, 64


class P2PArgs(C.Structure):
    """Mirror of `spmf_p2p_args` (include/spmf_b200.h)."""
    _fields_ = ([(n, i32) for n in ("world", "rank", "S", "slack")] + [("epoch", u32), ("skip_tail", i32)]
                + [(n, i64) for n in ("n_params", "n_block", "comm_off")]
                + [("w_entropy", C.c_double), ("w_prior", C.c_double)]
                + [("grads", p * P2P_MAX_WORLD), ("params", p * P2P_MAX_WORLD), ("flags", p * P2P_MAX_WORLD)]
                + [("parts", p), ("loss_out", p), ("adam", C.POINTER(AdamArgs))])


class StepArgs(C.Structure):
    """Mirror of `spmf_step_args` (include/spmf_b200.h), field for field."""
    _fields_ = (
        [(n, i32) for n in ("D", "K", "S", "world_size")]
        + [(n, f32) for n in ("u_tau_scale", "s_tau_scale", "decay", "w_entropy", "w_prior", "inv_xi")]
        + [("scale_rows", i32), ("fresh_noise", i32), ("rng_step", u32), ("seed", u64)]
        + [(n, p) for n in ("params", "grads", "adam_m", "adam_v", "noise", "dgda", "eta")]
        + [(n, i64) for n in ("n_params", "comm_off", "comm_slack")]
        + [(n, p) for n in ("Ap", "EV", "PH", "GAp", "GEV", "Gph", "z", "dzr", "rowacc", "scr_f",
                            "vsum", "phisum", "zcolsum", "datasums", "parts", "scr_d",
                            "rowptr", "cols", "vals", "rowsum", "lgam", "colptr", "crows", "cvals")]
        + [("nrows", i32), ("nnz", i32)]
        + [(n, f32) for n in ("adam_lr", "adam_beta1", "adam_beta2", "adam_eps", "clip_value")]
        + [("adam_t", i32)]
        + [(n, p) for n in ("caller_stream", "hot_stream", "side_stream", "ev_fork", "ev_join", "ev_done",
                            "ev_rows0", "ev_rows1", "ev_cols0", "ev_cols1")]
        + [("rank", p), ("hot_cols", i32), ("gemm_splits", i32)]
        + [("t3_qstride", i64)]
        + [(n, p) for n in ("rowmid", "xhot", "ApT3", "dzrT3",
                            "ev_gemm0", "ev_gemm1", "aux_stream1", "aux_stream2", "ev_aux_fork", "ev_aux_join1",
                            "ev_aux_join2")]
        + [("EVt", p), ("ev_tile0", p), ("ev_tile1", p), ("scr_dpre", p), ("ev_noise", p)]
        + [("link", i32), ("gs", p), ("xdense", p), ("xdense_in", p), ("step_state", p), ("model", i32), ("state_preset", i32), ("dense_raw", p), ("dense_raw_dtype", i32), ("adam_tail_early", i32)]
    )


_SIGS["spmf_advi_step"] = (i32, [C.POINTER(StepArgs)])
_SIGS["spmf_step_graph_create"] = (i32, [C.POINTER(StepArgs), C.POINTER(p)])
_SIGS["spmf_step_graph_launch"] = (i32, [p, u32, i32, f32, f32, f32, f32, f32, p])
_SIGS["spmf_step_graph_destroy"] = (i32, [p])
_SIGS["spmf_step_state_bytes"] = (i32, [])
_SIGS["spmf_step_state_set"] = (i32, [p, u32, i32, f32, f32, f32, f32, f32, p])
_SIGS["spmf_step_state_kernel_ptr"] = (p, [])
_SIGS["spmf_step_state_value"] = (i32, [u32, i32, f32, f32, f32, f32, f32, p])
_SIGS["spmf_fill_noise_dev"] = (i32, [p, p, i32, i32, i32, u64, u32, i32, p, p])
_SIGS["spmf_gamma_draw_grad_dev"] = (i32, [p, p, p, i32, i32, i32, u64, u32, p, p])
_SIGS["spmf_adam_step_dev"] = (i32, [p, p, p, p, i64, f32, f32, f32, f32, i32, f32, f32, p, p])
_SIGS["spmf_sample_m"] = (i32, [p, p, i32, i32, i32, p, i32, p])
_SIGS["spmf_draw_operands_ranked_m"] = (i32, [p, p, p, p, i32, i32, i32, p, p, p, p, p, p, i32, p])
_SIGS["spmf_backward_params_ranked_m"] = (i32, [p, p, p, p, p, i32, i32, i32, p, p, p, p, p, p, f32, f32, f32, f32,
                                                 f32, f32, i32, p, p, p, p, p, i32, p])
_SIGS["spmf_backward_pre_m"] = (i32, [p, p, p, p, i32, i32, i32, f32, f32, f32, f32, f32, f32, i32, p, p, p, i32, p])
_SIGS["spmf_backward_post_m"] = (i32, [p, p, p, p, i32, i32, i32, p, p, p, p, p, p, f32, f32, f32, f32, f32, f32, i32,
                                        p, p, p, p, p, i32, p])
_SIGS["spmf_prepare_batch"] = (i32, [p, p, p, p, p, i32, i64, i32, p, p, p, p, p, p, p])

_SIGS["spmf_p2p_alloc"] = (i32, [i64, p])
_SIGS["spmf_p2p_free"] = (i32, [p])
_SIGS["spmf_p2p_export"] = (i32, [p, p])
_SIGS["spmf_p2p_open"] = (i32, [p, p])
_SIGS["spmf_p2p_close"] = (i32, [p])
_SIGS["spmf_p2p_flag_bytes"] = (i64, [])
_SIGS["spmf_p2p_status"] = (i32, [p, p])
_SIGS["spmf_p2p_reduce_adam"] = (i32, [p, p])
_SIGS["spmf_p2p_owned_range"] = (i32, [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)])

EXPORTS = tuple(_SIGS)

for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(_lib, _name)      # AttributeError here = header / library mismatch
    _fn.restype = _res
    _fn.argtypes = _args


def _check(rc, name):
    if rc != 0:
        kind = {-1: "bad argument", -2: "unsupported configuration",
                -3: "a peer rank never reached the exchange"}.get(rc, f"CUDA error {rc}")
        raise SpmfError(f"{name} failed: {kind}")


def call(name, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    _check(getattr(_lib, name)(*args), name)


LINK_POISSON, LINK_POISSON_LOG, LINK_BERNOULLI, LINK_BERNOULLI_LOG = 0, 1, 2, 3
MODEL_POISSON, MODEL_BERNOULLI = 0, 1
DENSE_U8, DENSE_U16, DENSE_F32 = 1, 2, 4
DENSE_OPTIMISTIC, DENSE_STATS, DENSE_GUARDED = 0, 1, 2


def kpad(K):
    return _lib.spmf_kpad(K)


def draw_vec(S):
    return _lib.spmf_draw_vec(S)


def draw_vec_k(K, S):
    """Draws per gather record for latent dim K (what every device layout uses)."""
    return _lib.spmf_draw_vec_k(K, S)


_REC_PERM = {}


def rec_perm(KP, SV):
    """perm[sv*KP + k] = position of (sv,k) inside a gather record (list of ints, cached)."""
    key = (KP, SV)
    if key not in _REC_PERM:
        perm = [_lib.spmf_rec_pos(KP, SV, sv, k) for sv in range(SV) for k in range(KP)]
        if min(perm) < 0 or sorted(perm) != list(range(KP * SV)):
            raise SpmfError("spmf_rec_pos does not define a permutation")
        _REC_PERM[key] = perm
    return _REC_PERM[key]


def layout(D, K, S):
    t = (i64 * (NUM_TENSORS + 1))()
    n = (i64 * (NUM_VARS + 1))()
    _check(_lib.spmf_layout(D, K, S, t, n), "spmf_layout")
    return list(t), list(n)


def p2p_owned_range(comm_off, world, rank):
    """Floats [lo, hi) of the reduced block whose Adam moments `rank` holds under the peer-memory exchange."""
    lo, hi = i64(), i64()
    _check(_lib.spmf_p2p_owned_range(int(comm_off), int(world), int(rank), C.byref(lo), C.byref(hi)),
           "spmf_p2p_owned_range")
    return lo.value, hi.value


def backward_scratch(D, K, S):
    return (_lib.spmf_backward_scratch_floats(D, K, S), _lib.spmf_backward_scratch_doubles(D, K, S))


def version():
    return _lib.spmf_version().decode()
