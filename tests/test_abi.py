"""CPU tests of the drop-in boundary: the shared library loads, exports every symbol that
include/spmf_b200.h declares (and nothing the Python binding expects is missing), the host-only
helpers agree with the host-check build, and compute entry points reject bad arguments /
fail without a device instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "spmf_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(spmf_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from spmf_b200 import _abi
    lib = ctypes.CDLL(_abi.LIB_PATH)
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/spmf_b200.h but not exported"
    assert set(_abi.EXPORTS) == set(names), set(_abi.EXPORTS) ^ set(names)


def test_header_cites_reference_lines():
    src = open(HEADER).read()
    assert "poisson.py:156-184" in src and "poisson.py:113-154" in src and ":623-650" in src


def test_layout_matches_hostcheck_and_var_list():
    from spmf_b200 import _abi
    from spmf_b200.variables import VAR_LIST, VariableLayout
    import tests.hostcheck as hc
    for D, K, S in ((7, 3, 2), (100, 2, 4), (333, 50, 1), (2000, 128, 8)):
        t, n = _abi.layout(D, K, S)
        th, nh = hc.layout(D, K, S)
        assert t == list(th) and n == list(nh)
        L = VariableLayout(D, K, S)
        assert L.n_params == t[-1] and L.n_data_block == t[8]
        assert all(o % 32 == 0 for o in t)
    assert VAR_LIST == ['v', 'w', 'u', 'u_eta', 'u_tau', 's_eta', 's_tau', 's', 'u_eta_a', 'u_tau_a', 's_eta_a', 's_tau_a']
    assert _abi.kpad(50) == 64 and _abi.kpad(32) == 32 and _abi.kpad(1) == 1
    assert (_abi.draw_vec(4), _abi.draw_vec(6), _abi.draw_vec(3), _abi.draw_vec(80)) == (4, 2, 1, 4)


def test_bad_arguments_are_rejected():
    from spmf_b200 import _abi
    with pytest.raises(_abi.SpmfError):
        _abi.layout(10, 0, 1)
    with pytest.raises(_abi.SpmfError):
        _abi.layout(10, _abi.MAX_K + 1, 1)
    with pytest.raises(_abi.SpmfError):       # null pointers
        _abi.call("spmf_fill_noise", None, None, 10, 2, 1, 0, 0, 3, None)
    with pytest.raises(_abi.SpmfError):
        _abi.call("spmf_csr_rows", *([None] * 5), 1.0, 1, 4, 10, 2, 1, *([None] * 7), 0, None, None)
    with pytest.raises(_abi.SpmfError):       # dense-link entry points validate the same way
        _abi.call("spmf_dense_rows", *([None] * 3), 1.0, 1, 4, 10, 2, 1, 1, 0, 0, *([None] * 7))
    assert _abi._lib.spmf_guard_state_bytes() == 24


def test_no_cpu_fallback():
    """The product refuses to compute without a CUDA device (and never imports the oracle)."""
    import torch
    import spmf_b200
    if not torch.cuda.is_available():
        with pytest.raises((spmf_b200.SpmfError, RuntimeError, AssertionError)):
            spmf_b200.PoissonFactorization(latent_dim=2, feature_dim=5, device="cpu")
    import sys
    pkg = os.path.join(ROOT, "spmf_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f


def test_variable_views_roundtrip_on_host():
    """Views into the flat buffer have the reference shapes; v is stored transposed."""
    import torch
    from spmf_b200.variables import VariableLayout, var_shapes
    L = VariableLayout(6, 3, 2)
    flat = torch.zeros(L.n_params)
    L.fill_initial(flat, 0.01, 1.0)
    views = L.views(flat)
    sh = var_shapes(6, 3)
    assert list(views) == L.param_names()
    for name, v in views.items():
        assert tuple(v.shape) == sh[name.split('/')[0]]
    assert views['v/loc'].shape == (3, 6) and not views['v/loc'].is_contiguous()
    assert float(views['s/loc'][0, 0]) == -2.0 and float(views['s/loc'][1, 0]) == -1.0
    sp = torch.nn.functional.softplus
    assert abs(float(sp(views['u_tau_a/scale_raw'][0, 0])) - 1e4) < 1e-2
    views['v/loc'][1, 4] = 7.0
    assert flat[L.toff[0] + 4 * 3 + 1] == 7.0


def test_step_args_struct_matches_header(tmp_path):
    """ctypes mirror of spmf_step_args has the C layout (size and a few offsets), checked with gcc."""
    import subprocess
    from spmf_b200 import _abi
    src = tmp_path / "sz.c"
    fields = ["seed", "params", "n_params", "vsum", "rowptr", "nrows", "adam_lr", "adam_t", "caller_stream", "ev_cols1",
              "rank", "hot_cols", "t3_qstride", "rowmid", "xhot", "dzrT3", "ev_gemm1", "aux_stream2", "ev_aux_join2", "EVt", "ev_tile1", "scr_dpre", "ev_noise", "link", "step_state", "dense_raw", "dense_raw_dtype", "adam_tail_early"]
    prints = "".join(f'printf("%zu\\n", offsetof(spmf_step_args, {f}));' for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu\\n", sizeof(spmf_step_args));%s return 0;}\n'
                   % (HEADER, prints))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert out[0] == ctypes.sizeof(_abi.StepArgs)
    for f, off in zip(fields, out[1:]):
        assert getattr(_abi.StepArgs, f).offset == off, f


def test_p2p_args_struct_matches_header(tmp_path):
    """ctypes mirrors of spmf_p2p_args / spmf_adam_args have the C layout (gcc)."""
    import subprocess
    from spmf_b200 import _abi
    src = tmp_path / "sz.c"
    fields = ["epoch", "skip_tail", "n_params", "comm_off", "w_prior", "grads", "params", "flags", "parts", "loss_out", "adam"]
    prints = "".join(f'printf("%zu\\n", offsetof(spmf_p2p_args, {f}));' for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu\\n%%zu\\n", '
                   'sizeof(spmf_p2p_args), sizeof(spmf_adam_args));%s return 0;}\n' % (HEADER, prints))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert out[0] == ctypes.sizeof(_abi.P2PArgs) and out[1] == ctypes.sizeof(_abi.AdamArgs)
    for f, off in zip(fields, out[2:]):
        assert getattr(_abi.P2PArgs, f).offset == off, f
    assert _abi.P2P_MAX_WORLD == 8 and _abi.P2P_HANDLE_BYTES == 64
