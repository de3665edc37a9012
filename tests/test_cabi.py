"""C-ABI surface (no GPU needed): the library loads and exports every symbol include/vdb200.h declares,
and the ctypes signature table covers exactly that set."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "vdb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return set(re.findall(r"\b(vdb_[a-z0-9_]+)\s*\(", src))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from vdb200 import _lib
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(_lib.lib, s), f"{s} declared in include/vdb200.h but not exported by libvdb200.so"
    assert set(_lib.SIGNATURES) == syms, sorted(set(_lib.SIGNATURES) ^ syms)
    assert _lib.lib.vdb_version().startswith(b"vdb200")


def test_host_side_argument_checks_without_gpu():
    """Entry points validate arguments before touching the device: bad calls return VDB_ERR_INVALID + a message."""
    from vdb200._lib import lib
    assert lib.vdb_ddim_cfg_step(None, None, None, None, None, None, 1.0, 1.0, None, None, None, 0, None) == 1
    assert b"ddim_cfg_step" in lib.vdb_last_error()
    assert lib.vdb_gemm_bf16(None, 0, 0, 0, None, 0, 0, None, 0, 0, None, 0, 0, None, 0, None, 0, 0, 0, 1.0, 0, 0, None, 0, None) == 1
    assert lib.vdb_attention_dk_pad(40) == 64 and lib.vdb_attention_dv_pad(40) == 48
    assert lib.vdb_attention_dk_pad(160) == 192 and lib.vdb_attention_dv_pad(160) == 160
    # one (DK, DVP) pair per attention kernel: d_head 81..160 share the (192, 160) one
    assert [lib.vdb_attention_dk_pad(d) for d in (8, 64, 72, 80, 88, 96, 120, 128, 136)] == [64, 64, 128, 128, 192, 192, 192, 192, 192]
    assert [lib.vdb_attention_dv_pad(d) for d in (48, 56, 80, 88, 128)] == [48, 64, 80, 160, 160]
    assert lib.vdb_attention_dk_pad(168) == -1 and lib.vdb_attention_dv_pad(168) == -1
    assert lib.vdb_attention_dk_pad(512) == -1


def test_product_path_refuses_cpu_tensors():
    import pytest
    import torch
    from vdb200 import ops
    with pytest.raises(ValueError, match="no CPU fallback"):
        ops.layernorm(torch.zeros(4, 64, dtype=torch.bfloat16), torch.ones(64), torch.zeros(64))
