"""CPU tests of the boundary: the C-ABI library loads without a GPU, exports every symbol the header declares,
validates arguments before touching CUDA, and the product path refuses to run without it (no fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "ss2d_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ss2d_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from ceigm_unet_b200 import _lib
    L = _lib.lib()
    declared = _declared_symbols()
    assert declared, "no declarations parsed"
    assert sorted(_lib.EXPORTS) == declared
    for name in declared:
        assert hasattr(L, name), name


def test_version_and_strerror():
    from ceigm_unet_b200 import _lib
    assert "sm_100a" in _lib.version()
    L = _lib.lib()
    assert L.ss2d_strerror(0) == b"ok"
    assert b"256" in L.ss2d_strerror(-4)
    assert L.ss2d_strerror(-123) == b"unknown status"


def test_descriptor_validation_needs_no_gpu():
    from ceigm_unet_b200 import _lib
    L = _lib.lib()
    d = _lib.ScanDesc()
    d.batch, d.dim, d.seqlen, d.dstate, d.n_groups = 2, 12, 64, 16, 4
    assert L.ss2d_scan_ckpt_floats(ctypes.byref(d)) == 2 * 12 * 2 * 16
    assert L.ss2d_scan_bwd_workspace_bytes(ctypes.byref(d), 1) == 4 * (2 * 12 * 18)
    d.n_groups = 5                                   # 12 % 5 != 0
    assert L.ss2d_scan_ckpt_floats(ctypes.byref(d)) == 0
    assert L.ss2d_scan_fwd(ctypes.byref(d), None, None, None, None, None, None, None, None, None, None, None) == -2
    d.n_groups, d.dstate = 4, 257
    assert L.ss2d_scan_fwd(ctypes.byref(d), None, None, None, None, None, None, None, None, None, None, None) == -4
    d.dstate = 16
    assert L.ss2d_scan_fwd(ctypes.byref(d), None, None, None, None, None, None, None, None, None, None, None) == -1
    d.layout, d.H, d.W = 1, 8, 8
    d.dirs[0], d.dirs[1], d.dirs[2], d.dirs[3] = 1, 2, 3, 9
    assert L.ss2d_scan_fwd(ctypes.byref(d), None, None, None, None, None, None, None, None, None, None, None) == -5
    assert L.ss2d_out_gate_bwd_partials(24, 3136) == 592


def test_struct_layout_matches_header():
    from ceigm_unet_b200 import _lib
    # 11 int32 + 8 dirs + 12 int64 + 2 int32, 8-byte aligned: offsets must match the C struct
    assert _lib.ScanDesc.dirs.offset == 44
    assert _lib.ScanDesc.u_batch_stride.offset == 80
    assert _lib.ScanDesc.grads_prezeroed.offset == 80 + 12 * 8 + 8
    assert ctypes.sizeof(_lib.ScanDesc) == 80 + 12 * 8 + 16      # 3 trailing int32 padded to the struct's 8-byte alignment


def test_no_fallback_without_library(monkeypatch):
    from ceigm_unet_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libss2d_b200.so")
    with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def test_cpu_tensors_are_rejected():
    import torch
    from ceigm_unet_b200.dropin import selective_scan_cuda_core as core
    u = torch.randn(1, 4, 16)
    with pytest.raises(RuntimeError, match="is_cuda"):
        core.fwd(u, u, torch.randn(4, 2), torch.randn(1, 1, 2, 16), torch.randn(1, 1, 2, 16), None, None, True, 1)


def test_product_path_never_imports_oracle():
    pkg = os.path.join(ROOT, "ceigm-unet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, os.path.join(dirpath, f)


def test_constructors_reproduce_reference_init_bit_exactly():
    """Same seed -> same parameters as the reference constructors (RNG consumption order of mamba_init / __initv2__)."""
    import numpy as np
    import torch
    import ceigm_unet_b200 as P
    z = np.load(os.path.join(ROOT, "tests", "golden", "init_seed1234.npz"))
    cases = [("gm.", lambda: P.SS2D(d_model=32, d_state=1, ssm_ratio=1, d_conv=3)),
             ("vm.", lambda: P.SS2D(d_model=16, d_state=16, ssm_ratio=2.0, k_group=4)),
             ("layer.", lambda: P.GroupMambaLayer(64, 64))]
    for prefix, make in cases:
        torch.manual_seed(1234)
        sd = make().state_dict()
        ref = {k[len(prefix):]: z[k] for k in z.files if k.startswith(prefix)}
        assert list(sd.keys()) == list(ref.keys()), prefix
        for k, v in sd.items():
            assert np.array_equal(v.numpy(), ref[k]), prefix + k


def test_reference_python_picks_up_the_dropin_modules():
    """With install_dropin(), the UNMODIFIED reference csms6s.py (harness/install_ref.py) binds our extension modules."""
    from harness import refmodel
    if not refmodel.available():
        pytest.skip("reference tree not installed (harness/install_ref.py)")
    ref = os.path.join(refmodel.ref_root(), "model", "gm", "csms6s.py")
    import importlib.util
    import sys
    import warnings
    import ceigm_unet_b200 as P
    P.install_dropin()
    spec = importlib.util.spec_from_file_location("_ref_csms6s_probe", ref)
    mod = importlib.util.module_from_spec(spec)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        spec.loader.exec_module(mod)
    assert mod.selective_scan_cuda_core is sys.modules["selective_scan_cuda_core"]
    assert mod.selective_scan_cuda_core.__name__ == "ceigm_unet_b200.dropin.selective_scan_cuda_core"
    assert mod.selective_scan_cuda_oflex.__name__ == "ceigm_unet_b200.dropin.selective_scan_cuda_oflex"
    # the reference's own autograd wrapper now reaches our fwd(): on this CPU-only box it must fail loudly, not fall back
    import torch
    u = torch.randn(1, 4, 16)
    with pytest.raises(RuntimeError, match="is_cuda"):
        mod.SelectiveScanCore.apply(u, u, torch.randn(4, 2), torch.randn(1, 1, 2, 16), torch.randn(1, 1, 2, 16), None, None, True)
