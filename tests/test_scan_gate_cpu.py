"""CPU tests of the selective scan's output gate (ss2d_scan_fwd_gated / ss2d_scan_bwd_gated): the entry points exist, argument
validation, the workspace query, the drop-in's checks that run before any launch, and — from the SASS of the built library —
that the GATE scan_fwdr instantiations exist and that the deterministic dispatch still launches no global atomic."""
import ctypes
import re

import pytest
import torch

from ceigm_unet_b200 import _lib
from test_deterministic_cpu import _GLOBAL_ATOMIC, _desc, _det_launchable, _sass_functions, _ws

ERR_NULL, ERR_WORKSPACE, ERR_UNSUPPORTED, ERR_ALIGNMENT = -1, -6, -8, -9


def test_symbols_exist():
    L = _lib.lib()
    for name in ("ss2d_scan_fwd_gated", "ss2d_scan_bwd_gated", "ss2d_scan_bwd_gated_workspace_bytes"):
        assert hasattr(L, name) and name in _lib.EXPORTS, name


def _p(addr):
    return ctypes.c_void_p(addr) if addr else None


# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000
ODD = GOOD + 1        # misaligned for every element size


def _gws(d, have_ckpt=0):
    return int(_lib.lib().ss2d_scan_bwd_gated_workspace_bytes(ctypes.byref(d), have_ckpt))


def _fwd(d, z=GOOD, out=GOOD, out_z=GOOD, u=GOOD):
    return _lib.lib().ss2d_scan_fwd_gated(ctypes.byref(d), _p(u), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), None, None, None,
                                          _p(z), _p(out), _p(out_z), None, None, None)


def _bwd(d, z=GOOD, out=GOOD, dout_z=GOOD, dz=GOOD, du=GOOD, ws_bytes=None):
    ws_bytes = _gws(d) if ws_bytes is None else ws_bytes
    return _lib.lib().ss2d_scan_bwd_gated(
        ctypes.byref(d), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), None, None, None, _p(z), _p(out), _p(dout_z), None,
        None, _p(du), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), None, None, _p(dz), None, _p(GOOD), ctypes.c_size_t(ws_bytes), None)


def test_required_pointers():
    d = _desc()
    assert _fwd(d, z=0) == ERR_NULL
    assert _fwd(d, out=0) == ERR_NULL            # the backward reads y from out: it is always written
    assert _fwd(d, out_z=0) == ERR_NULL
    assert _fwd(d, u=0) == ERR_NULL
    for kw in ("z", "out", "dout_z", "dz", "du"):
        assert _bwd(d, **{kw: 0}) == ERR_NULL, kw


@pytest.mark.parametrize("dtype", [_lib.SS2D_F32, _lib.SS2D_BF16])
def test_misaligned_gate_operands_are_rejected(dtype):
    d = _desc()
    d.io_dtype = d.out_dtype = dtype
    for kw in ("z", "out", "out_z"):
        assert _fwd(d, **{kw: ODD}) == ERR_ALIGNMENT, kw
    for kw in ("z", "out", "dout_z", "dz"):
        assert _bwd(d, **{kw: ODD}) == ERR_ALIGNMENT, kw


def test_shared_dout_plane_is_unsupported():
    d = _desc()
    d.u_dim_modulo = 3
    assert _fwd(d) == ERR_UNSUPPORTED
    assert _bwd(d) == ERR_UNSUPPORTED


def test_invalid_descriptor_is_rejected_first():
    d = _desc(det=2)
    assert _gws(d) == 0
    assert _fwd(d, z=0) == -2 and _bwd(d, z=0) == -2


@pytest.mark.parametrize("shape", [
    (2, 12, 64, 16, 4),
    (24, 768, 3136, 16, 4),      # vm_d192
    (8, 1536, 2048, 16, 1),      # one Mamba-130m layer
    (2, 384, 784, 4, 4),
    (1, 64, 16384, 1, 4),
    (2, 64, 100, 40, 2),         # two state passes
])
@pytest.mark.parametrize("det", [0, 1])
@pytest.mark.parametrize("dtype", [(_lib.SS2D_F32, _lib.SS2D_F32), (_lib.SS2D_BF16, _lib.SS2D_BF16), (_lib.SS2D_F16, _lib.SS2D_F32)])
def test_gated_workspace_adds_one_fp32_plane(shape, det, dtype):
    b, dim, L, N, G = shape
    d = _desc(b, dim, L, N, G, det=det)
    d.io_dtype, d.out_dtype = dtype
    for have_ckpt in (0, 1):
        assert _gws(d, have_ckpt) == _ws(d, have_ckpt) + 4 * b * dim * L
    assert _bwd(d, ws_bytes=_gws(d) - 4) == ERR_WORKSPACE


def test_dropin_rejects_what_it_does_not_support_before_any_launch():
    from ceigm_unet_b200.dropin import selective_scan_cuda as m
    u = torch.randn(1, 4, 16)
    Bv = torch.randn(1, 1, 2, 16)
    with pytest.raises(RuntimeError, match="complex"):
        m.fwd(u, u, torch.randn(4, 2, dtype=torch.complex64), Bv, Bv, None, None, None, True)
    with pytest.raises(RuntimeError, match="vary along the sequence"):
        m.fwd(u, u, torch.randn(4, 2), torch.randn(4, 2), torch.randn(4, 2), None, None, None, True)
    with pytest.raises(RuntimeError, match="out_ is required"):
        m.bwd(u, u, torch.randn(4, 2), Bv, Bv, None, u, None, u, None, None, None, True, False)
    with pytest.raises(RuntimeError, match="is_cuda"):       # no CPU fallback
        m.fwd(u, u, torch.randn(4, 2), Bv, Bv, None, u, None, True)


def test_install_dropin_registers_mamba_ssm_module():
    import sys

    import ceigm_unet_b200 as P
    P.install_dropin()
    import selective_scan_cuda                            # noqa: F401  (resolved from sys.modules)
    assert sys.modules["selective_scan_cuda"].__name__ == "ceigm_unet_b200.dropin.selective_scan_cuda"


def _split(name):
    m = re.search(r"ss2d\d+(\w+?)I((?:L[a-z]+\d+E)+)EE", name)
    return (m.group(1), re.findall(r"L[a-z]+\d+E", m.group(2))) if m else (None, None)


def test_gate_instantiations_exist():
    """scan_fwdr_kernel<NS, R, SOFTPLUS, SEG, GATE, STATE>: the gated ones are whole-row, R = 1 and 2, with and without softplus."""
    funcs = _sass_functions()
    gated = sorted(tuple(a) for n in funcs for k, a in [_split(n)] if k == "scan_fwdr_kernel" and a[4] == "Lb1E")
    assert gated == sorted((ns, r, sp, "Lb0E", "Lb1E", "Lb0E") for ns, r in (("Li16E", "Li1E"), ("Li8E", "Li2E"))
                           for sp in ("Lb0E", "Lb1E"))
    # every gated scan_fwdr kernel stores out_z next to out: two 128-bit global stores per group
    for n in funcs:
        k, a = _split(n)
        if k == "scan_fwdr_kernel" and a[4] == "Lb1E":
            assert len(re.findall(r"\bSTG\.E\.128\b", funcs[n])) >= 2, n
    for k in ("scan_gate_fwd_kernel", "scan_gate_bwd_kernel"):
        assert sum(k in n for n in funcs) == 10, k         # 5 (io, out) dtype pairs x (8-wide, scalar)


def test_deterministic_dispatch_with_gate_issues_no_global_atomics():
    """A gated call adds the two gate kernels and the gated scan_fwdr to what the deterministic backward can launch."""
    funcs = _sass_functions()
    launchable = [n for n in funcs if _det_launchable(n) or "scan_gate_" in n]
    assert sum("scan_gate_" in n for n in launchable) == 20
    assert sum(_split(n)[0] == "scan_fwdr_kernel" and _split(n)[1][4] == "Lb1E" for n in launchable) == 4
    offenders = {n: sorted(set(m.group(0) for m in _GLOBAL_ATOMIC.finditer(funcs[n]))) for n in launchable}
    offenders = {n: v for n, v in offenders.items() if v}
    assert not offenders, offenders
