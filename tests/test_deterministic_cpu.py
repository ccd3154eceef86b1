"""CPU tests of the deterministic scan backward (ss2d_scan_desc.deterministic): descriptor layout, workspace size, argument
validation, and — from the SASS of the built library — that no kernel the deterministic dispatch can launch issues a global
atomic or reduction (the only way a sum's order could depend on timing)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from ceigm_unet_b200 import _lib

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def _desc(batch=2, dim=12, L=64, N=16, G=4, det=0):
    d = _lib.ScanDesc()
    d.batch, d.dim, d.seqlen, d.dstate, d.n_groups = batch, dim, L, N, G
    d.deterministic = det
    return d


def _ws(d, have_ckpt=1):
    return int(_lib.lib().ss2d_scan_bwd_workspace_bytes(ctypes.byref(d), have_ckpt))


def test_field_fills_the_tail_padding():
    assert _lib.ScanDesc.deterministic.offset == 80 + 96 + 12
    assert ctypes.sizeof(_lib.ScanDesc) == 80 + 12 * 8 + 16


def test_version_is_0_2():
    assert " 0.2.0 " in _lib.version()


@pytest.mark.parametrize("shape", [
    (2, 12, 64, 16, 4),          # the descriptor test_abi.py pins
    (24, 768, 3136, 16, 4),      # vm_d192: scan_bwd2, one slab per warp
    (2, 384, 784, 4, 4),         # generic scan_bwd
    (1, 64, 16384, 1, 4),        # d_state = 1, long rows
    (64, 256, 49, 1, 4),         # d_state = 1, short rows
    (2, 64, 100, 40, 2),         # two state passes
])
def test_workspace_grows_only_in_deterministic_mode(shape):
    b, dim, L, N, G = shape
    default = _ws(_desc(b, dim, L, N, G))
    nmax = min(N, 32)
    assert default == 4 * ((b * dim * (nmax + 2) + 3) & ~3)        # unchanged formula of the default mode
    det = _ws(_desc(b, dim, L, N, G, det=1))
    assert det >= default
    assert _ws(_desc(b, dim, L, N, G, det=1), have_ckpt=0) >= _ws(_desc(b, dim, L, N, G), have_ckpt=0)


def test_default_workspace_is_unchanged():
    assert _ws(_desc()) == 4 * (2 * 12 * 18)


def test_vm_d192_holds_one_slab_per_extra_warp():
    # 192 rows per group, 8 rows per warp of the fast backward: 24 slabs, slab 0 is dB / dC itself
    extra = _ws(_desc(24, 768, 3136, 16, 4, det=1)) - _ws(_desc(24, 768, 3136, 16, 4))
    assert extra == 4 * 2 * 23 * (24 * 4 * 16 * 3136)


def test_out_of_range_value_is_rejected():
    L = _lib.lib()
    d = _desc(det=2)
    assert _ws(d) == 0
    assert L.ss2d_scan_ckpt_floats(ctypes.byref(d)) == 0
    args = [None] * 17 + [ctypes.c_size_t(0), None]
    assert L.ss2d_scan_bwd(ctypes.byref(d), *args) == -2
    d.deterministic = -1
    assert L.ss2d_scan_bwd(ctypes.byref(d), *args) == -2


# every kernel template whose last parameter is the deterministic-mode flag; the value 1 is what DET mode launches
_DET_TEMPLATES = ("scan_bwd_kernel", "scan_bwd2_kernel", "scan_n1_bwd_kernel", "scan_n1_bwd_rows_kernel", "scan_par_bwd_kernel")
_GLOBAL_ATOMIC = re.compile(r"\b(REDG?|ATOMG?)[.\s]\S*")      # not ATOMS (shared memory) or REDUX (warp reduction)


def _sass_functions():
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not found")
    out = subprocess.run([CUOBJDUMP, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {}
    for chunk in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = chunk.split("\n", 1)
        funcs[name.strip()] = body
    return funcs


def _det_launchable(name):
    """Kernels the deterministic backward can launch: DET instantiations, the slab fold, the finalize pass, and the forward
    kernels that recompute the checkpoints when none are passed in."""
    m = re.search(r"ss2d\d+(\w+?)I((?:L[a-z]+\d+E)+)EE", name)
    if m and m.group(1) in _DET_TEMPLATES:
        return m.group(2).endswith("Lb1E")
    return any(k in name for k in ("scan_bwd_fold_kernel", "scan_bwd_finalize_kernel", "scan_fwd", "scan_n1_fwd", "scan_par_fwd"))


def test_det_instantiations_with_and_without_state_issue_no_global_atomics():
    funcs = _sass_functions()
    launchable = [n for n in funcs if _det_launchable(n)]
    det_instances = [n for n in launchable if any(t in n for t in _DET_TEMPLATES)]
    # 7 generic + 2 fast + 4 one-row + 2 rows-walking + 6 parallel-along-L instantiations, each with STATE = 0 and 1
    assert len(det_instances) == 42, det_instances
    assert any("scan_bwd_fold_kernel" in n for n in launchable)
    offenders = {n: sorted(set(m.group(0) for m in _GLOBAL_ATOMIC.finditer(funcs[n]))) for n in launchable}
    offenders = {n: v for n, v in offenders.items() if v}
    assert not offenders, offenders


def test_default_kernels_still_reduce_in_l2():
    """The check above would pass vacuously if the pattern never matched: the default scan_bwd2 kernel does use RED."""
    funcs = _sass_functions()
    default_bwd2 = [n for n in funcs if "scan_bwd2_kernel" in n and not _det_launchable(n)]
    assert default_bwd2 and all(_GLOBAL_ATOMIC.search(funcs[n]) for n in default_bwd2)
