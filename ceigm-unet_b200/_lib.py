"""ctypes binding of libss2d_b200.so (the C ABI declared in include/ss2d_b200.h).

The product path has NO fallback: if the shared library is missing or a call fails, a RuntimeError is
raised. Build it with `python __graft_entry__.py build` or `ceigm-unet_b200/csrc/build.sh`.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libss2d_b200.so")

SS2D_F32, SS2D_F16, SS2D_BF16 = 0, 1, 2
LAYOUT_SCAN, LAYOUT_NATURAL = 0, 1
MAX_GROUP_DIRS = 8
CHUNK = 32
MAX_DSTATE = 256

# every symbol include/ss2d_b200.h declares (tests/test_abi.py checks the library exports all of them)
EXPORTS = [
    "ss2d_scan_fwd", "ss2d_scan_ckpt_floats", "ss2d_scan_bwd", "ss2d_scan_bwd_workspace_bytes",
    "ss2d_scan_fwd_state", "ss2d_scan_bwd_state",
    "ss2d_scan_fwd_gated", "ss2d_scan_bwd_gated", "ss2d_scan_bwd_gated_workspace_bytes", "ss2d_state_update",
    "ss2d_conv1d_fwd", "ss2d_conv1d_bwd", "ss2d_conv1d_bwd_workspace_bytes", "ss2d_conv1d_update",
    "ss2d_ssd_fwd", "ss2d_ssd_fwd_workspace_bytes", "ss2d_ssd_bwd", "ss2d_ssd_bwd_workspace_bytes",
    "ss2d_cross_scan", "ss2d_cross_merge", "ss2d_out_gate_fwd", "ss2d_out_gate_bwd",
    "ss2d_out_gate_bwd_partials", "ss2d_group_gate_fwd", "ss2d_group_gate_bwd", "ss2d_out_gate_max_width", "ss2d_wgrad_ts", "ss2d_wgrad_ts_workspace_bytes",
    "ss2d_layernorm_fwd", "ss2d_layernorm_bwd", "ss2d_layernorm_bwd_partials",
    "ss2d_dwconv3_wgrad", "ss2d_dwconv3_wgrad_workspace_bytes", "ss2d_dwconv3_act", "ss2d_dwconv3_act_planes", "ss2d_gate_proj_fwd", "ss2d_gate_proj_supported", "ss2d_linear_tc", "ss2d_linear_tc_supported", "ss2d_strerror", "ss2d_last_cuda_error", "ss2d_version", "ss2d_launch_count", "ss2d_test_force_path", "ss2d_dwnhwc_stencil", "ss2d_dwnhwc_wgrad", "ss2d_dwnhwc_wgrad_workspace_bytes",
]


class ScanDesc(ctypes.Structure):
    """Mirror of `ss2d_scan_desc` (include/ss2d_b200.h)."""
    _fields_ = [
        ("batch", ctypes.c_int32), ("dim", ctypes.c_int32), ("seqlen", ctypes.c_int32),
        ("dstate", ctypes.c_int32), ("n_groups", ctypes.c_int32), ("io_dtype", ctypes.c_int32),
        ("out_dtype", ctypes.c_int32), ("delta_softplus", ctypes.c_int32), ("layout", ctypes.c_int32),
        ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("dirs", ctypes.c_int32 * MAX_GROUP_DIRS),
        ("u_batch_stride", ctypes.c_int64), ("u_dim_stride", ctypes.c_int64),
        ("delta_batch_stride", ctypes.c_int64), ("delta_dim_stride", ctypes.c_int64),
        ("out_batch_stride", ctypes.c_int64), ("out_dim_stride", ctypes.c_int64),
        ("B_batch_stride", ctypes.c_int64), ("B_group_stride", ctypes.c_int64), ("B_state_stride", ctypes.c_int64),
        ("C_batch_stride", ctypes.c_int64), ("C_group_stride", ctypes.c_int64), ("C_state_stride", ctypes.c_int64),
        ("u_dim_modulo", ctypes.c_int32), ("last_state_interleaved", ctypes.c_int32),
        ("grads_prezeroed", ctypes.c_int32), ("deterministic", ctypes.c_int32),
    ]


class StepDesc(ctypes.Structure):
    """Mirror of `ss2d_step_desc` (include/ss2d_b200.h)."""
    _fields_ = [
        ("batch", ctypes.c_int32), ("dim", ctypes.c_int32), ("dstate", ctypes.c_int32), ("n_groups", ctypes.c_int32),
        ("io_dtype", ctypes.c_int32), ("dt_softplus", ctypes.c_int32), ("io_batch_stride", ctypes.c_int64),
        ("B_batch_stride", ctypes.c_int64), ("B_group_stride", ctypes.c_int64),
        ("C_batch_stride", ctypes.c_int64), ("C_group_stride", ctypes.c_int64),
    ]


class Conv1dDesc(ctypes.Structure):
    """Mirror of `ss2d_conv1d_desc` (include/ss2d_b200.h)."""
    _fields_ = [
        ("batch", ctypes.c_int32), ("dim", ctypes.c_int32), ("seqlen", ctypes.c_int32), ("width", ctypes.c_int32),
        ("io_dtype", ctypes.c_int32), ("silu", ctypes.c_int32),
        ("x_batch_stride", ctypes.c_int64), ("x_dim_stride", ctypes.c_int64),
        ("out_batch_stride", ctypes.c_int64), ("out_dim_stride", ctypes.c_int64),
    ]


class SsdDesc(ctypes.Structure):
    """Mirror of `ss2d_ssd_desc` (include/ss2d_b200.h)."""
    _fields_ = [
        ("batch", ctypes.c_int32), ("seqlen", ctypes.c_int32), ("heads", ctypes.c_int32), ("headdim", ctypes.c_int32),
        ("n_groups", ctypes.c_int32), ("dstate", ctypes.c_int32), ("chunk_size", ctypes.c_int32), ("io_dtype", ctypes.c_int32),
        ("dt_softplus", ctypes.c_int32), ("d_mode", ctypes.c_int32), ("dt_min", ctypes.c_float), ("dt_max", ctypes.c_float),
    ] + [(f"{t}_{s}_stride", ctypes.c_int64) for t in ("x", "z", "out", "dt") for s in ("batch", "seq", "head")] + [
        ("bc_batch_stride", ctypes.c_int64), ("bc_seq_stride", ctypes.c_int64), ("bc_group_stride", ctypes.c_int64),
    ]


class LinearPart(ctypes.Structure):
    """Mirror of `ss2d_linear_part` (include/ss2d_b200.h)."""
    _fields_ = [("out", ctypes.c_void_p), ("ld", ctypes.c_int64), ("n_cols", ctypes.c_int32), ("planes_L", ctypes.c_int32),
                ("act", ctypes.c_int32)]


_lib = None


def build(verbose: bool = False) -> str:
    """Compile libss2d_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    script = os.path.join(_HERE, "csrc", "build.sh")
    out = subprocess.run(["bash", script], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libss2d_b200.so failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout.strip())
    global _lib
    _lib = None
    return LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run ceigm-unet_b200/csrc/build.sh "
            "(there is no CPU or PyTorch fallback for the SS2D scan).")
    L = ctypes.CDLL(LIB_PATH)
    vp, fp, i32, i64, sz = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
    dp = ctypes.POINTER(ScanDesc)
    L.ss2d_scan_fwd.argtypes = [dp, vp, vp, fp, vp, vp, fp, fp, vp, fp, fp, vp]
    L.ss2d_scan_fwd.restype = ctypes.c_int
    L.ss2d_scan_ckpt_floats.argtypes = [dp]
    L.ss2d_scan_ckpt_floats.restype = sz
    L.ss2d_scan_bwd.argtypes = [dp, vp, vp, fp, vp, vp, fp, fp, vp, fp, vp, vp, fp, fp, fp, fp, fp, vp, sz, vp]
    L.ss2d_scan_bwd.restype = ctypes.c_int
    L.ss2d_scan_fwd_state.argtypes = [dp, vp, vp, fp, vp, vp, fp, fp, fp, vp, fp, fp, vp]
    L.ss2d_scan_fwd_state.restype = ctypes.c_int
    L.ss2d_scan_bwd_state.argtypes = [dp, vp, vp, fp, vp, vp, fp, fp, fp, vp, fp, fp, vp, vp, fp, fp, fp, fp, fp, fp, vp, sz, vp]
    L.ss2d_scan_bwd_state.restype = ctypes.c_int
    L.ss2d_scan_fwd_gated.argtypes = [dp, vp, vp, fp, vp, vp, fp, fp, fp, vp, vp, vp, fp, fp, vp]
    L.ss2d_scan_fwd_gated.restype = ctypes.c_int
    L.ss2d_scan_bwd_gated.argtypes = [dp, vp, vp, fp, vp, vp, fp, fp, fp, vp, vp, vp, fp, fp, vp, vp, fp, fp, fp, fp, fp, vp, fp,
                                      vp, sz, vp]
    L.ss2d_scan_bwd_gated.restype = ctypes.c_int
    L.ss2d_scan_bwd_gated_workspace_bytes.argtypes = [dp, ctypes.c_int]
    L.ss2d_scan_bwd_gated_workspace_bytes.restype = sz
    L.ss2d_scan_bwd_workspace_bytes.argtypes = [dp, ctypes.c_int]
    L.ss2d_scan_bwd_workspace_bytes.restype = sz
    L.ss2d_state_update.argtypes = [ctypes.POINTER(StepDesc), fp, vp, vp, fp, vp, vp, fp, fp, vp, vp, vp]
    L.ss2d_state_update.restype = ctypes.c_int
    cd = ctypes.POINTER(Conv1dDesc)
    L.ss2d_conv1d_fwd.argtypes = [cd, vp, fp, fp, vp, vp]
    L.ss2d_conv1d_fwd.restype = ctypes.c_int
    L.ss2d_conv1d_bwd_workspace_bytes.argtypes = [cd]
    L.ss2d_conv1d_bwd_workspace_bytes.restype = sz
    L.ss2d_conv1d_bwd.argtypes = [cd, vp, fp, fp, vp, vp, fp, fp, vp, sz, vp]
    L.ss2d_conv1d_bwd.restype = ctypes.c_int
    L.ss2d_conv1d_update.argtypes = [cd, vp, vp, fp, fp, vp, vp]
    L.ss2d_conv1d_update.restype = ctypes.c_int
    sd = ctypes.POINTER(SsdDesc)
    L.ss2d_ssd_fwd_workspace_bytes.argtypes = [sd]
    L.ss2d_ssd_fwd_workspace_bytes.restype = sz
    L.ss2d_ssd_fwd.argtypes = [sd, vp, vp, fp, vp, vp, fp, fp, vp, fp, vp, fp, vp, sz, vp]
    L.ss2d_ssd_fwd.restype = ctypes.c_int
    L.ss2d_ssd_bwd_workspace_bytes.argtypes = [sd]
    L.ss2d_ssd_bwd_workspace_bytes.restype = sz
    L.ss2d_ssd_bwd.argtypes = [sd, vp, vp, fp, vp, vp, fp, fp, vp, fp, vp, fp, vp, vp, fp, vp, vp, fp, fp, vp, fp, vp, sz, vp]
    L.ss2d_ssd_bwd.restype = ctypes.c_int
    ip = ctypes.POINTER(ctypes.c_int32)
    L.ss2d_cross_scan.argtypes = [vp, vp, i32, i32, i32, i32, i32, ip, i32, vp]
    L.ss2d_cross_scan.restype = ctypes.c_int
    L.ss2d_cross_merge.argtypes = [vp, vp, i32, i32, i32, i32, i32, ip, i32, vp]
    L.ss2d_cross_merge.restype = ctypes.c_int
    L.ss2d_out_gate_fwd.argtypes = [fp, i32, fp, fp, vp, i64, i32, vp, fp, i32, i32, i32, ctypes.c_float, i32, i32, i32, i32,
                                    ctypes.c_uint32, vp]
    L.ss2d_out_gate_fwd.restype = ctypes.c_int
    L.ss2d_out_gate_bwd.argtypes = [fp, i32, fp, fp, vp, i64, i32, vp, fp, fp, vp, i64, fp, fp, i32, i32, i32, i32,
                                    i32, i32, i32, i32, ctypes.c_uint32, i32, vp]
    L.ss2d_out_gate_bwd.restype = ctypes.c_int
    L.ss2d_out_gate_max_width.argtypes = [i32]
    L.ss2d_out_gate_max_width.restype = i32
    u32 = ctypes.c_uint32
    L.ss2d_group_gate_fwd.argtypes = [fp, i32, ip, u32, fp, fp, vp, i64, i64, i64, vp, i64, fp, i32, i32, i32, ctypes.c_float,
                                      i32, i32, i32, i32, vp]
    L.ss2d_group_gate_fwd.restype = ctypes.c_int
    L.ss2d_group_gate_bwd.argtypes = [fp, i32, ip, u32, fp, fp, vp, i64, i64, i64, vp, i64, fp, fp, vp, i64, fp, fp, i32, i32,
                                      i32, i32, i32, i32, i32, i32, vp]
    L.ss2d_group_gate_bwd.restype = ctypes.c_int
    L.ss2d_out_gate_bwd_partials.argtypes = [i32, i32]
    L.ss2d_out_gate_bwd_partials.restype = i32
    L.ss2d_wgrad_ts.argtypes = [vp, vp, fp, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, i32, i32, vp, sz, vp]
    L.ss2d_wgrad_ts.restype = ctypes.c_int
    L.ss2d_wgrad_ts_workspace_bytes.argtypes = [i32, i32, i32, i32]
    L.ss2d_wgrad_ts_workspace_bytes.restype = sz
    L.ss2d_dwconv3_wgrad.argtypes = [fp, fp, fp, fp, i32, i32, i32, i32, vp, sz, vp]
    L.ss2d_dwconv3_wgrad.restype = ctypes.c_int
    L.ss2d_dwconv3_wgrad_workspace_bytes.argtypes = [i32, i32, i32, i32]
    L.ss2d_dwconv3_wgrad_workspace_bytes.restype = sz
    L.ss2d_layernorm_fwd.argtypes = [vp, fp, fp, vp, fp, i64, i32, ctypes.c_float, i32, vp]
    L.ss2d_layernorm_fwd.restype = ctypes.c_int
    L.ss2d_layernorm_bwd.argtypes = [vp, fp, vp, fp, vp, fp, fp, i32, i64, i32, i32, vp]
    L.ss2d_layernorm_bwd.restype = ctypes.c_int
    L.ss2d_layernorm_bwd_partials.argtypes = [i64]
    L.ss2d_layernorm_bwd_partials.restype = i32
    L.ss2d_dwconv3_act.argtypes = [i32, vp, fp, fp, vp, vp, i32, i32, i32, i32, i32, vp]
    L.ss2d_dwconv3_act.restype = ctypes.c_int
    L.ss2d_dwconv3_act_planes.argtypes = [i32, vp, i64, fp, fp, vp, i64, vp, i64, vp, i64, vp, i64, i32, i32, i32, i32, i32, vp]
    L.ss2d_dwconv3_act_planes.restype = ctypes.c_int
    L.ss2d_gate_proj_fwd.argtypes = [fp, i32, ctypes.c_uint32, fp, fp, ctypes.c_float, vp, i64, i32, vp, i64, fp, vp, i64, vp, i64, fp,
                                     i32, i32, i32, i32, i32, i32, i32, vp]
    L.ss2d_gate_proj_fwd.restype = ctypes.c_int
    L.ss2d_gate_proj_supported.argtypes = [i32, i32, i32, i32]
    L.ss2d_gate_proj_supported.restype = i32
    L.ss2d_linear_tc.argtypes = [vp, i64, vp, i64, fp, i32, i32, i32, i32, i32, ctypes.POINTER(LinearPart), vp]
    L.ss2d_linear_tc.restype = ctypes.c_int
    L.ss2d_linear_tc_supported.argtypes = [i32, i32, i32]
    L.ss2d_linear_tc_supported.restype = i32
    pp = ctypes.POINTER(ctypes.c_void_p)
    L.ss2d_dwnhwc_stencil.argtypes = [vp, vp, vp, i32, ip, ip, pp, pp, i32, i32, i32, i32, i32, i32, i32, vp]
    L.ss2d_dwnhwc_stencil.restype = ctypes.c_int
    L.ss2d_dwnhwc_wgrad.argtypes = [vp, vp, i32, i32, i32, fp, fp, i32, i32, i32, i32, i32, vp, sz, vp]
    L.ss2d_dwnhwc_wgrad.restype = ctypes.c_int
    L.ss2d_dwnhwc_wgrad_workspace_bytes.argtypes = [i32, i32, i32, i32, i32]
    L.ss2d_dwnhwc_wgrad_workspace_bytes.restype = sz
    L.ss2d_strerror.argtypes = [ctypes.c_int]
    L.ss2d_strerror.restype = ctypes.c_char_p
    L.ss2d_last_cuda_error.restype = ctypes.c_char_p
    L.ss2d_version.restype = ctypes.c_char_p
    L.ss2d_launch_count.argtypes = [ctypes.c_int]
    L.ss2d_launch_count.restype = ctypes.c_int64
    L.ss2d_test_force_path.argtypes = [ctypes.c_int32]
    L.ss2d_test_force_path.restype = ctypes.c_int32
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        L = lib()
        msg = L.ss2d_strerror(rc).decode()
        if rc == -7:
            msg += ": " + L.ss2d_last_cuda_error().decode()
        raise RuntimeError(f"{what} failed ({rc}): {msg}")


def test_force_path(policy: int) -> None:
    """TEST HOOK (include/ss2d_b200.h: ss2d_test_force_path): 0 automatic, 1 / 2 lane-owns-row forward (32 / 16-row warps), 3 the 8-row-warp forward (and the tiled FFN stencil), 4 the segmented forward; policy + 8: the same, with the output gate never fused into scan_fwdr."""
    rc = lib().ss2d_test_force_path(int(policy))
    if rc != 0:
        raise RuntimeError("ss2d_test_force_path(%d) -> %d" % (policy, rc))


def launch_count(reset: bool = False) -> int:
    return int(lib().ss2d_launch_count(1 if reset else 0))


def version() -> str:
    return lib().ss2d_version().decode()
