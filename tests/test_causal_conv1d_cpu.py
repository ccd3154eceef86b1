"""CPU tests of the causal depthwise conv1d (ss2d_conv1d_fwd / _bwd / _update, `causal_conv1d_fn` / `causal_conv1d_update`): the
entry points and descriptor, every error code of the C ABI (returned before any launch, so fake device addresses suffice), the
Python checks that raise before any launch, the registration of the two drop-in modules, and — from the SASS of the built
library — that the listed kernel instantiations exist, use no global atomics and no local memory, and that the vector ones move
their rows in 128-bit accesses."""
import ctypes
import re
import sys

import pytest
import torch

from ceigm_unet_b200 import _lib
from test_deterministic_cpu import _GLOBAL_ATOMIC, _sass_functions

OK, ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_LAYOUT, ERR_WORKSPACE, ERR_ALIGNMENT = 0, -1, -2, -3, -5, -6, -9
NAMES = ("ss2d_conv1d_fwd", "ss2d_conv1d_bwd", "ss2d_conv1d_bwd_workspace_bytes", "ss2d_conv1d_update")

# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000
ODD = GOOD + 1        # misaligned for every element size
MIS4 = GOOD + 2       # 2-byte aligned only


def test_symbols_and_descriptor():
    for n in NAMES:
        assert hasattr(_lib.lib(), n) and n in _lib.EXPORTS, n
    # 6 int32 then 4 int64: the C struct's offsets
    assert _lib.Conv1dDesc.x_batch_stride.offset == 24
    assert _lib.Conv1dDesc.out_dim_stride.offset == 24 + 3 * 8
    assert ctypes.sizeof(_lib.Conv1dDesc) == 56


def _desc(batch=2, dim=12, L=64, W=4, dtype=_lib.SS2D_F32, silu=1, update=False):
    d = _lib.Conv1dDesc()
    L = 1 if update else L
    d.batch, d.dim, d.seqlen, d.width, d.io_dtype, d.silu = batch, dim, L, W, dtype, silu
    d.x_batch_stride, d.x_dim_stride = dim * L, L
    d.out_batch_stride, d.out_dim_stride = dim * L, L
    return d


def _p(addr):
    return ctypes.c_void_p(addr) if addr else None


def _fwd(d, x=GOOD, w=GOOD, b=0, out=GOOD, desc=True):
    return _lib.lib().ss2d_conv1d_fwd(ctypes.byref(d) if desc else None, _p(x), _p(w), _p(b), _p(out), None)


def _bwd(d, x=GOOD, w=GOOD, b=0, dout=GOOD, dx=GOOD, dw=GOOD, db=0, ws=GOOD, ws_bytes=1 << 20, desc=True):
    return _lib.lib().ss2d_conv1d_bwd(ctypes.byref(d) if desc else None, _p(x), _p(w), _p(b), _p(dout), _p(dx), _p(dw), _p(db),
                                      _p(ws), ws_bytes, None)


def _upd(d, x=GOOD, state=GOOD, w=GOOD, b=0, out=GOOD, desc=True):
    return _lib.lib().ss2d_conv1d_update(ctypes.byref(d) if desc else None, _p(x), _p(state), _p(w), _p(b), _p(out), None)


CALLS = {"fwd": (_fwd, ("x", "w", "out"), ("x", "out")),
         "bwd": (_bwd, ("x", "w", "dout", "dx", "dw"), ("x", "dout", "dx")),
         "update": (_upd, ("x", "state", "w", "out"), ("x", "state", "out"))}


@pytest.mark.parametrize("call", list(CALLS))
def test_required_pointers(call):
    fn, required, _ = CALLS[call]
    d = _desc(update=call == "update")
    assert fn(d, desc=False) == ERR_NULL
    for kw in required:
        assert fn(d, **{kw: 0}) == ERR_NULL, kw


@pytest.mark.parametrize("call", list(CALLS))
@pytest.mark.parametrize("field,value", [("batch", 0), ("dim", -1), ("seqlen", 0), ("width", 1), ("width", 5)])
def test_bad_shapes_and_widths(call, field, value):
    fn = CALLS[call][0]
    d = _desc(update=call == "update")
    setattr(d, field, value)
    assert fn(d) == ERR_SHAPE


def test_update_takes_one_position():
    d = _desc(update=True)
    d.seqlen = 2
    assert _upd(d) == ERR_SHAPE


@pytest.mark.parametrize("call", list(CALLS))
@pytest.mark.parametrize("field,value", [("io_dtype", 3), ("io_dtype", -1), ("silu", 2), ("silu", -1)])
def test_bad_dtype_or_silu_flag(call, field, value):
    fn = CALLS[call][0]
    d = _desc(update=call == "update")
    setattr(d, field, value)
    assert fn(d) == ERR_DTYPE


@pytest.mark.parametrize("call", list(CALLS))
@pytest.mark.parametrize("field,delta", [("x_batch_stride", None), ("x_dim_stride", None), ("out_dim_stride", -1),
                                         ("out_batch_stride", -1)])
def test_bad_strides(call, field, delta):
    """negative x strides, and output rows that would overlap"""
    fn = CALLS[call][0]
    d = _desc(update=call == "update")
    setattr(d, field, -1 if delta is None else getattr(d, field) + delta)
    assert fn(d) == ERR_LAYOUT


@pytest.mark.parametrize("call", list(CALLS))
@pytest.mark.parametrize("dtype", [_lib.SS2D_F32, _lib.SS2D_F16, _lib.SS2D_BF16])
def test_alignment(call, dtype):
    fn, _, io = CALLS[call]
    d = _desc(dtype=dtype, update=call == "update")
    for kw in io:
        assert fn(d, **{kw: ODD}) == ERR_ALIGNMENT, kw
    fp32 = {"fwd": ("w", "b"), "bwd": ("w", "b", "dw", "db", "ws"), "update": ("w", "b")}[call]
    for kw in fp32:
        assert fn(d, **{kw: MIS4}) == ERR_ALIGNMENT, kw


def test_workspace():
    lib = _lib.lib()
    d = _desc(batch=1, dim=1, L=400 * 256, W=4)        # 400 segments of one channel: 100 slabs
    need = lib.ss2d_conv1d_bwd_workspace_bytes(ctypes.byref(d))
    assert need == 100 * (4 + 1) * 4
    assert _bwd(d, ws=0) == ERR_WORKSPACE
    assert _bwd(d, ws_bytes=need - 1) == ERR_WORKSPACE
    one = _desc(batch=16, dim=1536, L=2048)             # one slab per channel: no workspace
    assert lib.ss2d_conv1d_bwd_workspace_bytes(ctypes.byref(one)) == 0
    bad = _desc()
    bad.width = 7
    assert lib.ss2d_conv1d_bwd_workspace_bytes(ctypes.byref(bad)) == 0
    assert lib.ss2d_conv1d_bwd_workspace_bytes(None) == 0


def test_descriptor_errors_come_before_pointer_errors():
    d = _desc(W=5)
    assert _fwd(d, x=0) == ERR_SHAPE
    d = _desc(dtype=7)
    assert _bwd(d, x=ODD) == ERR_DTYPE


def test_no_launch_on_error():
    before = _lib.launch_count()
    _fwd(_desc(W=1))
    _bwd(_desc(batch=1, dim=1, L=400 * 256), ws=0)
    _upd(_desc(update=True), state=0)
    assert _lib.launch_count() == before


# ---- Python checks: RuntimeError before any launch ------------------------------------------------------------------
def _args(batch=2, dim=8, L=16, W=4, dtype=torch.float32, wdtype=torch.float32):
    return torch.randn(batch, dim, L, dtype=dtype), torch.randn(dim, W, dtype=wdtype), torch.randn(dim, dtype=wdtype)


def test_cpu_tensors_are_rejected():
    import ceigm_unet_b200 as P
    x, w, b = _args()
    with pytest.raises(RuntimeError, match="is_cuda"):          # no CPU fallback
        P.causal_conv1d_fn(x, w, b, activation="silu")
    with pytest.raises(RuntimeError, match="is_cuda"):
        P.causal_conv1d_fn(x, w.bfloat16(), None)
    with torch.no_grad(), pytest.raises(RuntimeError, match="is_cuda"):
        P.causal_conv1d_update(x[..., 0], torch.zeros(2, 8, 4), w, b, "silu")


@pytest.mark.parametrize("case,match", [
    ("seq_idx", "seq_idx is not supported"),
    ("activation", "activation must be None, silu, or swish"),
    ("width5", "2 <= width <= 4"),
    ("width1", "2 <= width <= 4"),
    ("weight3d", "2 <= width <= 4"),
    ("dim", "x must be .batch, dim, seqlen."),
    ("rank", "x must be .batch, dim, seqlen."),
    ("bias_shape", "bias must be .dim,. of weight's dtype"),
    ("bias_dtype", "bias must be .dim,. of weight's dtype"),
    ("x_dtype", "float32, float16 or bfloat16"),
    ("w_dtype", "weight must be float32, float16 or bfloat16"),
    ("channel_last", "channel-last x"),
])
def test_causal_conv1d_fn_checks(case, match):
    import ceigm_unet_b200 as P
    x, w, b = _args()
    kw = {}
    if case == "seq_idx":
        kw["seq_idx"] = torch.zeros(2, 16, dtype=torch.int32)
    elif case == "activation":
        kw["activation"] = "relu"
    elif case == "width5":
        w = torch.randn(8, 5)
    elif case == "width1":
        w = torch.randn(8, 1)
    elif case == "weight3d":
        w = w[:, None]                                   # nn.Conv1d's (dim, 1, width) is not causal-conv1d's layout
    elif case == "dim":
        w, b = torch.randn(9, 4), torch.randn(9)
    elif case == "rank":
        x = x[0]
    elif case == "bias_shape":
        b = torch.randn(9)
    elif case == "bias_dtype":
        b = b.half()
    elif case == "x_dtype":
        x = x.double()
    elif case == "w_dtype":
        w, b = w.double(), b.double()
    elif case == "channel_last":
        x = torch.randn(2, 16, 8).transpose(1, 2)
        assert x.stride(1) == 1 and x.stride(2) != 1
    with pytest.raises(RuntimeError, match=match):
        P.causal_conv1d_fn(x, w, b, activation=kw.pop("activation", "silu"), **kw)


def test_backward_and_update_checks():
    import ceigm_unet_b200 as P
    from ceigm_unet_b200 import ops
    x, w, b = _args()
    with pytest.raises(RuntimeError, match="dout must have x's shape"):
        ops.conv1d_bwd(x, w, b, x[..., :-1], True)
    with pytest.raises(RuntimeError, match="dx must have x's shape and dtype"):
        ops.conv1d_bwd(x, w, b, x, True, dx=x.half())
    xs = x[..., 0]
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="x must be .batch, dim."):
            P.causal_conv1d_update(x, torch.zeros(2, 8, 4), w, b)
        with pytest.raises(RuntimeError, match="conv_state must be .batch, dim, width. of x's dtype"):
            P.causal_conv1d_update(xs, torch.zeros(2, 8, 3), w, b)
        with pytest.raises(RuntimeError, match="conv_state must be .batch, dim, width. of x's dtype"):
            P.causal_conv1d_update(xs, torch.zeros(2, 8, 4, dtype=torch.bfloat16), w, b)
        with pytest.raises(RuntimeError, match="conv_state must be contiguous"):
            P.causal_conv1d_update(xs, torch.zeros(2, 4, 8).transpose(1, 2), w, b)
        with pytest.raises(RuntimeError, match="activation must be None, silu, or swish"):
            P.causal_conv1d_update(xs, torch.zeros(2, 8, 4), w, b, "gelu")


@pytest.mark.parametrize("name", ["x", "conv_state", "weight", "bias"])
def test_update_inputs_that_require_grad_are_rejected(name):
    import ceigm_unet_b200 as P
    x, w, b = _args()
    a = dict(x=x[..., 0].clone(), conv_state=torch.zeros(2, 8, 4), weight=w, bias=b)
    a[name] = a[name].clone().requires_grad_(True)
    with pytest.raises(RuntimeError, match=f"{name} requires grad"):
        P.causal_conv1d_update(**a)
    with torch.no_grad(), pytest.raises(RuntimeError, match="is_cuda"):
        P.causal_conv1d_update(**a)


def test_dropin_modules_are_registered():
    import ceigm_unet_b200 as P
    from ceigm_unet_b200.dropin import causal_conv1d as pkg
    from ceigm_unet_b200.dropin import causal_conv1d_cuda as ext
    saved = {k: sys.modules.get(k) for k in ("causal_conv1d", "causal_conv1d_cuda")}
    try:
        P.install_dropin()
        import causal_conv1d
        import causal_conv1d_cuda
        from causal_conv1d import causal_conv1d_fn, causal_conv1d_update
        assert causal_conv1d is pkg and causal_conv1d_cuda is ext
        assert causal_conv1d_fn is P.causal_conv1d_fn and causal_conv1d_update is P.causal_conv1d_update
        for n in ("causal_conv1d_fwd", "causal_conv1d_bwd", "causal_conv1d_update"):
            assert callable(getattr(causal_conv1d_cuda, n)), n
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    x, w, b = _args()
    with pytest.raises(RuntimeError, match="seq_idx is not supported"):
        ext.causal_conv1d_fwd(x, w, b, torch.zeros(2, 16, dtype=torch.int32), True)
    with pytest.raises(RuntimeError, match="seq_idx is not supported"):
        ext.causal_conv1d_bwd(x, w, b, x, torch.zeros(2, 16, dtype=torch.int32), None, True)
    with pytest.raises(RuntimeError, match="is_cuda"):
        ext.causal_conv1d_fwd(x, w, b, None, True)


# ---- SASS of the built library -------------------------------------------------------------------------------------
_TYPES = ("f", "6__half", "13__nv_bfloat16")
_KERNEL = re.compile(r"conv1d_(fwd|bwd|update)_kernelI(\w+?)Li(\d)ELb([01])E")


def _conv_kernels():
    return {n: b for n, b in _sass_functions().items() if "conv1d_" in n and "_kernel" in n}


def test_every_conv1d_instantiation_exists():
    """fwd / bwd: 3 io dtypes x width 2 / 3 / 4 x vector / scalar (18 each); update: 3 io dtypes x (width, vector) in
    (2, no), (2, yes), (3, no), (4, no), (4, yes) (15); and the finalize pass."""
    kernels = _conv_kernels()
    keys = set()
    for n in kernels:
        if "conv1d_wgrad_finalize_kernel" in n:
            continue
        m = _KERNEL.search(n)
        assert m, n
        keys.add((m.group(1), m.group(2), int(m.group(3)), m.group(4) == "1"))
    want = {(k, t, w, v) for k in ("fwd", "bwd") for t in _TYPES for w in (2, 3, 4) for v in (False, True)}
    want |= {("update", t, w, v) for t in _TYPES for w, v in ((2, False), (2, True), (3, False), (4, False), (4, True))}
    assert keys == want
    assert sum("conv1d_wgrad_finalize_kernel" in n for n in kernels) == 1
    assert len(kernels) == 52


def test_conv1d_kernels_use_no_global_atomics_and_no_local_memory():
    kernels = _conv_kernels()
    assert kernels
    offenders = {n: sorted(set(m.group(0) for m in _GLOBAL_ATOMIC.finditer(b))) for n, b in kernels.items()}
    assert not {n: v for n, v in offenders.items() if v}, offenders
    local = {n: sorted(set(re.findall(r"\b(?:LDL|STL)\S*", b))) for n, b in kernels.items()}
    assert not {n: v for n, v in local.items() if v}, local


def test_vector_instantiations_use_wide_accesses():
    """fwd / bwd VEC: runs move with 128-bit loads and stores. update VEC: the state row is stored in one access of width x the
    element size (32, 64 or 128 bits); at width 4 it is also loaded in one (at width 2 only the value that survives the shift is
    read)."""
    size = {"f": 4, "6__half": 2, "13__nv_bfloat16": 2}
    for n, b in _conv_kernels().items():
        m = _KERNEL.search(n)
        if not m or m.group(4) != "1":
            continue
        kind, W = m.group(1), int(m.group(3))
        bits = 128 if kind != "update" else 8 * W * size[m.group(2)]
        width = "" if bits == 32 else rf"\.{bits}"
        assert re.search(rf"\bSTG\.E{width}\b(?!\.U16)", b), n
        if kind != "update" or W == 4:
            assert re.search(rf"\bLDG\.E{width}\b", b), n
