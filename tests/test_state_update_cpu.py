"""CPU tests of the recurrent step (ss2d_state_update, `selective_state_update`): the entry point and descriptor, every error code
of the C ABI (returned before any launch, so fake device addresses suffice), the Python checks that raise before any launch, and
— from the SASS of the built library — that the ssm_step_kernel instantiations exist and use no global atomics and no local
memory."""
import ctypes
import re

import pytest
import torch

from ceigm_unet_b200 import _lib
from test_deterministic_cpu import _GLOBAL_ATOMIC, _sass_functions

OK, ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_DSTATE, ERR_ALIGNMENT = 0, -1, -2, -3, -4, -9

# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000
MIS16 = GOOD + 4      # 4-byte aligned, not 16-byte aligned
ODD = GOOD + 1        # misaligned for every element size


def test_symbol_and_descriptor():
    assert hasattr(_lib.lib(), "ss2d_state_update") and "ss2d_state_update" in _lib.EXPORTS
    # 6 int32 then 5 int64: the C struct's offsets
    assert _lib.StepDesc.io_batch_stride.offset == 24
    assert _lib.StepDesc.C_group_stride.offset == 24 + 4 * 8
    assert ctypes.sizeof(_lib.StepDesc) == 64


def _desc(batch=2, dim=12, N=16, G=4, dtype=_lib.SS2D_F32, softplus=1):
    d = _lib.StepDesc()
    d.batch, d.dim, d.dstate, d.n_groups, d.io_dtype, d.dt_softplus = batch, dim, N, G, dtype, softplus
    d.io_batch_stride, d.B_batch_stride, d.B_group_stride = dim, G * N, N
    d.C_batch_stride, d.C_group_stride = G * N, N
    return d


def _p(addr):
    return ctypes.c_void_p(addr) if addr else None


def _call(d, state=GOOD, x=GOOD, dt=GOOD, A=GOOD, B=GOOD, C=GOOD, D=0, dt_bias=0, z=0, out=GOOD, desc=True):
    return _lib.lib().ss2d_state_update(ctypes.byref(d) if desc else None, _p(state), _p(x), _p(dt), _p(A), _p(B), _p(C), _p(D),
                                        _p(dt_bias), _p(z), _p(out), None)


REQUIRED = ("state", "x", "dt", "A", "B", "C", "out")


def test_required_pointers():
    d = _desc()
    assert _call(d, desc=False) == ERR_NULL
    for kw in REQUIRED:
        assert _call(d, **{kw: 0}) == ERR_NULL, kw


@pytest.mark.parametrize("field,value", [("batch", 0), ("dim", -1), ("dstate", 0), ("n_groups", 0), ("n_groups", 5)])
def test_bad_shapes(field, value):
    d = _desc()
    setattr(d, field, value)
    assert _call(d) == ERR_SHAPE


def test_dstate_limit():
    assert _call(_desc(N=256), x=0) == ERR_NULL        # 256 passes the descriptor checks (a NULL x keeps it from launching)
    assert _call(_desc(N=257)) == ERR_DSTATE


@pytest.mark.parametrize("field,value", [("io_dtype", 3), ("io_dtype", -1), ("dt_softplus", 2), ("dt_softplus", -1)])
def test_bad_dtype_or_softplus_flag(field, value):
    d = _desc()
    setattr(d, field, value)
    assert _call(d) == ERR_DTYPE


@pytest.mark.parametrize("dtype", [_lib.SS2D_F32, _lib.SS2D_F16, _lib.SS2D_BF16])
def test_alignment(dtype):
    d = _desc(dtype=dtype)
    assert _call(d, state=MIS16) == ERR_ALIGNMENT
    for kw in ("x", "dt", "B", "C", "z", "out", "A", "D", "dt_bias"):
        assert _call(d, **{kw: ODD}) == ERR_ALIGNMENT, kw


def test_descriptor_errors_come_before_pointer_errors():
    d = _desc(G=5)
    assert _call(d, x=0) == ERR_SHAPE
    d = _desc(N=300)
    assert _call(d, state=MIS16) == ERR_DSTATE


# ---- Python checks: RuntimeError before any launch ------------------------------------------------------------------
def _cpu_args(batch=2, dim=8, N=4, G=1, dtype=torch.float32):
    return dict(state=torch.zeros(batch, dim, N), x=torch.randn(batch, dim, dtype=dtype), dt=torch.randn(batch, dim, dtype=dtype),
                A=-torch.rand(dim, N), B=torch.randn(batch, G, N, dtype=dtype), C=torch.randn(batch, G, N, dtype=dtype))


def test_cpu_tensors_are_rejected():
    import ceigm_unet_b200 as P
    a = _cpu_args()
    with torch.no_grad(), pytest.raises(RuntimeError, match="is_cuda"):      # no CPU fallback
        P.selective_state_update(**a)
    with torch.no_grad(), pytest.raises(RuntimeError, match="is_cuda"):
        P.selective_state_update(**a, D=torch.ones(8), z=torch.randn(2, 8), dt_bias=torch.zeros(8), dt_softplus=True)


@pytest.mark.parametrize("name", ["state", "x", "dt", "A", "B", "C", "D", "z", "dt_bias"])
def test_inputs_that_require_grad_are_rejected(name):
    import ceigm_unet_b200 as P
    a = dict(_cpu_args(), D=torch.ones(8), z=torch.randn(2, 8), dt_bias=torch.zeros(8))
    a[name] = a[name].clone().requires_grad_(True)
    with pytest.raises(RuntimeError, match=f"{name} requires grad"):
        P.selective_state_update(**a)
    # under no_grad the grad check passes and the device check is what stops the call
    with torch.no_grad(), pytest.raises(RuntimeError, match="is_cuda"):
        P.selective_state_update(**a)


def test_unsupported_dtype_is_rejected():
    from ceigm_unet_b200 import ops
    a = _cpu_args()
    a["x"] = a["x"].double()
    with pytest.raises(RuntimeError, match="float32, float16 or bfloat16"):
        ops.state_update(**a)


# ---- SASS of the built library -------------------------------------------------------------------------------------
def _step_kernels():
    funcs = _sass_functions()
    return {n: b for n, b in funcs.items() if "ssm_step_kernel" in n}


def test_every_step_instantiation_exists():
    """3 io dtypes x 7 lane mappings (S states per lane, P lanes per row) x vector / scalar state accesses."""
    kernels = _step_kernels()
    keys = set()
    for n in kernels:
        m = re.search(r"ssm_step_kernelI(\w+?)Li(\d+)ELi(\d+)ELb([01])E", n)
        assert m, n
        keys.add((m.group(1), int(m.group(2)), int(m.group(3)), m.group(4) == "1"))
    regimes = {(4, 1), (4, 2), (4, 4), (4, 8), (2, 32), (4, 32), (8, 32)}
    want = {(t, s, p, v) for t in ("f", "6__half", "13__nv_bfloat16") for s, p in regimes for v in (False, True)}
    assert keys == want and len(kernels) == 42


def test_step_kernels_use_no_global_atomics_and_no_local_memory():
    kernels = _step_kernels()
    assert kernels
    offenders = {n: sorted(set(m.group(0) for m in _GLOBAL_ATOMIC.finditer(b))) for n, b in kernels.items()}
    assert not {n: v for n, v in offenders.items() if v}, offenders
    local = {n: sorted(set(re.findall(r"\b(?:LDL|STL)\S*", b))) for n, b in kernels.items()}
    assert not {n: v for n, v in local.items() if v}, local


def test_vector_instantiations_move_the_state_in_wide_accesses():
    """VEC instantiations with 4 or 8 states per lane read and write the state with 128-bit accesses, with 2 with 64-bit ones."""
    for n, b in _step_kernels().items():
        m = re.search(r"Li(\d+)ELi\d+ELb1E", n)
        if m:
            width = "128" if int(m.group(1)) >= 4 else "64"
            assert re.search(rf"\bLDG?\.E\.{width}\b", b) and re.search(rf"\bSTG?\.E\.{width}\b", b), n
