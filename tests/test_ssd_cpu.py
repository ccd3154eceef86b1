"""CPU tests of Mamba-2's chunked selective scan (ss2d_ssd_fwd, `mamba_chunk_scan_combined`): the float64 chunked oracle
against the recurrence that defines the contract (values and autograd gradients), the descriptor and every error code of the
C ABI (returned before any launch, so fake device addresses suffice), the Python checks that raise before any launch, and —
from the SASS of the built library — that the listed kernel instantiations exist, use no global atomics and no local memory,
and that the product kernels run on the tensor cores (HMMA)."""
import ctypes
import math

import pytest
import torch

from ceigm_unet_b200 import _lib
from oracle.ssd_ref import ssd_chunked, ssd_recurrence
from test_deterministic_cpu import _GLOBAL_ATOMIC, _sass_functions

OK, ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_DSTATE, ERR_LAYOUT, ERR_WORKSPACE, ERR_UNSUPPORTED, ERR_ALIGNMENT = (
    0, -1, -2, -3, -4, -5, -6, -8, -9)

GOOD = 0x10000        # fake, never dereferenced device addresses
ODD = GOOD + 1
MIS4 = GOOD + 2


def _oracle_inputs(b, L, h, P, g, N, seed, grad=False):
    gen = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=gen, dtype=torch.float64)   # noqa: E731
    t = dict(x=r(b, L, h, P), dt=r(b, L, h) * 0.5 - 2.0, A=-(torch.rand(h, generator=gen, dtype=torch.float64) + 0.5),
             B=r(b, L, g, N), C=r(b, L, g, N), D=r(h, P), z=r(b, L, h, P), dt_bias=r(h) * 0.3, initial_states=r(b, h, P, N))
    if grad:
        for v in t.values():
            v.requires_grad_(True)
    return t


def _call(fn, t, *extra, **kw):
    return fn(t["x"], t["dt"], t["A"], t["B"], t["C"], *extra, D=t["D"], z=t["z"], dt_bias=t["dt_bias"],
              initial_states=t["initial_states"], dt_softplus=True, **kw)


@pytest.mark.parametrize("L,Q", [(1, 4), (7, 4), (16, 8), (37, 16)])
def test_chunked_oracle_matches_recurrence(L, Q):
    t = _oracle_inputs(2, L, 4, 3, 2, 5, seed=L)
    y0, h0 = _call(ssd_recurrence, t)
    y1, h1 = _call(ssd_chunked, t, Q)
    assert torch.allclose(y0, y1, rtol=1e-10, atol=1e-10) and torch.allclose(h0, h1, rtol=1e-10, atol=1e-10)


def test_chunked_oracle_with_clamp_and_no_options():
    t = _oracle_inputs(1, 19, 2, 3, 1, 4, seed=3)
    kw = dict(dt_softplus=True, dt_limit=(0.05, 0.15))
    y0, h0 = ssd_recurrence(t["x"], t["dt"], t["A"], t["B"], t["C"], **kw)
    y1, h1 = ssd_chunked(t["x"], t["dt"], t["A"], t["B"], t["C"], 8, **kw)
    assert torch.allclose(y0, y1, rtol=1e-10, atol=1e-10) and torch.allclose(h0, h1, rtol=1e-10, atol=1e-10)


def test_chunked_oracle_gradients_match_recurrence():
    t = _oracle_inputs(2, 21, 4, 3, 2, 4, seed=5, grad=True)
    gen = torch.Generator().manual_seed(6)
    wy = torch.randn(2, 21, 4, 3, generator=gen, dtype=torch.float64)
    wh = torch.randn(2, 4, 3, 4, generator=gen, dtype=torch.float64)
    grads = []
    for fn, extra in ((ssd_recurrence, ()), (ssd_chunked, (8,))):
        y, h = _call(fn, t, *extra)
        grads.append(torch.autograd.grad((y * wy).sum() + (h * wh).sum(), list(t.values())))
    for name, a, b in zip(t, *grads):
        assert torch.allclose(a, b, rtol=1e-9, atol=1e-9), name


def test_symbols_and_descriptor():
    for n in ("ss2d_ssd_fwd", "ss2d_ssd_fwd_workspace_bytes", "ss2d_ssd_bwd", "ss2d_ssd_bwd_workspace_bytes"):
        assert hasattr(_lib.lib(), n) and n in _lib.EXPORTS, n
    # 10 int32 and 2 floats, then 15 int64: the C struct's offsets
    assert _lib.SsdDesc.x_batch_stride.offset == 48
    assert _lib.SsdDesc.bc_group_stride.offset == 48 + 14 * 8
    assert ctypes.sizeof(_lib.SsdDesc) == 48 + 15 * 8


def _desc(b=2, L=100, h=4, P=64, g=2, N=32, Q=64, dtype=_lib.SS2D_BF16, softplus=1, d_mode=1):
    d = _lib.SsdDesc()
    d.batch, d.seqlen, d.heads, d.headdim, d.n_groups, d.dstate, d.chunk_size = b, L, h, P, g, N, Q
    d.io_dtype, d.dt_softplus, d.d_mode, d.dt_min, d.dt_max = dtype, softplus, d_mode, -math.inf, math.inf
    for t in ("x", "z", "out"):
        setattr(d, f"{t}_batch_stride", L * h * P)
        setattr(d, f"{t}_seq_stride", h * P)
        setattr(d, f"{t}_head_stride", P)
    d.dt_batch_stride, d.dt_seq_stride, d.dt_head_stride = L * h, h, 1
    d.bc_batch_stride, d.bc_seq_stride, d.bc_group_stride = L * g * N, g * N, N
    return d


def _fwd(d, x=GOOD, dt=GOOD, A=GOOD, B=GOOD, C=GOOD, D=GOOD, dt_bias=None, z=None, h0=None, out=GOOD, hT=None, ws=GOOD,
         ws_bytes=None):
    lib = _lib.lib()
    if ws_bytes is None:
        ws_bytes = lib.ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d)) if d is not None else 0
    desc = None if d is None else ctypes.byref(d)
    before = _lib.launch_count()
    rc = lib.ss2d_ssd_fwd(desc, x, dt, A, B, C, D, dt_bias, z, h0, out, hT, ws, ws_bytes, None)
    assert _lib.launch_count() == before, "no launch on error"
    return rc


def test_workspace_bytes():
    lib = _lib.lib()
    d = _desc(b=2, L=100, h=4, P=64, N=32, Q=64)
    assert lib.ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d)) == 4 * 2 * 4 * 2 * (2 * 64 + 64 * 32)
    d.chunk_size = 100
    assert lib.ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d)) == 0


def _with(**kw):
    d = _desc()
    for k, v in kw.items():
        setattr(d, k, v)
    return d


@pytest.mark.parametrize("field,value,code", [
    ("batch", 0, ERR_SHAPE), ("seqlen", 0, ERR_SHAPE), ("heads", 0, ERR_SHAPE), ("n_groups", 0, ERR_SHAPE),
    ("n_groups", 3, ERR_SHAPE), ("batch", 65536, ERR_SHAPE), ("heads", 65536, ERR_SHAPE), ("dt_min", math.nan, ERR_SHAPE),
    ("dt_min", 2.0, ERR_SHAPE),
    ("dstate", 0, ERR_SHAPE), ("dstate", 24, ERR_DSTATE), ("dstate", 272, ERR_DSTATE),
    ("headdim", 16, ERR_UNSUPPORTED), ("headdim", 96, ERR_UNSUPPORTED), ("chunk_size", 32, ERR_UNSUPPORTED),
    ("chunk_size", 512, ERR_UNSUPPORTED),
    ("io_dtype", 3, ERR_DTYPE), ("dt_softplus", 2, ERR_DTYPE), ("d_mode", 3, ERR_DTYPE), ("d_mode", -1, ERR_DTYPE),
    ("x_seq_stride", -1, ERR_LAYOUT), ("bc_group_stride", -2, ERR_LAYOUT), ("dt_head_stride", -1, ERR_LAYOUT),
    ("out_head_stride", 32, ERR_LAYOUT), ("out_seq_stride", 64 * 3, ERR_LAYOUT), ("out_batch_stride", 0, ERR_LAYOUT),
])
def test_descriptor_errors(field, value, code):
    d = _with(**{field: value})
    if field == "dt_min" and value == 2.0:
        d.dt_max = 1.0
    assert _fwd(d, ws_bytes=1 << 30) == code


def test_out_layouts_that_do_not_overlap_are_accepted():
    """The workspace size is 0 exactly when the descriptor is rejected: a (batch, heads, L, P) order, a padded head pitch
    and broadcast (stride 0) inputs pass."""
    ws = lambda d: _lib.lib().ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d))   # noqa: E731
    assert ws(_with(out_head_stride=100 * 64, out_seq_stride=64, out_batch_stride=4 * 100 * 64)) > 0
    assert ws(_with(out_head_stride=72, out_seq_stride=4 * 72, out_batch_stride=100 * 4 * 72)) > 0
    assert ws(_with(x_batch_stride=0, bc_batch_stride=0, dt_head_stride=0)) > 0


def test_pointer_errors():
    d = _desc()
    assert _fwd(None) == ERR_NULL
    for k in ("x", "dt", "A", "B", "C", "out"):
        assert _fwd(d, **{k: None}) == ERR_NULL, k
    assert _fwd(d, D=None) == ERR_NULL                      # d_mode 1 needs D
    for k in ("x", "dt", "B", "C", "out", "z"):
        assert _fwd(d, **{k: ODD}) == ERR_ALIGNMENT, k
    for k in ("A", "D", "dt_bias", "h0", "hT", "ws"):
        assert _fwd(d, **{k: MIS4}) == ERR_ALIGNMENT, k
    assert _fwd(d, ws=None) == ERR_WORKSPACE
    assert _fwd(d, ws_bytes=_lib.lib().ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d)) - 4) == ERR_WORKSPACE


def _t(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype)


def test_python_checks():
    import ceigm_unet_b200 as pkg
    x, dt, A, B, C = _t(1, 8, 2, 32), _t(1, 8, 2), _t(2), _t(1, 8, 1, 16), _t(1, 8, 1, 16)
    f = pkg.mamba_chunk_scan_combined
    for kw in (dict(seq_idx=_t(1, 8, dtype=torch.int32)), dict(cu_seqlens=_t(2, dtype=torch.int32)),
               dict(return_varlen_states=True)):
        with pytest.raises(RuntimeError, match="not supported"):
            f(x, dt, A, B, C, 64, **kw)
    with torch.no_grad():
        bad = [
            (dict(chunk_size=32), "chunk_size"), (dict(x=_t(1, 8, 2, 48)), "headdim|B must"),
            (dict(B=_t(1, 8, 1, 24), C=_t(1, 8, 1, 24)), "dstate"), (dict(B=_t(1, 8, 3, 16), C=_t(1, 8, 3, 16)), "multiple"),
            (dict(C=_t(1, 8, 1, 32)), "C must"), (dict(dt=_t(1, 8, 3)), "dt must"), (dict(A=_t(3)), "A must"),
            (dict(B=_t(1, 8, 1, 16, dtype=torch.float16)), "dtype"), (dict(x=_t(1, 8, 2, 32, dtype=torch.float64)), "float32"),
            (dict(D=_t(3)), "D must"), (dict(z=_t(1, 8, 2, 16)), "z must"), (dict(dt_bias=_t(3)), "dt_bias"),
            (dict(initial_states=_t(1, 2, 32, 8)), "initial_states"), (dict(dt_limit=(1.0, 0.5)), "dt_limit"),
            (dict(), "is_cuda"),
        ]
        for kw, msg in bad:
            args = dict(x=x, dt=dt, A=A, B=B, C=C, chunk_size=64)
            args.update(kw)
            with pytest.raises(RuntimeError, match=msg):
                f(**args)


def _ssd_kernels():
    return {n: b for n, b in _sass_functions().items() if "ssd_" in n and "_kernel" in n}


def test_sass_instantiations_atomics_local_memory_and_hmma():
    funcs = _ssd_kernels()
    product = []
    for t in ("f", "6__half", "13__nv_bfloat16"):
        for P in (32, 64, 128):
            product.append(f"_ZN4ss2d20ssd_chunk_out_kernelI{t}Li{P}EEEvNS_9SsdParamsE")
            for flag in ("0", "1"):
                product.append(f"_ZN4ss2d22ssd_chunk_state_kernelI{t}Li{P}ELb{flag}EEEvNS_9SsdParamsE")
                product.append(f"_ZN4ss2d20ssd_chunk_bwd_kernelI{t}Li{P}ELb{flag}EEEvNS_9SsdParamsE")
    for name in product:
        assert name in funcs, name
        assert "HMMA" in funcs[name], name
    for kern in ("ssd_state_pass_kernel", "ssd_state_pass_bwd_kernel", "ssd_param_grad_kernel"):
        assert any(kern in n for n in funcs), kern
    for kern in ("ssd_dt_bwd_kernel", "ssd_bc_grad_kernel"):
        assert sum(kern in n for n in funcs) == 3, kern
    assert len(funcs) == 54
    for n, body in funcs.items():
        assert not _GLOBAL_ATOMIC.search(body), n
        assert "LDL" not in body and "STL" not in body, n


def _bwd(d, dout=GOOD, dx=GOOD, ddt=GOOD, dA=GOOD, dB=GOOD, dC=GOOD, dD=GOOD, ws=GOOD, ws_bytes=None, D=GOOD, dz=None):
    lib = _lib.lib()
    if ws_bytes is None:
        ws_bytes = lib.ss2d_ssd_bwd_workspace_bytes(ctypes.byref(d))
    before = _lib.launch_count()
    rc = lib.ss2d_ssd_bwd(ctypes.byref(d), GOOD, GOOD, GOOD, GOOD, GOOD, D, None, None, None, dout, None, dx, ddt, dA, dB, dC, dD,
                          None, dz, None, ws, ws_bytes, None)
    assert _lib.launch_count() == before, "no launch on error"
    return rc


def test_bwd_errors():
    d = _desc()
    lib = _lib.lib()
    assert lib.ss2d_ssd_bwd_workspace_bytes(ctypes.byref(d)) > lib.ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d))
    assert lib.ss2d_ssd_bwd_workspace_bytes(ctypes.byref(_with(headdim=48))) == 0
    assert _bwd(_with(dstate=24), ws_bytes=1 << 30) == ERR_DSTATE
    assert _bwd(_with(chunk_size=32), ws_bytes=1 << 30) == ERR_UNSUPPORTED
    for k in ("dout", "dx", "ddt", "dA", "dB", "dC", "dD"):
        assert _bwd(d, **{k: None}) == ERR_NULL, k
    assert _bwd(_with(d_mode=0), D=None, dD=None, ws=None) == ERR_WORKSPACE     # dD may be NULL without D
    for k in ("dx", "ddt", "dB", "dC", "dz", "dout"):
        assert _bwd(d, **{k: ODD}) == ERR_ALIGNMENT, k
    for k in ("dA", "dD"):
        assert _bwd(d, **{k: MIS4}) == ERR_ALIGNMENT, k
    assert _bwd(d, ws=None) == ERR_WORKSPACE
    assert _bwd(d, ws_bytes=lib.ss2d_ssd_bwd_workspace_bytes(ctypes.byref(d)) - 4) == ERR_WORKSPACE
