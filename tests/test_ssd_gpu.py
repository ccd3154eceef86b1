"""GPU tests of Mamba-2's chunked selective scan, forward and backward (csrc/ssd.cu; C ABI ss2d_ssd_fwd / ss2d_ssd_bwd, Python
`mamba_chunk_scan_combined`).

Reference: the float64 recurrence of oracle/ssd_ref.py (the definition) for L <= 256, its float64 chunked restatement beyond.
16-bit inputs are rounded to their dtype first and used as they are (exact in float64). Bounds, as max|got - ref| / max|ref| per
tensor: fp32 1e-4 (the 3xTF32 products should land near 1e-6), fp16 / bf16 2e-2. Each test records its worst value per
quantity in its user properties (written to the junit report).

Also: agreement with the library's `selective_scan` on the expanded problem at a Mamba-2-130M layer, two calls chained
through final_states equal one call, a prefill stepped with `selective_state_update` equals one call over the longer sequence,
column slices of one in_proj output read in place, the gradients of every input (through out and final_states) against float64
autograd of the same references and against `selective_scan`'s, gradients of chained calls, C ABI calls writing exactly their region of NaN-filled buffers, identical
bits across calls and a CUDA-graph replay, and one call above 2^31 elements of x."""
import ctypes
import math

import pytest
import torch

import ceigm_unet_b200 as pkg
from ceigm_unet_b200 import _lib
from oracle.ssd_ref import ssd_chunked, ssd_recurrence

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
TOL = {F32: 1e-4, F16: 2e-2, BF16: 2e-2}
_DT = {F32: _lib.SS2D_F32, F16: _lib.SS2D_F16, BF16: _lib.SS2D_BF16}

_observed = {}


@pytest.fixture(autouse=True)
def _record_errors(request):
    _observed.clear()
    yield
    request.node.user_properties.extend(sorted(_observed.items()))


def _check(got, ref, what, tol, floor=1e-30):
    """max|got - ref| / max(max|ref|, floor)."""
    ref = ref.detach().double()
    rel = float((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(floor))
    _observed[what] = max(_observed.get(what, 0.0), rel)
    assert rel <= tol, f"{what}: rel err {rel:.3g} > {tol}"


def _inputs(b, L, h, P, g, N, dtype, seed, D_mode=1, z=True, dt_bias=True, softplus=True, h0=True):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)   # noqa: E731
    u = lambda *s: torch.rand(*s, device="cuda", generator=gen)    # noqa: E731
    inp = dict(
        x=r(b, L, h, P).to(dtype),
        dt=(r(b, L, h) * 0.5 - 3.0 if softplus else u(b, L, h) * 0.1).to(dtype),
        A=-(u(h) * 2.0 + 0.5),
        B=r(b, L, g, N).to(dtype),
        C=r(b, L, g, N).to(dtype),
        D=None if D_mode == 0 else (r(h) if D_mode == 1 else r(h, P)),
        z=r(b, L, h, P).to(dtype) if z else None,
        dt_bias=(r(h) * 0.5 if softplus else u(h) * 0.02) if dt_bias else None,
        initial_states=r(b, h, P, N) * 0.5 if h0 else None,
    )
    return inp


def _ref(inp, dt_softplus, dt_limit=(0.0, math.inf)):
    kw = dict(D=inp["D"], z=inp["z"], dt_bias=inp["dt_bias"], initial_states=inp["initial_states"], dt_softplus=dt_softplus,
              dt_limit=dt_limit)
    args = (inp["x"], inp["dt"], inp["A"], inp["B"], inp["C"])
    if inp["x"].shape[1] <= 256:
        return ssd_recurrence(*args, **kw)
    return ssd_chunked(*args, 64, **kw)


def _run(inp, chunk, dt_softplus, dt_limit=(0.0, math.inf)):
    with torch.no_grad():
        return pkg.mamba_chunk_scan_combined(inp["x"], inp["dt"], inp["A"], inp["B"], inp["C"], chunk, D=inp["D"], z=inp["z"],
                                             dt_bias=inp["dt_bias"], initial_states=inp["initial_states"],
                                             dt_softplus=dt_softplus, dt_limit=dt_limit, return_final_states=True)


def _parity(b, L, h, P, g, N, dtype, chunk, seed, D_mode=1, z=True, dt_bias=True, softplus=True, h0=True,
            dt_limit=(0.0, math.inf)):
    inp = _inputs(b, L, h, P, g, N, dtype, seed, D_mode, z, dt_bias, softplus, h0)
    out, fin = _run(inp, chunk, softplus, dt_limit)
    ref_out, ref_fin = _ref(inp, softplus, dt_limit)
    assert out.dtype == dtype and fin.dtype == F32 and tuple(fin.shape) == (b, h, P, N)
    _check(out, ref_out, "out", TOL[dtype])
    _check(fin, ref_fin, "final_states", TOL[dtype])


# every dtype x headdim x dstate, with chunk size, L, groups and the options cycling through their values
_GRID = []
for i, (dt_, P, N) in enumerate((d, p, n) for d in (F32, F16, BF16) for p in (32, 64, 128) for n in (16, 64, 128, 256)):
    Q = (64, 128, 256)[i % 3]
    L = (1, 63, Q, Q + 1, 1000, 2048)[i % 6]
    _GRID.append((dt_, P, N, Q, L, (1, 2, 4)[i % 3], i % 3, bool(i % 2), bool(i % 4 < 2), bool(i % 5 != 0), bool(i % 3 != 1)))


@pytest.mark.parametrize("dtype,P,N,Q,L,g,D_mode,z,dt_bias,softplus,h0", _GRID,
                         ids=[f"{str(c[0])[6:]}-P{c[1]}-N{c[2]}-Q{c[3]}-L{c[4]}-g{c[5]}" for c in _GRID])
def test_parity_grid(dtype, P, N, Q, L, g, D_mode, z, dt_bias, softplus, h0):
    _parity(2, L, 4, P, g, N, dtype, Q, seed=L + P + N, D_mode=D_mode, z=z, dt_bias=dt_bias, softplus=softplus, h0=h0)


@pytest.mark.parametrize("Q", [64, 128, 256])
@pytest.mark.parametrize("L", [1, 63, "Q", "Q+1", 1000, 2048])
def test_chunk_by_length(Q, L):
    L = {"Q": Q, "Q+1": Q + 1}.get(L, L)
    _parity(2, L, 4, 64, 2, 64, F32, Q, seed=Q + L)


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("h,g", [(4, 1), (4, 2), (4, 4), (6, 3), (8, 2)])
def test_groups_by_heads(dtype, h, g):
    _parity(2, 300, h, 64, g, 32, dtype, 128, seed=h * 10 + g)


@pytest.mark.parametrize("dtype", [F32, F16])
@pytest.mark.parametrize("z", [False, True])
@pytest.mark.parametrize("D_mode", [0, 1, 2])
def test_gate_by_skip(dtype, z, D_mode):
    _parity(1, 200, 4, 32, 1, 16, dtype, 64, seed=D_mode + 3 * z, D_mode=D_mode, z=z)


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("softplus,limit", [(True, (0.02, 0.08)), (False, (0.03, 0.06)), (True, (0.0, 0.05)),
                                            (False, (0.0, math.inf))])
def test_dt_limit(dtype, softplus, limit):
    """A clamp that is active for part of the positions; (0, inf) without softplus leaves t untouched, as in mamba_ssm."""
    _parity(2, 257, 4, 64, 2, 32, dtype, 128, seed=11, softplus=softplus, dt_limit=limit)


def test_unclamped_negative_dt():
    """dt + dt_bias < 0 without softplus and the default dt_limit: t stays negative (mamba_ssm clamps only a non-default
    limit)."""
    inp = _inputs(1, 130, 2, 32, 1, 16, F32, 5, softplus=False)
    inp["dt"] = inp["dt"] - 0.06
    out, fin = _run(inp, 64, False)
    ref_out, ref_fin = _ref(inp, False)
    _check(out, ref_out, "out", 1e-4)
    _check(fin, ref_fin, "final_states", 1e-4)


def test_returns_out_only_by_default():
    inp = _inputs(1, 70, 2, 32, 1, 16, F32, 1)
    with torch.no_grad():
        out = pkg.mamba_chunk_scan_combined(inp["x"], inp["dt"], inp["A"], inp["B"], inp["C"], 64, D=inp["D"])
    assert isinstance(out, torch.Tensor) and out.shape == inp["x"].shape


def test_against_selective_scan_expanded():
    """A Mamba-2-130M layer (24 heads x 64, dstate 128, one group, L 2048) in fp32 through the library's already-verified
    `selective_scan` with A, dt, D and dt_bias expanded over headdim."""
    b, L, h, P, g, N = 1, 2048, 24, 64, 1, 128
    inp = _inputs(b, L, h, P, g, N, F32, 7, D_mode=1)
    out, fin = _run(inp, 256, True)
    dim = h * P
    u = inp["x"].reshape(b, L, dim).transpose(1, 2).contiguous()
    delta = inp["dt"].repeat_interleave(P, dim=2).transpose(1, 2).contiguous()
    A = inp["A"].repeat_interleave(P)[:, None].expand(dim, N).contiguous()
    Bm = inp["B"].permute(0, 2, 3, 1).contiguous()
    Cm = inp["C"].permute(0, 2, 3, 1).contiguous()
    z = inp["z"].reshape(b, L, dim).transpose(1, 2).contiguous()
    with torch.no_grad():
        ref, last = pkg.selective_scan(u, delta, A, Bm, Cm, inp["D"].repeat_interleave(P), inp["dt_bias"].repeat_interleave(P),
                                       True, initial_state=inp["initial_states"].reshape(b, dim, N), return_last_state=True, z=z)
    _check(out.reshape(b, L, dim).transpose(1, 2), ref, "out_vs_scan", 1e-4)
    _check(fin.reshape(b, dim, N), last, "final_vs_scan", 1e-4)


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("m", [1, 100, 256])
def test_chained_calls(dtype, m):
    """[0, m) then [m, L) with initial_states = the first call's final_states equals one call over [0, L)."""
    L = 600
    inp = _inputs(2, L, 4, 64, 2, 64, dtype, m)
    out, fin = _run(inp, 128, True)
    first = {k: (v[:, :m] if k in ("x", "dt", "B", "C", "z") else v) for k, v in inp.items()}
    second = {k: (v[:, m:] if k in ("x", "dt", "B", "C", "z") else v) for k, v in inp.items()}
    o1, f1 = _run(first, 128, True)
    second["initial_states"] = f1
    o2, f2 = _run(second, 128, True)
    tol = 1e-5 if dtype == F32 else 1e-2
    _check(torch.cat([o1, o2], 1), out, "chained_out", tol)
    _check(f2, fin, "chained_final", tol)


def test_prefill_then_decode_steps():
    """A prefill's final_states stepped k times with selective_state_update (A and dt expanded per channel) equals one call
    over L + k."""
    b, L, k, h, P, g, N = 2, 500, 8, 4, 64, 2, 64
    inp = _inputs(b, L + k, h, P, g, N, F32, 3)
    out, _ = _run(inp, 256, True)
    pre = {kk: (v[:, :L] if kk in ("x", "dt", "B", "C", "z") else v) for kk, v in inp.items()}
    _, state = _run(pre, 256, True)
    state = state.reshape(b, h * P, N).contiguous()
    A = inp["A"].repeat_interleave(P)[:, None].expand(h * P, N).contiguous()
    D = inp["D"].repeat_interleave(P)
    bias = inp["dt_bias"].repeat_interleave(P)
    with torch.no_grad():
        for i in range(k):
            l = L + i
            y = pkg.selective_state_update(state, inp["x"][:, l].reshape(b, h * P), inp["dt"][:, l].repeat_interleave(P, dim=1),
                                           A, inp["B"][:, l], inp["C"][:, l], D, inp["z"][:, l].reshape(b, h * P), bias, True)
            _check(y, out[:, l].reshape(b, h * P), "decode_step", 1e-4)


def test_in_proj_column_slices():
    """x, z, B, C and dt as column slices of one (batch, L, width) projection output are read in place and give the bits of
    dense copies."""
    b, L, h, P, g, N = 2, 333, 4, 64, 2, 32
    gen = torch.Generator(device="cuda").manual_seed(9)
    d_in = h * P
    width = 2 * d_in + 2 * g * N + h
    zxbcdt = torch.randn(b, L, width, device="cuda", generator=gen).to(BF16)
    zxbcdt[..., -h:] = zxbcdt[..., -h:] * 0.5 - 3.0
    z, x, Bf, Cf, dt = torch.split(zxbcdt, [d_in, d_in, g * N, g * N, h], dim=-1)
    x, z = x.view(b, L, h, P), z.view(b, L, h, P)
    Bm, Cm = Bf.view(b, L, g, N), Cf.view(b, L, g, N)
    A = -torch.rand(h, device="cuda", generator=gen) - 0.5
    D = torch.randn(h, device="cuda", generator=gen)
    with torch.no_grad():
        got = pkg.mamba_chunk_scan_combined(x, dt, A, Bm, Cm, 128, D=D, z=z, dt_softplus=True, return_final_states=True)
        dense = pkg.mamba_chunk_scan_combined(x.contiguous(), dt.contiguous(), A, Bm.contiguous(), Cm.contiguous(), 128, D=D,
                                              z=z.contiguous(), dt_softplus=True, return_final_states=True)
    assert torch.equal(got[0], dense[0]) and torch.equal(got[1], dense[1])


def _desc(b, L, h, P, g, N, Q, dtype, x, z, out, dt, Bm, d_mode, softplus):
    d = _lib.SsdDesc()
    d.batch, d.seqlen, d.heads, d.headdim, d.n_groups, d.dstate, d.chunk_size = b, L, h, P, g, N, Q
    d.io_dtype, d.dt_softplus, d.d_mode, d.dt_min, d.dt_max = _DT[dtype], int(softplus), d_mode, -math.inf, math.inf
    d.x_batch_stride, d.x_seq_stride, d.x_head_stride = x.stride()[:3]
    d.z_batch_stride, d.z_seq_stride, d.z_head_stride = z.stride()[:3]
    d.out_batch_stride, d.out_seq_stride, d.out_head_stride = out.stride()[:3]
    d.dt_batch_stride, d.dt_seq_stride, d.dt_head_stride = dt.stride()
    d.bc_batch_stride, d.bc_seq_stride, d.bc_group_stride = Bm.stride()[:3]
    return d


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_abi_writes_exactly_its_region(dtype):
    """out with padded rows inside a NaN-filled buffer with guard bands, and hT between guard bands: exactly the documented
    elements change, and they equal the Python path's."""
    b, L, h, P, g, N, Q = 2, 150, 4, 32, 2, 32, 64
    inp = _inputs(b, L, h, P, g, N, dtype, 21, D_mode=2)
    pad_h, guard = P + 8, 64
    buf = torch.full((guard + b * L * h * pad_h + guard,), float("nan"), dtype=dtype, device="cuda")
    out = buf[guard:guard + b * L * h * pad_h].view(b, L, h, pad_h)[..., :P]
    hbuf = torch.full((guard + b * h * P * N + guard,), float("nan"), device="cuda")
    hT = hbuf[guard:guard + b * h * P * N]
    x, z, dt, Bm, Cm = inp["x"], inp["z"], inp["dt"], inp["B"], inp["C"]
    d = _desc(b, L, h, P, g, N, Q, dtype, x, z, out, dt, Bm, 2, True)
    lib = _lib.lib()
    ws_bytes = lib.ss2d_ssd_fwd_workspace_bytes(ctypes.byref(d))
    ws = torch.empty(ws_bytes // 4, device="cuda")
    h0 = inp["initial_states"].contiguous()
    p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    before = pkg.launch_count()
    rc = lib.ss2d_ssd_fwd(ctypes.byref(d), p(x), p(dt), p(inp["A"]), p(Bm), p(Cm), p(inp["D"]), p(inp["dt_bias"]), p(z), p(h0),
                          p(out), p(hT), p(ws), ws_bytes, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert rc == 0 and pkg.launch_count() - before == 3
    ref_out, ref_fin = _run(inp, Q, True)
    assert torch.equal(out, ref_out) and torch.equal(hT.view(b, h, P, N), ref_fin)
    assert buf[:guard].isnan().all() and buf[-guard:].isnan().all()
    assert buf[guard:guard + b * L * h * pad_h].view(b, L, h, pad_h)[..., P:].isnan().all()
    assert hbuf[:guard].isnan().all() and hbuf[-guard:].isnan().all()


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_bit_identical_repeat_and_graph(dtype):
    inp = _inputs(2, 700, 8, 64, 2, 128, dtype, 4, D_mode=2)
    first = _run(inp, 256, True)
    again = _run(inp, 256, True)
    assert torch.equal(first[0], again[0]) and torch.equal(first[1], again[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _run(inp, 256, True)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = _run(inp, 256, True)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured[0], first[0]) and torch.equal(captured[1], first[1])


def test_above_2_31_elements():
    """x with more than 2^31 elements (bf16, 4.3 GB): the last batch entry checked against the reference on its own."""
    b, L, h, P, g, N = 2, 65600, 128, 128, 1, 16
    assert b * L * h * P > 2 ** 31
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(b, L, h, P, device="cuda", generator=gen, dtype=BF16)
    dt = (torch.randn(b, L, h, device="cuda", generator=gen) * 0.5 - 3.0).to(BF16)
    A = -torch.rand(h, device="cuda", generator=gen) - 0.5
    Bm = torch.randn(b, L, g, N, device="cuda", generator=gen, dtype=BF16)
    Cm = torch.randn(b, L, g, N, device="cuda", generator=gen, dtype=BF16)
    with torch.no_grad():
        out, fin = pkg.mamba_chunk_scan_combined(x, dt, A, Bm, Cm, 256, dt_softplus=True, return_final_states=True)
    tail = slice(L - 300, L)
    heads = slice(h - 2, h)
    _, h_mid = ssd_chunked(x[1:, :L - 300, heads], dt[1:, :L - 300, heads], A[heads], Bm[1:, :L - 300], Cm[1:, :L - 300], 256,
                           dt_softplus=True)
    ref_out, ref_fin = ssd_recurrence(x[1:, tail, heads], dt[1:, tail, heads], A[heads], Bm[1:, tail], Cm[1:, tail],
                                      initial_states=h_mid, dt_softplus=True)
    _check(out[1:, tail, heads], ref_out, "large_out", 2e-2)
    _check(fin[1:, heads], ref_fin, "large_final", 2e-2)


# ---- backward ------------------------------------------------------------------------------------------------------------
_NAMES = ("x", "dt", "A", "B", "C", "D", "z", "dt_bias", "initial_states")


def _grad_parity(b, L, h, P, g, N, dtype, chunk, seed, D_mode=1, z=True, dt_bias=True, softplus=True, h0=True,
                 dt_limit=(0.0, math.inf), dfinal=True):
    inp = _inputs(b, L, h, P, g, N, dtype, seed, D_mode, z, dt_bias, softplus, h0)
    gen = torch.Generator(device="cuda").manual_seed(seed + 1)
    wy = torch.randn(b, L, h, P, device="cuda", generator=gen)
    wh = torch.randn(b, h, P, N, device="cuda", generator=gen) if dfinal else None
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in inp.items() if v is not None}
    args = {k: leaves.get(k) for k in _NAMES}
    out, fin = pkg.mamba_chunk_scan_combined(args["x"], args["dt"], args["A"], args["B"], args["C"], chunk, D=args["D"],
                                             z=args["z"], dt_bias=args["dt_bias"], initial_states=args["initial_states"],
                                             dt_softplus=softplus, dt_limit=dt_limit, return_final_states=True)
    loss = (out.float() * wy).sum() + ((fin * wh).sum() if dfinal else 0.0)
    got = torch.autograd.grad(loss, list(leaves.values()))
    ref_leaves = {k: v.detach().double().requires_grad_(True) for k, v in inp.items() if v is not None}
    rin = {k: ref_leaves.get(k) for k in _NAMES}
    ref_out, ref_fin = _ref(rin, softplus, dt_limit)
    ref_loss = (ref_out * wy.double()).sum() + ((ref_fin * wh.double()).sum() if dfinal else 0.0)
    ref = torch.autograd.grad(ref_loss, list(ref_leaves.values()))
    # a gradient that vanishes exactly (dA at L = 1 without an initial state: exp(t A) multiplies a zero state) is held to the
    # rounding noise of its terms: 1e-3 of the largest reference gradient as the floor of the scale
    floor = 1e-3 * max(float(r.abs().max()) for r in ref)
    for name, a, r in zip(leaves, got, ref):
        assert a.dtype == leaves[name].dtype and a.shape == leaves[name].shape, name
        # dA = sum_l d a_l t_l over batch and positions is a sum whose terms largely cancel; in 16-bit its terms carry the
        # rounding of the states to the I/O dtype, so it is held to 5e-2 (fp32: the common bar)
        tol = 5e-2 if name == "A" and dtype != F32 else TOL[dtype]
        _check(a, r, "d" + name, tol, floor)


_GGRID = []
for i, (dt_, P, N) in enumerate((d, p, n) for d in (F32, BF16, F16) for p in (32, 64, 128) for n in (16, 64, 128, 256)):
    if i % 2 and dt_ != F32:
        continue
    Q = (64, 128, 256)[i % 3]
    L = (1, 63, Q, Q + 1, 1000, 2048)[(i // 2) % 6]
    _GGRID.append((dt_, P, N, Q, L, (1, 2, 4)[i % 3], i % 3, bool(i % 2), bool(i % 4 < 2), bool(i % 5 != 0), bool(i % 3 != 1),
                   bool(i % 4 != 3)))


@pytest.mark.parametrize("dtype,P,N,Q,L,g,D_mode,z,dt_bias,softplus,h0,dfinal", _GGRID,
                         ids=[f"{str(c[0])[6:]}-P{c[1]}-N{c[2]}-Q{c[3]}-L{c[4]}-g{c[5]}" for c in _GGRID])
def test_grad_parity_grid(dtype, P, N, Q, L, g, D_mode, z, dt_bias, softplus, h0, dfinal):
    _grad_parity(2, L, 4, P, g, N, dtype, Q, seed=L + P + N + 7, D_mode=D_mode, z=z, dt_bias=dt_bias, softplus=softplus,
                 h0=h0, dfinal=dfinal)


@pytest.mark.parametrize("Q", [64, 128, 256])
@pytest.mark.parametrize("L", [1, 63, "Q", "Q+1", 1000])
def test_grad_chunk_by_length(Q, L):
    L = {"Q": Q, "Q+1": Q + 1}.get(L, L)
    _grad_parity(2, L, 4, 64, 2, 64, F32, Q, seed=Q + L)


@pytest.mark.parametrize("h,g", [(4, 1), (4, 4), (6, 3)])
def test_grad_groups_by_heads(h, g):
    _grad_parity(2, 300, h, 32, g, 32, F32, 128, seed=h + g)


@pytest.mark.parametrize("z", [False, True])
@pytest.mark.parametrize("D_mode", [0, 1, 2])
def test_grad_gate_by_skip(z, D_mode):
    _grad_parity(1, 200, 4, 32, 1, 16, F32, 64, seed=D_mode + 3 * z, D_mode=D_mode, z=z)


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("softplus,limit", [(True, (0.02, 0.08)), (False, (0.03, 0.06))])
def test_grad_dt_limit(dtype, softplus, limit):
    """Where the clamp is active the gradient to dt and dt_bias is zero."""
    _grad_parity(2, 257, 4, 64, 2, 32, dtype, 128, seed=13, softplus=softplus, dt_limit=limit)


def test_grad_against_selective_scan_expanded():
    """Mamba-2-130M layer in fp32: gradients against the library's `selective_scan` on the expanded problem, reduced over
    the expanded axes."""
    b, L, h, P, g, N = 1, 2048, 24, 64, 1, 128
    inp = _inputs(b, L, h, P, g, N, F32, 7, D_mode=1)
    gen = torch.Generator(device="cuda").manual_seed(8)
    wy = torch.randn(b, L, h, P, device="cuda", generator=gen)
    wh = torch.randn(b, h, P, N, device="cuda", generator=gen)
    la = {k: v.detach().clone().requires_grad_(True) for k, v in inp.items()}
    out, fin = pkg.mamba_chunk_scan_combined(la["x"], la["dt"], la["A"], la["B"], la["C"], 256, D=la["D"], z=la["z"],
                                             dt_bias=la["dt_bias"], initial_states=la["initial_states"], dt_softplus=True,
                                             return_final_states=True)
    got = torch.autograd.grad((out * wy).sum() + (fin * wh).sum(), list(la.values()))
    lb = {k: v.detach().clone().requires_grad_(True) for k, v in inp.items()}
    dim = h * P
    u = lb["x"].reshape(b, L, dim).transpose(1, 2)
    delta = lb["dt"].repeat_interleave(P, dim=2).transpose(1, 2)
    A = lb["A"].repeat_interleave(P)[:, None].expand(dim, N)
    z = lb["z"].reshape(b, L, dim).transpose(1, 2)
    ref, last = pkg.selective_scan(u.contiguous(), delta.contiguous(), A.contiguous(), lb["B"].permute(0, 2, 3, 1).contiguous(),
                                   lb["C"].permute(0, 2, 3, 1).contiguous(), lb["D"].repeat_interleave(P),
                                   lb["dt_bias"].repeat_interleave(P), True, initial_state=lb["initial_states"].reshape(b, dim, N),
                                   return_last_state=True, z=z.contiguous())
    loss = (ref.transpose(1, 2).reshape(b, L, h, P) * wy).sum() + (last.reshape(b, h, P, N) * wh).sum()
    want = torch.autograd.grad(loss, list(lb.values()))
    for name, a, r in zip(la, got, want):
        _check(a, r, "d" + name + "_vs_scan", 1e-4)


@pytest.mark.parametrize("m", [100, 256])
def test_grad_chained_calls(m):
    """Gradients of two calls joined by initial_states = final_states equal the gradients of one call."""
    L = 600
    inp = _inputs(2, L, 4, 64, 2, 64, F32, m)
    gen = torch.Generator(device="cuda").manual_seed(3)
    wy = torch.randn(2, L, 4, 64, device="cuda", generator=gen)
    wh = torch.randn(2, 4, 64, 64, device="cuda", generator=gen)
    seq = ("x", "dt", "B", "C", "z")

    def run(split):
        la = {k: v.detach().clone().requires_grad_(True) for k, v in inp.items()}
        kw = lambda d, sl: dict(D=la["D"], z=d["z"][:, sl], dt_bias=la["dt_bias"], dt_softplus=True,   # noqa: E731
                                return_final_states=True)
        if split:
            o1, f1 = pkg.mamba_chunk_scan_combined(*(la[k][:, :m] for k in ("x", "dt")), la["A"], la["B"][:, :m],
                                                   la["C"][:, :m], 128, initial_states=la["initial_states"],
                                                   **kw(la, slice(0, m)))
            o2, f2 = pkg.mamba_chunk_scan_combined(*(la[k][:, m:] for k in ("x", "dt")), la["A"], la["B"][:, m:],
                                                   la["C"][:, m:], 128, initial_states=f1, **kw(la, slice(m, L)))
            out, fin = torch.cat([o1, o2], 1), f2
        else:
            out, fin = pkg.mamba_chunk_scan_combined(la["x"], la["dt"], la["A"], la["B"], la["C"], 128,
                                                     initial_states=la["initial_states"], **kw(la, slice(0, L)))
        return torch.autograd.grad((out * wy).sum() + (fin * wh).sum(), list(la.values()))
    assert all(k in inp for k in seq)
    for name, a, r in zip(inp, run(True), run(False)):
        _check(a, r, "chained_d" + name, 1e-5)


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_grad_bit_identical_repeat_and_graph(dtype):
    inp = _inputs(2, 700, 8, 64, 2, 128, dtype, 4, D_mode=2)
    from ceigm_unet_b200 import ops
    prep = ops.ssd_prepare(inp["x"], inp["dt"], inp["A"], inp["B"], inp["C"], 256, inp["D"], inp["z"], inp["dt_bias"],
                           inp["initial_states"])
    gen = torch.Generator(device="cuda").manual_seed(2)
    dout = torch.randn(inp["x"].shape, device="cuda", generator=gen).to(dtype)
    dfin = torch.randn(inp["initial_states"].shape, device="cuda", generator=gen)
    call = lambda: ops.ssd_bwd(*prep[:5], 256, *prep[5:], True, (0.0, math.inf), dout, dfin)   # noqa: E731
    first, again = call(), call()
    for a, b in zip(first, again):
        assert torch.equal(a, b)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = call()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(captured, first):
        assert torch.equal(a, b)


def test_autograd_saves_only_inputs():
    """The Function keeps the prepared inputs and nothing the size of the chunk states."""
    inp = _inputs(1, 300, 4, 64, 1, 128, F32, 9)
    la = {k: v.detach().clone().requires_grad_(True) for k, v in inp.items()}
    out = pkg.mamba_chunk_scan_combined(la["x"], la["dt"], la["A"], la["B"], la["C"], 64, D=la["D"], z=la["z"],
                                        dt_bias=la["dt_bias"], initial_states=la["initial_states"], dt_softplus=True)
    saved = out.grad_fn.saved_tensors
    assert len(saved) == 9
    assert sum(t.numel() for t in saved if t is not None) == sum(v.numel() for v in inp.values())
