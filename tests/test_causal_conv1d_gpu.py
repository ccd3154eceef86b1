"""GPU tests of the causal depthwise conv1d (csrc/causal_conv1d.cu; C ABI ss2d_conv1d_*, Python `causal_conv1d_fn` /
`causal_conv1d_update`, drop-ins `causal_conv1d_cuda` / `causal_conv1d`).

Reference: a float64 restatement of causal-conv1d 1.1.x's contract (include/ss2d_b200.h):
    pre[l] = bias + sum_k w[k] x[l-(W-1)+k] (x = 0 before 0),  out = act(pre);
    g = dout act'(pre),  dx[l] = sum_k w[k] g[l+(W-1)-k] (g = 0 past L - 1),  dw[k] = sum_{b,l} g x[l-(W-1)+k],  db = sum_{b,l} g.
16-bit inputs are used as they are (exact in float64). Tolerances, as max|got - ref| / max|ref| per tensor: fp32 out and dx
1e-5, dweight and dbias 5e-5, the decode chain through the scan 1e-4. 16-bit outputs are checked elementwise:
|got - ref| <= u |ref| + tau max|ref| with u = 2^-8 (bf16) or 2^-11 (fp16) and tau the fp32 bound, i.e. correctly rounded up to
fp32 noise. Each test records the worst value per quantity in its user properties (written to the junit report).

Also: mamba's xz.chunk view and a misaligned x (the scalar path) give the bits of a dense aligned x, C ABI calls write exactly
their region of NaN-filled buffers with guard bands, one call above 2^31 elements, identical bits across calls and graph replays,
prefill + decode steps equal one forward, and a Mamba-mixer-shaped decode chain with `selective_state_update` equals one full pass."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from ceigm_unet_b200 import _lib

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
_DT = {F32: _lib.SS2D_F32, F16: _lib.SS2D_F16, BF16: _lib.SS2D_BF16}
ROUND = {BF16: 2.0 ** -8, F16: 2.0 ** -11}

_observed = {}


@pytest.fixture(autouse=True)
def _record_errors(request):
    _observed.clear()
    yield
    request.node.user_properties.extend(sorted(_observed.items()))


def _note(key, v):
    _observed[key] = max(_observed.get(key, 0.0), v)


def _check(got, ref, what, tol=1e-5):
    """fp32: max error relative to max|ref|; 16-bit: the elementwise rounding bound."""
    ref = ref.detach().double()
    err = (got.detach().double() - ref).abs()
    scale = ref.abs().max().clamp_min(1e-30)
    if got.dtype in ROUND:
        ratio = float((err / (ROUND[got.dtype] * ref.abs() + tol * scale)).max())
        _note(what + "16_ratio", ratio)
        assert ratio <= 1.0, f"{what}: {got.dtype} error {ratio:.3g} x the rounding bound"
    else:
        rel = float(err.max() / scale)
        _note(what, rel)
        assert rel <= tol, f"{what}: rel err {rel:.3g} > {tol}"


def _inputs(batch, dim, L, W, xdt, wdt, seed, bias=True):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    return dict(x=r(batch, dim, L).to(xdt), w=(0.5 * r(dim, W)).to(wdt), b=(0.5 * r(dim)).to(wdt) if bias else None,
                dout=r(batch, dim, L).to(xdt))


def _shifted(t, W, k):
    """t[..., l - (W-1) + k] with zeros before position 0"""
    return F.pad(t, (W - 1, 0))[..., k:k + t.shape[-1]]


def _ref_fwd(x, w, b, silu):
    x, w = x.double(), w.double()
    W = w.shape[1]
    pre = torch.zeros_like(x) + (b.double()[:, None] if b is not None else 0.0)
    for k in range(W):
        pre = pre + w[:, k, None] * _shifted(x, W, k)
    return (F.silu(pre) if silu else pre), pre


def _ref_bwd(x, w, b, dout, silu):
    _, pre = _ref_fwd(x, w, b, silu)
    x, w, g = x.double(), w.double(), dout.double()
    W, L = w.shape[1], x.shape[-1]
    if silu:
        s = torch.sigmoid(pre)
        g = g * s * (1 + pre * (1 - s))
    gp = F.pad(g, (0, W - 1))
    dx = sum(w[:, k, None] * gp[..., W - 1 - k:W - 1 - k + L] for k in range(W))
    dw = torch.stack([(g * _shifted(x, W, k)).sum((0, 2)) for k in range(W)], 1)
    return dx, dw, g.sum((0, 2))


def _fn(t, silu, x=None):
    import ceigm_unet_b200 as P
    return P.causal_conv1d_fn(t["x"] if x is None else x, t["w"], t["b"], activation="silu" if silu else None)


def _grads(t, silu, x=None):
    """forward + autograd backward -> out, dx, dw, db"""
    x = (t["x"] if x is None else x).detach().requires_grad_(True)
    w = t["w"].detach().requires_grad_(True)
    b = None if t["b"] is None else t["b"].detach().requires_grad_(True)
    out = _fn(dict(t, w=w, b=b), silu, x)
    out.backward(t["dout"])
    return out, x.grad, w.grad, None if b is None else b.grad


def _check_all(t, silu):
    out, dx, dw, db = _grads(t, silu)
    ref_out, _ = _ref_fwd(t["x"], t["w"], t["b"], silu)
    ref_dx, ref_dw, ref_db = _ref_bwd(t["x"], t["w"], t["b"], t["dout"], silu)
    assert out.dtype == t["x"].dtype and dx.dtype == t["x"].dtype and dw.dtype == t["w"].dtype
    assert tuple(out.shape) == tuple(t["x"].shape) and out.is_contiguous()
    _check(out, ref_out, "out")
    _check(dx, ref_dx, "dx")
    _check(dw, ref_dw, "dweight", 5e-5)
    if t["b"] is not None:
        assert db.dtype == t["b"].dtype
        _check(db, ref_db, "dbias", 5e-5)


# ---- coverage ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("silu", [False, True], ids=["noact", "silu"])
@pytest.mark.parametrize("bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("wdt", [F32, BF16], ids=["w_fp32", "w_bf16"])
@pytest.mark.parametrize("xdt", [F32, F16, BF16], ids=["x_fp32", "x_fp16", "x_bf16"])
@pytest.mark.parametrize("W", [2, 3, 4])
def test_dtypes_and_options(W, xdt, wdt, bias, silu):
    _check_all(_inputs(3, 64, 300, W, xdt, wdt, seed=W, bias=bias), silu)


LS = [1, 2, 3, 7, 8, 33, 2048, 4099]
DIMS = [1, 5, 64, 1536]


@pytest.mark.parametrize("batch", [1, 16])
@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("L", LS)
@pytest.mark.parametrize("W", [2, 3, 4])
def test_shapes(W, L, dim, batch):
    """Every length (L < width - 1 included), channel count and batch; the x dtype rotates over the grid, SiLU and bias on."""
    xdt = [F32, BF16, F16][(LS.index(L) + DIMS.index(dim) + batch) % 3]
    _check_all(_inputs(batch, dim, L, W, xdt, F32, seed=L + dim + batch), True)


# ---- layouts ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("L", [64, 1000])
def test_xz_chunk_view_gives_the_dense_bits(L, dtype):
    """x as mamba passes it, xz.chunk(2, dim=1)[0] (batch stride 2 dim L), read in place: the bits of a dense copy."""
    t = _inputs(4, 48, L, 4, dtype, F32, seed=L)
    xz = torch.cat([t["x"], torch.randn_like(t["x"])], 1)
    x = xz.chunk(2, dim=1)[0]
    assert x.stride(0) == 2 * 48 * L
    got = _grads(t, True, x)
    want = _grads(t, True, x.contiguous())
    assert all(torch.equal(a, b) for a, b in zip(got, want))


@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("W", [2, 4])
def test_misaligned_x_takes_the_scalar_path_with_the_same_bits(W, dtype):
    t = _inputs(2, 24, 777, W, dtype, F32, seed=W)
    raw = torch.empty(t["x"].numel() + 1, dtype=dtype, device="cuda")
    x = raw[1:].view(t["x"].shape)
    x.copy_(t["x"])
    assert x.data_ptr() % 16 != 0
    got = _grads(t, True, x)
    want = _grads(t, True)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    _check(got[0], _ref_fwd(t["x"], t["w"], t["b"], True)[0], "out")


GUARD = 64
_PATTERN = {F32: (torch.int32, 0x7FC0BEEF), F16: (torch.int16, 0x7FDA), BF16: (torch.int16, 0x7FDA)}   # NaN in every dtype


class Buf:
    """rows x rs elements of `dtype` in a NaN-pattern buffer with GUARD elements on both sides; columns [0, cols) are the region
    the call reads or writes."""

    def __init__(self, rows, rs, cols, dtype, fill=None):
        it, self.pat = _PATTERN[dtype]
        self.raw = torch.full((2 * GUARD + rows * rs,), self.pat, dtype=it, device="cuda")
        self.body = self.raw.view(dtype)[GUARD:GUARD + rows * rs].view(rows, rs)
        self.view = self.body[:, :cols]
        if fill is not None:
            self.view.copy_(fill.reshape(rows, cols))
        self.keep = torch.ones(self.raw.numel(), dtype=torch.bool, device="cuda")
        self.keep[GUARD:GUARD + rows * rs].view(rows, rs)[:, :cols] = False

    def ptr(self):
        return ctypes.c_void_p(self.view.data_ptr())

    def check(self, what):
        assert not torch.isnan(self.view.float()).any(), f"{what}: elements left unwritten"
        assert bool((self.raw[self.keep] == self.pat).all()), f"{what}: written outside its region"


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("L,pad", [(37, 5), (512, 8), (2048, 0)])
@pytest.mark.parametrize("W", [2, 3, 4])
def test_c_abi_writes_exactly_its_region(W, L, pad, dtype):
    """x, out, dout and dx with padded row strides (pad = 8 keeps the 128-bit path for 16-bit io, 5 forces the scalar one)."""
    batch, dim = 3, 10
    t = _inputs(batch, dim, L, W, dtype, F32, seed=L + W)
    rs = L + pad
    x, dout = (Buf(batch * dim, rs, L, dtype, t[k]) for k in ("x", "dout"))
    out, dx = Buf(batch * dim, rs, L, dtype), Buf(batch * dim, rs, L, dtype)
    dw, db = Buf(1, dim * W, dim * W, F32), Buf(1, dim, dim, F32)
    d = _lib.Conv1dDesc()
    d.batch, d.dim, d.seqlen, d.width, d.io_dtype, d.silu = batch, dim, L, W, _DT[dtype], 1
    d.x_batch_stride = d.out_batch_stride = dim * rs
    d.x_dim_stride = d.out_dim_stride = rs
    wp, bp = ctypes.c_void_p(t["w"].data_ptr()), ctypes.c_void_p(t["b"].data_ptr())
    L_ = _lib.lib()
    assert L_.ss2d_conv1d_fwd(ctypes.byref(d), x.ptr(), wp, bp, out.ptr(), _stream()) == 0
    nws = L_.ss2d_conv1d_bwd_workspace_bytes(ctypes.byref(d))
    ws = torch.empty(max(nws, 4) // 4, device="cuda")
    assert L_.ss2d_conv1d_bwd(ctypes.byref(d), x.ptr(), wp, bp, dout.ptr(), dx.ptr(), dw.ptr(), db.ptr(),
                              ctypes.c_void_p(ws.data_ptr()), nws, _stream()) == 0
    torch.cuda.synchronize()
    for buf, what in ((out, "out"), (dx, "dx"), (dw, "dweight"), (db, "dbias")):
        buf.check(what)
    ref_out, _ = _ref_fwd(t["x"], t["w"], t["b"], True)
    ref_dx, ref_dw, ref_db = _ref_bwd(t["x"], t["w"], t["b"], t["dout"], True)
    _check(out.view.view(batch, dim, L), ref_out, "out")
    _check(dx.view.view(batch, dim, L), ref_dx, "dx")
    _check(dw.view.view(dim, W), ref_dw, "dweight", 5e-5)
    _check(db.view.view(dim), ref_db, "dbias", 5e-5)


def test_a_call_above_two_to_the_31_elements():
    """bf16 8 x 4096 x 65600 = 2.15e9 elements: rows at the start, the middle and the end (offsets past 2^31), and the weight
    gradient of the first and the last channel."""
    batch, dim, L, W = 8, 4096, 65600, 4
    assert batch * dim * L > 2 ** 31
    from ceigm_unet_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(batch, dim, L, device="cuda", dtype=BF16, generator=gen)
    dout = torch.randn(batch, dim, L, device="cuda", dtype=BF16, generator=gen)
    w, b = 0.5 * torch.randn(dim, W, device="cuda", generator=gen), torch.randn(dim, device="cuda", generator=gen)
    out = ops.conv1d_fwd(x, w, b, True)
    dx, dw, db = ops.conv1d_bwd(x, w, b, dout, True)
    for bi, di in ((0, 0), (0, 1), (4, 2048), (7, 4094), (7, 4095)):
        sl = (slice(bi, bi + 1), slice(di, di + 1))
        ro, _ = _ref_fwd(x[sl], w[di:di + 1], b[di:di + 1], True)
        rdx, _, _ = _ref_bwd(x[sl], w[di:di + 1], b[di:di + 1], dout[sl], True)
        _check(out[sl], ro, "out")
        _check(dx[sl], rdx, "dx")
    for di in (0, dim - 1):
        _, rdw, rdb = _ref_bwd(x[:, di:di + 1], w[di:di + 1], b[di:di + 1], dout[:, di:di + 1], True)
        _check(dw[di:di + 1], rdw, "dweight", 5e-5)
        _check(db[di:di + 1], rdb, "dbias", 5e-5)


# ---- bits -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [1, 64, 1536])          # 1 slab and several (the finalize pass)
def test_backward_is_bit_identical_and_graph_replay_matches(dim):
    from ceigm_unet_b200 import ops
    t = _inputs(4, dim, 1031, 4, BF16, F32, seed=dim)

    def run():
        out = ops.conv1d_fwd(t["x"], t["w"], t["b"], True)
        return (out,) + ops.conv1d_bwd(t["x"], t["w"], t["b"], t["dout"], True)

    first, second = run(), run()
    assert all(torch.equal(a, b) for a, b in zip(first, second))
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        captured = run()
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(first, captured))


# ---- update -----------------------------------------------------------------------------------------------------------
def _update(x, state, w, b, silu):
    import ceigm_unet_b200 as P
    with torch.no_grad():
        return P.causal_conv1d_update(x, state, w, b, "silu" if silu else None)


@pytest.mark.parametrize("silu", [False, True], ids=["noact", "silu"])
@pytest.mark.parametrize("dtype", [F32, F16, BF16], ids=["fp32", "fp16", "bf16"])
@pytest.mark.parametrize("batch", [1, 16, 256])
@pytest.mark.parametrize("W", [2, 3, 4])
def test_update_step(W, batch, dtype, silu):
    dim = 1536
    gen = torch.Generator(device="cuda").manual_seed(W + batch)
    state = torch.randn(batch, dim, W, device="cuda", generator=gen).to(dtype)
    x = torch.randn(batch, dim, device="cuda", generator=gen).to(dtype)
    w, b = torch.randn(dim, W, device="cuda", generator=gen), torch.randn(dim, device="cuda", generator=gen)
    new = torch.cat([state[..., 1:], x[..., None]], -1)
    ref = (new.double() * w.double()).sum(-1) + b.double()
    ref = F.silu(ref) if silu else ref
    s = state.clone()
    out = _update(x, s, w, b, silu)
    assert torch.equal(s, new)
    assert out.dtype == dtype and tuple(out.shape) == (batch, dim)
    _check(out, ref, "update_out")


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("L0", [1, 2, 2048])
@pytest.mark.parametrize("W", [2, 3, 4])
def test_prefill_then_updates_equal_one_forward(W, L0, dtype):
    """conv_state = F.pad(x[..., :L0], (W - L0, 0)) after the prefill, as mamba sets it; 16 steps then give the forward over
    L0 + 16 positions at positions L0 .. L0 + 15."""
    import ceigm_unet_b200 as P
    t = _inputs(3, 96, L0 + 16, W, dtype, F32, seed=L0 + W)
    full = P.causal_conv1d_fn(t["x"], t["w"], t["b"], activation="silu")
    state = F.pad(t["x"][..., :L0], (W - L0, 0)).contiguous()
    steps = torch.stack([_update(t["x"][..., L0 + i], state, t["w"], t["b"], True) for i in range(16)], -1)
    _check(steps, full[..., L0:], "prefill_steps")
    ref, _ = _ref_fwd(t["x"], t["w"], t["b"], True)
    _check(steps, ref[..., L0:], "prefill_steps_ref")


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
def test_graph_replay_of_a_32_step_update_loop_matches_the_eager_loop(dtype):
    W, batch, dim = 4, 16, 1536
    gen = torch.Generator(device="cuda").manual_seed(1)
    xs = torch.randn(32, batch, dim, device="cuda", generator=gen).to(dtype)
    s0 = torch.randn(batch, dim, W, device="cuda", generator=gen).to(dtype)
    w, b = torch.randn(dim, W, device="cuda", generator=gen), torch.randn(dim, device="cuda", generator=gen)

    def loop(state):
        return [_update(xs[i], state, w, b, True) for i in range(32)]

    eager_state = s0.clone()
    eager = loop(eager_state)
    state = s0.clone()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        loop(s0.clone())
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        captured = loop(state)
    for _ in range(2):
        state.copy_(s0)
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(eager, captured))
        assert torch.equal(state, eager_state)


# ---- a Mamba decode chain: conv1d + selective scan, prefill then steps ------------------------------------------------
def test_mamba_mixer_decode_chain_matches_one_full_pass():
    """in_proj -> causal conv1d + SiLU -> x_proj / dt_proj -> selective scan with the z gate -> out_proj (mamba_simple's
    layout, fixed random projections). A prefill of L0 positions (causal_conv1d_fn, selective_scan with the final state),
    then 16 tokens (causal_conv1d_update, selective_state_update), against one pass over L0 + 16 positions."""
    import ceigm_unet_b200 as P
    torch.manual_seed(0)
    batch, d_model, d_inner, N, R, W, L0, T = 2, 64, 128, 16, 8, 4, 100, 16
    dev = "cuda"
    in_w = torch.randn(2 * d_inner, d_model, device=dev) / d_model ** 0.5
    conv_w, conv_b = 0.5 * torch.randn(d_inner, W, device=dev), 0.1 * torch.randn(d_inner, device=dev)
    xproj_w = torch.randn(R + 2 * N, d_inner, device=dev) / d_inner ** 0.5
    dt_w, dt_b = torch.randn(d_inner, R, device=dev) / R ** 0.5, torch.rand(d_inner, device=dev) - 4.0
    A = -torch.arange(1, N + 1, device=dev, dtype=torch.float32).repeat(d_inner, 1)
    D = torch.ones(d_inner, device=dev)
    out_w = torch.randn(d_model, d_inner, device=dev) / d_inner ** 0.5
    hidden = torch.randn(batch, L0 + T, d_model, device=dev)

    def project(xc):                                     # xc (batch, d_inner, L) -> dt (batch, d_inner, L), B, C (batch, N, L)
        dbl = torch.einsum("rd,bdl->brl", xproj_w, xc)
        dt, B, C = dbl.split([R, N, N], 1)
        return torch.einsum("dr,brl->bdl", dt_w, dt), B.contiguous(), C.contiguous()

    with torch.no_grad():
        xz = torch.einsum("ed,bld->bel", in_w, hidden)
        x, z = xz.chunk(2, dim=1)
        xc = P.causal_conv1d_fn(x, conv_w, conv_b, activation="silu")
        dt, B, C = project(xc)
        y = P.selective_scan(xc, dt, A, B, C, D, dt_b, True, z=z.contiguous())
        ref = torch.einsum("md,bdl->bml", out_w, y)

        xc0 = P.causal_conv1d_fn(x[..., :L0], conv_w, conv_b, activation="silu")
        conv_state = F.pad(x[..., :L0], (W - L0, 0)).contiguous()
        dt0, B0, C0 = project(xc0)
        _, ssm_state = P.selective_scan(xc0, dt0, A, B0, C0, D, dt_b, True, return_last_state=True,
                                        z=z[..., :L0].contiguous())
        outs = []
        for i in range(T):
            l = L0 + i
            xt = P.causal_conv1d_update(x[..., l], conv_state, conv_w, conv_b, "silu")
            dtt, Bt, Ct = (v[..., 0] for v in project(xt[..., None]))
            yt = P.selective_state_update(ssm_state, xt, dtt.contiguous(), A, Bt.contiguous(), Ct.contiguous(), D,
                                          z[..., l].contiguous(), dt_b, True)
            outs.append(out_w @ yt.T)
        got = torch.stack(outs, -1).permute(1, 0, 2)
    _check(got, ref[..., L0:], "decode_chain", 1e-4)


# ---- drop-ins ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("silu", [False, True], ids=["noact", "silu"])
def test_dropin_extension_matches_the_function_and_fills_dx_in_place(silu, bias):
    from ceigm_unet_b200.dropin import causal_conv1d_cuda as ext
    t = _inputs(2, 32, 500, 4, BF16, F32, seed=3, bias=bias)
    out, dx, dw, db = _grads(t, silu)
    assert torch.equal(ext.causal_conv1d_fwd(t["x"], t["w"], t["b"], None, silu), out)
    dxz = torch.full((2, 64, 500), float("nan"), dtype=BF16, device="cuda")
    dx_ = dxz.chunk(2, dim=1)[0]                          # mamba_inner_fn passes a view of dxz
    res = ext.causal_conv1d_bwd(t["x"], t["w"], t["b"], t["dout"], None, dx_, silu)
    assert len(res) == 3 and res[0] is dx_
    assert torch.equal(dx_, dx) and torch.equal(res[1], dw)
    assert (res[2] is None) if not bias else torch.equal(res[2], db)
    assert torch.isnan(dxz[:, 32:].float()).all()        # the other half of dxz untouched
    res2 = ext.causal_conv1d_bwd(t["x"], t["w"], t["b"], t["dout"], None, None, silu)
    assert torch.equal(res2[0], dx)
