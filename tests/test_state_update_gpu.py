"""GPU tests of the recurrent step (csrc/state_update.cu; C ABI ss2d_state_update, Python `selective_state_update`).

Reference: a float64 restatement of the header's contract,
    t = dt + dt_bias (softplus, threshold 20, when asked),  h = exp(t A) h + t x B_g,  out = C_g . h + D x  (* silu(z)).
Tolerances, as max|got - ref| / max|ref| per tensor: fp32 out and the state 1e-5 per step; 1e-4 for the chained comparisons with
`selective_scan` (the bound of the state-passing chaining tests). 16-bit outputs are checked elementwise:
|got - ref| <= u |ref| + 1e-5 max|ref| with u = 2^-8 (bf16) or 2^-11 (fp16), i.e. correctly rounded up to fp32 noise. Each
test records the worst value per quantity in its user properties (written to the junit report).

The guard-band tests call the C ABI directly with strided rows: the state and out live inside NaN-filled buffers, and exactly the
documented region must be written. Also: chaining steps equals one `selective_scan` over the same positions (from an initial
state, and after a 3136-position prefill), identical bits across calls, and a CUDA-graph replay of a 32-step loop reproduces the
eager loop bit for bit."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from ceigm_unet_b200 import _lib

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
_DT = {F32: _lib.SS2D_F32, F16: _lib.SS2D_F16, BF16: _lib.SS2D_BF16}
ROUND = {BF16: 2.0 ** -8, F16: 2.0 ** -11}
NS = [1, 2, 4, 8, 12, 16, 17, 32, 40, 64, 256]

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
    ref = ref.double()
    err = (got.double() - ref).abs()
    scale = ref.abs().max().clamp_min(1e-30)
    if got.dtype in ROUND:
        ratio = float((err / (ROUND[got.dtype] * ref.abs() + 1e-5 * scale)).max())
        _note(what + "16_ratio", ratio)
        assert ratio <= 1.0, f"{what}: {got.dtype} error {ratio:.3g} x the rounding bound"
    else:
        rel = float(err.max() / scale)
        _note(what, rel)
        assert rel <= tol, f"{what}: rel err {rel:.3g} > {tol}"


def _inputs(batch, dim, N, G, dtype, seed, dt_range=(-1.0, 1.0)):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    u = lambda lo, hi, *s: lo + (hi - lo) * torch.rand(*s, device="cuda", generator=gen)
    return dict(state=r(batch, dim, N), x=r(batch, dim).to(dtype), dt=u(*dt_range, batch, dim).to(dtype), A=u(-1.0, -0.05, dim, N),
                B=r(batch, G, N).to(dtype), C=r(batch, G, N).to(dtype), D=r(dim), z=r(batch, dim).to(dtype),
                dt_bias=u(-0.5, 0.5, dim))


def _reference(t, softplus, use_D=True, use_z=True, use_bias=True):
    """float64 -> (out, new state)"""
    h, x, A = t["state"].double(), t["x"].double(), t["A"].double()
    dim, G = A.shape[0], t["B"].shape[1]
    grp = torch.arange(dim, device=A.device) // (dim // G)
    Bg, Cg = t["B"].double()[:, grp], t["C"].double()[:, grp]                 # (batch, dim, N)
    dt = t["dt"].double() + (t["dt_bias"].double() if use_bias else 0.0)
    if softplus:
        dt = F.softplus(dt, threshold=20)
    h = torch.exp(dt[..., None] * A) * h + (dt * x)[..., None] * Bg
    y = (Cg * h).sum(-1) + (t["D"].double() * x if use_D else 0.0)
    if use_z:
        y = y * F.silu(t["z"].double())
    return y, h


def _step(t, state, softplus, use_D=True, use_z=True, use_bias=True):
    import ceigm_unet_b200 as P
    with torch.no_grad():
        return P.selective_state_update(state, t["x"], t["dt"], t["A"], t["B"], t["C"], t["D"] if use_D else None,
                                        t["z"] if use_z else None, t["dt_bias"] if use_bias else None, softplus)


def _run_and_check(t, softplus, **opts):
    ref_out, ref_h = _reference(t, softplus, **opts)
    state = t["state"].clone()
    out = _step(t, state, softplus, **opts)
    assert out.dtype == t["x"].dtype and tuple(out.shape) == tuple(t["x"].shape)
    _check(out, ref_out, "out")
    _check(state, ref_h, "state")


# ---- coverage ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("G", [1, 2, 4])
@pytest.mark.parametrize("N", NS)
def test_parity(N, G, dtype):
    _run_and_check(_inputs(3, 24, N, G, dtype, seed=N * 10 + G), True)


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("N", [5, 16])
@pytest.mark.parametrize("softplus", [False, True], ids=["nosp", "sp"])
@pytest.mark.parametrize("use_z", [False, True], ids=["noz", "z"])
@pytest.mark.parametrize("use_bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("use_D", [False, True], ids=["noD", "D"])
def test_options(use_D, use_bias, use_z, softplus, N, dtype):
    _run_and_check(_inputs(2, 32, N, 2, dtype, seed=3), softplus, use_D=use_D, use_z=use_z, use_bias=use_bias)


@pytest.mark.parametrize("N", [1, 16, 64])
@pytest.mark.parametrize("softplus", [False, True], ids=["nosp", "sp"])
def test_dt_on_both_sides_of_the_softplus_threshold(N, softplus):
    """dt + dt_bias spread over [17, 23]; with A in [-0.05, -0.01] the decay exp(t A) stays far from 0 and 1."""
    t = _inputs(4, 64, N, 2, F32, seed=11, dt_range=(17.5, 22.5))
    t["A"] = -0.01 - 0.04 * torch.rand_like(t["A"])
    pre = t["dt"].double() + t["dt_bias"].double()
    assert (pre < 20).any() and (pre > 20).any()
    _run_and_check(t, softplus)


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("batch", [1, 256])
def test_mamba_layer_sizes(batch, dtype):
    _run_and_check(_inputs(batch, 1536, 16, 1, dtype, seed=batch), True)


def test_two_dimensional_B_and_C_mean_one_group():
    t = _inputs(4, 32, 16, 1, F32, seed=5)
    s1, s2 = t["state"].clone(), t["state"].clone()
    o1 = _step(t, s1, True)
    o2 = _step(dict(t, B=t["B"][:, 0], C=t["C"][:, 0]), s2, True)
    assert torch.equal(o1, o2) and torch.equal(s1, s2)


def test_strided_python_inputs_are_accepted():
    """x / dt / z as views with a row stride (mamba's xz.chunk) and B / C with a padded group stride give the dense result."""
    t = _inputs(4, 32, 16, 2, F32, seed=6)
    wide = {k: torch.cat([t[k], torch.zeros_like(t[k])], -1)[:, :32] for k in ("x", "dt", "z")}
    padded = {k: torch.cat([t[k], torch.zeros(4, 2, 3, device="cuda")], -1)[..., :16] for k in ("B", "C")}
    s1, s2 = t["state"].clone(), t["state"].clone()
    o1 = _step(t, s1, True)
    o2 = _step(dict(t, **wide, **padded), s2, True)
    assert torch.equal(o1, o2) and torch.equal(s1, s2)


def test_python_checks_on_cuda_tensors():
    import ceigm_unet_b200 as P
    t = _inputs(2, 16, 8, 2, F32, seed=7)
    a = [t[k] for k in ("state", "x", "dt", "A", "B", "C")]
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="contiguous and 16-byte aligned"):
            P.selective_state_update(t["state"].transpose(0, 1), *a[1:])
        with pytest.raises(RuntimeError, match="x's dtype"):
            P.selective_state_update(a[0], a[1], a[2].half(), *a[3:])
        with pytest.raises(RuntimeError, match="dim % n_groups"):
            P.selective_state_update(*a[:4], t["B"][:, :1].expand(2, 3, 8), t["C"][:, :1].expand(2, 3, 8))
        with pytest.raises(RuntimeError, match="float32 .dim, dstate."):
            P.selective_state_update(a[0], a[1], a[2], a[3].double(), *a[4:])


# ---- strided rows and guard bands (C ABI) -----------------------------------------------------------------------------
GUARD = 64      # elements on each side; 64 fp32 keep the state 16-byte aligned
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


@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("N", [1, 16, 17, 64])
def test_strided_rows_write_exactly_their_region(N, dtype):
    batch, dim, G = 3, 40, 4
    t = _inputs(batch, dim, N, G, dtype, seed=N)
    ref_out, ref_h = _reference(t, True)
    io_rs = dim + 7                                       # x, dt, z and out share a padded row stride
    x, dt, z = (Buf(batch, io_rs, dim, dtype, t[k]) for k in ("x", "dt", "z"))
    gs, bs = N + 3, G * (N + 3) + 5                       # B / C: padded group and batch strides
    Bb, Cb = (Buf(1, batch * bs, batch * bs, dtype, torch.zeros(batch * bs, dtype=dtype, device="cuda")) for _ in range(2))
    for buf, k in ((Bb, "B"), (Cb, "C")):
        for b in range(batch):
            buf.view[0, b * bs:b * bs + G * gs].view(G, gs)[:, :N] = t[k][b]
    state = Buf(1, batch * dim * N, batch * dim * N, F32, t["state"])
    out = Buf(batch, io_rs, dim, dtype)
    d = _lib.StepDesc()
    d.batch, d.dim, d.dstate, d.n_groups, d.io_dtype, d.dt_softplus = batch, dim, N, G, _DT[dtype], 1
    d.io_batch_stride = io_rs
    d.B_batch_stride = d.C_batch_stride = bs
    d.B_group_stride = d.C_group_stride = gs
    rc = _lib.lib().ss2d_state_update(ctypes.byref(d), state.ptr(), x.ptr(), dt.ptr(), ctypes.c_void_p(t["A"].data_ptr()), Bb.ptr(),
                                      Cb.ptr(), ctypes.c_void_p(t["D"].data_ptr()), ctypes.c_void_p(t["dt_bias"].data_ptr()), z.ptr(),
                                      out.ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    state.check("state")
    out.check("out")
    _check(out.view, ref_out, "out")
    _check(state.view.view(batch, dim, N), ref_h, "state")


# ---- chaining with selective_scan -------------------------------------------------------------------------------------
def _seq_inputs(batch, dim, L, N, G, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    return dict(u=r(batch, dim, L), delta=0.5 * torch.rand(batch, dim, L, device="cuda", generator=gen) - 1.0,
                A=-0.1 - 0.9 * torch.rand(dim, N, device="cuda", generator=gen), B=r(batch, G, N, L), C=r(batch, G, N, L),
                D=r(dim), z=r(batch, dim, L), delta_bias=0.5 * torch.rand(dim, device="cuda", generator=gen), h0=r(batch, dim, N))


def _scan(s, a, b, h0):
    import ceigm_unet_b200 as P
    with torch.no_grad():
        return P.selective_scan(s["u"][..., a:b], s["delta"][..., a:b], s["A"], s["B"][..., a:b], s["C"][..., a:b], s["D"],
                                s["delta_bias"], True, initial_state=h0, return_last_state=True, z=s["z"][..., a:b].contiguous())


def _steps(s, a, b, state):
    import ceigm_unet_b200 as P
    outs = []
    with torch.no_grad():
        for l in range(a, b):
            outs.append(P.selective_state_update(state, s["u"][..., l], s["delta"][..., l], s["A"], s["B"][..., l], s["C"][..., l],
                                                 s["D"], s["z"][..., l], s["delta_bias"], True))
    return torch.stack(outs, -1)


@pytest.mark.parametrize("G", [1, 4])
@pytest.mark.parametrize("N", [1, 16, 64])
def test_64_steps_match_one_scan_from_h0(N, G):
    s = _seq_inputs(2, 64, 64, N, G, seed=N + G)
    ref_out, ref_last = _scan(s, 0, 64, s["h0"])
    state = s["h0"].clone()
    out = _steps(s, 0, 64, state)
    _check(out, ref_out, "chain_out", 1e-4)
    _check(state, ref_last, "chain_state", 1e-4)


def test_prefill_then_steps_match_one_scan():
    """selective_scan over 3136 positions (a 56 x 56 map) hands its last state to 16 steps: the same as one scan over 3152."""
    L0, L = 3136, 3152
    s = _seq_inputs(2, 64, L, 16, 4, seed=21)
    ref_out, ref_last = _scan(s, 0, L, None)
    _, state = _scan(s, 0, L0, None)
    out = _steps(s, L0, L, state)
    _check(out, ref_out[..., L0:], "prefill_out", 1e-4)
    _check(state, ref_last, "prefill_state", 1e-4)


# ---- bits -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 16, 40])
def test_identical_calls_give_identical_bits(N):
    t = _inputs(64, 256, N, 4, F32, seed=4)
    s1, s2 = t["state"].clone(), t["state"].clone()
    o1, o2 = _step(t, s1, True), _step(t, s2, True)
    assert torch.equal(o1, o2) and torch.equal(s1, s2)


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
def test_graph_replay_of_a_32_step_loop_matches_the_eager_loop(dtype):
    s = _seq_inputs(4, 128, 32, 16, 2, seed=9)
    for k in ("u", "delta", "B", "C", "z"):
        s[k] = s[k].to(dtype)
    s = {k: (v.movedim(-1, 0).contiguous() if v.dim() >= 3 and k not in ("h0",) else v) for k, v in s.items()}   # position first

    def loop(state):
        import ceigm_unet_b200 as P
        with torch.no_grad():
            return [P.selective_state_update(state, s["u"][l], s["delta"][l], s["A"], s["B"][l], s["C"][l], s["D"], s["z"][l],
                                             s["delta_bias"], True) for l in range(32)]

    eager_state = s["h0"].clone()
    eager = loop(eager_state)
    state = s["h0"].clone()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        loop(s["h0"].clone())                           # warm-up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        captured = loop(state)
    for _ in range(2):
        state.copy_(s["h0"])
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(eager, captured))
        assert torch.equal(state, eager_state)
