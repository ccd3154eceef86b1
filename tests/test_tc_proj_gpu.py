"""Float64 parity of the tcgen05 projection kernels, called straight through the C ABI with torch-allocated buffers:
ss2d_linear_tc (csrc/linear_tc.cu: in_proj / out_proj) and ss2d_gate_proj_fwd (csrc/gate_proj_tc.cu: merge + LayerNorm + gate,
with or without out_proj).

References. Both kernels round fp32 operands to nearest TF32 in shared memory (the tensor core would truncate them), with ties
away from zero on the bit pattern: (bits + 0x1000) & 0xFFFFE000. The fp32 reference rounds both operands the same way on the
host and multiplies in float64, so what is left between kernel and reference is the tensor core's fp32 accumulation. For
gate_proj the A operand is the kernel's own gated tensor G (requested through g_out) rounded that way: the kernel's operand is
bit for bit that value, so the projection is checked independently of the LayerNorm; G and the statistics are checked on their
own against the float64 composition. bf16 operands are multiplied exactly; the output must be the correctly rounded bf16 of the
float64 result up to fp32 noise.

Bars. TAU is a normwise error, max|got - ref| / max|ref|. fp32: error <= TAU, and every fp32 case asserts that its bar can see
the TF32 rounding: the same product from truncated operands lies more than 10 TAU from the reference on that case's data.
bf16: |got - ref| <= ulp_bf16(ref) / 2 + TAU max|ref| elementwise. G and the statistics: G_TOL. Largest values seen on a B200
(power limit 1000 W): fp32 outputs 8.9e-7 (TAU = 1e-5 leaves a factor 11), bf16 outputs 0.996 of their bound, G 2.2e-6 and the
statistics 7.4e-7 (both with eps = 1e-2 and ys offset by 50), G of the C = 0 mode against ss2d_out_gate_fwd 2.0e-7, the autograd
wiring 2.9e-4; the product from truncated operands was never closer than 61 TAU. Each test records its worst values in its user
properties (written to the junit report).

Every output lives inside a buffer pre-filled with a NaN pattern and padded by guard bands: the documented region must be fully
written and everything else (guards, row-stride gaps) must keep its bits. Operands are column slices of wider matrices whose
other columns hold NaN, and A is followed by NaN rows: nothing past K or M may be read."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from ceigm_unet_b200 import _lib, ops

pytestmark = pytest.mark.gpu

F32, BF16 = torch.float32, torch.bfloat16
_DT = {F32: _lib.SS2D_F32, BF16: _lib.SS2D_BF16}
TAU = 1e-5
G_TOL = 1e-5
ROUTES_TOL = 1e-6
N_SM = 148

_observed = {}


@pytest.fixture(autouse=True)
def _record_errors(request):
    _observed.clear()
    yield
    request.node.user_properties.extend(sorted(_observed.items()))


def _note(key, v, worst=max):
    _observed[key] = worst(_observed.get(key, v), v)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


# ---- TF32 rounding, as the kernels do it --------------------------------------------------------------------------------
def rna(t):
    """Round fp32 to nearest TF32, ties away from zero, on the bit pattern."""
    b = t.float().contiguous().view(torch.int32)
    return ((b + 0x1000) & -8192).view(torch.float32)


def trunc(t):
    """What the tensor core makes of an fp32 container: the 13 low mantissa bits dropped."""
    return (t.float().contiguous().view(torch.int32) & -8192).view(torch.float32)


def _normwise(got, ref):
    ref = ref.double()
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def check_f32(got, ref, ref_trunc, what):
    """got: the kernel's fp32 output; ref / ref_trunc: float64 results from rounded / truncated operands."""
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite output"
    err = _normwise(got, ref)
    _note("f32", err)
    assert err <= TAU, f"{what}: normwise error {err:.3g} > {TAU}"
    sep = _normwise(ref_trunc, ref)
    _note("trunc_sep_over_tau", sep / TAU, min)
    assert sep > 10 * TAU, f"{what}: the bar cannot see the TF32 rounding on this data ({sep:.3g})"


def half_ulp_bf16(ref):
    """Half an ulp of bf16 (8 significant bits) at each element of the float64 tensor ref."""
    _, e = torch.frexp(ref)
    return torch.ldexp(torch.ones_like(ref), e - 9)


def check_bf16(got, ref, what):
    ref = ref.double()
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite output"
    bound = half_ulp_bf16(ref) + TAU * ref.abs().max()
    ratio = float(((got.double() - ref).abs() / bound).max())
    _note("bf16_ratio", ratio)
    assert ratio <= 1.0, f"{what}: bf16 error {ratio:.3g} x (half an ulp + TAU max|ref|)"


def check_out(got, ref_fn, a, w, dtype, what):
    """ref_fn(a, w) -> float64 result from the operands as the tensor core sees them."""
    if dtype == F32:
        check_f32(got, ref_fn(rna(a), rna(w)), ref_fn(trunc(a), trunc(w)), what)
    else:
        check_bf16(got, ref_fn(a, w), what)


# ---- buffers ------------------------------------------------------------------------------------------------------------
_PATTERN = {F32: (torch.int32, 0x7FC0BEEF), BF16: (torch.int16, 0x7FDA)}   # NaN in either dtype
GUARD = 64


class Buf:
    """`rows` rows of `rs` elements inside a buffer pre-filled with a NaN pattern and padded by GUARD elements on both sides.
    ranges: the column ranges [c0, c1) the call is documented to write (or, for operands, that hold the operand)."""

    def __init__(self, rows, rs, ranges, dtype):
        it, self.pat = _PATTERN[dtype]
        self.raw = torch.full((2 * GUARD + rows * rs,), self.pat, dtype=it, device="cuda")
        self.body = self.raw.view(dtype)[GUARD:GUARD + rows * rs].view(rows, rs)
        self.rs, self.ranges, self.rows = rs, ranges, rows

    def cols(self, c0, n, rows=None):
        return self.body[:rows, c0:c0 + n]

    def ptr(self):
        return ctypes.c_void_p(self.body[:, self.ranges[0][0]].data_ptr())

    def check(self, what, rows=None):
        rows = self.rows if rows is None else rows
        keep = torch.ones(self.raw.numel(), dtype=torch.bool, device="cuda")
        for c0, c1 in self.ranges:
            assert not torch.isnan(self.body[:rows, c0:c1].float()).any(), f"{what}: elements left unwritten"
            keep[GUARD:GUARD + self.rows * self.rs].view(self.rows, self.rs)[:rows, c0:c1] = False
        assert bool((self.raw[keep] == self.pat).all()), f"{what}: written outside its region"


def operand(rows, cols, values, dtype, pad_rows=0):
    """`values` (rows, cols) as a column slice of a wider NaN matrix (16 bytes of NaN on either side of each row), followed by
    pad_rows NaN rows."""
    step = 16 // (4 if dtype == F32 else 2)
    b = Buf(rows + pad_rows, cols + 2 * step, [(step, step + cols)], dtype)
    b.cols(step, cols, rows).copy_(values.to(dtype))
    return b


def _bits_equal(a, b):
    return torch.equal(a.raw, b.raw)


# ---- ss2d_linear_tc -----------------------------------------------------------------------------------------------------
class LinearCase:
    """out = A W^T + bias on M rows, cut into parts (n_cols, planes_L or 0 for rows, act). Operands in NaN-padded slices,
    outputs in NaN-filled buffers; row-major parts get ld = n_cols + 16 bytes' worth of elements."""

    def __init__(self, M, K, parts, dtype, *, bias=True, seed=0, a=None, w=None):
        self.M, self.K, self.parts, self.dtype = M, K, parts, dtype
        self.N = sum(p[0] for p in parts)
        g = torch.Generator(device="cuda").manual_seed(seed)
        a = torch.randn(M, K, device="cuda", generator=g) if a is None else a
        w = torch.randn(self.N, K, device="cuda", generator=g) / K ** 0.5 if w is None else w
        self.a = a.to(dtype).float()
        self.w = w.to(dtype).float()
        # a bias that differs per column (and from part to part), so that indexing it by the part's column fails
        self.bias = (0.5 * torch.randn(self.N, device="cuda", generator=g) + torch.linspace(-1, 1, self.N, device="cuda")) if bias else None
        self.A = operand(M, K, self.a, dtype, pad_rows=130)
        self.W = operand(self.N, K, self.w, dtype)
        self.step = 16 // (4 if dtype == F32 else 2)

    def _outputs(self):
        outs = []
        for n, L, act in self.parts:
            if L:
                outs.append(Buf(self.M // L, n * L, [(0, n * L)], self.dtype))
            else:
                outs.append(Buf(self.M, n + self.step, [(0, n)], self.dtype))
        return outs

    def launch(self):
        outs = self._outputs()
        arr = (_lib.LinearPart * len(self.parts))()
        for i, ((n, L, act), o) in enumerate(zip(self.parts, outs)):
            arr[i].out, arr[i].ld, arr[i].n_cols, arr[i].planes_L, arr[i].act = o.ptr().value, 0 if L else o.rs, n, L, act
        rc = _lib.lib().ss2d_linear_tc(self.A.ptr(), self.A.rs, self.W.ptr(), self.W.rs, _p(self.bias), self.M, self.N, self.K,
                                       _DT[self.dtype], len(self.parts), arr, _stream())
        assert rc == 0, rc
        return outs

    def reference(self, a, w):
        """float64 results per part, each (M, n_cols) row-major."""
        full = a.double() @ w.double().t()
        if self.bias is not None:
            full = full + self.bias.double()
        res, n0 = [], 0
        for n, L, act in self.parts:
            r = full[:, n0:n0 + n]
            res.append(F.silu(r) if act else r)
            n0 += n
        return res

    def got(self, outs):
        """The kernel's parts as (M, n_cols) views."""
        res = []
        for (n, L, act), o in zip(self.parts, outs):
            res.append(o.body.view(self.M // L, n, L).transpose(1, 2).reshape(self.M, n) if L else o.cols(0, n))
        return res

    def run_and_check(self, what=""):
        outs = self.launch()
        torch.cuda.synchronize()
        for i, o in enumerate(outs):
            o.check(f"{what} part {i}")
        got = self.got(outs)
        for i, gp in enumerate(got):
            check_out(gp, lambda a, w: self.reference(a, w)[i], self.a, self.w, self.dtype, f"{what} part {i}")
        return outs, got


@pytest.mark.parametrize("dtype,K", [(F32, 4), (F32, 12), (F32, 36), (F32, 100), (F32, 160),
                                     (BF16, 8), (BF16, 72), (BF16, 200), (BF16, "max")])
def test_linear_k_tails(dtype, K):
    """K ends inside a 128-byte block (the TMA zero-fills the rest of it), and K at the shared-memory limit of a 256-wide part."""
    if K == "max":
        K = max(k for k in range(8, 4096, 8) if ops.linear_tc_supported(256, k, dtype))
        assert K == 320
    N = 256 if K in (160, 320) else 48
    LinearCase(129, K, [(N, 0, 0)], dtype, seed=K).run_and_check(f"K = {K}")


@pytest.mark.parametrize("n", [16, 48, 240, 256])
@pytest.mark.parametrize("M", [1, 127, 128, 129])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_part_widths_and_row_counts(n, M, dtype):
    """16-column chunk tails (48, 240), both extremes of the width, and M around one 128-row tile."""
    LinearCase(M, 36 if dtype == F32 else 72, [(n, 0, 0)], dtype, seed=n + M).run_and_check(f"n = {n}, M = {M}")


@pytest.mark.parametrize("K,N", [(160, 256), (64, 64)], ids=["K160_N256", "K64_N64"])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_many_tiles_per_cta(K, N, dtype):
    """5 x 148 full tiles + a 77-row tail: every CTA runs 5 or 6 tiles, so the A ring wraps many times and both accumulator
    stages are reused. fp32 K = 160, N = 256 leaves room for 2 ring stages, K = 64, N = 64 for 8."""
    M = 5 * N_SM * 128 + 77
    LinearCase(M, K, [(N, 0, 0)], dtype, seed=K).run_and_check(f"M = {M}")


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_north_star_in_proj_and_out_proj(dtype):
    """in_proj of SS2D(d_model = 96) at B = 24, 56 x 56: 96 -> planes of 192 channels + rows of 192 (the gate); out_proj 192 -> 96."""
    M, L = 24 * 3136, 3136
    LinearCase(M, 96, [(192, L, 0), (192, 0, 0)], dtype, seed=1).run_and_check("in_proj")
    LinearCase(M, 192, [(96, 0, 0)], dtype, seed=2).run_and_check("out_proj")


@pytest.mark.parametrize("parts", [
    [(64, 0, 1), (32, 49, 0), (16, 0, 0)],
    [(32, 49, 0), (48, 0, 1), (16, 49, 1), (64, 0, 0)],
    [(16, 0, 0), (16, 49, 1), (16, 0, 1), (256, 49, 0)],
], ids=["3_parts", "4_parts", "4_parts_wide_last"])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_three_and_four_parts(parts, dtype):
    """Planes, rows, rows + SiLU and planes + SiLU in one call, with a per-column bias: part i must read bias[n0_i + c]."""
    LinearCase(49 * 7, 64, parts, dtype, seed=len(parts)).run_and_check()


@pytest.mark.parametrize("L,Bn", [(1, 300), (49, 5), (130, 3), (3136, 2)])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_planes_lengths(L, Bn, dtype):
    """Channel-major planes whose image boundaries fall anywhere inside a 128-row tile (L = 1, 49, 130) or span many tiles."""
    LinearCase(L * Bn, 32, [(48, L, 0), (32, 0, 0)], dtype, seed=L).run_and_check(f"L = {L}")


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_silu_at_large_accumulators(dtype):
    """Accumulators from -200 to 200: SiLU must stay finite, vanish for large negative and pass large positive values."""
    M, K, N = 256, 64, 32
    g = torch.Generator(device="cuda").manual_seed(9)
    s = torch.linspace(-1, 1, M, device="cuda")[:, None]
    a = s * (torch.rand(M, K, device="cuda", generator=g) + 0.5)
    w = torch.rand(2 * N, K, device="cuda", generator=g) + 0.5
    acc = a @ w.t()
    a = a * (200 / acc.abs().max())
    case = LinearCase(M, K, [(N, 0, 1), (N, 32, 1)], dtype, bias=False, a=a, w=w)
    _, got = case.run_and_check()
    # the accumulators from the operands as the tensor core sees them; beyond +30 SiLU(x) = x to fp32 precision, so the output
    # is the accumulator up to the accumulation error and, in bf16, the output's rounding (half an ulp)
    a_op, w_op = (rna(case.a), rna(case.w)) if dtype == F32 else (case.a, case.w)
    pre = a_op.double() @ w_op.double().t()
    assert float(pre.min()) < -150 and float(pre.max()) > 150
    for i, gp in enumerate(got):
        pp = pre[:, i * N:(i + 1) * N]
        big = pp > 30
        bound = TAU * pp.abs().max() + (half_ulp_bf16(pp[big]) if dtype == BF16 else 0.0)
        assert bool((gp.double()[pp < -30].abs() <= 1e-6).all())
        assert bool(((gp.double() - pp)[big].abs() <= bound).all())


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_linear_repeatable_and_graph_replay(dtype):
    """Three tiles per CTA, planes + rows + SiLU: two calls and a CUDA-graph replay write the same bits."""
    case = LinearCase(18 * 3136, 96, [(192, 3136, 0), (64, 0, 1)], dtype, seed=4)
    first = case.launch()
    again = case.launch()
    torch.cuda.synchronize()
    for x, y in zip(first, again):
        assert _bits_equal(x, y)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = case.launch()
    for b in captured:
        b.raw.fill_(b.pat)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(first, captured):
        assert _bits_equal(x, y)


def _autograd_ref(fn, inputs):
    ins = [t.detach().double().requires_grad_() for t in inputs]
    outs = fn(*ins)
    return ins, outs


def test_functional_in_proj_planes_and_linear_wiring(monkeypatch):
    """functional.in_proj_planes / linear_tc with a bias and TF32 allowed: forward and dx, dW, db against float64 autograd of
    F.linear (+ chunk / permute). This checks which half of W and which slice of the bias feed xi and z. The backward runs on
    library GEMMs under TF32, hence the normwise bar of 1e-3."""
    from ceigm_unet_b200 import functional as Fn
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", True)
    g = torch.Generator(device="cuda").manual_seed(12)
    Bn, H, Wd, C, D = 2, 14, 10, 96, 192
    x = torch.randn(Bn, H, Wd, C, device="cuda", generator=g, requires_grad=True)
    W = (torch.randn(2 * D, C, device="cuda", generator=g) / C ** 0.5).requires_grad_()
    b = torch.randn(2 * D, device="cuda", generator=g).requires_grad_()
    launches = _lib.launch_count()
    res = Fn.in_proj_planes(x, W, b)
    assert res is not None and _lib.launch_count() > launches
    xi, z = res
    dxi, dz = torch.randn_like(xi), torch.randn_like(z)
    torch.autograd.backward([xi, z], [dxi, dz])

    def ref(x, W, b):
        xz = F.linear(x, W, b)
        xr, zr = xz.chunk(2, dim=-1)
        return xr.permute(0, 3, 1, 2), zr
    ins, (rxi, rz) = _autograd_ref(ref, [x, W, b])
    torch.autograd.backward([rxi, rz], [dxi.double(), dz.double()])
    for got, want, name in ((xi, rxi, "xi"), (z, rz, "z"), (x.grad, ins[0].grad, "dx"), (W.grad, ins[1].grad, "dW"),
                            (b.grad, ins[2].grad, "db")):
        err = _normwise(got.detach(), want.detach())
        _note("functional", err)
        assert err <= 1e-3, (name, err)

    y = torch.randn(Bn, H, Wd, D, device="cuda", generator=g, requires_grad=True)
    Wo = (torch.randn(C, D, device="cuda", generator=g) / D ** 0.5).requires_grad_()
    bo = torch.randn(C, device="cuda", generator=g).requires_grad_()
    launches = _lib.launch_count()
    out = Fn.linear_tc(y, Wo, bo)
    assert _lib.launch_count() > launches
    dout = torch.randn_like(out)
    out.backward(dout)
    ins, rout = _autograd_ref(F.linear, [y, Wo, bo])
    rout.backward(dout.double())
    for got, want, name in ((out, rout, "out"), (y.grad, ins[0].grad, "dy"), (Wo.grad, ins[1].grad, "dW"), (bo.grad, ins[2].grad, "db")):
        err = _normwise(got.detach(), want.detach())
        _note("functional", err)
        assert err <= 1e-3, (name, err)


# ---- ss2d_gate_proj_fwd -------------------------------------------------------------------------------------------------
def _merge_ref(ys, tmask, H, W):
    Bn, K, D, L = ys.shape
    y = 0
    for k in range(K):
        p = ys[:, k].double()
        if (tmask >> k) & 1:
            p = p.view(Bn, D, W, H).transpose(2, 3).reshape(Bn, D, L)
        y = y + p
    return y


class GateCase:
    """One ss2d_gate_proj_fwd call with its float64 reference. z, out and g live in NaN-filled row buffers; `pad` gives their
    rows 32 extra bytes and starts the data 16 bytes in."""

    def __init__(self, Bn, K, D, H, W, C, dtype, *, tmask=0b1010, z=True, z_act=1, affine="wb", bias=True, stats=True,
                 g_out=True, pad=False, eps=1e-5, offset=0.0, seed=0):
        self.Bn, self.K, self.D, self.H, self.W, self.C, self.dtype = Bn, K, D, H, W, C, dtype
        self.L = L = H * W
        self.tmask, self.z_act, self.eps, self.want_stats, self.want_g = tmask & ((1 << K) - 1), z_act, eps, stats, g_out
        g = torch.Generator(device="cuda").manual_seed(seed)
        self.ys = torch.randn(Bn, K, D, L, device="cuda", generator=g) + offset
        self.lnw = 1.0 + 0.5 * torch.randn(D, device="cuda", generator=g) if "w" in affine else None
        self.lnb = 0.5 * torch.randn(D, device="cuda", generator=g) if "b" in affine else None
        self.step = step = 16 // (4 if dtype == F32 else 2)
        self.c0 = step if pad else 0
        extra = 2 * step if pad else 0
        self.zb = None
        if z:
            self.zb = Buf(Bn * L, D + extra, [(self.c0, self.c0 + D)], dtype)
            self.zb.cols(self.c0, D).copy_(torch.randn(Bn * L, D, device="cuda", generator=g).to(dtype))
        self.w = (torch.randn(C, D, device="cuda", generator=g) / D ** 0.5).to(dtype).float() if C else None
        self.Wb = operand(C, D, self.w, dtype) if C else None
        self.bias = (0.5 * torch.randn(C, device="cuda", generator=g) + torch.linspace(-1, 1, C, device="cuda")) if C and bias else None
        self.out_rs = C + extra
        self.g_rs = D + extra

    def launch(self):
        Bn, L, D, C = self.Bn, self.L, self.D, self.C
        out = Buf(Bn * L, self.out_rs, [(self.c0, self.c0 + C)], self.dtype) if C else None
        gb = Buf(Bn * L, self.g_rs, [(self.c0, self.c0 + D)], self.dtype) if self.want_g else None
        st = Buf(Bn * L, 2, [(0, 2)], F32) if self.want_stats else None
        rc = _lib.lib().ss2d_gate_proj_fwd(
            _p(self.ys), self.K, ctypes.c_uint32(self.tmask), _p(self.lnw), _p(self.lnb), ctypes.c_float(self.eps),
            self.zb.ptr() if self.zb else None, self.zb.rs if self.zb else 0, self.z_act, self.Wb.ptr() if C else None,
            self.Wb.rs if C else 0, _p(self.bias), out.ptr() if out else None, self.out_rs, gb.ptr() if gb else None, self.g_rs,
            st.ptr() if st else None, Bn, D, L, self.H, self.W, C, _DT[self.dtype], _stream())
        assert rc == 0, rc
        return out, gb, st

    def reference_g(self):
        """float64 G (B L, D), mean and rstd (B L)."""
        Bn, D, L = self.Bn, self.D, self.L
        yt = _merge_ref(self.ys, self.tmask, self.H, self.W).transpose(1, 2).reshape(Bn * L, D)
        mean = yt.mean(-1)
        rstd = 1.0 / torch.sqrt(((yt - mean[:, None]) ** 2).mean(-1) + self.eps)
        g = (yt - mean[:, None]) * rstd[:, None]
        if self.lnw is not None:
            g = g * self.lnw.double()
        if self.lnb is not None:
            g = g + self.lnb.double()
        if self.zb is not None:
            z = self.zb.cols(self.c0, D).double()
            g = g * (F.silu(z) if self.z_act else z)
        return g, mean, rstd

    def projection_ref(self, a, w):
        r = a.double() @ w.double().t()
        return r if self.bias is None else r + self.bias.double()

    def run_and_check(self, what=""):
        out, gb, st = self.launch()
        torch.cuda.synchronize()
        for b, name in ((out, "out"), (gb, "g"), (st, "mean_rstd")):
            if b is not None:
                b.check(f"{what} {name}")
        g_ref, mean, rstd = self.reference_g()
        if gb is not None:
            g = gb.cols(self.c0, self.D)
            if self.dtype == F32:
                err = _normwise(g, g_ref)
                _note("g", err)
                assert err <= G_TOL, f"{what} G: {err:.3g}"
            else:
                ratio = float(((g.double() - g_ref).abs() / (2.0 ** -8 * g_ref.abs() + G_TOL * g_ref.abs().max())).max())
                _note("g16_ratio", ratio)
                assert ratio <= 1.0, f"{what} G: {ratio:.3g} x the bf16 rounding bound"
        if st is not None:
            for got, want, name in ((st.body[:, 0], mean, "mean"), (st.body[:, 1], rstd, "rstd")):
                err = _normwise(got, want)
                _note("stats", err)
                assert err <= G_TOL, f"{what} {name}: {err:.3g}"
        if out is not None and gb is not None:
            a = gb.cols(self.c0, self.D).float()
            check_out(out.cols(self.c0, self.C), self.projection_ref, a, self.w, self.dtype, f"{what} out")
        return out, gb, st


def _admitted():
    return [(D, C, dt) for dt in (F32, BF16) for D in (64, 128, 192, 256) for C in range(0, 257, 16)
            if ops.gate_proj_supported(D, C, 2, dt)]


def test_gate_admitted_shapes_table():
    adm = _admitted()
    assert len(adm) == 85 and sum(dt == F32 for _, _, dt in adm) == 43


@pytest.mark.parametrize("D", [64, 128, 192, 256])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_every_admitted_width(D, dtype):
    """Every C the predicate admits at this (D, dtype), on a ragged 12 x 20 image with K = 2."""
    Cs = [C for d, C, dt in _admitted() if d == D and dt == dtype]
    for C in Cs:
        GateCase(1, 2, D, 12, 20, C, dtype, tmask=0b10, seed=D + C).run_and_check(f"D = {D}, C = {C}")


@pytest.mark.parametrize("shape", [(24, 4, 192, 56, 56, 0), (24, 4, 192, 56, 56, 96), (16, 4, 64, 64, 64, 64)], ids=str)
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_many_tiles_per_cta(shape, dtype):
    """672 (24 x 56 x 56) or 512 tiles over at most 148 CTAs: every CTA reloads the weight over the plane ring, waits on
    `afree` and reuses both pixel tables. The first shape is the production ops.out_gate_fwd call."""
    Bn, K, D, H, W, C = shape
    if not ops.gate_proj_supported(D, C, K, dtype):
        pytest.skip("not admitted")
    case = GateCase(Bn, K, D, H, W, C, dtype, seed=C + 1)
    _, gb, st = case.run_and_check(str(shape))
    if C == 0 and dtype == F32:
        # the C = 0 mode and ss2d_out_gate_fwd agree
        L = H * W
        out_d, st_d = Buf(Bn * L, D, [(0, D)], F32), Buf(Bn * L, 2, [(0, 2)], F32)
        rc = _lib.lib().ss2d_out_gate_fwd(_p(case.ys), K, _p(case.lnw), _p(case.lnb), case.zb.ptr(), case.zb.rs, 1, out_d.ptr(),
                                          st_d.ptr(), Bn, D, L, ctypes.c_float(case.eps), _lib.SS2D_F32, _lib.SS2D_F32, H, W,
                                          ctypes.c_uint32(case.tmask), _stream())
        assert rc == 0, rc
        torch.cuda.synchronize()
        for a, b in ((gb.cols(0, D), out_d.body), (st.body, st_d.body)):
            rel = _normwise(a, b)
            _note("routes", rel)
            assert rel <= ROUTES_TOL, rel


def _masks(K):
    alt = int("10" * 4, 2) & ((1 << K) - 1)
    return {"natural": 0, "transposed": (1 << K) - 1, "alternating": alt}


@pytest.mark.parametrize("K", range(1, 9))
@pytest.mark.parametrize("mask", ["natural", "transposed", "alternating"])
def test_gate_direction_counts_and_masks(K, mask):
    dtype = F32 if K % 2 else BF16
    GateCase(2, K, 64, 8, 20, 32, dtype, tmask=_masks(K)[mask], seed=K).run_and_check(f"K = {K}")


@pytest.mark.parametrize("C", [0, 32])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_eight_directions_at_the_widest_d(C, dtype):
    """K = 8 at the largest D the predicate admits for this C and dtype."""
    Ds = [D for D in (64, 128, 192, 256) if ops.gate_proj_supported(D, C, 8, dtype)]
    D = max(Ds)
    GateCase(1, 8, D, 12, 20, C, dtype, tmask=0b10110100, seed=D).run_and_check(f"D = {D}")


@pytest.mark.parametrize("H,W", [(4, 4), (4, 12), (8, 36), (36, 4), (12, 20), (20, 8), (36, 36), (4, 36)])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_image_sizes(H, W, dtype):
    """Non-square images, partial tiles at both edges, and a single partial tile (H < 8, W < 16)."""
    GateCase(2, 4, 128, H, W, 48, dtype, seed=H * 64 + W).run_and_check(f"{H} x {W}")


OPTIONS = {
    "no_z": dict(z=False),
    "z_linear": dict(z_act=0),
    "no_affine": dict(affine=""),
    "weight_only": dict(affine="w"),
    "no_bias": dict(bias=False),
    "no_stats": dict(stats=False),
    "padded_rows": dict(pad=True),
    "eps_and_offset": dict(eps=1e-2, offset=50.0, K=2),
}


@pytest.mark.parametrize("opt", list(OPTIONS))
@pytest.mark.parametrize("C", [0, 64])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_options(opt, C, dtype):
    kw = dict(OPTIONS[opt])
    K = kw.pop("K", 4)
    if C == 0 and opt == "no_bias":
        pytest.skip("C = 0 has no bias")
    GateCase(2, K, 64, 12, 20, C, dtype, seed=len(opt), **kw).run_and_check(opt)


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_out_does_not_depend_on_g_out(dtype):
    """The kernel with and without the G output (two instantiations) writes the same bits to out, and to the statistics."""
    case = GateCase(3, 4, 192, 24, 20, 96, dtype, seed=5)
    out1, _, st1 = case.run_and_check()
    case.want_g = False
    out2, gb2, st2 = case.launch()
    torch.cuda.synchronize()
    assert gb2 is None
    out2.check("out without g")
    assert _bits_equal(out1, out2) and _bits_equal(st1, st2)


@pytest.mark.parametrize("C", [0, 96])
@pytest.mark.parametrize("dtype", [F32, BF16])
def test_gate_repeatable_and_graph_replay(C, dtype):
    case = GateCase(4, 4, 192, 56, 56, C, dtype, seed=7)
    first = case.launch()
    again = case.launch()
    torch.cuda.synchronize()
    for x, y in zip(first, again):
        if x is not None:
            assert _bits_equal(x, y)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = case.launch()
    for b in captured:
        if b is not None:
            b.raw.fill_(b.pat)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(first, captured):
        if x is not None:
            assert _bits_equal(x, y)
