"""GPU parity of the fused SS2D epilogue kernels (csrc/epilogue.cu; C ABI ss2d_out_gate_fwd / _bwd and ss2d_group_gate_fwd /
_bwd): merge over the K planes (transposed ones un-transposed) + (B, D, L) -> (B, L, D) + LayerNorm(D) + SiLU(z) gate, and its
backward, against a float64 torch composition of the contract in include/ss2d_b200.h, with gradients from autograd.

The calls go straight to the C ABI with torch-allocated buffers, so that strides, column offsets, NULL outputs and the kernel
that `ops.out_gate_fwd` would not pick can be chosen. Every output lives inside a buffer pre-filled with a NaN pattern and
padded by guard bands: the documented region must be fully written (no NaN left) and nothing else may change (the pattern
stays bit-identical in the guards, in row-stride gaps and in columns that belong to no group).

Tolerances, as max|got - ref| / max|ref| per tensor: fp32 out and statistics 1e-5, dy 5e-6, dz and the LayerNorm gradients
5e-5. The largest values seen on a B200 are out 8.3e-6 and stats 1.3e-6 (both with inputs offset by 50), dy 7.9e-7, dz 6.0e-6
and dln 8.1e-6. 16-bit outputs are checked elementwise: |got - ref| <= u |ref| + 1e-5 max|ref| with u = 2^-8 (bf16) or 2^-11
(fp16), i.e. correctly rounded up to fp32 noise (worst seen: 0.98 of that bound). Each test records the worst value per tensor
family in its user properties (written to the junit report)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from ceigm_unet_b200 import _lib, ops

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
_DT = {F32: _lib.SS2D_F32, F16: _lib.SS2D_F16, BF16: _lib.SS2D_BF16}
TOL = {"out": 1e-5, "stats": 1e-5, "dy": 5e-6, "dz": 5e-5, "dln": 5e-5}
ROUND = {BF16: 2.0 ** -8, F16: 2.0 ** -11}
ERR_UNSUPPORTED = -8

_observed = {}


@pytest.fixture(autouse=True)
def _record_errors(request):
    _observed.clear()
    yield
    request.node.user_properties.extend(sorted(_observed.items()))


def _note(key, v):
    _observed[key] = max(_observed.get(key, 0.0), v)


def _check(got, ref, family, what=""):
    """fp32: max error relative to max|ref|; 16-bit: the elementwise rounding bound."""
    ref = ref.double()
    err = (got.double() - ref).abs()
    scale = ref.abs().max().clamp_min(1e-30)
    if got.dtype in ROUND:
        ratio = float((err / (ROUND[got.dtype] * ref.abs() + 1e-5 * scale)).max())
        _note(family + "16_ratio", ratio)
        assert ratio <= 1.0, f"{family}{what}: {got.dtype} error {ratio:.3g} x the rounding bound"
    else:
        rel = float(err.max() / scale)
        _note(family, rel)
        assert rel <= TOL[family], f"{family}{what}: rel err {rel:.3g} > {TOL[family]}"


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


_PATTERN = {F32: (torch.int32, 0x7FC0BEEF), F16: (torch.int16, 0x7FDA), BF16: (torch.int16, 0x7FDA)}   # NaN in every dtype
GUARD = 64


class Buf:
    """`rows` rows of `rs` elements of `dtype` inside a buffer pre-filled with a NaN pattern and padded by GUARD elements on both
    sides. `ranges`: the column ranges [c0, c1) the call is documented to write (or, for inputs, that hold the operand)."""

    def __init__(self, rows, rs, ranges, dtype):
        it, self.pat = _PATTERN[dtype]
        self.raw = torch.full((2 * GUARD + rows * rs,), self.pat, dtype=it, device="cuda")
        self.body = self.raw.view(dtype)[GUARD:GUARD + rows * rs].view(rows, rs)
        self.rs, self.ranges = rs, ranges
        self.keep = torch.ones(self.raw.numel(), dtype=torch.bool, device="cuda")
        for c0, c1 in ranges:
            self.keep[GUARD:GUARD + rows * rs].view(rows, rs)[:, c0:c1] = False

    def cols(self, c0, n):
        return self.body[:, c0:c0 + n]

    def ptr(self, c0=None):
        return ctypes.c_void_p(self.body[:, self.ranges[0][0] if c0 is None else c0].data_ptr())

    def check(self, what):
        for c0, c1 in self.ranges:
            assert not torch.isnan(self.body[:, c0:c1].float()).any(), f"{what}: elements left unwritten"
        assert bool((self.raw[self.keep] == self.pat).all()), f"{what}: written outside its region"


def dense(rows, cols, dtype=F32):
    return Buf(rows, cols, [(0, cols)], dtype)


# ---- float64 reference of the header's contract ----------------------------------------------------------------------------
def _untranspose(p, transposed, H, W):
    Bn, D, L = p.shape
    return p.view(Bn, D, W, H).transpose(2, 3).reshape(Bn, D, L) if transposed else p


def _merge(planes):
    if len(planes) == 4:
        return (planes[0] + planes[2]) + (planes[1] + planes[3])
    y = planes[0]
    for p in planes[1:]:
        y = y + p
    return y


def _ln_gate(y, w, b, z, z_act, eps):
    """y (B, D, L) natural order -> out (B, L, D), mean, rstd (B, L)."""
    D = y.shape[1]
    yt = y.transpose(1, 2)
    out = F.layer_norm(yt, (D,), w, b, eps)
    if z is not None:
        out = out * (F.silu(z) if z_act else z)
    mean = yt.mean(-1)
    rstd = 1.0 / torch.sqrt(((yt - mean[..., None]) ** 2).mean(-1) + eps)
    return out, mean.detach(), rstd.detach()


def reference(ys, mask, lnw, lnb, z, z_act, eps, dout, H, W):
    """-> dict: out (B, L, D), mean / rstd (B, L), dy (merged, natural order), dys (per plane, each in its own order), dz,
    dlnw, dlnb. Without an affine LayerNorm the kernel still returns sum(go * yn) and sum(go): the gradients at w = 1, b = 0."""
    Bn, K, D, L = ys.shape
    ys64 = ys.double().requires_grad_()
    y = _merge([_untranspose(ys64[:, k], (mask >> k) & 1, H, W) for k in range(K)])
    y.retain_grad()
    w = (lnw.double() if lnw is not None else torch.ones(D, dtype=torch.float64, device=ys.device)).requires_grad_()
    b = (lnb.double() if lnb is not None else torch.zeros(D, dtype=torch.float64, device=ys.device)).requires_grad_()
    z64 = None if z is None else z.double().requires_grad_()
    out, mean, rstd = _ln_gate(y, w, b, z64, z_act, eps)
    out.backward(dout.double())
    return dict(out=out.detach(), mean=mean, rstd=rstd, dy=y.grad, dys=ys64.grad, dz=None if z is None else z64.grad,
                dlnw=w.grad, dlnb=b.grad)


def _transposed_order(t, H, W):
    """(B, D, L) natural order -> the transposed image's pixel order (offset w H + h)."""
    Bn, D, L = t.shape
    return t.reshape(Bn, D, H, W).transpose(2, 3).reshape(Bn, D, L)


# ---- single calls: ss2d_out_gate_fwd / ss2d_out_gate_bwd -----------------------------------------------------------------
def _inputs(Bn, K, D, L, affine, offset, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    ys = torch.randn(Bn, K, D, L, device="cuda", generator=g) + offset
    lnw = 1.0 + 0.5 * torch.randn(D, device="cuda", generator=g) if "w" in affine else None
    lnb = 0.5 * torch.randn(D, device="cuda", generator=g) if "b" in affine else None
    zv = torch.randn(Bn * L, D, device="cuda", generator=g)
    dv = torch.randn(Bn * L, D, device="cuda", generator=g)
    return ys, lnw, lnb, zv, dv


# z layouts: (z row stride, z column offset, dz row stride, dz column offset) as functions of D
Z_LAYOUTS = {
    "dense": lambda D: (D, 0, D, 0),
    "ss2d": lambda D: (2 * D, D, D, 0),                  # the second half of in_proj's rows; dz dense
    "misaligned": lambda D: (2 * D + 1, 1, D + 5, 3),    # rows not 16-byte aligned: the float4 row path must step aside
}


def run_single(Bn, K, D, H, W, mask, *, z="dense", z_act=1, affine="wb", zdt=F32, odt=F32, eps=1e-5, offset=0.0,
               dz_null=False, stats_null=False, two_planes=False, seed=0, backward=True):
    L = H * W
    lib = _lib.lib()
    ys, lnw, lnb, zv, dv = _inputs(Bn, K, D, L, affine, offset, seed)
    zb = None
    if z is not None:
        z_rs, z_c0, dz_rs, dz_c0 = Z_LAYOUTS[z](D)
        zb = Buf(Bn * L, z_rs, [(z_c0, z_c0 + D)], zdt)
        zb.cols(z_c0, D).copy_(zv.to(zdt))
    zval = None if zb is None else zb.cols(zb.ranges[0][0], D).float()
    dout = dv.to(odt)
    ref = reference(ys, mask, lnw, lnb, None if zval is None else zval.view(Bn, L, D), z_act, eps,
                    dout.float().view(Bn, L, D), H, W)

    out = dense(Bn * L, D, odt)
    stats = None if stats_null else dense(Bn * L, 2)
    rc = lib.ss2d_out_gate_fwd(_p(ys), K, _p(lnw), _p(lnb), zb.ptr() if zb else None, zb.rs if zb else 0, z_act, out.ptr(),
                               stats.ptr() if stats else None, Bn, D, L, ctypes.c_float(eps), _DT[zdt], _DT[odt], H, W,
                               ctypes.c_uint32(mask), _stream())
    assert rc == 0, rc
    out.check("out")
    _check(out.body, ref["out"].reshape(Bn * L, D), "out")
    if stats is not None:
        stats.check("mean_rstd")
        _check(stats.body[:, 0], ref["mean"].reshape(-1), "stats", " (mean)")
        _check(stats.body[:, 1], ref["rstd"].reshape(-1), "stats", " (rstd)")
    if not backward or stats is None:
        return ref
    res = run_bwd(ys, K, lnw, lnb, zb, z_act, dout, stats.body, D, H, W, mask, zdt, odt, dz_null, two_planes,
                  dz_layout=None if z is None else (dz_rs, dz_c0))
    check_bwd(res, ref, Bn, K, D, H, W, mask, two_planes)
    return ref


def run_bwd(ys, K, lnw, lnb, zb, z_act, dout, stats, D, H, W, mask, zdt, odt, dz_null=False, two_planes=False, dz_layout=None):
    Bn, L = ys.shape[0], H * W
    lib = _lib.lib()
    npart = int(lib.ss2d_out_gate_bwd_partials(Bn, L))
    dy = dense(Bn * (2 if two_planes else 1) * D, L)
    dz = None
    if zb is not None and not dz_null:
        dz_rs, dz_c0 = dz_layout
        dz = Buf(Bn * L, dz_rs, [(dz_c0, dz_c0 + D)], zdt)
    dw, db = dense(npart, D), dense(npart, D)
    rc = lib.ss2d_out_gate_bwd(_p(ys), K, _p(lnw), _p(lnb), zb.ptr() if zb else None, zb.rs if zb else 0, z_act, _p(dout),
                               _p(stats), dy.ptr(), dz.ptr() if dz else None, dz.rs if dz else 0, dw.ptr(), db.ptr(), npart, Bn,
                               D, L, _DT[zdt], _DT[odt], H, W, ctypes.c_uint32(mask), int(two_planes), _stream())
    assert rc == 0, rc
    for name, b in (("dy", dy), ("dz", dz), ("dln_w partials", dw), ("dln_b partials", db)):
        if b is not None:
            b.check(name)
    return dict(dy=dy, dz=dz, dw=dw, db=db)


def check_bwd(res, ref, Bn, K, D, H, W, mask, two_planes):
    L = H * W
    dy = res["dy"].body.view(Bn, 2 if two_planes else 1, D, L)
    if K == 1:                          # the single plane's gradient, in that plane's own pixel order
        _check(dy[:, 0], ref["dys"][:, 0], "dy")
    else:
        _check(dy[:, 0], ref["dy"], "dy")
    if two_planes:
        assert torch.equal(dy[:, 1], _transposed_order(dy[:, 0], H, W)), "second dy plane is not the first one transposed"
    if res["dz"] is not None:
        c0 = res["dz"].ranges[0][0]
        _check(res["dz"].cols(c0, D), ref["dz"].reshape(Bn * L, D), "dz")
    _check(res["dw"].body.double().sum(0), ref["dlnw"], "dln", " (weight)")
    _check(res["db"].body.double().sum(0), ref["dlnb"], "dln", " (bias)")


SHAPES = [   # (batch, K, D, H, W, transposed mask, two dy planes)
    (2, 1, 16, 56, 56, 0, False),            # small kernel DP = 16, float4 rows
    (2, 1, 16, 14, 14, 1, False),            # small kernel, transposed plane: dy in the plane's order
    (2, 1, 5, 7, 9, 1, False),               # D % 4 != 0: scalar rows; ragged
    (2, 1, 17, 5, 9, 0, False),              # DP = 32, lower edge
    (2, 1, 32, 13, 7, 1, False),             # DP = 32, upper edge
    (2, 1, 33, 13, 7, 1, False),             # tiled kernel with K = 1: transposed dy through o1 = lt; ragged patches
    (2, 2, 7, 5, 9, 0b10, False),            # PP = 32 pixel lanes
    (2, 2, 7, 5, 9, 0b10, True),
    (2, 3, 87, 7, 7, 0b101, False),          # odd D, K = 3 summation order
    (2, 4, 40, 14, 14, 0b1010, False),       # the VMamba-like mask
    (2, 4, 40, 14, 14, 0b1010, True),
    (2, 4, 100, 9, 17, 0b0101, False),       # PP = 2 with 56 idle threads; patches ragged in h and w
    (2, 4, 129, 12, 20, 0, False),           # PP = 1 below 256 channels; linear tiles, L % 32 != 0
    (2, 4, 192, 56, 56, 0b1010, True),       # north-star shape (ops.out_gate_fwd would take the TMA-fed kernel)
    (2, 2, 256, 6, 10, 0, False),            # backward m loop: one channel chunk
    (2, 2, 257, 5, 9, 0b11, False),          # two channel chunks
    (2, 2, 257, 5, 9, 0b01, True),
    (1, 1, 832, 4, 5, 0, False),             # backward width limit: four channel chunks
    (2, 8, 24, 6, 6, 0b10110100, False),     # K > 4, all eight mask bits in play
    (24, 4, 16, 56, 56, 0b1010, False),      # grid-stride: 2352 patch tiles, 1184 forward CTAs, 592 backward partials
    (100, 1, 16, 56, 56, 1, False),          # grid-stride of the small kernels: B L > 1184 x 256
]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "B%d_K%d_D%d_%dx%d_m%s%s" % (s[0], s[1], s[2], s[3], s[4], bin(s[5]),
                                                                                     "_two" if s[6] else ""))
def test_out_gate_matches_reference(shape):
    Bn, K, D, H, W, mask, two = shape
    run_single(Bn, K, D, H, W, mask, two_planes=two)


def test_forward_width_limit_and_backward_refusal():
    """D = 1664 is the widest forward; the backward of it is SS2D_ERR_UNSUPPORTED and writes nothing."""
    Bn, K, D, H, W = 2, 2, 1664, 3, 5
    L = H * W
    run_single(Bn, K, D, H, W, 0, backward=False)
    ys = torch.randn(Bn, K, D, L, device="cuda")
    lnw, lnb = torch.ones(D, device="cuda"), torch.zeros(D, device="cuda")
    z, dout, stats = (torch.randn(Bn * L, D, device="cuda") for _ in range(3))
    npart = int(_lib.lib().ss2d_out_gate_bwd_partials(Bn, L))
    dy, dz, dw, db = dense(Bn * D, L), dense(Bn * L, D), dense(npart, D), dense(npart, D)
    before = _lib.launch_count()
    rc = _lib.lib().ss2d_out_gate_bwd(_p(ys), K, _p(lnw), _p(lnb), _p(z), D, 1, _p(dout), _p(stats), dy.ptr(), dz.ptr(), D,
                                      dw.ptr(), db.ptr(), npart, Bn, D, L, _lib.SS2D_F32, _lib.SS2D_F32, H, W, ctypes.c_uint32(0), 0,
                                      _stream())
    assert rc == ERR_UNSUPPORTED and _lib.launch_count() == before
    torch.cuda.synchronize()
    for b in (dy, dz, dw, db):
        assert bool((b.raw == b.pat).all())


OPTIONS = [
    dict(),
    dict(z=None),
    dict(z_act=0),
    dict(affine="w"),
    dict(affine=""),
    dict(z="ss2d"),
    dict(z="misaligned"),
    dict(dz_null=True),
    dict(stats_null=True),
    dict(zdt=BF16, odt=BF16),
    dict(zdt=F16, odt=F16),
    dict(zdt=BF16, odt=F32),
    dict(zdt=F32, odt=BF16),
    dict(zdt=F16, odt=F32),
    dict(z="ss2d", zdt=BF16, odt=BF16),
    dict(eps=1e-2),
    dict(offset=50.0),
]
POINTS = {"small": (2, 1, 16, 7, 9, 1), "tiled": (2, 4, 40, 9, 13, 0b1010)}


def _opt_id(o):
    return "-".join("%s=%s" % (k, str(v).replace("torch.", "")) for k, v in o.items()) or "defaults"


@pytest.mark.parametrize("opts", OPTIONS, ids=_opt_id)
@pytest.mark.parametrize("point", list(POINTS))
def test_out_gate_options(point, opts):
    run_single(*POINTS[point], **opts)


# ---- the two forward routes ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 4, 192, 56, 56, 0b1010), (2, 2, 128, 12, 20, 0b10), (3, 4, 64, 8, 12, 0)], ids=str)
def test_forward_routes_agree(shape):
    """Where ops.out_gate_fwd takes the TMA-fed kernel (ss2d_gate_proj_fwd with C = 0), it and ss2d_out_gate_fwd give the same
    out and statistics, and the backward gives the same dy from either set of statistics."""
    Bn, K, D, H, W, mask = shape
    L = H * W
    assert ops.gate_proj_supported(D, 0, K, F32)
    ys, lnw, lnb, zv, dv = _inputs(Bn, K, D, L, "wb", 0.0, 3)
    z = zv.view(Bn, L, D)
    launches = _lib.launch_count()
    out_tma, st_tma = ops.out_gate_fwd(ys, lnw, lnb, z, True, 1e-5, F32, (H, W), mask)
    assert _lib.launch_count() == launches + 1
    ref = reference(ys, mask, lnw, lnb, z, 1, 1e-5, dv.view(Bn, L, D), H, W)
    _check(out_tma, ref["out"], "out")
    zb = Buf(Bn * L, D, [(0, D)], F32)
    zb.body.copy_(zv)
    out_d, st_d = dense(Bn * L, D), dense(Bn * L, 2)
    rc = _lib.lib().ss2d_out_gate_fwd(_p(ys), K, _p(lnw), _p(lnb), zb.ptr(), D, 1, out_d.ptr(), st_d.ptr(), Bn, D, L,
                                      ctypes.c_float(1e-5), _lib.SS2D_F32, _lib.SS2D_F32, H, W, ctypes.c_uint32(mask), _stream())
    assert rc == 0
    for a, b in ((out_tma.reshape(Bn * L, D), out_d.body), (st_tma.reshape(Bn * L, 2), st_d.body)):
        rel = float((a.double() - b.double()).abs().max() / b.double().abs().max())
        _note("routes", rel)
        assert rel <= 1e-6, rel
    two = K > 1 and mask != 0
    for st in (st_tma.reshape(Bn * L, 2), st_d.body):
        res = run_bwd(ys, K, lnw, lnb, zb, 1, dv, st, D, H, W, mask, F32, F32, two_planes=two, dz_layout=(D, 0))
        check_bwd(res, ref, Bn, K, D, H, W, mask, two)


def test_ops_out_gate_bwd_without_dz():
    """The header allows dz = NULL with a gate: ops.out_gate_bwd(dz_out=None) returns dy and the LayerNorm gradients."""
    Bn, K, D, H, W, mask = 2, 4, 40, 9, 13, 0b1010
    L = H * W
    ys, lnw, lnb, zv, dv = _inputs(Bn, K, D, L, "wb", 0.0, 5)
    z, dout = zv.view(Bn, L, D), dv.view(Bn, L, D)
    ref = reference(ys, mask, lnw, lnb, z, 1, 1e-5, dout, H, W)
    out, stats = ops.out_gate_fwd(ys, lnw, lnb, z, True, 1e-5, F32, (H, W), mask)
    _check(out, ref["out"], "out")
    dy, dlnw, dlnb = ops.out_gate_bwd(ys, lnw, lnb, z, True, dout, stats, None, (H, W), mask)
    _check(dy, ref["dy"], "dy")
    _check(dlnw, ref["dlnw"], "dln")
    _check(dlnb, ref["dlnb"], "dln")
    dz = torch.empty_like(z)
    dy2, _, _ = ops.out_gate_bwd(ys, lnw, lnb, z, True, dout, stats, dz, (H, W), mask)
    assert torch.equal(dy, dy2)
    _check(dz, ref["dz"], "dz")


# ---- grouped calls: ss2d_group_gate_fwd / ss2d_group_gate_bwd --------------------------------------------------------------
def group_reference(ys, plane_of, tbits, lnw, lnb, zgroups, dout_groups, eps, H, W):
    Bn, G, D, L = ys.shape
    ys64 = ys.double().requires_grad_()
    w, b = lnw.double().requires_grad_(), lnb.double().requires_grad_()
    zs = [zg.double().requires_grad_() for zg in zgroups]
    outs, means, rstds = [], [], []
    loss = 0.0
    for g in range(G):
        p = plane_of[g]
        y = _untranspose(ys64[:, p], (tbits >> p) & 1, H, W)
        o, m, r = _ln_gate(y, w[g], b[g], zs[g], 1, eps)
        loss = loss + (o * dout_groups[g].double()).sum()
        outs.append(o.detach()); means.append(m); rstds.append(r)
    loss.backward()
    return dict(out=outs, mean=means, rstd=rstds, dys=ys64.grad, dz=[zg.grad for zg in zs], dlnw=w.grad, dlnb=b.grad)


def _group_layout(G, D, z_gs):
    """z rows of width 2 G D (in_proj's output) with the gates at column G D; out / dout / dz rows with their own padding."""
    z_gs = D if z_gs is None else z_gs
    z_col0 = G * D
    span = (G - 1) * z_gs + D
    return dict(z_rs=z_col0 + max(span, G * D), z_col0=z_col0, z_gs=z_gs, out_rs=G * D + 24, dout_rs=G * D + 8,
                dz_rs=z_col0 + span + 16)


def run_grouped(Bn, G, D, H, W, plane_of, tbits, *, zdt=F32, odt=F32, z_gs=None, eps=1e-5, seed=0):
    L = H * W
    lib = _lib.lib()
    lay = _group_layout(G, D, z_gs)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    ys = torch.randn(Bn, G, D, L, device="cuda", generator=gen)
    lnw = 1.0 + 0.5 * torch.randn(G, D, device="cuda", generator=gen)
    lnb = 0.5 * torch.randn(G, D, device="cuda", generator=gen)
    zcols = [(lay["z_col0"] + g * lay["z_gs"], lay["z_col0"] + g * lay["z_gs"] + D) for g in range(G)]
    zb = Buf(Bn * L, lay["z_rs"], zcols, zdt)
    zb.body.copy_(torch.randn(Bn * L, lay["z_rs"], device="cuda", generator=gen).to(zdt))   # gaps hold other data
    dout = torch.randn(Bn * L, lay["dout_rs"], device="cuda", generator=gen).to(odt)
    zg = [zb.body[:, c0:c1].float().view(Bn, L, D) for c0, c1 in zcols]
    dg = [dout[:, g * D:(g + 1) * D].float().view(Bn, L, D) for g in range(G)]
    ref = group_reference(ys, plane_of, tbits, lnw, lnb, zg, dg, eps, H, W)
    arr = (ctypes.c_int32 * G)(*plane_of)

    out = Buf(Bn * L, lay["out_rs"], [(0, G * D)], odt)
    stats = dense(G * Bn * L, 2)
    rc = lib.ss2d_group_gate_fwd(_p(ys), G, arr, ctypes.c_uint32(tbits), _p(lnw), _p(lnb), zb.ptr(0), lay["z_rs"], lay["z_col0"],
                                 lay["z_gs"], out.ptr(0), lay["out_rs"], stats.ptr(), Bn, D, L, ctypes.c_float(eps), _DT[zdt],
                                 _DT[odt], H, W, _stream())
    assert rc == 0, rc
    out.check("out")
    stats.check("mean_rstd")
    st = stats.body.view(G, Bn * L, 2)
    for g in range(G):
        _check(out.cols(g * D, D), ref["out"][g].reshape(Bn * L, D), "out", f" (group {g})")
        _check(st[g, :, 0], ref["mean"][g].reshape(-1), "stats", f" (group {g} mean)")
        _check(st[g, :, 1], ref["rstd"][g].reshape(-1), "stats", f" (group {g} rstd)")

    npart = int(lib.ss2d_out_gate_bwd_partials(Bn, L))

    def backward():
        dy = dense(Bn * G * D, L)
        dz = Buf(Bn * L, lay["dz_rs"], zcols, zdt)
        dw, db = dense(G * npart, D), dense(G * npart, D)
        rc = lib.ss2d_group_gate_bwd(_p(ys), G, arr, ctypes.c_uint32(tbits), _p(lnw), _p(lnb), zb.ptr(0), lay["z_rs"],
                                     lay["z_col0"], lay["z_gs"], _p(dout), lay["dout_rs"], stats.ptr(), dy.ptr(), dz.ptr(0),
                                     lay["dz_rs"], dw.ptr(), db.ptr(), npart, Bn, D, L, _DT[zdt], _DT[odt], H, W, _stream())
        assert rc == 0, rc
        return dy, dz, dw, db

    dy, dz, dw, db = backward()
    for name, b in (("dy", dy), ("dz", dz), ("dln_w partials", dw), ("dln_b partials", db)):
        b.check(name)
    _check(dy.body.view(Bn, G, D, L), ref["dys"], "dy")       # plane p in its own pixel order
    for g, (c0, _) in enumerate(zcols):
        _check(dz.cols(c0, D), ref["dz"][g].reshape(Bn * L, D), "dz", f" (group {g})")
    _check(dw.body.view(G, npart, D).double().sum(1), ref["dlnw"], "dln", " (weight)")
    _check(db.body.view(G, npart, D).double().sum(1), ref["dlnb"], "dln", " (bias)")
    return backward, (dy, dz, dw, db)


GROUPED = [   # (batch, G, D, H, W, plane_of, transposed_planes, z_group_stride)
    (2, 4, 16, 14, 14, (0, 2, 1, 3), 0b1100, None),      # what GroupMambaLayer passes, small kernel
    (2, 4, 32, 14, 14, (3, 1, 0, 2), 0b0101, None),
    (2, 4, 87, 9, 13, (0, 1, 2, 3), 0b1111, None),       # tiled, odd D, non-square image
    (2, 4, 112, 14, 14, (0, 2, 1, 3), 0b1100, None),
    (2, 4, 16, 7, 11, (0, 2, 1, 3), 0b1100, 24),         # gate groups D + 8 columns apart
    (2, 3, 16, 7, 11, (2, 0, 1), 0b0101, None),
    (2, 3, 112, 6, 10, (1, 2, 0), 0b1111, None),
    (2, 2, 87, 5, 9, (1, 0), 0b0101, None),
    (2, 2, 32, 9, 6, (0, 1), 0b1100, None),
    (2, 1, 32, 9, 13, (0,), 0b1111, None),
    (2, 1, 112, 7, 7, (0,), 0b1100, None),
]


@pytest.mark.parametrize("case", GROUPED, ids=lambda c: "B%d_G%d_D%d_%dx%d_p%s_t%s%s" % (
    c[0], c[1], c[2], c[3], c[4], "".join(map(str, c[5])), bin(c[6]), "" if c[7] is None else "_zgs%d" % c[7]))
def test_group_gate_matches_reference(case):
    Bn, G, D, H, W, plane_of, tbits, z_gs = case
    run_grouped(Bn, G, D, H, W, plane_of, tbits, z_gs=z_gs)


@pytest.mark.parametrize("dt", [(BF16, BF16), (F16, F32), (F32, BF16)], ids=str)
@pytest.mark.parametrize("D", [16, 87])
def test_group_gate_dtypes(D, dt):
    run_grouped(2, 4, D, 7, 11, (0, 2, 1, 3), 0b1100, zdt=dt[0], odt=dt[1])


def test_ops_group_gate_matches_reference():
    Bn, G, D, H, W, plane_of, tbits = 2, 4, 16, 14, 14, (0, 2, 1, 3), 0b1100
    L = H * W
    ys = torch.randn(Bn, G, D, L, device="cuda")
    lnw, lnb = 1.0 + 0.5 * torch.randn(G, D, device="cuda"), 0.5 * torch.randn(G, D, device="cuda")
    z, dout = torch.randn(Bn, L, G * D, device="cuda"), torch.randn(Bn, L, G * D, device="cuda")
    ref = group_reference(ys, plane_of, tbits, lnw, lnb, list(z.split(D, -1)), list(dout.split(D, -1)), 1e-5, H, W)
    out, stats = ops.group_gate_fwd(ys, plane_of, tbits, lnw, lnb, z, 1e-5, F32, (H, W))
    _check(out, torch.cat(ref["out"], -1), "out")
    dy, dz, dlnw, dlnb = ops.group_gate_bwd(ys, plane_of, tbits, lnw, lnb, z, dout, stats, (H, W))
    _check(dy, ref["dys"], "dy")
    _check(dz, torch.cat(ref["dz"], -1), "dz")
    _check(dlnw, ref["dlnw"], "dln")
    _check(dlnb, ref["dlnb"], "dln")


# ---- determinism -------------------------------------------------------------------------------------------------------------
def _bits_equal(a, b):
    return torch.equal(a.raw, b.raw)


@pytest.mark.parametrize("shape", [(2, 1, 16, 14, 14, 1, False), (2, 4, 40, 14, 14, 0b1010, True), (1, 1, 832, 4, 5, 0, False),
                                   (24, 4, 16, 56, 56, 0b1010, False)], ids=str)
def test_backward_is_deterministic(shape):
    Bn, K, D, H, W, mask, two = shape
    L = H * W
    ys, lnw, lnb, zv, dv = _inputs(Bn, K, D, L, "wb", 0.0, 7)
    zb = Buf(Bn * L, D, [(0, D)], F32)
    zb.body.copy_(zv)
    stats = dense(Bn * L, 2)
    out = dense(Bn * L, D)
    assert _lib.lib().ss2d_out_gate_fwd(_p(ys), K, _p(lnw), _p(lnb), zb.ptr(), D, 1, out.ptr(), stats.ptr(), Bn, D, L,
                                        ctypes.c_float(1e-5), 0, 0, H, W, ctypes.c_uint32(mask), _stream()) == 0
    a = run_bwd(ys, K, lnw, lnb, zb, 1, dv, stats.body, D, H, W, mask, F32, F32, two_planes=two, dz_layout=(D, 0))
    b = run_bwd(ys, K, lnw, lnb, zb, 1, dv, stats.body, D, H, W, mask, F32, F32, two_planes=two, dz_layout=(D, 0))
    for k in ("dy", "dz", "dw", "db"):
        assert _bits_equal(a[k], b[k]), k


def test_grouped_backward_is_deterministic_and_graph_replays_it():
    backward, first = run_grouped(2, 4, 16, 14, 14, (0, 2, 1, 3), 0b1100)
    again = backward()
    for k, x, y in zip(("dy", "dz", "dw", "db"), first, again):
        assert _bits_equal(x, y), k
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = backward()
    for b in captured:
        b.raw.fill_(b.pat)
    graph.replay()
    torch.cuda.synchronize()
    for k, x, y in zip(("dy", "dz", "dw", "db"), first, captured):
        assert _bits_equal(x, y), k
