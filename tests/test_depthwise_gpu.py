"""GPU parity of the depthwise convolution kernels against a float64 restatement of their contract in include/ss2d_b200.h:
the FFN stack on channels-last tensors (csrc/ffn_dw.cu; C ABI ss2d_dwnhwc_stencil / ss2d_dwnhwc_wgrad: the column walker, the
tiled stencil and the row-walking weight gradient) and SS2D's 3 x 3 convolution + SiLU (csrc/dwconv.cu; ss2d_dwconv3_act,
ss2d_dwconv3_act_planes, ss2d_dwconv3_wgrad).

The calls go straight to the C ABI with torch-allocated buffers, so that pointer offsets, NULL biases and the kernel the
automatic choice would not take can be picked. Every output lives inside a buffer pre-filled with a NaN pattern and padded by
guard bands: the documented region must be fully written and every other element (guards, batch-stride gaps) keeps its bits.
The weight-gradient workspaces are NaN-filled too, so a partial the reduction never writes reaches the result. Shapes that
are meant to reach one branch of the host's dispatch (walker row segmentation, vector width, rows per CTA, slab count)
mirror that choice in Python and assert it, so the coverage does not drift when the dispatch changes.

The reference zero-pads, sums the k^2 shifted slices times the weights (flip: the reversed kernel), applies GELU as
0.5 x (1 + erf(x / sqrt 2)) (derivative Phi(x) + x phi(x)) or SiLU, and forms weight gradients as float64 sums over shifted
slices. 16-bit inputs are upcast exactly. Bounds:
  * linear stencil outputs (epi 0 / 2, flip, dwconv3 mode 2): |got - ref| <= tol (|b| + sum |w||x|) per element;
  * GELU / SiLU outputs: max |got - ref| / max |ref| per tensor;
  * weight gradients: |got - ref| <= tol sum |g||x| per channel and tap (sum |g| for the bias);
  * 16-bit outputs: |got - ref| <= u |ref| + 1e-5 max |ref|, u = 2^-8 (bf16) or 2^-11 (fp16).
Bounds (TOL) and the largest values seen on a B200 at a 1000 W power limit: stencil 1e-6 (seen 3.4e-7), GELU 1e-6 (3.6e-7),
FFN weight gradient 4e-7 (1.1e-7), SiLU 1.5e-6 (4.6e-7), dwconv3 mode 2 1e-6 (2.6e-7), dwconv3 weight gradient 2.5e-7
(7.2e-8); 16-bit outputs up to 0.99 of the rounding bound. Each test records its worst value per family in its user
properties (written to the junit report)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from ceigm_unet_b200 import _lib, ops

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
DTYPES = [F32, F16, BF16]
_DT = {F32: _lib.SS2D_F32, F16: _lib.SS2D_F16, BF16: _lib.SS2D_BF16}
TOL = {"stencil": 1e-6, "gelu": 1e-6, "wgrad": 4e-7, "silu": 1.5e-6, "act_lin": 1e-6, "dw3_wgrad": 2.5e-7}
ROUND = {BF16: 2.0 ** -8, F16: 2.0 ** -11}

_observed = {}


@pytest.fixture(autouse=True)
def _record_and_restore(request):
    """Records the worst value per family in the test's user properties; puts the kernel choice back to automatic."""
    _observed.clear()
    try:
        yield
    finally:
        _lib.test_force_path(0)
        request.node.user_properties.extend(sorted(_observed.items()))


def _note(key, v):
    _observed[key] = max(_observed.get(key, 0.0), v)


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


# ---- checks ---------------------------------------------------------------------------------------------------------------
def _check16(got, ref, family, what):
    err = (got.double() - ref).abs()
    ratio = float((err / (ROUND[got.dtype] * ref.abs() + 1e-5 * ref.abs().max().clamp_min(1e-30))).max())
    _note(family + "16_ratio", ratio)
    assert ratio <= 1.0, f"{family}{what}: {got.dtype} error {ratio:.3g} x the rounding bound"


def check_abs(got, ref, mag, family, what=""):
    """Linear outputs: elementwise against the same operation on absolute values (fp32), or the rounding bound (16-bit)."""
    if got.dtype in ROUND:
        return _check16(got, ref, family, what)
    rel = float(((got.double() - ref).abs() / mag.clamp_min(1e-30)).max())
    _note(family, rel)
    assert rel <= TOL[family], f"{family}{what}: error {rel:.3g} x sum|terms| > {TOL[family]}"


def check_max(got, ref, family, what=""):
    """Non-linear outputs: max error over max |ref| of the tensor (fp32), or the rounding bound (16-bit)."""
    if got.dtype in ROUND:
        return _check16(got, ref, family, what)
    rel = float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    _note(family, rel)
    assert rel <= TOL[family], f"{family}{what}: rel err {rel:.3g} > {TOL[family]}"


# ---- guarded buffers ------------------------------------------------------------------------------------------------------
_PATTERN = {F32: (torch.int32, 0x7FC0BEEF), F16: (torch.int16, 0x7FDA), BF16: (torch.int16, 0x7FDA)}   # NaN in every dtype
GUARD = 64


class Out:
    """n elements of `dtype` at element offset `off` of a buffer pre-filled with a NaN pattern, GUARD elements on both sides.
    `written`: bool mask of the n elements the call must write (default: all); the rest must keep the pattern."""

    def __init__(self, n, dtype, off=0, written=None):
        it, self.pat = _PATTERN[dtype]
        self.raw = torch.full((2 * GUARD + off + n,), self.pat, dtype=it, device="cuda")
        self.body = self.raw.view(dtype)[GUARD + off:GUARD + off + n]
        self.written = written
        self.keep = torch.ones(self.raw.numel(), dtype=torch.bool, device="cuda")
        self.keep[GUARD + off:GUARD + off + n] = False if written is None else ~written

    def ptr(self, elem=0):
        return ctypes.c_void_p(self.body.data_ptr() + elem * self.body.element_size())

    def check(self, what):
        vals = self.body if self.written is None else self.body[self.written]
        assert not torch.isnan(vals.float()).any(), f"{what}: elements left unwritten"
        assert bool((self.raw[self.keep] == self.pat).all()), f"{what}: written outside its region"


def placed(t, off=0):
    """A contiguous copy of t starting `off` elements into a fresh allocation (off > 0 lowers the pointer's alignment)."""
    buf = torch.empty(off + t.numel() + 8, dtype=t.dtype, device=t.device)
    v = buf[off:off + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def nan_workspace(nbytes):
    return torch.full((max(nbytes // 4, 1),), 0x7FC0BEEF, dtype=torch.int32, device="cuda")


# ---- float64 reference ----------------------------------------------------------------------------------------------------
def gelu64(a):
    return 0.5 * a * (1.0 + torch.erf(a / 2.0 ** 0.5))


def dgelu64(a):
    return 0.5 * (1.0 + torch.erf(a / 2.0 ** 0.5)) + a * torch.exp(-0.5 * a * a) / (2.0 * torch.pi) ** 0.5


def conv_nhwc(x, w, b, flip):
    """Depthwise k x k correlation of x (B, H, W, c) float64, zero padding k // 2; w (c, 1, k, k); -> (acc, sum of |terms|)."""
    Bn, H, W, c = x.shape
    k = w.shape[-1]
    P = k // 2
    wk = w.double().reshape(c, k, k)
    if flip:
        wk = wk.flip(1, 2)
    xp = F.pad(x, (0, 0, P, P, P, P))
    acc = torch.zeros_like(x) if b is None else b.double().expand_as(x).clone()
    mag = torch.zeros_like(x) if b is None else b.double().abs().expand_as(x).clone()
    for i in range(k):
        for j in range(k):
            sl = xp[:, i:i + H, j:j + W]
            acc += wk[:, i, j] * sl
            mag += wk[:, i, j].abs() * sl.abs()
    return acc, mag


def ref_stencil(x, aux, segs, flip, epi):
    """x, aux: (B, H, W, C) -> (y, sum of |terms| of the linear epilogues), float64. segs: [(c_end, k, w, b), ...]."""
    x = x.double()
    acc, mag = torch.zeros_like(x), torch.zeros_like(x)
    c0 = 0
    for c1, k, w, b in segs:
        if k == 1:
            acc[..., c0:c1] = x[..., c0:c1]
            mag[..., c0:c1] = x[..., c0:c1].abs()
        elif k > 1:
            acc[..., c0:c1], mag[..., c0:c1] = conv_nhwc(x[..., c0:c1], w, b, flip)
        c0 = c1
    if epi == 0:
        return acc, mag
    if epi == 1:
        return gelu64(acc), None
    if epi == 2:
        return x + acc, mag + x.abs()
    return aux.double() * dgelu64(acc), None


def ref_wgrad_nhwc(x, g, K):
    """x, g: (B, H, W, c) -> dW (c, K, K), its sum of |terms|, db (c), sum |g| (c), float64."""
    x, g = x.double(), g.double()
    Bn, H, W, c = x.shape
    P = K // 2
    xp = F.pad(x, (0, 0, P, P, P, P))
    dW = torch.empty(c, K, K, dtype=torch.float64, device=x.device)
    mag = torch.empty_like(dW)
    for i in range(K):
        for j in range(K):
            sl = xp[:, i:i + H, j:j + W]
            dW[:, i, j] = (g * sl).sum((0, 1, 2))
            mag[:, i, j] = (g.abs() * sl.abs()).sum((0, 1, 2))
    return dW, mag, g.sum((0, 1, 2)), g.abs().sum((0, 1, 2))


def _nhwc(t):         # (B, C, H, W) -> (B, H, W, C)
    return t.permute(0, 2, 3, 1)


# ---- ss2d_dwnhwc_stencil --------------------------------------------------------------------------------------------------
def dwn_vec(C, bounds, esz, ptrs):
    """Mirror of dwn_vec (csrc/ffn_dw.cu): the widest of 4 / 2 / 1 channels that divides C and every bound and keeps each
    pointer aligned to VEC elements."""
    for v in (4, 2):
        if C % v == 0 and all(b % v == 0 for b in bounds) and all(p % (v * esz) == 0 for p in ptrs if p):
            return v
    return 1


def walk_geometry(B, H, W, C, esz):
    """Mirror of walk3_launch's row segmentation: -> (rows per segment rs, number of segments nrs)."""
    tiles_w, nblk = _cdiv(W, 16), _cdiv(C, 64)
    slots = _sms() * (2 if esz == 2 else 1)
    base = B * tiles_w * nblk
    best, best_cost = 1, -1
    for n in range(1, min(16, H) + 1):
        rs = _cdiv(H, n)
        cost = _cdiv(base * _cdiv(H, rs), slots) * (rs + 2)
        if best_cost < 0 or cost < best_cost:
            best, best_cost = n, cost
    rs = _cdiv(H, best)
    return rs, _cdiv(H, rs)


def make_segs(widths, gen, bias=True, wscale=1.0):
    """widths: [(channels, k) or (channels, k, has_bias)] -> [(c_end, k, w, b)] with fp32 CUDA weights."""
    segs, c = [], 0
    for item in widths:
        n, k = item[0], item[1]
        hb = bias if len(item) < 3 else item[2]
        c += n
        w = wscale * torch.randn(n, 1, k, k, device="cuda", generator=gen) / k if k > 1 else None
        b = 0.5 * torch.randn(n, device="cuda", generator=gen) if (k > 1 and hb) else None
        segs.append((c, k, w, b))
    return segs


def run_stencil(B, H, W, widths, dtype=F32, epi=0, flip=0, bias=True, offsets=None, off=0, hook=0, want_vec=None,
                want_walker=None, seed=0):
    """One ss2d_dwnhwc_stencil call on a (B, H, W, C) image built from `widths`; x, aux and y start `off` elements into
    their allocations. offsets: per-image constants added to x (a halo that crosses images shows)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    segs = make_segs(widths, gen, bias, wscale=2.0 if epi in (1, 3) else 1.0)
    C = segs[-1][0]
    x = torch.randn(B, H, W, C, device="cuda", generator=gen)
    if offsets is not None:
        x += torch.tensor(offsets, dtype=torch.float32, device="cuda").view(B, 1, 1, 1)
    x = placed(x.to(dtype), off)
    aux = placed(torch.randn(B, H, W, C, device="cuda", generator=gen).to(dtype), off) if epi == 3 else None
    y = Out(B * H * W * C, dtype, off)
    bounds = [s[0] for s in segs]
    vec = dwn_vec(C, bounds, x.element_size(), [x.data_ptr(), None if aux is None else aux.data_ptr(), y.body.data_ptr()])
    walker = vec == 4 and len(segs) == 1 and segs[0][1] == 3 and hook != 3
    if want_vec is not None:
        assert vec == want_vec, f"the case meant for VEC {want_vec} gets VEC {vec}"
    if want_walker is not None:
        assert walker == want_walker
    n = len(segs)
    cbeg = (ctypes.c_int32 * (n + 1))(0, *bounds)
    ks = (ctypes.c_int32 * n)(*[s[1] for s in segs])
    wp = (ctypes.c_void_p * n)(*[None if s[2] is None else s[2].data_ptr() for s in segs])
    bp = (ctypes.c_void_p * n)(*[None if s[3] is None else s[3].data_ptr() for s in segs])
    _lib.test_force_path(hook)
    rc = _lib.lib().ss2d_dwnhwc_stencil(_p(x), _p(aux), y.ptr(), n, cbeg, ks, wp, bp, flip, epi, B, H, W, C, _DT[dtype], _stream())
    assert rc == 0, rc
    y.check("y")
    ref, mag = ref_stencil(x, aux, segs, flip, epi)
    got = y.body.view(B, H, W, C)
    what = f" (epi {epi}, flip {flip}, {'walker' if walker else 'tiled VEC %d' % vec})"
    if epi in (0, 2):
        check_abs(got, ref, mag, "stencil", what)
    else:
        check_max(got, ref, "gelu", what)
    return vec, walker


@pytest.mark.parametrize("bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("flip", [0, 1])
@pytest.mark.parametrize("epi", [0, 1, 2, 3])
def test_walker_epilogues(epi, flip, dtype, bias):
    """The column walker in every epilogue, both orientations and every I/O type; 72 channels leave 8 of the second block."""
    run_stencil(2, 7, 19, [(72, 3)], dtype, epi, flip, bias, want_vec=4, want_walker=True)


WALKER_IMAGES = [(1, 1, 12), (1, 37, 12), (29, 1, 12), (2, 3, 12), (5, 17, 12), (33, 4, 12), (56, 56, 64), (56, 56, 512)]


@pytest.mark.parametrize("H,W,C", WALKER_IMAGES, ids=lambda v: str(v))
def test_walker_images(H, W, C):
    """Degenerate and ragged images (a single row or column, edges of the 16-column tile and of the 3-fold unroll) and the
    live PVT2FFN width 512; two images offset by very different constants in the linear epilogues."""
    for epi, flip in ((0, 0), (0, 1), (1, 0), (2, 0), (3, 1)):
        run_stencil(2, H, W, [(C, 3)], F32, epi, flip, offsets=(0.0, 300.0) if epi in (0, 2) else None, want_walker=True,
                    seed=H * W + epi)


# (B, H, W, C, dtype, rs mod 3)
WALKER_SEGMENTS = [(1, 50, 16, 64, F32, 1), (2, 78, 23, 64, F32, 2), (1, 50, 16, 64, BF16, 1), (1, 78, 9, 8, F16, 2),
                   (3, 40, 16, 64, F32, 0)]


@pytest.mark.parametrize("case", WALKER_SEGMENTS, ids=lambda c: "B%d_%dx%d_C%d_%s" % (c[0], c[1], c[2], c[3], str(c[4])[6:]))
def test_walker_row_segments(case):
    """Images split into several row segments with a ragged last one, segment lengths 1 and 2 (mod 3) away from the walk's
    3-fold unroll; images offset by very different constants, so rows read across a segment or image border show."""
    B, H, W, C, dtype, rmod = case
    rs, nrs = walk_geometry(B, H, W, C, torch.finfo(dtype).bits // 8)
    assert nrs > 1 and H % rs != 0 and rs % 3 == rmod, (rs, nrs)
    offs = [(-1) ** b * 100.0 * (b + 1) for b in range(B)]
    for epi, flip in ((0, 0), (0, 1), (2, 1), (1, 0), (3, 0)):
        run_stencil(B, H, W, [(C, 3)], dtype, epi, flip, offsets=offs if epi in (0, 2) else None, want_walker=True, seed=epi)


# (B, H, W, [(channels, k[, bias])], VEC, dtype)
TILED = [
    (1, 56, 56, [(320, 1), (64, 3), (64, 5), (64, 7)], 4, F32),          # custom_ffn multi-scale stage, hidden 512
    (2, 14, 14, [(870, 1), (174, 3), (174, 5), (174, 7)], 2, F32),       # hidden 1392: segments on even, not 4-aligned bounds
    (2, 14, 14, [(870, 1), (174, 3), (174, 5), (174, 7)], 2, BF16),
    (2, 9, 17, [(4, 0), (12, 3), (20, 5), (12, 7)], 4, F32),             # every kernel size, NULL weight for k = 0
    (2, 7, 15, [(36, 3), (28, 5, False)], 4, F32),                       # blocks below 64 channels: idle lanes; NULL bias
    (2, 5, 33, [(100, 7)], 4, F32),                                      # one 7 x 7 segment: a full and a 36-channel block
    (2, 6, 16, [(1, 3), (6, 5, False), (3, 7)], 1, F32),                 # single-channel and odd-bounded segments
    (2, 6, 16, [(1, 3), (6, 5, False), (3, 7)], 1, F16),
    (2, 11, 17, [(2, 7), (6, 5), (2, 3, False)], 2, F32),                # even bounds
    (3, 1, 2, [(4, 7), (4, 5)], 4, F32),                                 # images smaller than the kernel
    (2, 3, 3, [(8, 7), (6, 3), (2, 1)], 2, BF16),
    (1, 13, 16, [(6, 3)], 2, F32),                                       # the single-segment 3 x 3 case at VEC 2
    (2, 9, 31, [(24, 3)], 4, F16),                                       # ... at VEC 4 through the test hook
]


@pytest.mark.parametrize("case", TILED, ids=lambda c: "B%d_%dx%d_%s_%s" % (
    c[0], c[1], c[2], "-".join("%dk%d%s" % (s[0], s[1], "nb" if len(s) > 2 else "") for s in c[3]), str(c[5])[6:]))
def test_tiled_segments(case):
    """The tiled kernel on segment lists mixing k in {0, 1, 3, 5, 7}, block tails, VEC 4 / 2 / 1 and small images; H is not a
    multiple of the 4 rows a thread owns and W lies around the 16-column tile."""
    B, H, W, widths, vec, dtype = case
    for epi, flip in ((0, 0), (0, 1), (1, 0), (2, 1), (3, 1)):
        run_stencil(B, H, W, widths, dtype, epi, flip, hook=3, want_vec=vec, want_walker=False, seed=epi,
                    offsets=[50.0 * b for b in range(B)] if epi in (0, 2) else None)


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("flip", [0, 1])
@pytest.mark.parametrize("epi", [0, 1, 2, 3])
def test_tiled_epilogues(epi, flip, dtype):
    """Every epilogue and orientation for 5 x 5 / 7 x 7 segments (weights staged in shared memory, flip applied there)."""
    run_stencil(2, 9, 17, [(4, 0), (12, 3), (20, 5, False), (12, 7)], dtype, epi, flip, want_vec=4, want_walker=False)


@pytest.mark.parametrize("dtype,off,vec", [(F32, 2, 2), (F16, 2, 2), (BF16, 2, 2), (F32, 4, 4)], ids=str)
def test_pointer_offsets_lower_the_vector_width(dtype, off, vec):
    """x, aux and y that start off the 16-byte (fp32) / 8-byte (16-bit) grid take narrower vectors — here a case the walker
    would otherwise take, and a multi-segment one."""
    for epi in (0, 3):
        run_stencil(2, 6, 13, [(16, 3)], dtype, epi, 0, off=off, want_vec=vec, want_walker=vec == 4)
        run_stencil(2, 6, 13, [(8, 1), (8, 5)], dtype, epi, 1, off=off, want_vec=vec, want_walker=False)


# ---- ss2d_dwnhwc_wgrad ----------------------------------------------------------------------------------------------------
def wgrad_rpl(B, H, nc, K, vec, esz):
    """Mirror of dwn_pick_rpl (csrc/ffn_dw.cu) for the instantiation the call takes."""
    groups = _cdiv(B * H, 16)
    cblocks = _cdiv(nc, 16 * vec)
    slots = _sms() * (2 if (K == 3 and esz == 2) else 1)
    rmin = _cdiv(groups, 65535)
    best, best_cost = rmin, -1
    for r in range(rmin, rmin + 8):
        cost = _cdiv(_cdiv(groups, r) * cblocks, slots) * r
        if best_cost < 0 or cost <= best_cost:
            best, best_cost = r, cost
    return best


def run_wgrad(B, H, W, C, c0, c1, K, dtype=F32, want_vec=None, bias=True, off=0, seed=0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = placed(torch.randn(B, H, W, C, device="cuda", generator=gen).to(dtype), off)
    g = placed(torch.randn(B, H, W, C, device="cuda", generator=gen).to(dtype), off)
    nc = c1 - c0
    vec = dwn_vec(C, [c0, c1], x.element_size(), [x.data_ptr(), g.data_ptr()])
    vec = min(vec, 2) if K > 3 else vec
    if want_vec is not None:
        assert vec == want_vec, f"the case meant for VEC {want_vec} gets VEC {vec}"
    lib = _lib.lib()
    ws_bytes = int(lib.ss2d_dwnhwc_wgrad_workspace_bytes(B, H, W, nc, K))
    assert ws_bytes == min(_cdiv(B * H, 16), 65535) * nc * (K * K + 1) * 4
    ws = nan_workspace(ws_bytes)
    dW, db = Out(nc * K * K, F32), (Out(nc, F32) if bias else None)
    rc = lib.ss2d_dwnhwc_wgrad(_p(x), _p(g), c0, c1, K, dW.ptr(), db.ptr() if db else None, B, H, W, C, _DT[dtype], _p(ws),
                               ctypes.c_size_t(ws_bytes), _stream())
    assert rc == 0, rc
    dW.check("dweight")
    ref, mag, rdb, dbmag = ref_wgrad_nhwc(x[..., c0:c1], g[..., c0:c1], K)
    what = f" (K {K}, VEC {vec})"
    check_abs(dW.body.view(nc, K, K), ref, mag, "wgrad", what)
    if db is not None:
        db.check("dbias")
        check_abs(db.body, rdb, dbmag, "wgrad", what + " bias")
    return dW, db, vec


# (C, c0, c1) per vector width: segment in the middle of C
WG_BOUNDS = {4: (40, 8, 32), 2: (38, 6, 30), 1: (37, 5, 26)}
WG_SHAPES = [(3, 1, 56), (2, 3, 11), (2, 14, 13), (3, 17, 2), (5, 3, 1), (2, 14, 6), (2, 17, 7)]


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("K,vec", [(3, 4), (3, 2), (3, 1), (5, 2), (5, 1), (7, 2), (7, 1)])
def test_wgrad_kernel_sizes_and_widths(K, vec, dtype):
    """Every (K, VEC) instantiation in every I/O type, on shapes whose 16-row groups straddle images (H 1, 3, 14, 17) and
    whose rows end inside the walk's K-fold unroll or the 3 x 3 ping-pong (W 1, 2, K - 1, 6k +- 1, 56)."""
    C, c0, c1 = WG_BOUNDS[vec]
    shapes = WG_SHAPES + [(2, 5, K - 1)]
    for i, (B, H, W) in enumerate(shapes):
        run_wgrad(B, H, W, C, c0, c1, K, dtype, want_vec=vec, seed=i)


def test_wgrad_several_row_groups_per_cta():
    """B = 64 at 56^2 with 64 channels: dwn_pick_rpl gives each CTA more than one 16-row group."""
    B, H, W, C = 64, 56, 56, 64
    assert wgrad_rpl(B, H, C, 3, 4, 4) > 1
    run_wgrad(B, H, W, C, 0, C, 3, F32, want_vec=4)


def test_wgrad_pointer_offset_and_null_bias_and_repeatability():
    """x and g at an 8-byte offset take VEC 2; dbias = NULL; a second call gives the same bits."""
    a = run_wgrad(2, 14, 13, 40, 8, 32, 3, F32, want_vec=2, off=2, seed=3)
    b = run_wgrad(2, 14, 13, 40, 8, 32, 3, F32, want_vec=2, off=2, seed=3)
    assert torch.equal(a[0].raw, b[0].raw) and torch.equal(a[1].raw, b[1].raw)
    for K in (3, 7):
        run_wgrad(3, 17, 9, 40, 8, 32, K, BF16, bias=False)


# ---- ss2d_dwconv3_act -----------------------------------------------------------------------------------------------------
def ref_act(mode, x, w, b, dy):
    """x, dy: (B, C, H, W) -> (y, sum of |terms| for mode 2), float64."""
    acc, mag = conv_nhwc(_nhwc(x.double()), w, None if mode == 2 else b, mode == 2)
    acc, mag = acc.permute(0, 3, 1, 2), mag.permute(0, 3, 1, 2)
    if mode == 2:
        return acc, mag
    s = torch.sigmoid(acc)
    if mode == 0:
        return acc * s, None
    return dy.double() * s * (1.0 + acc * (1.0 - s)), None


def run_act(mode, B, C, H, W, dtype, bias=True, seed=0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, C, H, W, device="cuda", generator=gen).to(dtype)
    w = 0.6 * torch.randn(C, 1, 3, 3, device="cuda", generator=gen)
    b = 0.5 * torch.randn(C, device="cuda", generator=gen) if bias else None
    dy = torch.randn(B, C, H, W, device="cuda", generator=gen).to(dtype) if mode == 1 else None
    y = Out(B * C * H * W, dtype)
    rc = _lib.lib().ss2d_dwconv3_act(mode, _p(x), _p(w), _p(b), _p(dy), y.ptr(), B, C, H, W, _DT[dtype], _stream())
    assert rc == 0, rc
    y.check("y")
    ref, mag = ref_act(mode, x, w, b, dy)
    got = y.body.view(B, C, H, W)
    if mode == 2:
        check_abs(got, ref, mag, "act_lin", " (mode 2)")
    else:
        check_max(got, ref, "silu", f" (mode {mode})")


@pytest.mark.parametrize("bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("W", [12, 13], ids=["px4", "px1"])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_dwconv3_act(mode, W, dtype, bias):
    run_act(mode, 2, 5, 9, W, dtype, bias)


@pytest.mark.parametrize("shape", [(8, 96, 64, 64), (2, 64, 75, 75)], ids=str)
def test_dwconv3_act_grid_stride(shape):
    """More work items than the 16 CTAs per SM x 256 threads of the launch: the grid-stride loop wraps."""
    B, C, H, W = shape
    items = B * C * H * (W // 4 if W % 4 == 0 else W)
    assert items > _sms() * 16 * 256
    for mode in (0, 1, 2):
        run_act(mode, B, C, H, W, F32, seed=mode)


# ---- ss2d_dwconv3_act_planes ----------------------------------------------------------------------------------------------
def _transposed(t):   # (B, C, H, W) -> (B, C, W * H): offset w * H + h
    Bn, C, H, W = t.shape
    return t.transpose(2, 3).reshape(Bn, C, W * H)


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("variant", ["y", "y+yT", "dy", "dy+dyT"])
@pytest.mark.parametrize("H,W", [(4, 4), (36, 28), (64, 32)], ids=str)
def test_dwconv3_act_planes(H, W, variant, dtype):
    """The 32 x 32 tile kernel on images that leave partial tiles. With yT, y and yT are the two halves of one (B, 2 C, L)
    buffer whose batch stride is padded: the gap stays untouched. Batch strides of x and dy are padded as well."""
    B, C, L = 2, 3, H * W
    pad = 8
    gen = torch.Generator(device="cuda").manual_seed(H + W)
    xs = C * L + pad
    xbuf = torch.randn(B, xs, device="cuda", generator=gen).to(dtype)
    x = xbuf[:, :C * L].view(B, C, H, W)
    w = 0.6 * torch.randn(C, 1, 3, 3, device="cuda", generator=gen)
    b = 0.5 * torch.randn(C, device="cuda", generator=gen)
    lib = _lib.lib()
    if variant.startswith("y"):
        two = variant == "y+yT"
        ys = (2 if two else 1) * C * L + pad
        written = torch.zeros(B, ys, dtype=torch.bool, device="cuda")
        written[:, :(2 if two else 1) * C * L] = True
        out = Out(B * ys, dtype, written=written.view(-1))
        rc = lib.ss2d_dwconv3_act_planes(0, _p(x), xs, _p(w), _p(b), None, 0, None, 0, out.ptr(), ys,
                                         out.ptr(C * L) if two else None, ys, B, C, H, W, _DT[dtype], _stream())
        assert rc == 0, rc
        out.check("y / yT")
        ref, _ = ref_act(0, x, w, b, None)
        body = out.body.view(B, ys)
        check_max(body[:, :C * L].view(B, C, H, W), ref, "silu", " (planes mode 0)")
        if two:
            check_max(body[:, C * L:2 * C * L].view(B, C, L), _transposed(ref), "silu", " (planes mode 0, yT)")
    else:
        two = variant == "dy+dyT"
        ds = 2 * C * L + pad
        dbuf = torch.randn(B, ds, device="cuda", generator=gen).to(dtype)
        dy = dbuf[:, :C * L]
        dyT = dbuf[:, C * L:2 * C * L] if two else None
        written = torch.zeros(B, xs, dtype=torch.bool, device="cuda")
        written[:, :C * L] = True
        out = Out(B * xs, dtype, written=written.view(-1))
        rc = lib.ss2d_dwconv3_act_planes(1, _p(x), xs, _p(w), _p(b), _p(dy), ds, _p(dyT), ds, out.ptr(), xs, None, 0, B, C, H, W,
                                         _DT[dtype], _stream())
        assert rc == 0, rc
        out.check("dpre")
        g = dy.double().view(B, C, H, W)
        if two:
            g = g + dyT.double().view(B, C, W, H).transpose(2, 3)
        ref, _ = ref_act(1, x, w, b, g)
        check_max(out.body.view(B, xs)[:, :C * L].view(B, C, H, W), ref, "silu", " (planes mode 1)")


# ---- ss2d_dwconv3_wgrad ---------------------------------------------------------------------------------------------------
def dw3_slabs(B, C, H, W):
    """Mirror of dwconv3_wgrad_slabs and the slab length of dwconv3_wgrad_kernel: -> (slabs, pixels per slab)."""
    total = B * H * W
    s = min(_cdiv(148 * 8, C), _cdiv(total, 256), 512)
    s = max(s, 1)
    return s, (_cdiv(total, s) + 3) & ~3


def run_dw3_wgrad(B, C, H, W, bias=True, seed=0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, C, H, W, device="cuda", generator=gen)
    dy = torch.randn(B, C, H, W, device="cuda", generator=gen)
    lib = _lib.lib()
    ws_bytes = int(lib.ss2d_dwconv3_wgrad_workspace_bytes(B, C, H, W))
    assert ws_bytes == C * dw3_slabs(B, C, H, W)[0] * 10 * 4
    ws = nan_workspace(ws_bytes)
    dW, db = Out(C * 9, F32), (Out(C, F32) if bias else None)
    rc = lib.ss2d_dwconv3_wgrad(_p(x), _p(dy), dW.ptr(), db.ptr() if db else None, B, C, H, W, _p(ws), ctypes.c_size_t(ws_bytes),
                                _stream())
    assert rc == 0, rc
    dW.check("dweight")
    ref, mag, rdb, dbmag = ref_wgrad_nhwc(_nhwc(x), _nhwc(dy), 3)
    check_abs(dW.body.view(C, 3, 3), ref, mag, "dw3_wgrad")
    if db is not None:
        db.check("dbias")
        check_abs(db.body, rdb, dbmag, "dw3_wgrad", " (bias)")
    return dW, db


@pytest.mark.parametrize("shape", [(2, 8, 12, 16), (2, 8, 11, 13), (3, 5, 1, 4), (2, 3, 7, 1), (24, 24, 28, 28)], ids=str)
def test_dwconv3_wgrad(shape):
    """The quad path (W % 4 == 0) and the scalar path, single-row and single-column images."""
    run_dw3_wgrad(*shape)
    run_dw3_wgrad(*shape, bias=False, seed=1)


@pytest.mark.parametrize("shape", [(2, 1, 257, 256), (3, 1, 1, 43691)], ids=["quads", "scalar"])
def test_dwconv3_wgrad_slab_cap_and_empty_slabs(shape):
    """C = 1: the slab count reaches its cap of 512, and the slab length rounded up to whole quads leaves trailing slabs
    with no pixels (they must still write their partials)."""
    B, C, H, W = shape
    slabs, per = dw3_slabs(B, C, H, W)
    assert slabs == 512 and (slabs - 1) * per >= B * H * W
    a = run_dw3_wgrad(*shape)
    b = run_dw3_wgrad(*shape)
    assert torch.equal(a[0].raw, b[0].raw) and torch.equal(a[1].raw, b[1].raw)


@pytest.mark.parametrize("off", [1, 2, 3])
def test_dwconv3_wgrad_op_accepts_misaligned_views(off):
    """ops.dwconv3_wgrad takes every contiguous fp32 tensor: views whose storage offset breaks the C ABI's 16-byte rule
    (W % 4 == 0) are copied before the call."""
    B, C, H, W = 2, 6, 8, 12
    n = B * C * H * W
    gen = torch.Generator(device="cuda").manual_seed(off)
    xb = torch.randn(n + 4, device="cuda", generator=gen)
    gb = torch.randn(n + 4, device="cuda", generator=gen)
    x = xb[off:off + n].view(B, C, H, W)
    dy = gb[4 - off:4 - off + n].view(B, C, H, W)
    assert x.is_contiguous() and x.data_ptr() % 16 != 0
    dW, db = ops.dwconv3_wgrad(x, dy, True)
    ref, mag, rdb, dbmag = ref_wgrad_nhwc(_nhwc(x), _nhwc(dy), 3)
    check_abs(dW.view(C, 3, 3), ref, mag, "dw3_wgrad")
    check_abs(db, rdb, dbmag, "dw3_wgrad", " (bias)")
