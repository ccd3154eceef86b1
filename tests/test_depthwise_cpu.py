"""CPU tests of the depthwise convolution C ABI (ss2d_dwnhwc_stencil, ss2d_dwnhwc_wgrad, ss2d_dwconv3_act,
ss2d_dwconv3_act_planes, ss2d_dwconv3_wgrad and the workspace queries): every argument check returns its error code before
anything is launched. The values the kernels compute are checked on the GPU by tests/test_depthwise_gpu.py."""
import ctypes

import pytest

from ceigm_unet_b200 import _lib

OK, ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_WORKSPACE, ERR_UNSUPPORTED, ERR_ALIGNMENT = 0, -1, -2, -3, -6, -8, -9
F32, F16, BF16 = _lib.SS2D_F32, _lib.SS2D_F16, _lib.SS2D_BF16

# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000


def _p(addr):
    return ctypes.c_void_p(addr) if addr else None


@pytest.fixture(autouse=True)
def no_launch():
    """Every call in this file is refused: none may launch."""
    before = _lib.launch_count()
    yield
    assert _lib.launch_count() == before


# ---- ss2d_dwnhwc_stencil --------------------------------------------------------------------------------------------------
def _stencil(x=GOOD, aux=GOOD, y=GOOD, nseg=1, cbeg=(0, 8), ks=(3,), w=(GOOD,), b=(GOOD,), flip=0, epi=0, batch=1, H=4, W=4,
             C=8, dtype=F32):
    ca = None if cbeg is None else (ctypes.c_int32 * len(cbeg))(*cbeg)
    ka = None if ks is None else (ctypes.c_int32 * len(ks))(*ks)
    wa = None if w is None else (ctypes.c_void_p * len(w))(*[a or None for a in w])
    ba = None if b is None else (ctypes.c_void_p * len(b))(*[a or None for a in b])
    return _lib.lib().ss2d_dwnhwc_stencil(_p(x), _p(aux), _p(y), nseg, ca, ka, wa, ba, flip, epi, batch, H, W, C, dtype, None)


def test_stencil_null_pointers():
    for kw in ("x", "y"):
        assert _stencil(**{kw: 0}) == ERR_NULL, kw
    for kw in ("cbeg", "ks", "w"):
        assert _stencil(**{kw: None}) == ERR_NULL, kw
    assert _stencil(epi=3, aux=0) == ERR_NULL                          # the GELU' epilogue needs aux
    assert _stencil(w=(0,)) == ERR_NULL                                # a k > 1 segment needs its weight
    assert _stencil(nseg=2, cbeg=(0, 4, 8), ks=(1, 7), w=(0, 0), b=(0, 0)) == ERR_NULL


@pytest.mark.parametrize("epi", [-1, 4])
def test_stencil_epilogue_out_of_range(epi):
    assert _stencil(epi=epi) == ERR_UNSUPPORTED


@pytest.mark.parametrize("k", [2, 4, -1, 9])
def test_stencil_kernel_size(k):
    assert _stencil(ks=(k,)) == ERR_UNSUPPORTED
    assert _stencil(nseg=2, cbeg=(0, 4, 8), ks=(3, k), w=(GOOD, GOOD), b=(GOOD, GOOD)) == ERR_UNSUPPORTED


@pytest.mark.parametrize("kw", [dict(batch=0), dict(H=0), dict(W=-1), dict(C=0),
                                dict(nseg=0), dict(nseg=5, cbeg=(0, 2, 4, 6, 7, 8), ks=(3,) * 5, w=(GOOD,) * 5, b=(GOOD,) * 5),
                                dict(batch=2, H=32768, W=32768), dict(batch=1, H=65536, W=32768),
                                dict(cbeg=(1, 8)), dict(cbeg=(0, 4)), dict(cbeg=(0, 12)),
                                dict(nseg=2, cbeg=(0, 4, 4), ks=(3, 3), w=(GOOD, GOOD), b=(GOOD, GOOD), C=4),
                                dict(nseg=3, cbeg=(0, 6, 4, 8), ks=(3, 3, 3), w=(GOOD,) * 3, b=(GOOD,) * 3),
                                dict(nseg=2, cbeg=(0, 0, 8), ks=(3, 3), w=(GOOD, GOOD), b=(GOOD, GOOD))], ids=str)
def test_stencil_bad_shape(kw):
    """Non-positive sizes, 0 or 5 segments, B H W >= 2^31, cbeg[0] != 0, cbeg[nseg] != C, non-increasing bounds."""
    assert _stencil(**kw) == ERR_SHAPE


@pytest.mark.parametrize("dtype", [3, -1])
def test_stencil_dtype(dtype):
    assert _stencil(dtype=dtype) == ERR_DTYPE


@pytest.mark.parametrize("kw", [dict(w=(GOOD + 2,)), dict(b=(GOOD + 2,)), dict(x=GOOD + 4), dict(y=GOOD + 4),
                                dict(aux=GOOD + 4, epi=3), dict(x=GOOD + 2, dtype=F16), dict(y=GOOD + 2, dtype=BF16),
                                dict(aux=GOOD + 6, dtype=F16, epi=3)], ids=str)
def test_stencil_alignment(kw):
    """Weights and biases 4-byte aligned; x, aux and y aligned to a channel pair (8 bytes fp32, 4 bytes 16-bit)."""
    assert _stencil(**kw) == ERR_ALIGNMENT


# ---- ss2d_dwnhwc_wgrad ----------------------------------------------------------------------------------------------------
def _wgq(batch=1, H=4, W=4, channels=8, k=3):
    return int(_lib.lib().ss2d_dwnhwc_wgrad_workspace_bytes(batch, H, W, channels, k))


def _wgrad(x=GOOD, g=GOOD, c0=0, c1=8, k=3, dW=GOOD, db=GOOD, batch=1, H=4, W=4, C=8, dtype=F32, ws=GOOD, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = max(_wgq(batch, H, W, max(c1 - c0, 1), k if k in (3, 5, 7) else 3), 4)
    return _lib.lib().ss2d_dwnhwc_wgrad(_p(x), _p(g), c0, c1, k, _p(dW), _p(db), batch, H, W, C, dtype, _p(ws),
                                        ctypes.c_size_t(ws_bytes), None)


@pytest.mark.parametrize("batch,H,W,channels,k", [(1, 4, 4, 8, 3), (3, 17, 9, 20, 5), (64, 56, 56, 64, 7), (1, 1, 1, 1, 3),
                                                  (8192, 128, 1, 3, 3)])
def test_wgrad_workspace_bytes(batch, H, W, channels, k):
    """One slab of partials per 16-row group, at most 65535 slabs."""
    slabs = min(-(-(batch * H) // 16), 65535)
    assert _wgq(batch, H, W, channels, k) == slabs * channels * (k * k + 1) * 4


@pytest.mark.parametrize("kw", [dict(k=0), dict(k=1), dict(k=2), dict(k=4), dict(k=9), dict(batch=0), dict(H=0), dict(W=-2),
                                dict(channels=0)], ids=str)
def test_wgrad_workspace_query_is_zero_when_unsupported(kw):
    assert _wgq(**kw) == 0


def test_wgrad_null_pointers():
    for kw in ("x", "g", "dW"):
        assert _wgrad(**{kw: 0}) == ERR_NULL, kw


@pytest.mark.parametrize("kw", [dict(batch=0), dict(H=0), dict(W=0), dict(C=0), dict(c0=-1), dict(c0=4, c1=4), dict(c0=6, c1=4),
                                dict(c1=9), dict(batch=2, H=32768, W=32768)], ids=str)
def test_wgrad_bad_shape(kw):
    assert _wgrad(**kw) == ERR_SHAPE


@pytest.mark.parametrize("k", [0, 1, 2, 4, 9])
def test_wgrad_kernel_size(k):
    assert _wgrad(k=k) == ERR_UNSUPPORTED


@pytest.mark.parametrize("dtype", [3, -1])
def test_wgrad_dtype(dtype):
    assert _wgrad(dtype=dtype) == ERR_DTYPE


@pytest.mark.parametrize("kw", [dict(x=GOOD + 2), dict(g=GOOD + 2), dict(x=GOOD + 1, dtype=F16), dict(g=GOOD + 1, dtype=BF16),
                                dict(dW=GOOD + 2), dict(db=GOOD + 2)], ids=str)
def test_wgrad_alignment(kw):
    """x and g aligned to their element size, dweight / dbias to 4 bytes."""
    assert _wgrad(**kw) == ERR_ALIGNMENT


def test_wgrad_workspace():
    need = _wgq()
    assert need > 0
    assert _wgrad(ws=0) == ERR_WORKSPACE
    assert _wgrad(ws_bytes=need - 4) == ERR_WORKSPACE
    assert _wgrad(ws_bytes=0) == ERR_WORKSPACE
    assert _wgrad(ws=GOOD + 2) == ERR_WORKSPACE


# ---- ss2d_dwconv3_act -----------------------------------------------------------------------------------------------------
def _act(mode=0, x=GOOD, w=GOOD, b=GOOD, dy=GOOD, y=GOOD, batch=1, C=4, H=4, W=8, dtype=F32):
    return _lib.lib().ss2d_dwconv3_act(mode, _p(x), _p(w), _p(b), _p(dy), _p(y), batch, C, H, W, dtype, None)


def test_act_null_pointers():
    for kw in ("x", "w", "y"):
        assert _act(**{kw: 0}) == ERR_NULL, kw
    assert _act(mode=1, dy=0) == ERR_NULL


@pytest.mark.parametrize("mode", [-1, 3])
def test_act_mode_out_of_range(mode):
    assert _act(mode=mode) == ERR_UNSUPPORTED


@pytest.mark.parametrize("kw", [dict(batch=0), dict(C=-1), dict(H=0), dict(W=0)], ids=str)
def test_act_bad_shape(kw):
    assert _act(**kw) == ERR_SHAPE


@pytest.mark.parametrize("dtype", [3, -1])
def test_act_dtype(dtype):
    assert _act(dtype=dtype) == ERR_DTYPE


@pytest.mark.parametrize("kw", [dict(x=GOOD + 4), dict(y=GOOD + 8), dict(dy=GOOD + 4, mode=1), dict(x=GOOD + 4, dtype=F16),
                                dict(y=GOOD + 2, dtype=BF16), dict(x=GOOD + 2, W=7), dict(y=GOOD + 1, W=7, dtype=F16),
                                dict(w=GOOD + 2)], ids=str)
def test_act_alignment(kw):
    """W % 4 == 0: x, dy and y aligned to four elements (the pixel quads move as one access), else to one; weights 4 bytes."""
    assert _act(**kw) == ERR_ALIGNMENT


# ---- ss2d_dwconv3_act_planes ----------------------------------------------------------------------------------------------
def _planes(mode=0, x=GOOD, xbs=128, w=GOOD, b=GOOD, dy=GOOD, dybs=256, dyT=GOOD, dyTbs=256, y=GOOD, ybs=256, yT=GOOD, yTbs=256,
            batch=1, C=4, H=4, W=8, dtype=F32):
    return _lib.lib().ss2d_dwconv3_act_planes(mode, _p(x), xbs, _p(w), _p(b), _p(dy), dybs, _p(dyT), dyTbs, _p(y), ybs, _p(yT),
                                              yTbs, batch, C, H, W, dtype, None)


def test_planes_null_pointers():
    for kw in ("x", "w", "y"):
        assert _planes(**{kw: 0}) == ERR_NULL, kw
    assert _planes(mode=1, dy=0) == ERR_NULL


@pytest.mark.parametrize("kw", [dict(mode=-1), dict(mode=2), dict(H=6), dict(W=10), dict(H=1, W=1)], ids=str)
def test_planes_unsupported(kw):
    """Modes 0 and 1 only; H and W must be multiples of 4 (whole pixel quads in both orientations)."""
    assert _planes(**kw) == ERR_UNSUPPORTED


@pytest.mark.parametrize("kw", [dict(batch=0), dict(C=0), dict(H=0), dict(W=-4), dict(C=65536), dict(batch=65536)], ids=str)
def test_planes_bad_shape(kw):
    """Non-positive sizes; C and batch above 65535 (grid dimensions y and z)."""
    assert _planes(**kw) == ERR_SHAPE


@pytest.mark.parametrize("dtype", [3, -1])
def test_planes_dtype(dtype):
    assert _planes(dtype=dtype) == ERR_DTYPE


@pytest.mark.parametrize("kw", [dict(x=GOOD + 4), dict(y=GOOD + 8), dict(yT=GOOD + 4), dict(dy=GOOD + 4, mode=1),
                                dict(dyT=GOOD + 12, mode=1), dict(x=GOOD + 4, dtype=F16), dict(yT=GOOD + 2, dtype=BF16),
                                dict(xbs=130), dict(ybs=258), dict(yTbs=257), dict(dybs=254, mode=1), dict(dyTbs=2, mode=1),
                                dict(xbs=130, dtype=F16), dict(w=GOOD + 2)], ids=str)
def test_planes_alignment(kw):
    """Pointers and batch strides in whole pixel quads (16 bytes fp32, 8 bytes 16-bit); weights 4 bytes."""
    assert _planes(**kw) == ERR_ALIGNMENT


# ---- ss2d_dwconv3_wgrad ---------------------------------------------------------------------------------------------------
def _dw3q(batch=1, C=4, H=4, W=8):
    return int(_lib.lib().ss2d_dwconv3_wgrad_workspace_bytes(batch, C, H, W))


def _dw3(x=GOOD, dy=GOOD, dW=GOOD, db=GOOD, batch=1, C=4, H=4, W=8, ws=GOOD, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = max(_dw3q(batch, C, H, W), 4)
    return _lib.lib().ss2d_dwconv3_wgrad(_p(x), _p(dy), _p(dW), _p(db), batch, C, H, W, _p(ws), ctypes.c_size_t(ws_bytes), None)


@pytest.mark.parametrize("batch,C,H,W", [(1, 4, 4, 8), (24, 192, 56, 56), (2, 1, 257, 256), (1, 2000, 3, 3), (1, 1, 1, 1)])
def test_dw3_workspace_bytes(batch, C, H, W):
    """C slabs of ten partials: about 8 CTAs per SM of a 148-SM B200, at least 256 pixels per slab, at most 512 slabs."""
    total = batch * H * W
    slabs = max(min(-(-1184 // C), -(-total // 256), 512), 1)
    assert _dw3q(batch, C, H, W) == C * slabs * 10 * 4


@pytest.mark.parametrize("kw", [dict(batch=0), dict(C=0), dict(H=-1), dict(W=0)], ids=str)
def test_dw3_workspace_query_of_empty_shapes_is_zero(kw):
    assert _dw3q(**kw) == 0


def test_dw3_null_pointers():
    for kw in ("x", "dy", "dW"):
        assert _dw3(**{kw: 0}) == ERR_NULL, kw


@pytest.mark.parametrize("kw", [dict(batch=0), dict(C=0), dict(H=0), dict(W=-1), dict(C=65536)], ids=str)
def test_dw3_bad_shape(kw):
    assert _dw3(**kw) == ERR_SHAPE


@pytest.mark.parametrize("kw", [dict(x=GOOD + 4), dict(dy=GOOD + 4), dict(x=GOOD + 8), dict(dy=GOOD + 12), dict(x=GOOD + 2, W=7),
                                dict(dy=GOOD + 1, W=7), dict(dW=GOOD + 2), dict(db=GOOD + 2)], ids=str)
def test_dw3_alignment(kw):
    """W % 4 == 0: x and dy are read as float4 pixel quads and must be 16-byte aligned (4-byte otherwise); dweight / dbias
    4-byte. A contiguous view at a storage offset that is not a multiple of four elements is refused, not read misaligned."""
    assert _dw3(**kw) == ERR_ALIGNMENT


def test_dw3_workspace():
    need = _dw3q()
    assert need > 0
    assert _dw3(ws=0) == ERR_WORKSPACE
    assert _dw3(ws_bytes=need - 4) == ERR_WORKSPACE
    assert _dw3(ws=GOOD + 2) == ERR_WORKSPACE
