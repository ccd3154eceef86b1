"""CPU tests of the fused SS2D epilogue's C ABI (ss2d_out_gate_fwd / _bwd, ss2d_group_gate_fwd / _bwd and the LayerNorm rule of
ss2d_gate_proj_fwd): argument validation returns its error code before anything is launched, and the partial-buffer query.
The values the kernels compute are checked on the GPU by tests/test_epilogue_gpu.py."""
import ctypes

import pytest
import torch

from ceigm_unet_b200 import _lib

OK, ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_LAYOUT, ERR_WORKSPACE, ERR_UNSUPPORTED = 0, -1, -2, -3, -5, -6, -8

# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000


def _p(addr):
    return ctypes.c_void_p(addr) if addr else None


def _partials(batch, L):
    return int(_lib.lib().ss2d_out_gate_bwd_partials(batch, L))


def _fwd(ys=GOOD, K=4, lnw=GOOD, lnb=GOOD, z=GOOD, out=GOOD, stats=GOOD, batch=2, D=16, H=4, W=6, L=None, tmask=0b1010,
         z_dtype=_lib.SS2D_F32, out_dtype=_lib.SS2D_F32):
    L = H * W if L is None else L
    return _lib.lib().ss2d_out_gate_fwd(_p(ys), K, _p(lnw), _p(lnb), _p(z), D, 1, _p(out), _p(stats), batch, D, L,
                                        ctypes.c_float(1e-5), z_dtype, out_dtype, H, W, ctypes.c_uint32(tmask), None)


def _bwd(ys=GOOD, K=4, lnw=GOOD, lnb=GOOD, z=GOOD, dout=GOOD, stats=GOOD, dy=GOOD, dz=GOOD, dw=GOOD, db=GOOD, batch=2, D=16,
         H=4, W=6, L=None, tmask=0b1010, two_planes=0, n_partials=None, z_dtype=_lib.SS2D_F32, out_dtype=_lib.SS2D_F32):
    L = H * W if L is None else L
    n_partials = _partials(batch, L) if n_partials is None else n_partials
    return _lib.lib().ss2d_out_gate_bwd(_p(ys), K, _p(lnw), _p(lnb), _p(z), D, 1, _p(dout), _p(stats), _p(dy), _p(dz), D, _p(dw),
                                        _p(db), n_partials, batch, D, L, z_dtype, out_dtype, H, W, ctypes.c_uint32(tmask),
                                        two_planes, None)


def _plane_arr(plane_of):
    return None if plane_of is None else (ctypes.c_int32 * max(len(plane_of), 1))(*plane_of)


def _gfwd(ys=GOOD, G=2, plane_of=(0, 1), lnw=GOOD, lnb=GOOD, z=GOOD, out=GOOD, stats=GOOD, batch=2, D=16, H=4, W=6, L=None,
          z_dtype=_lib.SS2D_F32, out_dtype=_lib.SS2D_F32):
    L = H * W if L is None else L
    return _lib.lib().ss2d_group_gate_fwd(_p(ys), G, _plane_arr(plane_of), ctypes.c_uint32(0b10), _p(lnw), _p(lnb), _p(z), G * D,
                                          0, D, _p(out), G * D, _p(stats), batch, D, L, ctypes.c_float(1e-5), z_dtype, out_dtype,
                                          H, W, None)


def _gbwd(ys=GOOD, G=2, plane_of=(0, 1), lnw=GOOD, lnb=GOOD, z=GOOD, dout=GOOD, stats=GOOD, dy=GOOD, dz=GOOD, dw=GOOD,
          db=GOOD, batch=2, D=16, H=4, W=6, L=None, n_partials=None, z_dtype=_lib.SS2D_F32, out_dtype=_lib.SS2D_F32):
    L = H * W if L is None else L
    n_partials = _partials(batch, L) if n_partials is None else n_partials
    return _lib.lib().ss2d_group_gate_bwd(_p(ys), G, _plane_arr(plane_of), ctypes.c_uint32(0b10), _p(lnw), _p(lnb), _p(z),
                                          G * D, 0, D, _p(dout), G * D, _p(stats), _p(dy), _p(dz), G * D, _p(dw), _p(db),
                                          n_partials, batch, D, L, z_dtype, out_dtype, H, W, None)


@pytest.fixture
def no_launch():
    """Asserts that the test's calls launched nothing."""
    before = _lib.launch_count()
    yield
    assert _lib.launch_count() == before


class _Mem:
    """Addresses for the calls a library without the check under test would launch. Without a GPU they are fake; with one
    they are zeroed device buffers large enough for the tiny shapes used with them, so that such a library still launches
    in bounds."""

    def __init__(self):
        self.keep, self.n = [], 0

    def __call__(self):
        if torch.cuda.is_available():
            self.keep.append(torch.zeros(1 << 14, device="cuda"))
            return self.keep[-1].data_ptr()
        self.n += 1
        return GOOD * (self.n + 1)


@pytest.mark.parametrize("batch,L", [(1, 1), (1, 32), (1, 33), (2, 3136), (24, 3136), (3, 5), (592, 1), (593, 1), (18, 1056),
                                     (19, 1000), (100, 3136)])
def test_bwd_partials(batch, L):
    assert _partials(batch, L) == min(batch * -(-L // 32), 592)


def test_bwd_partials_of_empty_shapes_is_zero():
    assert _partials(0, 16) == 0 and _partials(4, 0) == 0 and _partials(-1, 16) == 0


def test_max_width():
    assert _lib.lib().ss2d_out_gate_max_width(0) == 1664
    assert _lib.lib().ss2d_out_gate_max_width(1) == 832


def test_width_above_the_limit_is_unsupported(no_launch):
    fwd_max, bwd_max = _lib.lib().ss2d_out_gate_max_width(0), _lib.lib().ss2d_out_gate_max_width(1)
    assert _fwd(D=fwd_max + 1) == ERR_UNSUPPORTED
    assert _bwd(D=bwd_max + 1) == ERR_UNSUPPORTED
    assert _bwd(D=fwd_max) == ERR_UNSUPPORTED
    assert _gfwd(D=fwd_max + 1) == ERR_UNSUPPORTED
    assert _gbwd(D=bwd_max + 1) == ERR_UNSUPPORTED


@pytest.mark.parametrize("delta", [-1, 1, 100])
def test_wrong_partial_count_is_a_workspace_error(no_launch, delta):
    n = _partials(2, 24)
    assert _bwd(n_partials=n + delta) == ERR_WORKSPACE
    assert _gbwd(n_partials=n + delta) == ERR_WORKSPACE


def test_two_dy_planes_need_several_planes_and_a_transposed_one(no_launch):
    assert _bwd(K=1, tmask=1, two_planes=1) == ERR_UNSUPPORTED
    assert _bwd(K=4, tmask=0, two_planes=1) == ERR_UNSUPPORTED


def test_image_must_match_seqlen(no_launch):
    assert _fwd(L=25) == ERR_SHAPE                       # H * W = 24
    assert _bwd(L=25) == ERR_SHAPE
    assert _bwd(L=25, tmask=0, two_planes=1) == ERR_SHAPE
    assert _fwd(H=0, L=24, tmask=1) == ERR_SHAPE
    assert _gfwd(L=25) == ERR_SHAPE
    assert _gbwd(L=25) == ERR_SHAPE
    assert _gfwd(W=0, L=24) == ERR_SHAPE


@pytest.mark.parametrize("K", [0, -1, 9])
def test_plane_count_out_of_range(no_launch, K):
    assert _fwd(K=K) == ERR_SHAPE
    assert _bwd(K=K) == ERR_SHAPE


@pytest.mark.parametrize("G", [0, 5])
def test_group_count_out_of_range(no_launch, G):
    plane_of = tuple(range(max(G, 1)))
    assert _gfwd(G=G, plane_of=plane_of) == ERR_SHAPE
    assert _gbwd(G=G, plane_of=plane_of) == ERR_SHAPE


@pytest.mark.parametrize("kw", [dict(batch=0), dict(D=0), dict(D=-3)])
def test_non_positive_sizes(no_launch, kw):
    assert _fwd(**kw) == ERR_SHAPE
    assert _bwd(**kw) == ERR_SHAPE
    assert _gfwd(**kw) == ERR_SHAPE
    assert _gbwd(**kw) == ERR_SHAPE


@pytest.mark.parametrize("kw", [dict(z_dtype=3), dict(z_dtype=-1), dict(out_dtype=3), dict(out_dtype=-1)])
def test_bad_dtype(no_launch, kw):
    assert _fwd(**kw) == ERR_DTYPE
    assert _bwd(**kw) == ERR_DTYPE
    assert _gfwd(**kw) == ERR_DTYPE
    assert _gbwd(**kw) == ERR_DTYPE


@pytest.mark.parametrize("plane_of", [(0, 2), (-1, 0), (0, 1, 3), (4, 0, 1, 2)])
def test_plane_index_out_of_range(no_launch, plane_of):
    G = len(plane_of)
    assert _gfwd(G=G, plane_of=plane_of) == ERR_LAYOUT
    assert _gbwd(G=G, plane_of=plane_of) == ERR_LAYOUT


@pytest.mark.parametrize("plane_of", [(0, 0), (1, 1), (0, 1, 1), (2, 0, 2), (3, 1, 0, 1), (0, 0, 0, 0)])
def test_repeated_plane_is_rejected(no_launch, plane_of):
    """Two groups on one plane would write the same dy plane concurrently in the backward."""
    mem = _Mem()
    G = len(plane_of)
    args = dict(G=G, plane_of=plane_of, batch=1, D=16, H=4, W=4)
    assert _gfwd(ys=mem(), lnw=mem(), lnb=mem(), z=mem(), out=mem(), stats=mem(), **args) == ERR_LAYOUT
    assert _gbwd(ys=mem(), lnw=mem(), lnb=mem(), z=mem(), dout=mem(), stats=mem(), dy=mem(), dz=mem(), dw=mem(), db=mem(),
                 **args) == ERR_LAYOUT


def test_layernorm_bias_without_weight_is_unsupported(no_launch):
    """Every epilogue kernel applies the bias only together with the weight: the combination is rejected, not dropped."""
    mem = _Mem()
    for K, tmask, D in ((1, 1, 16), (4, 0b1010, 40)):          # the small and the tiled kernels
        args = dict(K=K, tmask=tmask, D=D, batch=1, H=4, W=4)
        assert _fwd(ys=mem(), lnw=0, lnb=mem(), z=mem(), out=mem(), stats=mem(), **args) == ERR_UNSUPPORTED
        assert _bwd(ys=mem(), lnw=0, lnb=mem(), z=mem(), dout=mem(), stats=mem(), dy=mem(), dz=mem(), dw=mem(), db=mem(),
                    **args) == ERR_UNSUPPORTED
    args = dict(G=2, batch=1, D=16, H=4, W=4)
    assert _gfwd(ys=mem(), lnw=0, lnb=mem(), z=mem(), out=mem(), stats=mem(), **args) == ERR_UNSUPPORTED
    assert _gbwd(ys=mem(), lnw=0, lnb=mem(), z=mem(), dout=mem(), stats=mem(), dy=mem(), dz=mem(), dw=mem(), db=mem(),
                 **args) == ERR_UNSUPPORTED


def test_gate_proj_layernorm_bias_without_weight_is_unsupported(no_launch):
    """ss2d_gate_proj_fwd (the TMA-fed epilogue) follows the same rule, and checks it before the operands' alignment."""
    L = _lib.lib()
    D, H, W = 64, 4, 4
    assert L.ss2d_gate_proj_supported(D, 0, 2, _lib.SS2D_F32) == 1

    def call(lnw, z):
        return L.ss2d_gate_proj_fwd(_p(GOOD), 2, ctypes.c_uint32(0b10), _p(lnw), _p(GOOD), ctypes.c_float(1e-5), _p(z), D, 1,
                                    None, 0, None, None, 0, _p(GOOD), D, _p(GOOD), 1, D, H * W, H, W, 0, _lib.SS2D_F32, None)
    assert call(0, GOOD + 4) == ERR_UNSUPPORTED
    assert call(GOOD, GOOD + 4) == -9                         # with the weight, the misaligned z is what is reported


def test_required_pointers(no_launch):
    for kw in ("ys", "out"):
        assert _fwd(**{kw: 0}) == ERR_NULL, kw
    for kw in ("ys", "dout", "stats", "dy", "dw", "db"):
        assert _bwd(**{kw: 0}) == ERR_NULL, kw
    for kw in ("ys", "z", "out", "plane_of"):
        assert _gfwd(**{kw: None if kw == "plane_of" else 0}) == ERR_NULL, kw
    for kw in ("ys", "z", "dout", "stats", "dy", "dz", "dw", "db", "plane_of"):
        assert _gbwd(**{kw: None if kw == "plane_of" else 0}) == ERR_NULL, kw
