"""CPU tests of the tensor-core projections' C ABI (ss2d_linear_tc, ss2d_gate_proj_fwd and their *_supported predicates):
every error code that is returned before a tensor map is built, and the boundaries of both predicates. The values the
kernels compute are checked on the GPU by tests/test_tc_proj_gpu.py."""
import ctypes

import pytest
import torch

from ceigm_unet_b200 import _lib

OK, ERR_NULL, ERR_SHAPE, ERR_DTYPE, ERR_LAYOUT, ERR_UNSUPPORTED, ERR_ALIGNMENT = 0, -1, -2, -3, -5, -8, -9
F32, F16, BF16 = _lib.SS2D_F32, _lib.SS2D_F16, _lib.SS2D_BF16

# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000
SMEM = 227 * 1024


def _p(addr):
    return ctypes.c_void_p(addr) if addr else None


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
            self.keep.append(torch.zeros(1 << 16, device="cuda"))
            return self.keep[-1].data_ptr()
        self.n += 1
        return GOOD * (self.n + 1)


# ---- ss2d_linear_tc ----------------------------------------------------------------------------------------------------
def _parts(specs):
    """specs: (out, ld, n_cols, planes_L, act) per part."""
    arr = (_lib.LinearPart * max(len(specs), 1))()
    for i, (out, ld, n, pl, act) in enumerate(specs):
        arr[i].out, arr[i].ld, arr[i].n_cols, arr[i].planes_L, arr[i].act = out, ld, n, pl, act
    return arr


def _linear(A=GOOD, lda=32, W=GOOD, ldw=32, bias=0, M=128, N=32, K=32, dtype=F32, parts=None, n_parts=None):
    specs = [(GOOD, 32, 32, 0, 0)] if parts is None else parts
    n_parts = len(specs) if n_parts is None else n_parts
    arr = None if specs == "null" else _parts(specs)
    return _lib.lib().ss2d_linear_tc(_p(A), lda, _p(W), ldw, _p(bias), M, N, K, dtype, n_parts, arr, None)


def test_linear_required_pointers(no_launch):
    assert _linear(A=0) == ERR_NULL
    assert _linear(W=0) == ERR_NULL
    assert _linear(parts="null", n_parts=1) == ERR_NULL
    assert _linear(parts=[(0, 32, 32, 0, 0)]) == ERR_NULL
    assert _linear(N=48, parts=[(GOOD, 32, 32, 0, 0), (0, 16, 16, 0, 0)]) == ERR_NULL


@pytest.mark.parametrize("kw", [dict(M=0), dict(M=-1), dict(N=0), dict(K=0), dict(K=-4), dict(n_parts=0), dict(N=48),
                                dict(n_parts=5, parts=[(GOOD, 16, 16, 0, 0)] * 5, N=80)])
def test_linear_bad_shape(no_launch, kw):
    assert _linear(**kw) == ERR_SHAPE


@pytest.mark.parametrize("planes_L", [-1, 3, 256])
def test_linear_planes_must_divide_the_rows(no_launch, planes_L):
    """M = 128 rows are not whole images of 3 or 256 pixels; a negative L is no layout at all."""
    assert _linear(parts=[(GOOD, 0, 32, planes_L, 0)]) == ERR_SHAPE


@pytest.mark.parametrize("dtype", [F16, 3, -1])
def test_linear_bad_dtype(no_launch, dtype):
    assert _linear(dtype=dtype) == ERR_DTYPE


@pytest.mark.parametrize("n_cols", [8, 24, 40, 272])
def test_linear_unsupported_part_width(no_launch, n_cols):
    assert _linear(N=n_cols, parts=[(GOOD, 288, n_cols, 0, 0)], lda=32) == ERR_UNSUPPORTED


def test_linear_unsupported_k(no_launch):
    assert _linear(K=2, lda=4, ldw=4) == ERR_UNSUPPORTED                  # 8 bytes of K: not a 16-byte multiple
    assert _linear(K=4, lda=8, ldw=8, dtype=BF16) == ERR_UNSUPPORTED
    assert _linear(K=164, lda=164, ldw=164, N=256, parts=[(GOOD, 256, 256, 0, 0)]) == ERR_UNSUPPORTED   # W part too large


@pytest.mark.parametrize("kw", [dict(lda=28), dict(ldw=28), dict(lda=16), dict(ldw=16), dict(lda=4, ldw=4)])
def test_linear_overlapping_operand_rows(kw):
    """lda or ldw below K would make rows of A or W overlap: rejected before anything is launched."""
    mem = _Mem()
    before = _lib.launch_count()
    assert _linear(A=mem(), W=mem(), parts=[(mem(), 32, 32, 0, 0)], **kw) == ERR_LAYOUT
    assert _lib.launch_count() == before


@pytest.mark.parametrize("ld", [16, 28, 0])
def test_linear_overlapping_output_rows(ld):
    """A row-major part with ld < n_cols would write rows over each other. The check precedes the alignment check."""
    mem = _Mem()
    before = _lib.launch_count()
    assert _linear(A=mem(), W=mem(), parts=[(mem(), ld, 32, 0, 0)]) == ERR_LAYOUT
    assert _linear(A=mem(), W=mem(), N=48, parts=[(mem(), 0, 16, 128, 0), (mem(), ld, 32, 0, 0)]) == ERR_LAYOUT
    assert _lib.launch_count() == before


@pytest.mark.parametrize("spec", [(GOOD, 33, 32, 0, 0), (GOOD + 4, 32, 32, 0, 0)])
def test_linear_misaligned_rows_part(no_launch, spec):
    assert _linear(parts=[spec]) == ERR_ALIGNMENT


def _linear_fits(n, K, esize):
    kblocks = -(-K * esize // 128)
    w = (kblocks * n * 128 + 1023) & ~1023
    return w + 2 * 128 * 128 + 2048 + 8 * 32 * 128 <= SMEM


@pytest.mark.parametrize("dtype,esize", [(F32, 4), (BF16, 2)])
def test_linear_supported_boundaries(dtype, esize):
    sup = _lib.lib().ss2d_linear_tc_supported
    step = 16 // esize
    # part width: a multiple of 16 in [16, 256]
    for n in (-16, 0, 8, 15, 17, 24, 248, 264, 272, 512):
        assert sup(n, 4 * step, dtype) == 0, n
    for n in range(16, 257, 16):
        assert sup(n, 4 * step, dtype) == 1, n
    # K: positive, K * esize a multiple of 16 bytes
    for K in (-step, 0, 1, step - 1, step + 1, 3 * step // 2):
        assert sup(64, K, dtype) == 0, K
    # shared memory: the resident W part next to a two-stage A ring
    for n in (16, 48, 128, 240, 256):
        kmax = max(K for K in range(step, 16384, step) if _linear_fits(n, K, esize))
        assert sup(n, kmax, dtype) == 1 and sup(n, kmax + step, dtype) == 0, (n, kmax)
    assert max(K for K in range(step, 16384, step) if sup(256, K, dtype)) == (160 if esize == 4 else 320)


@pytest.mark.parametrize("dtype", [F16, 3, -1])
def test_linear_supported_rejects_other_dtypes(dtype):
    assert _lib.lib().ss2d_linear_tc_supported(64, 64, dtype) == 0


# ---- ss2d_gate_proj_fwd ------------------------------------------------------------------------------------------------
def _gate(ys=GOOD, K=2, tmask=0b10, lnw=GOOD, lnb=GOOD, z=GOOD, z_rs=None, W=GOOD, ldw=None, bias=GOOD, out=GOOD,
          out_rs=None, g=GOOD, g_rs=None, stats=GOOD, batch=1, D=64, H=4, Wd=4, L=None, C=16, dtype=F32):
    L = H * Wd if L is None else L
    z_rs = D if z_rs is None else z_rs
    ldw = D if ldw is None else ldw
    out_rs = C if out_rs is None else out_rs
    g_rs = D if g_rs is None else g_rs
    return _lib.lib().ss2d_gate_proj_fwd(_p(ys), K, ctypes.c_uint32(tmask), _p(lnw), _p(lnb), ctypes.c_float(1e-5), _p(z), z_rs,
                                         1, _p(W), ldw, _p(bias), _p(out), out_rs, _p(g), g_rs, _p(stats), batch, D, L, H, Wd,
                                         C, dtype, None)


def test_gate_required_pointers(no_launch):
    assert _gate(ys=0) == ERR_NULL
    assert _gate(W=0) == ERR_NULL
    assert _gate(out=0) == ERR_NULL
    assert _gate(C=0, g=0, W=0, out=0) == ERR_NULL           # C = 0: the gated tensor is the output


@pytest.mark.parametrize("kw", [dict(batch=0), dict(L=0, H=0), dict(H=0, L=16), dict(Wd=-4, L=16), dict(L=20)])
def test_gate_bad_shape(no_launch, kw):
    assert _gate(**kw) == ERR_SHAPE


@pytest.mark.parametrize("kw", [dict(D=32), dict(D=96), dict(D=320), dict(K=0), dict(K=9), dict(C=8), dict(C=24), dict(C=272),
                                dict(dtype=F16), dict(dtype=3), dict(lnw=0), dict(D=256, C=0)])
def test_gate_unsupported(no_launch, kw):
    assert _gate(**kw) == ERR_UNSUPPORTED


@pytest.mark.parametrize("H,Wd", [(6, 4), (4, 6), (2, 8), (8, 2), (5, 7)])
@pytest.mark.parametrize("C", [0, 16])
def test_gate_image_sides_must_be_multiples_of_4(H, Wd, C):
    """The planes are read as TMA boxes over 16-byte aligned image rows: H % 4 or W % 4 is reported as unsupported before
    any tensor map is built, whatever the driver would make of such a map."""
    mem = _Mem()
    before = _lib.launch_count()
    args = dict(ys=mem(), lnw=mem(), lnb=mem(), z=mem(), W=mem(), bias=mem(), out=mem() if C else 0, g=mem(), stats=mem())
    assert _gate(H=H, Wd=Wd, C=C, **args) == ERR_UNSUPPORTED
    assert _lib.launch_count() == before


@pytest.mark.parametrize("kw", [dict(out_rs=8), dict(out_rs=0), dict(z_rs=60), dict(z_rs=0), dict(g_rs=32), dict(g_rs=0),
                                dict(C=0, out=0, g_rs=48)])
def test_gate_overlapping_rows(kw):
    """out_row_stride < C, z_row_stride < D or g_row_stride < D would make rows overlap: rejected before any launch."""
    mem = _Mem()
    before = _lib.launch_count()
    args = dict(ys=mem(), lnw=mem(), lnb=mem(), z=mem(), W=mem(), bias=mem(), out=mem(), g=mem(), stats=mem())
    args.update(kw)
    assert _gate(**args) == ERR_LAYOUT
    assert _lib.launch_count() == before


def test_gate_strides_of_absent_operands_are_ignored(no_launch):
    """Without z or g_out their strides mean nothing; C = 0 ignores out's stride. Such calls get past the layout check (and fail
    later on the fake pointers' alignment)."""
    assert _gate(z=0, z_rs=0, g=0, g_rs=0, out=GOOD + 4) == ERR_ALIGNMENT
    assert _gate(C=0, W=0, out=0, out_rs=0, g=GOOD + 4) == ERR_ALIGNMENT


@pytest.mark.parametrize("kw", [dict(out=GOOD + 4), dict(z=GOOD + 8), dict(g=GOOD + 4), dict(lnw=GOOD + 4), dict(lnb=GOOD + 4),
                                dict(out_rs=18), dict(z_rs=66), dict(g_rs=65)])
def test_gate_misaligned(no_launch, kw):
    assert _gate(**kw) == ERR_ALIGNMENT


# the (D, C) pairs ss2d_gate_proj_supported admits, from the shared-memory arithmetic of gp_smem_bytes
_GATE_TABLE = {
    (64, F32): range(0, 257, 16), (64, BF16): range(0, 257, 16),
    (128, F32): range(0, 257, 16), (128, BF16): range(0, 257, 16),
    (192, F32): range(0, 97, 16), (192, BF16): range(0, 113, 16),
    (256, F32): (16, 32), (256, BF16): (),
}


@pytest.mark.parametrize("K", [1, 2, 4, 8])
def test_gate_supported_table(K):
    sup = _lib.lib().ss2d_gate_proj_supported
    admitted = {(D, dt): tuple(C for C in range(0, 257, 16) if sup(D, C, K, dt)) for D in (64, 128, 192, 256) for dt in (F32, BF16)}
    assert admitted == {k: tuple(v) for k, v in _GATE_TABLE.items()}
    assert sum(len(v) for v in admitted.values()) == 85


def test_gate_supported_boundaries():
    sup = _lib.lib().ss2d_gate_proj_supported
    for dt in (F32, BF16):
        for D in (0, -64, 32, 96, 100, 160, 320, 512):
            assert sup(D, 16, 2, dt) == 0, D
        for K in (0, -1, 9, 16):
            assert sup(64, 16, K, dt) == 0, K
        for K in range(1, 9):
            assert sup(64, 16, K, dt) == 1 and sup(64, 0, K, dt) == 1, K
        for C in (-16, 8, 15, 17, 24, 264, 272):
            assert sup(64, C, 2, dt) == 0, C
    for dt in (F16, 3, -1):
        assert sup(64, 16, 2, dt) == 0, dt
