"""CPU tests of state passing in the selective scan (ss2d_scan_fwd_state / ss2d_scan_bwd_state): the entry points exist,
argument validation, the workspace query, and — from the SASS of the built library — that every STATE kernel is there and
that the ones the deterministic backward can launch issue no global atomic or reduction."""
import ctypes
import re

import pytest

from ceigm_unet_b200 import _lib
from test_deterministic_cpu import _GLOBAL_ATOMIC, _desc, _sass_functions, _ws

ERR_NULL, ERR_WORKSPACE, ERR_ALIGNMENT = -1, -6, -9


def test_symbols_exist():
    L = _lib.lib()
    assert hasattr(L, "ss2d_scan_fwd_state") and hasattr(L, "ss2d_scan_bwd_state")
    assert "ss2d_scan_fwd_state" in _lib.EXPORTS and "ss2d_scan_bwd_state" in _lib.EXPORTS


def _p(addr):
    return ctypes.c_void_p(addr)


# fake, never dereferenced device addresses: validation returns before anything is launched
GOOD = 0x10000
MIS = GOOD + 4        # 4-byte aligned, not 16-byte aligned


def _fwd(d, h0=GOOD, out=GOOD, u=GOOD):
    return _lib.lib().ss2d_scan_fwd_state(ctypes.byref(d), _p(u), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), None, None,
                                          _p(h0) if h0 else None, _p(out) if out else None, None, None, None)


def _bwd(d, h0=GOOD, dlast=GOOD, dh0=GOOD, dout=GOOD, ws_bytes=None):
    ws_bytes = _ws(d, 0) if ws_bytes is None else ws_bytes
    return _lib.lib().ss2d_scan_bwd_state(
        ctypes.byref(d), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), None, None, _p(h0) if h0 else None,
        _p(dout) if dout else None, _p(dlast) if dlast else None, None, _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD), _p(GOOD),
        None, None, _p(dh0) if dh0 else None, _p(GOOD), ctypes.c_size_t(ws_bytes), None)


def test_required_pointers():
    d = _desc()
    assert _fwd(d, u=0) == ERR_NULL
    assert _fwd(d, out=0) == ERR_NULL            # out, ckpt and last_state all NULL
    assert _bwd(d, dout=0) == ERR_NULL


def test_misaligned_states_are_rejected():
    d = _desc()
    assert _fwd(d, h0=MIS) == ERR_ALIGNMENT
    assert _bwd(d, h0=MIS) == ERR_ALIGNMENT
    assert _bwd(d, dlast=MIS) == ERR_ALIGNMENT
    assert _bwd(d, dh0=MIS) == ERR_ALIGNMENT


def test_workspace_is_checked_as_for_the_stateless_call():
    d = _desc()
    assert _bwd(d, ws_bytes=_ws(d, 0) - 4) == ERR_WORKSPACE


@pytest.mark.parametrize("shape", [
    (24, 768, 3136, 16, 4),      # vm_d192: scan_bwd2
    (2, 384, 784, 4, 4),         # generic scan_bwd
    (1, 64, 16384, 1, 4),        # d_state = 1, long rows
    (2, 64, 100, 40, 2),         # two state passes
])
@pytest.mark.parametrize("det", [0, 1])
def test_workspace_query_does_not_depend_on_states(shape, det):
    """One query serves both calls: the size takes no state argument, and a call with every state pointer set accepts exactly
    that size (a smaller one is refused before any launch)."""
    b, dim, L, N, G = shape
    d = _desc(b, dim, L, N, G, det=det)
    for have_ckpt in (0, 1):
        assert _ws(d, have_ckpt) > 0
    assert _bwd(d, ws_bytes=_ws(d, 0) - 16) == ERR_WORKSPACE


# backward kernel templates whose last two template flags are STATE, DET
_STATE_BWD = {"scan_bwd_kernel": 7, "scan_bwd2_kernel": 2, "scan_n1_bwd_kernel": 4, "scan_n1_bwd_rows_kernel": 2,
              "scan_par_bwd_kernel": 6}
# forward kernel templates whose last template flag is STATE
_STATE_FWD = {"scan_fwd_kernel": 6, "scan_fwdr_kernel": 4, "scan_fwd_carry_kernel": 2, "scan_fwd_fixup_kernel": 2,
              "scan_n1_fwd_kernel": 4, "scan_par_fwd_kernel": 6}


def _split(name):
    m = re.search(r"ss2d\d+(\w+?)I((?:L[a-z]+\d+E)+)EE", name)
    return (m.group(1), m.group(2)) if m else (None, None)


def _bwd_state(name):
    """STATE flag (second-to-last template flag) of a backward instantiation."""
    return re.findall(r"L[a-z]+\d+E", _split(name)[1])[-2] == "Lb1E"


def test_every_backward_template_has_its_state_instantiations():
    funcs = _sass_functions()
    bwd = {k: [n for n in funcs if _split(n)[0] == k and _bwd_state(n)] for k in _STATE_BWD}
    for k, per_det in _STATE_BWD.items():
        assert len(bwd[k]) == 2 * per_det, (k, bwd[k])          # DET = 0 and 1
    for k, count in _STATE_FWD.items():
        on = [n for n in funcs if _split(n)[0] == k and _split(n)[1].endswith("Lb1E")]
        assert len(on) == count, (k, on)


def test_state_det_instantiations_issue_no_global_atomics():
    funcs = _sass_functions()
    det_state = [n for n in funcs if _split(n)[0] in _STATE_BWD and _bwd_state(n) and _split(n)[1].endswith("Lb1E")]
    fwd_state = [n for n in funcs if _split(n)[0] in _STATE_FWD and _split(n)[1].endswith("Lb1E")]
    assert len(det_state) == sum(_STATE_BWD.values())
    offenders = {n: sorted(set(m.group(0) for m in _GLOBAL_ATOMIC.finditer(funcs[n]))) for n in det_state + fwd_state}
    offenders = {n: v for n, v in offenders.items() if v}
    assert not offenders, offenders


def test_state_instantiation_of_default_bwd2_still_reduces_in_l2():
    """The check above would pass vacuously if the pattern never matched: the non-deterministic STATE scan_bwd2 uses RED."""
    funcs = _sass_functions()
    plain = [n for n in funcs if _split(n)[0] == "scan_bwd2_kernel" and _bwd_state(n) and _split(n)[1].endswith("Lb0E")]
    assert plain and all(_GLOBAL_ATOMIC.search(funcs[n]) for n in plain)
