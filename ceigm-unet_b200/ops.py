"""Tensor-level wrappers over the C ABI: build a `ss2d_scan_desc` from torch tensors, allocate outputs with
torch on the current device/stream (exactly what the reference's host code does with ATen,
kernels/selective_scan/csrc/selective_scan/cus/selective_scan.cpp:217-233) and call libss2d_b200.so.

Error behaviour mirrors the reference's TORCH_CHECKs (selective_scan.cpp:165-215, 251-305): wrong dtype,
device, stride or shape raises RuntimeError before anything is launched.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Tuple

import torch

from . import _lib

_DT = {torch.float32: _lib.SS2D_F32, torch.float16: _lib.SS2D_F16, torch.bfloat16: _lib.SS2D_BF16}


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require(cond: bool, msg: str) -> None:
    if not cond:
        raise RuntimeError(msg)


def _round4(n: int) -> int:
    return (n + 3) & ~3


class ScanProblem:
    """Validated view of one selective-scan call.

    SCAN layout (reference extension API): u, delta (B, Dt, L); B, C (B, G, N, L) or (B, N, L).
    NATURAL layout (fused cross-scan/merge): pass hw=(H, W) and dirs (one direction 1..4 per group); u is
    (B, Dt | D, H*W) flattened images, u_mod=D shares one input across the K groups.
    """

    def __init__(self, u, delta, A, B, C, D=None, delta_bias=None, delta_softplus=False, *, out_float=False,
                 hw: Optional[Tuple[int, int]] = None, dirs: Optional[Sequence[int]] = None, u_mod: int = 0):
        _require(u.dtype in _DT, "u must be float32, float16 or bfloat16")                     # cpp:167
        _require(A.dtype == torch.float32, "A must be float32")                                 # cpp:168
        _require(delta.dtype == u.dtype and B.dtype == u.dtype and C.dtype == u.dtype,
                 "delta, B and C must have the dtype of u")                                     # cpp:170-172
        for name, t in (("u", u), ("delta", delta), ("A", A), ("B", B), ("C", C)):
            _require(t.is_cuda, f"Expected {name}.is_cuda() to be true")                        # cpp:174-178
        _require(u.dim() == 3 and delta.dim() == 3, "u and delta must be (batch, dim, seqlen)")
        _require(u.stride(-1) == 1 or u.size(-1) == 1, "u must be contiguous in its last dimension")          # cpp:180
        _require(delta.stride(-1) == 1 or delta.size(-1) == 1, "delta must be contiguous in its last dimension")
        self.squeeze_BC = B.dim() == 3
        if self.squeeze_BC:
            B, C = B.unsqueeze(1), C.unsqueeze(1)
        batch, dim, L = delta.shape
        N, G = A.shape[1], B.shape[1]
        _require(dim % G == 0, "dims should be dividable by n_groups")                          # cpp:190
        _require(N <= _lib.MAX_DSTATE, "selective_scan only supports state dimension <= 256")   # cpp:191
        _require(tuple(A.shape) == (dim, N) and A.is_contiguous(), "A must be a contiguous (dim, dstate) tensor")
        _require(tuple(B.shape) == (batch, G, N, L), "B must be (batch, n_groups, dstate, seqlen)")           # cpp:196
        _require(tuple(C.shape) == (batch, G, N, L), "C must be (batch, n_groups, dstate, seqlen)")           # cpp:198
        _require(B.stride(-1) == 1 or B.size(-1) == 1, "B must be contiguous in its last dimension")          # cpp:197
        _require(C.stride(-1) == 1 or C.size(-1) == 1, "C must be contiguous in its last dimension")          # cpp:199
        if u_mod:
            _require(tuple(u.shape) == (batch, u_mod, L) and dim % u_mod == 0, "u must be (batch, u_mod, seqlen)")
        else:
            _require(tuple(u.shape) == (batch, dim, L), "u must be (batch, dim, seqlen)")       # cpp:193
        for name, t in (("D", D), ("delta_bias", delta_bias)):
            if t is not None:
                _require(t.dtype == torch.float32, f"{name} must be float32")                   # cpp:203, 211
                _require(t.is_cuda, f"Expected {name}.is_cuda() to be true")
                _require(tuple(t.shape) == (dim,) and t.is_contiguous(), f"{name} must be a contiguous (dim,) tensor")
        self.u, self.delta, self.A, self.B, self.C, self.D, self.bias = u, delta, A, B, C, D, delta_bias
        self.batch, self.dim, self.L, self.N, self.G = batch, dim, L, N, G
        self.out_dtype = torch.float32 if out_float else u.dtype
        self.softplus = bool(delta_softplus)
        self.hw, self.dirs, self.u_mod = hw, dirs, int(u_mod)
        d = _lib.ScanDesc()
        d.batch, d.dim, d.seqlen, d.dstate, d.n_groups = batch, dim, L, N, G
        d.io_dtype, d.out_dtype, d.delta_softplus = _DT[u.dtype], _DT[self.out_dtype], int(self.softplus)
        if hw is not None:
            _require(dirs is not None and len(dirs) == G and G <= _lib.MAX_GROUP_DIRS, "one direction per group needed")
            _require(hw[0] * hw[1] == L, "H * W must equal seqlen")
            d.layout, d.H, d.W = _lib.LAYOUT_NATURAL, hw[0], hw[1]
            for i, k in enumerate(dirs):
                d.dirs[i] = int(k)
        else:
            d.layout = _lib.LAYOUT_SCAN
        d.u_batch_stride, d.u_dim_stride = u.stride(0), u.stride(1)
        d.delta_batch_stride, d.delta_dim_stride = delta.stride(0), delta.stride(1)
        d.B_batch_stride, d.B_group_stride, d.B_state_stride = B.stride(0), B.stride(1), B.stride(2)
        d.C_batch_stride, d.C_group_stride, d.C_state_stride = C.stride(0), C.stride(1), C.stride(2)
        d.u_dim_modulo = self.u_mod
        self.desc = d
        self.ckpt_floats = int(_lib.lib().ss2d_scan_ckpt_floats(ctypes.byref(d)))
        # 16-bit I/O: the kernels compute in fp32 either way, but only fp32 operands are staged by TMA and reach the fast
        # backward (csrc/scan_bwd2.cu); 16-bit tensors go through an index-mapped staging path that is 3 x slower
        # (fwd 1.47 vs 0.43 ms, bwd 3.21 vs 1.12 ms at B = 24, Dt = 768, L = 3136, N = 16). The scan is compute-bound there, so
        # the 16-bit call is routed through the fp32 kernels with cast passes around them (HBM-bound, ~15 % of the call):
        # identical arithmetic (the 16-bit values are exact in fp32), results rounded once on the way out.
        self._upcast = u.dtype != torch.float32
        self._inner = None

    def _fp32_twin(self):
        if self._inner is None:
            self._inner = ScanProblem(self.u.float(), self.delta.float(), self.A, self.B.float(), self.C.float(), self.D, self.bias,
                                      self.softplus, out_float=True, hw=self.hw, dirs=self.dirs, u_mod=self.u_mod)
        return self._inner

    def _state_arg(self, t: Optional[torch.Tensor], name: str) -> Optional[torch.Tensor]:
        """h0 / dlast: None, or a (batch, dim, dstate) fp32 CUDA tensor (made contiguous)."""
        if t is None:
            return None
        _require(t.is_cuda and t.dtype == torch.float32, f"{name} must be a float32 CUDA tensor")
        _require(tuple(t.shape) == (self.batch, self.dim, self.N), f"{name} must be (batch, dim, dstate)")
        t = t.contiguous()
        if t.data_ptr() % 16:
            t = t.clone()
        return t

    def _gate_arg(self, t: torch.Tensor, name: str, dtype) -> torch.Tensor:
        """z / out / dout of a gated call: a (batch, dim, seqlen) CUDA tensor of `dtype`, made contiguous (the C ABI gives the
        gate operands out's strides)."""
        _require(not self.u_mod, "the output gate needs one dout plane per channel (u_mod == 0)")
        _require(t.is_cuda and t.dtype == dtype, f"{name} must be a CUDA tensor of dtype {dtype}")
        _require(tuple(t.shape) == (self.batch, self.dim, self.L), f"{name} must be (batch, dim, seqlen)")
        return t.contiguous()

    # ---- forward ----
    def forward(self, want_state: bool = True, h0: Optional[torch.Tensor] = None, z: Optional[torch.Tensor] = None):
        """-> (out (B, Dt, L), x). `x` has the reference's shape convention (B, Dt, 1, 2N): x[:, :, -1, 1::2] is the
        final state; the chunk checkpoints for the backward live in front of it in the same storage.
        h0: optional (B, Dt, N) fp32 state before the first position (default zeros); a backward of this forward's `x` must
        be given the same h0.
        z: optional (B, Dt, L) gate of u's dtype: a third value out_z = out * silu(z) (out's dtype) is returned."""
        h0 = self._state_arg(h0, "h0")
        if z is not None:
            z = self._gate_arg(z, "z", self.u.dtype)
        if self._upcast:
            res = self._fp32_twin().forward(want_state, h0, None if z is None else z.float())
            return (res[0].to(self.out_dtype), res[1]) + tuple(r.to(self.out_dtype) for r in res[2:])
        d, dev = self.desc, self.delta.device
        out = torch.empty((self.batch, self.dim, self.L), dtype=self.out_dtype, device=dev)
        d.out_batch_stride, d.out_dim_stride = out.stride(0), out.stride(1)
        x = ckpt = last = None
        if want_state:
            head = _round4(self.ckpt_floats)
            buf = torch.empty(head + self.batch * self.dim * 2 * self.N, dtype=torch.float32, device=dev)
            ckpt = buf
            x = buf[head:].view(self.batch, self.dim, 1, 2 * self.N)
            last = x
            d.last_state_interleaved = 1
        out_z = None
        with torch.cuda.device(dev):
            if z is not None:
                out_z = torch.empty_like(out)
                rc = _lib.lib().ss2d_scan_fwd_gated(ctypes.byref(d), _ptr(self.u), _ptr(self.delta), _ptr(self.A), _ptr(self.B),
                                                    _ptr(self.C), _ptr(self.D), _ptr(self.bias), _ptr(h0), _ptr(z), _ptr(out),
                                                    _ptr(out_z), _ptr(ckpt), _ptr(last), _stream(dev))
            else:
                rc = _lib.lib().ss2d_scan_fwd_state(ctypes.byref(d), _ptr(self.u), _ptr(self.delta), _ptr(self.A), _ptr(self.B),
                                                    _ptr(self.C), _ptr(self.D), _ptr(self.bias), _ptr(h0), _ptr(out), _ptr(ckpt),
                                                    _ptr(last), _stream(dev))
        _lib.check(rc, "ss2d_scan_fwd")
        return (out, x) if z is None else (out, x, out_z)

    def _ckpt_from_x(self, x: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        """Recover the checkpoint buffer that `forward` placed in front of `x` (None if x is foreign)."""
        if x is None or x.dtype != torch.float32 or not x.is_cuda:
            return None
        head = _round4(self.ckpt_floats)
        total = head + self.batch * self.dim * 2 * self.N
        if x.storage_offset() != head or x.untyped_storage().nbytes() != total * 4 or not x.is_contiguous():
            return None
        return torch.empty(0, dtype=torch.float32, device=x.device).set_(x.untyped_storage(), 0, (head,), (1,))

    # ---- backward ----
    def backward(self, dout, x=None, h0: Optional[torch.Tensor] = None, dlast: Optional[torch.Tensor] = None,
                 want_dh0: bool = False, z: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None):
        """-> [du, ddelta, dA, dB, dC, dD, ddelta_bias] with the reference's dtypes (selective_scan.cpp:319-347):
        du/ddelta in u's dtype, dA/dD/ddelta_bias fp32, dB/dC accumulated in fp32 then cast to B's dtype.

        Under torch.use_deterministic_algorithms(True) (warn_only included) the kernels that take no global atomics run:
        the seven gradients are then bit-identical from call to call on the same GPU model (ss2d_scan_desc.deterministic).

        State passing: h0 is the forward's initial state (None: zeros), dlast the gradient of the final state (None: zeros).
        With any of h0 / dlast / want_dh0 given, an eighth entry dh0 (B, Dt, N) fp32 (or None unless want_dh0) is appended.

        Output gate: with z (the forward's gate) and out (the forward's ungated output y, required with z), dout is the
        gradient of out_z = out * silu(z), and dz (z's dtype) is appended after the seven gradients, before dh0."""
        d, dev = self.desc, self.delta.device
        dch = self.u_mod if self.u_mod else self.dim
        _require(dout.is_cuda and dout.dtype == self.out_dtype, "dout must be a CUDA tensor of out's dtype")
        _require(tuple(dout.shape) == (self.batch, dch, self.L), "dout must be (batch, dim, seqlen)")
        h0, dlast = self._state_arg(h0, "h0"), self._state_arg(dlast, "dlast")
        stateful = h0 is not None or dlast is not None or want_dh0
        gated = z is not None
        if gated:
            _require(out is not None, "out (the forward's ungated output) is required with z")
            z, out = self._gate_arg(z, "z", self.u.dtype), self._gate_arg(out, "out", self.out_dtype)
            dout = self._gate_arg(dout, "dout", self.out_dtype)
        if self._upcast:
            grads = self._fp32_twin().backward(dout.float(), x, h0, dlast, want_dh0, z=None if z is None else z.float(),
                                               out=None if out is None else out.float())
            du, ddelta, dA, dB, dC, dD, dbias = grads[:7]
            dB, dC = dB.to(self.B.dtype), dC.to(self.C.dtype)
            if self.squeeze_BC:
                dB, dC = dB[:, 0], dC[:, 0]
            rest = grads[7:]
            if gated:
                rest = [rest[0].to(self.u.dtype)] + rest[1:]
            return [du.to(self.u.dtype), ddelta.to(self.delta.dtype), dA, dB, dC, dD, dbias] + rest
        if dout.stride(-1) != 1:                                  # csms6s.py:360-361 does the same before calling bwd
            dout = dout.contiguous()
        d.out_batch_stride, d.out_dim_stride = dout.stride(0), dout.stride(1)
        # du / ddelta are written with u's / delta's strides: normalise strided views to dense tensors first
        u, delta = self.u, self.delta
        if not u.is_contiguous():
            u = u.contiguous()
            d.u_batch_stride, d.u_dim_stride = u.stride(0), u.stride(1)
        if not delta.is_contiguous():
            delta = delta.contiguous()
            d.delta_batch_stride, d.delta_dim_stride = delta.stride(0), delta.stride(1)
        du = torch.empty((self.batch, self.dim, self.L), dtype=u.dtype, device=dev) if self.u_mod else torch.empty_like(u)
        ddelta = torch.empty_like(delta)
        # one zero-fill launch for every accumulator (the live GM-UNet regime is launch-bound: 104 scan calls per step):
        # dB | dC always; for d_state = 1 also dA | dD | ddelta_bias, which the lean kernel then adds into directly —
        # except in deterministic mode, where those three are overwritten by the fixed-order finalize pass
        det = torch.are_deterministic_algorithms_enabled()
        d.deterministic = int(det)
        nbc = self.batch * self.G * self.N * self.L
        small = self.N == 1 and not det
        extra = self.dim * (self.N + 2) if small else 0
        zbuf = torch.zeros(2 * nbc + extra, dtype=torch.float32, device=dev)
        dB, dC = zbuf[:nbc].view(self.batch, self.G, self.N, self.L), zbuf[nbc:2 * nbc].view(self.batch, self.G, self.N, self.L)
        if small:
            dA = zbuf[2 * nbc:2 * nbc + self.dim * self.N].view(self.dim, self.N)
            dD = zbuf[2 * nbc + self.dim * self.N:2 * nbc + self.dim * (self.N + 1)] if self.D is not None else None
            dbias = zbuf[2 * nbc + self.dim * (self.N + 1):] if self.bias is not None else None
            d.grads_prezeroed = 1
        else:
            dA = torch.empty_like(self.A)
            dD = torch.empty_like(self.D) if self.D is not None else None
            dbias = torch.empty_like(self.bias) if self.bias is not None else None
            d.grads_prezeroed = 0
        ckpt = self._ckpt_from_x(x)
        L = _lib.lib()
        ws_query = L.ss2d_scan_bwd_gated_workspace_bytes if gated else L.ss2d_scan_bwd_workspace_bytes
        ws_bytes = int(ws_query(ctypes.byref(d), 1 if ckpt is not None else 0))
        ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=dev)
        dh0 = torch.empty((self.batch, self.dim, self.N), dtype=torch.float32, device=dev) if want_dh0 else None
        dz = torch.empty_like(z) if gated else None
        with torch.cuda.device(dev):
            if gated:
                rc = L.ss2d_scan_bwd_gated(ctypes.byref(d), _ptr(u), _ptr(delta), _ptr(self.A), _ptr(self.B), _ptr(self.C),
                                           _ptr(self.D), _ptr(self.bias), _ptr(h0), _ptr(z), _ptr(out), _ptr(dout), _ptr(dlast),
                                           _ptr(ckpt), _ptr(du), _ptr(ddelta), _ptr(dA), _ptr(dB), _ptr(dC), _ptr(dD),
                                           _ptr(dbias), _ptr(dz), _ptr(dh0), _ptr(ws), ctypes.c_size_t(ws_bytes), _stream(dev))
            else:
                rc = L.ss2d_scan_bwd_state(ctypes.byref(d), _ptr(u), _ptr(delta), _ptr(self.A), _ptr(self.B),
                                           _ptr(self.C), _ptr(self.D), _ptr(self.bias), _ptr(h0), _ptr(dout), _ptr(dlast),
                                           _ptr(ckpt), _ptr(du), _ptr(ddelta), _ptr(dA), _ptr(dB), _ptr(dC), _ptr(dD),
                                           _ptr(dbias), _ptr(dh0), _ptr(ws), ctypes.c_size_t(ws_bytes), _stream(dev))
        _lib.check(rc, "ss2d_scan_bwd")
        if self.B.dtype != torch.float32:
            dB, dC = dB.to(self.B.dtype), dC.to(self.C.dtype)
        if self.squeeze_BC:
            dB, dC = dB[:, 0], dC[:, 0]
        grads = [du, ddelta, dA, dB, dC, dD, dbias] + ([dz] if gated else [])
        return grads + [dh0] if stateful else grads


# ---- recurrent step ----------------------------------------------------------------------------
def state_update(state, x, dt, A, B, C, D=None, z=None, dt_bias=None, dt_softplus=False) -> torch.Tensor:
    """One step of the selective scan, `state` updated in place (ss2d_state_update) -> out (batch, dim) in x's dtype.
    state: fp32 (batch, dim, dstate) contiguous, 16-byte aligned; x, dt, z: (batch, dim); B, C: (batch, dstate) or
    (batch, n_groups, dstate), all of x's dtype; A: fp32 (dim, dstate) contiguous; D, dt_bias: fp32 (dim) or None.
    x, dt and z are made contiguous unless they already are (the C ABI gives them one shared row stride)."""
    _require(x.dtype in _DT, "x must be float32, float16 or bfloat16")
    for name, t in (("state", state), ("x", x), ("dt", dt), ("A", A), ("B", B), ("C", C), ("D", D), ("z", z), ("dt_bias", dt_bias)):
        if t is not None:
            _require(t.is_cuda, f"Expected {name}.is_cuda() to be true")
            _require(t.device == state.device, f"{name} must be on the device of state")
    _require(state.dtype == torch.float32 and state.dim() == 3, "state must be a float32 (batch, dim, dstate) tensor")
    batch, dim, N = state.shape
    _require(state.is_contiguous() and state.data_ptr() % 16 == 0, "state must be contiguous and 16-byte aligned (it is updated in place)")
    _require(N <= _lib.MAX_DSTATE, "selective_state_update only supports state dimension <= 256")
    _require(A.dtype == torch.float32 and tuple(A.shape) == (dim, N) and A.is_contiguous(), "A must be a contiguous float32 (dim, dstate) tensor")
    for name, t in (("x", x), ("dt", dt), ("z", z)):
        if t is not None:
            _require(t.dtype == x.dtype and tuple(t.shape) == (batch, dim), f"{name} must be (batch, dim) of x's dtype")
    if B.dim() == 2:
        B, C = B.unsqueeze(1), C.unsqueeze(1)
    _require(B.dim() == 3 and tuple(C.shape) == tuple(B.shape), "B and C must both be (batch, dstate) or (batch, n_groups, dstate)")
    G = B.shape[1]
    _require(tuple(B.shape) == (batch, G, N) and G > 0 and dim % G == 0, "B and C must be (batch, n_groups, dstate), dim % n_groups == 0")
    _require(B.dtype == x.dtype and C.dtype == x.dtype, "B and C must have x's dtype")
    for name, t in (("D", D), ("dt_bias", dt_bias)):
        if t is not None:
            _require(t.dtype == torch.float32 and tuple(t.shape) == (dim,) and t.is_contiguous(), f"{name} must be a contiguous float32 (dim,) tensor")
    B = B if B.stride(-1) == 1 else B.contiguous()
    C = C if C.stride(-1) == 1 else C.contiguous()
    x, dt = x.contiguous(), dt.contiguous()
    z = None if z is None else z.contiguous()
    out = torch.empty((batch, dim), dtype=x.dtype, device=x.device)
    d = _lib.StepDesc()
    d.batch, d.dim, d.dstate, d.n_groups = batch, dim, N, G
    d.io_dtype, d.dt_softplus, d.io_batch_stride = _DT[x.dtype], int(bool(dt_softplus)), dim
    d.B_batch_stride, d.B_group_stride = B.stride(0), B.stride(1)
    d.C_batch_stride, d.C_group_stride = C.stride(0), C.stride(1)
    with torch.cuda.device(state.device):
        rc = _lib.lib().ss2d_state_update(ctypes.byref(d), _ptr(state), _ptr(x), _ptr(dt), _ptr(A), _ptr(B), _ptr(C), _ptr(D),
                                          _ptr(dt_bias), _ptr(z), _ptr(out), _stream(state.device))
    _lib.check(rc, "ss2d_state_update")
    return out


# ---- stand-alone permutations ------------------------------------------------------------------
def cross_scan(x: torch.Tensor, dirs: Sequence[int]) -> torch.Tensor:
    """x (B, C, H, W) -> (B, K, C, H*W), plane k traversed in direction dirs[k] (csms6s.py:11-206)."""
    _require(x.is_cuda and x.dtype in _DT and x.dim() == 4, "x must be a CUDA (B, C, H, W) float tensor")
    x = x.contiguous()
    Bn, Cn, H, W = x.shape
    K = len(dirs)
    out = torch.empty((Bn, K, Cn, H * W), dtype=x.dtype, device=x.device)
    arr = (ctypes.c_int32 * K)(*[int(k) for k in dirs])
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_cross_scan(_ptr(x), _ptr(out), Bn, Cn, H, W, K, arr, _DT[x.dtype], _stream(x.device))
    _lib.check(rc, "ss2d_cross_scan")
    return out


def cross_merge(ys: torch.Tensor, hw: Tuple[int, int], dirs: Sequence[int]) -> torch.Tensor:
    """ys (B, K, C, L) in scan order -> (B, C, L) natural order, summed over K."""
    _require(ys.is_cuda and ys.dtype in _DT and ys.dim() == 4, "ys must be a CUDA (B, K, C, L) float tensor")
    ys = ys.contiguous()
    Bn, K, Cn, L = ys.shape
    H, W = hw
    _require(H * W == L and K == len(dirs), "shape mismatch in cross_merge")
    out = torch.empty((Bn, Cn, L), dtype=ys.dtype, device=ys.device)
    arr = (ctypes.c_int32 * K)(*[int(k) for k in dirs])
    with torch.cuda.device(ys.device):
        rc = _lib.lib().ss2d_cross_merge(_ptr(ys), _ptr(out), Bn, Cn, H, W, K, arr, _DT[ys.dtype], _stream(ys.device))
    _lib.check(rc, "ss2d_cross_merge")
    return out


# ---- fused epilogue ----------------------------------------------------------------------------
def out_gate_max_D(backward: bool) -> int:
    return int(_lib.lib().ss2d_out_gate_max_width(1 if backward else 0))


def out_gate_fwd(ys, ln_w, ln_b, z, z_act: bool, eps: float, out_dtype, hw=(0, 0), tmask: int = 0):
    """ys (B, K, D, L) fp32 natural order; z (B, L, D) view with stride(-1)==1 or None -> out (B, L, D), mean_rstd."""
    _require(ys.is_cuda and ys.dtype == torch.float32 and ys.is_contiguous(), "ys must be contiguous CUDA fp32")
    Bn, K, D, L = ys.shape
    out = torch.empty((Bn, L, D), dtype=out_dtype, device=ys.device)
    stats = torch.empty((Bn, L, 2), dtype=torch.float32, device=ys.device)
    zrs, zdt = 0, _lib.SS2D_F32
    if z is not None:
        _require(z.stride(-1) == 1 and z.shape[-1] == D and z.dtype in _DT, "z rows must be contiguous (.., D)")
        zrs, zdt = _row_stride(z, Bn, L), _DT[z.dtype]
    H, W = int(hw[0]), int(hw[1])
    if (H * W == L and H % 4 == 0 and W % 4 == 0 and out_dtype in (torch.float32, torch.bfloat16) and (z is None or z.dtype == out_dtype)
            and (z is None or (z.data_ptr() % 16 == 0 and (zrs * z.element_size()) % 16 == 0))
            and bool(_lib.lib().ss2d_gate_proj_supported(D, 0, K, _DT[out_dtype]))):
        # TMA-fed variant (csrc/gate_proj_tc.cu with C = 0): the K planes stream through a ring of tiled TMA boxes, a warp owns
        # whole pixel rows in the statistics / gate pass. Same results; 146 -> 129 us at B = 24, K = 4, D = 192, 56^2 (fp32 rows).
        with torch.cuda.device(ys.device):
            rc = _lib.lib().ss2d_gate_proj_fwd(_ptr(ys), K, ctypes.c_uint32(tmask), _ptr(ln_w), _ptr(ln_b), ctypes.c_float(eps), _ptr(z), zrs,
                                               int(z_act), None, 0, None, None, 0, _ptr(out), D, _ptr(stats), Bn, D, L, H, W, 0,
                                               _DT[out_dtype], _stream(ys.device))
        _lib.check(rc, "ss2d_gate_proj_fwd")
        return out, stats
    with torch.cuda.device(ys.device):
        rc = _lib.lib().ss2d_out_gate_fwd(_ptr(ys), K, _ptr(ln_w), _ptr(ln_b), _ptr(z), zrs, int(z_act), _ptr(out),
                                          _ptr(stats), Bn, D, L, ctypes.c_float(eps), zdt, _DT[out_dtype],
                                          int(hw[0]), int(hw[1]), ctypes.c_uint32(tmask), _stream(ys.device))
    _lib.check(rc, "ss2d_out_gate_fwd")
    return out, stats


def _row_stride(z, Bn, L) -> int:
    """Row stride of a (B, L, D) or (B, H, W, D) view whose rows are uniformly spaced in memory."""
    flat = z.reshape(Bn * L, z.shape[-1]) if z.is_contiguous() else None
    if flat is not None:
        return z.shape[-1]
    rs = z.stride(-2)
    # uniform spacing check: every outer stride must be the product of inner extents times rs
    exp = rs
    for dim in range(z.dim() - 2, -1, -1):
        _require(z.stride(dim) == exp, "z must be a uniformly strided view of (rows, D)")
        exp *= z.shape[dim]
    return rs


def out_gate_bwd(ys, ln_w, ln_b, z, z_act: bool, dout, stats, dz_out: Optional[torch.Tensor], hw=(0, 0), tmask: int = 0,
                 two_planes: bool = False):
    """-> dy (B, D, L) fp32, dln_w, dln_b. dz is written into `dz_out` (a (B, L, D) uniformly strided view), or not computed
    when `dz_out` is None.
    two_planes (K > 1, tmask != 0): dy is (B, 2, D, L) — the merged gradient in natural and in transposed pixel order."""
    Bn, K, D, L = ys.shape
    dout = dout.contiguous()
    dy = torch.empty((Bn, 2, D, L) if two_planes else (Bn, D, L), dtype=torch.float32, device=ys.device)
    npart = int(_lib.lib().ss2d_out_gate_bwd_partials(Bn, L))
    part = torch.empty((2, npart, D), dtype=torch.float32, device=ys.device)
    zrs, zdt, dzrs = 0, _lib.SS2D_F32, 0
    if z is not None:
        zrs, zdt = _row_stride(z, Bn, L), _DT[z.dtype]
        if dz_out is not None:
            _require(dz_out.dtype == z.dtype, "dz_out must have z's dtype (the kernel writes dz in it)")
            dzrs = _row_stride(dz_out, Bn, L)
    with torch.cuda.device(ys.device):
        rc = _lib.lib().ss2d_out_gate_bwd(_ptr(ys), K, _ptr(ln_w), _ptr(ln_b), _ptr(z), zrs, int(z_act), _ptr(dout),
                                          _ptr(stats), _ptr(dy), _ptr(dz_out) if z is not None else None, dzrs,
                                          _ptr(part[0]), _ptr(part[1]), npart, Bn, D, L, zdt, _DT[dout.dtype],
                                          int(hw[0]), int(hw[1]), ctypes.c_uint32(tmask), 1 if two_planes else 0, _stream(ys.device))
    _lib.check(rc, "ss2d_out_gate_bwd")
    sums = part.sum(dim=1)
    return dy, sums[0], sums[1]


# ---- grouped epilogue: the four SS2Ds of a GroupMambaLayer in one launch ------------------------------
def group_gate_fwd(ys, plane_of, tbits: int, ln_w, ln_b, z, eps: float, out_dtype, hw):
    """ys (B, G, D, L) fp32 planes (group g in plane plane_of[g]; bit p of tbits: plane p in transposed pixel order);
    ln_w / ln_b (G, D) fp32; z (B, L, G*D) raw gates, contiguous -> out (B, L, G*D) = concat_g LN_g(ys_g) * SiLU(z_g), stats."""
    _require(ys.is_cuda and ys.dtype == torch.float32 and ys.is_contiguous() and ys.dim() == 4, "ys must be contiguous CUDA fp32 (B, G, D, L)")
    Bn, G, D, L = ys.shape
    _require(z.is_contiguous() and tuple(z.shape) == (Bn, L, G * D) and z.dtype in _DT, "z must be a contiguous (B, L, G*D) tensor")
    _require(ln_w.is_contiguous() and ln_b.is_contiguous() and tuple(ln_w.shape) == (G, D), "ln_w / ln_b must be (G, D)")
    out = torch.empty((Bn, L, G * D), dtype=out_dtype, device=ys.device)
    stats = torch.empty((G, Bn, L, 2), dtype=torch.float32, device=ys.device)
    arr = (ctypes.c_int32 * G)(*[int(p) for p in plane_of])
    with torch.cuda.device(ys.device):
        rc = _lib.lib().ss2d_group_gate_fwd(_ptr(ys), G, arr, ctypes.c_uint32(tbits), _ptr(ln_w), _ptr(ln_b), _ptr(z), G * D, 0, D,
                                            _ptr(out), G * D, _ptr(stats), Bn, D, L, ctypes.c_float(eps), _DT[z.dtype],
                                            _DT[out_dtype], int(hw[0]), int(hw[1]), _stream(ys.device))
    _lib.check(rc, "ss2d_group_gate_fwd")
    return out, stats


def group_gate_bwd(ys, plane_of, tbits: int, ln_w, ln_b, z, dout, stats, hw):
    """-> dy (B, G, D, L) fp32 (plane p in its own pixel order), dz (B, L, G*D) like z, dln_w (G, D), dln_b (G, D)."""
    Bn, G, D, L = ys.shape
    dout = dout.contiguous()
    dy = torch.empty((Bn, G, D, L), dtype=torch.float32, device=ys.device)
    dz = torch.empty_like(z)
    npart = int(_lib.lib().ss2d_out_gate_bwd_partials(Bn, L))
    part = torch.empty((2, G, npart, D), dtype=torch.float32, device=ys.device)
    arr = (ctypes.c_int32 * G)(*[int(p) for p in plane_of])
    with torch.cuda.device(ys.device):
        rc = _lib.lib().ss2d_group_gate_bwd(_ptr(ys), G, arr, ctypes.c_uint32(tbits), _ptr(ln_w), _ptr(ln_b), _ptr(z), G * D, 0, D,
                                            _ptr(dout), G * D, _ptr(stats), _ptr(dy), _ptr(dz), G * D, _ptr(part[0]),
                                            _ptr(part[1]), npart, Bn, D, L, _DT[z.dtype], _DT[dout.dtype], int(hw[0]),
                                            int(hw[1]), _stream(ys.device))
    _lib.check(rc, "ss2d_group_gate_bwd")
    sums = part.sum(dim=2)
    return dy, dz, sums[0], sums[1]


# ---- tall-skinny weight gradient ---------------------------------------------------------------
def wgrad_ts_supported(M: int, N: int) -> bool:
    return 0 < M <= 256 and 0 < N <= 256 and ((M + 3) // 4) * ((N + 3) // 4) <= 256


def wgrad_ts(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """dW (M, N) fp32 = sum over (b, r) of dy[b, r, :, None] * x[b, r, None, :].
    dy (B, R, M), x (B, R, N): arbitrary strided views (a (B, C, L) tensor is passed as .transpose(1, 2))."""
    _require(dy.is_cuda and x.is_cuda and dy.dim() == 3 and x.dim() == 3 and dy.shape[:2] == x.shape[:2],
             "wgrad_ts: dy (B, R, M) and x (B, R, N) must be CUDA tensors with the same leading sizes")
    _require(dy.dtype in _DT and x.dtype in _DT, "wgrad_ts: float32, float16 or bfloat16 operands")
    Bn, R, M = dy.shape
    N = x.shape[2]
    _require(wgrad_ts_supported(M, N), "wgrad_ts: M x N too large for the tall-skinny kernel (use a library GEMM)")
    dev = dy.device
    L = _lib.lib()
    ws_bytes = int(L.ss2d_wgrad_ts_workspace_bytes(Bn, R, M, N))
    ws = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device=dev)
    dW = torch.empty((M, N), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = L.ss2d_wgrad_ts(_ptr(dy), _ptr(x), _ptr(dW), Bn, R, M, N, dy.stride(0), dy.stride(1), dy.stride(2),
                             x.stride(0), x.stride(1), x.stride(2), _DT[dy.dtype], _DT[x.dtype], _ptr(ws),
                             ctypes.c_size_t(ws_bytes), _stream(dev))
    _lib.check(rc, "ss2d_wgrad_ts")
    return dW


def dwconv3_act(mode: int, x: torch.Tensor, weight: torch.Tensor, bias, dy=None) -> torch.Tensor:
    """Depthwise 3 x 3 convolution (padding 1) fused with SiLU. mode 0: SiLU(b + conv(x)); 1: dy * SiLU'(b + conv(x));
    2: conv with the flipped kernel, no bias (input gradient of mode 1's result). x, dy: (B, C, H, W) contiguous."""
    _require(x.is_cuda and x.dim() == 4 and x.is_contiguous() and x.dtype in _DT, "dwconv3_act: contiguous CUDA (B, C, H, W) tensor")
    _require(dy is None or (dy.shape == x.shape and dy.dtype == x.dtype and dy.is_contiguous()), "dwconv3_act: dy must match x")
    Bn, C, H, W = x.shape
    w32 = weight.detach().float().contiguous()
    b32 = None if bias is None else bias.detach().float().contiguous()
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_dwconv3_act(mode, _ptr(x), _ptr(w32), _ptr(b32), _ptr(dy), _ptr(y), Bn, C, H, W, _DT[x.dtype],
                                         _stream(x.device))
    _lib.check(rc, "ss2d_dwconv3_act")
    return y


def dwconv3_act_planes_ok(x: torch.Tensor) -> bool:
    return x.dim() == 4 and x.shape[2] % 4 == 0 and x.shape[3] % 4 == 0 and x.shape[0] <= 65535 and x.shape[1] <= 65535


def dwconv3_act_planes_fwd(x: torch.Tensor, weight: torch.Tensor, bias) -> torch.Tensor:
    """u (B, 2 C, H W) = [SiLU(b + conv(x)) in natural pixel order | the same image transposed]: the two input planes of a
    K = 4 SS2D scan written by the convolution kernel itself (no permuted copy, no cat)."""
    _require(x.is_cuda and x.is_contiguous() and x.dtype in _DT and dwconv3_act_planes_ok(x), "dwconv3_act_planes: contiguous CUDA (B, C, H, W), H and W multiples of 4")
    Bn, C, H, W = x.shape
    w32 = weight.detach().float().contiguous()
    b32 = None if bias is None else bias.detach().float().contiguous()
    u = torch.empty((Bn, 2 * C, H * W), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_dwconv3_act_planes(0, _ptr(x), C * H * W, _ptr(w32), _ptr(b32), None, 0, None, 0, _ptr(u), 2 * C * H * W,
                                                ctypes.c_void_p(u.data_ptr() + C * H * W * u.element_size()), 2 * C * H * W,
                                                Bn, C, H, W, _DT[x.dtype], _stream(x.device))
    _lib.check(rc, "ss2d_dwconv3_act_planes")
    return u


def dwconv3_act_planes_bwd(x: torch.Tensor, weight: torch.Tensor, bias, du: torch.Tensor) -> torch.Tensor:
    """Gradient of the pre-activation from du (B, 2 C, H W) = [gradient of the natural plane | of the transposed plane]."""
    Bn, C, H, W = x.shape
    _require(du.is_cuda and du.is_contiguous() and du.dtype == x.dtype and du.shape == (Bn, 2 * C, H * W), "dwconv3_act_planes: du must be (B, 2 C, H W) like the forward's output")
    w32 = weight.detach().float().contiguous()
    b32 = None if bias is None else bias.detach().float().contiguous()
    dpre = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_dwconv3_act_planes(1, _ptr(x), C * H * W, _ptr(w32), _ptr(b32), _ptr(du), 2 * C * H * W,
                                                ctypes.c_void_p(du.data_ptr() + C * H * W * du.element_size()), 2 * C * H * W,
                                                _ptr(dpre), C * H * W, None, 0, Bn, C, H, W, _DT[x.dtype], _stream(x.device))
    _lib.check(rc, "ss2d_dwconv3_act_planes")
    return dpre


def gate_proj_supported(D: int, C: int, K: int, dtype: torch.dtype) -> bool:
    return dtype in (torch.float32, torch.bfloat16) and bool(_lib.lib().ss2d_gate_proj_supported(int(D), int(C), int(K), _DT[dtype]))


def gate_proj_fwd(ys, ln_w, ln_b, z, z_act: bool, eps: float, W, bias, hw, tmask: int, want_g: bool):
    """out (B, L, C) = out_proj(LayerNorm(merge_K(ys)) * SiLU(z)) in one kernel (ss2d.py:486-518).
    ys (B, K, D, L) fp32; z (B, L, D) rows (uniformly strided view) of W's dtype; W (C, D).
    -> (out, stats (B, L, 2) fp32, g (B, L, D) gated tensor or None)."""
    Bn, K, D, L = ys.shape
    C = W.shape[0]
    dt = W.dtype
    _require(ys.is_cuda and ys.dtype == torch.float32 and ys.is_contiguous(), "gate_proj: ys must be a contiguous fp32 CUDA tensor")
    _require(W.stride(1) == 1 and (z is None or z.dtype == dt), "gate_proj: z must have W's dtype")
    out = torch.empty((Bn, L, C), dtype=dt, device=ys.device)
    stats = torch.empty((Bn, L, 2), dtype=torch.float32, device=ys.device)
    g = torch.empty((Bn, L, D), dtype=dt, device=ys.device) if want_g else None
    zrs = _row_stride(z, Bn, L) if z is not None else 0
    b32 = None if bias is None else bias.float().contiguous()
    with torch.cuda.device(ys.device):
        rc = _lib.lib().ss2d_gate_proj_fwd(_ptr(ys), K, ctypes.c_uint32(tmask), _ptr(ln_w), _ptr(ln_b), ctypes.c_float(eps), _ptr(z), zrs,
                                           1 if z_act else 0, _ptr(W), W.stride(0), _ptr(b32), _ptr(out), C, _ptr(g), D, _ptr(stats),
                                           Bn, D, L, int(hw[0]), int(hw[1]), C, _DT[dt], _stream(ys.device))
    _lib.check(rc, "ss2d_gate_proj_fwd")
    return out, stats, g


# ---- tensor-core projections (tcgen05): out = A W^T (+ bias) with split / permuted epilogues ---------------
def linear_tc_supported(n_cols: int, K: int, dtype: torch.dtype) -> bool:
    return dtype in (torch.float32, torch.bfloat16) and bool(_lib.lib().ss2d_linear_tc_supported(int(n_cols), int(K), _DT[dtype]))


def linear_tc(x: torch.Tensor, W: torch.Tensor, bias, parts):
    """x (..., K) rows with unit inner stride, W (N, K) -> one tensor per part.
    parts: list of (n_cols, kind, act) with kind "rows" -> (..., n_cols) row-major, or ("planes", L) -> the rows are
    (B, L) pixels and the part is returned channel-major as (B, n_cols, L); act: apply SiLU.
    fp32 operands run as TF32 on the tensor cores, bf16 operands as bf16; accumulation is fp32 either way."""
    _require(x.is_cuda and W.is_cuda and x.dtype == W.dtype and x.dtype in (torch.float32, torch.bfloat16),
             "linear_tc: CUDA fp32 or bf16 operands of one dtype")
    K = x.shape[-1]
    N = W.shape[0]
    x2 = x.reshape(-1, K)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    _require(W.dim() == 2 and W.shape[1] == K and W.stride(1) == 1, "linear_tc: W must be (N, K) with unit inner stride")
    M = x2.shape[0]
    _require(sum(p[0] for p in parts) == N, "linear_tc: the parts must cover the N columns")
    arr = (_lib.LinearPart * len(parts))()
    outs = []
    for i, (n_cols, kind, act) in enumerate(parts):
        if kind == "rows":
            o = torch.empty(x.shape[:-1] + (n_cols,), dtype=x.dtype, device=x.device)
            arr[i].ld, arr[i].planes_L = n_cols, 0
        else:
            Lp = int(kind[1])
            _require(M % Lp == 0, "linear_tc: rows must be whole (batch, L) images for a planes part")
            o = torch.empty((M // Lp, n_cols, Lp), dtype=x.dtype, device=x.device)
            arr[i].ld, arr[i].planes_L = 0, Lp
        arr[i].out, arr[i].n_cols, arr[i].act = o.data_ptr(), n_cols, 1 if act else 0
        outs.append(o)
    b32 = None if bias is None else bias.float().contiguous()
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_linear_tc(_ptr(x2), x2.stride(0), _ptr(W), W.stride(0), _ptr(b32), M, N, K, _DT[x.dtype], len(parts),
                                       arr, _stream(x.device))
    _lib.check(rc, "ss2d_linear_tc")
    return outs


# ---- row-wise LayerNorm ------------------------------------------------------------------------
LN_MAX_C = 512


def layernorm_fwd(x: torch.Tensor, weight, bias, eps: float):
    """x (..., C) contiguous CUDA tensor, C <= 512 -> (y, mean_rstd (rows, 2) fp32)."""
    _require(x.is_cuda and x.dtype in _DT and x.is_contiguous(), "layernorm: contiguous CUDA float tensor expected")
    C = x.shape[-1]
    rows = x.numel() // C
    _require(0 < C <= LN_MAX_C and rows > 0, "layernorm: 0 < C <= 512 and at least one row")
    y = torch.empty_like(x)
    stats = torch.empty((rows, 2), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_layernorm_fwd(_ptr(x), _ptr(weight), _ptr(bias), _ptr(y), _ptr(stats), rows, C,
                                           ctypes.c_float(eps), _DT[x.dtype], _stream(x.device))
    _lib.check(rc, "ss2d_layernorm_fwd")
    return y, stats


def layernorm_bwd(x: torch.Tensor, weight, dy: torch.Tensor, stats: torch.Tensor):
    """-> dx (like x), dweight (C) fp32, dbias (C) fp32."""
    C = x.shape[-1]
    rows = x.numel() // C
    dy = dy.contiguous()
    _require(dy.dtype == x.dtype and dy.shape == x.shape, "layernorm: dy must match x")
    dx = torch.empty_like(x)
    L = _lib.lib()
    npart = int(L.ss2d_layernorm_bwd_partials(rows))
    part = torch.empty((2, npart, C), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        rc = L.ss2d_layernorm_bwd(_ptr(x), _ptr(weight), _ptr(dy), _ptr(stats), _ptr(dx), _ptr(part[0]), _ptr(part[1]), npart,
                                  rows, C, _DT[x.dtype], _stream(x.device))
    _lib.check(rc, "ss2d_layernorm_bwd")
    sums = part.sum(dim=1)
    return dx, sums[0], sums[1]


# ---- depthwise 3 x 3 convolution: parameter gradients ---------------------------------------------
def dwconv3_wgrad(x: torch.Tensor, dy: torch.Tensor, want_bias: bool):
    """x, dy: fp32 (B, C, H, W) contiguous CUDA tensors -> dweight (C, 1, 3, 3), dbias (C) or None."""
    _require(x.is_cuda and dy.is_cuda and x.dtype == torch.float32 and dy.dtype == torch.float32 and x.shape == dy.shape
             and x.dim() == 4 and x.is_contiguous() and dy.is_contiguous(), "dwconv3_wgrad: contiguous fp32 (B, C, H, W) tensors")
    Bn, C, H, W = x.shape
    va = 16 if W % 4 == 0 else 4          # the C ABI's alignment rule; a fresh copy of a misaligned view satisfies it
    x = x if x.data_ptr() % va == 0 else x.clone()
    dy = dy if dy.data_ptr() % va == 0 else dy.clone()
    L = _lib.lib()
    ws_bytes = int(L.ss2d_dwconv3_wgrad_workspace_bytes(Bn, C, H, W))
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=x.device)
    dW = torch.empty((C, 1, 3, 3), dtype=torch.float32, device=x.device)
    db = torch.empty((C,), dtype=torch.float32, device=x.device) if want_bias else None
    with torch.cuda.device(x.device):
        rc = L.ss2d_dwconv3_wgrad(_ptr(x), _ptr(dy), _ptr(dW), _ptr(db), Bn, C, H, W, _ptr(ws), ctypes.c_size_t(ws_bytes),
                                  _stream(x.device))
    _lib.check(rc, "ss2d_dwconv3_wgrad")
    return dW, db


# ---- depthwise stack of the GroupMamba FFNs on channels-last tensors (csrc/ffn_dw.cu) -------------------------------
EPI_NONE, EPI_GELU, EPI_RESIDUAL, EPI_DGELU_MUL = 0, 1, 2, 3


def dwnhwc_stencil(x: torch.Tensor, hw, segments, *, flip: bool = False, epi: int = EPI_NONE, aux=None) -> torch.Tensor:
    """y = epi(bias + depthwise conv(x)) on the (B, H, W, C) image behind a contiguous (B, L, C) token tensor.
    segments: [(c_end, ksize, weight (c, 1, k, k) or None, bias (c) or None), ...] in channel order (ksize 0: no taps)."""
    _require(x.is_cuda and x.dtype in _DT and x.is_contiguous() and x.dim() == 3, "dwnhwc_stencil: contiguous CUDA (B, L, C) tensor")
    Bn, L, C = x.shape
    H, W = int(hw[0]), int(hw[1])
    _require(H * W == L, "dwnhwc_stencil: H * W must equal the token count")
    _require(aux is None or (aux.shape == x.shape and aux.dtype == x.dtype and aux.is_contiguous()), "dwnhwc_stencil: aux must match x")
    n = len(segments)
    _require(1 <= n <= 4 and segments[-1][0] == C, "dwnhwc_stencil: 1..4 channel segments covering C")
    cbeg = (ctypes.c_int32 * (n + 1))(0, *[int(sg[0]) for sg in segments])
    ks = (ctypes.c_int32 * n)(*[int(sg[1]) for sg in segments])
    keep = []                      # fp32 contiguous copies stay alive until the launch is enqueued
    wp, bp = (ctypes.c_void_p * n)(), (ctypes.c_void_p * n)()
    for i, (_, k, w, b) in enumerate(segments):
        w32 = None if w is None else w.detach().float().contiguous()
        b32 = None if b is None else b.detach().float().contiguous()
        keep += [w32, b32]
        wp[i] = None if w32 is None else w32.data_ptr()
        bp[i] = None if b32 is None else b32.data_ptr()
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _lib.lib().ss2d_dwnhwc_stencil(_ptr(x), _ptr(aux), _ptr(y), n, cbeg, ks, wp, bp, 1 if flip else 0, int(epi), Bn, H, W, C,
                                            _DT[x.dtype], _stream(x.device))
    _lib.check(rc, "ss2d_dwnhwc_stencil")
    return y


def dwnhwc_wgrad(x: torch.Tensor, g: torch.Tensor, hw, c0: int, c1: int, ksize: int, want_bias: bool = True):
    """Weight / bias gradient of the depthwise segment [c0, c1): -> dweight (c1 - c0, 1, k, k) fp32, dbias (c1 - c0) or None."""
    _require(x.is_cuda and x.dtype in _DT and x.is_contiguous() and x.dim() == 3 and g.shape == x.shape and g.dtype == x.dtype
             and g.is_contiguous(), "dwnhwc_wgrad: contiguous CUDA (B, L, C) tensors of one dtype")
    Bn, L, C = x.shape
    H, W = int(hw[0]), int(hw[1])
    _require(H * W == L, "dwnhwc_wgrad: H * W must equal the token count")
    Lb = _lib.lib()
    nc = c1 - c0
    ws_bytes = int(Lb.ss2d_dwnhwc_wgrad_workspace_bytes(Bn, H, W, nc, ksize))
    _require(ws_bytes > 0, "dwnhwc_wgrad: unsupported segment")
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=x.device)
    dW = torch.empty((nc, 1, ksize, ksize), dtype=torch.float32, device=x.device)
    db = torch.empty((nc,), dtype=torch.float32, device=x.device) if want_bias else None
    with torch.cuda.device(x.device):
        rc = Lb.ss2d_dwnhwc_wgrad(_ptr(x), _ptr(g), c0, c1, ksize, _ptr(dW), _ptr(db), Bn, H, W, C, _DT[x.dtype], _ptr(ws),
                                  ctypes.c_size_t(ws_bytes), _stream(x.device))
    _lib.check(rc, "ss2d_dwnhwc_wgrad")
    return dW, db
