"""autograd.Function surface of the reference (boundary b2, SURVEY.md §8b), backed by libss2d_b200.so.

Same class names and `.apply` signatures as /root/reference/gm-unet/model/gm/csms6s.py:
  SelectiveScanCore / SelectiveScanOflex   csms6s.py:347-386
  CrossScan / CrossMerge (K = 4)           csms6s.py:11-53
  CrossScan_1.._4 / CrossMerge_1.._4       csms6s.py:56-206
plus the fused operator `ss2d_core_fused` (cross-scan + scan + cross-merge + out_norm + gate without any
permuted copy), which `modules.SS2D` uses when it recognises the (CrossScan_k, CrossMerge_k) pair it is given.
Backward passes of the single-direction scans are the TRUE adjoints (the reference's CrossScan_2/_4.backward
are only correct for H == W, SURVEY.md §8-a2; on square maps the results are identical).
"""
from __future__ import annotations

import torch

from . import ops


def _custom_fwd(fn):
    return torch.amp.custom_fwd(fn, device_type="cuda")


def _custom_bwd(fn):
    return torch.amp.custom_bwd(fn, device_type="cuda")


class SelectiveScanCore(torch.autograd.Function):
    """out = selective_scan(u, delta, A, B, C, D, delta_bias); output dtype = input dtype (csms6s.py:347-365)."""
    OUT_FLOAT = False

    @staticmethod
    @_custom_fwd
    def forward(ctx, u, delta, A, B, C, D=None, delta_bias=None, delta_softplus=False, nrows=1, backnrows=1,
                oflex=True):
        prob = ops.ScanProblem(u, delta, A, B, C, D, delta_bias, delta_softplus, out_float=False)
        out, x = prob.forward(want_state=True)
        ctx.delta_softplus = delta_softplus
        ctx.out_float = False
        ctx.save_for_backward(u, delta, A, B, C, D, delta_bias, x)
        return out

    @staticmethod
    @_custom_bwd
    def backward(ctx, dout, *args):
        u, delta, A, B, C, D, delta_bias, x = ctx.saved_tensors
        prob = ops.ScanProblem(u, delta, A, B, C, D, delta_bias, ctx.delta_softplus, out_float=ctx.out_float)
        du, ddelta, dA, dB, dC, dD, dbias = prob.backward(dout, x)
        return (du, ddelta, dA, dB, dC, dD, dbias, None, None, None, None)


class SelectiveScanOflex(torch.autograd.Function):
    """Same, but with oflex=True the output (and dout) are fp32 whatever the input dtype (csms6s.py:368-386)."""

    @staticmethod
    @_custom_fwd
    def forward(ctx, u, delta, A, B, C, D=None, delta_bias=None, delta_softplus=False, nrows=1, backnrows=1,
                oflex=True):
        prob = ops.ScanProblem(u, delta, A, B, C, D, delta_bias, delta_softplus, out_float=bool(oflex))
        out, x = prob.forward(want_state=True)
        ctx.delta_softplus = delta_softplus
        ctx.out_float = bool(oflex)
        ctx.save_for_backward(u, delta, A, B, C, D, delta_bias, x)
        return out

    backward = SelectiveScanCore.backward


class _SelectiveScanState(torch.autograd.Function):
    """selective_scan with an initial state and the final state as a differentiable output (see `selective_scan`).
    With a gate z the first output is out * silu(z); the ungated out is saved for the backward, as mamba_ssm does."""

    @staticmethod
    def forward(ctx, u, delta, A, B, C, D, delta_bias, delta_softplus, h0, z=None):
        prob = ops.ScanProblem(u, delta, A, B, C, D, delta_bias, delta_softplus, out_float=False)
        res = prob.forward(want_state=True, h0=h0, z=z)
        x = res[1]
        last = x[:, :, 0, 1::2].contiguous()
        ctx.delta_softplus = delta_softplus
        ctx.has_h0 = h0 is not None
        ctx.save_for_backward(u, delta, A, B, C, D, delta_bias, h0, x, z, res[0] if z is not None else None)
        return (res[0] if z is None else res[2]), last

    @staticmethod
    def backward(ctx, dout, dlast):
        u, delta, A, B, C, D, delta_bias, h0, x, z, y = ctx.saved_tensors
        prob = ops.ScanProblem(u, delta, A, B, C, D, delta_bias, ctx.delta_softplus, out_float=False)
        grads = prob.backward(dout.contiguous(), x, h0=h0, dlast=dlast, want_dh0=ctx.needs_input_grad[8], z=z, out=y)
        du, ddelta, dA, dB, dC, dD, dbias = grads[:7]
        dz = grads[7] if z is not None else None
        return du, ddelta, dA, dB, dC, dD, dbias, None, grads[-1], dz


def selective_scan(u, delta, A, B, C, D=None, delta_bias=None, delta_softplus=False, initial_state=None,
                   return_last_state=False, *, z=None):
    """Differentiable selective scan with state passing, in the reference extension's SCAN layout and dtype rules:
    u, delta (B, Dt, L) and B, C (B, G, N, L) or (B, N, L) of one dtype (fp32 / fp16 / bf16), A (Dt, N) fp32, D and
    delta_bias (Dt) fp32 or None; out has u's dtype.

        h_l = exp(delta_l A) * h_(l-1) + delta_l u_l B_l,  h_(-1) = initial_state (zeros when None),  out_l = C_l . h_l + D u_l

    initial_state: (B, Dt, N) fp32 or None; gradients flow to it. return_last_state: also return h_(L-1) as a (B, Dt, N)
    fp32 tensor whose gradient flows back through the scan, so a sequence split into pieces can be chained call by call.
    z: optional (B, Dt, L) gate of u's dtype (mamba_ssm's selective_scan_fn z): the result is then out * silu(z), with the
    gate applied inside the library (gradients flow to z too).
    Under torch.use_deterministic_algorithms(True) every gradient is bit-identical from call to call."""
    out, last = _SelectiveScanState.apply(u, delta, A, B, C, D, delta_bias, bool(delta_softplus), initial_state, z)
    return (out, last) if return_last_state else out


def selective_state_update(state, x, dt, A, B, C, D=None, z=None, dt_bias=None, dt_softplus=False):
    """One recurrent step of the selective scan with mamba_ssm's `selective_state_update` arguments; `state` is updated in place.

        t = dt + dt_bias (softplus(t) when dt_softplus),  state = exp(t A) * state + t x B,  out = C . state + D x  (* silu(z))

    state: fp32 (batch, dim, dstate), contiguous (the layout of `selective_scan`'s final state: a prefill's `last_state` is
    stepped from directly). x, dt, z: (batch, dim); B, C: (batch, dstate) or (batch, n_groups, dstate), all of one dtype (fp32 /
    fp16 / bf16); A: fp32 (dim, dstate); D, dt_bias: fp32 (dim) or None. Returns out (batch, dim) in x's dtype.
    Inference only, like mamba_ssm's function: with grad mode on, no input may require grad (train with `selective_scan`)."""
    if torch.is_grad_enabled():
        for name, t in (("state", state), ("x", x), ("dt", dt), ("A", A), ("B", B), ("C", C), ("D", D), ("z", z),
                        ("dt_bias", dt_bias)):
            if t is not None and t.requires_grad:
                raise RuntimeError(f"selective_state_update has no backward, but {name} requires grad: run it under torch.no_grad()")
    return ops.state_update(state, x, dt, A, B, C, D, z, dt_bias, dt_softplus)


# ---- causal depthwise conv1d (the causal-conv1d 1.1.x interface) ----------------------------------
def _silu_flag(activation):
    if activation not in (None, "silu", "swish"):
        raise NotImplementedError("activation must be None, silu, or swish")      # a RuntimeError, as in causal-conv1d
    return activation is not None


class _CausalConv1d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, silu):
        ctx.save_for_backward(x, weight, bias)
        ctx.silu = silu
        return ops.conv1d_fwd(x, weight, bias, silu)

    @staticmethod
    def backward(ctx, dout):
        x, weight, bias = ctx.saved_tensors
        dx, dweight, dbias = ops.conv1d_bwd(x, weight, bias, dout, ctx.silu)
        return dx, dweight, dbias, None


def causal_conv1d_fn(x, weight, bias=None, seq_idx=None, activation=None):
    """Causal depthwise conv1d with causal-conv1d's arguments, differentiable in x, weight and bias:

        out[b,d,l] = act(bias[d] + sum_{k<width} weight[d,k] x[b,d,l-(width-1)+k]),  x = 0 before position 0,

    that is nn.Conv1d(dim, dim, width, groups=dim, padding=width-1)(x)[..., :L] then act: SiLU for "silu" / "swish", none for None.
    x: (batch, dim, L) fp32 / fp16 / bf16 with stride 1 along L; weight: (dim, width), 2 <= width <= 4; bias: (dim) or None, of
    weight's dtype (fp32 parameters with a bf16 x, as under autocast, are fine). Math in fp32; out has x's dtype. seq_idx and
    channel-last x are not supported (RuntimeError)."""
    if seq_idx is not None:
        raise RuntimeError("causal_conv1d_fn: seq_idx is not supported")
    return _CausalConv1d.apply(x, weight, bias, _silu_flag(activation))


def causal_conv1d_update(x, conv_state, weight, bias=None, activation=None):
    """One decode position with causal-conv1d's arguments: conv_state (batch, dim, width) of x's dtype is shifted left by one in
    place and x (batch, dim) stored in its last slot; returns act(bias + sum_k weight[:, k] conv_state[..., k]) (batch, dim).
    After a prefill over L positions, conv_state = F.pad(x, (width - L, 0)) holds the last width inputs, and step t returns the
    forward over L + t + 1 positions at position L + t. Inference only: with grad mode on, no input may require grad."""
    if torch.is_grad_enabled():
        for name, t in (("x", x), ("conv_state", conv_state), ("weight", weight), ("bias", bias)):
            if t is not None and t.requires_grad:
                raise RuntimeError(f"causal_conv1d_update has no backward, but {name} requires grad: run it under torch.no_grad()")
    return ops.conv1d_update(x, conv_state, weight, bias, _silu_flag(activation))


# ---- Mamba-2 chunked selective scan (the mamba_ssm 2.x interface) -----------------------------------
class _ChunkScan(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, dt, A, B, C, D, z, dt_bias, initial_states, chunk_size, dt_softplus, dt_limit):
        ops_in = ops.ssd_prepare(x, dt, A, B, C, chunk_size, D, z, dt_bias, initial_states, dt_limit)
        out, final = ops.ssd_fwd(*ops_in[:5], chunk_size, *ops_in[5:], dt_softplus, dt_limit, True)
        ctx.save_for_backward(*ops_in)      # the inputs only: the backward recomputes the chunk states
        ctx.cfg = (chunk_size, dt_softplus, dt_limit)
        ctx.dtypes = tuple(None if t is None else t.dtype for t in (dt, A, D, dt_bias))
        return out, final

    @staticmethod
    def backward(ctx, dout, dfinal):
        x, dt, A, B, C, D, z, dt_bias, h0 = ctx.saved_tensors
        chunk_size, dt_softplus, dt_limit = ctx.cfg
        if dout is None:
            dout = torch.zeros_like(x)
        dx, ddt, dA, dB, dC, dD, dz, ddt_bias, dh0 = ops.ssd_bwd(x, dt, A, B, C, chunk_size, D, z, dt_bias, h0, dt_softplus,
                                                                 dt_limit, dout, dfinal)
        dt_t, A_t, D_t, bias_t = ctx.dtypes
        cast = lambda g, t: None if g is None else g.to(t)   # noqa: E731
        return (dx, cast(ddt, dt_t), cast(dA, A_t), dB, dC, cast(dD, D_t), dz, cast(ddt_bias, bias_t), dh0, None, None, None)


def mamba_chunk_scan_combined(x, dt, A, B, C, chunk_size, D=None, z=None, dt_bias=None, initial_states=None, seq_idx=None,
                              cu_seqlens=None, dt_softplus=False, dt_limit=(0.0, float("inf")), return_final_states=False,
                              return_varlen_states=False):
    """Mamba-2's scan (SSD) with mamba_ssm's arguments, computed in chunks of chunk_size positions on the tensor cores:

        t_l = clamp(softplus?(dt_l + dt_bias), dt_limit),  H_l = exp(t_l A) H_{l-1} + t_l x_l (x) B_l,  H_{-1} = initial_states,
        y_l = C_l . H_l + D x_l,  out_l = y_l * silu(z_l) (with z).

    x, z (batch, seqlen, heads, headdim), dt (batch, seqlen, heads), A (heads), B, C (batch, seqlen, n_groups, dstate), D (heads)
    or (heads, headdim), dt_bias (heads), initial_states (batch, heads, headdim, dstate). x, z, B and C share one dtype (fp32 /
    fp16 / bf16); math in fp32; out has x's dtype. headdim in {32, 64, 128}, dstate a multiple of 16 up to 256, chunk_size in
    {64, 128, 256}. The default dt_limit (0, inf) does not clamp, as in mamba_ssm. Returns out, or (out, final_states) with
    final_states = H_{seqlen-1} fp32 (batch, heads, headdim, dstate): the (batch, heads * headdim, dstate) state that
    selective_scan(..., initial_state=) and selective_state_update take.
    Differentiable in x, dt, A, B, C, D, z, dt_bias and initial_states, and through final_states; the gradients are
    bit-identical from call to call, and autograd keeps only the inputs. seq_idx, cu_seqlens and return_varlen_states are not
    supported (RuntimeError)."""
    if seq_idx is not None or cu_seqlens is not None or return_varlen_states:
        raise RuntimeError("mamba_chunk_scan_combined: seq_idx, cu_seqlens and return_varlen_states are not supported")
    out, final = _ChunkScan.apply(x, dt, A, B, C, D, z, dt_bias, initial_states, chunk_size, bool(dt_softplus),
                                  tuple(dt_limit))
    return (out, final) if return_final_states else out


# ---- cross scan / merge ---------------------------------------------------------------------------
def _make_cross_pair(dirs, suffix):
    dirs = tuple(dirs)
    K = len(dirs)

    class _Scan(torch.autograd.Function):
        DIRS = dirs

        @staticmethod
        def forward(ctx, x: torch.Tensor):
            Bn, Cn, H, W = x.shape
            ctx.shape = (Bn, Cn, H, W)
            return ops.cross_scan(x, dirs)                              # (B, K, C, L)

        @staticmethod
        def backward(ctx, ys: torch.Tensor):
            Bn, Cn, H, W = ctx.shape
            return ops.cross_merge(ys.contiguous(), (H, W), dirs).view(Bn, Cn, H, W)

    class _Merge(torch.autograd.Function):
        DIRS = dirs

        @staticmethod
        def forward(ctx, ys: torch.Tensor):
            Bn, Kn, D, H, W = ys.shape
            ctx.shape = (H, W)
            return ops.cross_merge(ys.reshape(Bn, Kn, D, H * W), (H, W), dirs)     # (B, D, L)

        @staticmethod
        def backward(ctx, x: torch.Tensor):
            H, W = ctx.shape
            Bn, Cn, L = x.shape
            return ops.cross_scan(x.reshape(Bn, Cn, H, W), dirs).view(Bn, K, Cn, H, W)

    _Scan.__name__ = _Scan.__qualname__ = "CrossScan" + suffix
    _Merge.__name__ = _Merge.__qualname__ = "CrossMerge" + suffix
    return _Scan, _Merge


CrossScan, CrossMerge = _make_cross_pair((1, 2, 3, 4), "")
CrossScan_1, CrossMerge_1 = _make_cross_pair((1,), "_1")
CrossScan_2, CrossMerge_2 = _make_cross_pair((2,), "_2")
CrossScan_3, CrossMerge_3 = _make_cross_pair((3,), "_3")
CrossScan_4, CrossMerge_4 = _make_cross_pair((4,), "_4")


def directions_of(cross_scan_cls, cross_merge_cls):
    """Directions encoded by a (CrossScan*, CrossMerge*) class pair — ours or the reference's (matched by class
    name, since the reference passes the classes themselves into SS2D.forward, groupmamba.py:143-146)."""
    table = {"CrossScan": (1, 2, 3, 4), "CrossScan_1": (1,), "CrossScan_2": (2,), "CrossScan_3": (3,), "CrossScan_4": (4,)}
    sname, mname = cross_scan_cls.__name__, cross_merge_cls.__name__
    if sname not in table or mname != sname.replace("Scan", "Merge"):
        return None
    return table[sname]


# ---- fused SS2D core ------------------------------------------------------------------------------
class _SS2DScanNatural(torch.autograd.Function):
    """Selective scan over K groups in NATURAL layout, each group traversed in its direction.

    u: (B, P*D, L) — P input planes shared cyclically by the groups (group g reads plane g % P): P = 1 when every
    direction scans the same image, P = 2 for (natural, transposed) pairs. delta (B, K*D, L), Bs/Cs (B, K, N, L), all
    in the pixel order of the plane their group reads. Returns ys (B, K/P, P, D, L) fp32 in that same pixel order."""

    @staticmethod
    @_custom_fwd
    def forward(ctx, u, dts, A, Bs, Cs, Ds, delta_bias, H, W, dirs, P):
        Bn, PD, L = u.shape
        D, K = PD // P, len(dirs)
        prob = ops.ScanProblem(u, dts, A, Bs, Cs, Ds, delta_bias, True, out_float=True, hw=(H, W), dirs=dirs, u_mod=PD)
        out, st = prob.forward(want_state=True)
        ctx.meta = (H, W, tuple(dirs), D, P)
        ctx.save_for_backward(u, dts, A, Bs, Cs, Ds, delta_bias, st)
        return out.view(Bn, K // P, P, D, L)

    @staticmethod
    @_custom_bwd
    def backward(ctx, dys):
        """dys: (B, K/P, P, D, L). When it is a stride-0 expansion over dim 1 (what `_OutGate.backward` returns:
        CrossMerge's adjoint hands every direction the same gradient, csms6s.py:42-53) the kernel reads the P shared
        (B, D, L) planes for all groups; otherwise the per-direction planes are used as they are."""
        u, dts, A, Bs, Cs, Ds, delta_bias, st = ctx.saved_tensors
        H, W, dirs, D, P = ctx.meta
        K = len(dirs)
        Bn, L = u.shape[0], H * W
        if K == P or dys.stride(1) == 0:
            prob = ops.ScanProblem(u, dts, A, Bs, Cs, Ds, delta_bias, True, out_float=True, hw=(H, W), dirs=dirs, u_mod=P * D)
            du, ddelta, dA, dB, dC, dD, dbias = prob.backward(dys[:, 0].reshape(Bn, P * D, L).float(), st)
        else:
            u_full = u.view(Bn, 1, P * D, L).expand(Bn, K // P, P * D, L).reshape(Bn, K * D, L)
            prob = ops.ScanProblem(u_full, dts, A, Bs, Cs, Ds, delta_bias, True, out_float=True, hw=(H, W), dirs=dirs, u_mod=0)
            du, ddelta, dA, dB, dC, dD, dbias = prob.backward(dys.reshape(Bn, K * D, L).float().contiguous(), st)
        du = du.view(Bn, K // P, P * D, L).sum(dim=1) if K > P else du.view_as(u)
        return du, ddelta, dA, dB, dC, dD, dbias, None, None, None, None


class _OutGate(torch.autograd.Function):
    """merge over K + un-transpose + (B,D,L)->(B,L,D) + LayerNorm(D) + SiLU(z) gate (ops.out_gate_fwd/bwd).
    ys: (B, K/P, P, D, L); plane (i, j) is in transposed pixel order when bit j of `tplanes` is set."""

    @staticmethod
    @_custom_fwd
    def forward(ctx, ys, ln_w, ln_b, z, z_act, eps, out_dtype, H, W, tplanes):
        Bn, G, P, D, L = ys.shape
        K = G * P
        tmask = 0
        for k in range(K):
            if (tplanes >> (k % P)) & 1:
                tmask |= 1 << k
        out, stats = ops.out_gate_fwd(ys.view(Bn, K, D, L), ln_w, ln_b, z, z_act, eps, out_dtype, (H, W), tmask)
        ctx.meta = (z_act, z is not None, H, W, tmask, tplanes)
        ctx.save_for_backward(ys, ln_w, ln_b, z, stats)
        return out

    @staticmethod
    @_custom_bwd
    def backward(ctx, dout):
        ys, ln_w, ln_b, z, stats = ctx.saved_tensors
        z_act, has_z, H, W, tmask, tplanes = ctx.meta
        Bn, G, P, D, L = ys.shape
        dz = torch.empty(z.shape, dtype=z.dtype, device=z.device) if has_z else None
        two = P == 2 and tplanes == 0b10 and G * P > 1          # (natural, transposed) plane pairs: the kernel writes both orientations
        dy, dw, db = ops.out_gate_bwd(ys.view(Bn, G * P, D, L), ln_w, ln_b, z, z_act, dout, stats, dz, (H, W), tmask, two_planes=two)
        if two:      # (B, 2, D, L) straight from the kernel: no transposed copy, no stack
            return (dy.unsqueeze(1).expand(Bn, G, P, D, L), (dw if ln_w is not None else None), (db if ln_b is not None else None), dz,
                    None, None, None, None, None, None)
        # dy is the gradient of the merged y in natural pixel order; every group receives it (transposed for the groups
        # that ran on the transposed image). Returned as a stride-0 expansion over the K/P repeats: no K-fold copy.
        if G * P == 1:      # a single plane: the kernel already wrote dy in that plane's own (possibly transposed) pixel order
            return (dy.view(Bn, 1, 1, D, L), (dw if ln_w is not None else None), (db if ln_b is not None else None), dz,
                    None, None, None, None, None, None)
        planes = [dy.view(Bn, D, H, W).transpose(2, 3).reshape(Bn, D, L) if (tplanes >> j) & 1 else dy for j in range(P)]
        base = planes[0].unsqueeze(1) if P == 1 else torch.stack(planes, dim=1)          # (B, P, D, L)
        dys = base.unsqueeze(1).expand(Bn, G, P, D, L)
        return (dys, (dw if ln_w is not None else None), (db if ln_b is not None else None), dz,
                None, None, None, None, None, None)


class _OutGateProj(torch.autograd.Function):
    """out = out_proj(LayerNorm(merge_K(ys)) * SiLU(z)) in ONE tcgen05 kernel (ops.gate_proj_fwd; ss2d.py:486-518): the gated
    tensor is built in shared memory in the tensor core's operand layout and only written out (g) when a backward will need it.
    Backward: dG = dout W (library GEMM), then ops.out_gate_bwd as for _OutGate; dW from g."""

    @staticmethod
    def forward(ctx, ys, ln_w, ln_b, z, W, bias, eps, H, Wd, tplanes):
        Bn, G, P, D, L = ys.shape
        K = G * P
        tmask = 0
        for k in range(K):
            if (tplanes >> (k % P)) & 1:
                tmask |= 1 << k
        zc, Wc = _tc_operands(z, W)
        need_bwd = any(ctx.needs_input_grad)
        out, stats, g = ops.gate_proj_fwd(ys.view(Bn, K, D, L), ln_w, ln_b, zc, True, eps, Wc, bias, (H, Wd), tmask, need_bwd)
        ctx.meta = (H, Wd, tmask, tplanes, bias is not None, z.dtype, W.dtype)
        ctx.save_for_backward(ys, ln_w, ln_b, zc, stats, g, Wc)
        return out

    @staticmethod
    def backward(ctx, dout):
        ys, ln_w, ln_b, zc, stats, g, Wc = ctx.saved_tensors
        H, Wd, tmask, tplanes, has_bias, z_dtype, W_dtype = ctx.meta
        Bn, G, P, D, L = ys.shape
        C = Wc.shape[0]
        d2 = dout.reshape(Bn * L, C).to(Wc.dtype)
        dG = torch.matmul(d2, Wc).view(Bn, L, D)
        dz = torch.empty_like(zc)
        two = P == 2 and tplanes == 0b10 and G * P > 1
        dy, dlw, dlb = ops.out_gate_bwd(ys.view(Bn, G * P, D, L), ln_w, ln_b, zc, True, dG, stats, dz, (H, Wd), tmask, two_planes=two)
        if two:
            dys = dy.unsqueeze(1).expand(Bn, G, P, D, L)
        elif G * P == 1:
            dys = dy.view(Bn, 1, 1, D, L)
        else:
            planes = [dy.view(Bn, D, H, Wd).transpose(2, 3).reshape(Bn, D, L) if (tplanes >> j) & 1 else dy for j in range(P)]
            base = planes[0].unsqueeze(1) if P == 1 else torch.stack(planes, dim=1)
            dys = base.unsqueeze(1).expand(Bn, G, P, D, L)
        dW = _wgrad_rows(d2.contiguous(), g.reshape(Bn * L, D)).to(W_dtype) if ctx.needs_input_grad[4] else None
        db = d2.float().sum(dim=0) if has_bias and ctx.needs_input_grad[5] else None
        return dys, dlw, dlb, dz.to(z_dtype), dW, db, None, None, None, None


def out_gate_proj_ok(ys, z, W, H, Wd) -> bool:
    """Eligibility of the fused epilogue + out_proj kernel: a gate is present, the operand dtype is allowed on the tensor cores
    (_tc_dtype_ok) and the shape fits (ops.gate_proj_supported; the backward goes through out_gate_bwd: D <= its limit)."""
    if z is None or not _tc_dtype_ok(z):
        return False
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else z.dtype
    Bn, G, P, D, L = ys.shape
    return (ys.dtype == torch.float32 and ops.gate_proj_supported(D, W.shape[0], G * P, dt) and W.shape[1] == D
            and H % 4 == 0 and Wd % 4 == 0              # the planes are read as TMA boxes: 16-byte aligned image rows
            and D <= ops.out_gate_max_D(backward=True))


class _GroupGate(torch.autograd.Function):
    """The epilogues of the four single-direction SS2Ds of a GroupMambaLayer in one launch (ops.group_gate_fwd/bwd):
    per group out_norm LayerNorm(D) + SiLU(z) gate (ss2d.py:498, 515-517), un-transposition of the column-major planes,
    (B,D,L)->(B,L,D), and the concatenation over the groups (groupmamba.py:149) as the column placement of the stores."""

    @staticmethod
    @_custom_fwd
    def forward(ctx, ys, ln_w, ln_b, z, eps, out_dtype, H, W, plane_of, tbits):
        out, stats = ops.group_gate_fwd(ys, plane_of, tbits, ln_w, ln_b, z, eps, out_dtype, (H, W))
        ctx.meta = (H, W, tuple(plane_of), tbits)
        ctx.save_for_backward(ys, ln_w, ln_b, z, stats)
        return out

    @staticmethod
    @_custom_bwd
    def backward(ctx, dout):
        ys, ln_w, ln_b, z, stats = ctx.saved_tensors
        H, W, plane_of, tbits = ctx.meta
        dy, dz, dw, db = ops.group_gate_bwd(ys, plane_of, tbits, ln_w, ln_b, z, dout, stats, (H, W))
        return dy, dw, db, dz, None, None, None, None, None, None


class _InProjSplit(torch.autograd.Function):
    """x_all, z_all = xn @ Wx^T, xn @ Wz^T for block-structured (C, C) weights: the four in_proj layers of a GroupMambaLayer
    (ss2d.py:504-506) as two GEMMs whose outputs are separate dense tensors, so that neither the split nor its backward costs
    a pass over memory (a chunk() of one GEMM output would: slice_backward zero-fills and copies). Library GEMMs under the
    ambient autocast; the backward accumulates the two input-gradient products inside the second GEMM."""

    @staticmethod
    def forward(ctx, xn, Wx, Wz):
        ctx.save_for_backward(xn, Wx, Wz)
        return torch.nn.functional.linear(xn, Wx), torch.nn.functional.linear(xn, Wz)

    @staticmethod
    def backward(ctx, dx, dz):
        xn, Wx, Wz = ctx.saved_tensors
        C = Wx.shape[1]
        dx2, dz2, x2 = dx.reshape(-1, Wx.shape[0]), dz.reshape(-1, Wz.shape[0]), xn.reshape(-1, C)
        dxn = dWx = dWz = None
        if ctx.needs_input_grad[0]:
            acc = torch.matmul(dx2, Wx.to(dx2.dtype))
            acc.addmm_(dz2.to(acc.dtype), Wz.to(acc.dtype))
            dxn = acc.view(xn.shape).to(xn.dtype)
        if ctx.needs_input_grad[1]:
            dWx = torch.matmul(dx2.t(), x2.to(dx2.dtype)).to(Wx.dtype)
        if ctx.needs_input_grad[2]:
            dWz = torch.matmul(dz2.t(), x2.to(dz2.dtype)).to(Wz.dtype)
        return dxn, dWx, dWz


class _ToPlanes(torch.autograd.Function):
    """(B, H, W, 4 D) channels-last, channel blocks in PLANE order -> (B, 4 D, H, W) channel-major with the last two blocks
    TRANSPOSED (stored as (W, H) images; H == W): the NHWC->NCHW copy of ss2d.py:510 for the four SS2Ds at once, with the
    transposition that turns the column-major scans 2 / 4 into row-major scans folded into the same copy."""

    @staticmethod
    def forward(ctx, x, D2):
        Bn, H, W, C = x.shape
        out = torch.empty((Bn, C, H, W), dtype=x.dtype, device=x.device)
        out[:, :D2].copy_(x[..., :D2].permute(0, 3, 1, 2))
        out[:, D2:].copy_(x[..., D2:].permute(0, 3, 2, 1))
        ctx.D2 = D2
        return out

    @staticmethod
    def backward(ctx, dout):
        D2 = ctx.D2
        Bn, C, H, W = dout.shape
        dx = torch.empty((Bn, H, W, C), dtype=dout.dtype, device=dout.device)
        dx[..., :D2].copy_(dout[:, :D2].permute(0, 2, 3, 1))
        dx[..., D2:].copy_(dout[:, D2:].permute(0, 3, 2, 1))
        return dx, None


# ---- small projections with a tall-skinny weight gradient -------------------------------------------
_TS_MIN_ROWS = 8192      # below this a library GEMM is as good (measured on the four GM-UNet stage shapes)


class _LinearTS(torch.autograd.Function):
    """y = F.linear(x, W, b) (cuBLAS; runs under the ambient autocast like nn.Linear). Backward: dx by cuBLAS, dW by
    ops.wgrad_ts when W is tiny and the number of rows huge (in_proj / out_proj / proj of the live GM-UNet stages)."""

    @staticmethod
    def forward(ctx, x, W, bias):
        ctx.save_for_backward(x, W)
        ctx.has_bias = bias is not None
        return torch.nn.functional.linear(x, W, bias)

    @staticmethod
    def backward(ctx, dy):
        x, W = ctx.saved_tensors
        M, N = W.shape
        dy2, x2 = dy.reshape(-1, M), x.reshape(-1, N)
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.matmul(dy2, W.to(dy2.dtype)).view(x.shape).to(x.dtype)
        if ctx.needs_input_grad[1]:
            if dy2.shape[0] >= _TS_MIN_ROWS and ops.wgrad_ts_supported(M, N):
                dW = ops.wgrad_ts(dy2.unsqueeze(0), x2.unsqueeze(0)).to(W.dtype)
            else:
                dW = _wgrad_rows(dy2.contiguous(), x2.to(dy2.dtype).contiguous()).to(W.dtype)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy2.sum(dim=0)
        return dx, dW, db


def _wgrad_rows(dy2: torch.Tensor, x2: torch.Tensor) -> torch.Tensor:
    """dW (M, N) = dy2 (R, M)^T @ x2 (R, N) for R >> M, N. As ONE GEMM this is a handful of output tiles walking the whole
    reduction (6 CTAs on 148 SMs for 96 x 192 over 75 264 rows: 77 us); cut into S slabs it is a batched GEMM with S times the
    CTAs plus a tiny sum (split-K done by hand, deterministic)."""
    R = dy2.shape[0]
    S = 128
    while S > 1 and (R % S != 0 or R // S < 256):
        S //= 2
    if S == 1:
        return torch.matmul(dy2.t(), x2)
    part = torch.bmm(dy2.view(S, R // S, -1).transpose(1, 2), x2.view(S, R // S, -1))
    return part.sum(dim=0)


def _need_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:      # the modules have no CPU path: fail here rather than silently run a library op on the host
        raise RuntimeError(f"{what}: CUDA tensor expected (ceigm_unet_b200 has no CPU fallback)")


def _ts_eligible(rows: int, M: int, N: int, t: torch.Tensor) -> bool:
    _need_cuda(t, "projection")
    return rows >= _TS_MIN_ROWS and ops.wgrad_ts_supported(M, N)


def linear_ts(x, W, bias=None):
    """nn.Linear's forward; its weight gradient comes from ops.wgrad_ts when the shape is tall and skinny."""
    if not _ts_eligible(x.numel() // max(x.shape[-1], 1), W.shape[0], W.shape[1], x):
        return torch.nn.functional.linear(x, W, bias)
    return _LinearTS.apply(x, W, bias)


class _ProjCM(torch.autograd.Function):
    """out (B, M, L) = W (M, D) @ u (B, D, L): the 1 x 1 projections of SS2D.forward_core on channel-major tensors
    (x_proj, dt_proj; ss2d.py:465-477). Backward: du by cuBLAS, dW by ops.wgrad_ts on the operands in place."""

    @staticmethod
    def forward(ctx, W, u):
        ctx.save_for_backward(W, u)
        return _bmm_w(W, u)

    @staticmethod
    def backward(ctx, dout):
        W, u = ctx.saved_tensors
        M, D = W.shape
        dW = du = None
        if ctx.needs_input_grad[1]:
            du = _bmm_w(W.t().to(dout.dtype), dout).to(u.dtype)
        if ctx.needs_input_grad[0]:
            if dout.shape[0] * dout.shape[2] >= _TS_MIN_ROWS and ops.wgrad_ts_supported(M, D):
                dW = ops.wgrad_ts(dout.transpose(1, 2), u.transpose(1, 2)).to(W.dtype)
            else:
                dW = torch.matmul(dout, u.transpose(1, 2).to(dout.dtype)).sum(dim=0).to(W.dtype)
        return dW, du


def _bmm_w(W, u):
    """W (M, D) @ u (B, D, L) -> (B, M, L) as ONE strided-batched GEMM with a stride-0 weight. torch.matmul folds this case
    into a 2-D GEMM by materialising u^T (and copying the transposed result back): 190 us of copies around a 31 us GEMM at
    the north-star shape."""
    return torch.bmm(W.unsqueeze(0).expand(u.shape[0], W.shape[0], W.shape[1]), u)


def proj_cm(W, u):
    if not _ts_eligible(u.shape[0] * u.shape[2], W.shape[0], W.shape[1], u):
        return _bmm_w(W, u)
    return _ProjCM.apply(W, u)


# ---- tensor-core projections (ops.linear_tc: tcgen05, TMA-fed, accumulators in tensor memory) ---------------
def _tc_operands(x, W):
    """The operand dtype nn.Linear would compute in: the autocast dtype when autocast is on, else x's own."""
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        return x.to(dt), W.to(dt)
    return x, W.to(x.dtype)


def _tc_dtype_ok(x) -> bool:
    """bf16 operands always (the tensor core multiplies them exactly); fp32 operands only when the user has allowed TF32
    matmuls (torch.backends.cuda.matmul.allow_tf32 / set_float32_matmul_precision("high" | "medium"), as the reference's
    train_synapse.py:21 does) — the same switch that governs cuBLAS."""
    _need_cuda(x, "projection")
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    return dt == torch.bfloat16 or (dt == torch.float32 and torch.backends.cuda.matmul.allow_tf32)


def _tc_shape_ok(n_cols: int, K: int, x) -> bool:
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    return ops.linear_tc_supported(n_cols, K, dt)


class _InProjPlanes(torch.autograd.Function):
    """xi (B, D, H, W), z (B, H, W, D) = in_proj + chunk + the NHWC -> NCHW copy of the x half (ss2d.py:504-510): ONE
    tcgen05 launch whose epilogue stores the x half as channel-major planes and the gate half as rows."""

    @staticmethod
    def forward(ctx, x, W, bias):
        xc, Wc = _tc_operands(x, W)
        Bn, H, Wd, _ = x.shape
        D = W.shape[0] // 2
        xi, z = ops.linear_tc(xc, Wc, bias, [(D, ("planes", H * Wd), False), (D, "rows", False)])
        ctx.save_for_backward(xc, Wc)
        ctx.meta = (bias is not None, x.dtype, W.dtype)
        return xi.view(Bn, D, H, Wd), z

    @staticmethod
    def backward(ctx, dxi, dz):
        xc, Wc = ctx.saved_tensors
        has_bias, x_dtype, W_dtype = ctx.meta
        Bn, H, Wd, C = xc.shape
        D, L = Wc.shape[0] // 2, H * Wd
        dxi3 = dxi.reshape(Bn, D, L).to(Wc.dtype)             # channel-major, as the forward wrote it
        dz2 = dz.reshape(Bn * L, D).to(Wc.dtype)
        x3 = xc.reshape(Bn, L, C)
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            # batched GEMM on the channel-major gradient in place (torch.matmul would first copy it to pixel-major)
            acc = torch.bmm(dxi3.transpose(1, 2), Wc[:D].unsqueeze(0).expand(Bn, D, C)).view(Bn * L, C)
            acc.addmm_(dz2, Wc[D:])
            dx = acc.view(xc.shape).to(x_dtype)
        if ctx.needs_input_grad[1]:
            dWx = torch.matmul(dxi3, x3).sum(dim=0)
            dWz = _wgrad_rows(dz2.contiguous(), x3.reshape(Bn * L, C))
            dW = torch.cat([dWx, dWz], dim=0).to(W_dtype)
        if has_bias and ctx.needs_input_grad[2]:
            db = torch.cat([dxi3.float().sum(dim=(0, 2)), dz2.float().sum(dim=0)])
        return dx, dW, db


class _LinearTC(torch.autograd.Function):
    """y = x W^T + b on the tensor cores (out_proj, ss2d.py:518); backward as _LinearTS."""

    @staticmethod
    def forward(ctx, x, W, bias):
        xc, Wc = _tc_operands(x, W)
        (out,) = ops.linear_tc(xc, Wc, bias, [(W.shape[0], "rows", False)])
        ctx.save_for_backward(xc, Wc)
        ctx.meta = (bias is not None, x.dtype, W.dtype)
        return out

    @staticmethod
    def backward(ctx, dy):
        xc, Wc = ctx.saved_tensors
        has_bias, x_dtype, W_dtype = ctx.meta
        M, N = Wc.shape
        dy2, x2 = dy.reshape(-1, M).to(Wc.dtype), xc.reshape(-1, N)
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.matmul(dy2, Wc).view(xc.shape).to(x_dtype)
        if ctx.needs_input_grad[1]:
            if dy2.shape[0] >= _TS_MIN_ROWS and ops.wgrad_ts_supported(M, N):
                dW = ops.wgrad_ts(dy2.unsqueeze(0), x2.unsqueeze(0)).to(W_dtype)
            else:
                dW = _wgrad_rows(dy2.contiguous(), x2.contiguous()).to(W_dtype)
        if has_bias and ctx.needs_input_grad[2]:
            db = dy2.float().sum(dim=0)
        return dx, dW, db


def in_proj_planes(x, W, bias=None):
    """(xi (B, D, H, W), z (B, H, W, D)) through the tensor-core kernel, or None when the shape / dtype is not eligible
    (the caller then composes F.linear + chunk + permute as the reference does)."""
    D = W.shape[0] // 2
    if x.dim() != 4 or W.shape[0] != 2 * D or not _tc_dtype_ok(x) or not _tc_shape_ok(D, W.shape[1], x):
        return None
    return _InProjPlanes.apply(x, W, bias)


def linear_tc(x, W, bias=None):
    """nn.Linear on the tensor-core kernel when eligible, else linear_ts (library GEMM, tall-skinny weight gradient)."""
    if _tc_dtype_ok(x) and _tc_shape_ok(W.shape[0], W.shape[1], x):
        return _LinearTC.apply(x, W, bias)
    return linear_ts(x, W, bias)


# ---- row-wise LayerNorm (GroupMambaLayer.norm) ------------------------------------------------------
class _LayerNormRows(torch.autograd.Function):
    """nn.LayerNorm over the last dimension (C <= 512) of a channels-last tensor: ops.layernorm_fwd/bwd. Runs in the
    dtype of x with fp32 statistics (under autocast nn.LayerNorm runs in fp32 as well; x is fp32 there)."""

    @staticmethod
    @_custom_fwd
    def forward(ctx, x, weight, bias, eps):
        xc = x.contiguous()
        w = weight.float() if weight is not None else None
        b = bias.float() if bias is not None else None
        y, stats = ops.layernorm_fwd(xc, w, b, eps)
        ctx.save_for_backward(xc, w, stats)
        ctx.has = (weight is not None, bias is not None)
        return y

    @staticmethod
    @_custom_bwd
    def backward(ctx, dy):
        xc, w, stats = ctx.saved_tensors
        dx, dw, db = ops.layernorm_bwd(xc, w, dy.to(xc.dtype), stats)
        return dx, (dw if ctx.has[0] else None), (db if ctx.has[1] else None), None


def layer_norm_rows(x, weight, bias, eps):
    _need_cuda(x, "layer_norm_rows")
    if torch.is_autocast_enabled("cuda") and x.dtype in (torch.float16, torch.bfloat16):
        x = x.float()      # nn.LayerNorm is on autocast's fp32 list: 16-bit inputs are normalised in, and returned as, fp32
    if x.shape[-1] > ops.LN_MAX_C or x.dtype not in (torch.float32, torch.float16, torch.bfloat16):
        return torch.nn.functional.layer_norm(x, (x.shape[-1],), weight, bias, eps)      # wide rows: library kernel
    return _LayerNormRows.apply(x, weight, bias, eps)


# ---- SS2D's depthwise 3 x 3 convolution with a reduction-shaped parameter gradient -----------------------
class _DWConv3(torch.autograd.Function):
    """y = conv2d(x, W (C,1,3,3), b, padding=1, groups=C) (library forward and input gradient); dW / db by
    ops.dwconv3_wgrad (ss2d.py:316-325, 512)."""

    @staticmethod
    def forward(ctx, x, W, bias):
        ctx.save_for_backward(x, W)
        ctx.has_bias = bias is not None
        return torch.nn.functional.conv2d(x, W, bias, padding=1, groups=W.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x, W = ctx.saved_tensors
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.nn.grad.conv2d_input(x.shape, W.to(dy.dtype), dy, padding=1, groups=W.shape[0]).to(x.dtype)
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dW, db = ops.dwconv3_wgrad(x.float().contiguous(), dy.float().contiguous(), ctx.has_bias)
            dW = dW.to(W.dtype)
        return dx, dW, db


class _DWConv3SiLU(torch.autograd.Function):
    """SiLU(conv2d(x, W (C,1,3,3), b, padding=1, groups=C)) (ss2d.py:512-513) as ONE kernel (ops.dwconv3_act); backward: the
    pre-activation gradient is recomputed from x in one pass, the input gradient is the flipped-kernel pass over it, dW / db
    come from ops.dwconv3_wgrad. Runs in the autocast dtype like nn.Conv2d."""

    @staticmethod
    def forward(ctx, x, W, bias):
        if torch.is_autocast_enabled("cuda"):
            x = x.to(torch.get_autocast_dtype("cuda"))
        x = x.contiguous()
        ctx.save_for_backward(x, W, bias)
        return ops.dwconv3_act(0, x, W, bias)

    @staticmethod
    def backward(ctx, dy):
        x, W, bias = ctx.saved_tensors
        dpre = ops.dwconv3_act(1, x, W, bias, dy.to(x.dtype).contiguous())
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = ops.dwconv3_act(2, dpre, W, None)
        if ctx.needs_input_grad[1] or (bias is not None and ctx.needs_input_grad[2]):
            dW, db = ops.dwconv3_wgrad(x.float(), dpre.float(), bias is not None)
            dW = dW.to(W.dtype)
            db = None if db is None else db.to(bias.dtype)
        return dx, dW, db


class _DWConv3SiLUPlanes(torch.autograd.Function):
    """u (B, 2 D, L) = [SiLU(conv(x)) | its transposed image]: ss2d.py:512-513 and the two input planes of the K = 4 scan
    (directions 1 / 3 read the natural plane, 2 / 4 the transposed one as row-major traversals) in ONE kernel — what the
    reference does with conv, SiLU and CrossScan's permuted copies (csms6s.py:11-29). Backward: one pass adds the two planes'
    gradients (the transposed one through a shared-memory tile) and applies SiLU'; then the flipped-kernel pass."""

    @staticmethod
    def forward(ctx, x, W, bias):
        if torch.is_autocast_enabled("cuda"):
            x = x.to(torch.get_autocast_dtype("cuda"))
        x = x.contiguous()
        ctx.save_for_backward(x, W, bias)
        return ops.dwconv3_act_planes_fwd(x, W, bias)

    @staticmethod
    def backward(ctx, du):
        x, W, bias = ctx.saved_tensors
        dpre = ops.dwconv3_act_planes_bwd(x, W, bias, du.to(x.dtype).contiguous())
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = ops.dwconv3_act(2, dpre, W, None)
        if ctx.needs_input_grad[1] or (bias is not None and ctx.needs_input_grad[2]):
            dW, db = ops.dwconv3_wgrad(x.float(), dpre.float(), bias is not None)
            dW = dW.to(W.dtype)
            db = None if db is None else db.to(bias.dtype)
        return dx, dW, db


def dwconv3_silu_planes(x, W, bias):
    """(B, 2 D, H W) natural + transposed planes of SiLU(conv(x)), or None when the shape is not eligible."""
    _need_cuda(x, "dwconv3_silu_planes")
    if not ops.dwconv3_act_planes_ok(x):
        return None
    return _DWConv3SiLUPlanes.apply(x, W, bias)


def dwconv3_silu(x, W, bias):
    """SiLU(depthwise 3 x 3 conv) as one kernel (weights given explicitly: the grouped layer assembles them per call)."""
    _need_cuda(x, "dwconv3_silu")
    return _DWConv3SiLU.apply(x, W, bias)


def dwconv3(x, conv: "torch.nn.Conv2d"):
    """SS2D.conv2d through _DWConv3 when it is the reference's depthwise 3 x 3 / padding 1 layer on a CUDA tensor."""
    _need_cuda(x, "dwconv3")
    ok = (conv.kernel_size == (3, 3) and conv.padding == (1, 1) and conv.stride == (1, 1) and
          conv.dilation == (1, 1) and conv.groups == conv.in_channels == conv.out_channels and conv.padding_mode == "zeros" and
          x.shape[0] * x.shape[2] * x.shape[3] >= _TS_MIN_ROWS)
    return _DWConv3.apply(x, conv.weight, conv.bias) if ok else conv(x)


class _FFNDepthwise(torch.autograd.Function):
    """The depthwise stack between fc1 and fc2 of PVT2FFN / custom_ffn on the channels-last token tensor (csrc/ffn_dw.cu):
        y1  = GELU(dw3x3(h) + b)                                                   groupmamba.py:76-78, custom_mlp.py:363-364
        out = y1 + cat(y1_id, dw3x3(y1_3), dw5x5(y1_5), dw7x7(y1_7))   (custom_ffn)  custom_mlp.py:323-336
    h: (B, L, C) contiguous, hw = (H, W). ms = None (PVT2FFN) or the six multi-scale tensors (w3, b3, w5, b5, w7, b7).
    Two launches forward (one without the multi-scale block); backward: the data gradient is three stencil launches
    (multi-scale transposed + residual; GELU' on the recomputed pre-activation; 3x3 transposed), the parameter gradients
    one reduction per convolution. Saved: h and y1 — what the reference's autograd keeps is h, the pre-activation, y1, the
    three splits and their outputs."""

    @staticmethod
    @_custom_fwd
    def forward(ctx, h, hw, w3, b3, *ms):
        C = h.shape[-1]
        h = h.contiguous()
        y1 = ops.dwnhwc_stencil(h, hw, [(C, 3, w3, b3)], epi=ops.EPI_GELU)
        ctx.hw, ctx.has_ms = hw, len(ms) > 0
        if ctx.has_ms:
            gc = ms[0].shape[0]
            ctx.gc = gc
            segs = [(C - 3 * gc, 1, None, None), (C - 2 * gc, 3, ms[0], ms[1]), (C - gc, 5, ms[2], ms[3]), (C, 7, ms[4], ms[5])]
            out = ops.dwnhwc_stencil(y1, hw, segs, epi=ops.EPI_RESIDUAL)
            ctx.save_for_backward(h, y1, w3, b3, *ms)
        else:
            out = y1
            ctx.save_for_backward(h, w3, b3)
        return out

    @staticmethod
    @_custom_bwd
    def backward(ctx, dout):
        hw = ctx.hw
        dout = dout.contiguous()
        if ctx.has_ms:
            h, y1, w3, b3, *ms = ctx.saved_tensors
        else:
            h, w3, b3 = ctx.saved_tensors
            ms = []
        C = h.shape[-1]
        if dout.dtype != h.dtype:
            dout = dout.to(h.dtype)
        grads_ms = []
        if ctx.has_ms:
            gc = ctx.gc
            segs = [(C - 3 * gc, 1, None, None), (C - 2 * gc, 3, ms[0], None), (C - gc, 5, ms[2], None), (C, 7, ms[4], None)]
            dy1 = ops.dwnhwc_stencil(dout, hw, segs, flip=True, epi=ops.EPI_RESIDUAL)
            for i, k in enumerate((3, 5, 7)):
                c0 = C - (3 - i) * gc
                dW, db = ops.dwnhwc_wgrad(y1, dout, hw, c0, c0 + gc, k, True)
                grads_ms += [dW.to(ms[2 * i].dtype), db.to(ms[2 * i + 1].dtype)]
        else:
            dy1 = dout
        dz = ops.dwnhwc_stencil(h, hw, [(C, 3, w3, b3)], epi=ops.EPI_DGELU_MUL, aux=dy1)
        dh = ops.dwnhwc_stencil(dz, hw, [(C, 3, w3, None)], flip=True, epi=ops.EPI_NONE) if ctx.needs_input_grad[0] else None
        dW3, db3 = ops.dwnhwc_wgrad(h, dz, hw, 0, C, 3, True)
        return (dh, None, dW3.to(w3.dtype), db3.to(b3.dtype), *grads_ms)


def ffn_depthwise(h, hw, conv3: "torch.nn.Conv2d", ms_convs=None):
    """h (B, L, C) -> the input of fc2. conv3: the DWConv's nn.Conv2d; ms_convs: (dwconv_3x3, dwconv_5x5, dwconv_7x7) or None."""
    _need_cuda(h, "ffn_depthwise")
    ms = []
    if ms_convs is not None:
        for m in ms_convs:
            ms += [m.weight, m.bias]
    return _FFNDepthwise.apply(h, hw, conv3.weight, conv3.bias, *ms)
