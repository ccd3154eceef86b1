"""Float64 references for Mamba-2's chunked selective scan (mamba_ssm 2.x's mamba_chunk_scan_combined).

`ssd_recurrence` is the definition: the per-position recurrence
    t_l = clamp(softplus?(dt_l + dt_bias), dt_limit),  H_l = exp(t_l A) H_{l-1} + t_l x_l (x) B_l,  y_l = C_l . H_l + D x_l,
    out_l = y_l silu(z_l) (with z),
with H_{-1} = initial_states (zeros when None). `ssd_chunked` restates it in chunks (mamba_ssm's `ssd_minimal_discrete`:
intra-chunk scores, chunk states, state passing, state-to-output), in a handful of einsums, so that long sequences and
autograd gradients are cheap. Both take torch tensors of any dtype and device and compute in float64 there.
Shapes: x, z (b, L, h, p), dt (b, L, h), A (h), B, C (b, L, g, n), D (h) or (h, p), dt_bias (h), initial_states (b, h, p, n).
Both return (out, final_states (b, h, p, n)).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def _prep(x, dt, A, B, C, D, z, dt_bias, dt_softplus, dt_limit):
    f = lambda t: None if t is None else t.double()   # noqa: E731
    x, dt, A, B, C, D, z, dt_bias = map(f, (x, dt, A, B, C, D, z, dt_bias))
    h, g = x.shape[2], B.shape[2]
    if dt_bias is not None:
        dt = dt + dt_bias
    if dt_softplus:
        dt = F.softplus(dt)
    if tuple(dt_limit) != (0.0, math.inf):
        dt = dt.clamp(dt_limit[0], dt_limit[1])
    B = B.repeat_interleave(h // g, dim=2)
    C = C.repeat_interleave(h // g, dim=2)
    return x, dt, A, B, C, D, z


def _finish(y, x, D, z):
    if D is not None:
        y = y + x * (D[:, None] if D.dim() == 1 else D)
    if z is not None:
        y = y * F.silu(z)
    return y


def ssd_recurrence(x, dt, A, B, C, D=None, z=None, dt_bias=None, initial_states=None, dt_softplus=False,
                   dt_limit=(0.0, math.inf)):
    x, t, A, B, C, D, z = _prep(x, dt, A, B, C, D, z, dt_bias, dt_softplus, dt_limit)
    b, L, h, p = x.shape
    n = B.shape[-1]
    H = x.new_zeros(b, h, p, n) if initial_states is None else initial_states.double()
    ys = []
    for l in range(L):
        H = torch.exp(t[:, l] * A)[..., None, None] * H + (t[:, l, :, None] * x[:, l])[..., None] * B[:, l, :, None, :]
        ys.append(torch.einsum("bhpn,bhn->bhp", H, C[:, l]))
    return _finish(torch.stack(ys, 1), x, D, z), H


def _segsum(a):
    """a (..., T) -> (..., T, T) with [i, j] = sum_{j < k <= i} a_k for j <= i and -inf above the diagonal."""
    T = a.shape[-1]
    cs = torch.cumsum(a, -1)
    s = cs[..., :, None] - cs[..., None, :]
    mask = torch.tril(torch.ones(T, T, dtype=torch.bool, device=a.device))
    return s.masked_fill(~mask, -math.inf)


def ssd_chunked(x, dt, A, B, C, chunk_size, D=None, z=None, dt_bias=None, initial_states=None, dt_softplus=False,
                dt_limit=(0.0, math.inf)):
    x, t, A, B, C, D, z = _prep(x, dt, A, B, C, D, z, dt_bias, dt_softplus, dt_limit)
    b, L, h, p = x.shape
    n = B.shape[-1]
    Q = chunk_size
    pad = (-L) % Q
    X = F.pad(x * t[..., None], (0, 0, 0, 0, 0, pad))          # padded positions: t = 0, x = B = C = 0
    a = F.pad(t * A, (0, 0, 0, pad))
    Bp = F.pad(B, (0, 0, 0, 0, 0, pad))
    Cp = F.pad(C, (0, 0, 0, 0, 0, pad))
    c = (L + pad) // Q
    X, Bp, Cp = (v.reshape(b, c, Q, h, -1) for v in (X, Bp, Cp))
    a = a.reshape(b, c, Q, h).permute(0, 3, 1, 2)               # (b, h, c, Q)
    cum = torch.cumsum(a, -1)
    Ld = torch.exp(_segsum(a))                                   # (b, h, c, Q, Q)
    y_diag = torch.einsum("bclhn,bcshn,bhcls,bcshp->bclhp", Cp, Bp, Ld, X)
    decay_states = torch.exp(cum[..., -1:] - cum)
    states = torch.einsum("bclhn,bhcl,bclhp->bchpn", Bp, decay_states, X)
    h0 = x.new_zeros(b, 1, h, p, n) if initial_states is None else initial_states.double()[:, None]
    states = torch.cat([h0, states], 1)
    decay_chunk = torch.exp(_segsum(F.pad(cum[..., -1], (1, 0))))   # (b, h, c + 1, c + 1)
    new_states = torch.einsum("bhzc,bchpn->bzhpn", decay_chunk, states)
    states, final = new_states[:, :-1], new_states[:, -1]
    y_off = torch.einsum("bclhn,bchpn,bhcl->bclhp", Cp, states, torch.exp(cum))
    y = (y_diag + y_off).reshape(b, c * Q, h, p)[:, :L]
    return _finish(y, x, D, z), final
