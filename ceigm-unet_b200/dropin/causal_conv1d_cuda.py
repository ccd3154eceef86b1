"""Drop-in for `causal_conv1d_cuda`, the extension module of causal-conv1d 1.1.x, which mamba_ssm's `mamba_inner_fn` calls:

    causal_conv1d_fwd(x, weight, bias_, seq_idx_, silu_activation) -> out
    causal_conv1d_bwd(x, weight, bias_, dout, seq_idx_, dx_, silu_activation) -> [dx, dweight, dbias]
    causal_conv1d_update(x, conv_state, weight, bias_, silu_activation) -> out       (conv_state updated in place)

x (batch, dim, L) with stride 1 along L, weight (dim, width), bias_ (dim) or None. dx is written into dx_ when it is given;
dweight / dbias have weight's dtype, and dbias is None without a bias. seq_idx_ must be None: RuntimeError otherwise.
"""
from .. import ops


def _no_seq_idx(seq_idx_):
    if seq_idx_ is not None:
        raise RuntimeError("causal_conv1d_cuda: seq_idx is not supported")


def causal_conv1d_fwd(x, weight, bias_, seq_idx_, silu_activation):
    _no_seq_idx(seq_idx_)
    return ops.conv1d_fwd(x, weight, bias_, bool(silu_activation))


def causal_conv1d_bwd(x, weight, bias_, dout, seq_idx_, dx_, silu_activation):
    _no_seq_idx(seq_idx_)
    return list(ops.conv1d_bwd(x, weight, bias_, dout, bool(silu_activation), dx=dx_))


def causal_conv1d_update(x, conv_state, weight, bias_, silu_activation):
    return ops.conv1d_update(x, conv_state, weight, bias_, bool(silu_activation))
