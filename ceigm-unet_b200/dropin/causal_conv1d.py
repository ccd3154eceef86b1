"""Drop-in for the `causal_conv1d` package (1.1.x), which mamba_ssm's `mamba_simple.Mamba` imports:
`causal_conv1d_fn(x, weight, bias=None, seq_idx=None, activation=None)` and
`causal_conv1d_update(x, conv_state, weight, bias=None, activation=None)`."""
from ..functional import causal_conv1d_fn, causal_conv1d_update  # noqa: F401
