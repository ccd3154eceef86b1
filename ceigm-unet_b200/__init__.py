"""ceigm-unet_b200 — B200-native (sm_100a) implementation of GM-UNet's SS2D selective-scan hot path.

Layers (SURVEY.md §8b):
  b1  dropin/selective_scan_cuda_core.py, dropin/selective_scan_cuda_oflex.py, dropin/selective_scan_cuda.py (mamba_ssm's
      module, with the z gate) — the reference extension modules' `fwd` / `bwd` functions; `install_dropin()` registers them
      in sys.modules so that the reference's own `model/gm/csms6s.py` picks them up unchanged. dropin/causal_conv1d_cuda.py and
      dropin/causal_conv1d.py serve causal-conv1d 1.1.x, the convolution in front of every Mamba block's scan.
  b2  functional.py — SelectiveScanCore/Oflex, CrossScan[_k], CrossMerge[_k] autograd Functions; the Mamba functions
      selective_scan, selective_state_update, causal_conv1d_fn / _update, and mamba_chunk_scan_combined (Mamba-2's chunked
      scan, mamba_ssm 2.x's arguments, differentiable).
  b3  modules.py — SS2D, GroupMambaLayer (and the FFNs next to them: PVT2FFN, custom_ffn) with the reference's state_dict.
Underneath: ops.py -> _lib.py (ctypes) -> libss2d_b200.so (csrc/*.cu, C ABI in include/ss2d_b200.h).
There is no CPU or PyTorch fallback: without the built library every operator raises RuntimeError.
"""
from . import _lib, dist, functional, modules, ops                 # noqa: F401
from ._lib import build, launch_count, version                    # noqa: F401
from .functional import (CrossMerge, CrossMerge_1, CrossMerge_2, CrossMerge_3, CrossMerge_4, CrossScan,   # noqa: F401
                         CrossScan_1, CrossScan_2, CrossScan_3, CrossScan_4, SelectiveScanCore, SelectiveScanOflex,
                         causal_conv1d_fn, causal_conv1d_update, mamba_chunk_scan_combined, selective_scan,
                         selective_state_update)
from .modules import SS2D, GroupMambaLayer, LayerNormRows, PVT2FFN, custom_ffn, mamba_init             # noqa: F401


def graphed(module, sample_args, num_warmup_iters: int = 3):
    """Capture the forward AND backward of `module` (an SS2D / GroupMambaLayer, or any nn.Module built from this
    package's autograd Functions) into CUDA graphs and return the graphed callable (torch.cuda.make_graphed_callables).

    The live GM-UNet regime is launch-bound — about 120 small kernels per GroupMambaLayer call (groupmamba.py:127-159),
    2 650 per model forward (SURVEY.md §8-f2) — so replaying one graph per layer takes the host launches off the
    critical path. Everything the operators do is capturable: outputs are allocated with torch on the capturing
    stream, the C ABI never synchronises, and the TMA tensor maps are passed by value as kernel parameters.
    `sample_args`: a tuple of tensors with the shapes / dtypes / requires_grad flags of the real inputs.
    Capture BEFORE the module's first eager backward: autograd pins every parameter's gradient accumulator to the stream
    of its first use, and an accumulator created on the legacy default stream cannot be joined from a capturing stream
    (cudaErrorStreamCaptureImplicit).
    torch.use_deterministic_algorithms() is read when the graph is captured: the captured backward keeps the scan kernels
    (atomic or deterministic) of that moment, whatever the switch says at replay."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("graphed() needs a CUDA device: there is no CPU fallback")
    return torch.cuda.make_graphed_callables(module, tuple(sample_args), num_warmup_iters=num_warmup_iters)


def install_dropin() -> None:
    """Make `import selective_scan_cuda_core` / `selective_scan_cuda_oflex` / `selective_scan_cuda` (mamba_ssm's module)
    resolve to this package's modules (the reference imports them at module import time inside try/except:
    model/gm/csms6s.py:209-220), and `import causal_conv1d_cuda` / `from causal_conv1d import causal_conv1d_fn,
    causal_conv1d_update` (mamba_ssm's convolution) too."""
    import sys

    from .dropin import causal_conv1d, causal_conv1d_cuda, selective_scan_cuda, selective_scan_cuda_core, selective_scan_cuda_oflex
    sys.modules["selective_scan_cuda_core"] = selective_scan_cuda_core
    sys.modules["selective_scan_cuda_oflex"] = selective_scan_cuda_oflex
    sys.modules["selective_scan_cuda"] = selective_scan_cuda
    sys.modules["causal_conv1d_cuda"] = causal_conv1d_cuda
    sys.modules["causal_conv1d"] = causal_conv1d
