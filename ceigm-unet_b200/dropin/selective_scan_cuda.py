"""Drop-in for `selective_scan_cuda`, the extension module of mamba_ssm (requirements.txt:2), which the reference's
`SelectiveScanMamba` (model/gm/csms6s.py:324-344, model/vmamba/csms6s.py) calls:

    fwd(u, delta, A, B, C, D_, z_, delta_bias_, delta_softplus) -> [out, x] (+ [out_z] if z_ is given)
    bwd(u, delta, A, B, C, D_, z_, delta_bias_, dout, x_, out_, dz_, delta_softplus, recompute_out_z)
        -> [du, ddelta, dA, dB, dC, dD, ddelta_bias] (+ [dz] if z_) (+ [out_z] if recompute_out_z)

out_z = out * silu(z). With z_, dout is the gradient of out_z, out_ (the forward's out) is required, and dz_, when given, receives
dz in place. out has u's dtype. `x` keeps the convention x[:, :, -1, 1::2] == final state, as in the other two drop-ins; the
chunk checkpoints `bwd` uses sit in front of it in the same storage. recompute_out_z reruns the gated forward scan to produce
out_z (the bits the forward returned). Complex A and time-invariant (2-D) B / C are not supported: RuntimeError before any launch.
"""
from .. import ops


def _check(A, B, C):
    if A.is_complex():
        raise RuntimeError("selective_scan_cuda: complex A is not supported")
    if B.dim() < 3 or C.dim() < 3:
        raise RuntimeError("selective_scan_cuda: B and C must vary along the sequence ((batch, [groups,] dstate, seqlen))")


def fwd(u, delta, A, B, C, D_=None, z_=None, delta_bias_=None, delta_softplus=False):
    _check(A, B, C)
    res = ops.ScanProblem(u, delta, A, B, C, D_, delta_bias_, delta_softplus, out_float=False).forward(True, z=z_)
    return list(res)


def bwd(u, delta, A, B, C, D_, z_, delta_bias_, dout, x_=None, out_=None, dz_=None, delta_softplus=False,
        recompute_out_z=False):
    _check(A, B, C)
    if z_ is not None and out_ is None:
        raise RuntimeError("selective_scan_cuda.bwd: out_ is required when z_ is given")
    prob = ops.ScanProblem(u, delta, A, B, C, D_, delta_bias_, delta_softplus, out_float=False)
    grads = prob.backward(dout, x_, z=z_, out=out_)
    if z_ is not None and dz_ is not None:
        dz_.copy_(grads[7])
        grads[7] = dz_
    if z_ is not None and recompute_out_z:
        grads.append(prob.forward(True, z=z_)[2])       # with checkpoints: the forward's kernels, so the forward's bits
    return grads
