"""GPU tests of the deterministic scan backward: under torch.use_deterministic_algorithms(True) every backward kernel family
(scan_bwd2, scan_bwd, the two d_state = 1 kernels of scan_n1, scan_par) gives bit-identical gradients across calls, streams
and CUDA-graph replays, with groups split over several CTAs (the case the default mode reduces with atomics). Each case is
also checked against the C/f64 oracle (rel <= 1e-3) and against the default mode (rel <= 1e-5: the two differ only in the
order of the fp32 sums; 16-bit outputs are compared after their rounding, within 1e-2).
Module level (SS2D, GroupMambaLayer, both FFNs, eager and graphed) runs in a subprocess that sets CUBLAS_WORKSPACE_CONFIG
before CUDA starts, so that torch's own GEMMs are reproducible too."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias"]


@pytest.fixture(autouse=True)
def _restore_defaults():
    yield
    from ceigm_unet_b200 import _lib
    torch.use_deterministic_algorithms(False)
    _lib.test_force_path(0)


def _order(k, H, W):
    """Natural pixel index of each scan position of direction k (1 row-major, 2 column-major, 3 / 4 reversed)."""
    idx = np.arange(H * W).reshape(H, W)
    o = (idx if k in (1, 3) else idx.T).reshape(-1)
    return o[::-1].copy() if k in (3, 4) else o


# id: (batch, dim, L, N, G, hw, dirs, dtype, out_float). Every case splits a group over more than one CTA.
CASES = {
    "bwd2_dirs13": (2, 384, 784, 16, 4, (28, 28), [1, 3, 1, 3], torch.float32, False),
    "bwd2_scan": (2, 384, 784, 16, 1, None, None, torch.float32, False),
    "bwd_N4": (2, 256, 784, 4, 2, None, None, torch.float32, False),
    "bwd_N16_dirs24": (2, 384, 784, 16, 4, (28, 28), [1, 2, 3, 4], torch.float32, False),
    "bwd_N40_two_passes": (2, 128, 300, 40, 2, None, None, torch.float32, False),
    "n1_rows": (2, 256, 784, 1, 4, (28, 28), [1, 3, 1, 3], torch.float32, False),
    "n1_rows_long_4100": (1, 32, 4100, 1, 1, None, None, torch.float32, False),
    "n1_rows_long_16384": (1, 64, 16384, 1, 4, None, None, torch.float32, False),
    "n1_one_row_L20": (4, 64, 20, 1, 2, None, None, torch.float32, False),
    "n1_one_row_L49": (4, 64, 49, 1, 2, (7, 7), [1, 3], torch.float32, False),
    "par_dirs24": (2, 64, 196, 1, 4, (14, 14), [1, 2, 3, 4], torch.float32, False),
    "bf16": (2, 384, 784, 16, 4, (28, 28), [1, 3, 1, 3], torch.bfloat16, False),
    "bf16_out_float": (2, 256, 196, 1, 4, (14, 14), [1, 3, 1, 3], torch.bfloat16, True),
}


def _inputs(b, dt, L, N, G, dtype, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    return dict(u=r(b, dt, L).to(dtype), delta=(0.5 * torch.rand(b, dt, L, device="cuda", generator=gen)).to(dtype),
                A=-0.5 * torch.rand(dt, N, device="cuda", generator=gen), B=r(b, G, N, L).to(dtype), C=r(b, G, N, L).to(dtype),
                D=r(dt), bias=0.5 * torch.rand(dt, device="cuda", generator=gen), dout=r(b, dt, L))


def _oracle(a, hw, dirs, G):
    """Reference gradients in the natural layout: the inputs of each group are permuted into its scan order, the oracle
    runs the sequential scan, and the results are permuted back."""
    from oracle import c_oracle
    n = {k: v.float().cpu().numpy() for k, v in a.items()}
    b, dt, L = n["u"].shape
    dpg = dt // G
    orders = [_order(k, *hw) for k in dirs] if hw else [np.arange(L)] * G
    def to_scan(x, per):      # per: channels per group on axis 1
        return np.concatenate([x[:, g * per:(g + 1) * per][..., orders[g]] for g in range(G)], axis=1)
    ref = c_oracle.scan_bwd(to_scan(n["u"], dpg), to_scan(n["delta"], dpg), n["A"], to_scan(n["B"], 1), to_scan(n["C"], 1),
                            n["D"], n["bias"], to_scan(n["dout"], dpg), True, acc="f64")
    for name, per in (("du", dpg), ("ddelta", dpg), ("dB", 1), ("dC", 1)):
        x, out = ref[name], np.empty_like(ref[name])
        for g in range(G):
            out[:, g * per:(g + 1) * per][..., orders[g]] = x[:, g * per:(g + 1) * per]
        ref[name] = out
    return ref


def _rel(got, want):
    got = got.float().cpu().numpy().astype(np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))


def _equal(g1, g2):
    return all((x is None and y is None) or torch.equal(x, y) for x, y in zip(g1, g2))


@pytest.mark.parametrize("case", sorted(CASES))
def test_deterministic_backward(case):
    from ceigm_unet_b200 import ops
    b, dt, L, N, G, hw, dirs, dtype, out_float = CASES[case]
    a = _inputs(b, dt, L, N, G, dtype, seed=len(case))
    pr = ops.ScanProblem(a["u"], a["delta"], a["A"], a["B"], a["C"], a["D"], a["bias"], True, out_float=out_float, hw=hw, dirs=dirs)
    out, x = pr.forward(True)
    dout = a["dout"].to(out.dtype)
    default = pr.backward(dout, x)
    torch.use_deterministic_algorithms(True)
    g1 = pr.backward(dout, x)
    assert _equal(g1, pr.backward(dout, x)) and _equal(g1, pr.backward(dout, x))
    # no checkpoints: the states are recomputed by a forward sweep into the workspace first
    g_nockpt = pr.backward(dout, None)
    assert _equal(g_nockpt, pr.backward(dout, None))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g_side = pr.backward(dout, x)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    assert _equal(g1, g_side)
    # captured once, replayed twice
    with torch.cuda.stream(side):
        pr.backward(dout, x)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_graph = pr.backward(dout, x)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert _equal(g1, g_graph)
    # accuracy: oracle, and the default mode (same arithmetic, other summation order)
    tol_ref, tol_def = (1e-3, 1e-5) if dtype == torch.float32 else (1e-2, 1e-2)
    ref = _oracle(dict(a, dout=dout), hw, dirs, G)
    for name, g, gn, gd in zip(NAMES, g1, g_nockpt, default):
        assert _rel(g, ref[name]) < tol_ref, name
        assert _rel(gn, ref[name]) < tol_ref, name
        assert _rel(g, gd.float().cpu().numpy()) < tol_def, name


def test_warn_only_also_takes_the_deterministic_kernels():
    import ceigm_unet_b200 as P
    from ceigm_unet_b200 import ops
    a = _inputs(2, 64, 16384, 1, 4, torch.float32, seed=3)
    pr = ops.ScanProblem(a["u"], a["delta"], a["A"], a["B"], a["C"], a["D"], a["bias"], True)
    _, x = pr.forward(True)
    P.launch_count(reset=True)
    pr.backward(a["dout"], x)
    default_launches = P.launch_count(reset=True)          # one kernel: atomics into the zeroed buffer
    torch.use_deterministic_algorithms(True, warn_only=True)
    g1, g2 = pr.backward(a["dout"], x), pr.backward(a["dout"], x)
    assert P.launch_count() == 2 * (default_launches + 2)   # + the slab fold and the finalize pass
    assert _equal(g1, g2)


def test_dropin_core_bwd_is_deterministic():
    from ceigm_unet_b200.dropin import selective_scan_cuda_core as core
    from oracle.selective_scan_ref import make_inputs
    inp = make_inputs(4, 384, 784, 16, groups=4, seed=1, device="cuda")
    args = (inp["u"], inp["delta"], inp["A"], inp["B"], inp["C"], inp["D"], inp["delta_bias"])
    _, x = core.fwd(*args, True, 1)
    torch.use_deterministic_algorithms(True)
    g = [core.bwd(*args, inp["dout"], x, True, 1) for _ in range(3)]
    assert _equal(g[0], g[1]) and _equal(g[0], g[2])


_MODULE_SCRIPT = textwrap.dedent("""
    import copy, sys
    import torch
    sys.path.insert(0, ROOT)
    import ceigm_unet_b200 as P
    torch.use_deterministic_algorithms(True)

    class Wrap(torch.nn.Module):
        def __init__(self, m, hw):
            super().__init__()
            self.m, self.hw = m, hw
        def forward(self, x):
            return self.m(x, *self.hw)

    def cases():
        yield "ss2d_k4_n16", lambda: P.SS2D(d_model=96, d_state=16, ssm_ratio=2.0, k_group=4), (2, 28, 28, 96)
        yield "gml_stage1", lambda: Wrap(P.GroupMambaLayer(64, 64), (56, 56)), (2, 3136, 64)
        yield "gml_stage4", lambda: Wrap(P.GroupMambaLayer(448, 448), (7, 7)), (2, 49, 448)
        yield "pvt2ffn", lambda: Wrap(P.PVT2FFN(64, 256), (56, 56)), (2, 3136, 64)
        yield "custom_ffn", lambda: Wrap(P.custom_ffn(64, 256), (56, 56)), (2, 3136, 64)

    def grads(fn, mod, x, gy):
        x.grad = None
        for p in mod.parameters():
            p.grad = None
        fn(x).backward(gy)
        torch.cuda.synchronize()
        return [x.grad.clone()] + [p.grad.clone() for p in mod.parameters() if p.grad is not None]

    bad = []
    for name, make, shape in cases():
        torch.manual_seed(0)
        eager = make().cuda()
        captured = copy.deepcopy(eager)
        x = torch.randn(*shape, device="cuda", requires_grad=True)
        gy = torch.randn(*shape, device="cuda")
        graphed = P.graphed(captured, (x.detach().clone().requires_grad_(True),))
        for tag, fn, mod in (("eager", eager, eager), ("graphed", graphed, captured)):
            a, b = grads(fn, mod, x, gy), grads(fn, mod, x, gy)
            if len(a) < 2 or not all(torch.equal(u, v) for u, v in zip(a, b)):
                bad.append(name + "/" + tag)
    print("NOT BIT-IDENTICAL:", bad)
    sys.exit(1 if bad else 0)
""")


def test_modules_are_bit_reproducible():
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    r = subprocess.run([sys.executable, "-c", "ROOT = %r\n" % ROOT + _MODULE_SCRIPT], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
