"""GPU tests of the selective scan's output gate, out_z = y * silu(z) with dz from the backward (ss2d_scan_fwd_gated /
ss2d_scan_bwd_gated, `selective_scan(..., z=)`, and the mamba_ssm drop-in `selective_scan_cuda`), through every forward family.

Reference: the float64 recurrence of test_scan_state_gpu.py differentiated by autograd, composed with the gate by the chain
rule (the scan's gradients are those of dout = dout_z * silu(z); out_z = y silu(z) and dz = dout_z y silu'(z) in float64), and
the oracle's selective_scan_ref(..., z=) for the drop-in. Tolerance: max|got - ref| / max|ref| per tensor, 1e-3 for fp32 and
2e-2 for 16-bit I/O."""
import pytest
import torch
import torch.nn.functional as F

from test_scan_state_gpu import NAMES, _inputs, _reference, _rel

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _restore_defaults():
    yield
    from ceigm_unet_b200 import _lib
    torch.use_deterministic_algorithms(False)
    _lib.test_force_path(0)


def _gate_inputs(t, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    b, dim, L = t["delta"].shape
    t["z"] = (2 * torch.randn(b, dim, L, device="cuda", generator=gen)).to(t["u"].dtype)
    return t


def _gated_reference(t, softplus, hw=None, dirs=None):
    z = t["z"].double().requires_grad_(True)
    s = F.silu(z)
    ref = _reference(dict(t, dout=t["dout"].double() * s.detach()), softplus, hw, dirs)
    y = ref["out"]
    out_z = y * s
    (out_z * t["dout"].double()).sum().backward()
    return dict(ref, out_z=out_z.detach(), dz=z.grad)


def _run_gated(t, softplus, hw=None, dirs=None, states=True, use_ckpt=True, z=None):
    from ceigm_unet_b200 import _lib, ops
    pr = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], softplus, hw=hw, dirs=dirs)
    z = t["z"] if z is None else z
    _lib.launch_count(reset=True)
    out, x, out_z = pr.forward(want_state=True, h0=t["h0"] if states else None, z=z)
    fwd_launches = _lib.launch_count()
    last = x[:, :, -1, 1::2].clone()
    grads = pr.backward(t["dout"].to(pr.out_dtype), x if use_ckpt else None, h0=t["h0"] if states else None,
                        dlast=t["dlast"] if states else None, want_dh0=states, z=z, out=out)
    got = {"out": out, "out_z": out_z, "last": last, **dict(zip(NAMES + ["dz"], grads))}
    if states:
        got["dh0"] = grads[8]
    return got, fwd_launches


# id: (batch, dim, L, N, G, hw, dirs, dtype, softplus, forced path policy, scan_fwdr applies the gate itself)
CASES = {
    "fwdr32": (2, 64, 256, 16, 2, None, None, torch.float32, True, 1, True),             # scan_fwdr R = 1
    "fwdr32_N8_nosp": (2, 64, 256, 8, 1, None, None, torch.float32, False, 1, True),
    "fwdr16_dirs13": (2, 48, 400, 12, 2, (20, 20), [1, 3], torch.float32, True, 2, True),  # scan_fwdr R = 2, reversed rows
    "segmented": (2, 32, 640, 16, 1, None, None, torch.float32, False, 4, False),         # gate after the fix-up
    "fwd8_dirs1234": (2, 64, 144, 16, 4, (12, 12), [1, 2, 3, 4], torch.float32, True, 3, False),   # scan_fwd
    "N1_n1": (2, 64, 784, 1, 4, (28, 28), [1, 3, 1, 3], torch.float32, True, 0, False),  # scan_n1
    "N1_par_dirs24": (2, 32, 196, 1, 4, (14, 14), [1, 2, 3, 4], torch.float32, True, 0, False),   # scan_par
    "N4_L60": (2, 32, 60, 4, 1, None, None, torch.float32, True, 0, False),
    "N40_two_passes": (2, 16, 100, 40, 2, None, None, torch.float32, True, 0, False),   # gate after the last state pass
    "N16_bf16": (2, 64, 256, 16, 2, None, None, torch.bfloat16, True, 0, False),
    "N1_bf16_dirs": (2, 32, 196, 1, 4, (14, 14), [1, 3, 1, 3], torch.bfloat16, True, 0, False),
}
_REF = {}


def _case_inputs(case, seed=11):
    b, dim, L, N, G, hw, dirs, dtype, sp, policy, fused = CASES[case]
    return _gate_inputs(_inputs(b, dim, L, N, G, dtype, seed=seed), seed + 1)


@pytest.mark.parametrize("use_ckpt", [True, False], ids=["ckpt", "no_ckpt"])
@pytest.mark.parametrize("states", [True, False], ids=["states", "no_states"])
@pytest.mark.parametrize("case", list(CASES))
def test_gated_parity(case, states, use_ckpt):
    from ceigm_unet_b200 import _lib
    b, dim, L, N, G, hw, dirs, dtype, sp, policy, fused = CASES[case]
    t = _case_inputs(case)
    if not states:
        t["h0"], t["dlast"] = torch.zeros_like(t["h0"]), torch.zeros_like(t["dlast"])
    _lib.test_force_path(policy)
    got, launches = _run_gated(t, sp, hw, dirs, states=states, use_ckpt=use_ckpt)
    if fused:
        assert launches == 1, launches          # scan_fwdr wrote out_z: no separate gate pass
    key = (case, states)
    if key not in _REF:
        _REF[key] = _gated_reference(t, sp, hw, dirs)
    ref = _REF[key]
    tol = 1e-3 if dtype == torch.float32 else 2e-2
    bad = {k: _rel(got[k], ref[k]) for k in got if got[k] is not None and _rel(got[k], ref[k]) > tol}
    assert not bad, bad


@pytest.mark.parametrize("case", ["fwdr32", "fwdr16_dirs13"])
def test_misaligned_gate_takes_the_standalone_pass(case):
    """z one element off a 16-byte boundary: scan_fwdr runs ungated and the scalar gate kernel follows, same results."""
    from ceigm_unet_b200 import _lib
    b, dim, L, N, G, hw, dirs, dtype, sp, policy, _ = CASES[case]
    t = _case_inputs(case)
    _lib.test_force_path(policy)
    zbuf = torch.empty(t["z"].numel() + 1, dtype=t["z"].dtype, device="cuda")
    z = zbuf[1:].view_as(t["z"])
    z.copy_(t["z"])
    got, launches = _run_gated(t, sp, hw, dirs, z=z)
    assert launches == 2, launches
    ref, _ = _run_gated(t, sp, hw, dirs)
    for k in ref:
        assert _rel(got[k], ref[k]) <= 1e-6, k


def test_oracle_selective_scan_ref_with_z():
    """The drop-in against the oracle's restatement of the reference (fp32 autograd), stateless, SCAN layout."""
    from ceigm_unet_b200.dropin import selective_scan_cuda as m
    from oracle.selective_scan_ref import make_inputs, selective_scan_ref
    inp = make_inputs(2, 64, 256, 16, groups=2, seed=3, device="cuda")
    z = torch.randn_like(inp["u"])
    leaf = {k: inp[k].clone().requires_grad_(True) for k in ("u", "delta", "A", "B", "C", "D", "delta_bias")}
    zl = z.clone().requires_grad_(True)
    ref = selective_scan_ref(leaf["u"], leaf["delta"], leaf["A"], leaf["B"], leaf["C"], leaf["D"], zl, leaf["delta_bias"], True)
    ref.backward(inp["dout"])
    out, x, out_z = m.fwd(inp["u"], inp["delta"], inp["A"], inp["B"], inp["C"], inp["D"], z, inp["delta_bias"], True)
    grads = m.bwd(inp["u"], inp["delta"], inp["A"], inp["B"], inp["C"], inp["D"], z, inp["delta_bias"], inp["dout"], x, out,
                  None, True, False)
    assert _rel(out_z, ref.detach()) <= 1e-3
    for name, g, k in zip(NAMES, grads, ("u", "delta", "A", "B", "C", "D", "delta_bias")):
        assert _rel(g, leaf[k].grad) <= 1e-3, name
    assert _rel(grads[7], zl.grad) <= 1e-3


# SCAN-layout calls of `selective_scan`: (batch, dim, L, N, G, forced path policy)
EQ_CASES = {"fwdr_R1": (2, 64, 256, 16, 2, 1), "fwdr_R2": (2, 64, 256, 16, 2, 2), "fwd8": (2, 64, 144, 16, 4, 3),
            "segmented": (2, 32, 640, 16, 1, 4), "N1": (2, 64, 784, 1, 4, 0), "N4": (2, 32, 64, 4, 1, 0),
            "N40": (2, 16, 100, 40, 2, 0)}


@pytest.mark.parametrize("case", list(EQ_CASES))
def test_gated_equals_ungated_then_torch_gate(case):
    """selective_scan(z=) == selective_scan() * F.silu(z) through autograd, every gradient included."""
    import ceigm_unet_b200 as P
    b, dim, L, N, G, policy = EQ_CASES[case]
    t = _gate_inputs(_inputs(b, dim, L, N, G, torch.float32, seed=5), 6)
    P._lib.test_force_path(policy)
    keys = ("u", "delta", "A", "B", "C", "D", "delta_bias", "h0", "z")
    res = []
    for gated in (True, False):
        lf = {k: t[k].clone().requires_grad_(True) for k in keys}
        args = [lf[k] for k in keys[:7]]
        y, last = P.selective_scan(*args, delta_softplus=True, initial_state=lf["h0"], return_last_state=True,
                                   z=lf["z"] if gated else None)
        if not gated:
            y = y * F.silu(lf["z"])
        ((y * t["dout"]).sum() + (last * t["dlast"]).sum()).backward()
        res.append({"y": y.detach(), "last": last.detach(), **{k: lf[k].grad for k in keys}})
    for k in res[1]:
        assert _rel(res[0][k], res[1][k]) <= 1e-5, k


@pytest.mark.parametrize("case", ["fwdr32", "segmented", "N1_n1", "N40_two_passes", "N16_bf16"])
def test_deterministic_gated_is_bit_identical(case):
    """Three eager calls and two CUDA-graph replays of the gated forward + backward give the same bits."""
    from ceigm_unet_b200 import _lib, ops
    b, dim, L, N, G, hw, dirs, dtype, sp, policy, _ = CASES[case]
    t = _case_inputs(case)
    _lib.test_force_path(policy)
    torch.use_deterministic_algorithms(True)

    def step():
        pr = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], sp, hw=hw, dirs=dirs)
        out, x, out_z = pr.forward(True, h0=t["h0"], z=t["z"])
        g = pr.backward(t["dout"].to(pr.out_dtype), x, h0=t["h0"], dlast=t["dlast"], want_dh0=True, z=t["z"], out=out)
        return [out, out_z, x] + [v for v in g if v is not None]

    first = [v.clone() for v in step()]
    for _ in range(2):
        assert all(torch.equal(a, b) for a, b in zip(first, step()))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()                                   # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(first, static))


def test_selective_scan_z_in_a_cuda_graph():
    import ceigm_unet_b200 as P
    t = _case_inputs("fwdr32")
    keys = ("u", "delta", "A", "B", "C", "D", "delta_bias", "z")
    lf = {k: t[k].clone().requires_grad_(True) for k in keys}

    def step():
        for v in lf.values():
            v.grad = None
        y = P.selective_scan(*[lf[k] for k in keys[:7]], delta_softplus=True, z=lf["z"])
        (y * t["dout"]).sum().backward()
        return [y.detach()] + [lf[k].grad for k in keys]

    eager = [v.clone() for v in step()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, static):
        assert _rel(b, a) <= 1e-5


def test_dropin_without_z_equals_core_bit_for_bit():
    """SelectiveScanMamba's calls (csms6s.py:324-344) pass z_ = None: the results are those of selective_scan_cuda_core.
    (Deterministic mode: the default backward sums dB / dC with atomics, so two of its calls may differ in the last bits.)"""
    from ceigm_unet_b200.dropin import selective_scan_cuda as m
    from ceigm_unet_b200.dropin import selective_scan_cuda_core as core
    torch.use_deterministic_algorithms(True)
    for dtype in (torch.float32, torch.bfloat16):
        t = _inputs(2, 64, 256, 16, 2, dtype, seed=21)
        t["dout"] = t["dout"].to(dtype)
        a = [t[k] for k in ("u", "delta", "A", "B", "C", "D")]
        out, x = m.fwd(*a, None, t["delta_bias"], True)
        out_c, x_c = core.fwd(*a, t["delta_bias"], True, 1)
        assert torch.equal(out, out_c) and torch.equal(x[:, :, -1, 1::2], x_c[:, :, -1, 1::2])
        g = m.bwd(*a, None, t["delta_bias"], t["dout"], x, None, None, True, False)
        g_c = core.bwd(*a, t["delta_bias"], t["dout"], x_c, True, 1)
        assert len(g) == 7 and all(torch.equal(p, q) for p, q in zip(g, g_c))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_dropin_with_z(dtype):
    from ceigm_unet_b200 import ops
    from ceigm_unet_b200.dropin import selective_scan_cuda as m
    torch.use_deterministic_algorithms(True)          # bit-for-bit comparisons of two backward calls below
    t = _gate_inputs(_inputs(2, 64, 256, 16, 2, dtype, seed=23), 24)
    t["dout"] = t["dout"].to(dtype)
    a = [t[k] for k in ("u", "delta", "A", "B", "C", "D")]
    out, x, out_z = m.fwd(*a, t["z"], t["delta_bias"], True)
    assert out_z.dtype == dtype
    g = m.bwd(*a, t["z"], t["delta_bias"], t["dout"], x, out, None, True, False)
    assert len(g) == 8 and g[7].dtype == dtype
    dz_buf = torch.full_like(t["z"], float("nan"))
    g2 = m.bwd(*a, t["z"], t["delta_bias"], t["dout"], x, out, dz_buf, True, True)
    assert len(g2) == 9 and g2[7] is dz_buf
    assert torch.equal(dz_buf, g[7]) and all(torch.equal(p, q) for p, q in zip(g[:7], g2[:7]))
    assert torch.equal(g2[8], out_z)
    # against the ScanProblem path the module is built on
    pr = ops.ScanProblem(*a, t["delta_bias"], True)
    o2, _, oz2 = pr.forward(True, z=t["z"])
    assert torch.equal(o2, out) and torch.equal(oz2, out_z)
