"""GPU tests of state passing in the selective scan: a forward that starts from a given state h0, and a backward that takes the
gradient of the final state (dlast) and returns the gradient of h0 (dh0), through every kernel family.

Reference: the recurrence h_l = exp(delta_l A) h_(l-1) + delta_l u_l B_l, h_(-1) = h0, out_l = C_l . h_l + D u_l in float64 on
the GPU, differentiated by torch autograd with loss = <out, dout> + <h_(L-1), dlast>. Tolerance: max|got - ref| / max|ref| per
tensor, 1e-3 for fp32 and 2e-2 for 16-bit I/O.
Also: chaining two calls equals one call; zero states reproduce the stateless call bit for bit; the public `selective_scan`
through autograd; deterministic mode is bit-identical across calls and CUDA-graph replays."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

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


def _inputs(b, dim, L, N, G, dtype, seed, u_mod=0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    ud = u_mod or dim
    t = dict(u=r(b, ud, L).to(dtype), delta=(0.5 * torch.rand(b, dim, L, device="cuda", generator=gen)).to(dtype),
             A=-0.5 * torch.rand(dim, N, device="cuda", generator=gen), B=r(b, G, N, L).to(dtype), C=r(b, G, N, L).to(dtype),
             D=r(dim), delta_bias=0.5 * torch.rand(dim, device="cuda", generator=gen))
    t["h0"] = r(b, dim, N)
    t["dlast"] = r(b, dim, N)
    t["dout"] = r(b, ud, L)
    return t


def _reference(t, softplus, hw=None, dirs=None, u_mod=0):
    """float64 forward + autograd backward -> dict of out, last, and the gradients (du per channel when u_mod > 0)."""
    b, dim, L = t["delta"].shape
    G, N = t["B"].shape[1], t["A"].shape[1]
    dpg, dev = dim // G, t["delta"].device
    leaf = {k: t[k].detach().double().requires_grad_(True) for k in ("delta", "A", "B", "C", "D", "delta_bias", "h0")}
    ch = torch.arange(dim, device=dev)
    u_full = t["u"].detach().double()[:, ch % u_mod] if u_mod else t["u"].detach().double()
    leaf["u"] = u_full.requires_grad_(True)
    if hw is not None:
        perms = torch.tensor(np.stack([_order(k, *hw) for k in dirs]), device=dev)        # (G, L) natural index per position
    else:
        perms = torch.arange(L, device=dev).expand(G, L)
    pc = perms[ch // dpg]                                                                    # (dim, L)
    gather_c = lambda x: x.gather(2, pc.expand(b, dim, L))
    us, ds = gather_c(leaf["u"]), gather_c(leaf["delta"])
    pg = perms[None, :, None, :].expand(b, G, N, L)
    Bs, Cs = leaf["B"].gather(3, pg)[:, ch // dpg], leaf["C"].gather(3, pg)[:, ch // dpg]   # (b, dim, N, L)
    dt = ds + leaf["delta_bias"][:, None]
    if softplus:
        dt = F.softplus(dt)
    a = torch.exp(dt[:, :, None, :] * leaf["A"][None, :, :, None])
    bu = (dt * us)[:, :, None, :] * Bs
    h, ys = leaf["h0"], []
    for l in range(L):
        h = a[..., l] * h + bu[..., l]
        ys.append((Cs[..., l] * h).sum(-1))
    y = torch.stack(ys, -1) + leaf["D"][:, None] * us
    out = torch.empty_like(y).scatter(2, pc.expand(b, dim, L), y)                            # back to natural order
    dout = t["dout"].double()[:, ch % u_mod] if u_mod else t["dout"].double()
    ((out * dout).sum() + (h * t["dlast"].double()).sum()).backward()
    g = {"du": leaf["u"].grad, "ddelta": leaf["delta"].grad, "dA": leaf["A"].grad, "dB": leaf["B"].grad,
         "dC": leaf["C"].grad, "dD": leaf["D"].grad, "ddelta_bias": leaf["delta_bias"].grad, "dh0": leaf["h0"].grad}
    return {"out": out.detach(), "last": h.detach(), **g}


def _run(t, softplus, hw=None, dirs=None, u_mod=0, use_ckpt=True, out_float=False):
    from ceigm_unet_b200 import ops
    pr = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], softplus, out_float=out_float,
                         hw=hw, dirs=dirs, u_mod=u_mod)
    out, x = pr.forward(want_state=True, h0=t["h0"])
    last = x[:, :, -1, 1::2].clone()
    dout = t["dout"].to(pr.out_dtype)
    grads = pr.backward(dout, x if use_ckpt else None, h0=t["h0"], dlast=t["dlast"], want_dh0=True)
    return {"out": out, "last": last, **dict(zip(NAMES + ["dh0"], grads))}


def _rel(got, ref):
    got, ref = got.double(), ref.double()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def _check(got, ref, tol):
    bad = {k: _rel(got[k], ref[k]) for k in ref if ref[k] is not None and _rel(got[k], ref[k]) > tol}
    assert not bad, bad


# id: (batch, dim, L, N, G, hw, dirs, dtype, softplus, u_mod, forced path policy). The kernel families each case reaches:
CASES = {
    "fwdr32_bwd2_scan": (2, 64, 256, 16, 2, None, None, torch.float32, True, 0, 1),          # scan_fwdr R=1, scan_bwd2
    "fwdr16_bwd2_dirs13": (2, 48, 400, 12, 2, (20, 20), [1, 3], torch.float32, True, 0, 2),  # scan_fwdr R=2, reversed
    "segmented_b1_north_star": (1, 768, 3136, 16, 4, (56, 56), [1, 3, 1, 3], torch.float32, True, 0, 0),
    "segmented_forced": (2, 32, 640, 16, 1, None, None, torch.float32, False, 0, 4),
    "fwd8_N16_dirs1234": (2, 64, 144, 16, 4, (12, 12), [1, 2, 3, 4], torch.float32, True, 0, 3),   # scan_fwd, scan_bwd
    "N1_n1": (2, 64, 784, 1, 4, (28, 28), [1, 3, 1, 3], torch.float32, True, 0, 0),          # scan_n1 fwd + bwd
    "N1_n1_rows_long": (1, 64, 16384, 1, 4, None, None, torch.float32, True, 0, 0),          # gm_s1_b64_512 row geometry
    "N1_n1_L20": (4, 16, 20, 1, 2, None, None, torch.float32, False, 0, 0),                  # L < 32, one-row kernel
    "N1_par_dirs24": (2, 32, 196, 1, 4, (14, 14), [1, 2, 3, 4], torch.float32, True, 0, 0),  # scan_par
    "N1_par_bf16": (2, 32, 196, 1, 4, (14, 14), [1, 3, 1, 3], torch.bfloat16, True, 0, 0),
    "N2_L50": (2, 32, 50, 2, 2, None, None, torch.float32, True, 0, 0),
    "N4_L30": (2, 32, 30, 4, 1, None, None, torch.float32, True, 0, 0),
    "N8_L97": (2, 32, 97, 8, 2, None, None, torch.float32, False, 0, 0),
    "N24": (2, 32, 128, 24, 2, None, None, torch.float32, True, 0, 0),
    "N64_two_passes": (2, 16, 100, 64, 2, None, None, torch.float32, True, 0, 0),
    "N16_u_mod": (2, 64, 196, 16, 2, (14, 14), [1, 3], torch.float32, True, 32, 0),
    "N16_fp16_dirs": (2, 64, 196, 16, 4, (14, 14), [1, 2, 3, 4], torch.float16, True, 0, 0),
    "N16_bf16": (2, 64, 256, 16, 2, None, None, torch.bfloat16, True, 0, 0),
}


_REF_CACHE = {}


@pytest.mark.parametrize("use_ckpt", [True, False], ids=["ckpt", "no_ckpt"])
@pytest.mark.parametrize("case", list(CASES))
def test_parity_with_states(case, use_ckpt):
    from ceigm_unet_b200 import _lib
    b, dim, L, N, G, hw, dirs, dtype, sp, u_mod, policy = CASES[case]
    t = _inputs(b, dim, L, N, G, dtype, seed=7, u_mod=u_mod)
    _lib.test_force_path(policy)
    got = _run(t, sp, hw, dirs, u_mod, use_ckpt=use_ckpt)
    if case not in _REF_CACHE:          # the inputs are seeded: both checkpoint modes compare with one reference
        _REF_CACHE[case] = _reference(t, sp, hw, dirs, u_mod)
    _check(got, _REF_CACHE[case], 1e-3 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("case", ["fwdr32_bwd2_scan", "fwd8_N16_dirs1234", "N1_n1", "N1_n1_rows_long", "N1_par_dirs24",
                                  "N64_two_passes"])
def test_parity_with_states_deterministic(case):
    from ceigm_unet_b200 import _lib
    b, dim, L, N, G, hw, dirs, dtype, sp, u_mod, policy = CASES[case]
    t = _inputs(b, dim, L, N, G, dtype, seed=8, u_mod=u_mod)
    _lib.test_force_path(policy)
    torch.use_deterministic_algorithms(True)
    runs = [_run(t, sp, hw, dirs, u_mod) for _ in range(3)]
    for r in runs[1:]:
        for k in runs[0]:
            assert torch.equal(r[k], runs[0][k]), k
    _check(runs[0], _reference(t, sp, hw, dirs, u_mod), 1e-3)


def _slice(t, a, z):
    s = dict(t)
    for k in ("u", "delta", "dout"):
        s[k] = t[k][..., a:z].contiguous()
    for k in ("B", "C"):
        s[k] = t[k][..., a:z].contiguous()
    return s


@pytest.mark.parametrize("m", [1024, 1000], ids=["m_mult32", "m_not_mult32"])
@pytest.mark.parametrize("shape", [(24, 768, 3136, 16, 4), (24, 64, 3136, 1, 4)], ids=["vm_d192", "gm_s1_g4"])
def test_chaining_equals_one_call(shape, m):
    """Forward of [0, m) hands its last state to [m, L) as h0; backward of [m, L) hands its dh0 to [0, m) as dlast."""
    from ceigm_unet_b200 import ops
    b, dim, L, N, G = shape
    t = _inputs(b, dim, L, N, G, torch.float32, seed=3)
    t["h0"] = torch.zeros_like(t["h0"])
    t["dlast"] = torch.zeros_like(t["dlast"])
    full = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], True)
    out, x = full.forward()
    g_full = full.backward(t["dout"], x)
    last_full = x[:, :, -1, 1::2]

    s0, s1 = _slice(t, 0, m), _slice(t, m, L)
    p0 = ops.ScanProblem(s0["u"], s0["delta"], s0["A"], s0["B"], s0["C"], s0["D"], s0["delta_bias"], True)
    p1 = ops.ScanProblem(s1["u"], s1["delta"], s1["A"], s1["B"], s1["C"], s1["D"], s1["delta_bias"], True)
    o0, x0 = p0.forward()
    mid = x0[:, :, -1, 1::2].contiguous()
    o1, x1 = p1.forward(h0=mid)
    g1 = p1.backward(s1["dout"], x1, h0=mid, want_dh0=True)
    g0 = p0.backward(s0["dout"], x0, dlast=g1[7])

    def close(a, ref, what):
        assert _rel(a, ref) <= 1e-4, (what, _rel(a, ref))
    close(torch.cat([o0, o1], -1), out, "out")
    close(x1[:, :, -1, 1::2], last_full, "last_state")
    for i, name in enumerate(NAMES):
        if name in ("du", "ddelta", "dB", "dC"):
            close(torch.cat([g0[i], g1[i]], -1), g_full[i], name)
        else:
            close(g0[i] + g1[i], g_full[i], name)


@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
@pytest.mark.parametrize("case", ["fwdr32_bwd2_scan", "segmented_forced", "fwd8_N16_dirs1234", "N1_n1", "N1_n1_rows_long",
                                  "N1_par_dirs24", "N64_two_passes", "N16_bf16"])
def test_zero_states_reproduce_the_stateless_call(case, det):
    from ceigm_unet_b200 import _lib, ops
    b, dim, L, N, G, hw, dirs, dtype, sp, u_mod, policy = CASES[case]
    t = _inputs(b, dim, L, N, G, dtype, seed=5, u_mod=u_mod)
    _lib.test_force_path(policy)
    torch.use_deterministic_algorithms(det)
    pr = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], sp, hw=hw, dirs=dirs, u_mod=u_mod)
    dout = t["dout"].to(pr.out_dtype)
    out0, x0 = pr.forward()
    g0 = pr.backward(dout, x0)
    z = torch.zeros_like(t["h0"])
    out1, x1 = pr.forward(h0=z)
    g1 = pr.backward(dout, x1, h0=z, dlast=z, want_dh0=True)
    assert torch.equal(out0, out1)
    assert torch.equal(x0[:, :, -1, 1::2], x1[:, :, -1, 1::2])
    # the default mode sums dB / dC (and, for d_state = 1, dA / dD / d(delta_bias)) with atomics: two calls may differ in the
    # order of those additions whatever the states, so there they are compared to 1e-5; everything else bit for bit
    atomic = set() if det else {"dA", "dB", "dC", "dD", "ddelta_bias"}
    for name, a, c in zip(NAMES, g0, g1[:7]):
        if a is not None:
            assert torch.equal(a, c) if name not in atomic else _rel(c, a) <= 1e-5, name
    assert g1[7] is not None and torch.isfinite(g1[7]).all()


def _autograd_case(dtype, seed=11):
    b, dim, L, N, G = 2, 64, 300, 16, 2
    t = _inputs(b, dim, L, N, G, dtype, seed)
    leaves = {k: t[k].detach().clone().requires_grad_(True)
              for k in ("u", "delta", "A", "B", "C", "D", "delta_bias", "h0")}
    return t, leaves


def _autograd_step(t, leaves):
    import ceigm_unet_b200 as P
    out, last = P.selective_scan(leaves["u"], leaves["delta"], leaves["A"], leaves["B"], leaves["C"], leaves["D"],
                                 leaves["delta_bias"], delta_softplus=True, initial_state=leaves["h0"], return_last_state=True)
    return out, last, torch.autograd.grad((out * t["dout"].to(out.dtype)).sum() + (last * t["dlast"]).sum(), list(leaves.values()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_selective_scan_autograd(dtype):
    t, leaves = _autograd_case(dtype)
    out, last, grads = _autograd_step(t, leaves)
    assert out.dtype == dtype and last.dtype == torch.float32 and tuple(last.shape) == tuple(t["h0"].shape)
    ref = _reference(t, True)
    got = {"out": out, "last": last, **dict(zip(["du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dh0"], grads))}
    _check(got, ref, 1e-3 if dtype == torch.float32 else 2e-2)


def test_selective_scan_plain_call_and_no_initial_state():
    import ceigm_unet_b200 as P
    t, _ = _autograd_case(torch.float32)
    out = P.selective_scan(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], delta_softplus=True)
    t0 = dict(t, h0=torch.zeros_like(t["h0"]))
    assert _rel(out, _reference(t0, True)["out"]) <= 1e-3


def test_selective_scan_deterministic_calls_and_graph_replays():
    torch.use_deterministic_algorithms(True)
    t, leaves = _autograd_case(torch.float32)
    first = _autograd_step(t, leaves)[2]
    for _ in range(2):
        again = _autograd_step(t, leaves)[2]
        assert all(torch.equal(a, b) for a, b in zip(first, again))
    # the same step captured into a CUDA graph and replayed
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        _autograd_step(t, leaves)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        captured = _autograd_step(t, leaves)[2]
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(first, captured))
