"""b4 (SURVEY.md §8b): the UNMODIFIED reference modules and model run on the B200 through this repo's drop-in, and are
checked against the CPU oracle at the LIVE shapes of GM-UNet (stage widths 64 / 128 / 348 / 448 on 56^2 ... 7^2 maps) and of
the north-star regime (VMamba SS2D, K = 4, d_state = 16, d_model = 96 on 56^2).

  level 1: reference `model.gm.groupmamba.GroupMambaLayer` / `model.gm.ss2d.SS2D` / `model.vmamba.vmamba.SS2D` /
           `model.build_model` with `install_dropin()` — every selective scan goes through libss2d_b200.so;
  level 2: `ceigm_unet_b200.GroupMambaLayer` / `SS2D` (fused kernels: wgrad_ts, dwconv3_wgrad, layernorm, out_gate) with the
           reference's weights loaded through `state_dict`, at the shapes that select those kernels.
The checker is oracle/ss2d_ref.py with the C-backed scan (oracle/fast_scan.py) on the host; the reference tree comes from the
git-ignored baseline/_ref/ (harness/install_ref.py). Without it only the level-2 layer and SS2D cases run: this repo's
constructors draw the reference's parameters under the same seed, so they need no reference code.
Tolerances (BASELINE.json north_star): rel <= 1e-3 fp32 (max |diff| / max |ref| per tensor; 2e-3 for parameter gradients, which
sum 6 272 ... 98 rows in fp32 on both sides), <= 2e-2 under bf16 autocast; argmax label maps are compared pixel by pixel.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STAGES = [(64, 56), (128, 28), (348, 14), (448, 7)]          # (C, H = W) of the four GM-UNet stages at 224^2


@pytest.fixture(autouse=True)
def _fp32_math():
    """fp32 parity means fp32 arithmetic in the library convolutions / GEMMs around the path too: cuDNN convolutions
    default to TF32 in PyTorch (10-bit mantissa, ~1e-3 per layer), which would mask or fake errors of the operators under test."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _ref():
    from harness import refmodel
    if not refmodel.available():
        pytest.skip("reference tree not installed: run harness/install_ref.py (populates baseline/_ref/)")
    return refmodel


def rel_err(got, ref):
    got = got.detach().double().cpu().numpy()
    ref = ref.detach().double().cpu().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))


def allclose_table(got, ref, rtol=6e-4, atol=2e-3):
    """The reference test's own per-element criterion (test_selective_scan.py:398-401, fp32 row) as a second check."""
    return torch.allclose(got.detach().float().cpu(), ref.detach().float().cpu(), rtol=rtol, atol=atol)


def _oracle_layer(sd, x, dy, H, W):
    from oracle import ss2d_ref
    ss2d_ref.use_fast_scan(True)
    try:
        p = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in sd.items()}
        xr = x.detach().cpu().clone().requires_grad_(True)
        y = ss2d_ref.group_layer(xr, p, H, W)
        y.backward(dy.cpu())
    finally:
        ss2d_ref.use_fast_scan(False)
    return y.detach(), xr.grad, {k: v.grad for k, v in p.items()}


def _randomise(layer, seed):
    """Block_mamba re-initialises Linear/LayerNorm/Conv2d weights (groupmamba.py:206-221); a bare GroupMambaLayer keeps
    nn defaults. Perturb the parameters whose defaults would hide errors (LayerNorm = identity, skip_scale = 1, biases 0)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in layer.named_parameters():
            if n.endswith("norm.weight") or n.endswith("out_norm.weight") or n == "skip_scale":
                p.add_(0.2 * torch.randn(p.shape, generator=g))
            elif n.endswith("norm.bias") or n.endswith("out_norm.bias"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))


def _run_layer(layer, x, dy, H, W):
    layer = layer.cuda()
    xg = x.cuda().requires_grad_(True)
    y = layer(xg, H, W)
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    return y.detach(), xg.grad, {n: p.grad for n, p in layer.named_parameters()}


def _compare(got, ref, tol=1e-3):
    y, dx, grads = got
    yr, dxr, gr = ref
    errs = {"y": rel_err(y, yr), "dx": rel_err(dx, dxr)}
    for n, gval in grads.items():
        errs["grad." + n] = rel_err(gval, gr[n])
    bad = {k: v for k, v in errs.items() if v > (tol if k in ("y", "dx") else 2 * tol)}
    assert not bad, bad
    assert allclose_table(y, yr) and allclose_table(dx, dxr, rtol=1.2e-3, atol=4e-3)
    return errs


@pytest.mark.parametrize("C,H", STAGES, ids=[f"C{c}_{h}x{h}" for c, h in STAGES])
@pytest.mark.parametrize("level", ["ref_dropin", "fused"])
def test_group_mamba_layer_live_shapes(C, H, level):
    import ceigm_unet_b200 as P
    torch.manual_seed(100 + C)
    if level == "ref_dropin":
        R = _ref()
        R.load_reference(scan="dropin")
        _, _, gmb = R.reference_modules()
        layer = gmb.GroupMambaLayer(C, C)                      # the reference's own module (CPU construction)
    else:
        layer = P.GroupMambaLayer(C, C)                        # the reference's parameters (test_abi.py pins the init)
    _randomise(layer, C)
    sd = {k: v.clone() for k, v in layer.state_dict().items()}
    x = torch.randn(2, H * H, C)
    dy = torch.randn(2, H * H, C)
    P.launch_count(reset=True)
    got = _run_layer(layer, x, dy, H, H)
    assert P.launch_count() >= 8                               # 4 scans fwd + 4 bwd at the very least went through the C ABI
    _compare(got, _oracle_layer(sd, x, dy, H, H))


@pytest.mark.parametrize("level", ["ref_dropin", "fused"])
def test_vmamba_ss2d_k4_n16_live_shape(level):
    """North-star regime at its real size: VMamba SS2D(d_model=96, d_state=16, ssm_ratio=2) -> K=4, D=192, L=56^2."""
    import ceigm_unet_b200 as P
    from oracle import ss2d_ref
    torch.manual_seed(7)
    if level == "ref_dropin":
        R = _ref()
        R.load_reference(scan="dropin")
        import importlib
        vm = importlib.import_module("model.vmamba.vmamba")
        mod = vm.SS2D(d_model=96, d_state=16, ssm_ratio=2.0, forward_type="v2")
    else:
        mod = P.SS2D(d_model=96, d_state=16, ssm_ratio=2.0, k_group=4)      # the reference's parameters (test_abi.py)
    _randomise(mod, 3)
    sd = {k: v.clone() for k, v in mod.state_dict().items()}
    x = torch.randn(2, 56, 56, 96)
    dy = torch.randn(2, 56, 56, 96)
    mod = mod.cuda()
    xg = x.cuda().requires_grad_(True)
    y = mod(xg)
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    ss2d_ref.use_fast_scan(True)
    try:
        p = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
        xr = x.clone().requires_grad_(True)
        yr = ss2d_ref.ss2d_forward(xr, p, (1, 2, 3, 4))
        yr.backward(dy)
    finally:
        ss2d_ref.use_fast_scan(False)
    _compare((y.detach(), xg.grad, {n: q.grad for n, q in mod.named_parameters()}),
             (yr.detach(), xr.grad, {k: v.grad for k, v in p.items()}))


def _dice_per_class(pred, label, num_classes):
    """eval.py:9-45 / utils.py:30-55 (SegMeter + calc_dice_gpu) on label maps."""
    out = []
    for c in range(1, num_classes):
        a, b = pred == c, label == c
        sa, sb = int(a.sum()), int(b.sum())
        out.append(2.0 * int((a & b).sum()) / (sa + sb) if sa > 0 and sb > 0 else (1.0 if sa > 0 and sb == 0 else 0.0))
    return out


@pytest.mark.parametrize("level", ["ref_dropin", "fused"])
def test_build_model_224_forward_backward(level):
    """BASELINE config 1 on the GPU: `model.build_model(in_channels=3, num_classes=9)` at 1 x 3 x 224 x 224 against the same
    model on the host with the oracle scan — logits, DiceCE loss (train_synapse.py:90-93), gradients of the first and last
    parameters, argmax label map (mismatching pixels) and per-class Dice (eval.py)."""
    R = _ref()
    m_cpu = R.load_reference(scan="cpu_fast")
    torch.manual_seed(42)
    net_cpu = m_cpu.build_model(in_channels=3, num_classes=9)
    sd = {k: v.clone() for k, v in net_cpu.state_dict().items()}
    loss_mod = R.load_losses()
    crit = loss_mod.DiceCELoss(ce_weight=0.4, dc_weight=0.6)
    g = torch.Generator().manual_seed(42)
    x = torch.randn(1, 3, 224, 224, generator=g)
    label = torch.randint(0, 9, (1, 1, 224, 224), generator=g).float()
    # eval(): stochastic depth (DropPath, groupmamba.py:327) draws from the device's own RNG stream, so train() mode is not
    # comparable across devices sample by sample; BatchNorm then uses its running statistics on both sides. Gradients still flow.
    net_cpu.eval()
    out_cpu = net_cpu(x)
    loss_cpu = crit(out_cpu, label)
    loss_cpu.backward()
    names = [n for n, _ in net_cpu.named_parameters()]
    probe = [names[0], names[len(names) // 2], names[-2]]
    g_cpu = {n: p.grad.clone() for n, p in net_cpu.named_parameters() if n in probe}

    m_gpu = R.load_reference(scan="dropin", fused=(level == "fused"))
    torch.manual_seed(42)
    net = m_gpu.build_model(in_channels=3, num_classes=9)
    if level == "fused":
        assert R.reclass_layernorms(net) > 0              # the encoder's LayerNorms on this repo's row kernel (level 2)
    missing, unexpected = net.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    net = net.cuda().eval()
    import ceigm_unet_b200 as P
    P.launch_count(reset=True)
    out = net(x.cuda())
    loss = crit(out, label.cuda())
    loss.backward()
    torch.cuda.synchronize()
    assert P.launch_count() >= 104                             # 104 scan calls per forward (SURVEY.md §3.1)
    e_logits = rel_err(out, out_cpu)
    assert e_logits < 1e-3, e_logits
    assert abs(loss.item() - loss_cpu.item()) <= 1e-3 * abs(loss_cpu.item())
    for n, p in net.named_parameters():
        if n in probe:
            assert rel_err(p.grad, g_cpu[n]) < 2e-3, n
    pred, pred_cpu = out.argmax(1).cpu(), out_cpu.argmax(1)
    mism = int((pred != pred_cpu).sum())
    d_gpu, d_cpu = _dice_per_class(pred, label[:, 0].long(), 9), _dice_per_class(pred_cpu, label[:, 0].long(), 9)
    ddice = max(abs(a - b) for a, b in zip(d_gpu, d_cpu))
    print(f"[{level}] logits rel {e_logits:.2e}, argmax mismatching pixels {mism} / {pred.numel()}, max |dDice| {ddice:.2e}")
    assert mism <= 0.001 * pred.numel() and ddice < 1e-3


def test_reference_autograd_functions_bound_to_dropin():
    """The reference's csms6s.py must have picked up THIS repo's extension modules (not a stub, not mamba_ssm)."""
    R = _ref()
    R.load_reference(scan="dropin")
    import sys
    core = sys.modules["selective_scan_cuda_core"]
    assert "ceigm" in (core.__file__ or "") and hasattr(core, "fwd") and hasattr(core, "bwd")
    cs, ss, _ = R.reference_modules()
    assert ss.SelectiveScanCore is cs.SelectiveScanCore       # the reference's own autograd.Function, unmodified


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_harness_min_pool_rebinding_is_bit_identical(dtype):
    """harness.graph_step.make_capturable() replaces AdaptiveMinPool2d.forward (F.unfold of the whole map + min) by the same
    min on the flattened view: identical values and identical gradient routing — including ties (post-ReLU zeros)."""
    import importlib
    R = _ref()
    R.load_reference(scan="dropin")
    from harness import graph_step
    bd = importlib.import_module("model.best_decoder")
    pool = bd.AdaptiveMinPool2d()
    orig = getattr(bd.AdaptiveMinPool2d, "_ss2d_harness_orig_forward", bd.AdaptiveMinPool2d.forward)
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.relu(torch.randn(3, 40, 28, 28, device="cuda", generator=gen)).to(dtype)      # many exact ties at 0
    x[:, ::2] -= 1.0                                                                          # and channels with a unique minimum
    g = torch.randn(3, 40, 1, 1, device="cuda", generator=gen).to(dtype)
    xa = x.clone().requires_grad_(True)
    ya = orig(pool, xa)
    ya.backward(g)
    graph_step.make_capturable()
    assert bd.AdaptiveMinPool2d.forward is graph_step._min_pool_direct
    xb = x.clone().requires_grad_(True)
    yb = pool(xb)
    yb.backward(g)
    assert torch.equal(ya, yb) and torch.equal(xa.grad, xb.grad)
    # non-square maps keep the reference code path
    xr = torch.randn(1, 4, 6, 6, device="cuda")
    assert torch.equal(pool(xr), orig(pool, xr))
