"""Cost of the causal depthwise conv1d (`causal_conv1d_fn`, `causal_conv1d_update`) against what a Mamba user runs without
causal-conv1d, mamba_simple's fallbacks:
  - forward: act(nn.Conv1d(dim, dim, width, groups=dim, padding=width - 1)(x)[..., :L]) with SiLU, and its autograd backward;
  - update: the `step` fallback, conv_state.copy_(roll(conv_state, -1)), conv_state[..., -1] = x, sum(conv_state * w, -1) + bias,
    SiLU.

Each route is captured into a CUDA graph and the graphs of one workload are replayed alternately in one process, L2 overwritten
(256 MB) before every timed replay; each number is the median (and min ... max) of the repeats. Forward / backward workloads
time three graphs per route: the forward, the forward + backward (autograd.grad of x, weight and bias), and for the library its
backward call alone. Algorithmic bytes per element of x: forward 2 s (x read, out written), backward 3 s (x and dout read, dx
written), s = element size; GB/s and the share of 7.7 TB/s (one B200's HBM3e bandwidth on the data sheet) are computed from them.
The update workloads time a 64-step decode loop (each step with its own x) and report the time per step. Before timing, the
routes' outputs are compared (max error over max |value|). The GPU name and power limit are read in the same run.

usage: python tools/bench_causal_conv1d.py [--repeats 15] [--out profiles/r6_bench_causal_conv1d.jsonl]"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from bench_scan_state import alternate, capture, gpu_info  # noqa: E402

HBM = 7.7e12
W = 4
STEPS = 64
CONV_SHAPES = [(1536, 16, 2048, "fp32"), (1536, 16, 2048, "bf16"), (5120, 8, 2048, "bf16")]   # (d_inner, batch, L, dtype)
UPDATE_DIMS, UPDATE_BATCHES = [1536, 5120], [1, 16, 256]
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def torch_fwd(x, w, b):
    return F.silu(F.conv1d(x, w.unsqueeze(1).to(x.dtype), b.to(x.dtype), padding=w.shape[1] - 1, groups=w.shape[0])[..., :x.shape[-1]])


def lib_fwd(x, w, b):
    import ceigm_unet_b200 as P
    return P.causal_conv1d_fn(x, w, b, activation="silu")


def stats(ts, scale=1.0):
    per = [scale * t for t in ts]
    return statistics.median(per), [round(min(per), 4), round(max(per), 4)]


def conv_workload(dim, batch, L, dtype_name, repeats, flush):
    from ceigm_unet_b200 import ops
    dtype = DTYPES[dtype_name]
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(batch, dim, L, device="cuda", generator=gen).to(dtype).requires_grad_(True)
    dout = torch.randn(batch, dim, L, device="cuda", generator=gen).to(dtype)
    w = (0.5 * torch.randn(dim, W, device="cuda", generator=gen)).requires_grad_(True)
    b = (0.1 * torch.randn(dim, device="cuda", generator=gen)).requires_grad_(True)
    agree = {"out_rel": rel(lib_fwd(x, w, b), torch_fwd(x, w, b))}
    g_lib = torch.autograd.grad(lib_fwd(x, w, b), (x, w, b), dout)
    g_ref = torch.autograd.grad(torch_fwd(x, w, b), (x, w, b), dout)
    agree.update({k: rel(a, r) for k, a, r in zip(("dx_rel", "dweight_rel", "dbias_rel"), g_lib, g_ref)})

    def fwd(route):
        def run():
            with torch.no_grad():
                route(x, w, b)
        return run

    def fwd_bwd(route):
        return lambda: torch.autograd.grad(route(x, w, b), (x, w, b), dout)

    graphs = {"lib_fwd": capture(fwd(lib_fwd)), "torch_fwd": capture(fwd(torch_fwd)),
              "lib_fwd_bwd": capture(fwd_bwd(lib_fwd)), "torch_fwd_bwd": capture(fwd_bwd(torch_fwd)),
              "lib_bwd": capture(lambda: ops.conv1d_bwd(x.detach(), w.detach(), b.detach(), dout, True))}
    times = alternate({m: g.replay for m, g in graphs.items()}, repeats, flush)
    del graphs
    torch.cuda.empty_cache()
    n, s = batch * dim * L, torch.finfo(dtype).bits // 8
    nbytes = {"fwd": 2 * s * n, "bwd": 3 * s * n, "fwd_bwd": 5 * s * n}
    rec = {"workload": f"d_inner {dim}, batch {batch}, L {L}, width {W}, SiLU, bias", "io": dtype_name, "weights": "fp32"}
    for m, ts in times.items():
        med, spread = stats(ts)
        kind = m.split("_", 1)[1]
        rec[f"{m}_ms"] = round(med, 4)
        rec[f"{m}_spread_ms"] = spread
        rec[f"{m}_GBps"] = round(nbytes[kind] / (med * 1e-3) / 1e9, 1)
        rec[f"{m}_hbm_share"] = round(nbytes[kind] / (med * 1e-3) / HBM, 3)
    rec["speedup_fwd"] = round(rec["torch_fwd_ms"] / rec["lib_fwd_ms"], 2)
    rec["speedup_fwd_bwd"] = round(rec["torch_fwd_bwd_ms"] / rec["lib_fwd_bwd_ms"], 2)
    rec["bytes"] = nbytes
    rec["agreement"] = {k: float("%.2e" % v) for k, v in agree.items()}
    return rec


def torch_step(state, x, w, b):
    state.copy_(torch.roll(state, shifts=-1, dims=-1))
    state[:, :, -1] = x
    return F.silu(torch.sum(state * w, dim=-1) + b).to(x.dtype)


def lib_step(state, x, w, b):
    import ceigm_unet_b200 as P
    return P.causal_conv1d_update(x, state, w, b, "silu")


def update_workload(dim, batch, dtype_name, repeats, flush):
    dtype = DTYPES[dtype_name]
    gen = torch.Generator(device="cuda").manual_seed(1)
    xs = torch.randn(STEPS, batch, dim, device="cuda", generator=gen).to(dtype)
    s0 = torch.randn(batch, dim, W, device="cuda", generator=gen).to(dtype)
    w, b = 0.5 * torch.randn(dim, W, device="cuda", generator=gen), 0.1 * torch.randn(dim, device="cuda", generator=gen)
    sa, sb = s0.clone(), s0.clone()
    agree = {"out_rel": rel(lib_step(sa, xs[0], w, b), torch_step(sb, xs[0], w, b)), "state_equal": bool(torch.equal(sa, sb))}
    states = {"lib": s0.clone(), "torch": s0.clone()}

    def loop(route, state):
        def run():
            for i in range(STEPS):
                route(state, xs[i], w, b)
        return run

    graphs = {"lib": capture(loop(lib_step, states["lib"])), "torch": capture(loop(torch_step, states["torch"]))}
    times = alternate({m: g.replay for m, g in graphs.items()}, repeats, flush)
    del graphs
    rec = {"workload": f"update d_inner {dim}, width {W}, SiLU, bias", "batch": batch, "io": dtype_name, "weights": "fp32"}
    for m, ts in times.items():
        med, spread = stats(ts, 1e3 / STEPS)                  # ms per replay -> us per step
        rec[f"{m}_us_per_step"] = round(med, 3)
        rec[f"{m}_spread_us"] = [round(v, 3) for v in spread]
    rec["speedup"] = round(rec["torch_us_per_step"] / rec["lib_us_per_step"], 2)
    rec["first_step_agreement"] = agree
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_causal_conv1d.py needs a CUDA device")
    import ceigm_unet_b200 as P
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > 126 MB of L2
    lines = [{"gpu": gpu_info(), "library": P.version(), "repeats": args.repeats, "update_steps_per_replay": STEPS}]
    print(json.dumps(lines[0]), flush=True)
    for dim, batch, L, dtype_name in CONV_SHAPES:
        lines.append(conv_workload(dim, batch, L, dtype_name, args.repeats, flush))
        print(json.dumps(lines[-1]), flush=True)
    with torch.no_grad():
        for dtype_name in DTYPES:
            for dim in UPDATE_DIMS:
                for batch in UPDATE_BATCHES:
                    lines.append(update_workload(dim, batch, dtype_name, args.repeats, flush))
                    print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
