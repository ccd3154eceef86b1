"""Cost of one recurrent step of the selective scan: `selective_state_update` (ss2d_state_update: one kernel, the state updated in
place) against what a caller had before it, `selective_scan` over L = 1 from `initial_state` with `return_last_state=True`, followed
by the copy of the returned state back into the state buffer.

Both routes run a decode loop of 64 steps with D, dt_bias, softplus and a z gate (the Mamba block's configuration), each step with
its own x, dt, z, B and C. Each loop is captured into a CUDA graph; the two graphs are replayed alternately in one process, L2
overwritten (256 MB) before every timed replay (inside a loop the state stays in L2 after the first step, as it does for one layer
of a decoding model whose states fit there). Reports the time per step (replay time / 64) as the median and spread (min ... max)
of the repeats, and the algorithmic GB/s of a step: the state read and written (8 B dim N bytes), x, dt, z and out (4 B dim
elements of the io dtype) and B and C (2 B G N elements); A, D and dt_bias are not counted. Before timing, one step of each route
from the same state is compared (max error over max |value| of out and of the new state). The GPU name and power limit are read in
the same run.

Shapes (dim, dstate, G): (1536, 16, 1), a Mamba-130M layer; (768, 16, 4), vm_d192's channels; (448, 1, 4), GM-UNet's stage 4
(d_state = 1). Batch 1, 16 and 256; fp32 and bf16 io.

usage: python tools/bench_state_update.py [--repeats 15] [--out profiles/r5_bench_state_update.jsonl]"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from bench_scan_state import alternate, capture, gpu_info  # noqa: E402

STEPS = 64
SHAPES = [("mamba130m", 1536, 16, 1), ("vm_d192", 768, 16, 4), ("gm_stage4", 448, 1, 4)]
BATCHES = [1, 16, 256]
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def make_inputs(batch, dim, N, G, dtype, seed=0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    return dict(x=r(STEPS, batch, dim).to(dtype), dt=(0.5 * torch.rand(STEPS, batch, dim, device="cuda", generator=gen) - 2.0).to(dtype),
                z=r(STEPS, batch, dim).to(dtype), B=r(STEPS, batch, G, N).to(dtype), C=r(STEPS, batch, G, N).to(dtype),
                A=-torch.arange(1, N + 1, device="cuda", dtype=torch.float32).repeat(dim, 1), D=torch.ones(dim, device="cuda"),
                dt_bias=0.1 * r(dim), h0=r(batch, dim, N))


def step_route(t, state, l):
    import ceigm_unet_b200 as P
    return P.selective_state_update(state, t["x"][l], t["dt"][l], t["A"], t["B"][l], t["C"][l], t["D"], t["z"][l], t["dt_bias"], True)


def scan_route(t, state, l):
    import ceigm_unet_b200 as P
    out, last = P.selective_scan(t["x"][l].unsqueeze(-1), t["dt"][l].unsqueeze(-1), t["A"], t["B"][l].unsqueeze(-1),
                                 t["C"][l].unsqueeze(-1), t["D"], t["dt_bias"], True, initial_state=state, return_last_state=True,
                                 z=t["z"][l].unsqueeze(-1))
    state.copy_(last)
    return out[..., 0]


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def workload(name, dim, N, G, batch, dtype_name, repeats, flush):
    dtype = DTYPES[dtype_name]
    t = make_inputs(batch, dim, N, G, dtype)
    s_step, s_scan = t["h0"].clone(), t["h0"].clone()
    agree = {"out_rel": rel(step_route(t, s_step, 0), scan_route(t, s_scan, 0)), "state_rel": rel(s_step, s_scan)}
    states = {"step": t["h0"].clone(), "scan": t["h0"].clone()}

    def loop(route, state):
        def run():
            for l in range(STEPS):
                route(t, state, l)
        return run

    graphs = {"step": capture(loop(step_route, states["step"])), "scan": capture(loop(scan_route, states["scan"]))}
    times = alternate({m: g.replay for m, g in graphs.items()}, repeats, flush)
    del graphs
    torch.cuda.empty_cache()
    es = torch.finfo(dtype).bits // 8
    nbytes = 8 * batch * dim * N + 4 * batch * dim * es + 2 * batch * G * N * es
    rec = {"workload": f"{name} (dim {dim}, dstate {N}, G {G})", "batch": batch, "io": dtype_name}
    for m, ts in times.items():
        per = [1e3 * x / STEPS for x in ts]                    # ms per replay -> us per step
        med = statistics.median(per)
        rec[f"{m}_us_per_step"] = round(med, 3)
        rec[f"{m}_spread_us"] = [round(min(per), 3), round(max(per), 3)]
        rec[f"{m}_GBps"] = round(nbytes / (med * 1e-6) / 1e9, 1)
    rec["speedup"] = round(rec["scan_us_per_step"] / rec["step_us_per_step"], 2)
    rec["bytes_per_step"] = nbytes
    rec["first_step_agreement"] = {k: float("%.2e" % v) for k, v in agree.items()}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_state_update.py needs a CUDA device")
    import ceigm_unet_b200 as P
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > 126 MB of L2
    lines = [{"gpu": gpu_info(), "library": P.version(), "repeats": args.repeats, "steps_per_replay": STEPS}]
    print(json.dumps(lines[0]), flush=True)
    with torch.no_grad():
        for name, dim, N, G in SHAPES:
            for dtype_name in DTYPES:
                for batch in BATCHES:
                    rec = workload(name, dim, N, G, batch, dtype_name, args.repeats, flush)
                    lines.append(rec)
                    print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
