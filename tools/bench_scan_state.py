"""Cost of state passing in the selective scan: the call with an initial state h0 (forward) or with h0, the final-state
gradient dlast and the h0 gradient dh0 (backward) against the stateless call, on bench.py's workloads and input recipe.

Each call of one step is captured into a CUDA graph per variant (stateless / state), forward and backward separately; the
graphs are replayed alternately in one process, L2 overwritten (256 MB) before every timed replay. Reports the median and the
spread (min ... max) over the repeats, the ratio of the medians, and the GPU name and power limit read in the same run.

usage: python tools/bench_scan_state.py [--repeats 15] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import WORKLOADS, build_inputs  # noqa: E402

SCAN_WORKLOADS = ["vm_d192", "vm_d192_b1", "gm_live_g4", "gm_s1_b64_512"]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def capture(fn):
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        fn()
    torch.cuda.synchronize()
    return g


def alternate(runs, repeats, flush):
    """runs: {variant: callable}. Times each callable `repeats` times, variants interleaved, L2 overwritten before each."""
    times = {m: [] for m in runs}
    for _ in range(3):
        for fn in runs.values():
            fn()
    torch.cuda.synchronize()
    for _ in range(repeats):
        for m, fn in runs.items():
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[m].append(e0.elapsed_time(e1))
    return times


def summary(name, times):
    med = {m: statistics.median(t) for m, t in times.items()}
    return {"workload": name,
            **{f"{m}_ms": round(med[m], 4) for m in times},
            **{f"{m}_spread_ms": [round(min(t), 4), round(max(t), 4)] for m, t in times.items()},
            "ratio": round(med["state"] / med["stateless"], 3)}


def scan_workload(name, repeats, flush):
    from ceigm_unet_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(1)
    sets = []
    for count, inp in build_inputs(WORKLOADS[name], "cuda", on_device=True):
        t = {k: v.cuda() for k, v in inp.items()}
        pr = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], True)
        shape = (pr.batch, pr.dim, pr.N)
        h0 = torch.randn(shape, device="cuda", generator=gen)
        dlast = torch.randn(shape, device="cuda", generator=gen)
        x0, x1 = pr.forward()[1], pr.forward(h0=h0)[1]
        sets.append((count, pr, t["dout"], h0, dlast, x0, x1))

    def fwd(state):
        def step():
            for count, pr, _, h0, _, _, _ in sets:
                for _ in range(count):
                    pr.forward(h0=h0 if state else None)
        return step

    def bwd(state):
        def step():
            for count, pr, dout, h0, dlast, x0, x1 in sets:
                for _ in range(count):
                    if state:
                        pr.backward(dout, x1, h0=h0, dlast=dlast, want_dh0=True)
                    else:
                        pr.backward(dout, x0)
        return step

    res = []
    for leg, make in (("forward", fwd), ("backward", bwd)):
        graphs = {"stateless": capture(make(False)), "state": capture(make(True))}
        res.append(summary(f"{name} ({leg})", alternate({m: g.replay for m, g in graphs.items()}, repeats, flush)))
        del graphs
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_scan_state.py needs a CUDA device")
    import ceigm_unet_b200 as P
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > 126 MB of L2
    lines = [{"gpu": gpu_info(), "library": P.version(), "repeats": args.repeats}]
    print(json.dumps(lines[0]), flush=True)
    for name in SCAN_WORKLOADS:
        for rec in scan_workload(name, args.repeats, flush):
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
