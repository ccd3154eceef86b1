"""Cost of the deterministic scan backward (torch.use_deterministic_algorithms(True)) against the default one.

Scan workloads (bench.py's WORKLOADS and input recipe): the backward calls of one step captured into a CUDA graph per mode
(the switch is read at capture), replayed alternately in the same process, L2 overwritten (256 MB) before every timed
replay. Module workloads: forward + backward of a graphed stage-1 GroupMambaLayer (batch 24, 56^2, 64 channels) and of a
K = 4 SS2D(d_model=96, d_state=16) (batch 24, 56^2), one graphed copy per mode. Reports the median and the spread
(min ... max) over the repeats, the ratio of the medians, and the GPU name and power limit read in the same run.

usage: python tools/bench_deterministic.py [--repeats 15] [--out FILE]"""
import argparse
import copy
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


def capture(fn, det):
    """CUDA graph of fn() captured with the deterministic switch at `det`."""
    torch.use_deterministic_algorithms(det)
    try:
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
    finally:
        torch.use_deterministic_algorithms(False)


def alternate(runs, repeats, flush):
    """runs: {mode: callable}. Times each callable `repeats` times, modes interleaved, L2 overwritten before each."""
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
            "ratio": round(med["deterministic"] / med["default"], 3)}


def scan_workload(name, repeats, flush):
    from ceigm_unet_b200.dropin import selective_scan_cuda_core as core
    sets = [(c, {k: v.cuda() for k, v in inp.items()}) for c, inp in build_inputs(WORKLOADS[name], "cuda", on_device=True)]
    xs = []
    for _, t in sets:
        xs.append(core.fwd(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], True, 1)[1])

    def bwd_step():
        for (count, t), x in zip(sets, xs):
            for _ in range(count):
                core.bwd(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], t["dout"], x, True, 1)

    graphs = {"default": capture(bwd_step, False), "deterministic": capture(bwd_step, True)}
    res = summary(name + " (backward)", alternate({m: g.replay for m, g in graphs.items()}, repeats, flush))
    del graphs
    torch.cuda.empty_cache()
    return res


def module_workload(name, make, shape, hw, repeats, flush):
    import ceigm_unet_b200 as P

    class Wrap(torch.nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m = m

        def forward(self, x):
            return self.m(x, *hw) if hw else self.m(x)

    torch.manual_seed(0)
    base = Wrap(make()).cuda()
    x = torch.randn(*shape, device="cuda", requires_grad=True)
    gy = torch.randn(*shape, device="cuda")
    runs = {}
    for mode, det in (("default", False), ("deterministic", True)):
        mod = copy.deepcopy(base)
        torch.use_deterministic_algorithms(det)
        g = P.graphed(mod, (x.detach().clone().requires_grad_(True),))
        torch.use_deterministic_algorithms(False)

        def step(g=g):
            g(x).backward(gy)
        runs[mode] = step
    return summary(name + " (fwd+bwd, graphed)", alternate(runs, repeats, flush))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_deterministic.py needs a CUDA device")
    import ceigm_unet_b200 as P
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > 126 MB of L2
    lines = [{"gpu": gpu_info(), "library": P.version(), "repeats": args.repeats}]
    print(json.dumps(lines[0]), flush=True)
    for name in SCAN_WORKLOADS:
        lines.append(scan_workload(name, args.repeats, flush))
        print(json.dumps(lines[-1]), flush=True)
    mods = [("GroupMambaLayer stage 1 (b24, 56^2, C64)", lambda: P.GroupMambaLayer(64, 64), (24, 3136, 64), (56, 56)),
            ("SS2D K4 N16 (b24, 56^2, d_model 96)", lambda: P.SS2D(d_model=96, d_state=16, ssm_ratio=2.0, k_group=4),
             (24, 56, 56, 96), None)]
    for name, make, shape, hw in mods:
        lines.append(module_workload(name, make, shape, hw, args.repeats, flush))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
