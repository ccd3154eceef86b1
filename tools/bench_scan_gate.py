"""Cost of the selective scan's output gate out_z = y * silu(z): the ungated scan followed by torch's gate, the gated call with the
gate in its own pass (scan_gate_fwd_kernel / scan_gate_bwd_kernel), and the gated call with the gate inside scan_fwdr.

Shapes: mamba_d1536 (B = 8, Dt = 1536, L = 2048, N = 16, G = 1, fp32, softplus: one Mamba-130m layer) and bench.py's vm_d192 with
a z. At mamba_d1536 the automatic forward is scan_fwd (too few 16-row warps to fill the machine, sequence too short to split), so
the fused gate cannot apply; a second record forces scan_fwdr with 16-row warps (test hook policy 2) to compare the two gate
placements there too.

Each variant is captured into a CUDA graph, forward and backward separately; the graphs are replayed alternately in one process,
L2 overwritten (256 MB) before every timed replay. Reports the median and the spread (min ... max) over the repeats, and the GPU
name and power limit read in the same run.
Rows: forward  torch_gate = scan + out * F.silu(z); standalone = gated call, gate pass after the scan (policy + 8);
                fused = gated call as dispatched (the gate inside scan_fwdr where it applies);
      backward torch_gate = the three elementwise kernels autograd runs for out * F.silu(z) + the scan backward;
                gated = ss2d_scan_bwd_gated (gate prologue + the scan backward).

usage: python tools/bench_scan_gate.py [--repeats 15] [--out profiles/r4_bench_scan_gate.jsonl]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from bench import WORKLOADS, build_inputs  # noqa: E402
from bench_scan_state import alternate, capture, gpu_info  # noqa: E402


def summary(name, times, base):
    import statistics
    med = {m: statistics.median(t) for m, t in times.items()}
    return {"workload": name,
            **{f"{m}_ms": round(med[m], 4) for m in times},
            **{f"{m}_spread_ms": [round(min(t), 4), round(max(t), 4)] for m, t in times.items()},
            **{f"{m}_vs_{base}": round(med[m] / med[base], 3) for m in times if m != base}}


def mamba_inputs():
    gen = torch.Generator(device="cuda").manual_seed(0)
    b, dim, L, N = 8, 1536, 2048, 16
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    t = dict(u=r(b, dim, L), delta=0.5 * torch.rand(b, dim, L, device="cuda", generator=gen) - 2.0,
             A=-torch.arange(1, N + 1, device="cuda", dtype=torch.float32).repeat(dim, 1), B=r(b, 1, N, L), C=r(b, 1, N, L),
             D=torch.ones(dim, device="cuda"), delta_bias=0.1 * r(dim), dout=r(b, dim, L))
    return [(1, t)]


def gate_workload(name, sets_in, policy, repeats, flush):
    from ceigm_unet_b200 import _lib, ops
    gen = torch.Generator(device="cuda").manual_seed(1)
    _lib.test_force_path(policy)
    sets = []
    for count, t in sets_in:
        pr = ops.ScanProblem(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], True)
        z = torch.randn(pr.batch, pr.dim, pr.L, device="cuda", generator=gen)
        out, x, out_z = pr.forward(z=z)
        _lib.launch_count(reset=True)
        pr.forward(z=z)
        fused = _lib.launch_count() == 1
        sets.append(dict(count=count, pr=pr, z=z, dout=t["dout"], out=out, x=x, silu_z=F.silu(z), fused=fused))

    def fwd(variant):
        def step():
            _lib.test_force_path(policy + 8 if variant == "standalone" else policy)
            for s in sets:
                for _ in range(s["count"]):
                    if variant == "torch_gate":
                        y = s["pr"].forward()[0]
                        y * F.silu(s["z"])
                    else:
                        s["pr"].forward(z=s["z"])
            _lib.test_force_path(policy)
        return step

    def bwd(variant):
        def step():
            for s in sets:
                for _ in range(s["count"]):
                    if variant == "torch_gate":          # what autograd runs for out * F.silu(z), then the scan backward
                        dy = s["dout"] * s["silu_z"]
                        torch.ops.aten.silu_backward(s["dout"] * s["out"], s["z"])
                        s["pr"].backward(dy, s["x"])
                    else:
                        s["pr"].backward(s["dout"], s["x"], z=s["z"], out=s["out"])
        return step

    res = []
    tag = f"{name}" + (f" (policy {policy})" if policy else "")
    for leg, make, variants in (("forward", fwd, ("torch_gate", "standalone", "fused")), ("backward", bwd, ("torch_gate", "gated"))):
        graphs = {v: capture(make(v)) for v in variants}
        rec = summary(f"{tag} ({leg})", alternate({v: g.replay for v, g in graphs.items()}, repeats, flush), "torch_gate")
        if leg == "forward":
            rec["gate_inside_scan_fwdr"] = all(s["fused"] for s in sets)
        res.append(rec)
        del graphs
        torch.cuda.empty_cache()
    _lib.test_force_path(0)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_scan_gate.py needs a CUDA device")
    import ceigm_unet_b200 as P
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > 126 MB of L2
    lines = [{"gpu": gpu_info(), "library": P.version(), "repeats": args.repeats}]
    print(json.dumps(lines[0]), flush=True)
    vm = [(c, {k: v.cuda() for k, v in inp.items()}) for c, inp in build_inputs(WORKLOADS["vm_d192"], "cuda", on_device=True)]
    for name, sets, policy in (("mamba_d1536", mamba_inputs(), 0), ("mamba_d1536", mamba_inputs(), 2), ("vm_d192", vm, 0)):
        for rec in gate_workload(name, sets, policy, args.repeats, flush):
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
