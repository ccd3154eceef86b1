#!/usr/bin/env python
"""bench.py — throughput of the SS2D selective-scan hot path on B200 (contract: task statement ④).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one forward + one backward pass of the selective scan over one batch of synthetic input
(the reference test's seeded recipe, kernels/selective_scan/test_selective_scan.py:406-441), called through
the reference-facing drop-in API `selective_scan_cuda_core.fwd / .bwd`.

Metric (BASELINE.json): selective-scan algorithmic HBM GB/s (fwd+bwd), whole job over all ranks.
Algorithmic bytes (SURVEY.md §8d, level 1): fwd s(3 B Dt L + 2 B K N L), bwd s(5 B Dt L + 4 B K N L).

Workloads (`--workload`):
  vm_d192 (default)  K=4 directions, d_state N=16, D=192 (Dt=768), L=56^2, batch 24, fp32 — the north-star
                     SS2D regime on the stage-1 map of a 224^2 Synapse slice at the config-2 batch.
  vm_d96 / vm_d384 / vm_d768_l112 ... other points of BASELINE config 4.
  gm_live            the 104 single-direction N=1 scan calls of one GM-UNet forward+backward at batch 24
                     (gm_live_g4: the same scans as 26 grouped G=4 calls, the way the fused GroupMambaLayer issues them).
Multi-GPU: the batch is sharded, every rank runs an independent replica of the per-GPU workload (weak scaling,
no data-path collective — SURVEY.md §8e); the timed region is bracketed by barrier + synchronize and the
slowest rank's device time is used.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: importing its modules must not write __pycache__ into it

import torch  # noqa: E402

# name -> list of (count, batch, Dt, L, N, G) scan calls making up one step
WORKLOADS = {
    "vm_d96": [(1, 24, 384, 3136, 16, 4)],
    "vm_d192": [(1, 24, 768, 3136, 16, 4)],
    "vm_d384": [(1, 24, 1536, 3136, 16, 4)],
    "vm_d192_l80": [(1, 24, 768, 6400, 16, 4)],
    "vm_d192_l112": [(1, 24, 768, 12544, 16, 4)],
    "vm_d768_l112": [(1, 24, 3072, 12544, 16, 4)],
    # live GM-UNet census (SURVEY.md §8 table): per forward 20/24/48/12 calls on the four stages
    "gm_live": [(20, 24, 16, 3136, 1, 1), (24, 24, 32, 784, 1, 1), (48, 24, 87, 196, 1, 1), (12, 24, 112, 49, 1, 1)],
}
# single calls of the live regime, alone and with the 4 SS2Ds of a GroupMambaLayer grouped into one launch (G=4)
for _i, (_c, _b, _d, _l, _n, _g) in enumerate(WORKLOADS["gm_live"], 1):
    WORKLOADS[f"gm_s{_i}"] = [(1, _b, _d, _l, _n, _g)]
    WORKLOADS[f"gm_s{_i}_g4"] = [(1, _b, 4 * _d, _l, _n, 4)]
WORKLOADS["gm_s1_b64_512"] = [(1, 64, 64, 16384, 1, 4)]
# the same 104 scans as the fused GroupMambaLayer issues them: the four SS2Ds of a layer in one G = 4 launch (26 calls)
WORKLOADS["gm_live_g4"] = [(c // 4, b, 4 * d, l, n, 4) for c, b, d, l, n, g in WORKLOADS["gm_live"]]
# small-batch points of the north-star shape (BASELINE config 1 runs batch 1): grid-fill regime
WORKLOADS["vm_d192_b1"] = [(1, 1, 768, 3136, 16, 4)]
WORKLOADS["vm_d192_b2"] = [(1, 2, 768, 3136, 16, 4)]
DEFAULT_WORKLOAD = "vm_d192"
# BASELINE config 4: the whole sweep goes into the driver-run line (other_workloads)
SWEEP_CONFIG4 = ["vm_d96", "vm_d192", "vm_d384", "vm_d192_l80", "vm_d192_l112", "vm_d768_l112"]


def alg_bytes(calls, esize=4):
    fwd = sum(c * esize * (3 * b * dt * L + 2 * b * g * n * L) for c, b, dt, L, n, g in calls)
    bwd = sum(c * esize * (5 * b * dt * L + 4 * b * g * n * L) for c, b, dt, L, n, g in calls)
    return fwd, bwd


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe). The sampler is started
    before the warm-up (nvidia-smi takes a few hundred ms to produce its first line); samples are time-stamped and the
    ones inside the timed region are used, falling back to every sample of the run when the region was too short."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc = gpu_index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        import datetime
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[2]), float(f[3]), [n for n, v in zip(names, f[6:10]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if t_begin is not None and t_begin <= r[0] <= t_end]
        used, scope = (inside, "timed region") if len(inside) >= 2 else (rows, "whole run (timed region shorter than the sampling period)")
        sm = [r[1] for r in used]
        reasons = sorted({n for r in used for n in r[3]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max((r[2] for r in used), default=None),
                "samples": len(sm), "scope": scope, "reasons": reasons}


def build_inputs(calls, device, on_device=False):
    """One input set per distinct shape (reused across the `count` repetitions of that shape). Host tensors by default (the
    end-to-end leg starts from pinned host memory); on_device=True draws the same recipe with the device generator (the
    sweep's largest point is 11 GB of inputs)."""
    sets = []
    gen = torch.Generator(device=device if on_device else "cpu").manual_seed(0)
    kw = dict(generator=gen, device=device if on_device else "cpu")
    for count, b, dt, L, n, g in calls:
        A = (-0.5 * torch.rand(dt, n, **kw)).float()
        inp = dict(A=A, B=torch.randn(b, g, n, L, **kw), C=torch.randn(b, g, n, L, **kw),
                   D=torch.randn(dt, **kw), delta_bias=0.5 * torch.rand(dt, **kw),
                   u=torch.randn(b, dt, L, **kw), delta=0.5 * torch.rand(b, dt, L, **kw),
                   dout=torch.randn(b, dt, L, **kw))
        sets.append((count, inp))
    return sets


GRAD_NAMES = ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias")
DUMP_BUDGET_BYTES = 60_000_000      # under 64 MB with the .npy headers


def dump_outputs(out_dir, kept):
    """Writes what fwd / bwd returned for each input set as <out_dir>/<name>.npy in float32: out, the final state
    (x[:, :, -1, 1::2]) and the seven gradients, prefixed `call<i>_` when the step has several input sets. An array larger
    than its equal share of the budget is replaced by a fixed sample of its flattened elements: the first `share` indices
    of a permutation drawn from a CPU generator seeded 0, in ascending order, so that two builds run with the same
    arguments can be compared element by element."""
    import numpy as np
    arrays = {}
    for i, (out, x, grads) in enumerate(kept):
        named = {"out": out, "last_state": x[:, :, -1, 1::2], **dict(zip(GRAD_NAMES, grads))}
        prefix = f"call{i}_" if len(kept) > 1 else ""
        arrays.update({prefix + k: v for k, v in named.items() if v is not None})
    share = DUMP_BUDGET_BYTES // 4 // len(arrays)
    os.makedirs(out_dir, exist_ok=True)
    samples = {}
    for name, v in arrays.items():
        v = v.detach()
        if v.numel() > share:
            if v.numel() not in samples:
                gen = torch.Generator().manual_seed(0)
                samples[v.numel()] = torch.randperm(v.numel(), generator=gen)[:share].sort().values.to(v.device)
            v = v.reshape(-1)[samples[v.numel()]]
        np.save(os.path.join(out_dir, name + ".npy"), v.float().cpu().numpy())


def run_ours(args, rank, world, local_rank):
    import ceigm_unet_b200 as pkg
    from ceigm_unet_b200 import dist as D
    from ceigm_unet_b200.dropin import selective_scan_cuda_core as core
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl ours) needs a CUDA device: there is no CPU fallback")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    calls = WORKLOADS[args.workload]
    fwd_b, bwd_b = alg_bytes(calls)
    host_sets = build_inputs(calls, device)
    dev_sets = [(c, {k: v.to(device) for k, v in inp.items()}) for c, inp in host_sets]
    resident = sum(v.numel() * 4 for _, inp in dev_sets for v in inp.values())

    def step(record=None, keep=False):
        """One step; with keep=True returns (out, x, grads) of the last call of every input set."""
        kept = []
        for count, t in dev_sets:
            for _ in range(count):
                if record is not None:
                    record[0].record()
                out, x = core.fwd(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], True, 1)
                if record is not None:
                    record[1].record()
                grads = core.bwd(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], t["dout"], x, True, 1)
                if record is not None:
                    record[2].record()
            if keep:
                kept.append((out, x, grads))
        return kept

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(device)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    # ---- timed region: K steps, device time via CUDA events on the launching (current) stream ----
    single_call = len(calls) == 1 and calls[0][0] == 1
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)] if single_call else None
    pkg.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        last = step(evs[i] if evs else None, keep=args.dump_outputs is not None and i == args.steps - 1)
    e1.record()
    barrier()
    clocks = sampler.stop(wall0, time.time())
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    launches = pkg.launch_count()
    ms = D.max_over_ranks(e0.elapsed_time(e1), device)      # slowest rank's device time
    ms_per_step = ms / args.steps
    value = world * (fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9

    peak, peak_src = load_peaks()
    roofline = None
    extra = {}
    if evs:
        fwd_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)
        bwd_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in evs)
        ach = bwd_b / (bwd_ms * 1e-3) / 1e9
        if all(c[4] == 1 for c in calls):
            kname = "scan_n1_bwd_rows_kernel"
        elif all(8 < c[4] <= 16 for c in calls):
            kname = "scan_bwd2_kernel"         # fp32 + TMA fast path (csrc/scan_bwd2.cu)
        else:
            kname = "scan_bwd_kernel"
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                for key, rec in json.load(f).items():
                    if key.startswith(kname) and key.endswith("@ " + args.workload):
                        traffic, traffic_src = rec["traffic"], f"profiles/r2_traffic.json ({rec['report']}, dram read+write of one launch)"
        roofline = {"bound": "hbm", "kernel": kname + " (+ finalize and dB/dC memsets inside the bwd call)",
                    "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": traffic, "traffic_source": traffic_src, "alg_bytes_per_launch": bwd_b, "peak_source": peak_src,
                    "note": "d_state=16 is instruction-issue / MUFU.EX2 bound on B200, not HBM-bound: see DESIGN.md §3"}
        extra = {"fwd_ms": round(fwd_ms, 4), "bwd_ms": round(bwd_ms, 4),
                 "fwd_GBps": round(fwd_b / (fwd_ms * 1e-3) / 1e9, 1), "bwd_GBps": round(ach, 1),
                 "fwd_frac_of_peak": round(fwd_b / (fwd_ms * 1e-3) / 1e9 / peak, 4)}

    # ---- end to end: host buffers in pinned memory; every step copies every input host->device and every result
    #      device->host. The batch is cut into chunks that are pipelined over two streams so that H2D, the scan
    #      kernels and D2H of different chunks overlap (samples are independent; dA/dD/dbias are summed on the host).
    pinned = [(c, {k: v.pin_memory() for k, v in inp.items()}) for c, inp in host_sets]
    h2d = sum(c * sum(v.numel() * 4 for v in inp.values()) for c, inp in pinned)
    streams = [torch.cuda.Stream(device) for _ in range(args.e2e_streams)]
    res_host = {}
    BATCHED = ("u", "delta", "B", "C", "dout")

    def e2e_step():
        d2h = 0
        for ci, (count, inp) in enumerate(pinned):
            nb = inp["u"].shape[0]
            nchunk = min(args.e2e_chunks, nb) if nb >= 8 else 1
            for rep in range(count):
                for ch in range(nchunk):
                    a, bnd = D.shard_batch(nb, ch, nchunk)
                    st = streams[ch % len(streams)]
                    with torch.cuda.stream(st):
                        t_ = {k: (v[a:bnd] if k in BATCHED else v).to(device, non_blocking=True) for k, v in inp.items()}
                        out, x = core.fwd(t_["u"], t_["delta"], t_["A"], t_["B"], t_["C"], t_["D"], t_["delta_bias"], True, 1)
                        grads = core.bwd(t_["u"], t_["delta"], t_["A"], t_["B"], t_["C"], t_["D"], t_["delta_bias"],
                                         t_["dout"], x, True, 1)
                        outs = [out] + list(grads)
                        key = (ci, ch)
                        if key not in res_host:
                            res_host[key] = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
                        for hbuf, o in zip(res_host[key], outs):
                            hbuf.copy_(o, non_blocking=True)
                            d2h += o.numel() * o.element_size()
        for st in streams:
            st.synchronize()
        return d2h

    d2h = e2e_step()
    e2e_steps = max(3, min(args.steps, 10))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    dt_e2e = D.max_over_ranks(time.perf_counter() - t0, device)
    e2e_val = world * (fwd_b + bwd_b) * e2e_steps / dt_e2e / 1e9

    line = {
        "metric": "selective-scan fwd+bwd algorithmic HBM GB/s", "value": round(value, 1), "unit": "GB/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": our_config(args.workload),
        "frac_of_hbm_peak": round(value / world / peak, 4),
        "e2e": {"value": round(e2e_val, 1), "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "note": "pinned host buffers; every input copied in and every result copied out per step; %d batch chunks pipelined over %d streams (PCIe-bound)" % (args.e2e_chunks, args.e2e_streams)},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
    }
    line.update(extra)
    # secondary ceilings for d_state > 1 (DESIGN.md): one MUFU.EX2 per (row, position, state) forward, two backward,
    # plus softplus; measured MUFU rate 16 lanes/clk/SM (tools/ubench/pipes.cu: 4.6e12 ex2/s at 1.965 GHz)
    ex2 = sum(c * b * dt * L * (3 * n + 6) for c, b, dt, L, n, g in calls)
    line["mufu_roofline"] = {"ex2_per_step": ex2, "peak_ex2_per_s": 4.6e12, "floor_ms": round(ex2 / 4.6e12 * 1e3, 4),
                             "frac": round(ex2 / 4.6e12 * 1e3 / ms_per_step, 4)}
    if rank == 0 and world == 1 and not args.no_extras:
        line["other_workloads"] = other_workloads(core, device, peak, exclude=args.workload)
        line["projections"] = projection_workloads(device, peak)
        line["ffn_depthwise"] = ffn_workloads(device, peak)
    if not args.no_model:
        # every rank takes part (batch-sharded data parallel, gradient all-reduce on NCCL); rank 0 reports
        line["model"] = model_workloads(device, rank, world)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_port(args.workload)
    return line


def graph_time_ms(core, sets, iters=10, with_bwd=True):
    """GPU time of one step (all calls) replayed from a CUDA graph: no host launch overhead between kernels."""
    def run():
        for count, t in sets:
            for _ in range(count):
                out, x = core.fwd(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], True, 1)
                if with_bwd:
                    core.bwd(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], t["delta_bias"], t["dout"], x, True, 1)
    g, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.stream(st):
        run()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=st):
            run()
    torch.cuda.synchronize()
    for _ in range(3):
        g.replay()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def other_workloads(core, device, peak, exclude):
    """Context numbers in the same run (not the headline), each one CUDA-graph replay of fwd+bwd, median of 10:
    the whole BASELINE config-4 sweep, two small-batch points, the live GM-UNet regime (d_state = 1: the scan calls of one
    224^2 batch-24 training step, one layer's grouped call, the 512^2 batch-64 stage-1 shape of config 5), and — when
    baseline/_ref/ext holds it — the REFERENCE's own CUDA kernel recompiled for sm_100 on the same box and inputs."""
    out = []
    names = [n for n in SWEEP_CONFIG4 if n != exclude] + ["vm_d192_b1", "vm_d192_b2", "gm_live", "gm_live_g4", "gm_s1_g4", "gm_s1_b64_512"]
    ref_ext = None
    try:
        from harness import refmodel
        ref_ext = refmodel.load_ref_cuda_ext()
    except Exception:      # noqa: BLE001  (the baseline column is optional; never let it break the bench line)
        ref_ext = None
    ref_points = {"vm_d192", "gm_live", "gm_s1_b64_512"}
    for name in names + ([exclude] if exclude in ref_points else []):
        calls = WORKLOADS[name]
        sets = build_inputs(calls, device, on_device=True)
        fb, bb = alg_bytes(calls)
        rec = {"workload": name, "calls_per_step": [list(c) for c in calls]}
        if name != exclude:
            ms_f = graph_time_ms(core, sets, with_bwd=False)
            ms = graph_time_ms(core, sets, with_bwd=True)
            rec.update({"fwd_ms": round(ms_f, 4), "fwd_bwd_ms": round(ms, 4), "fwd_GBps": round(fb / ms_f / 1e6, 1),
                        "fwd_bwd_GBps": round((fb + bb) / ms / 1e6, 1), "frac_of_hbm_peak": round((fb + bb) / ms / 1e6 / peak, 4),
                        "timing": "CUDA graph replay"})
            if name in ("gm_live", "gm_live_g4"):
                rec["scan_only_slices_per_s"] = round(calls[0][1] / (ms * 1e-3), 1)
        if ref_ext is not None and name in ref_points:
            try:
                rf = graph_time_ms(ref_ext, sets, with_bwd=False)
                rfb = graph_time_ms(ref_ext, sets, with_bwd=True)
                rec["ref_cuda_kernel"] = {"fwd_ms": round(rf, 4), "fwd_bwd_ms": round(rfb, 4),
                                          "fwd_bwd_GBps": round((fb + bb) / rfb / 1e6, 1),
                                          "what": "reference cus/ extension (setup.py flags) recompiled for sm_100, same inputs, CUDA graph replay"}
                if "fwd_bwd_ms" in rec:
                    rec["speedup_vs_ref_cuda_kernel"] = round(rfb / rec["fwd_bwd_ms"], 2)
            except Exception as e:      # noqa: BLE001
                rec["ref_cuda_kernel"] = {"error": str(e)[:200]}
        out.append(rec)
        del sets
        torch.cuda.empty_cache()
    return out


def projection_workloads(device, peak):
    """The dense contractions around the scan on the tcgen05 kernel (csrc/linear_tc.cu) at the north-star SS2D shape
    (d_model 96, d_inner 192, batch 24, 56 x 56): in_proj + chunk + NHWC->NCHW in one launch and out_proj, next to the
    library composition they replace (F.linear [+ chunk + permute().contiguous()]); CUDA-graph replay, L2 flushed between
    replays, algorithmic bytes = operands read once + outputs written once."""
    import torch.nn.functional as F
    from ceigm_unet_b200 import ops
    Bn, H, W, C, D = 24, 56, 56, 96, 192
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def timed(fn, iters=10):
        g, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.stream(st):
            fn()
            torch.cuda.synchronize()
            with torch.cuda.graph(g, stream=st):
                fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    out = []
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    try:
        for dtype, name in ((torch.float32, "f32 (tf32 math)"), (torch.bfloat16, "bf16")):
            es = 4 if dtype == torch.float32 else 2
            x = torch.randn(Bn, H, W, C, device=device).to(dtype)
            y = torch.randn(Bn, H, W, D, device=device).to(dtype)
            Win = (torch.randn(2 * D, C, device=device) / C ** 0.5).to(dtype)
            Wout = (torch.randn(C, D, device=device) / D ** 0.5).to(dtype)
            M = Bn * H * W
            torch.backends.cuda.matmul.allow_tf32 = True      # the library column gets tensor cores too

            def lib_in():
                xi, z = F.linear(x, Win).chunk(2, dim=-1)
                return xi.permute(0, 3, 1, 2).contiguous(), z
            for op, ours, lib, nbytes in (
                    ("in_proj + chunk + NHWC->NCHW (ss2d.py:504-510)",
                     lambda: ops.linear_tc(x, Win, None, [(D, ("planes", H * W), False), (D, "rows", False)]), lib_in, es * M * (C + 2 * D)),
                    ("out_proj (ss2d.py:518)", lambda: ops.linear_tc(y, Wout, None, [(C, "rows", False)]),
                     lambda: F.linear(y, Wout), es * M * (C + D))):
                ms, ms_lib = timed(ours), timed(lib)
                out.append({"op": op, "kernel": "linear_tc_kernel (tcgen05.mma, TMA, TMEM)", "dtype": name, "rows": M, "K_N": [x.shape[-1] if "in_proj" in op else D, 2 * D if "in_proj" in op else C],
                            "ms": round(ms, 4), "alg_GBps": round(nbytes / ms / 1e6, 1), "frac_of_hbm_peak": round(nbytes / ms / 1e6 / peak, 4),
                            "library_ms": round(ms_lib, 4), "speedup_vs_library": round(ms_lib / ms, 2)})
    except Exception as e:      # noqa: BLE001
        out.append({"error": repr(e)[:300]})
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old_tf32
    return out


def ffn_workloads(device, peak):
    """The depthwise stack of the GroupMamba FFNs (SURVEY.md §8-f3; csrc/ffn_dw.cu) at the stage-1 encoder shape of a 224^2
    batch-24 step (hidden 512 @ 56 x 56, bf16 — the autocast training configuration): the module's forward + backward
    between fc1 and fc2 (ceigm_unet_b200.functional.ffn_depthwise) next to the reference composition (transpose to NCHW,
    F.conv2d depthwise, GELU, [split, three depthwise convs, cat, residual], transpose back: groupmamba.py:446-455, 76-78,
    custom_mlp.py:323-336, 363-366); CUDA-graph replay, L2 flushed between replays. Algorithmic bytes per element of the
    (B, L, C) tensor (s = 2): PVT2FFN forward 2 s, backward 3 s (GELU' on the recomputed pre-activation) + 2 s (transposed conv) + 2 s
    (weight gradient) = 9 s; custom_ffn adds the multi-scale pass forward (2 s), its transposed pass (2 s) and three 1/8-width
    reductions (0.75 s) = 13.75 s."""
    import torch.nn.functional as F
    import ceigm_unet_b200 as pkg
    from ceigm_unet_b200 import functional as Fn
    Bn, H, W, C = 24, 56, 56, 512
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    out = []
    try:
        for name, ctor in (("PVT2FFN", pkg.PVT2FFN), ("custom_ffn", pkg.custom_ffn)):
            torch.manual_seed(0)
            mod = ctor(C // 8, C).to(device)
            h = torch.randn(Bn, H * W, C, device=device).to(torch.bfloat16).requires_grad_(True)
            dy = torch.randn(Bn, H * W, C, device=device).to(torch.bfloat16)
            conv3 = mod.dwconv.dwconv
            ms_convs = (mod.custom.dwconv_3x3, mod.custom.dwconv_5x5, mod.custom.dwconv_7x7) if name == "custom_ffn" else None
            params = [p for m in ((conv3,) + (ms_convs or ())) for p in m.parameters()]

            def ours():
                y = Fn.ffn_depthwise(h, (H, W), conv3, ms_convs)
                return torch.autograd.grad(y, [h] + params, dy)

            def lib():
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    img = h.transpose(1, 2).reshape(Bn, C, H, W)
                    y = F.gelu(conv3(img))
                    if ms_convs is not None:
                        gc = ms_convs[0].weight.shape[0]
                        a, b3, b5, b7 = torch.split(y, (C - 3 * gc, gc, gc, gc), dim=1)
                        y = y + torch.cat((a, ms_convs[0](b3), ms_convs[1](b5), ms_convs[2](b7)), dim=1)
                    y = y.flatten(2).transpose(1, 2)
                return torch.autograd.grad(y, [h] + params, dy.to(y.dtype))

            def timed(fn, iters=10):
                g, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
                with torch.cuda.stream(st):
                    fn()
                    torch.cuda.synchronize()
                    with torch.cuda.graph(g, stream=st):
                        fn()
                torch.cuda.synchronize()
                ts = []
                for _ in range(iters):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                return statistics.median(ts)

            ms, ms_lib = timed(ours), timed(lib)
            passes = 9.0 if name == "PVT2FFN" else 13.75      # tensor passes of one forward + backward (docstring)
            nbytes = passes * 2 * h.numel()
            out.append({"op": f"{name} depthwise stack fwd+bwd (hidden {C} @ {H}x{W}, batch {Bn})", "kernel": "dwnhwc_stencil_kernel / dwnhwc_wgrad_kernel",
                        "dtype": "bf16", "ms": round(ms, 4), "alg_GBps": round(nbytes / ms / 1e6, 1),
                        "frac_of_hbm_peak": round(nbytes / ms / 1e6 / peak, 4), "reference_composition_ms": round(ms_lib, 4),
                        "speedup_vs_reference_composition": round(ms_lib / ms, 2)})
    except Exception as e:      # noqa: BLE001
        out.append({"error": repr(e)[:300]})
    return out


def model_workloads(device, rank, world):
    """BASELINE configs 2 / 3 / 5 (and 1 as the CPU column): the UNMODIFIED reference GM-UNet through the drop-in
    (harness/workloads.py) — 224^2 batch-24 bf16 training slices/s (with the NCCL gradient all-reduce inside the timed
    region when world > 1) and 512^2 batch-64 inference slices/s. Needs baseline/_ref (harness/install_ref.py)."""
    try:
        from harness import refmodel, workloads as W
        if not refmodel.available():
            return {"unavailable": "baseline/_ref not installed (harness/install_ref.py)"}
        res = {}
        for key, kw in (("train_224_b24_dropin_eager", dict(level="dropin", graphs=False)),
                        ("train_224_b24_fused_graphs", dict(level="fused", graphs=True))):
            try:
                res[key] = W.train_bench(device, rank, world, per_gpu_batch=24, steps=5, warmup=3, **kw)
            except Exception as e:      # noqa: BLE001
                res[key] = {"error": repr(e)[:300]}
        if world > 1:
            try:
                res["train_acdc_224_b24_fused_graphs"] = W.train_bench(device, rank, world, per_gpu_batch=24, num_classes=4, steps=5,
                                                                        warmup=3, level="fused", graphs=True, weight_decay=1e-4)
            except Exception as e:      # noqa: BLE001
                res["train_acdc_224_b24_fused_graphs"] = {"error": repr(e)[:300]}
        for key, kw in (("infer_512_b64_dropin_eager", dict(level="dropin", graphs=False)),
                        ("infer_512_b64_fused_graphs", dict(level="fused", graphs=True))):
            try:
                res[key] = W.infer_bench(device, rank, world, per_gpu_batch=64, size=512, steps=3, warmup=2, **kw)
            except Exception as e:      # noqa: BLE001
                res[key] = {"error": repr(e)[:300]}
        if rank == 0 and world == 1:
            try:
                res["cpu_reference_224_b1"] = W.cpu_reference_step()
            except Exception as e:      # noqa: BLE001
                res["cpu_reference_224_b1"] = {"error": repr(e)[:300]}
        return res
    except Exception as e:      # noqa: BLE001
        return {"error": repr(e)[:300]}


def cpu_baseline_port(workload, sample_batch=8, min_seconds=10.0):
    """The C oracle (oracle/scan_oracle.c, OpenMP over rows, f64 accumulate) on a bounded sample of the same workload:
    fwd+bwd on `sample_batch` samples of the largest call, repeated until at least `min_seconds` of CPU work."""
    from oracle import c_oracle
    calls = WORKLOADS[workload]
    count, b, dt, L, n, g = max(calls, key=lambda c: c[0] * c[1] * c[2] * c[3] * c[4])
    sb = min(sample_batch, b)
    gen = torch.Generator().manual_seed(0)
    A = (-0.5 * torch.rand(dt, n, generator=gen)).numpy()
    Bm, Cm = torch.randn(sb, g, n, L, generator=gen).numpy(), torch.randn(sb, g, n, L, generator=gen).numpy()
    Dv, bias = torch.randn(dt, generator=gen).numpy(), (0.5 * torch.rand(dt, generator=gen)).numpy()
    u, dl = torch.randn(sb, dt, L, generator=gen).numpy(), (0.5 * torch.rand(sb, dt, L, generator=gen)).numpy()
    dy = torch.randn(sb, dt, L, generator=gen).numpy()
    c_oracle.scan_fwd(u[:1], dl[:1], A, Bm[:1], Cm[:1], Dv, bias, True)          # warm-up (page-in, thread pool)
    reps, t0 = 0, time.perf_counter()
    while True:
        c_oracle.scan_fwd(u, dl, A, Bm, Cm, Dv, bias, True, acc="f64")
        c_oracle.scan_bwd(u, dl, A, Bm, Cm, Dv, bias, dy, True, acc="f64")
        reps += 1
        dt_s = time.perf_counter() - t0
        if dt_s >= min_seconds or reps >= 200:
            break
    fwd_b, bwd_b = alg_bytes([(1, sb, dt, L, n, g)])
    return {"value": round(reps * (fwd_b + bwd_b) / dt_s / 1e9, 4), "unit": "GB/s", "cores": c_oracle.num_threads(),
            "kind": "port", "seconds": round(dt_s, 2),
            "sample": f"C oracle (OpenMP) fwd+bwd on batch {sb} of {b} of the largest call of '{workload}' "
                      f"(Dt={dt}, L={L}, N={n}, G={g}), {reps} repetitions"}


def our_config(workload):
    """The `config` object of a bench line: identical in the `ours` and the `reference` arm (the driver compares them)."""
    calls = WORKLOADS[workload]
    fwd_b, bwd_b = alg_bytes(calls)
    resident = sum(4 * (3 * b * dt * L + 2 * b * g * n * L + 2 * dt + dt * n) for c, b, dt, L, n, g in calls)
    return {"workload": workload, "calls_per_step": [list(c) for c in calls],
            "call_fields": ["count", "batch", "Dt=K*D", "L", "d_state", "groups"],
            "api": "selective_scan_cuda_core.fwd/bwd drop-in -> C ABI ss2d_scan_fwd/bwd",
            "l2_policy": "inputs larger than L2 (resident working set %.0f MB vs 126 MB L2)" % (resident / 1e6),
            "alg_bytes_fwd": fwd_b, "alg_bytes_bwd": bwd_b, "per_gpu_batch": calls[0][1]}


def run_reference(args):
    """Reference arm: the reference's own CPU path for the scan — its pure-PyTorch `selective_scan_ref`
    (kernels/selective_scan/test_selective_scan.py:168-234) forward + autograd backward, restated in
    oracle/selective_scan_ref.py (the reference has no native CPU code to compile: DESIGN.md §4) — on all host threads.

    Same workload and metric as the `ours` arm. One step processes a BOUNDED SAMPLE of it: a slab of whole channel rows of one
    (batch, group) — a quarter of the group's rows with their shared B / C, the way the workload itself amortises B / C over
    the rows of a group (a whole 192-row group takes 70 s per step in this implementation: its autograd backward moves
    O(L^2) memory, SURVEY.md §8c). The value is the workload's algorithmic bytes x (rows processed / rows in the workload) /
    time, i.e. the speed at which this implementation would get through the SAME step."""
    from oracle.selective_scan_ref import selective_scan_ref
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    calls = WORKLOADS[args.workload]
    count, b, dt, L, n, g = max(calls, key=lambda c: c[0] * c[1] * c[2] * c[3] * c[4])
    dpg = dt // g
    total_rows = sum(c * bb * dd for c, bb, dd, _, _, _ in calls)
    fwd_all, bwd_all = alg_bytes(calls)

    def make(rows):
        gen = torch.Generator().manual_seed(0)
        t = dict(u=torch.randn(1, rows, L, generator=gen), delta=0.5 * torch.rand(1, rows, L, generator=gen),
                 A=-0.5 * torch.rand(rows, n, generator=gen), B=torch.randn(1, 1, n, L, generator=gen),
                 C=torch.randn(1, 1, n, L, generator=gen), D=torch.randn(rows, generator=gen),
                 delta_bias=0.5 * torch.rand(rows, generator=gen))
        for v in t.values():
            v.requires_grad_(True)
        t["dout"] = torch.randn(1, rows, L, generator=gen)
        return t

    def one(t):
        for k, v in t.items():
            if k != "dout":
                v.grad = None
        out = selective_scan_ref(t["u"], t["delta"], t["A"], t["B"], t["C"], t["D"], None, t["delta_bias"], True)
        out.backward(t["dout"])

    # slab = a quarter of a group's rows (48 of 192 for vm_d192); shrink only if (steps + warmup) slabs would not fit ~4 min
    rows = max(1, min(dpg, max(dpg // 4, 1)))
    t = make(rows)
    t0 = time.perf_counter(); one(t); first = time.perf_counter() - t0
    budget = 240.0 / max(1, args.steps + args.warmup)
    while rows > 4 and first > budget:
        rows = max(4, rows // 2)
        t = make(rows)
        t0 = time.perf_counter(); one(t); first = time.perf_counter() - t0
    for _ in range(max(args.warmup - 1, 0)):
        one(t)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one(t)
    sec = (time.perf_counter() - t0) / args.steps
    val = (fwd_all + bwd_all) * (rows / total_rows) / sec / 1e9
    sample = (f"selective_scan_ref fwd + autograd bwd on a slab of {rows} whole rows (1 batch, 1 group of {dpg}, shared B/C, "
              f"L={L}, N={n}) of the {total_rows} (batch x channel) rows of '{args.workload}' per step; bytes counted as the "
              f"workload's algorithmic bytes x {rows}/{total_rows}")
    return {
        "impl": "reference", "metric": "selective-scan fwd+bwd algorithmic HBM GB/s", "value": round(val, 6),
        "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(sec * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": our_config(args.workload),
        "cpu_baseline": {"value": round(val, 6), "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample,
                         "sample_rows": rows, "seconds_per_slab": round(sec, 3),
                         "whole_step_would_take_s": round(sec * total_rows / rows, 1)},
        "e2e": {"value": round(val, 6), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=8, help="batch chunks of the end-to-end leg (H2D / scan / D2H pipelining)")
    ap.add_argument("--e2e-streams", type=int, default=4)
    ap.add_argument("--no-extras", action="store_true", help="skip the other_workloads context block")
    ap.add_argument("--no-model", action="store_true", help="skip the model-level (GM-UNet train / inference) block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what fwd / bwd returned in the last timed step as DIR/<name>.npy (float32, at most 64 MB in "
                         "all: larger arrays are replaced by a fixed seeded sample of their elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs dumps the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(run_reference(args)), flush=True)
        return 0

    if world > 1:
        from ceigm_unet_b200 import dist as D
        D.init_from_env("nccl")
    try:
        line = run_ours(args, rank, world, local_rank)
        if rank == 0:
            print(json.dumps(line), flush=True)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
