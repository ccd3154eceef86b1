"""Cost of Mamba-2's chunked scan (`mamba_chunk_scan_combined`, csrc/ssd.cu), forward and forward + backward, against the two
routes a user of this library has without it:
  (a) scan: the library's `selective_scan` on the expanded problem: x as u (batch, heads * headdim, L), dt repeated over
      headdim as delta, A[k] repeated into a (heads * headdim, dstate) matrix, D and dt_bias repeated, B and C as
      (batch, groups, dstate, L). The layout copies are part of the route, since the Mamba-2 tensors do not come in that layout;
  (b) torch: the chunked composition of mamba_ssm's `ssd_minimal_discrete` (einsums on cuBLAS, (batch, heads, chunks, Q, Q)
      score tensors) in the I/O dtype.
Mamba-2 settings: D per head, dt_bias, softplus, no z (Mamba2 gates in its RMSNorm), one group, chunk 256, L 2048.

Each route is captured into a CUDA graph and the graphs of one workload are replayed alternately in one process, L2 overwritten
(256 MB) before every timed replay; each number is the median (and min ... max) of the repeats. Before timing, the routes'
outputs are compared with the library's (max error over max |value|).
FLOPs per (batch, head, chunk of Q positions), the products the chunked algorithm needs with the causal half of the Q x Q
scores: 2 Q P N (chunk state) + 2 Q P N (state to output) + Q^2 N (scores) + Q^2 P (scores times x). Bytes: x and out
(2 s b L h P), B and C (2 s b L g N), dt (s b L h), final states not written; s = element size. The shares are of one B200's
data-sheet bf16 dense peak (2,250 TFLOP/s; the fp32 path runs three TF32 products per product, counted once) and of 7.7 TB/s
of HBM3e; "roofline_bound" names the larger of the two lower limits on time, not what limits the kernels.
Forward + backward: autograd.grad of every input of each route, given dout, in the same graphs-and-alternation scheme.
The GPU name and power limit are read in the same run.

usage: python tools/bench_ssd.py [--repeats 15] [--out profiles/r7_bench_ssd.jsonl]"""
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
BF16_PEAK = 2.25e15
Q = 256
MODELS = {"mamba2-130m": 24, "mamba2-2.7b": 80}     # heads of headdim 64, dstate 128, one group
P, N, G, L = 64, 128, 1, 2048
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def flops(b, h):
    chunks = (L + Q - 1) // Q
    return b * h * chunks * (4 * Q * P * N + Q * Q * (N + P))


def nbytes(b, h, s):
    return s * (2 * b * L * h * P + 2 * b * L * G * N + b * L * h)


def lib_route(x, dt, A, B, C, D, dt_bias):
    import ceigm_unet_b200 as pkg
    return pkg.mamba_chunk_scan_combined(x, dt, A, B, C, Q, D=D, dt_bias=dt_bias, dt_softplus=True)


def scan_route(x, dt, A, B, C, D, dt_bias):
    import ceigm_unet_b200 as pkg
    b, _, h, p = x.shape
    dim = h * p
    u = x.reshape(b, L, dim).transpose(1, 2).contiguous()
    delta = dt.repeat_interleave(p, dim=2).transpose(1, 2).contiguous()
    Ae = A.repeat_interleave(p)[:, None].expand(dim, B.shape[-1]).contiguous()
    y = pkg.selective_scan(u, delta, Ae, B.permute(0, 2, 3, 1).contiguous(), C.permute(0, 2, 3, 1).contiguous(),
                           D.repeat_interleave(p), dt_bias.repeat_interleave(p), True)
    return y.transpose(1, 2).reshape(b, L, h, p)


def _segsum(a):
    T = a.shape[-1]
    cs = torch.cumsum(a, -1)
    s = cs[..., :, None] - cs[..., None, :]
    return s.masked_fill(~torch.tril(torch.ones(T, T, dtype=torch.bool, device=a.device)), -torch.inf)


def torch_route(x, dt, A, B, C, D, dt_bias):
    """ssd_minimal_discrete in x's dtype, with the softplus of dt and the D skip."""
    b, _, h, p = x.shape
    t = F.softplus(dt.float() + dt_bias).to(x.dtype)
    X = (x * t[..., None]).reshape(b, L // Q, Q, h, p)
    a = (t * A.to(x.dtype)).reshape(b, L // Q, Q, h).permute(0, 3, 1, 2)
    Bc = B.reshape(b, L // Q, Q, G, -1).repeat_interleave(h // G, dim=3)
    Cc = C.reshape(b, L // Q, Q, G, -1).repeat_interleave(h // G, dim=3)
    cum = torch.cumsum(a, -1)
    y_diag = torch.einsum("bclhn,bcshn,bhcls,bcshp->bclhp", Cc, Bc, torch.exp(_segsum(a)), X)
    states = torch.einsum("bclhn,bhcl,bclhp->bchpn", Bc, torch.exp(cum[..., -1:] - cum), X)
    states = torch.cat([torch.zeros_like(states[:, :1]), states], 1)
    new_states = torch.einsum("bhzc,bchpn->bzhpn", torch.exp(_segsum(F.pad(cum[..., -1], (1, 0)))), states)[:, :-1]
    y_off = torch.einsum("bclhn,bchpn,bhcl->bclhp", Cc, new_states, torch.exp(cum))
    return (y_diag + y_off).reshape(b, L, h, p) + x * D.to(x.dtype)[:, None]


def stats(ts):
    return statistics.median(ts), [round(min(ts), 4), round(max(ts), 4)]


def workload(model, b, dtype_name, repeats, flush):
    h = MODELS[model]
    dtype = DTYPES[dtype_name]
    gen = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)   # noqa: E731
    args = (r(b, L, h, P).to(dtype), (r(b, L, h) * 0.5 - 3.0).to(dtype), -(torch.rand(h, device="cuda", generator=gen) + 0.5),
            r(b, L, G, N).to(dtype), r(b, L, G, N).to(dtype), r(h), r(h) * 0.5)
    routes = {"lib": lib_route, "scan": scan_route, "torch": torch_route}
    with torch.no_grad():
        ref = lib_route(*args)
        agree = {f"{m}_vs_lib_rel": rel(fn(*args), ref) for m, fn in routes.items() if m != "lib"}

    def fwd(fn):
        def run():
            with torch.no_grad():
                fn(*args)
        return run

    leaves = [a.detach().clone().requires_grad_(True) for a in args]
    dout = torch.randn(args[0].shape, device="cuda", generator=gen).to(dtype)

    def fwd_bwd(fn):
        return lambda: torch.autograd.grad(fn(*leaves), leaves, dout)

    graphs = {m: capture(fwd(fn)) for m, fn in routes.items()}
    graphs.update({m + "_fwd_bwd": capture(fwd_bwd(fn)) for m, fn in routes.items()})
    times = alternate({m: g.replay for m, g in graphs.items()}, repeats, flush)
    del graphs
    torch.cuda.empty_cache()
    fl, by = flops(b, h), nbytes(b, h, torch.finfo(dtype).bits // 8)
    rec = {"workload": f"{model}: {h} heads x {P}, dstate {N}, groups {G}, chunk {Q}, L {L}, D, dt_bias, softplus, no z",
           "batch": b, "io": dtype_name, "flops_fwd": fl, "bytes_fwd": by}
    for m, ts in times.items():
        med, spread = stats(ts)
        rec[f"{m}_ms"] = round(med, 4)
        rec[f"{m}_spread_ms"] = spread
    t = rec["lib_ms"] * 1e-3
    rec["lib_TFLOPs"] = round(fl / t / 1e12, 2)
    rec["lib_bf16_peak_share"] = round(fl / t / BF16_PEAK, 4)
    rec["lib_hbm_share"] = round(by / t / HBM, 4)
    rec["roofline_bound"] = "compute" if fl / BF16_PEAK > by / HBM else "memory"   # the larger lower limit, not the observed limiter
    rec["speedup_vs_scan"] = round(rec["scan_ms"] / rec["lib_ms"], 2)
    rec["speedup_vs_torch"] = round(rec["torch_ms"] / rec["lib_ms"], 2)
    rec["fwd_bwd_speedup_vs_scan"] = round(rec["scan_fwd_bwd_ms"] / rec["lib_fwd_bwd_ms"], 2)
    rec["fwd_bwd_speedup_vs_torch"] = round(rec["torch_fwd_bwd_ms"] / rec["lib_fwd_bwd_ms"], 2)
    rec["agreement"] = {k: float("%.2e" % v) for k, v in agree.items()}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_ssd.py needs a CUDA device")
    import ceigm_unet_b200 as pkg
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > 126 MB of L2
    lines = [{"gpu": gpu_info(), "library": pkg.version(), "repeats": args.repeats}]
    print(json.dumps(lines[0]), flush=True)
    for model in MODELS:
        for b in (1, 8):
            for dtype_name in DTYPES:
                lines.append(workload(model, b, dtype_name, args.repeats, flush))
                print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
