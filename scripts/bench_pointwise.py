"""Time the element-wise squashing layers (csrc/fc_pointwise.cu) against the eager composition of the reference's
formulas (flowcon/transforms/nonlinearities.py; autograd for the backward) on the same GPU, at 4 M rows, and their share
of the bounded_maf workload.

Passes, for each op (sigmoid, tanh, leaky_relu, exp, cauchy) and D in {2, 6, 32, 64, 256}:
  forward, inverse        8 B per element + 4 B per row (x in, y out, logabsdet out)
  backward                12 B per element + 4 B per row (x, grad_y in, grad_x out, grad_logabsdet in), in the layer's
                          forward direction; for sigmoid also `backward_T`, with the temperature gradient reduced
Every pass reports its median time over --iters calls (each after overwriting the L2 with a 256 MB buffer, so it streams
from HBM; ours and eager alternate), the eager composition's time, the rate as a fraction of the device-to-device copy rate
measured in the same run (`copy_GBps`), and the GPU's name and power limit.  Then `share` lines: the new layers' share of
bounded_maf log_prob, sample and an Adam training step (torch.profiler CUDA time of fc_pointwise_* over all kernels).

    python scripts/bench_pointwise.py --out profiles/r08_pointwise_bench.jsonl
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, ops, workloads  # noqa: E402

ROWS = 1 << 22
DS = [2, 6, 32, 64, 256]
OPS = {"sigmoid": _cabi.POINTWISE_SIGMOID, "tanh": _cabi.POINTWISE_TANH, "leaky_relu": _cabi.POINTWISE_LEAKY_RELU,
       "exp": _cabi.POINTWISE_EXP, "cauchy": _cabi.POINTWISE_CAUCHY_CDF}
_FLUSH = []


def timed_pair(fa, fb, iters):
    """Median ms of fa and of fb over `iters` alternated calls, each after overwriting the L2."""
    if not _FLUSH:
        _FLUSH.append(torch.empty(1 << 26, dtype=torch.float32, device="cuda"))
    for _ in range(3):
        fa()
        fb()
    times = ([], [])
    for _ in range(iters):
        for fn, out in ((fa, times[0]), (fb, times[1])):
            _FLUSH[0].zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            out.append(a.elapsed_time(b))
    return tuple(sorted(t)[len(t) // 2] for t in times)


def copy_peak(dev, iters):
    src = torch.empty(1 << 28, dtype=torch.float32, device=dev)  # 1 GB
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return 2 * src.numel() * 4 / (sorted(ts)[len(ts) // 2] * 1e-3) / 1e9


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def eager(op, x, inverse, T):
    """The reference's formulas, eager (the inverse's host-synchronising domain checks included)."""
    if op == "sigmoid":
        if not inverse:
            u = T * x
            return torch.sigmoid(u), (torch.log(T) - F.softplus(-u) - F.softplus(u)).sum(1)
        if torch.min(x) < 0 or torch.max(x) > 1:
            raise ValueError
        xc = torch.clamp(x, 1e-6, 1 - 1e-6)
        y = (1 / T) * (torch.log(xc) - torch.log1p(-xc))
        return y, -(torch.log(T) - F.softplus(-T * y) - F.softplus(T * y)).sum(1)
    if op == "tanh":
        if not inverse:
            y = torch.tanh(x)
            return y, torch.log(1 - y ** 2).sum(1)
        if torch.min(x) <= -1 or torch.max(x) >= 1:
            raise ValueError
        return 0.5 * torch.log((1 + x) / (1 - x)), -torch.log(1 - x ** 2).sum(1)
    if op == "leaky_relu":
        s = 1e-2
        ls = math.log(s)
        mask = (x < 0).float()
        return F.leaky_relu(x, 1 / s if inverse else s), ((-ls if inverse else ls) * mask).sum(1)
    if op == "exp":
        if not inverse:
            return torch.exp(x), x.sum(1)
        if torch.min(x) <= 0:
            raise ValueError
        y = torch.log(x)
        return y, -y.sum(1)
    if not inverse:
        return torch.atan(x) / math.pi + 0.5, (-math.log(math.pi) - torch.log(1 + x ** 2)).sum(1)
    if torch.min(x) < 0 or torch.max(x) > 1:
        raise ValueError
    y = torch.tan(math.pi * (x - 0.5))
    return y, (math.log(math.pi) + torch.log(1 + y ** 2)).sum(1)


def inputs(op, inverse, R, D, g, dev):
    z = torch.randn(R, D, generator=g, device=dev)
    if not inverse or op == "leaky_relu":
        return z
    if op == "exp":
        return torch.exp(z)
    u = torch.sigmoid(z)
    return 2 * u - 1 if op == "tanh" else u


def workload_shares(dev, iters):
    """fc_pointwise_* share of the CUDA time of bounded_maf log_prob, sample and an Adam step (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile

    wl = workloads.get_workload("bounded_maf")
    flow = workloads.build_flow(wl)
    flow.load_state_dict(workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl))
    flow = flow.to(dev)
    x = workloads.sample_data(wl, wl["batch"], seed=0).to(dev)
    opt = torch.optim.Adam(flow.parameters(), lr=1e-4)

    def log_prob():
        with torch.no_grad():
            flow.log_prob(x)

    def sample():
        with torch.no_grad():
            flow.sample(wl["batch"])

    def train():
        opt.zero_grad(set_to_none=True)
        (-flow.log_prob(x).mean()).backward()
        opt.step()

    out = []
    for name, fn in (("log_prob", log_prob), ("sample", sample), ("train_step", train)):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(iters):
                fn()
            torch.cuda.synchronize()
        total = pw = 0.0
        for ev in prof.key_averages():
            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                total += t
                if "pw_" in ev.key:
                    pw += t
        out.append({"pass": "share", "workload": "bounded_maf", "call": name, "rows": wl["batch"],
                    "pointwise_us_per_call": round(pw / iters, 1), "all_kernels_us_per_call": round(total / iters, 1),
                    "share": round(pw / total, 4) if total else None})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r08_pointwise_bench.jsonl")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rows", type=int, default=ROWS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pointwise needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu, watts = torch.cuda.get_device_name(dev), power_limit()
    peak = copy_peak(dev, args.iters)
    R = args.rows
    lines = []

    def emit(rec):
        rec.update({"gpu": gpu, "power_limit_w": watts})
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    def rel(a, b):
        ok = torch.isfinite(b)
        return float(((a - b).abs() / b.abs().clamp_min(1.0))[ok].max())

    T = torch.tensor([1.0], device=dev)
    for D in DS:
        g = torch.Generator(device=dev).manual_seed(D)
        for name, op in OPS.items():
            tp = T if op == _cabi.POINTWISE_SIGMOID else None
            for inverse in (False, True):
                x = inputs(name, inverse, R, D, g, dev)
                ours = lambda: ops.pointwise_layer(x, tp, op, inverse, 1e-2, 1e-6)  # noqa: E731
                ref = lambda: eager(name, x, inverse, T)  # noqa: E731
                t_ours, t_ref = timed_pair(ours, ref, args.iters)
                a, b = ours(), ref()
                nbytes = 8 * R * D + 4 * R
                emit({"pass": "inverse" if inverse else "forward", "op": name, "D": D, "rows": R,
                      "ours_ms": round(t_ours, 4), "eager_ms": round(t_ref, 4), "speedup": round(t_ref / t_ours, 2),
                      "bytes": nbytes, "ours_GBps": round(nbytes / (t_ours * 1e-3) / 1e9, 1),
                      "frac_copy_peak": round(nbytes / (t_ours * 1e-3) / 1e9 / peak, 3), "copy_GBps": round(peak, 1),
                      "max_rel_diff_vs_eager": max(rel(a[0], b[0]), rel(a[1], b[1]))})
                del a, b
            x = inputs(name, False, R, D, g, dev)
            gy = torch.randn(R, D, generator=g, device=dev)
            gl = torch.randn(R, generator=g, device=dev)
            for want_t in ((False, True) if tp is not None else (False,)):
                xg = x.clone().requires_grad_(True)
                tg = T.clone().requires_grad_(want_t)
                y, lad = eager(name, xg, False, tg)
                wrt = (xg, tg) if want_t else (xg,)
                outs = [(t, g_) for t, g_ in ((y, gy), (lad, gl)) if t.requires_grad]  # LeakyReLU: constant log-det
                ours = lambda: ops.pointwise_layer_backward(x, tp, gy, gl, op, False, 1e-2, 1e-6, want_t)  # noqa: E731
                ref = lambda: torch.autograd.grad([t for t, _ in outs], wrt, [g_ for _, g_ in outs],
                                                    retain_graph=True)  # noqa: E731
                t_ours, t_ref = timed_pair(ours, ref, args.iters)
                a, b = ours(), ref()
                nbytes = 12 * R * D + 4 * R
                emit({"pass": "backward_T" if want_t else "backward", "op": name, "D": D, "rows": R,
                      "ours_ms": round(t_ours, 4), "eager_ms": round(t_ref, 4), "speedup": round(t_ref / t_ours, 2),
                      "bytes": nbytes, "ours_GBps": round(nbytes / (t_ours * 1e-3) / 1e9, 1),
                      "frac_copy_peak": round(nbytes / (t_ours * 1e-3) / 1e9 / peak, 3), "copy_GBps": round(peak, 1),
                      "max_rel_diff_vs_eager": rel(a[0], b[0])})
                del xg, tg, y, lad, outs, a, b
            del x, gy, gl
        torch.cuda.empty_cache()
    for rec in workload_shares(dev, 5):
        emit(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        for rec in lines:
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
