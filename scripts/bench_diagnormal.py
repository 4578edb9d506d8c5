"""Time the diagonal-Gaussian base density kernels (csrc/fc_diagnormal.cu) against the reference's eager torch
composition (flowcon/distributions/normal.py) on the same GPU, at 4 M rows.

Passes, for D in {2, 6, 32, 64, 256}:
  log_prob        conditional log-density (G = 1, parameters = an encoder output [R, 2D])
  log_prob_bwd    its backward: grad_x and grad_params [R, 2D]
  shared_bwd      backward with one shared parameter row (DiagonalNormal, G = R): grad_x and the ordered column sums
  sample          n = 1 and n = 1024 draws per context row (R / n context rows)
  sample_bwd      its backward: grad_params [R / n, 2D] (n = 1024: group sums)
Every pass reports its time, the eager composition's time, the bytes it has to move (computed from the shapes below)
and that rate as a fraction of the device-to-device copy rate measured in the same run (`copy_GBps`), with the GPU's
name and power limit.  The L2 is overwritten before every timed call (medians of --iters calls), so every pass streams
from HBM.

    python scripts/bench_diagnormal.py --out profiles/r07_diagnormal_bench.jsonl
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import ops  # noqa: E402

ROWS = 1 << 22
DS = [2, 6, 32, 64, 256]


_FLUSH = []


def timed(fn, iters, flush=True):
    """Median ms of `iters` calls, each after overwriting the L2 with a 256 MB buffer (so it streams from HBM)."""
    if flush and not _FLUSH:
        _FLUSH.append(torch.empty(1 << 26, dtype=torch.float32, device="cuda"))
    for _ in range(3):
        fn()
    times = []
    for _ in range(iters):
        if flush:
            _FLUSH[0].zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def copy_peak(dev, iters):
    src = torch.empty(1 << 28, dtype=torch.float32, device=dev)  # 1 GB
    dst = torch.empty_like(src)
    ms = timed(lambda: dst.copy_(src), iters, flush=False)
    return 2 * src.numel() * 4 / (ms * 1e-3) / 1e9


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def eager_log_prob(x, params, D):
    means, log_stds = params[..., :D], params[..., D:]
    norm = (x - means) * torch.exp(-log_stds)
    lp = -0.5 * torch.sum(norm ** 2, dim=1)
    lp = lp - torch.sum(log_stds, dim=1)
    return lp - 0.5 * D * math.log(2 * math.pi)


def eager_sample(noise, params, D, n):
    means, stds = params[:, :D], torch.exp(params[:, D:])
    return torch.repeat_interleave(means, n, dim=0) + torch.repeat_interleave(stds, n, dim=0) * noise


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07_diagnormal_bench.jsonl")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rows", type=int, default=ROWS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_diagnormal needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu, watts = torch.cuda.get_device_name(dev), power_limit()
    peak = copy_peak(dev, args.iters)
    R, f = args.rows, 4
    lines = []

    def emit(name, D, n, ours_ms, eager_ms, nbytes, check):
        rec = {"pass": name, "D": D, "rows": R, "n": n, "ours_ms": round(ours_ms, 4), "eager_ms": round(eager_ms, 4),
               "speedup": round(eager_ms / ours_ms, 2), "bytes": nbytes,
               "ours_GBps": round(nbytes / (ours_ms * 1e-3) / 1e9, 1),
               "frac_copy_peak": round(nbytes / (ours_ms * 1e-3) / 1e9 / peak, 3), "copy_GBps": round(peak, 1),
               "max_rel_diff_vs_eager": check, "gpu": gpu, "power_limit_w": watts}
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    def rel(a, b):
        return float(((a - b).abs() / b.abs().clamp_min(1.0)).max())

    for D in DS:
        g = torch.Generator(device=dev).manual_seed(D)
        x = torch.randn(R, D, generator=g, device=dev)
        params = torch.randn(R, 2 * D, generator=g, device=dev) * 0.3
        w = torch.randn(R, generator=g, device=dev)
        ours = lambda: ops.diagnormal_log_prob(x, params, 1, None)  # noqa: E731
        eager = lambda: eager_log_prob(x, params, D)  # noqa: E731
        emit("log_prob", D, 1, timed(ours, args.iters), timed(eager, args.iters), f * R * (3 * D + 1),
             rel(ours(), eager()))

        xg, pg = x.clone().requires_grad_(True), params.clone().requires_grad_(True)
        lp = eager_log_prob(xg, pg, D)
        ours = lambda: ops.diagnormal_log_prob_backward(x, params, 1, w)  # noqa: E731
        eager = lambda: torch.autograd.grad(lp, (xg, pg), w, retain_graph=True)  # noqa: E731
        a, b = ours(), eager()
        emit("log_prob_bwd", D, 1, timed(ours, args.iters), timed(eager, args.iters), f * R * (6 * D + 1),
             max(rel(a[0], b[0]), rel(a[1], b[1])))
        del lp, xg, pg, a, b

        shared = params[:1].clone()
        sg = shared.clone().requires_grad_(True)
        xg = x.clone().requires_grad_(True)
        lp = eager_log_prob(xg, sg, D)
        ours = lambda: ops.diagnormal_log_prob_backward(x, shared, R, w)  # noqa: E731
        eager = lambda: torch.autograd.grad(lp, (xg, sg), w, retain_graph=True)  # noqa: E731
        a, b = ours(), eager()
        emit("shared_bwd", D, R, timed(ours, args.iters), timed(eager, args.iters), f * R * (2 * D + 1),
             rel(a[0], b[0]))
        del lp, xg, sg, a, b

        for n in (1, 1024):
            C = R // n
            p = params[:C].contiguous()
            ours = lambda: ops.diagnormal_sample(x, p, n)  # noqa: E731
            eager = lambda: eager_sample(x, p, D, n)  # noqa: E731
            emit("sample", D, n, timed(ours, args.iters), timed(eager, args.iters), f * (2 * R * D + 2 * C * D),
                 rel(ours(), eager()))
            pg = p.clone().requires_grad_(True)
            y = eager_sample(x, pg, D, n)
            gy = torch.randn(R, D, generator=g, device=dev)
            ours = lambda: ops.diagnormal_sample_backward(x, p, n, gy)  # noqa: E731
            eager = lambda: torch.autograd.grad(y, (pg,), gy, retain_graph=True)  # noqa: E731
            a, b = ours(), eager()[0]
            emit("sample_bwd", D, n, timed(ours, args.iters), timed(eager, args.iters), f * (2 * R * D + 4 * C * D),
                 rel(a, b))
            del pg, y, gy, a, b
        del x, params, w
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        for rec in lines:
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
