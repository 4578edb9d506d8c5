"""LULinear on the GPU: fc_lulinear against the cuBLAS composition it replaces, per layer and inside a neural spline flow.

    python scripts/bench_lulinear.py [--rows 4194304] [--iters 20] [--out lines.jsonl]

Per D in {2, 8, 16, 32, 48, 63}, 4 M rows, one LULinear layer (trained-like entries), alternating in the same run:
  forward   layer(x)                       vs  F.linear(x, M, c) + the log-det fill (ld * ones(B))
  inverse   layer.inverse(x)               vs  the same with the inverse operands
  backward  ops.lulinear_layer_backward    vs  gy @ M, gy^T @ x, gy.sum(0)
Every timed pass is preceded by overwriting a 256 MB buffer, so that x is read from HBM, not from the 126 MB L2.  Times are
CUDA events around the call alone.  Bytes: the algorithmic traffic (x and y, plus 4 B of log-det per row; backward x, grad_y
and grad_x), reported against a device-to-device copy measured in the same run.  Then nsf_lu (D = 32, 8 RQ couplings each
followed by an LULinear, 1 M rows): log_prob, sample and one Adam training step, with the device time of the LU kernels
(launch events of fc_lulinear_apply / fc_lulinear_backward) as a share of each.  One JSON line per result.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
from torch.nn import functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, ops, transforms, workloads  # noqa: E402

DS = [2, 8, 16, 32, 48, 63]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit": power}


class Timer:
    def __init__(self, flush):
        self.flush = flush

    def __call__(self, fn):
        self.flush.add_(1.0)  # evicts the operands from L2
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        return a, b


def alternate(timer, fns, iters, warmup=3):
    """Median ms of each callable, the callables interleaved in every round."""
    for _ in range(warmup):
        for fn in fns.values():
            fn()
    events = {k: [] for k in fns}
    for _ in range(iters):
        for k, fn in fns.items():
            events[k].append(timer(fn))
    torch.cuda.synchronize()
    out = {}
    for k, ev in events.items():
        ts = sorted(a.elapsed_time(b) for a, b in ev)
        out[k] = ts[len(ts) // 2]
    return out


def copy_peak(timer, iters):
    src = torch.empty(1 << 28, device="cuda")  # 1 GB
    dst = torch.empty_like(src)
    ms = alternate(timer, {"copy": lambda: dst.copy_(src)}, iters)["copy"]
    return 2 * src.numel() * 4 / (ms * 1e-3) / 1e9


def layer_bench(D, rows, timer, iters, peak, emit):
    torch.manual_seed(D)
    layer = transforms.LULinear(D, identity_init=False).cuda()
    with torch.no_grad():
        for p in layer.parameters():
            p.uniform_(-D ** -0.5, D ** -0.5)
    x = torch.randn(rows, D, device="cuda")
    gy = torch.randn(rows, D, device="cuda")
    with torch.no_grad():
        for direction, inverse in (("forward", False), ("inverse", True)):
            M, c, ld = layer._operands(inverse)
            call = layer.inverse if inverse else layer.forward
            ours, lo = call(x)
            ref = F.linear(x, M, c)
            diff = (ours - ref).abs().max().item() / max(1.0, ref.abs().max().item())
            ms = alternate(timer, {"kernel": lambda: call(x),
                                   "cublas": lambda: (F.linear(x, M, c), ld * x.new_ones(rows))}, iters)
            nbytes = rows * D * 8 + rows * 4
            emit({"bench": "lulinear_layer", "direction": direction, "D": D, "rows": rows, "kernel_ms": ms["kernel"],
                  "cublas_ms": ms["cublas"], "speedup": ms["cublas"] / ms["kernel"],
                  "kernel_GBps": nbytes / (ms["kernel"] * 1e-3) / 1e9, "cublas_GBps": nbytes / (ms["cublas"] * 1e-3) / 1e9,
                  "kernel_of_copy_peak": nbytes / (ms["kernel"] * 1e-3) / 1e9 / peak,
                  "flop_per_byte": 2.0 * rows * D * D / nbytes, "max_rel_diff_vs_cublas": diff})
        M = torch.randn(D, D, device="cuda") * D ** -0.5
        gx, gM, gc = ops.lulinear_layer_backward(x, M, gy)
        diff = max((gx - gy @ M).abs().max().item() / max(1.0, gx.abs().max().item()),
                   (gM - gy.t() @ x).abs().max().item() / max(1.0, gM.abs().max().item()),
                   (gc - gy.sum(0)).abs().max().item() / max(1.0, gc.abs().max().item()))
        ms = alternate(timer, {"kernel": lambda: ops.lulinear_layer_backward(x, M, gy),
                               "cublas": lambda: (torch.mm(gy, M), torch.mm(gy.t(), x), gy.sum(0))}, iters)
        nbytes = rows * D * 12
        emit({"bench": "lulinear_layer", "direction": "backward", "D": D, "rows": rows, "kernel_ms": ms["kernel"],
              "cublas_ms": ms["cublas"], "speedup": ms["cublas"] / ms["kernel"],
              "kernel_GBps": nbytes / (ms["kernel"] * 1e-3) / 1e9, "cublas_GBps": nbytes / (ms["cublas"] * 1e-3) / 1e9,
              "kernel_of_copy_peak": nbytes / (ms["kernel"] * 1e-3) / 1e9 / peak,
              "flop_per_byte": 4.0 * rows * D * D / nbytes, "max_rel_diff_vs_cublas": diff})


def flow_bench(timer, iters, emit):
    wl = workloads.get_workload("nsf_lu")
    flow = workloads.build_flow(wl)
    flow.load_state_dict(workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl))
    flow = flow.cuda()
    rows = wl["batch"]
    x = torch.randn(rows, wl["features"], device="cuda")
    opt = torch.optim.Adam(flow.parameters(), lr=1e-5)

    def train_step():
        opt.zero_grad(set_to_none=True)
        (-flow.log_prob(x).mean()).backward()
        opt.step()

    def no_grad(fn):
        def run():
            with torch.no_grad():
                fn()
        return run

    calls = {"log_prob": no_grad(lambda: flow.log_prob(x)), "sample": no_grad(lambda: flow._transform.inverse(x)),
             "train_step": train_step}
    for name, fn in calls.items():
        ms = alternate(timer, {name: fn}, iters)[name]
        _cabi.STATS.reset()
        _cabi.STATS.timing = True
        fn()
        torch.cuda.synchronize()
        _cabi.STATS.timing = False
        lu_ms = sum(_cabi.STATS.elapsed_ms(k)[1] for k in ("fc_lulinear_apply", "fc_lulinear_backward"))
        emit({"bench": "nsf_lu", "call": name, "rows": rows, "features": wl["features"], "ms": ms,
              "rows_per_s": rows / (ms * 1e-3), "lu_kernel_ms": lu_ms, "lu_share": lu_ms / ms,
              "lu_launches": sum(_cabi.STATS.counts.get(k, 0) for k in ("fc_lulinear_apply", "fc_lulinear_backward"))})


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=1 << 22)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lulinear.py needs a CUDA device")
    out = open(args.out, "a") if args.out else None

    def emit(d):
        d.update(info)
        line = json.dumps(d)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    info = card()
    timer = Timer(torch.empty(1 << 26, device="cuda"))  # 256 MB
    peak = copy_peak(timer, args.iters)
    emit({"bench": "copy_peak", "GBps": peak})
    for D in DS:
        layer_bench(D, args.rows, timer, args.iters, peak, emit)
    flow_bench(timer, max(3, args.iters // 4), emit)
    if out:
        out.close()


if __name__ == "__main__":
    main()
