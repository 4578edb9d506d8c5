"""BatchNorm on the GPU: the fc_batchnorm kernels against the eager composition they replace, per layer and inside a
masked autoregressive flow.

    python scripts/bench_batchnorm.py [--rows 4194304] [--iters 20] [--out lines.jsonl]

Per D in {6, 21, 43, 64, 256}, 4 M rows, one BatchNorm (trained-like weights and running statistics), alternating in the
same run with the eager torch composition of the reference's formulas:
  train_forward   ops.batchnorm_train (statistics + forward)          12 algorithmic bytes per element (x twice, y)
  eval_forward    ops.batchnorm_eval                                   8 (x, y)
  eval_inverse    ops.batchnorm_eval(inverse=True)                     8
  train_backward  ops.batchnorm_backward(BATCHNORM_TRAIN)             20 (x and grad_y twice, grad_x)
  eval_backward   ops.batchnorm_backward(BATCHNORM_EVAL_FORWARD)      12 (x, grad_y, grad_x)
The eager backward is autograd through the composition (torch.autograd.grad on a retained graph).  Every timed pass is
preceded by overwriting a 256 MB buffer, so that x is read from HBM, not from the 126 MB L2; medians of alternated passes;
the share of a device-to-device copy measured in the same run.  Then maf_bn (MAF-affine, D = 43, H = 256, 5 layers with
BatchNorm between them, 262 144 rows): one Adam training step, with the device time of the BatchNorm launches as a share
of it.  One JSON line per result, with the GPU name and power limit.
"""
import argparse
import json
import os
import sys

import torch
from torch.nn import functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, ops, workloads  # noqa: E402
from scripts.bench_lulinear import Timer, alternate, card, copy_peak  # noqa: E402

DS = [6, 21, 43, 64, 256]
EPS = 1e-5
BN_ENTRIES = ("fc_batchnorm_stats", "fc_batchnorm_apply", "fc_batchnorm_backward")


def eager_train(x, uw, bias):
    w = F.softplus(uw) + EPS
    mean, var = x.mean(0), x.var(0)
    y = w * ((x - mean) / torch.sqrt(var + EPS)) + bias
    return y, torch.sum(torch.log(w) - 0.5 * torch.log(var + EPS)) * x.new_ones(x.shape[0])


def eager_eval(x, rm, rv, uw, bias, inverse):
    w = F.softplus(uw) + EPS
    if inverse:
        y = torch.sqrt(rv + EPS) * ((x - bias) / w) + rm
        return y, torch.sum(-torch.log(w) + 0.5 * torch.log(rv + EPS)) * x.new_ones(x.shape[0])
    y = w * ((x - rm) / torch.sqrt(rv + EPS)) + bias
    return y, torch.sum(torch.log(w) - 0.5 * torch.log(rv + EPS)) * x.new_ones(x.shape[0])


def rel_diff(a, b):
    return (a - b).abs().max().item() / max(1.0, b.abs().max().item())


def layer_bench(D, rows, timer, iters, peak, emit):
    g = torch.Generator(device="cuda").manual_seed(D)
    x = 3.0 + torch.randn(rows, D, device="cuda", generator=g)
    gy = torch.randn(rows, D, device="cuda", generator=g)
    gl = torch.randn(rows, device="cuda", generator=g)
    uw = 0.4 * torch.randn(D, device="cuda", generator=g)
    bias = 0.5 * torch.randn(D, device="cuda", generator=g)
    rm = 3.0 + 0.1 * torch.randn(D, device="cuda", generator=g)
    rv = torch.exp(0.3 * torch.randn(D, device="cuda", generator=g))

    def record(call, nbytes, ms, diff):
        gbps = nbytes / (ms["kernel"] * 1e-3) / 1e9
        emit({"bench": "batchnorm_layer", "call": call, "D": D, "rows": rows, "kernel_ms": ms["kernel"],
              "eager_ms": ms["eager"], "speedup": ms["eager"] / ms["kernel"], "bytes_per_element": nbytes // (rows * D),
              "kernel_GBps": gbps, "kernel_of_copy_peak": gbps / peak, "max_rel_diff_vs_eager": diff})

    with torch.no_grad():
        ours, ref = ops.batchnorm_train(x, uw, bias, EPS), eager_train(x, uw, bias)
        ms = alternate(timer, {"kernel": lambda: ops.batchnorm_train(x, uw, bias, EPS),
                               "eager": lambda: eager_train(x, uw, bias)}, iters)
        record("train_forward", 12 * rows * D, ms, rel_diff(ours[0], ref[0]))
        for call, inverse in (("eval_forward", False), ("eval_inverse", True)):
            ours = ops.batchnorm_eval(x, rm, rv, uw, bias, EPS, inverse)
            ref = eager_eval(x, rm, rv, uw, bias, inverse)
            ms = alternate(timer, {"kernel": lambda: ops.batchnorm_eval(x, rm, rv, uw, bias, EPS, inverse),
                                   "eager": lambda: eager_eval(x, rm, rv, uw, bias, inverse)}, iters)
            record(call, 8 * rows * D, ms, rel_diff(ours[0], ref[0]))
    _, _, mean, var = ops.batchnorm_train(x, uw, bias, EPS)
    for call, mode in (("train_backward", _cabi.BATCHNORM_TRAIN), ("eval_backward", _cabi.BATCHNORM_EVAL_FORWARD)):
        xr, uwr, br = (t.detach().clone().requires_grad_(True) for t in (x, uw, bias))
        y, lad = eager_train(xr, uwr, br) if mode == _cabi.BATCHNORM_TRAIN else eager_eval(xr, rm, rv, uwr, br, False)
        ref = torch.autograd.grad((y, lad), (xr, uwr, br), (gy, gl), retain_graph=True)
        stats = (mean, var) if mode == _cabi.BATCHNORM_TRAIN else (rm, rv)
        ours = ops.batchnorm_backward(x, *stats, uw, bias, EPS, gy, gl, mode)
        diff = max(rel_diff(a, b) for a, b in zip(ours, ref))
        ms = alternate(timer, {"kernel": lambda: ops.batchnorm_backward(x, *stats, uw, bias, EPS, gy, gl, mode),
                               "eager": lambda: torch.autograd.grad((y, lad), (xr, uwr, br), (gy, gl),
                                                                    retain_graph=True)}, iters)
        record(call, (20 if mode == _cabi.BATCHNORM_TRAIN else 12) * rows * D, ms, diff)
        del y, lad


def flow_bench(timer, iters, emit):
    wl = workloads.get_workload("maf_bn")
    flow = workloads.build_flow(wl)
    flow.load_state_dict(workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl))
    flow = flow.cuda().train()
    rows = wl["batch"]
    x = torch.randn(rows, wl["features"], device="cuda")
    opt = torch.optim.Adam(flow.parameters(), lr=1e-5)

    def train_step():
        opt.zero_grad(set_to_none=True)
        (-flow.log_prob(x).mean()).backward()
        opt.step()

    ms = alternate(timer, {"train_step": train_step}, iters)["train_step"]
    _cabi.STATS.reset()
    _cabi.STATS.timing = True
    train_step()
    torch.cuda.synchronize()
    _cabi.STATS.timing = False
    bn_ms = sum(_cabi.STATS.elapsed_ms(k)[1] for k in BN_ENTRIES)
    emit({"bench": "maf_bn", "call": "train_step", "rows": rows, "features": wl["features"], "ms": ms,
          "rows_per_s": rows / (ms * 1e-3), "bn_kernel_ms": bn_ms, "bn_share": bn_ms / ms,
          "bn_launches": {k: _cabi.STATS.counts.get(k, 0) for k in BN_ENTRIES}})


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=1 << 22)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_batchnorm.py needs a CUDA device")
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
