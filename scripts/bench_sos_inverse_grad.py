#!/usr/bin/env python
"""Gradients through the numerical sum-of-sigmoids inverse, measured at cfg 4 shapes (262 144 rows x 32 features,
n = 10 sigmoids).

* kernel: the forward adjoint (fc_sos_backward) and the inverse adjoint (fc_sos_inverse_backward), timed alternately
  with CUDA events on a working set above the L2 (params and their gradient are 1 GB each).  Bytes as in
  scripts/bench_kernels.py, B (8 D P + 12 D + 4); the copy peak is a device-to-device copy measured in the same run.
* end to end: one reverse-KL step (Flow.sample_and_log_prob + backward) of the cfg 4 flow, against the same step computed
  by the reference algorithm (oracle/restated.py: eager fp32, bisection + autograd Newton inverse) on the same GPU.

Writes one JSON line per measurement to --out, each with the GPU name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from flowconductor_b200 import ops, workloads  # noqa: E402
from oracle import restated  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
    except Exception:  # the power limit is then reported as unknown, never guessed
        name, power = torch.cuda.get_device_name(0), None
    return {"gpu": name, "power_limit": power}


def events(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def median(ts):
    ts = sorted(ts)
    return ts[len(ts) // 2]


def copy_peak_gbs(dev, reps):
    src = torch.empty(1 << 29, device=dev)  # 2 GiB
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    ms = median([events(lambda: dst.copy_(src)) for _ in range(reps)])
    return 2 * src.numel() * 4 / ms / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=262144)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--ref-steps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_sos_inverse_grad.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("this benchmark needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    records = []

    def emit(rec):
        rec = dict(rec, **info)
        records.append(rec)
        print(json.dumps(rec), flush=True)

    peak = copy_peak_gbs(dev, args.reps)
    emit({"what": "device-to-device copy", "GB/s": peak})

    B, D, n = args.rows, 32, 10
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(B, D, generator=g, device=dev)
    p = torch.randn(B, D * (3 * n + 1), generator=g, device=dev) * 2
    gy, gl = torch.randn(B, D, generator=g, device=dev), torch.randn(B, generator=g, device=dev)
    nbytes = B * (8 * D * (3 * n + 1) + 12 * D + 4)
    kernels = {"fc_sos_backward": lambda: ops.sos_layer_backward(x, p, gy, gl, n),
               "fc_sos_inverse_backward": lambda: ops.sos_layer_inverse_backward(x, p, gy, gl, n)}
    for fn in kernels.values():
        for _ in range(5):
            fn()
    times = {k: [] for k in kernels}
    for _ in range(args.reps):
        for k, fn in kernels.items():
            times[k].append(events(fn))
    for k, ts in times.items():
        ms = median(ts)
        emit({"what": "kernel " + k, "rows": B, "D": D, "n_sigmoids": n, "ms_median": ms, "ms_best": min(ts),
              "bytes": nbytes, "GB/s": nbytes / ms / 1e6, "frac_of_copy_peak": nbytes / ms / 1e6 / peak})
    ratio = median(times["fc_sos_inverse_backward"]) / median(times["fc_sos_backward"])
    emit({"what": "inverse adjoint / forward adjoint", "ratio": ratio})
    del x, p, gy, gl

    # end to end: one reverse-KL step of the cfg 4 flow against a standard-normal target
    wl = workloads.get_workload("cfg4")
    flow = workloads.build_flow(wl, seed=0).to(dev)
    ctx = torch.randn(B, wl["context_features"], generator=g, device=dev)

    def target_log_prob(t):
        return -0.5 * (t.reshape(-1, D) ** 2).sum(-1)

    def ours():
        flow.zero_grad(set_to_none=True)
        xs, lq = flow.sample_and_log_prob(1, context=ctx)
        loss = (lq.reshape(-1) - target_log_prob(xs)).mean()
        loss.backward()
        return loss

    state = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in flow.state_dict().items()}
    specs = workloads.oracle_specs(wl)

    def reference():
        for v in state.values():
            v.grad = None
        noise = torch.randn(B, D, device=dev)
        xr, ladr = restated.composite(state, specs, noise, ctx, inverse=True)
        loss = (restated.standard_normal_log_prob(noise) - ladr - target_log_prob(xr)).mean()
        loss.backward()
        return loss

    torch.cuda.reset_peak_memory_stats(dev)
    for name, fn, steps in (("flowconductor_b200", ours, args.steps), ("reference algorithm", reference, args.ref_steps)):
        fn()
        ts = []
        for _ in range(steps):
            out = {}
            ts.append(events(lambda: out.update(loss=fn())))
        emit({"what": "reverse-KL step cfg4 (sample_and_log_prob + backward)", "impl": name, "rows": B,
              "ms_median": median(ts), "ms_best": min(ts), "steps": steps, "loss": float(out["loss"]),
              "peak_mem_GB": torch.cuda.max_memory_allocated(dev) / 1e9})
        torch.cuda.reset_peak_memory_stats(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in records:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
