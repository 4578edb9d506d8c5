"""A/B of conditional flows (coupling / MAF conditioners with `context_features`): the fused conditioner kernel with
precomputed context terms against the path these flows took before it (torch modules + element-wise kernels,
`tensorcore.ENABLED = False`), alternated in one process.

Workloads (inference, trained-like weights, random context):
  cfg 2 shapes (8 PRQ coupling layers, D = 64, H = 256, K = 8) with C = 16 and C = 96: log_prob and sampling at 2^20 rows
  cfg 3 shapes (5 masked PRQ layers, D = 16, K = 16, H = 256) with C = 8: log_prob at 262 144 rows, sampling at 32 768
"Sampling" times the inverse cascade on fixed noise (Flow._sample without the noise draw), so both paths see the same
inputs.  Per call: CUDA-event time (mean of the rounds), the per-launch device time of every C-ABI kernel of the new path
(`_cabi.STATS.timing`, a separate pass), max |new - old| and parity of both against the fp64 oracle on 512 rows.  The
same shapes without a context give the reference time of the context-free conditioner kernel.

    python scripts/bench_context.py --out profiles/r03_context_ab.jsonl
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, workloads  # noqa: E402
from flowconductor_b200.nn import tensorcore  # noqa: E402
from oracle import restated  # noqa: E402
from tests.helpers import assert_parity  # noqa: E402


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip()
        lim, sm, smax = [v.strip() for v in q.split(",")]
        info.update(power_limit_w=float(lim), sm_mhz=int(sm), sm_max_mhz=int(smax))
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = "unavailable: {}".format(e)
    return info


def build(name, C):
    wl = workloads.get_workload(name)
    wl["context_features"] = C
    flow = workloads.build_flow(wl)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    g = torch.Generator().manual_seed(7)
    for k in state:  # context layers and second block layers away from their (near-identity) initialisation
        if "context_layer" in k or "linear_layers.1" in k:
            fan = state[k].shape[-1]
            state[k] = torch.randn(state[k].shape, generator=g) * (1.0 / math.sqrt(fan) if state[k].dim() == 2 else 0.3)
    flow.load_state_dict(state)
    return wl, flow.cuda().eval()


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def launches(fn):
    """{entry point: [launches, mean device ms per launch]} of one call."""
    _cabi.STATS.reset()
    _cabi.STATS.timing = True
    try:
        fn()
        torch.cuda.synchronize()
        out = {}
        for name in _cabi.STATS.counts:
            n, ms = _cabi.STATS.elapsed_ms(name)
            out[name] = [n, round(ms / max(n, 1), 4)]
        return out
    finally:
        _cabi.STATS.timing = False
        _cabi.STATS.reset()


def parity(ours, o32, o64):
    try:
        assert_parity(ours, o32, o64, 1e-5, 1.0, "bench", max_ratio=30.0)
        ok = True
    except AssertionError:
        ok = False
    d = (ours.double().cpu() - o64).abs()
    return {"parity_ok": ok, "max_abs_vs_fp64": float(d.max()), "max_abs_oracle32_vs_fp64": float((o32.double() - o64).abs().max())}


def run_case(name, C, direction, rows, rounds, reps):
    wl, flow = build(name, C)
    D = wl["features"]
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(rows, D, generator=g, device="cuda")
    ctx = torch.randn(rows, C, generator=g, device="cuda") if C else None
    if direction == "log_prob":
        fn = lambda: flow.log_prob(x, context=ctx)  # noqa: E731
    else:
        fn = lambda: flow._transform.inverse(x, context=ctx)[0]  # noqa: E731
    out = {"workload": name, "context_features": C, "call": direction, "rows": rows}
    times = {"new": [], "old": []}
    results = {}
    with torch.no_grad():
        for enabled in (True, False):  # warm-up (packing, kernel attributes, allocator)
            tensorcore.ENABLED = enabled
            results["new" if enabled else "old"] = fn()
            fn()
        torch.cuda.synchronize()
        for _ in range(rounds):
            for enabled in (True, False):
                tensorcore.ENABLED = enabled
                times["new" if enabled else "old"].append(timed(fn, reps))
        tensorcore.ENABLED = True
        out["launches_new"] = launches(fn)
    tensorcore.ENABLED = True
    out["new_ms"] = round(sum(times["new"]) / rounds, 3)
    out["old_ms"] = round(sum(times["old"]) / rounds, 3)
    out["new_ms_rounds"] = [round(t, 3) for t in times["new"]]
    out["old_ms_rounds"] = [round(t, 3) for t in times["old"]]
    out["speedup"] = round(out["old_ms"] / out["new_ms"], 3)
    new, old = results["new"], results["old"]
    out["max_abs_new_minus_old"] = float((new - old).abs().max())
    sample = torch.cat([torch.arange(256), torch.arange(rows - 256, rows)])
    specs = workloads.oracle_specs(wl)
    state = {k: v.cpu() for k, v in flow.state_dict().items()}
    state64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    xs = x[sample.cuda()].cpu()
    cs = ctx[sample.cuda()].cpu() if C else None
    with torch.no_grad():
        if direction == "log_prob":
            o32 = restated.flow_log_prob(state, specs, xs, cs)
            o64 = restated.flow_log_prob(state64, specs, xs.double(), cs.double() if C else None)
        else:
            o32 = restated.flow_sample_from_noise(state, specs, xs, cs)
            o64 = restated.flow_sample_from_noise(state64, specs, xs.double(), cs.double() if C else None)
    out["new_vs_oracle"] = parity(new[sample.cuda()], o32, o64)
    out["old_vs_oracle"] = parity(old[sample.cuda()], o32, o64)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSONL file to append to (default: stdout only)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small row counts (a functional rehearsal, not a measurement)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_context.py measures on the GPU"
    info = gpu_info()
    q = 1 / 64 if args.quick else 1
    cases = [("cfg2", 16, "log_prob", 1 << 20), ("cfg2", 16, "sample", 1 << 20),
             ("cfg2", 96, "log_prob", 1 << 20), ("cfg2", 96, "sample", 1 << 20),
             ("cfg3", 8, "log_prob", 262144), ("cfg3", 8, "sample", 32768)]
    lines = []
    for name, C, direction, rows in cases:
        res = run_case(name, C, direction, max(512, int(rows * q)), args.rounds, args.reps)
        res.update(info)
        lines.append(res)
        print(json.dumps(res), flush=True)
    # the context-free conditioner kernel at the same shape: per-launch time for the C = 16 / no-context ratio
    for C in (None,):
        wl, flow = build("cfg2", C)
        x = torch.randn(max(512, int((1 << 20) * q)), 64, device="cuda")
        with torch.no_grad():
            flow.log_prob(x)
            res = {"workload": "cfg2", "context_features": None, "call": "log_prob", "rows": x.shape[0],
                   "launches_new": launches(lambda: flow.log_prob(x))}
        res.update(info)
        lines.append(res)
        print(json.dumps(res), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for res in lines:
                f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
