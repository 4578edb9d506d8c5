"""Sampling from conditional masked autoregressive flows (`context_features`): the incremental MADE inverse with the
context prefill (csrc/fc_made_inverse.cuh, one term launch + one fc_made_inverse_* launch per layer) against the D-pass
inverse (`made_inverse.ENABLED = False`), alternated in one process on the same seeded inputs.

  1. a narrow conditional MAF stack (5 masked PRQ layers, D = 16, H = 48, K = 16, C = 8) — below the fused conditioner's
     widths, so the D-pass path runs the torch modules D times per layer — sampled (the inverse cascade on fixed noise)
     at 4096, 32 768 and 262 144 rows;
  2. one cfg 3-shape layer (D = 16, H = 256, K = 16, C = 8) at 32 768 rows: the conditional kernel against the same
     layer's context-free kernel (same weights, context layers dropped), and against the fused D-pass path
     (fc_conditioner_rqs_apply x D), which is what `layer.inverse` runs for this net.

Per case: CUDA-event time per call (mean over alternating rounds), the device time of each C-ABI launch of one call (a
separate pass with per-launch events), max |incremental - D-pass| and both against the fp64 oracle on 512 rows.  The
card name, power limit and SM clocks are read in the same run.

    python scripts/bench_made_inverse_context.py --out profiles/r04_made_inverse_context.jsonl
"""
import argparse
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, made_inverse, workloads  # noqa: E402
from flowconductor_b200.transforms import made as made_module  # noqa: E402
from oracle import restated  # noqa: E402
from scripts.bench_context import gpu_info, launches, timed  # noqa: E402
from tests.helpers import assert_parity  # noqa: E402


def _randomise_context(state, seed=7):
    """Context layers and second block layers away from their (near-identity) initialisation, so the terms matter (their
    weights and biases only: the masks and degrees are buffers under the same names)."""
    g = torch.Generator().manual_seed(seed)
    for k in state:
        if ("context_layer" in k or "linear_layers.1" in k) and k.endswith((".weight", ".bias")):
            fan = state[k].shape[-1]
            state[k] = torch.randn(state[k].shape, generator=g) * (1.0 / math.sqrt(fan) if state[k].dim() == 2 else 0.3)
    return state


def parity(ours, o32, o64, tol=1e-3):
    try:
        assert_parity(ours, o32, o64, tol, 1.0, "bench", max_ratio=30.0)
        ok = True
    except AssertionError:
        ok = False
    return {"parity_ok": ok, "max_abs_vs_fp64": float((ours.double().cpu() - o64).abs().max()),
            "max_abs_oracle32_vs_fp64": float((o32.double() - o64).abs().max())}


def alternate(fns, rounds, reps):
    """{name: mean ms per call} of the callables, alternated round by round."""
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            times[k].append(timed(fn, reps))
    return {k: round(sum(v) / len(v), 4) for k, v in times.items()}


def with_made_inverse(enabled, fn):
    def call():
        made_inverse.ENABLED = enabled
        try:
            return fn()
        finally:
            made_inverse.ENABLED = True
    return call


def narrow_stack(rows_list, rounds, reps):
    wl = {"name": "maf_narrow_ctx", "features": 16, "context_features": 8, "batch": 4096,
          "layers": workloads._maf_prq_stack(16, 5, 16, 48)}
    flow = workloads.build_flow(wl)
    state = _randomise_context(workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl))
    flow.load_state_dict(state)
    flow = flow.cuda().eval()
    specs = workloads.oracle_specs(wl)
    out = []
    for rows in rows_list:
        g = torch.Generator(device="cuda").manual_seed(rows)
        z = torch.randn(rows, 16, generator=g, device="cuda")
        ctx = torch.randn(rows, 8, generator=g, device="cuda")
        fn = lambda: flow._transform.inverse(z, context=ctx)  # noqa: E731
        fns = {"incremental": with_made_inverse(True, fn), "d_pass": with_made_inverse(False, fn)}
        with torch.no_grad():
            res = {k: f() for k, f in fns.items()}
            for f in fns.values():
                f()
            torch.cuda.synchronize()
            ms = alternate(fns, rounds, reps)
            rec = {"case": "narrow conditional MAF stack sampling", "layers": 5, "D": 16, "H": 48, "K": 16, "C": 8,
                   "rows": rows, "incremental_ms": ms["incremental"], "d_pass_ms": ms["d_pass"],
                   "speedup": round(ms["d_pass"] / ms["incremental"], 2),
                   "launches_incremental": launches(fns["incremental"]),
                   "launches_d_pass": launches(fns["d_pass"]),
                   "max_abs_incremental_vs_d_pass": float((res["incremental"][0] - res["d_pass"][0]).abs().max())}
        sel = torch.arange(min(rows, 512))
        cpu = {k: v.cpu() for k, v in flow.state_dict().items()}
        with torch.no_grad():
            o32, _ = restated.composite(cpu, specs, z[sel].cpu(), ctx[sel].cpu(), inverse=True)
            o64, _ = restated.composite({k: (v.double() if v.is_floating_point() else v) for k, v in cpu.items()}, specs,
                                        z[sel].cpu().double(), ctx[sel].cpu().double(), inverse=True)
        assert rec["launches_incremental"].get("fc_made_inverse_rqs", [0])[0] == 5, rec["launches_incremental"]
        rec["oracle_incremental"] = parity(res["incremental"][0][sel.cuda()], o32, o64)
        rec["oracle_d_pass"] = parity(res["d_pass"][0][sel.cuda()], o32, o64)
        out.append(rec)
        print(json.dumps(rec), flush=True)
    return out


def cfg3_layer(rows, rounds, reps):
    wl = {"name": "cfg3_layer_ctx", "features": 16, "context_features": 8, "batch": rows,
          "layers": [{"kind": "maf_prq", "num_bins": 16, "tails": "linear", "tail_bound": 3.0, "hidden_features": 256,
                      "num_blocks": 2}]}
    flow = workloads.build_flow(wl)
    state = _randomise_context(workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl))
    flow.load_state_dict(state)
    layer = flow._transform._transforms[0].cuda().eval()
    net = layer.autoregressive_net
    plain = made_module.MADE(16, 256, num_blocks=2, output_multiplier=net.final_layer.weight.shape[0] // 16)
    plain.load_state_dict({k: v for k, v in net.state_dict().items() if "context_layer" not in k})
    plain = plain.cuda().eval()
    P = layer._spline.params_per_feature()
    cfg, _ = layer._spline.config(True, None)
    g = torch.Generator(device="cuda").manual_seed(3)
    z = torch.randn(rows, 16, generator=g, device="cuda")
    ctx = torch.randn(rows, 8, generator=g, device="cuda")
    with torch.no_grad():
        prog, prog_plain = made_inverse.program_for(net, P), made_inverse.program_for(plain, P)
        assert prog is not None and prog_plain is not None
        fns = {"conditional_kernel": lambda: made_inverse.apply_rqs(prog, z, cfg, None, context=ctx),
               "context_free_kernel": lambda: made_inverse.apply_rqs(prog_plain, z, cfg),
               "fused_d_pass": lambda: layer.inverse(z, context=ctx)}
        res = {k: f() for k, f in fns.items()}
        for f in fns.values():
            f()
        torch.cuda.synchronize()
        ms = alternate(fns, rounds, reps)
        lc = launches(fns["conditional_kernel"])
        lp = launches(fns["context_free_kernel"])
        lf = launches(fns["fused_d_pass"])
    rec = {"case": "cfg3-shape conditional layer", "D": 16, "H": 256, "K": 16, "C": 8, "rows": rows,
           "call_ms": ms, "launches_conditional": lc, "launches_context_free": lp, "launches_fused_d_pass": lf,
           "kernel_ratio_conditional_over_context_free": round(lc["fc_made_inverse_rqs"][1] / lp["fc_made_inverse_rqs"][1],
                                                               4),
           "call_ratio_conditional_over_fused_d_pass": round(ms["conditional_kernel"] / ms["fused_d_pass"], 3),
           "max_abs_conditional_vs_fused_d_pass": float((res["conditional_kernel"][0] - res["fused_d_pass"][0]).abs().max())}
    sel = torch.cat((torch.arange(256), torch.arange(rows - 256, rows)))
    cpu = {k: v.cpu() for k, v in layer.state_dict().items()}
    spec = workloads.oracle_specs(wl)[0]
    spec = dict(spec, prefix="")
    with torch.no_grad():
        o32, _ = restated.apply_layer(cpu, spec, z[sel].cpu(), ctx[sel].cpu(), inverse=True)
        o64, _ = restated.apply_layer({k: (v.double() if v.is_floating_point() else v) for k, v in cpu.items()}, spec,
                                      z[sel].cpu().double(), ctx[sel].cpu().double(), inverse=True)
    rec["oracle_conditional_kernel"] = parity(res["conditional_kernel"][0][sel.cuda()], o32, o64)
    rec["oracle_fused_d_pass"] = parity(res["fused_d_pass"][0][sel.cuda()], o32, o64)
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rows", type=int, nargs="+", default=[4096, 32768, 262144])
    ap.add_argument("--cfg3-rows", type=int, default=32768)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_made_inverse_context.py measures the GPU kernels: no CUDA device found")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    recs = narrow_stack(args.rows, args.rounds, args.reps)
    recs.append(cfg3_layer(args.cfg3_rows, args.rounds, args.reps))
    if args.out:
        with open(args.out, "w") as f:
            for r in recs:
                f.write(json.dumps(dict(info, **r)) + "\n")


if __name__ == "__main__":
    main()
