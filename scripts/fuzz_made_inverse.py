#!/usr/bin/env python
"""Random-shape stress of the incremental autoregressive inverse (csrc/fc_made_inverse.cuh) against the D-pass path:
features 1..48, hidden 4..256, 1..3 blocks, every autoregressive layer family, ragged batch sizes.

    python scripts/fuzz_made_inverse.py [seed] [cases] [context]

`context`: conditional MADEs instead (context width 1..80, 1..6 blocks); the nets the fused conditioner covers keep the
D-pass path and are counted as falling back."""
import os
import random
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, made_inverse, transforms  # noqa: E402
from oracle import restated  # noqa: E402  (checker only)


def oracle_inverse(layer, fam, z, blocks, ctx=None):
    """fp64 D-pass inverse of the reference algorithm with the layer's weights."""
    st = {k: (v.detach().cpu().double() if v.is_floating_point() else v.cpu()) for k, v in layer.state_dict().items()}
    spec = {"prefix": "", "num_blocks": blocks, "hidden_features": layer.autoregressive_net.initial_layer.weight.shape[0]}
    if fam in ("rqs", "rqs_none"):
        spec.update(kind="maf_prq", num_bins=layer.num_bins, tails=layer.tails, tail_bound=layer.tail_bound)
    elif fam == "affine":
        spec.update(kind="maf_affine")
    elif fam == "sos":
        spec.update(kind="maf_sos", n_sigmoids=layer.n_sigmoids)
    elif fam == "lin":
        spec.update(kind="maf_plin", num_bins=layer.num_bins, tails=None, tail_bound=1.0)
    elif fam == "quad":
        spec.update(kind="maf_pquad", num_bins=layer.num_bins, tails=layer.tails, tail_bound=layer.tail_bound)
    else:
        spec.update(kind="maf_pcubic", num_bins=layer.num_bins, tails=None, tail_bound=1.0)
    with torch.no_grad():
        ctx = None if ctx is None else ctx.detach().cpu().double()
        return restated.apply_layer(st, spec, z.detach().cpu().double(), ctx, inverse=True)

def main():
    dev = torch.device("cuda:0")
    random.seed(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
    n_cases = int(sys.argv[2]) if len(sys.argv) > 2 else 40
    conditional = len(sys.argv) > 3 and sys.argv[3] == "context"
    worst = 0.0
    ran = skipped = 0
    for case in range(n_cases):
        D = random.choice([1, 2, 3, 5, 8, 13, 16, 24, 33, 48])
        H = random.choice([4, 12, 32, 64, 100, 128, 256])
        blocks = random.choice([1, 2, 3])
        fam = random.choice(["rqs", "rqs_none", "affine", "sos", "lin", "quad", "cubic"])
        rows = random.choice([1, 31, 32, 33, 500, 4100])
        C = None
        if conditional:
            blocks = random.randint(1, 6)
            C = random.randint(1, 80)
        only = os.environ.get("FUZZ_ONLY")
        skip = only is not None and str(case) not in only.split(",")
        torch.manual_seed(case)
        if fam == "rqs":
            layer = transforms.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(
                D, H, num_bins=random.choice([4, 8, 10, 16]), tails="linear", tail_bound=3.0, num_blocks=blocks, context_features=C)
        elif fam == "rqs_none":
            layer = transforms.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(
                D, H, num_bins=random.choice([5, 8]), tails=None, num_blocks=blocks, context_features=C)
        elif fam == "affine":
            layer = transforms.MaskedAffineAutoregressiveTransform(D, H, num_blocks=blocks, context_features=C)
        elif fam == "sos":
            layer = transforms.MaskedSumOfSigmoidsTransform(D, H, n_sigmoids=random.choice([3, 10]), num_blocks=blocks,
                                                        context_features=C)
        elif fam == "lin":
            layer = transforms.MaskedPiecewiseLinearAutoregressiveTransform(random.choice([4, 8, 10]), D, H, num_blocks=blocks,
                                                                            context_features=C)
        elif fam == "quad":
            layer = transforms.MaskedPiecewiseQuadraticAutoregressiveTransform(
                D, H, num_bins=random.choice([4, 8]), tails=random.choice([None, "linear"]), tail_bound=3.0, num_blocks=blocks,
                context_features=C)
        else:
            layer = transforms.MaskedPiecewiseCubicAutoregressiveTransform(random.choice([4, 8]), D, H, num_blocks=blocks,
                                                                           context_features=C)
        if skip:
            continue
        layer = layer.to(dev).eval()
        unit_box = fam in ("lin", "cubic") or (fam == "quad" and layer.tails is None)
        with torch.no_grad():
            for p in layer.parameters():
                p.add_(torch.randn_like(p) * 0.05)
            if fam == "rqs_none":
                z = (torch.rand(rows, D, device=dev) * 2 - 1) * 1.15
            elif unit_box:
                z = torch.rand(rows, D, device=dev) * 0.98 + 0.01
            else:
                z = torch.randn(rows, D, device=dev)
            ctx = None if C is None else torch.randn(rows, C, device=dev)
            _cabi.STATS.reset()
            try:
                x, lad = layer.inverse(z, context=ctx)
                used = any(k.startswith("fc_made_inverse") for k in _cabi.STATS.counts)
                made_inverse.ENABLED = False
                xd, ladd = layer.inverse(z, context=ctx)
            except Exception as e:  # noqa: BLE001
                print("case %2d %-8s D=%2d H=%3d blocks=%d rows=%4d: %s raised %s: %s   <<<<<< MISMATCH" % (
                    case, fam, D, H, blocks, rows, "incremental" if made_inverse.ENABLED else "D-pass", type(e).__name__, e))
                made_inverse.ENABLED = True
                continue
            finally:
                made_inverse.ENABLED = True
        if not used:
            skipped += 1
            continue
        ran += 1
        ex = ((x - xd).abs() / xd.abs().clamp_min(1.0)).max().item()
        el = ((lad - ladd).abs() / ladd.abs().clamp_min(1.0)).max().item()
        worst = max(worst, ex, el)
        flag = "" if (ex < 2e-3 and el < 2e-2 and torch.isfinite(x).all()) else "   <<<<<< MISMATCH"
        print("case %2d %-8s D=%2d H=%3d blocks=%d C=%s rows=%4d: outputs %.2e logabsdet %.2e%s" % (
            case, fam, D, H, blocks, C, rows, ex, el, flag))
        if flag:
            xr, lr = oracle_inverse(layer, fam, z[:64], blocks, None if ctx is None else ctx[:64])
            print("        vs the fp64 oracle: incremental %.2e / %.2e, D-pass path %.2e / %.2e" % (
                (x[:64].cpu().double() - xr).abs().max(), (lad[:64].cpu().double() - lr).abs().max(),
                (xd[:64].cpu().double() - xr).abs().max(), (ladd[:64].cpu().double() - lr).abs().max()))
    print("ran %d (fell back to the D-pass path: %d), worst relative difference %.2e" % (ran, skipped, worst))


if __name__ == "__main__":
    main()
