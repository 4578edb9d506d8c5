"""GPU bring-up check + micro-benchmark of the tensor-core linear kernels (fc_linear_apply / fc_linear_rqs_apply).

    python scripts/check_linear.py [--bench]

Compares against fp64 torch matmul (and the fp32 cuBLAS result for scale), then the fused spline epilogue against
fc_linear_apply -> fc_rqs_apply on the same packed weights.
"""
import argparse
import math
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, linear as fl, ops  # noqa: E402


def rel_err(got, want64):
    scale = want64.abs().max().item()
    return (got.double() - want64).abs().max().item() / scale


def check_store(M, K, N, relu_in, relu_out, use_res, gen, dev, a_t128=False, o_t128=False):
    a = torch.randn(M, K, generator=gen, device=dev)
    w = torch.randn(N, K, generator=gen, device=dev) / math.sqrt(K)
    b = torch.randn(N, generator=gen, device=dev)
    res = torch.randn(M, N, generator=gen, device=dev) if use_res else None
    pk = fl.pack(w, b)
    a_in = fl.T128.from_rows(a) if a_t128 else a
    res_in = fl.T128.from_rows(res) if (o_t128 and use_res) else res
    out = fl.linear(a_in, pk, relu_in=relu_in, relu_out=relu_out, residual=res_in, out_t128=o_t128)
    if o_t128:
        out = out.to_rows()
    torch.cuda.synchronize()
    a64 = a.double().relu() if relu_in else a.double()
    want = a64 @ w.double().t() + b.double()
    if use_res:
        want = want + res.double()
    if relu_out:
        want = want.relu()
    a32 = a.relu() if relu_in else a
    ref32 = torch.nn.functional.linear(a32, w, b)
    if use_res:
        ref32 = ref32 + res
    if relu_out:
        ref32 = ref32.relu()
    e, e32 = rel_err(out, want), rel_err(ref32, want)
    ok = e < 5e-6
    print("store M={} K={} N={} relu_in={} relu_out={} res={} t128(a,out)={}{}: ours {:.2e}  cublas-fp32 {:.2e}  {}".format(
        M, K, N, relu_in, relu_out, use_res, int(a_t128), int(o_t128), e, e32, "OK" if ok else "FAIL"))
    return ok


def error_profile(gen, dev):
    """Where does the 3xTF32 error come from?  Signed relative error statistics on large outputs."""
    M, K, N = 4096, 256, 256
    a = torch.randn(M, K, generator=gen, device=dev).abs()     # same-sign operands: accumulator grows monotonically
    w = torch.randn(N, K, generator=gen, device=dev).abs() / K
    b = torch.zeros(N, device=dev)
    pk = fl.pack(w, b)
    out = fl.linear(a, pk).double()
    want = a.double() @ w.double().t()
    ref = torch.nn.functional.linear(a, w, b).double()
    for name, got in (("ours", out), ("cublas-fp32", ref)):
        r = (got - want) / want
        print("  positive operands  {:12s}: mean signed rel err {:+.3e}  rms {:.3e}  max {:.3e}".format(
            name, r.mean().item(), r.pow(2).mean().sqrt().item(), r.abs().max().item()))
    for K in (32, 64, 256):
        a = torch.randn(M, K, generator=gen, device=dev)
        w = torch.randn(N, K, generator=gen, device=dev) / math.sqrt(K)
        pk = fl.pack(w, b)
        out = fl.linear(a, pk).double()
        want = a.double() @ w.double().t()
        ref = torch.nn.functional.linear(a, w, b).double()
        for name, got in (("ours", out), ("cublas-fp32", ref)):
            e = (got - want)
            print("  gaussian operands K={:3d} {:12s}: rms abs err {:.3e}  max {:.3e}  (rms |out| {:.3f})".format(
                K, name, e.pow(2).mean().sqrt().item(), e.abs().max().item(), want.pow(2).mean().sqrt().item()))


def check_colmap(gen, dev):
    # coupling first layer: weight columns scattered to the identity columns of the full-width input
    M, D, H = 777, 64, 256
    x = torch.randn(M, D, generator=gen, device=dev)
    ident = torch.arange(1, D, 2, device=dev)
    w = torch.randn(H, ident.numel(), generator=gen, device=dev)
    b = torch.randn(H, generator=gen, device=dev)
    pk = fl.pack(w, b, col_map=ident.to(torch.int32), k_in=D)
    out = fl.linear(x, pk)
    want = x[:, ident].double() @ w.double().t() + b.double()
    e = rel_err(out, want)
    print("col_map first layer: {:.2e} {}".format(e, "OK" if e < 5e-6 else "FAIL"))
    return e < 5e-6


def rqs_cfg(K, H, inverse=False, identity_init=False):
    return _cabi.RqsConfig(K, _cabi.TAILS_LINEAR, int(identity_init), int(inverse), -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3,
                           1e-3, 1.0 / math.sqrt(H))


def check_rqs(M, D, K, H, gen, dev, inverse=False, coupling=True, h_t128=False):
    P = 3 * K - 1
    ppad = fl.RQS_PPAD[K]
    if coupling:
        tcols = torch.arange(0, D, 2, device=dev, dtype=torch.int32)
        ccols = torch.arange(1, D, 2, device=dev, dtype=torch.int32)
    else:
        tcols, ccols = None, None
    d_t = tcols.numel() if coupling else D
    x = torch.randn(M, D, generator=gen, device=dev) * 1.5
    hid = torch.randn(M, H, generator=gen, device=dev)
    w = torch.randn(d_t * P, H, generator=gen, device=dev) * (4.0 / math.sqrt(H))
    b = torch.randn(d_t * P, generator=gen, device=dev)
    pk = fl.pack(w, b, row_map=fl.grouped_row_map(d_t, P, ppad, dev), n_tile=fl.N_TILE_RQS)
    cfg = rqs_cfg(K, H, inverse)
    y = torch.empty_like(x)
    lad = torch.empty(M, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    fl.linear_rqs(fl.T128.from_rows(hid) if h_t128 else hid, pk, x, y, lad, False, d_t, tcols, ccols, cfg, status)
    torch.cuda.synchronize()
    # reference: fp64 GEMM -> fp32 params -> standalone spline kernel; yardstick: the same with the fp32 cuBLAS GEMM
    # (what the unfused path does).  The spline amplifies parameter noise (1/slope in the inverse), so the fused path
    # is judged against the yardstick's own error, quantile by quantile.
    args = (K, _cabi.TAILS_LINEAR, inverse, False, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3, 1.0 / math.sqrt(H))
    params = (hid.double() @ w.double().t() + b.double()).float()
    y2, lad2, _ = ops.rqs_layer(x, params, tcols, ccols, *args)
    y3, lad3, _ = ops.rqs_layer(x, torch.nn.functional.linear(hid, w, b), tcols, ccols, *args)
    q = torch.tensor([0.5, 0.99, 0.999, 1.0], device=dev)

    def quant(t):
        return torch.quantile(t.flatten()[: 1 << 22].float(), q)

    ey, ey3 = quant((y - y2).abs()), quant((y3 - y2).abs())
    el, el3 = quant((lad - lad2).abs()), quant((lad3 - lad2).abs())
    ok = bool((ey <= 3 * ey3 + 2e-6).all()) and bool((el <= 3 * el3 + 2e-5).all())
    print("rqs-fused M={} D={} K={} H={} inv={} coupling={}: |dy| q50/99/99.9/max {} (cuBLAS path {})  |dlad| {} ({}) {}"
          .format(M, D, K, H, inverse, coupling, ["%.1e" % v for v in ey.tolist()], ["%.1e" % v for v in ey3.tolist()],
                  ["%.1e" % v for v in el.tolist()], ["%.1e" % v for v in el3.tolist()], "OK" if ok else "FAIL"))
    return ok


def check_affine(M, D, H, gen, dev, layout, activation, inverse, h_t128):
    if layout == _cabi.AFFINE_BLOCKED:
        tcols = torch.arange(0, D, 2, device=dev, dtype=torch.int32)
        ccols = torch.arange(1, D, 2, device=dev, dtype=torch.int32)
        d_t = tcols.numel()
    else:
        tcols, ccols, d_t = None, None, D
    x = torch.randn(M, D, generator=gen, device=dev)
    hid = torch.randn(M, H, generator=gen, device=dev)
    w = torch.randn(2 * d_t, H, generator=gen, device=dev) / math.sqrt(H)
    b = torch.randn(2 * d_t, generator=gen, device=dev) * 0.5
    pk = fl.pack(w, b, row_map=fl.affine_row_map(d_t, layout, dev), n_tile=fl.N_TILE_AFFINE)
    y = torch.empty_like(x)
    lad = torch.empty(M, device=dev)
    fl.linear_affine(fl.T128.from_rows(hid) if h_t128 else hid, pk, x, y, lad, False, d_t, tcols, ccols, activation,
                     inverse)
    params = (hid.double() @ w.double().t() + b.double()).float()
    y2, lad2 = ops.affine_layer(x, params, tcols, ccols, layout, activation, inverse)
    ey = (y - y2).abs().max().item()
    el = (lad - lad2).abs().max().item()
    ok = ey < 2e-5 * max(1.0, y2.abs().max().item()) and el < 2e-4
    print("affine-fused M={} D={} H={} layout={} act={} inv={} t128={}: max|dy| {:.2e} max|dlad| {:.2e} {}".format(
        M, D, H, layout, activation, inverse, int(h_t128), ey, el, "OK" if ok else "FAIL"))
    return ok


def bench(dev, gen):
    M, H = 1 << 20, 256
    a = torch.randn(M, H, generator=gen, device=dev)
    w = torch.randn(H, H, generator=gen, device=dev) / 16
    b = torch.randn(H, generator=gen, device=dev)
    pk = fl.pack(w, b)
    out = torch.empty(M, H, device=dev)

    def timeit(fn, n=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(n):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / n

    t = timeit(lambda: fl.linear(a, pk, relu_in=True, out=out))
    flops = 2.0 * M * H * H
    at, ot, rt = fl.T128.from_rows(a), fl.T128(M, H, dev), fl.T128.from_rows(out)
    tt = timeit(lambda: fl.linear(at, pk, relu_in=True, residual=rt, out=ot, out_t128=True))
    print("hidden linear T128 in/out + residual: {:.3f} ms  {:.1f} TFLOP/s fp32-equivalent".format(tt, flops / tt / 1e9))
    print("hidden linear 1M x 256 x 256: {:.3f} ms  {:.1f} TFLOP/s fp32-equivalent ({:.1f} tf32 tensor TFLOP/s)".format(
        t, flops / t / 1e9, 3 * flops / t / 1e9))
    t2 = timeit(lambda: torch.nn.functional.linear(a, w, b))
    print("  cuBLAS fp32 same shape: {:.3f} ms  {:.1f} TFLOP/s".format(t2, flops / t2 / 1e9))
    # final layer + spline
    D, K = 64, 8
    P, ppad, d_t = 23, 24, 32
    x = torch.randn(M, D, generator=gen, device=dev)
    wf = torch.randn(d_t * P, H, generator=gen, device=dev) / 4
    bf = torch.randn(d_t * P, generator=gen, device=dev)
    pkf = fl.pack(wf, bf, row_map=fl.grouped_row_map(d_t, P, ppad, dev), n_tile=fl.N_TILE_RQS)
    tcols = torch.arange(0, D, 2, device=dev, dtype=torch.int32)
    ccols = torch.arange(1, D, 2, device=dev, dtype=torch.int32)
    cfg = rqs_cfg(K, H)
    y = x.clone()
    lad = torch.zeros(M, device=dev)
    t3 = timeit(lambda: fl.linear_rqs(a, pkf, x, y, lad, False, d_t, tcols, ccols, cfg, None))
    flops_f = 2.0 * M * H * 768
    t3t = timeit(lambda: fl.linear_rqs(at, pkf, x, y, lad, False, d_t, tcols, ccols, cfg, None))
    print("final layer + spline, T128 hidden: {:.3f} ms".format(t3t))
    print("final layer + spline 1M x 256 x 768: {:.3f} ms  {:.1f} TFLOP/s fp32-equivalent".format(t3, flops_f / t3 / 1e9))

    def unfused():
        p = torch.nn.functional.linear(a, wf, bf)
        return ops.rqs_layer(x, p, tcols, ccols, K, _cabi.TAILS_LINEAR, False, False, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3,
                             1e-3, 1.0 / 16)
    t4 = timeit(unfused, n=5)
    print("  cuBLAS fp32 + standalone spline kernel: {:.3f} ms".format(t4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bench", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(0)
    ok = True
    t0 = time.time()
    ok &= check_store(128, 32, 256, False, False, False, gen, dev)
    ok &= check_store(1000, 256, 256, False, False, False, gen, dev)
    ok &= check_store(1000, 256, 256, True, True, True, gen, dev)
    ok &= check_store(40000, 256, 512, True, False, True, gen, dev)
    ok &= check_store(5000, 8, 64, False, True, False, gen, dev)
    ok &= check_store(1000, 256, 256, False, False, False, gen, dev, a_t128=True)
    ok &= check_store(1000, 64, 256, False, False, False, gen, dev, o_t128=True)
    ok &= check_store(1000, 256, 256, True, True, True, gen, dev, a_t128=True, o_t128=True)
    ok &= check_store(70000, 32, 64, True, False, True, gen, dev, a_t128=True, o_t128=True)
    ok &= check_store(128, 752, 32, False, False, False, gen, dev)       # input-gradient shapes (K = layer width)
    ok &= check_store(5000, 736, 256, False, False, False, gen, dev)
    ok &= check_store(128, 48, 16, False, False, False, gen, dev)
    ok &= check_colmap(gen, dev)
    ok &= check_rqs(1000, 64, 8, 256, gen, dev, h_t128=True)
    ok &= check_rqs(1000, 64, 8, 256, gen, dev)
    ok &= check_rqs(30000, 64, 8, 256, gen, dev, inverse=True)
    ok &= check_rqs(5000, 16, 16, 256, gen, dev, coupling=False)
    ok &= check_rqs(3000, 20, 8, 64, gen, dev, coupling=True)
    ok &= check_affine(1000, 64, 256, gen, dev, _cabi.AFFINE_BLOCKED, _cabi.SCALE_SIGMOID2, False, True)
    ok &= check_affine(5000, 10, 16, gen, dev, _cabi.AFFINE_BLOCKED, _cabi.SCALE_SOFTPLUS_CLAMP3, True, False)
    ok &= check_affine(3000, 100, 64, gen, dev, _cabi.AFFINE_INTERLEAVED, _cabi.SCALE_SOFTPLUS_EPS, False, True)
    ok &= check_affine(300, 2, 32, gen, dev, _cabi.AFFINE_INTERLEAVED, _cabi.SCALE_SOFTPLUS_EPS, True, False)
    print("checks {} in {:.1f}s".format("PASSED" if ok else "FAILED", time.time() - t0))
    error_profile(gen, dev)
    if args.bench:
        bench(dev, gen)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
