"""Micro-benchmark of the two tensor-core kernels on cfg-2 shapes (FC_LINEAR_DEBUG=4 with a profiling build also prints
the wait-cycle counters)."""
import math, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import _cabi, linear as fl  # noqa: E402

dev = torch.device("cuda:0")
gen = torch.Generator(device=dev).manual_seed(0)
M, H, D, K = 1 << 20, 256, 64, 8
a = torch.randn(M, H, generator=gen, device=dev)
w = torch.randn(H, H, generator=gen, device=dev) / 16
b = torch.randn(H, generator=gen, device=dev)
pk = fl.pack(w, b)
out = torch.empty(M, H, device=dev)
P, ppad, d_t = 23, 24, 32
x = torch.randn(M, D, generator=gen, device=dev)
wf = torch.randn(d_t * P, H, generator=gen, device=dev) / 4
bf = torch.randn(d_t * P, generator=gen, device=dev)
pkf = fl.pack(wf, bf, row_map=fl.grouped_row_map(d_t, P, ppad, dev), n_tile=fl.N_TILE_RQS)
tcols = torch.arange(0, D, 2, device=dev, dtype=torch.int32)
ccols = torch.arange(1, D, 2, device=dev, dtype=torch.int32)
cfg = _cabi.RqsConfig(K, _cabi.TAILS_LINEAR, 0, 0, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3, 1.0 / math.sqrt(H))
y = x.clone()
lad = torch.zeros(M, device=dev)


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


t1 = timeit(lambda: fl.linear(a, pk, relu_in=True, out=out))
at, ot, rt = fl.T128.from_rows(a), fl.T128(M, H, dev), fl.T128.from_rows(out)
res = torch.randn(M, H, generator=gen, device=dev)
v = {}
v["rowA,rowO,res"] = timeit(lambda: fl.linear(a, pk, relu_in=True, out=out, residual=res))
v["t128A,rowO"] = timeit(lambda: fl.linear(at, pk, relu_in=True, out=out))
v["rowA,t128O"] = timeit(lambda: fl.linear(a, pk, relu_in=True, out=ot, out_t128=True))
v["t128A,t128O"] = timeit(lambda: fl.linear(at, pk, relu_in=True, out=ot, out_t128=True))
v["t128A,t128O,res"] = timeit(lambda: fl.linear(at, pk, relu_in=True, out=ot, residual=rt, out_t128=True))
print("  " + "  ".join("{} {:.3f}".format(k, t) for k, t in v.items()))
t2 = timeit(lambda: fl.linear_rqs(a, pkf, x, y, lad, False, d_t, tcols, ccols, cfg, None))
t2i = timeit(lambda: fl.linear_rqs(at, pkf, x, x, lad, False, d_t, tcols, ccols, cfg, None))
print("final+spline in place, T128 hidden: {:.3f} ms".format(t2i))
print("hidden {:.3f} ms   final+spline {:.3f} ms".format(t1, t2))

if int(os.environ.get("FC_LINEAR_DEBUG", "0")) & 4:
    import ctypes
    L = _cabi.lib()
    buf = (ctypes.c_ulonglong * 16)()
    names = ["mma_total", "w_tempty", "", "w_conv", "", "stages", "", "", "epi_total", "e_init", "e_wait",
             "e_drain", "conv_wait_tma", "conv_work"]
    for label, fn in (("hidden t128 res", lambda: fl.linear(at, pk, relu_in=True, out=ot, residual=rt, out_t128=True)),
                      ("final+spline", lambda: fl.linear_rqs(at, pkf, x, y, lad, False, d_t, tcols, ccols, cfg, None)),
                      ("final+spline in place", lambda: fl.linear_rqs(at, pkf, x, x, lad, False, d_t, tcols, ccols, cfg, None))):
        fn()
        torch.cuda.synchronize()
        L.fc_linear_debug_profile(ctypes.byref(buf))
        print("  prof " + label + ": " + "  ".join("{}={}".format(n, buf[i]) for i, n in enumerate(names) if n))
