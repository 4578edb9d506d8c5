"""Weight-gradient product grad_W = grad_y^T x: torch.mm against the split-K tensor-core product, and its k-slice sweep."""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowconductor_b200 import linear as fl  # noqa: E402

dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)


def timeit(fn, n=20):
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


for B, N, K in [(262144, 256, 256), (262144, 752, 256), (32768, 256, 256)]:
    gy = torch.randn(B, N, generator=g, device=dev)
    x = torch.randn(B, K, generator=g, device=dev)
    t_mm = timeit(lambda: gy.t().mm(x))
    t_new = timeit(lambda: fl.linear_splitk_t(gy, fl.pack_transposed(x)))
    t_pack = timeit(lambda: fl.pack_transposed(x))
    pk = fl.pack_transposed(x)
    t_gemm = timeit(lambda: fl.linear_splitk_t(gy, pk))
    print("B={} N={} K={}: torch.mm {:.3f} ms | split-K {:.3f} (pack x^T {:.3f}, product + slice sum {:.3f})".format(
        B, N, K, t_mm, t_new, t_pack, t_gemm), flush=True)

# reduction ranges per product at a small per-GPU shard (the 8-GPU cfg-3 step: 32768 rows per rank)
B, N, K = 32768, 256, 256
gy = torch.randn(B, N, generator=g, device=dev)
pk = fl.pack_transposed(torch.randn(B, K, generator=g, device=dev))
print("k_slices sweep at B=32768, 256x256:", "  ".join(
    "{}: {:.3f} ms".format(ks, timeit(lambda: fl.linear_splitk_t(gy, pk, k_slices=ks))) for ks in (16, 32, 64, 128)))
