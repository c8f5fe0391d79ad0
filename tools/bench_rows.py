"""Micro-benchmark of the hypernet streaming kernels (fp32 vs bf16 weights) on one head-sized matrix."""
import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hypernet_image_captioning_b200 import ops

def t(fn, n=5):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n

for (N, K) in ((90000, 11250), (67500, 8437), (240000, 480)):
    for dt in (torch.float32, torch.bfloat16):
        W = torch.randn(N, K, device="cuda").to(dt)
        A = torch.randn(1, K, device="cuda"); dY = torch.randn(1, N, device="cuda")
        bytes_w = N * K * W.element_size()
        f = t(lambda: ops.rows_linear_fwd(W, None, A, 0))
        b = t(lambda: ops.rows_linear_bwd(W, A, None, dY, 0))
        print(f"N={N} K={K} {str(dt):16s} fwd {f*1e3:8.1f} us {bytes_w/f/1e6:7.0f} GB/s | bwd {b*1e3:8.1f} us "
              f"{2*bytes_w/b/1e6:7.0f} GB/s", flush=True)
        del W
