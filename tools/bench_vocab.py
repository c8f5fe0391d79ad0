"""Vocabulary-projection chain at the benchmark shapes: logits GEMM (A-stationary schedule on / off), cross-entropy forward
+ gradient operand (one pass vs ce_fwd + ce_bwd_split), the two backward products.  `python tools/bench_vocab.py`."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hypernet_image_captioning_b200 import functional as Fn  # noqa: E402
from hypernet_image_captioning_b200 import ops  # noqa: E402


def timed(fn, n=10, reps=5):
    """n calls captured into one CUDA graph and replayed: device time, no host launch overhead (the host-side tensor-map
    encoding of a GEMM call costs about as much as these ~100 us kernels run)."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(n):
            fn()
    gr.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        gr.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (n * reps) * 1e3


g = torch.Generator().manual_seed(0)
M, V = 10240, 9684
for H in (150, 200):
    X = torch.randn(M, H, generator=g).cuda()
    W = (torch.randn(V, H, generator=g) * 0.2).cuda()
    b = torch.randn(V, generator=g).cuda()
    tgt = torch.randint(0, V, (M,), generator=g).cuda()
    xs, ws = ops.split_bf16(X), ops.split_bf16(W)
    out = torch.empty(M, V, device="cuda")
    res = {}
    for mode in ("0", "1"):
        os.environ["CAPHN_TC_ASTAT"] = mode
        us = timed(lambda: ops.gemm_tc(xs, ws, bias=b, out=out))
        res[mode] = out.clone()
        print(f"H={H} logits GEMM astat={mode}: {us:7.1f} us ({4.0 * M * V / us / 1e3:5.0f} GB/s of output)", flush=True)
    os.environ.pop("CAPHN_TC_ASTAT", None)
    print(f"    bit-identical: {torch.equal(res['0'], res['1'])}")
    t_set = timed(lambda: out.zero_())
    print(f"    (memset of the same [M, V] fp32 buffer: {t_set:6.1f} us = {4.0 * M * V / t_set / 1e3:5.0f} GB/s)")
    logits = res["0"]
    gs = torch.ones(1, device="cuda")
    t_fwd = timed(lambda: ops.ce_fwd(logits, tgt, 0))
    lb, lse = ops.ce_fwd(logits, tgt, 0)
    t_bwd = timed(lambda: ops.ce_bwd_split(logits, tgt, 0, lse, lb, gs))
    t_one = timed(lambda: ops.ce_fwd_split(logits, tgt, 0))
    print(f"H={H} ce_fwd {t_fwd:6.1f} us + ce_bwd_split {t_bwd:6.1f} us = {t_fwd + t_bwd:6.1f} us;  one pass (ce_fwd_split) "
          f"{t_one:6.1f} us = {(4.0 + 4.0) * M * V / t_one / 1e3:5.0f} GB/s", flush=True)
    lb1, lse1, hi, lo = ops.ce_fwd_split(logits, tgt, 0)
    t_old = timed(lambda: Fn.vocab_bwd_fused(logits, tgt, 0, lse, lb, gs, X, W))
    t_new = timed(lambda: Fn.vocab_bwd_fused(logits, tgt, 0, lse1, lb1, gs, X, W, hi, lo))
    print(f"H={H} backward of the projection: ce_bwd_split + dH + dW + colsum {t_old:6.1f} us;  scaled dH + [dW | db] "
          f"{t_new:6.1f} us", flush=True)
    d = ops.SplitOperand(hi, lo, M, V, hi.shape[1])
    dT = ops.SplitOperand(hi, lo, V, M, hi.shape[1], True)
    wt = ops.split_bf16_t(W)
    ht = ops.split_bf16_t(X, ones_row=True)
    wbuf = torch.empty(V, ops.round4(H + 1), device="cuda")[:, :H + 1]
    print(f"H={H} dH product alone {timed(lambda: ops.gemm_tc(d, wt, scale=(gs, lb1[1:]))):6.1f} us, "
          f"[dW | db] product alone {timed(lambda: ops.gemm_tc(dT, ht, scale=(gs, lb1[1:]), out=wbuf)):6.1f} us", flush=True)

