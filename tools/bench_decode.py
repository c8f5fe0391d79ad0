"""Greedy-decode throughput of both variants (B=512, T=20), CUDA events: `python tools/bench_decode.py [tag]`."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hypernet_image_captioning_b200 as C  # noqa: E402
from hypernet_image_captioning_b200.synth import synth_captions  # noqa: E402

B, T, V = 512, 20, 9684
dev = torch.device("cuda", 0)
N_TIMED = int(os.environ.get("CAPHN_DECODE_ITERS", "20"))
if os.environ.get("CAPHN_NO_GRAPH") == "1":      # eager launches (for an ncu launch list: ncu cannot follow stream capture)
    from hypernet_image_captioning_b200 import graphs
    graphs.ENABLED = False


def timed(fn, n=N_TIMED):
    for _ in range(3 if n > 2 else 1):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


torch.manual_seed(0)
with torch.device(dev):
    m = C.HyperNetPooled(200, 150, V, None)
g = torch.Generator().manual_seed(1)
pooled = torch.relu(torch.randn(B, 2048, generator=g)).to(dev)
h0 = torch.rand(B, 150, generator=g).to(dev)


def dec_pooled():
    with torch.no_grad():
        cap = m.forward(m.captioner.embed.weight[4:5])
        return cap.infer(m.image_encoder(pooled), max_len=T, h0=h0)


def hyper_only():
    with torch.no_grad():
        return m.generate_theta(m.captioner.embed.weight[4:5])


ms = timed(dec_pooled)
ms_h = timed(hyper_only)
print(f"{sys.argv[1] if len(sys.argv) > 1 else ''} pooled greedy decode: {ms:.3f} ms ({B / ms * 1e3:.0f} captions/s); "
      f"hypernet forward alone {ms_h:.3f} ms; decode loop {ms - ms_h:.3f} ms = {(ms - ms_h) / T * 1e3:.1f} us/step")
del m
torch.cuda.empty_cache()
with torch.device(dev):
    ma = C.HyperNetAttention(200, 200, 200, V, None)
feats = torch.randn(B, 49, 2048, generator=g).to(dev)
caps = synth_captions(B, T, V, g).to(dev)


def dec_att():
    with torch.no_grad():
        cap = ma.forward(ma.captioner.embed.weight[4:5])
        return cap(feats, caps, 1.0)


ms = timed(dec_att)
print(f"{sys.argv[1] if len(sys.argv) > 1 else ''} attention greedy decode: {ms:.3f} ms ({B / ms * 1e3:.0f} captions/s)")
ma.async_hypernet = True          # hypernet weight streaming next to the feature branch (streams.py)
ms = timed(dec_att)
print(f"{sys.argv[1] if len(sys.argv) > 1 else ''} attention greedy decode, async hypernet: {ms:.3f} ms ({B / ms * 1e3:.0f} captions/s)")
