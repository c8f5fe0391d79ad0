"""Micro-benchmark: attention recurrence forward and backward -- persistent L2-streaming kernel vs step-split path."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hypernet_image_captioning_b200 import ops

B, T, Fo, E, H, P = 512, 20, 200, 200, 200, 49
dev = "cuda"
g = torch.Generator(device=dev).manual_seed(1)
r = lambda *s: torch.randn(*s, generator=g, device=dev)
Kp, f, GIw = r(B, P, H) * 0.5, r(B, P, Fo) * 0.5, r(T * B, 3 * H) * 0.5
Ua, W_ih, W_hh = r(H, H) / H ** 0.5, r(3 * H, E + Fo) / (E + Fo) ** 0.5, r(3 * H, H) / H ** 0.5
bu, va, bv, bhh, h0 = r(H) * 0.1, r(H) * 0.3, r(1), r(3 * H) * 0.1, r(B, H) * 0.5
Hall = torch.empty(T + 1, B, H, device=dev); Hall[0] = h0
Hbm, attn = torch.empty(B, T, H, device=dev), torch.empty(B, T, P, device=dev)
XC, saved = torch.zeros(T * B, E + Fo, device=dev), torch.empty(5, T, B, H, device=dev)
lw = ops.AttGruWeights(W_ih, W_hh, Ua, E, P, step=False)
lws = ops.AttGruWeights(W_ih, W_hh, Ua, E, P, step=True)

def run(step):
    if step:
        ops.attgru_fwd(Kp, f, GIw, lws, bu, va, bv, bhh, Hall, Hbm, attn, XC, E, saved, 0, T)
    else:
        ops.attgru_seq_fwd(Kp, f, GIw, lw, bu, va, bv, bhh, Hall, Hbm, attn, XC, E, saved, 0, T)

for step in (False, True):
    for _ in range(2):
        run(step)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        run(step)
    e1.record(); torch.cuda.synchronize()
    print("step-split        " if step else "streaming         ", f"{e0.elapsed_time(e1) / 5 * 1e3:9.1f} us  ({e0.elapsed_time(e1) / 5 / T * 1e3:.1f} us/step)")

# ---- backward: persistent streaming kernel vs step-split ----
ops.attgru_fwd(Kp, f, GIw, lws, bu, va, bv, bhh, Hall, Hbm, attn, XC, E, saved, 0, T)
dHbm = r(B, T, H) * 0.3
for step in (False, True):
    for _ in range(2):
        ops.attgru_bwd(dHbm, None, Kp, f, attn, saved, Hall, Ua, va, W_ih, W_hh, E, step=step)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        ops.attgru_bwd(dHbm, None, Kp, f, attn, saved, Hall, Ua, va, W_ih, W_hh, E, step=step)
    e1.record(); torch.cuda.synchronize()
    print("bwd step-split        " if step else "bwd streaming         ", f"{e0.elapsed_time(e1) / 5 * 1e3:9.1f} us  ({e0.elapsed_time(e1) / 5 / T * 1e3:.1f} us/step)")
