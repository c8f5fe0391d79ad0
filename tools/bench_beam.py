"""Batched beam-search throughput of both captioners (B = 512, k = 3, max_steps = 20), CUDA events:
`python tools/bench_beam.py [--iters N]`.

The hypernet forward (weight generation) and the image encoder run before the timer: a call is the search alone.  Both
models are default-initialised, on synthetic features; with such weights </s> rarely wins, so the searches run to their
step limit (the step count is printed) and the numbers are the cost of a full-length search.  Context lines: the pooled
search with one beam against greedy ``infer`` at the same shape, and the [V, 3H] projection-table GEMM the pooled search
builds on every call."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hypernet_image_captioning_b200 as C  # noqa: E402
from hypernet_image_captioning_b200 import ops  # noqa: E402

B, K, MAX_STEPS, V = 512, 3, 20, 9684


def timed(fn, n):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def steps_run(fn):
    """Decoder steps one call runs: its caphn_beam_step launches."""
    n, call = [0], ops._cabi.call

    def counting(name, *args):
        n[0] += name == "caphn_beam_step"
        return call(name, *args)
    ops._cabi.call = counting
    try:
        out = fn()
    finally:
        ops._cabi.call = call
    return n[0], sum(x is not None for x in out)


def report(tag, ms, steps, n_cap):
    print(f"{tag}: {ms:.3f} ms per call ({B / ms * 1e3:.0f} captions/s), {steps} steps run "
          f"({ms / steps * 1e3:.1f} us/step), {n_cap}/{B} images with a caption")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_beam.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True)
    print(q.stdout.strip())
    dev = torch.device("cuda", 0)
    n = args.iters
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(1)

    with torch.device(dev):
        m = C.HyperNetPooled(200, 150, V, None)
    pooled = torch.relu(torch.randn(B, 2048, generator=g)).to(dev)
    h0 = torch.rand(B, 150, generator=g).to(dev)
    with torch.no_grad():
        cap = m.forward(m.captioner.embed.weight[4:5])
        feats = m.image_encoder(pooled)
    beam = lambda k: cap.beam_search_batched(feats, beam_size=k, max_steps=MAX_STEPS, h0=h0)
    report(f"pooled beam search k={K}", timed(lambda: beam(K), n), *steps_run(lambda: beam(K)))
    report("pooled beam search k=1", timed(lambda: beam(1), n), *steps_run(lambda: beam(1)))
    ms = timed(lambda: cap.infer(feats, max_len=MAX_STEPS + 1, h0=h0), n)
    print(f"pooled greedy infer, max_len={MAX_STEPS + 1}: {ms:.3f} ms per call ({B / ms * 1e3:.0f} captions/s)")
    W_ih, _, b_ih, _ = [t.detach().contiguous() for t in cap._cells()[0]]
    emb = cap.embed.weight.detach()
    ms = timed(lambda: ops.linear(emb, W_ih, b_ih), n)
    print(f"projection table [{V}, {3 * 150}] alone: {ms:.3f} ms")
    del m, cap, feats
    torch.cuda.empty_cache()

    with torch.device(dev):
        ma = C.HyperNetAttention(200, 200, 200, V, None)
    fa = torch.randn(B, 49, 2048, generator=g).to(dev)
    with torch.no_grad():
        capa = ma.forward(ma.captioner.embed.weight[4:5])
    beam_a = lambda: capa.beam_search_batched(fa, beam_size=K, max_steps=MAX_STEPS)
    report(f"attention beam search k={K}", timed(beam_a, n), *steps_run(beam_a))


if __name__ == "__main__":
    main()
