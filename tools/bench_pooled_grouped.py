"""Many-style training step of the pooled captioners: `python tools/bench_pooled_grouped.py [--iters N] [--warmup W]`.

BASELINE configs[1] shapes (B=512, T=20, E=200, H=150, V=9684), fp32 mode, G = 1, 3 and 100 style groups of random sizes
(every row draws its group uniformly).  One timed step = hypernet forward for all G styles, captioner forward, mean
cross-entropy (padding index 0) and the whole backward; gradients are dropped between steps, no optimizer.

    GRU   forward_loss(groups=)          the fused many-style loss node
          forward(groups=) + cross_entropy   logits materialised, loss and its backward as separate passes
    LSTM  forward_loss(groups=)          grouped kernels, fused loss
          forward(groups=) + cross_entropy   grouped kernels
          per-group loop                 modules._run_grouped: one complete single-style decoder call per group

Each variant is timed with CUDA events over --iters steps after --warmup steps; the variants of one (cell, G) alternate
over --rounds rounds and the median round is printed, with the loss of the last step (variants of one cell compute the
same loss up to rounding).  The card name and power limit are printed first: the times belong to them."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, T, E, H, V = 512, 20, 200, 150, 9684


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)} | {q}: {out}"


def variants(m, cell, styles, pooled, caps, groups, G):
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200.modules import _run_grouped

    def fused():
        cap = m.forward_grouped(styles)
        loss, _ = cap.forward_loss(m.image_encoder(pooled), caps, ignore_index=0, groups=groups)
        return loss

    def unfused():
        cap = m.forward_grouped(styles)
        return C.cross_entropy(cap(m.image_encoder(pooled), caps, True, groups=groups), caps, 0)

    def loop():
        cap = m.forward_grouped(styles)
        feats = m.image_encoder(pooled)
        h0 = cap._h0(feats)
        logits = _run_grouped(lambda g, f, c, h: cap._forward_one(f, c, h, cap._cells(g)), groups, [feats, caps, h0], G)[0]
        return C.cross_entropy(logits, caps, 0)

    out = {"forward_loss(groups=)": fused, "forward(groups=) + cross_entropy": unfused}
    if cell == "lstm":
        out["per-group loop (_run_grouped)"] = loop
    return out


def time_steps(m, fn, n):
    loss = None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        m.zero_grad(set_to_none=True)
        loss = fn()
        loss.backward()
        m.release_graph()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, loss.item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--groups", type=int, nargs="+", default=[1, 3, 100])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import hypernet_image_captioning_b200 as C
    from oracle import caption_hn_oracle as O
    print(card())
    print(f"B={B} T={T} E={E} H={H} V={V} fp32; {args.iters} timed steps after {args.warmup} warm-up steps per round, "
          f"median of {args.rounds} rounds")
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(0)
    pooled = torch.relu(torch.randn(B, 2048, generator=gen)).to(dev)
    caps = O.synth_captions(B, T, V, gen).to(dev)
    for cell in ("gru", "lstm"):
        torch.manual_seed(0)
        with torch.device(dev):
            m = C.HyperNetPooled(E, H, V, None, num_layers=1, type=cell)
        for G in args.groups:
            groups = torch.randint(0, G, (B,), generator=gen)
            styles = torch.randn(G, E, generator=gen).to(dev)
            sizes = torch.bincount(groups, minlength=G)
            vs = variants(m, cell, styles, pooled, caps, groups, G)
            for fn in vs.values():
                time_steps(m, fn, args.warmup)
            ms = {k: [] for k in vs}
            loss = {}
            for _ in range(args.rounds):
                for k, fn in vs.items():
                    t, loss[k] = time_steps(m, fn, args.iters)
                    ms[k].append(t)
            print(f"\n{cell.upper()} G={G} (group sizes {int(sizes.min())}..{int(sizes.max())}, "
                  f"{int((sizes == 0).sum())} empty)")
            for k in vs:
                med = statistics.median(ms[k])
                print(f"  {k:34s} {med:8.3f} ms/step  {B / med:7.1f} k captions/s  "
                      f"(rounds {', '.join(f'{t:.3f}' for t in ms[k])})  loss {loss[k]:.6f}")
        del m
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
