#!/usr/bin/env python
"""bench.py -- captions/s of the Caption-HN hot path on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR] # our CUDA path (default N=1)
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]     # the reference's CPU path (oracle port)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N # N > 1 (one rank per GPU, NCCL)

Workload (BASELINE.json configs[1]): pooled-feature hypernet-GRU (hypernet.py HyperNet + DecoderGRU), batch 512 per
GPU, T=20, E=200, H=150, V=9684, L=1, fp32, teacher-forced forward + backward with the gradient flowing through the
generated weights into the hypernet heads ("flow"), hypernet forward included, no optimizer step (SURVEY 8(d)).
A "step" = hypernet -> theta -> image_encoder.fc -> decoder -> cross-entropy -> full backward on one batch.
Synthetic data, default-init weights.  Weak scaling: the per-GPU batch is fixed.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(B=512, T=20, E=200, H=150, V=9684, L=1, D=2048)
CPU_SAMPLE_B = 512  # same batch as the GPU arm: the per-step hypernet cost amortises over the batch, so a smaller sample would understate the CPU
DUMP_LOGIT_ROWS = 256          # (caption, position) rows of the [B*T, V] logits that --dump-outputs writes
DUMP_GRAD_ENTRIES = 1 << 19    # entries written per parameter gradient (all of them when it has fewer)
DUMP_MAX_BYTES = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=CFG["B"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (loss, logits, parameter gradients) "
                         "as DIR/<name>.npy, float32; large arrays as a fixed seeded sample, %d MB in all at most"
                         % (DUMP_MAX_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


# ----------------------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        load = [s for s, p in zip(sm, power) if p > 250] or sm
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle port of the reference's PyTorch path on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_arm(steps, warmup, B=CPU_SAMPLE_B):
    """Times hypernet fwd + image_encoder.fc + DecoderGRU fwd + CE + backward (flow) on the CPU, all host threads."""
    from oracle import caption_hn_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = CFG
    p = O.init_params_pooled(c["D"], c["E"], c["H"], c["V"], L=c["L"], seed=0)
    p = {k: v.requires_grad_(True) for k, v in p.items()}
    g = torch.Generator().manual_seed(1234)
    pooled = torch.relu(torch.randn(B, c["D"], generator=g))
    caps = O.synth_captions(B, c["T"], c["V"], g)
    h0 = torch.rand(B, c["H"], generator=g)

    def step():
        for v in p.values():
            v.grad = None
        style = p["captioner.embed.weight"][4:5]
        logits, _, _ = O.path_pooled(p, style, pooled, caps, h0, L=c["L"], flow=True)
        loss = O.caption_loss(logits, caps, None)
        loss.backward()
        return float(loss)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"value": B * steps / dt, "unit": "captions/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"oracle port (torch CPU fp32) of the same workload at batch {B} x {steps} steps "
                      f"(+{warmup} warm-up), flow-mode fwd+bwd incl. hypernet", "ms_per_step": dt / steps * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    r = cpu_reference_arm(steps, warmup)
    line = {
        "impl": "reference", "metric": "hypernet-GRU train captions/s", "value": r["value"], "unit": "captions/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),   # our arm's config; the bounded sample actually run is in `cpu_baseline`
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "captions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    c = CFG
    return {
        "workload": (f"BASELINE configs[1]: pooled-feature hypernet-GRU (hypernet.py HyperNet + DecoderGRU) teacher-forced "
                     f"fwd+bwd, flow mode, hypernet fwd included, no optimizer; B={args.batch}/GPU T={c['T']} E={c['E']} "
                     f"H={c['H']} V={c['V']} L={c['L']} D={c['D']}"),
        "global_batch": args.batch * world, "seq_len": c["T"], "parallelism": f"dp{world}",
        "l2": "inputs larger than L2: 6.46 GB of hypernet head weights are streamed every step",
    }


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import _cabi, ops, parallel
    from hypernet_image_captioning_b200.synth import synth_captions   # (the oracle is used by the cpu_baseline leg only)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl=ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _cabi.load()

    c = CFG
    B, T = args.batch, c["T"]
    torch.manual_seed(0)
    with torch.device(dev):
        model = C.HyperNetPooled(c["E"], c["H"], c["V"], None, num_layers=c["L"])
    model.grad_mode = "flow"
    model.async_hypernet = True        # hypernet weight streaming on its own stream (streams.py)
    model.dp_enabled = world > 1
    shared = parallel.shared_parameters(model)
    if world > 1:      # the 15 MB shared-gradient bucket is reduced on a side stream while the head backward runs
        parallel.enable_overlap(shared)

    g = torch.Generator().manual_seed(1234 + rank)
    pooled_h = torch.relu(torch.randn(B, c["D"], generator=g)).pin_memory()
    caps_h = synth_captions(B, T, c["V"], g).pin_memory()
    pooled_d, caps_d = pooled_h.to(dev), caps_h.to(dev)
    h0_d = torch.rand(B, c["H"], generator=g).to(dev)
    inv_world = 1.0 / world

    def step(pooled, caps, h0):
        model.zero_grad(set_to_none=True)
        style = model.captioner.embed.weight[4:5]          # 'factual' row, hypernet_attention.py:139-142 idiom
        captioner = model.forward(style)
        feats = model.image_encoder(pooled)
        loss, logits = captioner.forward_loss(feats, caps, h0=h0, ignore_index=None)   # decoder + CE (hypernet.py:139-145)
        (loss * inv_world if world > 1 else loss).backward()
        if world > 1:
            parallel.allreduce_shared_grads(shared)
        return loss, logits

    # End to end through the module API, the way a training loop with a pinned-memory loader runs it: every step's
    # inputs are copied host->device inside the timed region (on a copy stream, one step ahead, into one of two device
    # buffers), and every step's loss is read back to the host (asynchronously; the host waits for step i-1's value
    # before it enqueues step i+1, so it never runs more than one step ahead of the device).
    # The whole step (forward + backward + gradient all-reduces) is captured into ONE CUDA graph and replayed
    # (graphs.GraphedStep; CAPHN_BENCH_GRAPH=0 or a failed capture runs the same kernels eagerly).
    from hypernet_image_captioning_b200 import graphs
    gstep = None
    if os.environ.get("CAPHN_BENCH_GRAPH", "1") != "0":
        gstep = graphs.GraphedStep(step, (pooled_d, caps_d, h0_d), params=list(model.parameters()),
                                   release=model.release_graph)
        if not gstep.captured:
            gstep = None
    run_step = gstep if gstep is not None else step

    copy_stream = torch.cuda.Stream(device=dev)
    dbuf = [(torch.empty_like(pooled_d), torch.empty_like(caps_d), torch.empty_like(h0_d)) for _ in range(2)]
    h0_pin = [torch.empty(B, c["H"]).pin_memory() for _ in range(2)]
    ev_copied = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_loss = [torch.cuda.Event() for _ in range(2)]
    loss_ring = [torch.empty(1, pin_memory=True) for _ in range(2)]
    e2e_state = {"i": 0, "primed": False, "losses": []}

    def _issue_copy(j):
        ev_copied[j % 2].synchronize()                        # the last copy out of this pinned h0 buffer is done
        torch.rand(B, c["H"], out=h0_pin[j % 2])              # h0 drawn on the host per call like the reference (later.py:393)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[j % 2])            # the step that last used this buffer has finished
            dbuf[j % 2][0].copy_(pooled_h, non_blocking=True)
            dbuf[j % 2][1].copy_(caps_h, non_blocking=True)
            dbuf[j % 2][2].copy_(h0_pin[j % 2], non_blocking=True)
            ev_copied[j % 2].record(copy_stream)

    def step_e2e():
        i = e2e_state["i"]
        cur = torch.cuda.current_stream()
        if not e2e_state["primed"]:
            _issue_copy(i)
            e2e_state["primed"] = True
        _issue_copy(i + 1)                                    # next step's inputs fly while this step computes
        cur.wait_event(ev_copied[i % 2])
        loss, _ = run_step(*dbuf[i % 2])
        ev_free[i % 2].record(cur)
        loss_ring[i % 2].copy_(loss.detach().reshape(1), non_blocking=True)
        ev_loss[i % 2].record(cur)
        if i >= 1:
            ev_loss[(i - 1) % 2].synchronize()                # read the previous step's loss on the host
            e2e_state["losses"].append(float(loss_ring[(i - 1) % 2]))
        e2e_state["i"] = i + 1
        return loss_ring[i % 2]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        run_step(pooled_d, caps_d, h0_d)
    l0 = _cabi.launches()
    last = [None]

    def headline_step():
        last[0] = run_step(pooled_d, caps_d, h0_d)
    ms = timed(headline_step, args.steps)
    launches = _cabi.launches() - l0
    if gstep is not None:                                     # replayed launches are not seen by the library's counter
        launches = gstep.launches_per_step * args.steps
    value = B * world * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last[0], model)
    last = None

    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = B * world * args.steps / (ms_e2e * 1e-3)
    h2d = pooled_h.numel() * 4 + caps_h.numel() * 8 + B * c["H"] * 4
    torch.cuda.synchronize()
    final_loss = float(loss_ring[(e2e_state["i"] - 1) % 2])

    # ---- roofline of the dominant kernel: the fused head backward (reads W2 once, writes dW2 once), timed alone ----
    head = model.hn_heads[0]
    W2 = head[2].weight.detach()
    N, K = W2.shape
    a1 = torch.randn(1, K, device=dev)
    dY = torch.randn(1, N, device=dev)
    for _ in range(2):
        ops.rows_linear_bwd(W2, a1, None, dY, ops.ACT_NONE)
    torch.cuda.synchronize()
    evs = []
    for _ in range(5):
        dWs = torch.empty(N, K, device=dev)
        dP, db, dA = torch.empty(1, N, device=dev), torch.empty(N, device=dev), torch.zeros(1, K, device=dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        _cabi.call("caphn_rows_linear_bwd", W2.data_ptr(), a1.data_ptr(), K, None, 0, dY.data_ptr(), N, dP.data_ptr(),
                   dWs.data_ptr(), db.data_ptr(), dA.data_ptr(), K, 1, N, K, 0, 0.01,
                   torch.cuda.current_stream().cuda_stream)
        e.record()
        evs.append((s, e))
        del dWs
    torch.cuda.synchronize()
    k_ms = statistics.mean(s.elapsed_time(e) for s, e in evs)
    alg_bytes = 2.0 * N * K * 4
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("rows_bwd_kernel")
    except Exception:  # noqa: BLE001
        pass
    roofline = {"kernel": "rows_bwd_kernel<1> (hn_heads.0.2 backward: dW2 + dA1 in one pass)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json (burst copy)" if peaks else "fallback 6650 GB/s",
                "alg_bytes_per_launch": alg_bytes, "ms_per_launch": k_ms}

    # ---- sustained run: >= 2 s of back-to-back headline steps with its own clock samples (power steady state) ----
    sustained = None
    if not args.no_extras:
        n_sus = max(args.steps, int(2200.0 / (ms / args.steps)) + 1)
        sus_sampler = ClockSampler(local)
        if rank == 0:
            sus_sampler.start()
        ms_sus = timed(lambda: run_step(pooled_d, caps_d, h0_d), n_sus)
        sus_clocks = sus_sampler.stop() if rank == 0 else None
        sustained = {"steps": n_sus, "seconds": ms_sus * 1e-3, "ms_per_step": ms_sus / n_sus,
                     "captions_per_s": B * world * n_sus / (ms_sus * 1e-3), "clocks": sus_clocks}

    graphed = gstep is not None
    gstep = run_step = None                                   # release the graph's memory pool (gradients + activations)
    model.async_hypernet = False          # the eager extras below run single-stream (the side stream pays off under a graph)
    model.zero_grad(set_to_none=True)
    torch.cuda.empty_cache()

    extras = {}
    rooflines = {}
    hn_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters() if n_.startswith("hn_"))
    sh_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters()
                     if not n_.startswith("hn_") and not n_.startswith("captioner.lstm_cell"))
    w2_b = 4.0 * sum(h_[2].weight.numel() for h_ in model.hn_heads)
    # flow-mode training step, SURVEY 8(d): parameters read once, gradients written once, head second-layer weights read
    # once more for dA1, per caption: pooled feature + caption + logits written and re-read once
    step_bytes = 2 * hn_b + w2_b + 2 * sh_b + B * (c["D"] * 4.0 + 8.0 * T + 2.0 * T * c["V"] * 4.0)
    rooflines["pooled_train_step"] = roofline_block(step_bytes, ms / args.steps, peak,
                                                    "whole fwd+bwd step (headline `value`), compulsory traffic only")
    if sustained is not None:
        rooflines["pooled_train_step_sustained"] = roofline_block(step_bytes, sustained["ms_per_step"], peak,
                                                                  f"same, {sustained['seconds']:.1f} s back to back")
    def pooled_extras():
        # literal mode (the reference's actual behaviour: graph cut at utils.py:57, no head backward)
        model.grad_mode = "literal"
        for _ in range(3):
            step(pooled_d, caps_d, h0_d)
        ms_lit = timed(lambda: step(pooled_d, caps_d, h0_d), args.steps)
        model.grad_mode = "flow"
        extras["literal_mode_captions_per_s"] = B * world * args.steps / (ms_lit * 1e-3)
        # the reference's own call shape (hypernet.py:139-145): captioner(features, captions, True) returns the logits and the
        # SCRIPT computes the loss -- with torch's F.cross_entropy (the unedited script) or caphn.cross_entropy (one changed
        # line); the headline uses the fused decoder + loss node (forward_loss).  Eager launches, flow mode.
        import torch.nn.functional as F_
        def step_shape(ce):
            model.zero_grad(set_to_none=True)
            captioner = model.forward(model.captioner.embed.weight[4:5])
            logits = captioner(model.image_encoder(pooled_d), caps_d, True, h0=h0_d)
            loss = ce(logits)
            (loss * inv_world if world > 1 else loss).backward()
            if world > 1:
                parallel.allreduce_shared_grads(shared)
        ces = {"torch_F_cross_entropy": lambda lg: F_.cross_entropy(lg.view(-1, c["V"]), caps_d.view(-1)),
               "caphn_cross_entropy": lambda lg: C.cross_entropy(lg, caps_d, None)}
        extras["reference_call_shape_captions_per_s"] = {}
        for name_, ce_ in ces.items():
            for _ in range(3):
                step_shape(ce_)
            ms_s = timed(lambda: step_shape(ce_), args.steps)
            extras["reference_call_shape_captions_per_s"][name_] = B * world * args.steps / (ms_s * 1e-3)
        # greedy decode (DecoderGRU.infer, max_len = T), hypernet forward included
        def decode():
            with torch.no_grad():
                cap = model.forward(model.captioner.embed.weight[4:5])
                return cap.infer(model.image_encoder(pooled_d), max_len=T, h0=h0_d)
        for _ in range(3):
            decode()
        ms_dec = timed(decode, args.steps)
        extras["greedy_decode_captions_per_s"] = B * world * args.steps / (ms_dec * 1e-3)
        hn_bytes = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters() if n_.startswith("hn_"))
        dec_shared = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters()
                               if not n_.startswith("hn_") and not n_.startswith("captioner.lstm_cell"))
        # SURVEY 8(d) compulsory traffic: every parameter read once, pooled feature + int64 caption read, T*V probabilities written
        dec_bytes = hn_bytes + dec_shared + B * (c["D"] * 4.0 + T * c["V"] * 4.0)
        rooflines["pooled_greedy_decode"] = roofline_block(dec_bytes, ms_dec / args.steps, peak,
                                                           "heads + shared params read once, probabilities [B,T,V] written once")
        lit_bytes = hn_bytes + dec_shared * 2 + B * (c["D"] * 4.0 + 8.0 * T + 2.0 * T * c["V"] * 4.0)
        rooflines["pooled_train_literal"] = roofline_block(lit_bytes, ms_lit / args.steps, peak,
                                                           "heads read once (no head backward: graph cut of utils.py:57), decoder as in flow mode")
        # optimizer step (SURVEY 8(f) rank 1): FusedAdam with the global-norm clip folded in, on the gradients of the
        # last training step; Adam moves 28 bytes per parameter (p,g,m,v read; p,m,v written) + 4 for the norm pass
        from hypernet_image_captioning_b200 import FusedAdam
        step(pooled_d, caps_d, h0_d)
        opt_params = [p_ for p_ in model.parameters() if p_.grad is not None]
        n_opt = sum(p_.numel() for p_ in opt_params)
        opt = FusedAdam(opt_params, lr=1e-6, max_grad_norm=5.0)
        for _ in range(2):
            opt.step()
        ms_opt = timed(opt.step, 5) / 5
        extras["optimizer"] = {"kind": "FusedAdam + clip_grad_norm 5.0 (hypernet heads/base, embed, image fc)",
                               "params": n_opt, "ms_per_step": ms_opt,
                               "alg_bytes": 32.0 * n_opt, "achieved_gbs": 32.0 * n_opt / (ms_opt * 1e-3) / 1e9,
                               "hbm_frac": 32.0 * n_opt / (ms_opt * 1e-3) / 1e9 / peak}
        def step_opt():
            step(pooled_d, caps_d, h0_d)
            opt.step()
        for _ in range(2):
            step_opt()
        ms_full = timed(step_opt, args.steps)
        extras["train_with_optimizer_captions_per_s"] = B * world * args.steps / (ms_full * 1e-3)
        del opt, opt_params
        model.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
        # rank-G head gradients: dW2 = dtheta^T a stays a (dtheta, a) pair; FusedAdam forms it on the fly
        model.head_grad_mode = "lowrank"
        opt = FusedAdam([p_ for p_ in model.parameters() if not any(p_ is q_ for q_ in model.captioner.lstm_cell.parameters())],
                        lr=1e-6, max_grad_norm=5.0)
        def step_lr():
            step(pooled_d, caps_d, h0_d)
            opt.step()
        for _ in range(3):
            step_lr()
        ms_bwd_lr = timed(lambda: step(pooled_d, caps_d, h0_d), args.steps)
        step(pooled_d, caps_d, h0_d)
        ms_full_lr = timed(step_lr, args.steps)
        extras["lowrank_head_grad"] = {
            "train_fwd_bwd_captions_per_s": B * world * args.steps / (ms_bwd_lr * 1e-3),
            "train_with_optimizer_captions_per_s": B * world * args.steps / (ms_full_lr * 1e-3),
            "note": "head dW kept as (dtheta, a): backward streams W once (dA only), Adam reads/writes p,m,v only"}
        model.head_grad_mode = "materialize"
        del opt
        for p_ in model.parameters():
            p_.grad_lowrank = None
        model.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
        # bf16 mode (BASELINE configs[1] "fp32 and bf16"): hypernet weights + gradients in bf16, plain-bf16 tensor-core
        # products, fp32 accumulation / recurrent state; tolerance vs the fp32 oracle stated in tests/test_gpu_bf16.py
        model.set_precision("bf16")
        for _ in range(3):
            step(pooled_d, caps_d, h0_d)
        ms_bf = timed(lambda: step(pooled_d, caps_d, h0_d), args.steps)
        extras["bf16_mode_train_captions_per_s"] = B * world * args.steps / (ms_bf * 1e-3)
        ops.set_precision("fp32")

    if not args.no_extras:
        # a failure in one of the secondary measurements is recorded under its name and must not cost the headline line
        # (every rank runs the same code, so a deterministic failure is the same on every rank)
        try:
            pooled_extras()
        except Exception as e:  # noqa: BLE001
            extras["pooled_extras_error"] = f"{type(e).__name__}: {e}"[:300]
            model.grad_mode, model.head_grad_mode = "flow", "materialize"
            ops.set_precision("fp32")
            torch.cuda.synchronize()
        model = None
        torch.cuda.empty_cache()
        # the other workloads: each builds its own model
        for name_, fn_ in (("attention", lambda: attention_extras(args, dev, world, timed, rooflines, peak)),
                           ("cc", lambda: cc_extras(args, dev, world, timed, rooflines, peak)),
                           ("lstm", lambda: lstm_extras(args, dev, world, timed)),
                           ("pooled_l2", lambda: pooled_l2_extras(args, dev, world, timed, rooflines, peak))):
            try:
                extras.update(fn_())
            except Exception as e:  # noqa: BLE001
                extras[f"{name_}_extras_error"] = f"{type(e).__name__}: {e}"[:300]
                if world > 1:
                    parallel.disable_overlap()
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
        if sustained is not None:
            extras["sustained_headline"] = sustained

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        model = None
        torch.cuda.empty_cache()
        if not args.no_extras:
            # third column of SURVEY 8(d): the reference's PyTorch path run by stock torch eager ON THIS GPU (cuBLAS / ATen
            # kernels; none of ours) -- "the only existing Blackwell path".  Part of the baseline leg: it executes the oracle.
            try:
                extras["torch_eager_gpu_captions_per_s"] = torch_eager_gpu_arm(dev, timed, B)
            except Exception as e:  # noqa: BLE001
                extras["torch_eager_gpu_captions_per_s"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
            torch.cuda.empty_cache()
        cpu = cpu_reference_arm(steps=3, warmup=1)

    if rank == 0:
        line = {
            "metric": "hypernet-GRU train captions/s", "value": value, "unit": "captions/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),      # identical to the reference arm's config
            "cuda_graph": graphed,
            "e2e": {"value": e2e_value, "unit": "captions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "rooflines": rooflines,
            "cpu_baseline": ({k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")} if cpu else None),
            "loss": final_loss, "extras": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(dirname, loss, logits, model):
    """What one headline step returns to its caller, as float32 .npy files under `dirname`: loss.npy, logits_rows.npy
    (DUMP_LOGIT_ROWS rows of the [B*T, V] logits) and grad.<parameter>.npy for every parameter gradient (flattened;
    DUMP_GRAD_ENTRIES entries of the larger ones).  The rows and entries are drawn from generators seeded by the array's
    name, so every run with the same arguments writes the same positions and two builds compare entry for entry."""
    import zlib
    import numpy as np

    def pick(name, x, k):
        """k rows of x (all of them when it has no more)."""
        if x.shape[0] <= k:
            return x
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        return x[torch.randint(x.shape[0], (k,), generator=g).sort().values.to(x.device)]

    out = {"loss": loss.detach().reshape(1)}
    lg = logits.detach()
    out["logits_rows"] = pick("logits_rows", lg.reshape(-1, lg.shape[-1]), DUMP_LOGIT_ROWS)
    for name, p in model.named_parameters():
        if p.grad is not None:
            out["grad." + name] = pick(name, p.grad.detach().reshape(-1), DUMP_GRAD_ENTRIES)
    total = sum(v.numel() * 4 for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs would write {total} bytes, more than {DUMP_MAX_BYTES}")
    os.makedirs(dirname, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(dirname, name + ".npy"), v.float().cpu().numpy())


def roofline_block(alg_bytes, ms, peak, what):
    """End-to-end HBM roofline of a whole workload: algorithmic (compulsory) bytes / measured time against the measured peak."""
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "alg_bytes": alg_bytes, "ms": ms, "achieved": gbs, "peak": peak, "unit": "GB/s",
            "frac": gbs / peak, "floor_ms": alg_bytes / (peak * 1e9) * 1e3, "what": what}


def torch_eager_gpu_arm(dev, timed, B):
    """Oracle port (plain torch ops) with every tensor on the GPU: hypernet fwd + fc + DecoderGRU + CE + backward, flow mode."""
    from oracle import caption_hn_oracle as O
    c = CFG
    p = O.init_params_pooled(c["D"], c["E"], c["H"], c["V"], L=c["L"], seed=0)
    p = {k: v.to(dev).requires_grad_(True) for k, v in p.items()}
    g = torch.Generator().manual_seed(1234)
    pooled = torch.relu(torch.randn(B, c["D"], generator=g)).to(dev)
    caps = O.synth_captions(B, c["T"], c["V"], g).to(dev)
    h0 = torch.rand(B, c["H"], generator=g).to(dev)

    def step():
        for v in p.values():
            v.grad = None
        logits, _, _ = O.path_pooled(p, p["captioner.embed.weight"][4:5], pooled, caps, h0, L=c["L"], flow=True)
        O.caption_loss(logits, caps, None).backward()

    for _ in range(3):
        step()
    ms = timed(step, 10)
    out = {"pooled_train": B * 10 / (ms * 1e-3), "ms_per_step": ms / 10,
           "what": "oracle port, torch eager CUDA kernels (cuBLAS/ATen), same workloads, fp32 (TF32 off)"}
    del p
    torch.cuda.empty_cache()
    # configs[2]: attention variant, teacher-forced fwd+bwd and greedy decode
    import numpy as np
    pa = O.init_params_attention(2048, 200, 200, 200, c["V"], 200, seed=0)
    pa = {k: v.to(dev).requires_grad_(True) for k, v in pa.items()}
    feats = torch.randn(B, 49, 2048, generator=g).to(dev)

    def astep():
        for v in pa.values():
            v.grad = None
        logits = O.path_attention(pa, pa["captioner.embed.weight"][4:5], feats, caps, 0.0, np.random.RandomState(0))[0]
        O.caption_loss(logits, caps, 0).backward()

    def adec():
        with torch.no_grad():
            O.path_attention(pa, pa["captioner.embed.weight"][4:5], feats, caps, 1.0, np.random.RandomState(0))

    for name, fn in (("attention_train", astep), ("attention_greedy_decode", adec)):
        for _ in range(2):
            fn()
        ms = timed(fn, 5)
        out[name] = B * 5 / (ms * 1e-3)
    return out


def pooled_l2_extras(args, dev, world, timed, rooflines, peak):
    """The reference launcher's own operating point (hypernet.py:209): num_layers = 2 -- 2.78 G hypernet parameters
    (11.1 GB), the second GRU cell reads theta from offset 0 again (utils.py:45,68); L2-streaming multi-layer recurrence."""
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import graphs, parallel as par
    from hypernet_image_captioning_b200.synth import synth_captions
    c = CFG
    B, T, V = args.batch, c["T"], c["V"]
    torch.manual_seed(0)
    with torch.device(dev):
        model = C.HyperNetPooled(c["E"], c["H"], V, None, num_layers=2)
    model.async_hypernet = True
    model.dp_enabled = world > 1
    shared = par.shared_parameters(model)
    if world > 1:
        par.enable_overlap(shared)
    g = torch.Generator().manual_seed(4321)
    pooled = torch.relu(torch.randn(B, c["D"], generator=g)).to(dev)
    caps = synth_captions(B, T, V, g).to(dev)
    h0 = torch.rand(B, c["H"], generator=g).to(dev)

    def train():
        model.zero_grad(set_to_none=True)
        cap = model.forward(model.captioner.embed.weight[4:5])
        loss, _ = cap.forward_loss(model.image_encoder(pooled), caps, h0=h0)
        ((loss / world) if world > 1 else loss).backward()
        if world > 1:
            par.allreduce_shared_grads(shared)

    run = train
    if os.environ.get("CAPHN_BENCH_GRAPH", "1") != "0":
        gtrain = graphs.GraphedStep(train, (), params=list(model.parameters()), release=model.release_graph)
        run = gtrain if gtrain.captured else train
    for _ in range(3):
        run()
    ms = timed(run, args.steps) / args.steps
    hn_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters() if n_.startswith("hn_"))
    w2_b = 4.0 * sum(h_[2].weight.numel() for h_ in model.hn_heads)
    sh_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters()
                     if not n_.startswith("hn_") and not n_.startswith("captioner.lstm_cell") and not n_.startswith("captioner.layers"))
    step_bytes = 2 * hn_b + w2_b + 2 * sh_b + B * (c["D"] * 4.0 + 8.0 * T + 2.0 * T * V * 4.0)
    rooflines["pooled_l2_train_step"] = roofline_block(step_bytes, ms, peak, "num_layers=2 (hypernet.py:209), flow mode fwd+bwd")
    if world > 1:
        par.disable_overlap()
    return {"pooled_l2_train_captions_per_s": B * world / (ms * 1e-3), "pooled_l2_hypernet_params": int(hn_b / 4)}


def attention_extras(args, dev, world, timed, rooflines=None, peak=6537.6):
    """BASELINE configs[2]/[1b]: attention variant (hypernet_attention.HyperNet + AttentionGru), F=E=H=200, P=49, D=2048,
    B=512/GPU, T=20: teacher-forced fwd+bwd (flow, ignore_index=<pad>) and greedy decode (sample_prob=1.0, test_hn.py)."""
    import numpy as np
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200.synth import synth_captions
    B, T, V = args.batch, CFG["T"], CFG["V"]
    torch.manual_seed(0)
    with torch.device(dev):
        model = C.HyperNetAttention(200, 200, 200, V, None)
    model.dp_enabled = world > 1
    g = torch.Generator().manual_seed(4321)
    feats = torch.randn(B, 49, 2048, generator=g).to(dev)
    caps = synth_captions(B, T, V, g).to(dev)

    from hypernet_image_captioning_b200 import parallel as par
    shared = par.shared_parameters(model)
    if world > 1:
        par.enable_overlap(shared)

    def train():
        model.zero_grad(set_to_none=True)
        captioner = model.forward(model.captioner.embed.weight[4:5])
        loss, _, _ = captioner.forward_loss(feats, caps, 0.0, ignore_index=0)
        if world > 1:      # exact global-batch masked mean: weight by this rank's share of the non-pad tokens
            (loss * par.loss_weight(caps, 0)).backward()
            par.allreduce_shared_grads(shared)
        else:
            loss.backward()

    def greedy():
        with torch.no_grad():
            model.async_hypernet = True       # the hypernet streams its weights while the feature branch runs
            captioner = model.forward(model.captioner.embed.weight[4:5])
            out = captioner(feats, caps, 1.0)
            model.async_hypernet = False
            return out

    out = {}
    for name, fn in (("attention_train_captions_per_s", train), ("attention_greedy_decode_captions_per_s", greedy)):
        for _ in range(3):
            fn()
        ms = timed(fn, args.steps)
        out[name] = B * world * args.steps / (ms * 1e-3)
    if os.environ.get("CAPHN_BENCH_GRAPH", "1") != "0":       # the same training step replayed from one CUDA graph
        from hypernet_image_captioning_b200 import graphs
        model.async_hypernet = True       # hypernet / feature branch / recurrence on three streams inside the graph
        gtrain = graphs.GraphedStep(train, (), params=list(model.parameters()), release=model.release_graph)
        model.async_hypernet = False
        if gtrain.captured:
            for _ in range(3):
                gtrain()
            ms = timed(gtrain, args.steps)
            out["attention_train_eager_captions_per_s"] = out["attention_train_captions_per_s"]
            out["attention_train_captions_per_s"] = B * world * args.steps / (ms * 1e-3)
        del gtrain
    if rooflines is not None:
        P, D = 49, 2048
        hn_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters() if n_.startswith("hn_"))
        w2_b = 4.0 * sum(h_[2].weight.numel() for h_ in model.hn_heads)
        sh_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters()
                         if not n_.startswith("hn_") and not n_.startswith("captioner.gru"))
        per_cap_fwd = P * D * 4.0 + 8.0 * T + T * V * 4.0 + T * P * 4.0          # SURVEY 8(d): 1.18 MB
        tr_bytes = 2 * hn_b + w2_b + 2 * sh_b + B * (per_cap_fwd + T * V * 4.0)  # + logits re-read: 1.95 MB / caption
        de_bytes = hn_b + sh_b + B * per_cap_fwd
        rooflines["attention_train_step"] = roofline_block(
            tr_bytes, B * world / out["attention_train_captions_per_s"] * 1e3, peak,
            "configs[2] fwd+bwd, flow mode, compulsory traffic (SURVEY 8(d) worked example: 2.78 GB)")
        rooflines["attention_greedy_decode"] = roofline_block(
            de_bytes, B * world / out["attention_greedy_decode_captions_per_s"] * 1e3, peak,
            "configs[2] greedy decode (sample_prob=1.0), compulsory traffic (SURVEY 8(d): 1.20 GB)")
    if world > 1:
        par.disable_overlap()
    return out


def cc_extras(args, dev, world, timed, rooflines, peak):
    """BASELINE configs[3]: Conceptual-Captions domain-conditioned hypernet (hypernet_attention.HyperNet(cc=True), one-hot
    domain vectors, he = #domains = 100 / 150, cc_train_hypernet.py:86-89,134-153), F=E=H=200, B=512/GPU, T=20, teacher-forced
    fwd+bwd (flow).  G = 1 is the reference's own step (one domain per batch, :136); G = 3 / 100 / 150 put that many domains in
    ONE batch (rows assigned round-robin, SURVEY 8(d)) and run the grouped kernels: one hypernet pass for all G, grouped
    tensor-core x-projection / dX / dW products, per-group weight packs in the recurrence.  Under DP the d(theta) [G, theta]
    all-reduce (144 MB at G = 100) runs on the hypernet stream next to the feature branch's backward."""
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import graphs, parallel as par
    from hypernet_image_captioning_b200.synth import synth_captions
    B, T, V = args.batch, CFG["T"], CFG["V"]
    g = torch.Generator().manual_seed(777)
    feats = torch.randn(B, 49, 2048, generator=g).to(dev)
    caps = synth_captions(B, T, V, g).to(dev)
    out = {}
    for he, Gs in ((100, (1, 3, 100)), (150, (150,))):
        torch.manual_seed(0)
        with torch.device(dev):
            model = C.HyperNetAttention(200, 200, 200, V, None, cc=True, hyper_emb=he)
        model.dp_enabled = world > 1
        shared = par.shared_parameters(model)
        if world > 1:
            par.enable_overlap(shared)
        eye = torch.eye(he, device=dev)
        for G in Gs:
            groups = torch.arange(B) % G                     # host tensor: the batch composition is loader (host) data
            styles = eye[:G].contiguous()

            def train():
                model.zero_grad(set_to_none=True)
                if G == 1:
                    captioner = model.forward(styles[0])                      # 1-D one-hot, as cc_train_hypernet.py:141-143
                    loss, _, _ = captioner.forward_loss(feats, caps, 0.0, ignore_index=0)
                else:
                    captioner = model.forward_grouped(styles)
                    loss, _, _ = captioner.forward_loss(feats, caps, 0.0, ignore_index=0, groups=groups)
                if world > 1:
                    (loss * par.loss_weight(caps, 0)).backward()
                    par.allreduce_shared_grads(shared)
                else:
                    loss.backward()

            run = train
            if os.environ.get("CAPHN_BENCH_GRAPH", "1") != "0":
                model.async_hypernet = True
                gtrain = graphs.GraphedStep(train, (), params=list(model.parameters()), release=model.release_graph)
                model.async_hypernet = False
                run = gtrain if gtrain.captured else train
            for _ in range(3):
                run()
            ms = timed(run, args.steps) / args.steps
            out[f"cc_onehot_he{he}_G{G}_train_captions_per_s"] = B * world / (ms * 1e-3)
            hn_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters() if n_.startswith("hn_"))
            w2_b = 4.0 * sum(h_[2].weight.numel() for h_ in model.hn_heads)
            sh_b = 4.0 * sum(p_.numel() for n_, p_ in model.named_parameters()
                             if not n_.startswith("hn_") and not n_.startswith("captioner.gru"))
            theta = sum(p_.numel() for p_ in model.captioner.gru.parameters())
            per_cap = 49 * 2048 * 4.0 + 8.0 * T + 2.0 * T * V * 4.0 + T * 49 * 4.0
            alg = 2 * hn_b + w2_b + 2 * sh_b + B * per_cap + 2.0 * G * theta * 4.0      # + theta, d(theta) per group
            rooflines[f"cc_he{he}_G{G}_train_step"] = roofline_block(
                alg, ms, peak, f"configs[3], {G} domain(s) in the batch, flow mode fwd+bwd, compulsory traffic")
            run = None
            model.zero_grad(set_to_none=True)
        if world > 1:
            par.disable_overlap()
        del model
        torch.cuda.empty_cache()
    return out


def lstm_extras(args, dev, world, timed):
    """The LSTM captioner of the pooled hypernet (hypernet.py:53, DecoderRNN): same sizes as the headline workload;
    the generated cell is 4H x (E + H) instead of 3H x (E + H), so the hypernet heads are 8.6 GB instead of 6.46 GB."""
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import parallel as par
    from hypernet_image_captioning_b200.synth import synth_captions
    c = CFG
    B, T, V = args.batch, c["T"], c["V"]
    torch.manual_seed(0)
    with torch.device(dev):
        model = C.HyperNetPooled(c["E"], c["H"], V, None, num_layers=c["L"], type="lstm")
    model.async_hypernet = True
    model.dp_enabled = world > 1
    shared = par.shared_parameters(model)
    if world > 1:
        par.enable_overlap(shared)
    g = torch.Generator().manual_seed(4321)
    pooled = torch.relu(torch.randn(B, c["D"], generator=g)).to(dev)
    caps = synth_captions(B, T, V, g).to(dev)

    def train():
        model.zero_grad(set_to_none=True)
        cap = model.forward(model.captioner.embed.weight[4:5])
        loss, _ = cap.forward_loss(model.image_encoder(pooled), caps)
        ((loss / world) if world > 1 else loss).backward()
        if world > 1:
            par.allreduce_shared_grads(shared)

    run = train
    if os.environ.get("CAPHN_BENCH_GRAPH", "1") != "0":
        from hypernet_image_captioning_b200 import graphs
        gtrain = graphs.GraphedStep(train, (), params=list(model.parameters()), release=model.release_graph)
        run = gtrain if gtrain.captured else train
    for _ in range(3):
        run()
    ms = timed(run, args.steps)
    n_head = sum(p_.numel() for n_, p_ in model.named_parameters() if n_.startswith("hn_"))
    return {"lstm_train_captions_per_s": B * world * args.steps / (ms * 1e-3), "lstm_hypernet_params": n_head}


def main():
    args = parse()
    # The contract is ONE JSON line on stdout.  Libraries write banners to file descriptor 1 from native code (the
    # "NCCL version ..." line at communicator creation, on every rank): park fd 1 on stderr while the benchmark runs and
    # hand the real stdout back to Python's sys.stdout only for the final print.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
