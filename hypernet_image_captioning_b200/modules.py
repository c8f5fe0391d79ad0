"""Host-side mirror of the reference module API (constructor / forward signatures and state_dict layout unchanged).

  reference class                                   ->  class here
  hypernet.HyperNet              (hypernet.py:26)    ->  HyperNetPooled  (alias ``hypernet.HyperNet`` in dropin/)
  later.DecoderGRU               (later.py:362)      ->  DecoderGRU
  hypernet_attention.HyperNet    (hypernet_attention.py:32) -> HyperNetAttention   (modules_attention.py)
  models.decoderlstm.AttentionGru (models/decoderlstm.py:11) -> AttentionGru       (modules_attention.py)

All arithmetic runs in the CUDA kernels behind the C-ABI; the nn.Module objects here only own parameters.
``grad_mode``: "flow" (default) lets the caption loss reach the hypernet heads through the generated weights (the
intended semantics, BASELINE.json north_star); "literal" reproduces the reference's graph cut (utils.py:57): the
generated weights become leaves and their gradient lands on ``captioner.<cell>.weight_*.grad``.
"""
from typing import List

import torch
from torch import nn

from . import functional as Fn
from . import ops, streams

try:  # the reference classes are LightningModules; use the real base when it exists
    import pytorch_lightning as _pl
    _Base = _pl.LightningModule
except Exception:  # noqa: BLE001
    class _Base(nn.Module):
        def __init__(self):
            super().__init__()
            object.__setattr__(self, "hparams", {})

        def log(self, *a, **k):
            pass

        @property
        def device(self):
            return next(self.parameters()).device


class RowsLinear(nn.Linear):
    """nn.Linear of the hypernet (``hn_base`` / ``hn_heads`` layers; same parameters, same ``state_dict`` keys) whose
    ``forward`` runs the weight-streaming kernels.  ``HyperNet.forward`` does not go through it (it runs the whole stack as
    one autograd node); this is for callers that apply the layers themselves -- ``train_init.py:78-91`` calls
    ``hn_base(style_embed)`` and ``hn_heads[i](base)`` directly in its regression pre-training loop."""

    def forward(self, x):
        x2 = x.reshape(-1, x.shape[-1])
        if x2.shape[0] > 8 or self.weight.dtype != torch.float32:
            y = Fn.linear(x2.to(torch.float32), self.weight.to(torch.float32), self.bias.to(torch.float32))
        else:
            y = Fn.rows_linear(x2.to(torch.float32).contiguous(), self.weight, self.bias, leaky=False)
        return y.reshape(*x.shape[:-1], self.out_features)


def _hn_params(hn) -> List[torch.Tensor]:
    ps = [hn.hn_base[0].weight, hn.hn_base[0].bias, hn.hn_base[2].weight, hn.hn_base[2].bias]
    for head in hn.hn_heads:
        ps += [head[0].weight, head[0].bias, head[2].weight, head[2].bias]
    return ps


class _HyperNetMixin:
    """theta generation + injection shared by both variants (reference utils.py:24-69 flip/set_all_parameters)."""

    grad_mode = "flow"
    dp_group = None      # set dp_enabled = True under torch.distributed to all-reduce d(theta) (parallel.py)
    dp_enabled = False

    # "materialize" (default): .grad of every hypernet parameter is a dense tensor, as torch autograd gives.
    # "lowrank": the backward keeps dW2 = dtheta^T a of the large head matrices as the pair (dtheta, a) on
    # ``param.grad_lowrank`` (param.grad stays None) -- for caphn.FusedAdam, which forms the gradient on the fly.
    head_grad_mode = "materialize"
    lowrank_min_numel = 1 << 22

    # True: ``forward(x)`` launches the hypernet on a side stream and returns at once; the captioner waits for the generated
    # weights right before it needs them, so whatever it runs first (feature_fc, the input gather) overlaps with the weight
    # streaming, and the autograd engine runs the head backward on that stream too (streams.py).  Opt-in, because code that
    # reads ``captioner.<cell>.weight_*`` directly after ``forward`` must then call ``sync_generated()`` first.
    async_hypernet = False

    def sync_generated(self):
        """Order the current stream after an asynchronous hypernet forward (no-op otherwise)."""
        streams.wait_pending()

    def zero_grad(self, set_to_none: bool = True):
        super().zero_grad(set_to_none)
        for p in self.parameters():            # rank-G gradients live beside .grad
            if getattr(p, "grad_lowrank", None) is not None:
                p.grad_lowrank = None

    def release_graph(self):
        """Forget the generated weights of the last ``forward`` (flow mode: they carry the hypernet's autograd graph, which
        the captioner otherwise keeps alive until the next ``forward``).  The injected ``captioner.<cell>.weight_*`` values
        stay, as in the reference."""
        self.captioner._generated = None
        self.captioner._generated_groups = None

    def _generate_and_inject(self, x: torch.Tensor, grouped: bool = False):
        """theta (+ its per-cell views, + the copy into the captioner's cell parameters) -- on the hypernet side stream when
        ``async_hypernet`` is set."""
        streams.clear_ranges()      # readiness marks of an earlier forward must not be mistaken for this one's
        def run():
            theta = self.generate_theta(x)
            if grouped:
                self.captioner._theta_groups = theta        # [G, theta]: the grouped kernels take the whole matrix
                return [self._split_theta(theta[g]) for g in range(theta.shape[0])]
            if hasattr(self, "_split_theta_node"):
                return self._split_theta_node(theta)
            return self._split_theta(theta[0], write_params=True)
        if self.async_hypernet and x.is_cuda and streams.ENABLED is not False:      # explicit opt-in: also in eager mode
            with streams.fork("hypernet") as s:
                out = run()
            streams.defer(s)
            return out
        return run()

    def generate_theta(self, x: torch.Tensor) -> torch.Tensor:
        x2 = x.reshape(1, -1) if x.dim() == 1 else x
        x2 = x2.to(torch.float32).contiguous()
        Fn.LOWRANK_MIN_NUMEL = self.lowrank_min_numel if self.head_grad_mode == "lowrank" else 0
        if self.grad_mode == "literal":
            with torch.no_grad():
                return Fn.hypernet_theta(x2, _hn_params(self))
        if self.dp_enabled:
            from . import parallel
            world = parallel.world_size(self.dp_group)
            if world > 1 and x2.requires_grad:
                leaf = parallel.route_style_grad(x) if self.grad_mode == "flow" else None
                if leaf is not None:      # style = a row of a shared parameter: keep that parameter's gradient "early"
                    x2 = (leaf.reshape(1, -1) if leaf.dim() == 1 else leaf).to(torch.float32).contiguous()
                else:
                    x2 = parallel.ScaleGradFn.apply(x2, 1.0 / world)   # the style gradient leaves the replicated hypernet already global
        ps = _hn_params(self)
        if x2.shape[0] > 8 and ps[0].dtype == torch.float32:
            # many style vectors: the layers as dense tensor-core GEMMs (one pass over the head weights for all G)
            from .grouped import HyperNetThetaManyFn
            theta = HyperNetThetaManyFn.apply(x2, *ps)
        else:
            theta = Fn.hypernet_theta(x2, ps)
        if self.dp_enabled:
            theta = parallel.allreduce_grad(theta, self.dp_group)
        return theta

    def regression_loss(self, style_embed: torch.Tensor, target_params):
        """Hypernet regression pre-training objective of train_init.py:70-123: sum over the generated GRU parameters of
        MSE(head_i(hn_base(style)).flatten(), target_i.flatten()).  ``target_params`` = the pretrained cell's parameters
        in named_parameters() order (weight_ih, weight_hh, bias_ih, bias_hh[, next cell ...]).  The head forward /
        backward run in the weight-streaming kernels; the MSE itself is a few hundred thousand elements."""
        theta = self.generate_theta(style_embed)[0]
        loss, a = theta.new_zeros(()), 0
        for tgt in target_params:
            n = tgt.numel()
            loss = loss + torch.nn.functional.mse_loss(theta[a:a + n], tgt.detach().reshape(-1).to(theta.dtype))
            a += n
        if a != theta.numel():
            raise ValueError(f"target parameters cover {a} of {theta.numel()} generated values")
        return loss

    def set_precision(self, mode: str):
        """"fp32" (default; parity mode) or "bf16": the hypernet base/head parameters -- and therefore their gradients --
        are stored in bf16 (half the HBM traffic of the dominant kernels) and the decoder's tensor-core products use
        plain bf16 operands; activations, theta, the recurrent state and every accumulation stay fp32."""
        dt = {"fp32": torch.float32, "bf16": torch.bfloat16}[mode]
        self.hn_base.to(dt)
        self.hn_heads.to(dt)
        ops.set_precision(mode)
        return self

    def forward_grouped(self, X: torch.Tensor):
        """Grouped generalisation (BASELINE.json north_star "per-style grouped"): ``X`` = [G, he] style/domain vectors.
        One pass over the hypernet weights generates all G weight sets (the reference would stream them G times, one
        ``forward`` per style); the captioner then decodes every batch row with the weights of its group:
        ``captioner(features, captions, ..., groups=group_ids)``.  Oracle = one reference call per group, concatenated."""
        self.captioner._generated_groups = self._generate_and_inject(X, grouped=True)
        return self.captioner


def _run_grouped(fn, groups: torch.Tensor, tensors, n_groups: int):
    """Apply ``fn(g, *row_subsets)`` per group and put the rows back in their original order (differentiable glue)."""
    groups = groups.to(tensors[0].device)
    order = torch.argsort(groups, stable=True)
    counts = torch.bincount(groups, minlength=n_groups).tolist()
    outs, start = None, 0
    for g, n in enumerate(counts):
        if n == 0:
            continue
        idx = order[start:start + n]
        start += n
        res = fn(g, *[t.index_select(0, idx) for t in tensors])
        res = res if isinstance(res, tuple) else (res,)
        outs = [[r] for r in res] if outs is None else [o + [r] for o, r in zip(outs, res)]
    inv = torch.empty_like(order)
    inv[order] = torch.arange(order.numel(), device=order.device)
    return tuple(torch.cat(o, 0).index_select(0, inv) for o in outs)


def _beam_search(setup, beam_size, V, max_steps, end_sentence, sync_every):
    """Device-resident beam search of HyperNet.test_step (hypernet_attention.py:247-326) for B images at once, around a
    captioner's decoder step; returns a list of B results, each the best complete token sequence (leading 0, trailing
    ``end_sentence``) or ``None`` where a beam is still open after ``max_steps`` + 1 steps.

    ``setup(rep)`` runs after the argument checks and returns ``(h0 [B, H], step_fn)``; ``rep`` repeats a [B, ...] tensor
    for the beams (rows b*k + j: beam j of image b).  ``step_fn(step, h, prev_tok, words)`` runs decoder step ``step``
    (1-based) from the state ``h`` [B*k, H] -- ``rep(h0)`` at step 1 -- and the tokens the previous step chose
    (``prev_tok`` int32, or ``words``: the embedding rows to feed, -1 = zero vector) and returns ``(logits [B*k, V],
    h_out [B*k, H])``; it must not write ``h``.  Between steps ONE kernel per step (csrc/beam.cu, a CTA per image) does
    the reference's host bookkeeping on the device; the host reads the results in one copy at the end and only peeks at
    an 'all images finished' flag every ``sync_every`` steps to stop early."""
    k = int(beam_size)
    if not 1 <= k <= 8:
        raise ValueError(f"beam_size {k} outside [1, 8]")
    if k > V:
        raise ValueError(f"beam_size {k} exceeds the vocabulary size {V}")
    rep = lambda x: x.unsqueeze(1).expand(-1, k, *x.shape[1:]).reshape(x.shape[0] * k, *x.shape[1:]).contiguous()
    h0, step_fn = setup(rep)
    (B, H), dev = h0.shape, h0.device
    R, L = B * k, int(max_steps) + 3
    h = rep(h0)
    i32 = lambda *s: torch.zeros(*s, device=dev, dtype=torch.int32)
    h_next = torch.zeros(R, H, device=dev, dtype=torch.float32)     # rows of finished beams stay finite
    scores = torch.zeros(R, device=dev, dtype=torch.float32)
    live = torch.full((B,), k, device=dev, dtype=torch.int32)
    prev_tok, ncomp, failed = i32(R), i32(B), i32(B)
    words = torch.full((R,), -1, device=dev, dtype=torch.int64)  # every beam starts from word 0 -> zero embeddings (:265-266)
    seq = [i32(R, L), i32(R, L)]                                  # histories start with the token 0
    comp_score = torch.zeros(R, device=dev, dtype=torch.float32)
    comp_seq, comp_len = i32(R, L), i32(R)
    n_steps = int(max_steps) + 1
    for step in range(1, n_steps + 1):
        logits, h_out = step_fn(step, h, prev_tok, words)
        ops.beam_step(logits, h_out, h_next, scores, live, prev_tok, words, seq[(step - 1) & 1], seq[step & 1],
                      comp_score, comp_seq, comp_len, ncomp, failed, k, step, int(end_sentence), step == n_steps)
        h = h_next
        if sync_every and step % sync_every == 0 and step < n_steps and int(live.max()) == 0:
            break
    nc, fl = ncomp.cpu().tolist(), failed.cpu().tolist()           # the one read-back of the search
    cs, cq, cl = comp_score.cpu().view(B, k), comp_seq.cpu().view(B, k, L), comp_len.cpu().view(B, k)
    out = []
    for b in range(B):
        if fl[b] or nc[b] == 0:
            out.append(None)
            continue
        sc = cs[b, :nc[b]].tolist()
        j = sc.index(max(sc))                                     # first maximum, as list.index does (:319-321)
        out.append(cq[b, j, :int(cl[b, j])].tolist())
    return out


class PooledFeatureEncoder(nn.Module):
    """Stands in for the frozen ResNet-101 + trainable fc of hypernet.py:40-48: the CNN trunk is out of scope
    (BASELINE.json), so ``forward`` takes the precomputed pooled 2048-d feature and applies ``fc``."""

    def __init__(self, num_ftrs, embed_size):
        super().__init__()
        self.fc = nn.Linear(num_ftrs, embed_size)

    def forward(self, pooled):
        return Fn.linear(pooled, self.fc.weight, self.fc.bias)


class DecoderGRU(nn.Module):
    """Drop-in for later.py:362 DecoderGRU (constructor signature, forward/infer signatures, state_dict keys).

    ``data/vocab.pkl`` is *not* opened (reference later.py:372 loads it only for the discarded per-token text loop at
    :451-452); the hard-coded V = 9684 of :449 is likewise not required."""

    def __init__(self, embed_size, hidden_size, vocab_size, num_layers=1, dropout=False):
        super().__init__()
        self.embed_size, self.hidden_size, self.vocab_size = embed_size, hidden_size, vocab_size
        self.dropout, self.num_layers = dropout, num_layers
        self.lstm_cell = nn.GRUCell(input_size=embed_size, hidden_size=hidden_size)
        self.layers = None
        if num_layers > 1:
            self.layers = nn.ModuleList([nn.GRUCell(hidden_size, hidden_size) for _ in range(num_layers - 1)])
        self.fc_out = nn.Linear(hidden_size, vocab_size)
        self.embed = nn.Embedding(vocab_size, embed_size)
        self._generated = None  # per-cell (W_ih, W_hh, b_ih, b_hh) carrying the hypernet graph (flow mode)
        self._generated_groups = None  # list over style groups of the above (forward_grouped)
        self._theta_groups = None

    def _cells(self, group=None):
        if group is not None:
            return self._generated_groups[group]
        if self._generated is not None:
            return self._generated
        cells = [self.lstm_cell] + (list(self.layers) if self.layers else [])
        return [(c.weight_ih, c.weight_hh, c.bias_ih, c.bias_hh) for c in cells]

    def _h0(self, features):
        # reference later.py:393-394: global CPU RNG, then type_as(features).  Same CPU random stream, but drawn into
        # pinned memory and copied asynchronously: a pageable copy would block the host until the device has drained.
        h0 = torch.rand(size=(features.size(0), self.hidden_size), pin_memory=features.is_cuda)
        return h0.to(features.device, features.dtype, non_blocking=True)

    def forward(self, features, captions, teacher_forcing=True, h0=None, groups=None):
        if not teacher_forcing:
            raise NotImplementedError("multinomial-sampled decoding (later.py:424-434) is outside the hot path")
        streams.wait_pending()      # an asynchronous hypernet forward (async_hypernet) must have produced the weights
        if groups is not None:
            if h0 is None:
                h0 = self._h0(features)
            if self._grouped_kernels_ok(features):
                # many-style batch on the grouped kernels (grouped.py): batch sorted by group, one grouped tensor-core launch
                # per time-batched product, a recurrence that runs every row tile with THEIR group's W_hh
                from . import grouped as Gp
                Theta = self._theta_groups
                plan = Gp.GroupPlan.get(groups, Theta.shape[0], captions.shape[1], features.device)
                fs = Gp.RowPermuteFn.apply(features, plan.order, plan.inv)
                hs = Gp.RowPermuteFn.apply(h0, plan.order, plan.inv)
                return self._grouped_fns()[0].apply(plan, fs, captions.index_select(0, plan.order), hs, Theta,
                                                    self.embed.weight, self.fc_out.weight, self.fc_out.bias)
            return _run_grouped(lambda g, f, c, h: self._forward_one(f, c, h, self._cells(g)), groups,
                                [features, captions, h0], len(self._generated_groups))[0]
        if h0 is None:
            h0 = self._h0(features)
        return self._forward_one(features, captions, h0, self._cells())

    def _grouped_kernels_ok(self, features):
        """Grouped kernels: single-layer GRU captioner whose W_hh fits the weights-resident cluster kernel, fp32 mode."""
        return (self.num_layers == 1 and getattr(self, "_theta_groups", None) is not None and features.is_cuda
                and ops.TC_SPLIT and ops.gru_cluster_size(self.hidden_size) > 0)

    def _grouped_fns(self):
        """(forward node, forward + loss node) of the grouped kernels for this cell type."""
        from . import grouped as Gp
        return Gp.DecoderGRUGroupedFn, Gp.DecoderGRUGroupedLossFn

    def _forward_loss_grouped(self, features, captions, h0, ignore_index, groups):
        """forward_loss for a many-style batch: one autograd node (grouped.py) whose loss and logits are the numbers of
        ``cross_entropy(self(features, captions, h0=h0, groups=groups), captions, ignore_index)``."""
        fallback = "use forward(..., groups=...) + cross_entropy instead"
        if self.num_layers > 1:
            raise NotImplementedError(f"forward_loss(groups=...) covers single-layer captioners; {fallback}")
        Theta = getattr(self, "_theta_groups", None)
        if Theta is None:
            raise ValueError("forward_loss(groups=...) needs the weights of every group: call the hypernet's "
                             "forward_grouped(X) after its last forward(x)")
        from . import grouped as Gp
        plan = Gp.GroupPlan.get(groups, Theta.shape[0], captions.shape[1], features.device)     # checks the group ids
        if not self._grouped_kernels_ok(features):
            raise NotImplementedError("forward_loss(groups=...) runs on the grouped CUDA kernels: CUDA tensors, fp32 "
                                      f"precision and a hidden size their recurrence covers; {fallback}")
        if h0 is None:
            h0 = self._h0(features)
        streams.wait_pending()
        fs = Gp.RowPermuteFn.apply(features, plan.order, plan.inv)
        hs = Gp.RowPermuteFn.apply(h0, plan.order, plan.inv)
        return self._grouped_fns()[1].apply(ignore_index, plan, captions.contiguous(), fs,
                                            captions.index_select(0, plan.order), hs, Theta, self.embed.weight,
                                            self.fc_out.weight, self.fc_out.bias)

    def forward_loss(self, features, captions, h0=None, ignore_index=None, groups=None):
        """Teacher-forced forward fused with the mean cross-entropy of hypernet.py:145 (``ignore_index=None``: no
        masking): returns ``(loss, logits)``.  Same numbers as ``cross_entropy(self(features, captions), captions)``
        but one autograd node whose backward writes the softmax gradient straight into tensor-core operands.
        ``groups`` ([B] group id per row, after the hypernet's ``forward_grouped``): many-style batch, single layer, fp32
        mode, CUDA tensors; elsewhere ``NotImplementedError`` (use ``forward(..., groups=...)`` + ``cross_entropy``)."""
        if groups is not None:
            return self._forward_loss_grouped(features, captions, h0, ignore_index, groups)
        if h0 is None:
            h0 = self._h0(features)
        # (no wait_pending here: the fused node waits for the generated weights slice by slice, Fn._gru_decoder_forward)
        flat = [w for cell in self._cells() for w in cell]
        return Fn.DecoderGRULossFn.apply(ignore_index, features, captions, h0, self.embed.weight, self.fc_out.weight,
                                         self.fc_out.bias, *flat)

    def _forward_one(self, features, captions, h0, cells):
        if len(cells) > 4:
            raise NotImplementedError("DecoderGRU with more than 4 layers")
        flat = [w for cell in cells for w in cell]
        return Fn.DecoderGRUSeqFn.apply(features, captions, h0, self.embed.weight, self.fc_out.weight,
                                        self.fc_out.bias, *flat)

    @torch.no_grad()
    def infer(self, features, max_len=50, h0=None):
        """Greedy decode, reference later.py:459-490: argmax feedback, first cell only, returns softmax probs.
        The whole loop (~5 launches per step) is captured into a CUDA graph per (batch, max_len) and replayed."""
        from . import graphs
        streams.wait_pending()
        W_ih, W_hh, b_ih, b_hh = [t.detach().contiguous() for t in self._cells()[0]]
        if h0 is None:
            h0 = self._h0(features)
        key = ("DecoderGRU.infer", id(self), tuple(features.shape), int(max_len), features.device.index,
               self.embed.weight.data_ptr(), self.fc_out.weight.data_ptr(), self.fc_out.bias.data_ptr())
        return graphs.graphed_call(key, lambda f, h, wi, wh, bi, bh: self._infer_loop(f, h, wi, wh, bi, bh, max_len),
                                   [features.contiguous().float(), h0.contiguous().float(), W_ih, W_hh, b_ih, b_hh])[0]

    def _infer_loop(self, features, h0, W_ih, W_hh, b_ih, b_hh, max_len):
        B, H = features.size(0), self.hidden_size
        emb, fc_w, fc_b = self.embed.weight.detach(), self.fc_out.weight.detach(), self.fc_out.bias.detach()
        WhhT = ops.transpose_pad(W_hh, ops.round4(3 * H))
        outputs = torch.empty(B, max_len, self.vocab_size, device=features.device, dtype=torch.float32)
        h = h0.contiguous()
        x = features.contiguous()
        logits = torch.empty(B, self.vocab_size, device=features.device, dtype=torch.float32)
        xproj, vocab = ops.LinearPlan(W_ih, b_ih), ops.LinearPlan(fc_w, fc_b)   # weight splits made once, not per step
        # From step 1 on the input is a word embedding, so its projection is a row of  P = Emb W_ih^T + b_ih  [V, 3H]:
        # one GEMM per call instead of (gather + operand split + GEMM) per step -- same products, same order per element.
        table = ops.linear(emb, W_ih, b_ih) if ops.use_projection_table(B, max_len, emb.shape[0]) else None
        words = None
        # Fast path (projection table + tensor-core vocabulary projection): the arg-max that feeds step t+1 comes out of the
        # vocabulary GEMM's epilogue as per-tile partials and is finished inside the gather of the next input row, so the
        # softmax that produces the RETURNED probabilities (later.py:472) is off the dependency chain: the logits are written
        # straight into outputs[:, t] and normalised in place on a side stream while the next step runs.
        fast = table is not None and ops._tc_ok(B, self.vocab_size, H)
        if not fast:
            for t in range(max_len):
                if t == 0:
                    GI = xproj(x)
                elif table is not None:
                    GI = ops.gather_rows(table, words)
                else:
                    GI = xproj(ops.gather_rows(emb, words))
                Hall, _, _, _ = ops.gru_seq_fwd(GI, WhhT, b_hh, h, 1, save=False, want_bm=False)
                h = Hall[1]
                vocab(h, out=logits)
                _, words = ops.softmax_argmax(logits, want_probs=True, probs_out=outputs[:, t, :])
            return outputs
        # The dependency chain -- ONE fused launch per step for (arg-max finish, table gather, GRU cell, bf16 operand rows of
        # the new state: ops.gru_decode_step) followed by the vocabulary GEMM -- runs on a HIGH-PRIORITY stream; the in-place
        # softmax of each step's logits follows on the caller's stream, so its 512 CTAs fill the gaps of the chain instead of
        # delaying it.
        nslot = 2 * ((self.vocab_size + 127) // 128)
        pv = torch.empty(B, nslot, device=x.device, dtype=torch.float32)
        pi = torch.empty(B, nslot, device=x.device, dtype=torch.int32)
        Kp = ops.round64(H)
        hhi = torch.empty(B, Kp, device=x.device, dtype=torch.bfloat16)
        hlo = torch.empty(B, Kp, device=x.device, dtype=torch.bfloat16) if ops.TC_SPLIT else None
        hop = ops.SplitOperand(hhi, hlo, B, H, Kp)
        hbuf = [torch.empty(B, H, device=x.device, dtype=torch.float32) for _ in range(2)]
        GIb = torch.empty(B, 3 * H, device=x.device, dtype=torch.float32)
        fused_step = ops.gru_decode_step_ok(H, self.vocab_size)      # else: arg-max finish + gather, GRU step, operand split as three launches
        nparts = 0
        import contextlib
        cur = torch.cuda.current_stream()
        chain = streams.side("decode_chain", priority=-1) if streams.enabled(x) else None     # None: everything in order
        if chain is not None:
            chain.wait_stream(cur)
        for t in range(max_len):
            with (torch.cuda.stream(chain) if chain is not None else contextlib.nullcontext()):
                lg = outputs[:, t, :]
                if fused_step:
                    hn = hbuf[t & 1]
                    ops.gru_decode_step(xproj(x) if t == 0 else None, pv, pi, nparts, table, W_hh, b_hh, h, hn, hhi, hlo)
                    h = hn
                    nparts = ops.gemm_tc_amax(hop, vocab.operand(), fc_b, lg, pv, pi)
                else:
                    if t == 0:
                        GI = xproj(x)
                    else:
                        ops.argmax_finish_gather(pv, pi, nparts, table, None, GIb)
                        GI = GIb
                    h = ops.gru_seq_fwd(GI, WhhT, b_hh, h, 1, save=False, want_bm=False)[0][1]
                    nparts = ops.gemm_tc_amax(ops.split_bf16(h), vocab.operand(), fc_b, lg, pv, pi)
            if chain is not None:
                cur.wait_stream(chain)                               # (up to this step's GEMM)
            ops.softmax_argmax(lg, want_probs=True, probs_out=lg, want_argmax=False)         # in place, off the chain
        return outputs

    @torch.no_grad()
    def beam_search_batched(self, features, beam_size=3, end_sentence=2, max_steps=50, h0=None, sync_every=8):
        """Beam search over the decoder step of ``infer`` for a whole batch, device-resident: ``features`` [B, E] (what
        ``infer`` takes, ``image_encoder(pooled)``) -> list of B results, each the best complete token sequence (leading 0,
        trailing ``end_sentence``) or ``None`` where a beam is still open after ``max_steps`` + 1 steps.  Same result format
        and bookkeeping as ``AttentionGru.beam_search_batched`` (hypernet_attention.py:268-312: step 1 ranks row 0 only,
        summed log-probabilities without length normalisation, finished beams leave, ties to the lower flat index).

        Step 1 feeds ``features`` with ``h0`` (``None``: ``torch.rand(B, H)`` as ``infer`` draws it), each image's row
        repeated for its k beams; later steps feed Emb[w] for the word w each beam chose -- the true word, without the
        attention search's zero-embedding quirk (hypernet_attention.py:265-266), so ``beam_size=1`` gives ``infer``'s
        greedy tokens.  First cell only, as in ``infer``.  Per step: one fused decode-step launch (projection-table row
        -> GRU cell -> bf16 operand rows), the vocabulary GEMM and the bookkeeping kernel (csrc/beam.cu); the host reads
        the results once at the end and peeks at an 'all images finished' flag every ``sync_every`` steps."""
        streams.wait_pending()
        W_ih, W_hh, b_ih, b_hh = [t.detach().contiguous() for t in self._cells()[0]]
        if features.dim() != 2 or features.shape[1] != W_ih.shape[1]:
            raise ValueError(f"beam_search_batched expects features [B, {W_ih.shape[1]}], got {list(features.shape)}")
        H, V = self.hidden_size, self.vocab_size

        def setup(rep):
            feats = features.contiguous().float()
            h_init = self._h0(feats) if h0 is None else h0
            dev = feats.device
            emb, fc_w, fc_b = self.embed.weight.detach(), self.fc_out.weight.detach(), self.fc_out.bias.detach()
            xproj, vocab = ops.LinearPlan(W_ih, b_ih), ops.LinearPlan(fc_w, fc_b)
            table = ops.linear(emb, W_ih, b_ih)                       # [V, 3H]: the input projection of every word
            GI0 = rep(xproj(feats))
            R = GI0.shape[0]
            fused = ops.gru_decode_step_tok_ok(H)                     # else: table gather + GRU step as two launches
            hop = hhi = hlo = None                                    # hop: the new state's operand rows for the GEMM
            if fused:
                hout = torch.empty(R, H, device=dev, dtype=torch.float32)
                if ops._tc_ok(R, V, H):
                    Kp = ops.round64(H)
                    hhi = torch.empty(R, Kp, device=dev, dtype=torch.bfloat16)
                    hlo = torch.empty(R, Kp, device=dev, dtype=torch.bfloat16) if ops.TC_SPLIT else None
                    hop = ops.SplitOperand(hhi, hlo, R, H, Kp)
            else:
                WhhT = ops.transpose_pad(W_hh, ops.round4(3 * H))
            logits = torch.empty(R, V, device=dev, dtype=torch.float32)

            def step_fn(step, h, prev_tok, words):                    # (``words`` is the attention search's input)
                if fused:
                    if step == 1:
                        ops.gru_decode_step(GI0, None, None, 0, None, W_hh, b_hh, h, hout, hhi, hlo)
                    else:
                        ops.gru_decode_step_tok(prev_tok, table, W_hh, b_hh, h, hout, hhi, hlo)
                    h_out = hout
                else:
                    GI = GI0 if step == 1 else ops.gather_rows(table, prev_tok.long())
                    h_out = ops.gru_seq_fwd(GI, WhhT, b_hh, h, 1, save=False, want_bm=False)[0][1]
                if hop is not None:
                    ops.gemm_tc(hop, vocab.operand(), bias=fc_b, out=logits)
                else:
                    vocab(h_out, out=logits)
                return logits, h_out
            return h_init.contiguous().float(), step_fn
        return _beam_search(setup, beam_size, V, max_steps, end_sentence, sync_every)


class DecoderRNN(DecoderGRU):
    """Drop-in for later.py:227 DecoderRNN: the LSTM captioner the pooled hypernet builds when ``type != 'gru'``
    (hypernet.py:50-53).  Same attribute names as the reference (``lstm_cell``, ``layers``, ``fc_out``, ``embed``);
    (h, c) start at zero (later.py:256-259: no RNG draw); extra cells are applied as ``(h, c) = cell(h, (h, c))``."""

    def __init__(self, embed_size, hidden_size, vocab_size, num_layers=1, dropout=False):
        super().__init__(embed_size, hidden_size, vocab_size, num_layers=num_layers, dropout=dropout)
        self.lstm_cell = nn.LSTMCell(input_size=embed_size, hidden_size=hidden_size)
        if num_layers > 1:
            self.layers = nn.ModuleList([nn.LSTMCell(hidden_size, hidden_size) for _ in range(num_layers - 1)])
        # re-register in the reference's order: lstm_cell, layers, fc_out, embed (later.py:241-249)
        fc_out, embed = self.fc_out, self.embed
        del self.fc_out, self.embed
        self.fc_out, self.embed = fc_out, embed

    def _h0(self, features):
        return torch.zeros(features.size(0), self.hidden_size, device=features.device, dtype=features.dtype)

    def beam_search_batched(self, *args, **kwargs):
        raise NotImplementedError("beam search is implemented for the GRU captioner (DecoderGRU) only: the LSTM cell state "
                                  "would have to follow the beams, and there is no LSTM decode-step kernel")

    def _grouped_kernels_ok(self, features):
        """Grouped kernels: single-layer LSTM captioner whose recurrence fits one CTA's shared memory, fp32 mode."""
        return (self.num_layers == 1 and getattr(self, "_theta_groups", None) is not None and features.is_cuda
                and ops.TC_SPLIT and ops.lstm_seq_fits(self.hidden_size))

    def _grouped_fns(self):
        from . import grouped as Gp
        return Gp.DecoderRNNGroupedFn, Gp.DecoderRNNGroupedLossFn

    def forward_loss(self, features, captions, h0=None, ignore_index=None, groups=None):
        if groups is not None:
            return self._forward_loss_grouped(features, captions, h0, ignore_index, groups)
        if h0 is None:
            h0 = self._h0(features)
        streams.wait_pending()
        flat = [w for cell in self._cells() for w in cell]
        return Fn.DecoderRNNLossFn.apply(ignore_index, features, captions, h0, self.embed.weight, self.fc_out.weight,
                                         self.fc_out.bias, *flat)

    def _forward_one(self, features, captions, h0, cells):
        if len(cells) > 4:
            raise NotImplementedError("DecoderRNN with more than 4 layers")
        flat = [w for cell in cells for w in cell]
        return Fn.DecoderRNNSeqFn.apply(features, captions, h0, self.embed.weight, self.fc_out.weight,
                                        self.fc_out.bias, *flat)

    def _infer_loop(self, features, h0, W_ih, W_hh, b_ih, b_hh, max_len):
        """Greedy decode of later.py:326-360: argmax feedback, first cell only, returns softmax probs."""
        B, H = features.size(0), self.hidden_size
        emb, fc_w, fc_b = self.embed.weight.detach(), self.fc_out.weight.detach(), self.fc_out.bias.detach()
        WhhT = ops.transpose_pad(W_hh, ops.round4(4 * H))
        outputs = torch.empty(B, max_len, self.vocab_size, device=features.device, dtype=torch.float32)
        h, c = h0.contiguous(), None
        x = features.contiguous()
        logits = torch.empty(B, self.vocab_size, device=features.device, dtype=torch.float32)
        xproj, vocab = ops.LinearPlan(W_ih, b_ih), ops.LinearPlan(fc_w, fc_b)
        table = ops.linear(emb, W_ih, b_ih) if ops.use_projection_table(B, max_len, emb.shape[0]) else None   # [V, 4H]
        words = None
        for t in range(max_len):
            if t == 0:
                GI = xproj(x)
            elif table is not None:
                GI = ops.gather_rows(table, words)
            else:
                GI = xproj(ops.gather_rows(emb, words))
            Hall, _, _, _, c = ops.lstm_seq_fwd(GI, WhhT, b_hh, h, 1, save=False, want_bm=False, c0=c, want_c=True)
            h = Hall[1]
            vocab(h, out=logits)
            _, words = ops.softmax_argmax(logits, want_probs=True, probs_out=outputs[:, t, :])
        return outputs


class HyperNetPooled(_HyperNetMixin, _Base):
    """Drop-in for hypernet.py:26 HyperNet (pooled-feature variant)."""

    def __init__(self, embed_size, hidden_size, vocab_size, vocab, num_layers=1, type='gru', lr=1e-6):
        super().__init__()
        self.hparams['vocab_size'] = vocab_size
        self.hparams['embed_size'] = embed_size
        self.hparams['hidden_size'] = hidden_size
        self.vocab = vocab
        self.hparams['lr'] = lr
        self.hparams['num_layers'] = num_layers
        self.teacher_forcing_proba = 1.0
        self.image_encoder = PooledFeatureEncoder(2048, embed_size)
        if type == 'gru':       # hypernet.py:50-53
            self.captioner = DecoderGRU(embed_size, hidden_size, vocab_size, num_layers=num_layers, dropout=False)
        else:
            self.captioner = DecoderRNN(embed_size, hidden_size, vocab_size, num_layers=num_layers)
        E = embed_size
        self.hn_base = nn.Sequential(RowsLinear(E, 4 * E), nn.LeakyReLU(), RowsLinear(4 * E, 8 * E), nn.LeakyReLU())
        heads = []
        for name, W in self.captioner.named_parameters():  # hypernet.py:62-89
            if name in ('embed.weight', 'fc_out.weight', 'fc_out.bias'):
                continue
            w = W.numel()
            if w < 8 * E:
                dims = (8 * E, w, w)
            elif w // 8 < 8 * E:
                dims = (8 * E, 8 * E, 8 * E)
            else:
                dims = (8 * E, w // 8, w // 8)
            heads.append(nn.Sequential(RowsLinear(dims[0], dims[1]), nn.LeakyReLU(), RowsLinear(dims[2], w)))
        self.hn_heads = nn.ModuleList(heads)

    def forward(self, x):
        """theta = heads(base(x)); inject into the captioner's GRU cells; returns self.captioner (hypernet.py:104-114)."""
        gen = self._generate_and_inject(x)
        self.captioner._generated = gen if self.grad_mode == "flow" else None
        self.captioner._generated_groups = None
        self.captioner._theta_groups = None
        return self.captioner

    def _split_theta_node(self, theta):
        """Single-style form of ``_split_theta(theta[0], write_params=True)`` as one autograd node (Fn.ThetaSplitFn)."""
        cells_mod = [self.captioner.lstm_cell] + (list(self.captioner.layers) if self.captioner.layers else [])
        names = ("weight_ih", "weight_hh", "bias_ih", "bias_hh")
        shapes = tuple(tuple(tuple(getattr(c, n).shape) for n in names) for c in cells_mod)
        flat = Fn.ThetaSplitFn.apply(theta, shapes)
        gen = [tuple(flat[4 * ci: 4 * ci + 4]) for ci in range(len(cells_mod))]
        with torch.no_grad():
            for cell, ws in zip(cells_mod, gen):
                for n, w in zip(names, ws):
                    getattr(cell, n).copy_(w)  # state_dict keeps the last generated weights, as the reference does
        return gen

    def _split_theta(self, theta, write_params=False):
        cells_mod = [self.captioner.lstm_cell] + (list(self.captioner.layers) if self.captioner.layers else [])
        gen = []
        for ci, cell in enumerate(cells_mod):
            a = 0  # utils.py:45 -- every recursive call restarts at offset 0, so extra layers alias theta[0:...]
            ws = []
            for name in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                p = getattr(cell, name)
                w = theta[a:a + p.numel()].reshape(p.shape)
                a += p.numel()
                if write_params:
                    with torch.no_grad():
                        p.copy_(w)  # state_dict keeps the last generated weights, as the reference does
                ws.append(w)
            gen.append(tuple(ws))
        return gen

    def configure_optimizers(self):  # hypernet.py:116-124
        params = list(self.hn_heads.parameters()) + list(self.hn_base.parameters())
        params += list(self.captioner.embed.parameters()) + list(self.image_encoder.fc.parameters())
        opt = torch.optim.Adam(params, lr=self.hparams['lr'])
        sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, cooldown=2)
        return [opt], [{'scheduler': sch, 'monitor': 'val_loss'}]
