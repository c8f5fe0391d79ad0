"""Attention variant ("Variant B"): hypernet_attention.HyperNet + models.decoderlstm.AttentionGru, drop-in API.

Reference: hypernet_attention.py:32-131 (HyperNet), models/decoderlstm.py:11-135 (AttentionGru),
models/attention.py:5-46 (BahdanauAttention).  The CNN trunk (models/encoder.py EncoderCNN) is out of scope: features are
the precomputed 7x7x2048 ResNet maps ``[B, 49, 2048]``.
"""
import numpy as np
import torch
from torch import nn
from torch.autograd import Function

from . import functional as Fn
from . import ops, streams
from .modules import RowsLinear, _Base, _HyperNetMixin, _beam_search, _run_grouped


class FeatureFn(Function):
    """Loop-invariant branch of AttentionGru.forward as its own autograd node: feature_fc (models/decoderlstm.py:61), the
    attention keys K = W_a f + b_a hoisted out of the time loop (the reference recomputes them every step,
    models/attention.py:34) and h0 = init_h(mean_p f) (:63, 133-134).  Returns (f [B,P,F], K [B,P,H], h0 [B,H]).

    A separate node so that it can live on its own stream (streams.py): forward next to the hypernet's weight streaming,
    backward (four tensor-core weight-gradient GEMMs) next to the hypernet head backward."""

    @staticmethod
    def forward(ctx, features, fc0_w, fc0_b, fc2_w, fc2_b, Wa_w, Wa_b, init_w, init_b):
        B, P, D = features.shape
        Fd, H = fc2_w.shape[0], Wa_w.shape[0]
        feats2 = features.reshape(B * P, D)
        if not feats2.is_contiguous():
            feats2 = feats2.contiguous()
        # the bf16x3 split of the image features (the largest input, 205 MB at B=512) is made once and reused by the
        # backward as the in-place MN-major operand of dW1 = df1^T . features
        fsplit = ops.split_bf16(feats2) if ops._tc_ok(B * P, Fd, D) else None
        if fsplit is not None:
            f1 = ops.gemm_tc(fsplit, ops.split_bf16(fc0_w.contiguous()), bias=fc0_b, relu=True)   # [B*P, F]
        else:
            f1 = ops.linear(feats2, fc0_w, fc0_b, relu=True)
        f = ops.linear(f1, fc2_w, fc2_b)                                  # [B*P, F]
        Kp = ops.linear(f, Wa_w, Wa_b)                                    # [B*P, H]
        fmean = ops.mean_pos(f.view(B, P, Fd))                            # [B, F]
        h0 = ops.linear(fmean, init_w, init_b)                            # [B, H]
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(feats2, f1, f, fmean, fc0_w, fc2_w, Wa_w, init_w,
                                  fsplit.hi if fsplit is not None else None, fsplit.lo if fsplit is not None else None)
            ctx.dims = (B, P, D, Fd, H)
        return f.view(B, P, Fd), Kp.view(B, P, H), h0

    @staticmethod
    def backward(ctx, df_in, dK, dh0):
        feats2, f1, f, fmean, fc0_w, fc2_w, Wa_w, init_w, fs_hi, fs_lo = ctx.saved_tensors
        B, P, D, Fd, H = ctx.dims
        # attention keys: dW_a = dK^T f, df = dK W_a
        dK2 = dK.reshape(B * P, H).contiguous()
        dh0 = dh0.contiguous()
        with streams.Branches("ftail", like=dK2) as br:
            with br.on(0):                                                 # off the critical path: only parameter gradients
                dWa_w = ops.matmul_tn(dK2, f)                              # [H, F]
                dWa_b = ops.colsum(dK2)
                dinit_w = ops.matmul_tn(dh0, fmean)                        # [H, F]
                dinit_b = ops.colsum(dh0)
            df = ops.matmul_nn(dK2, Wa_w.contiguous())                     # [B*P, F]
            # init_h's input gradient and the recurrence's df contribution are added to df in one pass
            dfmean = ops.matmul_nn(dh0, init_w.contiguous())               # [B, F]
            ops.mean_pos_bwd(dfmean, df.view(B, P, Fd), extra=df_in.contiguous() if df_in is not None else None)
            # feature_fc (no gradient w.r.t. the image features: they are a leaf input)
            with br.on(1):                                                 # (df is complete at this point)
                dfc2_w = ops.matmul_tn(df, f1)
                dfc2_b = ops.colsum(df)
            df1 = ops.matmul_nn(df, fc2_w.contiguous())
            ops.relu_mask_(f1, df1)
            with br.on(2):                                                 # (df1 is masked at this point)
                dfc0_b = ops.colsum(df1)
            if fs_hi is not None and (fs_lo is not None) == ops.TC_SPLIT:
                feats_op = ops.SplitOperand(fs_hi, fs_lo, D, B * P, fs_hi.shape[1], True)      # features^T, read in place
                dfc0_w = ops.gemm_tc(ops.split_bf16(df1, mn=True), feats_op)                   # [F, D]
            else:
                dfc0_w = ops.matmul_tn(df1, feats2)                                            # [F, D]
        return (None, dfc0_w, dfc0_b, dfc2_w, dfc2_b, dWa_w, dWa_b, dinit_w, dinit_b)


def _attgru_forward(need_grad, f3, K3, h0, captions, use_sampling, emb_w, W_ih, W_hh, b_ih, b_hh, fc_w, fc_b, Ua_w, Ua_b,
                    va_w, va_b):
    """The time loop of AttentionGru.forward (models/decoderlstm.py:78-108) + the vocabulary projection, given the
    loop-invariant tensors of FeatureFn.  Returns (logits, attn, tensors to save, dims)."""
    B, P, Fd = f3.shape
    T = captions.shape[1]
    E = emb_w.shape[1]
    H = W_hh.shape[1]
    V = fc_w.shape[0]
    dev = f3.device
    caps = captions.contiguous()
    f3, K3 = f3.contiguous(), K3.contiguous()
    emb_w = emb_w.contiguous()
    W_ih, W_hh = W_ih.contiguous(), W_hh.contiguous()
    lw = ops.AttGruWeights(W_ih, W_hh, Ua_w.contiguous(), E, P)
    va = va_w.reshape(-1).contiguous()
    bv = va_b.reshape(1).contiguous()
    Ua_b = Ua_b.contiguous()
    b_hh = b_hh.contiguous()
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32)
    attn = torch.empty(B, T, P, device=dev, dtype=torch.float32)
    XC = torch.empty(T * B, E + Fd, device=dev, dtype=torch.float32)   # [x_word | ctx] per (t,b)
    saved = torch.empty(5, T, B, H, device=dev, dtype=torch.float32) if need_grad else None
    logits = torch.empty(B, T, V, device=dev, dtype=torch.float32)
    W_ih_w = W_ih[:, :E]
    fed = torch.full((T, B), -1, device=dev, dtype=torch.int64)        # token whose embedding was fed at (t,b)

    if not any(use_sampling):
        # x_0 = x_1 = 0 (in-place aliasing, :83-88), x_t = Emb[caps[:, t-1]] for t >= 2
        if T > 2:
            fed[2:] = caps[:, 1:T - 1].t()
        Xw = ops.build_inputs(None, emb_w, caps, 1)                    # [T*B, E]
        XC[:, :E].copy_(Xw)
        GIw = ops.linear(Xw, W_ih_w, b_ih.contiguous())                # [T*B, 3H]
        ops.attgru_fwd(K3, f3, GIw, lw, Ua_b, va, bv, b_hh, Hall, Hbm, attn, XC, E, saved, 0, T)
        ops.linear(Hbm.view(B * T, H), fc_w, fc_b, out=logits.view(B * T, V))
    else:
        GIw = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
        xproj, vocab = ops.LinearPlan(W_ih_w, b_ih.contiguous()), ops.LinearPlan(fc_w, fc_b)   # split once, reuse per step
        # Decode without a backward pass: the word half of the input projection is a row of
        # P = [Emb; 0] W_ih[:, :E]^T + b_ih  [V+1, 3H]  (row V = the zero input of t = 0, 1) -- one GEMM per call instead
        # of (gather + copy + operand split + GEMM) per step.  Training keeps the per-step path: it needs x_word itself.
        table = None
        if not need_grad and ops.use_projection_table(B, T + 1, V):
            emb_ext = torch.cat([emb_w, emb_w.new_zeros(1, E)], 0)
            table = ops.linear(emb_ext, W_ih_w.contiguous(), b_ih.contiguous())
            fed.fill_(V)
        # Decode fast path (projection table + step-split kernels + tensor-core vocabulary projection): 5 dependent launches
        # per step instead of 7 -- the arg-max of the logits comes out of the vocabulary GEMM's epilogue as per-tile partials
        # and is finished inside the gather of the next step's input row; h_t goes to the GEMM as the bf16 hi/lo rows the
        # gates kernel has already written for the next step (no separate operand split).
        fast = table is not None and lw.pack is not None and ops._tc_ok(B, V, H)
        if fast:
            pv = torch.empty(B, 2 * ((V + 127) // 128), device=dev, dtype=torch.float32)
            pi = torch.empty(B, 2 * ((V + 127) // 128), device=dev, dtype=torch.int32)
            nparts = 0
        for t in range(T):
            if fast and use_sampling[t] and nparts:
                # tokens of step t-1 from the partials + the table row they select, one launch
                ops.argmax_finish_gather(pv, pi, nparts, table, fed[t], GIw[t * B:(t + 1) * B])
            else:
                if use_sampling[t]:
                    # :91-96  argmax of log_softmax(logits/0.5) == argmax of logits (lowest index on ties)
                    _, top = ops.softmax_argmax(logits[:, t - 1, :], want_probs=False)
                    fed[t].copy_(top)
                elif t >= 2:
                    fed[t].copy_(caps[:, t - 1])
                if table is not None:
                    ops.gather_rows(table, fed[t], out=GIw[t * B:(t + 1) * B])
                else:
                    xw = ops.gather_rows(emb_w, fed[t])                    # zeros where fed == -1
                    XC[t * B:(t + 1) * B, :E].copy_(xw)
                    xproj(xw, out=GIw[t * B:(t + 1) * B])
            ops.attgru_fwd(K3, f3, GIw, lw, Ua_b, va, bv, b_hh, Hall, Hbm, attn, XC, E, saved, t, t + 1)
            if fast:
                nparts = ops.gemm_tc_amax(ops.attstep_h_operand(lw, B, H, Fd, t), vocab.operand(), fc_b, logits[:, t, :],
                                          pv, pi)
            else:
                vocab(Hall[t + 1], out=logits[:, t, :])
    sv = (f3, K3, XC, Hall, Hbm, attn, saved, fed, emb_w, W_ih, W_hh, fc_w, Ua_w, va)
    return logits, attn, sv, (B, T, P, E, H, Fd, V)


def _attgru_backward(sv, dims, vocab, dattn):
    """vocab = (dfc_w, dfc_b, dHbm [B*T,H]).  Returns the gradients of (f, K, h0) and of the 11 parameters in
    AttentionGruFn argument order."""
    f3, K3, XC, Hall, Hbm, attn, saved, fed, emb_w, W_ih, W_hh, fc_w, Ua_w, va = sv
    B, T, P, E, H, Fd, V = dims
    dfc_w, dfc_b, dHbm = vocab
    if dattn is not None:
        dattn = dattn.contiguous()
    dGI, dGH, dU, dCTX, dK, dva, dbv, dh0 = ops.attgru_bwd(
        dHbm.view(B, T, H), dattn, K3, f3, attn, saved, Hall, Ua_w.contiguous(), va, W_ih, W_hh, E)
    Hprev = Hall[:-1].reshape(T * B, H)
    # four independent chains of small launches (each: operand splits + a GEMM that fills <= 80 of the 148 SMs + a bias
    # sum): side by side on branch streams instead of back to back
    with streams.Branches("atail", like=dGI) as br:
        with br.on(0):
            dW_ih = ops.matmul_tn(dGI, XC)                             # [3H, E+F]
            db_ih = ops.colsum(dGI)
        with br.on(1):
            dW_hh = ops.matmul_tn(dGH, Hprev)
            db_hh = ops.colsum(dGH)
        with br.on(2):
            dUa_w = ops.matmul_tn(dU, Hprev)                           # [H, H]
            dUa_b = ops.colsum(dU)
        with br.on(3):
            # features through the context vectors: df[b,p,:] = sum_t alpha[b,t,p] dctx[t,b,:]  (the K / init_h paths are
            # FeatureFn's); 72 us of fill + kernel that only need the BPTT's dctx: on their own branch, not behind a GEMM chain
            df = torch.zeros(B, P, Fd, device=f3.device, dtype=torch.float32)
            ops.attn_df(attn, dCTX, df)
        # word embeddings (t >= 2 teacher-forced rows, or the fed-back argmax rows)
        dXw = ops.matmul_nn(dGI, W_ih[:, :E])                          # [T*B, E]
        demb = torch.zeros_like(emb_w)
        ops.scatter_add_rows(dXw, fed.reshape(-1), demb)
    return (df, dK, dh0, demb, dW_ih, dW_hh, db_ih, db_hh, dfc_w, dfc_b, dUa_w, dUa_b, dva.view(1, H), dbv.view(1))


class AttentionGruFn(Function):
    """The time loop of AttentionGru.forward (models/decoderlstm.py:78-108) + vocabulary projection as one autograd node.
    Inputs: (f, K, h0) from FeatureFn, captions, the scheduled-sampling decisions, then emb_w, the generated
    (W_ih, W_hh, b_ih, b_hh), fc_w, fc_b, U_a (w, b), v_a (w, b).

    ``use_sampling[t]`` are the host-side scheduled-sampling decisions of :79-80 (already drawn by the caller from
    NumPy's global RNG, one per step).  All-False = teacher forcing: one persistent launch covers every step and the
    vocabulary projection is a single GEMM.  Otherwise the recurrence runs step by step with the argmax feedback of
    :91-96 between steps (greedy decode = all True after t = 0, the test_hn.py path).
    """

    @staticmethod
    def forward(ctx, f3, K3, h0, captions, use_sampling, *params):
        need_grad = any(ctx.needs_input_grad)
        logits, attn, sv, dims = _attgru_forward(need_grad, f3, K3, h0, captions, use_sampling, *params)
        if need_grad:
            ctx.save_for_backward(*sv)
            ctx.dims = dims
        return logits, attn

    @staticmethod
    def backward(ctx, dlogits, dattn):
        sv = ctx.saved_tensors
        B, T, P, E, H, Fd, V = ctx.dims
        dl = dlogits.reshape(B * T, V).contiguous()
        vocab = Fn.vocab_bwd_from_dlogits(dl, sv[4].view(B * T, H), sv[11])
        g = _attgru_backward(sv, ctx.dims, vocab, dattn)
        return (*g[:3], None, None, *g[3:])


class AttentionGruLossFn(Function):
    """AttentionGruFn + F.cross_entropy(ignore_index) (cc_train_hypernet.py:152-153) as ONE autograd node:
    returns (loss, logits, attn); the CE gradient goes straight into tensor-core operands (no fp32 dlogits)."""

    @staticmethod
    def forward(ctx, ignore_index, f3, K3, h0, captions, use_sampling, *params):
        logits, attn, sv, dims = _attgru_forward(True, f3, K3, h0, captions, use_sampling, *params)
        B, T, V = logits.shape
        targets = captions.reshape(-1).contiguous()
        lossbuf, lse, dhi, dlo = Fn.ce_fwd_for_loss(logits.view(B * T, V), targets, ignore_index, dims[4],
                                                    any(ctx.needs_input_grad))
        ctx.save_for_backward(*sv, logits, targets, lse, lossbuf, dhi, dlo)
        ctx.dims = dims
        ctx.ignore_index = ignore_index
        ctx.mark_non_differentiable(logits, attn)
        ctx.set_materialize_grads(False)
        return lossbuf[0].clone(), logits, attn

    @staticmethod
    def backward(ctx, g, _dl, _da):
        allsv = ctx.saved_tensors
        sv, (logits, targets, lse, lossbuf, dhi, dlo) = allsv[:-6], allsv[-6:]
        B, T, P, E, H, Fd, V = ctx.dims
        g = g.reshape(1).to(torch.float32).contiguous()
        vocab = Fn.vocab_bwd_fused(logits.view(B * T, V), targets, ctx.ignore_index, lse, lossbuf, g,
                                   sv[4].view(B * T, H), sv[11], dhi, dlo)
        gr = _attgru_backward(sv, ctx.dims, vocab, None)
        return (None, *gr[:3], None, None, *gr[3:])


class BahdanauAttention(nn.Module):
    """Parameter holder with the reference layout (models/attention.py:9-19); the math runs inside the recurrence."""

    def __init__(self, num_features, hidden_dim, output_dim=1):
        super().__init__()
        self.num_features, self.hidden_dim, self.output_dim = num_features, hidden_dim, output_dim
        self.W_a = nn.Linear(num_features, hidden_dim)
        self.U_a = nn.Linear(hidden_dim, hidden_dim)
        self.v_a = nn.Linear(hidden_dim, output_dim)


class AttentionGru(nn.Module):
    """Drop-in for models/decoderlstm.py:11 AttentionGru (num_layers = 1, dropout p = 0 as in every hypernet launcher)."""

    def __init__(self, num_features, feature_out, embedding_dim, hidden_dim, vocab_size, num_layers=1, p=0.0):
        super().__init__()
        if num_layers != 1:
            raise NotImplementedError("AttentionGru with extra GRU layers is not used by any hypernet launcher")
        if p != 0.0:
            raise NotImplementedError("dropout p > 0 is outside the hot path (HyperNet passes p=0.0)")
        self.num_features, self.embedding_dim, self.hidden_dim = num_features, embedding_dim, hidden_dim
        self.vocab_size, self.num_layers, self.sample_temp = vocab_size, num_layers, 0.5
        self.feature_fc = nn.Sequential(nn.Linear(num_features, feature_out), nn.ReLU(),
                                        nn.Linear(feature_out, feature_out))
        self.embed = nn.Embedding(vocab_size, embedding_dim)
        self.gru = nn.GRUCell(embedding_dim + feature_out, hidden_dim)
        self.layers = None
        self.fc = nn.Linear(hidden_dim, vocab_size)
        self.attention = BahdanauAttention(feature_out, hidden_dim)
        self.drop = nn.Dropout(p=p)
        self.init_h = nn.Linear(feature_out, hidden_dim)
        self._generated = None
        self._generated_groups = None
        self._theta_groups = None

    def _gru_weights(self, group=None):
        if group is not None:
            return self._generated_groups[group]
        if self._generated is not None:
            return self._generated
        g = self.gru
        return (g.weight_ih, g.weight_hh, g.bias_ih, g.bias_hh)

    def forward(self, features, captions, sample_prob=0.0, groups=None):
        """Returns (outputs [B,T,V], atten_weights [B,T,P]) -- models/decoderlstm.py:49-120.
        Consumes one np.random.random() per time step from NumPy's global RNG exactly like the reference (:79-80).
        ``groups`` ([B] int64 group id per row, after ``HyperNet.forward_grouped``) decodes every row with the generated
        weights of its style group; the scheduled-sampling draws are shared by all groups of the call."""
        T = captions.size(1)
        use = []
        for t in range(T):
            sp = 0.0 if t == 0 else sample_prob
            use.append(bool(np.random.random() < sp))
        if groups is not None:
            streams.wait_pending()
            if not any(use) and self._grouped_kernels_ok(features):
                return self._forward_grouped(features, captions, groups, None)
            # scheduled sampling / decode or a shape the step-split kernels do not cover: one call per group
            return _run_grouped(lambda g, f, c: self._forward_one(f, c, tuple(use), self._gru_weights(g)), groups,
                                [features, captions], len(self._generated_groups))
        if any(use) and not torch.is_grad_enabled():
            # decode (test_hn.py path, cc_train_hypernet.py:230): ~10 launches per step -> captured into a CUDA graph
            from . import graphs
            # the loop-invariant feature branch runs eagerly on its own stream (next to an asynchronous hypernet forward);
            # the graph holds only the time loop
            f3, K3, h0 = self._features(features.contiguous().float())
            streams.wait_pending()
            rp = [p.detach() for p in self._recurrence_params(self._gru_weights())]
            gen = [rp[1].contiguous(), rp[2].contiguous(), rp[3].contiguous(), rp[4].contiguous()]   # generated weights
            key = ("AttentionGru.decode", id(self), tuple(features.shape), tuple(captions.shape), tuple(use),
                   features.device.index) + tuple(p.data_ptr() for i, p in enumerate(rp) if i not in (1, 2, 3, 4))

            def run(f_, k_, h_, c, wi, wh, bi, bh):
                q = list(rp)
                q[1], q[2], q[3], q[4] = wi, wh, bi, bh
                return AttentionGruFn.apply(f_, k_, h_, c, tuple(use), *q)

            out = graphs.graphed_call(key, run, [f3.detach(), K3.detach(), h0.detach(), captions.contiguous()] + gen)
            return out[0], out[1]
        return self._forward_one(features, captions, tuple(use), self._gru_weights())

    def _feature_params(self):
        a = self.attention
        return (self.feature_fc[0].weight, self.feature_fc[0].bias, self.feature_fc[2].weight, self.feature_fc[2].bias,
                a.W_a.weight, a.W_a.bias, self.init_h.weight, self.init_h.bias)

    def _recurrence_params(self, gru_w):
        W_ih, W_hh, b_ih, b_hh = gru_w
        a = self.attention
        return (self.embed.weight, W_ih, W_hh, b_ih, b_hh, self.fc.weight, self.fc.bias, a.U_a.weight, a.U_a.bias,
                a.v_a.weight, a.v_a.bias)

    def _features(self, features):
        """FeatureFn on the "features" side stream: it overlaps with an asynchronous hypernet forward, and its backward
        node (which the autograd engine runs on the same stream) with the hypernet head backward."""
        if streams.enabled(features):
            # high priority: the backward of this branch (tensor-core GEMMs, the long feature_fc weight gradient last) runs
            # next to the hypernet head backward, whose thousands of short CTAs otherwise fill every SM slot first and push
            # the branch -- the end of the step -- behind them (tools/timeline_step.py attention)
            with streams.fork("features_hp", priority=-1) as s:
                out = FeatureFn.apply(features, *self._feature_params())
            torch.cuda.current_stream().wait_stream(s)
            return out
        return FeatureFn.apply(features, *self._feature_params())

    def _forward_one(self, features, captions, use, gru_w):
        f3, K3, h0 = self._features(features)
        streams.wait_pending()                    # generated weights of an asynchronous hypernet forward
        return AttentionGruFn.apply(f3, K3, h0, captions, use, *self._recurrence_params(gru_w))

    def _grouped_kernels_ok(self, features):
        """The grouped kernels cover teacher forcing on shapes the step-split recurrence handles (fp32 mode)."""
        P = features.shape[1]
        Fd = self.feature_fc[2].out_features
        return (getattr(self, "_theta_groups", None) is not None and features.is_cuda and ops.ATT_STEP
                and ops._attstep_bytes(self.hidden_dim, Fd, P, 0)[0] > 0
                and ops._attstep_bwd_bytes(self.hidden_dim, Fd, P, features.shape[0], 1)[0] > 0)

    def _forward_grouped(self, features, captions, groups, ignore_index):
        """Many-style batch on the grouped kernels (grouped.py): rows sorted by style group, one grouped tensor-core launch
        per time-batched product, the step-split recurrence with one weight pack per group.  ``ignore_index`` None:
        returns (logits, attn); else (loss, logits, attn) with the loss fused."""
        from . import grouped as Gp
        Theta = self._theta_groups
        plan = Gp.GroupPlan.get(groups, Theta.shape[0], captions.shape[1], features.device)
        f3, K3, h0 = self._features(features)
        f3s = Gp.RowPermuteFn.apply(f3, plan.order, plan.inv)
        K3s = Gp.RowPermuteFn.apply(K3, plan.order, plan.inv)
        h0s = Gp.RowPermuteFn.apply(h0, plan.order, plan.inv)
        caps_s = captions.index_select(0, plan.order)
        a = self.attention
        shared = (self.embed.weight, self.fc.weight, self.fc.bias, a.U_a.weight, a.U_a.bias, a.v_a.weight, a.v_a.bias)
        if ignore_index is None:
            return Gp.AttentionGruGroupedFn.apply(plan, f3s, K3s, h0s, caps_s, Theta, *shared)
        return Gp.AttentionGruGroupedLossFn.apply(ignore_index, plan, captions.contiguous(), f3s, K3s, h0s, caps_s, Theta,
                                                  *shared)

    def forward_loss(self, features, captions, sample_prob=0.0, ignore_index=0, groups=None):
        """``forward`` fused with ``F.cross_entropy(outputs.view(-1,V), captions.view(-1), ignore_index=<pad>)``
        (cc_train_hypernet.py:152-153): returns ``(loss, outputs, atten_weights)``; one autograd node.
        ``groups``: many-style batch after ``HyperNet.forward_grouped`` (teacher forcing only)."""
        T = captions.size(1)
        use = tuple(bool(np.random.random() < (0.0 if t == 0 else sample_prob)) for t in range(T))
        if groups is not None:
            streams.wait_pending()
            if any(use) or not self._grouped_kernels_ok(features):
                raise NotImplementedError("forward_loss(groups=...) covers teacher forcing on step-split shapes; use "
                                          "forward(..., groups=...) + cross_entropy otherwise")
            return self._forward_grouped(features, captions, groups, ignore_index)
        f3, K3, h0 = self._features(features)
        streams.wait_pending()
        return AttentionGruLossFn.apply(ignore_index, f3, K3, h0, captions, use,
                                        *self._recurrence_params(self._gru_weights()))

    @torch.no_grad()
    def beam_search(self, features, beam_size=3, end_sentence=2, max_steps=50):
        """Beam search for ONE image -- the loop of HyperNet.test_step, hypernet_attention.py:247-326 (``beam_size`` = 3 at
        :44).  ``features`` [1, P, D] are the encoder features (``feature_fc`` is applied here, :249).  Returns the best
        complete sequence as a list of token ids (leading 0, trailing ``end_sentence``) or ``None`` when the reference
        computes no beam caption (a beam is still open after ``max_steps`` + 1 steps, :308-311).

        Reference quirks kept: every row starts from word 0 and ALL rows get a zero word embedding whenever the first
        row's previous word is 0 (:265-266); step 1 ranks ``scores[0]`` only (:274-275); scores are summed
        log-probabilities without length normalisation; finished beams leave the batch (:296-303).
        Runs ``beam_search_batched`` on the one image, so ``beam_size`` must lie in [1, 8] and not exceed V."""
        if features.dim() != 3 or features.shape[0] != 1:
            raise ValueError("beam_search expects the features of one image: [1, P, D]")
        return self.beam_search_batched(features, beam_size, end_sentence, max_steps)[0]

    @torch.no_grad()
    def beam_search_batched(self, features, beam_size=3, end_sentence=2, max_steps=50, sync_every=8):
        """Beam search of HyperNet.test_step (hypernet_attention.py:247-326) for a whole batch at once, device-resident:
        ``features`` [B, P, D] -> list of B results, each the best complete token sequence (leading 0, trailing
        ``end_sentence``) or ``None`` where the reference computes no beam caption (a beam still open after
        ``max_steps`` + 1 steps).  ``beam_size`` in [1, 8], at most V.

        All B*k beams go through the decoder step kernels together; between steps ONE kernel per step
        (csrc/beam.cu, a CTA per image) does the reference's host bookkeeping on the device: log-softmax + running scores,
        top-k over the k*V candidates, completed beams to the complete list, survivors compacted (history, score, hidden
        state gathered from the parent beam), next input words.  The host reads the results in one copy at the end; it
        only peeks at an 'all images finished' flag every ``sync_every`` steps to stop early."""
        streams.wait_pending()
        if features.dim() != 3:
            raise ValueError("beam_search_batched expects features [B, P, D]")
        E, H, V = self.embedding_dim, self.hidden_dim, self.vocab_size

        def setup(rep):
            feats = features.contiguous().float()
            P, dev = feats.shape[1], feats.device
            W_ih, W_hh, b_ih, b_hh = [w.detach().contiguous() for w in self._gru_weights()]
            a = self.attention
            emb_w = self.embed.weight.detach()
            f3, K3, h0 = FeatureFn.apply(feats, *[p.detach() for p in self._feature_params()])
            f3k, K3k = rep(f3), rep(K3)
            R, Fd = f3k.shape[0], f3.shape[2]
            lw = ops.AttGruWeights(W_ih, W_hh, a.U_a.weight.detach().contiguous(), E, P)
            va, bv = a.v_a.weight.detach().reshape(-1).contiguous(), a.v_a.bias.detach().reshape(1).contiguous()
            bu = a.U_a.bias.detach().contiguous()
            xproj, vocab = ops.LinearPlan(W_ih[:, :E], b_ih), ops.LinearPlan(self.fc.weight.detach(), self.fc.bias.detach())
            Hall = torch.empty(2, R, H, device=dev, dtype=torch.float32)
            attn = torch.empty(R, 1, P, device=dev, dtype=torch.float32)
            XC = torch.empty(R, E + Fd, device=dev, dtype=torch.float32)
            GIw = torch.empty(R, 3 * H, device=dev, dtype=torch.float32)
            logits = torch.empty(R, V, device=dev, dtype=torch.float32)

            def step_fn(step, h, prev_tok, words):
                xproj(ops.gather_rows(emb_w, words), out=GIw)          # zeros where words == -1
                Hall[0].copy_(h)
                ops.attgru_fwd(K3k, f3k, GIw, lw, bu, va, bv, b_hh, Hall, None, attn, XC, E, None, 0, 1)
                return vocab(Hall[1], out=logits), Hall[1]
            return h0, step_fn
        return _beam_search(setup, beam_size, V, max_steps, end_sentence, sync_every)

    @torch.no_grad()
    def greedy_search(self, features, end_sentence=2, max_sentence=20):
        """B = 1 greedy decoding with EOS stop -- models/decoderlstm.py:138-175.  ``features`` have ALREADY been through
        ``feature_fc`` ([1, P, F]); the first input word is index 0; returns (tokens list[int], list of attention
        weights [1, P]).  All ``max_sentence`` steps run on the device without host round trips; the token list is cut
        after the first ``end_sentence`` (the steps after it do not influence the ones before)."""
        streams.wait_pending()
        f3 = features.contiguous().float()
        B, P, Fd = f3.shape
        W_ih, W_hh, b_ih, b_hh = [w.detach().contiguous() for w in self._gru_weights()]
        E, H, T = self.embedding_dim, self.hidden_dim, int(max_sentence)
        dev = f3.device
        a = self.attention
        emb_w = self.embed.weight.detach()
        Kp = ops.linear(f3.view(B * P, Fd), a.W_a.weight.detach(), a.W_a.bias.detach()).view(B, P, H)
        h0 = ops.linear(ops.mean_pos(f3), self.init_h.weight.detach(), self.init_h.bias.detach())
        lw = ops.AttGruWeights(W_ih, W_hh, a.U_a.weight.detach().contiguous(), E, P)
        va, bv = a.v_a.weight.detach().reshape(-1).contiguous(), a.v_a.bias.detach().reshape(1).contiguous()
        Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
        Hall[0].copy_(h0)
        attn = torch.empty(B, T, P, device=dev, dtype=torch.float32)
        XC = torch.empty(T * B, E + Fd, device=dev, dtype=torch.float32)
        GIw = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
        logits = torch.empty(B, self.vocab_size, device=dev, dtype=torch.float32)
        tokens = torch.zeros(T + 1, B, device=dev, dtype=torch.int64)          # tokens[0] = 0: the first input word
        W_ih_w = W_ih[:, :E]
        for t in range(T):
            xw = ops.gather_rows(emb_w, tokens[t])
            ops.linear(xw, W_ih_w, b_ih, out=GIw[t * B:(t + 1) * B])
            ops.attgru_fwd(Kp, f3, GIw, lw, a.U_a.bias.detach(), va, bv, b_hh, Hall, None, attn, XC, E, None, t, t + 1)
            ops.linear(Hall[t + 1], self.fc.weight.detach(), self.fc.bias.detach(), out=logits)
            _, top = ops.softmax_argmax(logits, want_probs=False)
            tokens[t + 1].copy_(top)
        sent = tokens[1:, 0].tolist()
        if end_sentence in sent:
            sent = sent[:sent.index(end_sentence) + 1]
        return sent, [attn[0:1, t, :].clone() for t in range(len(sent))]

    def init_hidden(self, features):
        """h0 = init_h(mean over positions) -- models/decoderlstm.py:122-135 (features already through feature_fc)."""
        B, P, Fd = features.shape
        return Fn.linear(ops.mean_pos(features.contiguous()), self.init_h.weight, self.init_h.bias)


class SpatialFeatureEncoder(nn.Module):
    """Stands in for models/encoder.py EncoderCNN (ResNet-152 trunk, out of scope): passes precomputed [B,49,2048]
    feature maps through unchanged."""

    def forward(self, feats):
        return feats


class HyperNetAttention(_HyperNetMixin, _Base):
    """Drop-in for hypernet_attention.py:32 HyperNet."""

    def __init__(self, feature_size, embed_size, hidden_size, vocab_size, vocab, num_layers=1, lr=1e-6, mixup=False,
                 alpha=0.3, cc=False, hyper_emb=10):
        super().__init__()
        self.hparams['feature_size'] = feature_size
        self.hparams['vocab_size'] = vocab_size
        self.hparams['embed_size'] = embed_size
        self.hparams['hidden_size'] = hidden_size
        self.vocab = vocab
        self.hparams['lr'] = lr
        self.hparams['num_layers'] = num_layers
        self.teacher_forcing_proba = 0.0
        self.beam_size = 3
        self.mixup, self.alpha = mixup, alpha
        self.image_encoder = SpatialFeatureEncoder()
        self.captioner = AttentionGru(2048, feature_size, embed_size, hidden_size, vocab_size, p=0.0)
        N, M = 1, 500
        he = hyper_emb if cc else embed_size
        self.hn_base = nn.Sequential(RowsLinear(he, N * he), nn.LeakyReLU(), RowsLinear(N * he, N * he), nn.LeakyReLU())
        heads = []
        for name, W in self.captioner.gru.named_parameters():  # hypernet_attention.py:69-96
            w = W.numel()
            if w < N * he:
                heads.append(nn.Sequential(RowsLinear(N * he, N), nn.LeakyReLU(), RowsLinear(w, w)))
            elif w // M < N * he:
                heads.append(nn.Sequential(RowsLinear(N * he, N * he), nn.LeakyReLU(), RowsLinear(N * he, w)))
            else:
                heads.append(nn.Sequential(RowsLinear(N * he, w // M), nn.LeakyReLU(), RowsLinear(w // M, w)))
        self.hn_heads = nn.ModuleList(heads)

    def forward(self, x):
        """theta -> captioner.gru weights; returns self.captioner (hypernet_attention.py:111-121)."""
        ws = self._generate_and_inject(x)
        self.captioner._generated = ws if self.grad_mode == "flow" else None
        self.captioner._generated_groups = None
        self.captioner._theta_groups = None
        return self.captioner

    def _split_theta(self, theta, write_params=False):
        gru = self.captioner.gru
        a, ws = 0, []
        for name in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
            p = getattr(gru, name)
            w = theta[a:a + p.numel()].reshape(p.shape)
            a += p.numel()
            if write_params:
                with torch.no_grad():
                    p.copy_(w)
            ws.append(w)
        return tuple(ws)

    def configure_optimizers(self):  # hypernet_attention.py:123-134
        c = self.captioner
        params = list(self.hn_heads.parameters()) + list(self.hn_base.parameters())
        for m in (c.feature_fc, c.embed, c.fc, c.attention, c.init_h):
            params += list(m.parameters())
        opt = torch.optim.Adam(params, lr=self.hparams['lr'])
        sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, cooldown=2, factor=0.5)
        return [opt], [{'scheduler': sch, 'monitor': 'val_loss with TF', 'interval': 'epoch'}]
