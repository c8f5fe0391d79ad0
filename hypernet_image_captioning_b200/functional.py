"""autograd.Function wrappers: forward and backward both run the hand-written CUDA kernels (no torch math)."""
from typing import List, Optional, Sequence

import torch
from torch.autograd import Function

from . import ops, parallel, streams
from .ops import ACT_LEAKY, ACT_NONE


# ----------------------------------------------------------------------------------------------------------------------
# hypernetwork: X[G,he] -> Theta[G,theta]      (reference hypernet_attention.py:111-118 / hypernet.py:104-111)
# ----------------------------------------------------------------------------------------------------------------------
# Rank-G head gradients (see optim.FusedAdam): when > 0, the backward of a head's second Linear whose weight has at least
# this many elements does NOT materialise dW2 = dtheta^T a; it attaches ``(dtheta_slice [G,N], a [G,K])`` to the parameter
# as ``.grad_lowrank`` and leaves ``.grad`` untouched.  Set by ``hypernet.head_grad_mode = "lowrank"``.
LOWRANK_MIN_NUMEL = 0
LOWRANK_MAX_G = 4


class HyperNetThetaFn(Function):
    """params = [base0.W, base0.b, base2.W, base2.b, (head_i.0.W, head_i.0.b, head_i.2.W, head_i.2.b) * n_heads]."""

    @staticmethod
    def forward(ctx, x, *params):
        nh = (len(params) - 4) // 4
        b0 = ops.rows_linear_fwd(params[0], params[1], x, ACT_LEAKY)
        b1 = ops.rows_linear_fwd(params[2], params[3], b0, ACT_LEAKY)
        sizes = [params[4 + 4 * i + 2].shape[0] for i in range(nh)]
        theta = torch.empty(x.shape[0], sum(sizes), device=x.device, dtype=torch.float32)
        mids, offs, off = [None] * nh, [], 0
        for i in range(nh):
            offs.append(off)
            off += sizes[i]
        # the heads are independent chains (small first layer -> second layer); the two that generate the weight matrices
        # stream hundreds of MB, the bias heads are a few 4 us launches: side by side instead of back to back
        streams.clear_ranges()
        with streams.Branches("hnf", like=x, enable=nh > 1) as br:
            # tiny (bias) heads first, the matrix heads after them in parameter order (W_ih before W_hh: the input projection
            # starts when W_ih and b_ih are there): the big heads' persistent CTAs fill every SM for hundreds of microseconds,
            # and a bias head queued behind them (12 us of work) would only run when they drain
            for i in sorted(range(nh), key=lambda q: (sizes[q] >= 4096, q)):
                W1, c1, W2, c2 = params[4 + 4 * i: 8 + 4 * i]
                with br.on(i % 4):
                    a = ops.rows_linear_fwd(W1, c1, b1, ACT_LEAKY)
                    seg = theta[:, offs[i]:offs[i] + sizes[i]]
                    ops.rows_linear_fwd(W2, c2, a, ACT_NONE, out=seg)
                    mids[i] = a
                    if x.shape[0] == 1:
                        streams.mark_range(seg)      # consumers of this slice alone need not wait for the other heads
        ctx.save_for_backward(x, b0, b1, *mids, *params)
        ctx.lowrank_targets = [params[4 + 4 * i + 2] for i in range(nh)]    # the Parameter objects (saved tensors are views)
        ctx.lowrank_min = LOWRANK_MIN_NUMEL
        ctx.nh = nh
        ctx.sizes = sizes
        return theta

    @staticmethod
    def backward(ctx, dtheta):
        nh, sizes = ctx.nh, ctx.sizes
        sv = ctx.saved_tensors
        x, b0, b1 = sv[0], sv[1], sv[2]
        mids = sv[3:3 + nh]
        params = sv[3 + nh:]
        need = ctx.needs_input_grad  # [x, *params]
        dtheta = dtheta.contiguous()
        grads: List[Optional[torch.Tensor]] = [None] * len(params)
        db1 = torch.zeros_like(b1)
        offs, off = [], 0
        for i in range(nh):
            offs.append(off)
            off += sizes[i]

        def head_bwd(i):
            W1, c1, W2, c2 = params[4 + 4 * i: 8 + 4 * i]
            pi = 4 + 4 * i
            off = offs[i]
            tgt = ctx.lowrank_targets[i]
            prev = getattr(tgt, "grad_lowrank", None)
            lowrank = (ctx.lowrank_min > 0 and need[1 + pi + 2] and W2.numel() >= ctx.lowrank_min
                       and W2.dtype == torch.float32
                       and x.shape[0] + (prev[0].shape[0] if prev is not None else 0) <= LOWRANK_MAX_G)
            if lowrank:
                _, dc2, da, dP = ops.rows_linear_bwd(W2, mids[i], None, dtheta[:, off:off + sizes[i]], ACT_NONE,
                                                     need_dW=False, return_dP=True)
                # a second backward before the optimizer step accumulates by growing the rank
                tgt.grad_lowrank = (dP, mids[i]) if prev is None else (torch.cat([prev[0], dP], 0),
                                                                        torch.cat([prev[1], mids[i]], 0))
                dW2 = None
            else:
                dW2, dc2, da = ops.rows_linear_bwd(W2, mids[i], None, dtheta[:, off:off + sizes[i]], ACT_NONE,
                                                   need_dW=need[1 + pi + 2])
            dW1, dc1, _ = ops.rows_linear_bwd(W1, b1, mids[i], da, ACT_LEAKY, need_dW=need[1 + pi], dA=db1)   # db1 += (atomics)
            grads[pi], grads[pi + 1], grads[pi + 2], grads[pi + 3] = dW1, dc1, dW2, dc2

        # independent per-head chains side by side (the bias heads' 6-7 us launches fit next to the big heads' streaming)
        with streams.Branches("hnb", like=x, enable=nh > 1) as br:
            for i in range(nh):
                with br.on(i % 4):
                    head_bwd(i)
        dWb1, dcb1, db0 = ops.rows_linear_bwd(params[2], b0, b1, db1, ACT_LEAKY, need_dW=need[3])
        dWb0, dcb0, dx = ops.rows_linear_bwd(params[0], x, b0, db0, ACT_LEAKY, need_dW=need[1], need_dA=need[0])
        grads[0], grads[1], grads[2], grads[3] = dWb0, dcb0, dWb1, dcb1
        for j in range(len(grads)):
            if not need[1 + j]:
                grads[j] = None
            elif grads[j] is not None and grads[j].dtype != params[j].dtype:
                grads[j] = grads[j].to(params[j].dtype)   # bf16 mode: bias gradients (weights are already bf16)
        if dx is not None and dx.dtype != x.dtype:
            dx = dx.to(x.dtype)
        parallel.join()   # data parallel: whatever consumes these gradients is ordered after the overlapped bucket all-reduce
        return (dx if need[0] else None, *grads)


class ThetaSplitFn(Function):
    """theta [1, n] -> the generated parameter tensors of every cell, as views (the injection of utils.py:24-69: cell c's
    (weight_ih, weight_hh, bias_ih, bias_hh) are consecutive slices that start again at offset 0 for every extra cell,
    utils.py:45).  One autograd node whose backward assembles d(theta) with ONE concatenation per cell, instead of autograd's
    select + slice + view chain (a zero fill, a copy and an add per slice, all in front of the head backward)."""

    @staticmethod
    def forward(ctx, theta, shapes):
        ctx.shapes, ctx.n = shapes, theta.shape[1]
        outs = []
        for cell in shapes:
            a = 0
            for shp in cell:
                n = 1
                for d in shp:
                    n *= d
                outs.append(theta[0, a:a + n].view(shp))
                a += n
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        out, i = None, 0
        ref = next(g for g in grads if g is not None)
        for cell in ctx.shapes:
            parts = []
            for shp in cell:
                n = 1
                for d in shp:
                    n *= d
                g = grads[i]
                i += 1
                parts.append(g.reshape(-1) if g is not None else ref.new_zeros(n))
            used = sum(p.numel() for p in parts)
            if used < ctx.n:
                parts.append(ref.new_zeros(ctx.n - used))
            flat = torch.cat(parts)
            out = flat if out is None else out + flat
        return out.view(1, ctx.n), None


def hypernet_theta(x2d: torch.Tensor, params: Sequence[torch.Tensor]) -> torch.Tensor:
    return HyperNetThetaFn.apply(x2d, *params)


class RowsLinearFn(Function):
    """y = act(x W^T + b) for a handful of rows (G <= a few) on the weight-streaming kernels; act = LeakyReLU(0.01) or none.
    Used by the domain-embedding front-ends (cc_train_hypernet.py:90-106), whose input is one vector per step."""

    @staticmethod
    def forward(ctx, x, W, b, leaky):
        act = ACT_LEAKY if leaky else ops.ACT_NONE
        y = ops.rows_linear_fwd(W, b, x, act)
        ctx.save_for_backward(x, W, y)
        ctx.act = act
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, y = ctx.saved_tensors
        need = ctx.needs_input_grad
        dW, db, dx = ops.rows_linear_bwd(W, x, y if ctx.act != ops.ACT_NONE else None, dy.contiguous(), ctx.act,
                                         need_dW=need[1], need_dA=need[0])
        return (dx if need[0] else None, dW if need[1] else None, db if need[2] else None, None)


def rows_linear(x, W, b, leaky=False):
    return RowsLinearFn.apply(x, W, b, leaky)


# ----------------------------------------------------------------------------------------------------------------------
# y = x W^T + b (ReLU optional)        -- nn.Linear replacement (image_encoder.fc hypernet.py:46, feature_fc, init_h ...)
# ----------------------------------------------------------------------------------------------------------------------
class LinearFn(Function):
    @staticmethod
    def forward(ctx, x, W, b, relu):
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        y = ops.linear(x2, W.contiguous(), b, relu=relu)
        ctx.save_for_backward(x2, W, y if relu else None)
        ctx.relu = relu
        ctx.xshape = x.shape
        return y.reshape(*x.shape[:-1], W.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, W, y = ctx.saved_tensors
        dy2 = dy.reshape(-1, dy.shape[-1]).contiguous()
        if ctx.relu:
            dy2 = dy2.clone()
            ops._cabi.call("caphn_relu_mask", y.data_ptr(), dy2.data_ptr(), dy2.numel(), ops._stream())
        dx = ops.matmul_nn(dy2, W.contiguous()).reshape(ctx.xshape) if ctx.needs_input_grad[0] else None
        dW = ops.matmul_tn(dy2, x2) if ctx.needs_input_grad[1] else None
        db = ops.colsum(dy2) if ctx.needs_input_grad[2] else None
        return dx, dW, db, None


def linear(x, W, b, relu=False):
    return LinearFn.apply(x, W, b, relu)


# ----------------------------------------------------------------------------------------------------------------------
# fused softmax cross-entropy (mean over non-ignored rows)      -- F.cross_entropy at cc_train_hypernet.py:153
# ----------------------------------------------------------------------------------------------------------------------
class CrossEntropyFn(Function):
    @staticmethod
    def forward(ctx, logits, targets, ignore_index):
        l2 = logits.reshape(-1, logits.shape[-1])
        if l2.stride(1) != 1:
            l2 = l2.contiguous()
        t = targets.reshape(-1).contiguous()
        lossbuf, lse = ops.ce_fwd(l2, t, ignore_index)
        ctx.save_for_backward(l2, t, lse, lossbuf)
        ctx.ignore_index = ignore_index
        ctx.shape = logits.shape
        return lossbuf[0].clone()

    @staticmethod
    def backward(ctx, g):
        l2, t, lse, lossbuf = ctx.saved_tensors
        g = g.reshape(1).to(torch.float32).contiguous()
        dX = ops.ce_bwd(l2, t, ctx.ignore_index, lse, lossbuf, g)
        return dX.reshape(ctx.shape), None, None


def cross_entropy(logits, targets, ignore_index: Optional[int] = None):
    """Mean CE over rows whose target != ignore_index (None = no masking, hypernet.py:145)."""
    return CrossEntropyFn.apply(logits, targets, ignore_index)


# ----------------------------------------------------------------------------------------------------------------------
# vocabulary projection backward, shared by both decoders
# ----------------------------------------------------------------------------------------------------------------------
def vocab_bwd_from_dlogits(dl, Hbm2, fc_w, need_w=True, need_b=True):
    """dl [B*T, V] fp32 (as handed over by autograd).  Returns (dfc_w, dfc_b, dHbm)."""
    dfc_w = ops.matmul_tn(dl, Hbm2) if need_w else None
    dfc_b = ops.colsum(dl) if need_b else None
    dHbm = ops.matmul_nn(dl, fc_w.contiguous())
    return dfc_w, dfc_b, dHbm


# The fused loss nodes compute the cross-entropy AND its (unscaled) gradient operand in one pass over the logits during the
# forward (ops.ce_fwd_split: 0.4 GB read + 0.4 GB written at [10240, 9684], instead of ce_fwd's read followed by
# ce_bwd_split's read + write in the backward); the scalar grad_output / #valid rows is applied by the epilogues of the two
# backward products, and the bias gradient is one more output column of the dW product (a row of ones appended to H).
def ce_fwd_for_loss(logits2d, targets, ignore_index, H, need_grad):
    """Forward of the fused loss nodes.  Returns (lossbuf, lse, hi, lo): hi / lo = the unscaled gradient operand when the
    one-pass kernel applies (gradients wanted, both backward products on the tensor cores, row fits in shared memory), else
    None / None and the backward runs ce_bwd_split."""
    M, V = logits2d.shape
    if need_grad and V <= ops.CE_FWD_SPLIT_MAX_V and ops._tc_ok(M, H, V) and ops._tc_ok(V, H + 1, M):
        return ops.ce_fwd_split(logits2d, targets, ignore_index)
    lossbuf, lse = ops.ce_fwd(logits2d, targets, ignore_index)
    return lossbuf, lse, None, None


class VocabPrep:
    """Operand preparation of the vocabulary projection moved off the step's dependency chain (fused loss nodes, while a CUDA
    graph is captured -- eagerly the same launches simply run in order): the two bf16 splits of the projection weight do not
    depend on the step's activations, so they run on a branch stream from the start of the decoder forward (next to the input
    projection and the recurrence); the transposed split of the hidden states [H | 1] that only the BACKWARD needs runs on a
    second branch next to the logits product instead of in front of the dW product."""

    def __init__(self, M, V, H, need_grad, like):
        self.on = bool(need_grad and V <= ops.CE_FWD_SPLIT_MAX_V and ops._tc_ok(M, H, V) and ops._tc_ok(V, H + 1, M)
                       and ops._tc_ok(M, V, H))
        self.w = self.wt = self.ht = None
        self.br = streams.Branches("vprep", like=like) if self.on else None

    def start(self, fc_w):
        if not self.on:
            return
        self.br.__enter__()
        with self.br.on(0):
            wc = fc_w.contiguous()
            self.w = ops.split_bf16(wc)                    # B operand of the logits product
            self.wt = ops.split_bf16_t(wc)                 # B operand of dH = d W_out

    def logits(self, Hbm2, fc_b):
        """Called right after the recurrence: logits = Hbm2 W^T + b with the prepared weight operand."""
        with self.br.on(1):                                # after the recurrence (queued so far on the caller's stream)
            self.ht = ops.split_bf16_t(Hbm2, ones_row=True)    # B operand of [dW_out | db] = d^T [H | 1]
        self.br.join(0)
        return ops.gemm_tc(ops.split_bf16(Hbm2), self.w, bias=fc_b)

    def finish(self):
        if self.on:
            self.br.__exit__(None, None, None)

    def saved(self):
        """Tensors for save_for_backward (None entries when the preparation is off)."""
        if not self.on:
            return (None, None, None, None)
        return (self.wt.hi, self.wt.lo, self.ht.hi, self.ht.lo)


def vocab_bwd_fused(logits2d, targets, ignore_index, lse, lossbuf, gscale, Hbm2, fc_w, hi=None, lo=None, pre=None):
    """Loss fused with the projection: the cross-entropy gradient is written directly as bf16x3 tensor-core operands
    (row-major for dH = d W_out, transposed for dW_out = d^T H) and the bias gradient is reduced in the same pass, so
    the fp32 dlogits tensor never exists.  hi / lo: the unscaled operand ce_fwd_for_loss produced in the forward."""
    M, V = logits2d.shape
    H = Hbm2.shape[1]
    if hi is not None:
        Vp = hi.shape[1]
        d, dT = ops.SplitOperand(hi, lo, M, V, Vp), ops.SplitOperand(hi, lo, V, M, Vp, True)
        scale = (gscale, lossbuf[1:])
        if pre is not None and pre[0] is not None:         # operands prepared in the forward (VocabPrep)
            Mp = pre[2].shape[1]
            wt = ops.SplitOperand(pre[0], pre[1], H, V, pre[0].shape[1])
            ht = ops.SplitOperand(pre[2], pre[3], H + 1, M, Mp)
        else:
            wt = ops.split_bf16_t(fc_w.contiguous(), want_lo=lo is not None)
            ht = ops.split_bf16_t(Hbm2, want_lo=lo is not None, ones_row=True)
        dHbm = ops.gemm_tc(d, wt, scale=scale)             # [B*T, H]
        # [V, H+1] with a row pitch that is a multiple of 4 floats: the split-K epilogue adds 16-byte vectors per row
        wb = torch.empty(V, ops.round4(H + 1), device=Hbm2.device, dtype=torch.float32)[:, :H + 1]
        ops.gemm_tc(dT, ht, scale=scale, out=wb)
        return wb[:, :H].contiguous(), wb[:, H].contiguous(), dHbm
    if not (ops._tc_ok(M, H, V) and ops._tc_ok(V, H, M)):
        dl = ops.ce_bwd(logits2d, targets, ignore_index, lse, lossbuf, gscale)
        return vocab_bwd_from_dlogits(dl, Hbm2, fc_w)
    d, dT, dfc_b = ops.ce_bwd_split(logits2d, targets, ignore_index, lse, lossbuf, gscale)
    dHbm = ops.gemm_tc(d, ops.split_bf16_t(fc_w.contiguous()))            # [B*T, H]   (K = V)
    dfc_w = ops.gemm_tc(dT, ops.split_bf16_t(Hbm2))                       # [V, H]     (K = B*T)
    return dfc_w, dfc_b, dHbm


# ----------------------------------------------------------------------------------------------------------------------
# Variant A decoder: teacher-forced DecoderGRU.forward  (reference later.py:389-457)
# ----------------------------------------------------------------------------------------------------------------------
def _gru_decoder_forward(feats, captions, h0, emb_w, fc_w, fc_b, cells, prep=None):
    B, T = captions.shape
    NL = len(cells) // 4
    W_ih, W_hh, b_ih, b_hh = cells[0:4]
    H = W_hh.shape[1]
    if prep is not None:
        prep.start(fc_w)
    caps = captions.contiguous()
    feats = feats.contiguous()
    emb_w = emb_w.contiguous()
    X = ops.build_inputs(feats, emb_w, caps, 0)                       # [T*B, E]
    # the input projection needs only the W_ih / b_ih slices of the generated weights: with an asynchronous hypernet forward
    # (modules.py async_hypernet) it runs while the head that generates W_hh is still streaming
    if not streams.wait_ranges((W_ih, b_ih)):
        streams.wait_pending()
    GI = ops.linear(X, W_ih.contiguous(), b_ih.contiguous())          # [T*B, 3H]
    late_join = streams.wait_ranges(tuple(cells))                    # every generated slice (not the parameter injection copies)
    if not late_join:
        streams.wait_pending()
    if NL == 1 and ops.gru_resident_ok(H):
        # weights-resident path: the whole W_hh lives in ONE CTA (shared memory + registers) for all T steps, 4 rows per CTA
        Hall, Hbm, saved, Hmid = ops.gru_resident_fwd(GI, W_hh.contiguous(), b_hh.contiguous(), h0.contiguous(), T)
    elif NL == 1 and ops.gru_cluster_size(H):
        # weights-resident path: W_hh stays in shared memory (cluster-split) for all T steps
        Hall, Hbm, saved, Hmid = ops.gru_cluster_fwd(GI, W_hh.contiguous(), b_hh.contiguous(), h0.contiguous(), T)
    else:
        ld3 = ops.round4(3 * H)
        WhhT = ops.transpose_pad(W_hh.contiguous(), ld3)                  # [H, ld3]
        extra = []
        for l in range(1, NL):
            Wi, Wh, bi, bh = cells[4 * l: 4 * l + 4]
            extra.append((ops.transpose_pad(Wi.contiguous(), ld3), ops.transpose_pad(Wh.contiguous(), ld3),
                          bi.contiguous(), bh.contiguous()))
        Hall, Hbm, saved, Hmid = ops.gru_seq_fwd(GI, WhhT, b_hh.contiguous(), h0.contiguous(), T, save=True,
                                                 extra=extra)
    if late_join:
        streams.wait_pending()      # (whatever else the forked hypernet computation queued; done long before this point)
    if prep is not None and prep.on:
        logits = prep.logits(Hbm.view(B * T, H), fc_b)
    else:
        logits = ops.linear(Hbm.view(B * T, H), fc_w.contiguous(), fc_b)
    return logits.view(B, T, -1), (caps, X, Hall, Hbm, saved, Hmid, emb_w, fc_w)


def _gru_decoder_backward(saved_tensors, NL, need, vocab):
    """need = needs_input_grad of (feats, captions, h0, emb_w, fc_w, fc_b, *cells); vocab = (dfc_w, dfc_b, dHbm)."""
    caps, X, Hall, Hbm, saved, Hmid, emb_w, fc_w = saved_tensors[:8]
    cells = saved_tensors[8:]
    W_ih, W_hh = cells[0], cells[1]
    B, T = caps.shape
    H = W_hh.shape[1]
    dfc_w, dfc_b, dHbm = vocab
    if NL == 1 and ops.gru_resident_ok(H):
        dGI, dGH, xdGI, xdGH, dh0 = ops.gru_resident_bwd(dHbm.view(B, T, H), saved, Hall, W_hh.contiguous())
    elif NL == 1 and ops.gru_cluster_size(H):
        dGI, dGH, xdGI, xdGH, dh0 = ops.gru_cluster_bwd(dHbm.view(B, T, H), saved, Hall, W_hh.contiguous())
    else:
        ldh = ops.round4(H)
        Whh_p = ops.copy_pad(W_hh.contiguous(), ldh)
        extra = [(ops.copy_pad(cells[4 * l].contiguous(), ldh), ops.copy_pad(cells[4 * l + 1].contiguous(), ldh))
                 for l in range(1, NL)]
        dGI, dGH, xdGI, xdGH, dh0 = ops.gru_seq_bwd(dHbm.view(B, T, H), saved, Hall, Hmid, Whh_p, extra=extra)
    Hprev = Hall[:-1].reshape(T * B, H)
    # independent chains of small launches (operand splits + a weight-gradient GEMM + a bias sum): side by side
    br = streams.Branches("ptail", like=dGI)
    br.__enter__()
    with br.on(0):
        g_wih = ops.matmul_tn(dGI, X) if need[6] else None
    with br.on(1):
        g_whh = ops.matmul_tn(dGH, Hprev) if need[7] else None
    with br.on(2):      # the bias sums only read dGI / dGH: on their own branch they are done long before the GEMM chains
        g_bih = ops.colsum(dGI) if need[8] else None
        g_bhh = ops.colsum(dGH) if need[9] else None
    cell_grads = [g_wih, g_whh, g_bih, g_bhh]
    for l in range(1, NL):
        Hin = Hmid[l - 1].reshape(T * B, H)                            # input == state of layer l
        n0 = 6 + 4 * l
        cell_grads += [ops.matmul_tn(xdGI[l - 1], Hin) if need[n0] else None,
                       ops.matmul_tn(xdGH[l - 1], Hin) if need[n0 + 1] else None,
                       ops.colsum(xdGI[l - 1]) if need[n0 + 2] else None,
                       ops.colsum(xdGH[l - 1]) if need[n0 + 3] else None]
    dfeats = demb = None
    if need[0] or need[3]:
        dX = ops.matmul_nn(dGI, W_ih.contiguous())                     # [T*B, E]
        if need[0]:
            dfeats = dX[:B].clone()
        if need[3]:
            demb = torch.zeros_like(emb_w)
            ops.embed_scatter_add(dX, caps, demb, 1)
    br.__exit__(None, None, None)
    return (dfeats, None, (dh0 if need[2] else None), demb, dfc_w if need[4] else None,
            dfc_b if need[5] else None, *cell_grads)


# ----------------------------------------------------------------------------------------------------------------------
# Variant A decoder with LSTM cells: teacher-forced DecoderRNN.forward  (reference later.py:254-324)
# ----------------------------------------------------------------------------------------------------------------------
def _lstm_decoder_forward(feats, captions, h0, emb_w, fc_w, fc_b, cells):
    B, T = captions.shape
    NL = len(cells) // 4
    W_ih, W_hh, b_ih, b_hh = cells[0:4]
    H = W_hh.shape[1]
    caps = captions.contiguous()
    X = ops.build_inputs(feats.contiguous(), emb_w.contiguous(), caps, 0)      # [T*B, E]: features at t = 0 (:277)
    GI = ops.linear(X, W_ih.contiguous(), b_ih.contiguous())                   # [T*B, 4H]
    ld4 = ops.round4(4 * H)
    WhhT = ops.transpose_pad(W_hh.contiguous(), ld4)
    extra = []
    for l in range(1, NL):
        Wi, Wh, bi, bh = cells[4 * l: 4 * l + 4]
        extra.append((ops.transpose_pad(Wi.contiguous(), ld4), ops.transpose_pad(Wh.contiguous(), ld4),
                      bi.contiguous(), bh.contiguous()))
    Hall, Hbm, saved, Hmid = ops.lstm_seq_fwd(GI, WhhT, b_hh.contiguous(), h0.contiguous(), T, save=True, extra=extra)
    logits = ops.linear(Hbm.view(B * T, H), fc_w.contiguous(), fc_b)
    return logits.view(B, T, -1), (caps, X, Hall, Hbm, saved, Hmid if Hmid is not None else Hall.new_empty(0),
                                   emb_w.contiguous(), fc_w)


def _lstm_decoder_backward(saved_tensors, NL, need, vocab):
    """need = needs_input_grad of (feats, captions, h0, emb_w, fc_w, fc_b, *cells); vocab = (dfc_w, dfc_b, dHbm)."""
    caps, X, Hall, Hbm, saved, Hmid, emb_w, fc_w = saved_tensors[:8]
    cells = saved_tensors[8:]
    W_ih, W_hh = cells[0], cells[1]
    B, T = caps.shape
    H = W_hh.shape[1]
    dfc_w, dfc_b, dHbm = vocab
    ldh = ops.round4(H)
    Whh_p = ops.copy_pad(W_hh.contiguous(), ldh)
    extra = [(ops.copy_pad(cells[4 * l].contiguous(), ldh), ops.copy_pad(cells[4 * l + 1].contiguous(), ldh))
             for l in range(1, NL)]
    dG, dh0 = ops.lstm_seq_bwd(dHbm.view(B, T, H), saved, Hall, Whh_p, extra=extra)
    Hprev = Hall[:-1].reshape(T * B, H)
    db0 = ops.colsum(dG[0]) if (need[8] or need[9]) else None
    cell_grads = [ops.matmul_tn(dG[0], X) if need[6] else None, ops.matmul_tn(dG[0], Hprev) if need[7] else None,
                  db0 if need[8] else None, (db0.clone() if need[8] else db0) if need[9] else None]
    for l in range(1, NL):
        Hin = Hmid[l - 1].reshape(T * B, H)                            # input == state of cell l
        n0 = 6 + 4 * l
        dWl = ops.matmul_tn(dG[l], Hin) if (need[n0] or need[n0 + 1]) else None
        dbl = ops.colsum(dG[l]) if (need[n0 + 2] or need[n0 + 3]) else None
        cell_grads += [dWl if need[n0] else None, (dWl.clone() if need[n0] else dWl) if need[n0 + 1] else None,
                       dbl if need[n0 + 2] else None, (dbl.clone() if need[n0 + 2] else dbl) if need[n0 + 3] else None]
    dfeats = demb = None
    if need[0] or need[3]:
        dX = ops.matmul_nn(dG[0], W_ih.contiguous())                   # [T*B, E]
        if need[0]:
            dfeats = dX[:B].clone()
        if need[3]:
            demb = torch.zeros_like(emb_w)
            ops.embed_scatter_add(dX, caps, demb, 1)
    return (dfeats, None, (dh0 if need[2] else None), demb, dfc_w if need[4] else None,
            dfc_b if need[5] else None, *cell_grads)


class DecoderRNNSeqFn(Function):
    """LSTM counterpart of DecoderGRUSeqFn: inputs feats, captions, h0, emb_w, fc_w, fc_b, then (W_ih, W_hh, b_ih, b_hh)
    of every LSTM cell.  Extra cells are applied as (h, c) = cell_l(h, (h, c)) (later.py:279-281)."""

    @staticmethod
    def forward(ctx, feats, captions, h0, emb_w, fc_w, fc_b, *cells):
        logits, sv = _lstm_decoder_forward(feats, captions, h0, emb_w, fc_w, fc_b, cells)
        ctx.save_for_backward(*sv, *cells)
        ctx.NL = len(cells) // 4
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        sv = ctx.saved_tensors
        Hbm, fc_w = sv[3], sv[7]
        B, T, H = Hbm.shape
        need = ctx.needs_input_grad
        dl = dlogits.reshape(B * T, -1).contiguous()
        vocab = vocab_bwd_from_dlogits(dl, Hbm.view(B * T, H), fc_w, need[4], need[5])
        return _lstm_decoder_backward(sv, ctx.NL, need, vocab)


class DecoderRNNLossFn(Function):
    """DecoderRNN + mean cross-entropy as one autograd node (see DecoderGRULossFn)."""

    @staticmethod
    def forward(ctx, ignore_index, feats, captions, h0, emb_w, fc_w, fc_b, *cells):
        logits, sv = _lstm_decoder_forward(feats, captions, h0, emb_w, fc_w, fc_b, cells)
        B, T, V = logits.shape
        targets = captions.reshape(-1).contiguous()
        lossbuf, lse, dhi, dlo = ce_fwd_for_loss(logits.view(B * T, V), targets, ignore_index, sv[3].shape[-1],
                                                 any(ctx.needs_input_grad))
        ctx.save_for_backward(*sv, *cells, logits, targets, lse, lossbuf, dhi, dlo)
        ctx.NL = len(cells) // 4
        ctx.ignore_index = ignore_index
        ctx.mark_non_differentiable(logits)
        ctx.set_materialize_grads(False)
        return lossbuf[0].clone(), logits

    @staticmethod
    def backward(ctx, g, _unused):
        allsv = ctx.saved_tensors
        sv, (logits, targets, lse, lossbuf, dhi, dlo) = allsv[:-6], allsv[-6:]
        Hbm, fc_w = sv[3], sv[7]
        B, T, H = Hbm.shape
        need = ctx.needs_input_grad[1:]
        g = g.reshape(1).to(torch.float32).contiguous()
        vocab = vocab_bwd_fused(logits.view(B * T, -1), targets, ctx.ignore_index, lse, lossbuf, g,
                                Hbm.view(B * T, H), fc_w, dhi, dlo)
        return (None, *_lstm_decoder_backward(sv, ctx.NL, need, vocab))


class DecoderGRUSeqFn(Function):
    """inputs: feats, captions, h0, emb_w, fc_w, fc_b, then (W_ih, W_hh, b_ih, b_hh) for every GRU cell (layer 0 first).
    Extra layers are applied as h = cell_l(h, h) at every step (later.py:413-414, 420-421).  Returns logits [B,T,V]."""

    @staticmethod
    def forward(ctx, feats, captions, h0, emb_w, fc_w, fc_b, *cells):
        logits, sv = _gru_decoder_forward(feats, captions, h0, emb_w, fc_w, fc_b, cells)
        ctx.save_for_backward(*sv, *cells)
        ctx.NL = len(cells) // 4
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        sv = ctx.saved_tensors
        Hbm, fc_w = sv[3], sv[7]
        B, T, H = Hbm.shape
        need = ctx.needs_input_grad
        dl = dlogits.reshape(B * T, -1).contiguous()
        vocab = vocab_bwd_from_dlogits(dl, Hbm.view(B * T, H), fc_w, need[4], need[5])
        return _gru_decoder_backward(sv, ctx.NL, need, vocab)


class DecoderGRULossFn(Function):
    """Decoder + mean cross-entropy as ONE autograd node (hypernet.py:139-145 computes exactly this pair): returns
    (loss, logits) with logits non-differentiable; the backward never materialises fp32 dlogits."""

    @staticmethod
    def forward(ctx, ignore_index, feats, captions, h0, emb_w, fc_w, fc_b, *cells):
        Bc, Tc = captions.shape
        prep = VocabPrep(Bc * Tc, fc_w.shape[0], cells[1].shape[1], any(ctx.needs_input_grad), feats)
        logits, sv = _gru_decoder_forward(feats, captions, h0, emb_w, fc_w, fc_b, cells, prep=prep)
        B, T, V = logits.shape
        targets = captions.reshape(-1).contiguous()
        lossbuf, lse, dhi, dlo = ce_fwd_for_loss(logits.view(B * T, V), targets, ignore_index, sv[3].shape[-1],
                                                 any(ctx.needs_input_grad))
        prep.finish()
        ctx.save_for_backward(*sv, *cells, logits, targets, lse, lossbuf, dhi, dlo, *prep.saved())
        ctx.NL = len(cells) // 4
        ctx.ignore_index = ignore_index
        ctx.mark_non_differentiable(logits)
        ctx.set_materialize_grads(False)   # do not zero-fill a [B,T,V] gradient for the unused logits output
        return lossbuf[0].clone(), logits

    @staticmethod
    def backward(ctx, g, _unused):
        allsv = ctx.saved_tensors
        sv, (logits, targets, lse, lossbuf, dhi, dlo), pre = allsv[:-10], allsv[-10:-4], allsv[-4:]
        Hbm, fc_w = sv[3], sv[7]
        B, T, H = Hbm.shape
        need = ctx.needs_input_grad[1:]
        g = g.reshape(1).to(torch.float32).contiguous()
        vocab = vocab_bwd_fused(logits.view(B * T, -1), targets, ctx.ignore_index, lse, lossbuf, g,
                                Hbm.view(B * T, H), fc_w, dhi, dlo, pre)
        return (None, *_gru_decoder_backward(sv, ctx.NL, need, vocab))
