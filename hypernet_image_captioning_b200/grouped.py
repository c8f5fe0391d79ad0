"""Many-style ("grouped") execution of the attention variant: one batch whose rows use G different generated weight sets.

BASELINE.json configs[3] / north star: "Conceptual Captions domain-conditioned hypernet-GRU with many domains -> many-group
grouped GEMM", "the per-style grouped GEMM that projects all timesteps' word embeddings", "keeps each style group's
generated W_hh resident".  Reference semantics: one ``HyperNet.forward`` + captioner call per sample's style
(train_cc.py:90-123; cc_train_hypernet.py:134-153 is the G = 1 case) -- the oracle of the tests is exactly that loop.

Layouts.  The batch is sorted by group (``order``).  The recurrence keeps the time-major layout ``row = t*B + b`` of the
single-style path, so a row tile of one group is contiguous at every step and the step-split kernels only need a tile
table (first row, rows, group) and one weight pack per group.  The time-batched tensor-core products want every group's
rows of ALL steps contiguous: "group-major" ``row = gm_off[g] + t*cnt[g] + j`` with each group's block padded to a
multiple of 64 rows (the K block of the weight-gradient products).  ``ops.split_bf16_gather`` produces the bf16 hi/lo
operands directly in that order, and the x-projection's epilogue scatters its rows back through the same map, so the
permutation never costs a pass of its own.

    x-projection   GIw[row]  = X[row] . W_ih[g][:, :E]^T + b_ih[g]        grouped GEMM, A = X (group-major), B = W_ih[g]
    dX             dXw[row]  = dGI[row] . W_ih[g][:, :E]                  grouped GEMM, B read MN-major from the same split
    dW_ih[g]       = dGI_g^T . [x | ctx]_g      dW_hh[g] = dGH_g^T . Hprev_g        grouped GEMMs over each group's K range,
                                                                                   written straight into dTheta[g]
    db_ih[g], db_hh[g]                                                    ops.group_colsum
"""
from typing import Dict, Tuple

import numpy as np
import torch
from torch.autograd import Function

from . import functional as Fn
from . import ops


def _r64(n):
    return (n + 63) // 64 * 64


class GroupPlan:
    """Host-side description of one batch composition (which row belongs to which style group), built once per distinct
    ``groups`` vector and cached: permutation, group-major row map, recurrence tile tables, grouped-GEMM unit tables."""

    _cache: Dict[Tuple, "GroupPlan"] = {}

    @classmethod
    def get(cls, groups: torch.Tensor, G: int, T: int, device) -> "GroupPlan":
        """``groups``: [B] integer group id per batch row.  Pass a CPU tensor (the domain of a sample is host data in the
        reference's loaders, cc_train_hypernet.py:135-137): a CUDA tensor costs a device->host copy + synchronisation per
        call and cannot be used while a CUDA graph is being captured."""
        g_host = groups.detach().to("cpu", torch.int64).numpy()
        key = (g_host.tobytes(), G, T, str(device))
        plan = cls._cache.get(key)
        if plan is None:
            if len(cls._cache) > 64:
                cls._cache.clear()
            plan = cls._cache[key] = GroupPlan(g_host, G, T, device)
        return plan

    def __init__(self, g_host: np.ndarray, G: int, T: int, device):
        B = int(g_host.shape[0])
        if B == 0 or g_host.min() < 0 or g_host.max() >= G:
            raise ValueError("group ids must lie in [0, G)")
        self.B, self.G, self.T, self.device = B, G, T, device
        order = np.argsort(g_host, kind="stable")
        inv = np.empty_like(order)
        inv[order] = np.arange(B)
        cnt = np.bincount(g_host, minlength=G).astype(np.int64)
        goff = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
        self.cnt, self.goff = cnt, goff
        self.present = [int(g) for g in range(G) if cnt[g] > 0]
        gm_cnt = T * cnt
        gm_pad = (gm_cnt + 63) // 64 * 64
        gm_off = np.concatenate([[0], np.cumsum(gm_pad)]).astype(np.int64)
        self.gm_cnt, self.gm_pad, self.gm_off = gm_cnt, gm_pad, gm_off
        self.R_gm = int(gm_off[-1])
        gm2tm = np.full(self.R_gm, -1, np.int32)
        for g in self.present:
            c = int(cnt[g])
            tm = (np.arange(T)[:, None] * B + goff[g] + np.arange(c)[None, :]).reshape(-1)   # (t, j) -> t*B + goff + j
            gm2tm[gm_off[g]: gm_off[g] + T * c] = tm
        i64 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(device)
        i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device)
        self.order, self.inv = i64(order), i64(inv)
        self.gm2tm = i32(gm2tm)
        self.goff_dev = i32(goff)
        # recurrence row tiles: groups of <= 8 rows (a many-domain batch) take the small-tile kernels
        small = int(cnt.max()) <= 8
        self.tile_rows_fwd, self.tile_rows_bwd = (8, 8) if small else (64, 32)
        self.tiles_fwd = i32(self._tiles(self.tile_rows_fwd))
        self.tiles_bwd = i32(self._tiles(self.tile_rows_bwd))
        self.tiles8 = i32(self._tiles(8))                           # 8-row tiles: the weights-resident cluster GRU (pooled variant)
        self.tiles4 = i32(self._tiles(4))                           # 4-row tiles: the streaming LSTM recurrence (pooled variant)
        absent = [g for g in range(G) if cnt[g] == 0]
        self.absent_dev = i64(absent) if absent else None         # groups without rows: their d(theta) rows are zero
        self._units: Dict[Tuple, torch.Tensor] = {}

    def _tiles(self, nb):
        out = []
        for g in self.present:
            for r in range(int(self.goff[g]), int(self.goff[g + 1]), nb):
                out.append((r, min(nb, int(self.goff[g + 1]) - r), g, 0))
        return np.array(out, np.int32).reshape(-1, 4)

    # -- grouped-GEMM unit tables: rows of 12 int32 {a_row, b_row, ka0, kb0, nkb, m_valid, n_valid, bias_off, map0, c_lo, c_hi, 0}
    def _dev_units(self, key, rows):
        if key not in self._units:
            arr = np.array(rows, np.int64).reshape(-1, 12)
            c = arr[:, 9].copy()                       # 64-bit C offset -> low / high words
            arr[:, 9] = c & 0xFFFFFFFF
            arr[:, 10] = c >> 32
            arr[:, 9] = np.where(arr[:, 9] >= 2 ** 31, arr[:, 9] - 2 ** 32, arr[:, 9])   # as a signed 32-bit pattern
            self._units[key] = torch.from_numpy(arr.astype(np.int32)).to(self.device)
        return self._units[key]

    def units_xproj(self, H3, K, BN):
        """GIw (time-major, through gm2tm) = X_gm . W[g]^T + b[g]; B rows g*H3.., K columns from 0."""
        rows = []
        nkb = (K + 63) // 64
        for g in self.present:
            n = int(self.gm_cnt[g])
            for m0 in range(0, n, 128):
                a_row = int(self.gm_off[g]) + m0
                for n0 in range(0, H3, BN):
                    rows.append((a_row, g * H3 + n0, 0, 0, nkb, min(128, n - m0), min(BN, H3 - n0), g * H3 + n0, a_row,
                                 n0, 0, 0))
        return self._dev_units(("xproj", H3, K, BN), rows)

    def units_dx(self, H3, E, BN):
        """dX (time-major, through gm2tm) = dGI_gm . W[g][:, :E]; B = the W split read MN-major: k rows g*H3.., N columns 0..E."""
        rows = []
        nkb = (H3 + 63) // 64
        for g in self.present:
            n = int(self.gm_cnt[g])
            for m0 in range(0, n, 128):
                a_row = int(self.gm_off[g]) + m0
                for n0 in range(0, E, BN):
                    rows.append((a_row, n0, 0, g * H3, nkb, min(128, n - m0), min(BN, E - n0), 0, a_row, n0, 0, 0))
        return self._dev_units(("dx", H3, E, BN), rows)

    def units_dw(self, H3, N, BN, theta, base, ldc):
        """dW[g] [H3, N] = dG_gm[g]^T . X_gm[g] over the group's (padded) K range, written at dTheta[g, base:]."""
        rows = []
        for g in self.present:
            k0, nkb = int(self.gm_off[g]), int(self.gm_pad[g]) // 64
            for m0 in range(0, H3, 128):
                for n0 in range(0, N, BN):
                    rows.append((m0, n0, k0, k0, nkb, min(128, H3 - m0), min(BN, N - n0), 0, 0,
                                 g * theta + base + m0 * ldc + n0, 0, 0))
        return self._dev_units(("dw", H3, N, BN, theta, base, ldc), rows)


class RowPermuteFn(Function):
    """y[i] = x[idx[i]] for a permutation idx (rows of a [B, ...] tensor); backward gathers with the inverse permutation."""

    @staticmethod
    def forward(ctx, x, idx, inv):
        ctx.save_for_backward(inv)
        ctx.shape = x.shape
        x2 = x.reshape(x.shape[0], -1).contiguous()
        return ops.gather_rows(x2, idx).reshape(x.shape)

    @staticmethod
    def backward(ctx, g):
        (inv,) = ctx.saved_tensors
        g2 = g.reshape(g.shape[0], -1).contiguous()
        return ops.gather_rows(g2, inv).reshape(ctx.shape), None, None


def _layout(E, Fd, H):
    """Offsets of (W_ih [3H, E+F], W_hh [3H, H], b_ih [3H], b_hh [3H]) inside one row of Theta (utils.py:55-60 order)."""
    H3 = 3 * H
    o_hh = H3 * (E + Fd)
    o_bi = o_hh + H3 * H
    o_bh = o_bi + H3
    return H3, o_hh, o_bi, o_bh, o_bh + H3


def _grouped_forward(plan: GroupPlan, f3, K3, h0, caps, Theta, emb_w, fc_w, fc_b, Ua_w, Ua_b, va_w, va_b):
    """Teacher-forced AttentionGru time loop for a batch SORTED by style group (f3, K3, h0, caps already permuted).
    Returns logits / attention weights in the ORIGINAL batch order and the tensors the backward needs."""
    B, P, Fd = f3.shape
    T = caps.shape[1]
    E, H, V = emb_w.shape[1], Ua_w.shape[0], fc_w.shape[0]
    G, theta = Theta.shape
    H3, o_hh, o_bi, o_bh, total = _layout(E, Fd, H)
    assert theta == total and plan.B == B and plan.T == T and plan.G == G
    dev = f3.device
    Theta = Theta.contiguous()
    f3, K3 = f3.contiguous(), K3.contiguous()
    emb_w = emb_w.contiguous()
    # per-group weight packs for the recurrence; bias tables [G, 3H]
    gw = ops.AttGruGroupWeights(Theta, Ua_w.contiguous(), E, Fd, H, P)
    b_ih_g = Theta[:, o_bi:o_bh].contiguous()
    b_hh_g = Theta[:, o_bh:].contiguous()
    va, bv = va_w.reshape(-1).contiguous(), va_b.reshape(1).contiguous()
    # word inputs (time-major, sorted batch): x_0 = x_1 = 0, x_t = Emb[caps[:, t-1]]  (models/decoderlstm.py:82-88)
    fed = torch.full((T, B), -1, device=dev, dtype=torch.int64)
    if T > 2:
        fed[2:] = caps[:, 1:T - 1].t()
    Xw = ops.build_inputs(None, emb_w, caps, 1)                            # [T*B, E]
    XC = torch.empty(T * B, E + Fd, device=dev, dtype=torch.float32)       # [x_word | ctx] per (t, b)
    XC[:, :E].copy_(Xw)
    # grouped x-projection: A = X in group-major order, B = W_ih of every group (one operand array [G*3H, Kp])
    Wsp = ops.split_bf16_batched(Theta, theta, E + Fd, G, H3, E + Fd)
    Xgm = ops.split_bf16_gather(Xw, plan.gm2tm, plan.R_gm)
    GIw = torch.empty(T * B, H3, device=dev, dtype=torch.float32)
    ops.gemm_tc_grouped(Xgm, False, Wsp, False, GIw, H3, plan.units_xproj(H3, E, 128), 128, bias=b_ih_g,
                        rowmap=plan.gm2tm)
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32)
    attn = torch.empty(B, T, P, device=dev, dtype=torch.float32)
    saved = torch.empty(5, T, B, H, device=dev, dtype=torch.float32)
    ops.attgru_fwd_grouped(K3, f3, GIw, gw, Ua_b.contiguous(), va, bv, b_hh_g, Hall, Hbm, attn, XC, E, saved,
                           plan.tiles_fwd, plan.tile_rows_fwd)
    # back to the caller's batch order before the vocabulary projection: logits [B, T, V] (0.4 GB) are never permuted
    Hbm_o = ops.gather_rows(Hbm.view(B, T * H), plan.inv).view(B, T, H)
    attn_o = ops.gather_rows(attn.view(B, T * P), plan.inv).view(B, T, P)
    logits = ops.linear(Hbm_o.view(B * T, H), fc_w, fc_b).view(B, T, V)
    sv = (f3, K3, XC, Hall, Hbm_o, attn, saved, fed, emb_w, Theta, fc_w, Ua_w, va, Wsp.hi, Wsp.lo)
    return logits, attn_o, sv, (B, T, P, E, H, Fd, V, G)


def _grouped_backward(plan: GroupPlan, sv, dims, vocab, dattn_o):
    """vocab = (dfc_w, dfc_b, dHbm in the ORIGINAL batch order [B*T, H]).  Returns gradients of
    (f3, K3, h0 [sorted order], Theta, emb_w, fc_w, fc_b, Ua_w, Ua_b, va_w, va_b)."""
    f3, K3, XC, Hall, Hbm_o, attn, saved, fed, emb_w, Theta, fc_w, Ua_w, va, Wsp_hi, Wsp_lo = sv
    B, T, P, E, H, Fd, V, G = dims
    H3, o_hh, o_bi, o_bh, theta = _layout(E, Fd, H)
    dfc_w, dfc_b, dHbm_o = vocab
    dev = f3.device
    dHbm = ops.gather_rows(dHbm_o.reshape(B, T * H).contiguous(), plan.order).view(B, T, H)
    dattn = None
    if dattn_o is not None:
        dattn = ops.gather_rows(dattn_o.reshape(B, T * P).contiguous(), plan.order).view(B, T, P)
    dGI, dGH, dU, dCTX, dK, dva, dbv, dh0 = ops.attgru_bwd_grouped(dHbm, dattn, K3, f3, attn, saved, Hall, Theta,
                                                                    Ua_w.contiguous(), va, E, plan.tiles_bwd,
                                                                    plan.tile_rows_bwd)
    Hprev = Hall[:-1].reshape(T * B, H)
    # shared attention parameter U_a: plain products over all rows
    dUa_w = ops.matmul_tn(dU, Hprev)
    dUa_b = ops.colsum(dU)
    # group-major bf16 operands of the gate gradients and of the cell inputs
    R = plan.R_gm
    dGI_gm = ops.split_bf16_gather(dGI, plan.gm2tm, R)
    dGH_gm = ops.split_bf16_gather(dGH, plan.gm2tm, R)
    XC_gm = ops.split_bf16_gather(XC, plan.gm2tm, R)
    Hp_gm = ops.split_bf16_gather(Hprev, plan.gm2tm, R)
    dTheta = torch.empty(G, theta, device=dev, dtype=torch.float32)
    dTheta[:, o_bi:].zero_()
    if plan.absent_dev is not None:
        dTheta.index_fill_(0, plan.absent_dev, 0.0)
    mn = lambda op: ops.SplitOperand(op.hi, op.lo, op.K, op.rows, op.ld, True)
    ops.gemm_tc_grouped(mn(dGI_gm), True, mn(XC_gm), True, dTheta, E + Fd,
                        plan.units_dw(H3, E + Fd, 128, theta, 0, E + Fd), 128)
    ops.gemm_tc_grouped(mn(dGH_gm), True, mn(Hp_gm), True, dTheta, H,
                        plan.units_dw(H3, H, 128, theta, o_hh, H), 128)
    ops.group_colsum(dGI, plan.goff_dev, G, B, T, dTheta[:, o_bi:o_bh])
    ops.group_colsum(dGH, plan.goff_dev, G, B, T, dTheta[:, o_bh:])
    # word embeddings: dXw = dGI . W_ih[g][:, :E] (grouped), scattered to the rows that were fed
    Wsp = ops.SplitOperand(Wsp_hi, Wsp_lo, E + Fd, G * H3, Wsp_hi.shape[1], True)
    dXw = torch.empty(T * B, E, device=dev, dtype=torch.float32)
    ops.gemm_tc_grouped(dGI_gm, False, Wsp, True, dXw, E, plan.units_dx(H3, E, 128), 128, rowmap=plan.gm2tm)
    demb = torch.zeros_like(emb_w)
    ops.scatter_add_rows(dXw, fed.reshape(-1), demb)
    df = torch.zeros(B, P, Fd, device=dev, dtype=torch.float32)
    ops.attn_df(attn, dCTX, df)
    return (df, dK, dh0, dTheta, demb, dfc_w, dfc_b, dUa_w, dUa_b, dva.view(1, H), dbv.view(1))


class AttentionGruGroupedFn(Function):
    """Teacher-forced AttentionGru.forward for a many-style batch as one autograd node.  Inputs: plan, then f3, K3, h0,
    captions (all SORTED by group), Theta [G, theta], emb_w, fc_w, fc_b, U_a (w, b), v_a (w, b).  Outputs in the original
    batch order."""

    @staticmethod
    def forward(ctx, plan, f3, K3, h0, caps, *params):
        logits, attn_o, sv, dims = _grouped_forward(plan, f3, K3, h0, caps, *params)
        ctx.save_for_backward(*sv)
        ctx.plan, ctx.dims = plan, dims
        return logits, attn_o

    @staticmethod
    def backward(ctx, dlogits, dattn):
        sv = ctx.saved_tensors
        B, T, P, E, H, Fd, V, G = ctx.dims
        dl = dlogits.reshape(B * T, V).contiguous()
        vocab = Fn.vocab_bwd_from_dlogits(dl, sv[4].view(B * T, H), sv[10])
        g = _grouped_backward(ctx.plan, sv, ctx.dims, vocab, dattn)
        return (None, *g[:3], None, *g[3:])


class AttentionGruGroupedLossFn(Function):
    """AttentionGruGroupedFn + F.cross_entropy(ignore_index) as one node (cc_train_hypernet.py:152-153 for a many-style
    batch): returns (loss, logits, attn); the captions of the loss are in the ORIGINAL order (``caps_o``)."""

    @staticmethod
    def forward(ctx, ignore_index, plan, caps_o, f3, K3, h0, caps, *params):
        logits, attn_o, sv, dims = _grouped_forward(plan, f3, K3, h0, caps, *params)
        B, T, V = logits.shape
        targets = caps_o.reshape(-1).contiguous()
        lossbuf, lse, dhi, dlo = Fn.ce_fwd_for_loss(logits.view(B * T, V), targets, ignore_index, dims[4],
                                                    any(ctx.needs_input_grad))
        ctx.save_for_backward(*sv, logits, targets, lse, lossbuf, dhi, dlo)
        ctx.plan, ctx.dims, ctx.ignore_index = plan, dims, ignore_index
        ctx.mark_non_differentiable(logits, attn_o)
        ctx.set_materialize_grads(False)
        return lossbuf[0].clone(), logits, attn_o

    @staticmethod
    def backward(ctx, g, _dl, _da):
        allsv = ctx.saved_tensors
        sv, (logits, targets, lse, lossbuf, dhi, dlo) = allsv[:-6], allsv[-6:]
        B, T, P, E, H, Fd, V, G = ctx.dims
        g = g.reshape(1).to(torch.float32).contiguous()
        vocab = Fn.vocab_bwd_fused(logits.view(B * T, V), targets, ctx.ignore_index, lse, lossbuf, g,
                                   sv[4].view(B * T, H), sv[10], dhi, dlo)
        gr = _grouped_backward(ctx.plan, sv, ctx.dims, vocab, None)
        return (None, None, None, *gr[:3], None, *gr[3:])


# ----------------------------------------------------------------------------------------------------------------------
# pooled variant (hypernet.HyperNet + DecoderGRU / DecoderRNN, single layer): grouped x-projection, then either the
# weights-resident cluster GRU whose clusters each keep THEIR group's W_hh in shared memory for all T steps, or the
# streaming LSTM recurrence whose CTAs each run a <= 4-row tile of one group against that group's slice of a W_hh pack
# ----------------------------------------------------------------------------------------------------------------------
def _layout_pooled(E, H, gates=3):
    """Offsets of (W_ih [gH, E], W_hh [gH, H], b_ih, b_hh) inside one row of Theta (hypernet.py:62-68 parameter order);
    g = 3 gates for the GRU cell, 4 for the LSTM cell."""
    NG = gates * H
    o_hh = NG * E
    o_bi = o_hh + NG * H
    o_bh = o_bi + NG
    return NG, o_hh, o_bi, o_bh, o_bh + NG


def _pooled_grouped_forward(plan: GroupPlan, lstm, feats, caps, h0, Theta, emb_w, fc_w, fc_b):
    """Teacher-forced DecoderGRU.forward (later.py:389-457) or, with ``lstm``, DecoderRNN.forward (later.py:254-324), one
    layer, for a batch SORTED by style group.  Returns logits in the ORIGINAL batch order."""
    B, T = caps.shape
    E, H, V = emb_w.shape[1], fc_w.shape[1], fc_w.shape[0]
    G, theta = Theta.shape
    NG, o_hh, o_bi, o_bh, total = _layout_pooled(E, H, 4 if lstm else 3)
    assert theta == total and plan.B == B and plan.T == T and plan.G == G
    dev = feats.device
    Theta = Theta.contiguous()
    emb_w = emb_w.contiguous()
    X = ops.build_inputs(feats.contiguous(), emb_w, caps, 0)                # [T*B, E] time-major: x_0 = feature, x_t = Emb[caps[:, t-1]]
    b_ih_g = Theta[:, o_bi:o_bh].contiguous()
    Wsp = ops.split_bf16_batched(Theta, theta, E, G, NG, E)                  # W_ih of every group: [G*gH, Kp]
    Xgm = ops.split_bf16_gather(X, plan.gm2tm, plan.R_gm)
    GI = torch.empty(T * B, NG, device=dev, dtype=torch.float32)
    ops.gemm_tc_grouped(Xgm, False, Wsp, False, GI, NG, plan.units_xproj(NG, E, 128), 128, bias=b_ih_g, rowmap=plan.gm2tm)
    if lstm:
        WhhT = ops.transpose_pad_batched(Theta[:, o_hh:o_bi], NG, H, ops.round4(NG))     # [G, H, ld4]
        Hall, Hbm, saved = ops.lstm_seq_fwd_grouped(GI, WhhT, Theta[:, o_bh:], h0, T, plan.tiles4)
    else:
        Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
        Hall[0].copy_(h0)
        Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32)
        saved = torch.empty(1, 4, T, B, H, device=dev, dtype=torch.float32)
        ops._cabi.call("caphn_gru_cluster_fwd_grouped", GI.data_ptr(), Theta.data_ptr() + 4 * o_hh,
                       Theta.data_ptr() + 4 * o_bh, Hall.data_ptr(), Hbm.data_ptr(), saved.data_ptr(), B, T, H,
                       plan.tiles8.data_ptr(), plan.tiles8.shape[0], theta, theta, ops._stream())
    Hbm_o = ops.gather_rows(Hbm.view(B, T * H), plan.inv).view(B, T, H)
    logits = ops.linear(Hbm_o.view(B * T, H), fc_w.contiguous(), fc_b).view(B, T, V)
    sv = (caps, X, Hall, Hbm_o, saved, emb_w, Theta, fc_w, Wsp.hi, Wsp.lo)
    return logits, sv, (B, T, E, H, V, G)


def _pooled_grouped_backward(plan: GroupPlan, lstm, sv, dims, vocab, need_feats):
    caps, X, Hall, Hbm_o, saved, emb_w, Theta, fc_w, Wsp_hi, Wsp_lo = sv
    B, T, E, H, V, G = dims
    NG, o_hh, o_bi, o_bh, theta = _layout_pooled(E, H, 4 if lstm else 3)
    dfc_w, dfc_b, dHbm_o = vocab
    dev = X.device
    dHbm = ops.gather_rows(dHbm_o.reshape(B, T * H).contiguous(), plan.order).view(B, T, H)
    if lstm:
        # the LSTM pre-activation is the plain sum gi + gh: one gate gradient dG serves both weight products and both biases
        Whh_p = ops.copy_pad_batched(Theta[:, o_hh:o_bi], NG, H, ops.round4(H))          # [G, 4H, ldh]
        dGI, dh0 = ops.lstm_seq_bwd_grouped(dHbm, saved, Hall, Whh_p, plan.tiles4)
        dGH = dGI
    else:
        dGI = torch.empty(T * B, NG, device=dev, dtype=torch.float32)
        dGH = torch.empty(T * B, NG, device=dev, dtype=torch.float32)
        dh0 = torch.empty(B, H, device=dev, dtype=torch.float32)
        ops._cabi.call("caphn_gru_cluster_bwd_grouped", dHbm.data_ptr(), saved.data_ptr(), Hall.data_ptr(),
                       Theta.data_ptr() + 4 * o_hh, dGI.data_ptr(), dGH.data_ptr(), dh0.data_ptr(), B, T, H,
                       plan.tiles8.data_ptr(), plan.tiles8.shape[0], theta, ops._stream())
    Hprev = Hall[:-1].reshape(T * B, H)
    R = plan.R_gm
    dGI_gm = ops.split_bf16_gather(dGI, plan.gm2tm, R)
    dGH_gm = dGI_gm if dGH is dGI else ops.split_bf16_gather(dGH, plan.gm2tm, R)
    X_gm = ops.split_bf16_gather(X, plan.gm2tm, R)
    Hp_gm = ops.split_bf16_gather(Hprev, plan.gm2tm, R)
    dTheta = torch.empty(G, theta, device=dev, dtype=torch.float32)
    dTheta[:, o_bi:].zero_()
    if plan.absent_dev is not None:
        dTheta.index_fill_(0, plan.absent_dev, 0.0)
    mn = lambda op: ops.SplitOperand(op.hi, op.lo, op.K, op.rows, op.ld, True)
    ops.gemm_tc_grouped(mn(dGI_gm), True, mn(X_gm), True, dTheta, E, plan.units_dw(NG, E, 128, theta, 0, E), 128)
    ops.gemm_tc_grouped(mn(dGH_gm), True, mn(Hp_gm), True, dTheta, H, plan.units_dw(NG, H, 128, theta, o_hh, H), 128)
    ops.group_colsum(dGI, plan.goff_dev, G, B, T, dTheta[:, o_bi:o_bh])
    ops.group_colsum(dGH, plan.goff_dev, G, B, T, dTheta[:, o_bh:])
    Wsp = ops.SplitOperand(Wsp_hi, Wsp_lo, E, G * NG, Wsp_hi.shape[1], True)
    dX = torch.empty(T * B, E, device=dev, dtype=torch.float32)
    ops.gemm_tc_grouped(dGI_gm, False, Wsp, True, dX, E, plan.units_dx(NG, E, 128), 128, rowmap=plan.gm2tm)
    dfeats = dX[:B].clone() if need_feats else None                       # rows of t = 0 (sorted order)
    demb = torch.zeros_like(emb_w)
    ops.embed_scatter_add(dX, caps, demb, 1)
    return dfeats, dh0, dTheta, demb, dfc_w, dfc_b


class DecoderGRUGroupedFn(Function):
    """Teacher-forced DecoderGRU.forward (single layer) for a many-style batch.  Inputs: plan, then feats [B,E], captions,
    h0 (all SORTED by group), Theta [G, theta], emb_w, fc_w, fc_b.  Logits come back in the original batch order."""

    @staticmethod
    def forward(ctx, plan, feats, caps, h0, Theta, emb_w, fc_w, fc_b):
        return _pooled_fn_forward(ctx, False, plan, feats, caps, h0, Theta, emb_w, fc_w, fc_b)

    @staticmethod
    def backward(ctx, dlogits):
        sv = ctx.saved_tensors
        B, T, E, H, V, G = ctx.dims
        dl = dlogits.reshape(B * T, V).contiguous()
        vocab = Fn.vocab_bwd_from_dlogits(dl, sv[3].view(B * T, H), sv[7])
        dfeats, dh0, dTheta, demb, dfc_w, dfc_b = _pooled_grouped_backward(ctx.plan, ctx.lstm, sv, ctx.dims, vocab,
                                                                         ctx.needs_input_grad[1])
        return None, dfeats, None, dh0 if ctx.needs_input_grad[3] else None, dTheta, demb, dfc_w, dfc_b


class DecoderRNNGroupedFn(DecoderGRUGroupedFn):
    """DecoderGRUGroupedFn for the LSTM captioner (DecoderRNN, single layer): same inputs and outputs."""

    @staticmethod
    def forward(ctx, plan, feats, caps, h0, Theta, emb_w, fc_w, fc_b):
        return _pooled_fn_forward(ctx, True, plan, feats, caps, h0, Theta, emb_w, fc_w, fc_b)


def _pooled_fn_forward(ctx, lstm, plan, *args):
    logits, sv, dims = _pooled_grouped_forward(plan, lstm, *args)
    ctx.save_for_backward(*sv)
    ctx.plan, ctx.dims, ctx.lstm = plan, dims, lstm
    return logits


class DecoderGRUGroupedLossFn(Function):
    """DecoderGRUGroupedFn + mean cross-entropy (hypernet.py:139-145 for a many-style batch; ``ignore_index`` None = no
    masking) as one node: returns (loss, logits).  The captions of the loss are in the ORIGINAL order (``caps_o``); the
    one-pass CE kernel writes the softmax gradient as tensor-core operands, so fp32 dlogits never exist."""

    @staticmethod
    def forward(ctx, ignore_index, plan, caps_o, feats, caps, h0, Theta, emb_w, fc_w, fc_b):
        return _pooled_loss_forward(ctx, False, ignore_index, plan, caps_o, feats, caps, h0, Theta, emb_w, fc_w, fc_b)

    @staticmethod
    def backward(ctx, g, _dl):
        allsv = ctx.saved_tensors
        sv, (logits, targets, lse, lossbuf, dhi, dlo) = allsv[:-6], allsv[-6:]
        B, T, E, H, V, G = ctx.dims
        g = g.reshape(1).to(torch.float32).contiguous()
        vocab = Fn.vocab_bwd_fused(logits.view(B * T, V), targets, ctx.ignore_index, lse, lossbuf, g,
                                   sv[3].view(B * T, H), sv[7], dhi, dlo)
        dfeats, dh0, dTheta, demb, dfc_w, dfc_b = _pooled_grouped_backward(ctx.plan, ctx.lstm, sv, ctx.dims, vocab,
                                                                         ctx.needs_input_grad[3])
        return (None, None, None, dfeats, None, dh0 if ctx.needs_input_grad[5] else None, dTheta, demb, dfc_w, dfc_b)


class DecoderRNNGroupedLossFn(DecoderGRUGroupedLossFn):
    """DecoderGRUGroupedLossFn for the LSTM captioner (DecoderRNN, single layer): same inputs and outputs."""

    @staticmethod
    def forward(ctx, ignore_index, plan, caps_o, feats, caps, h0, Theta, emb_w, fc_w, fc_b):
        return _pooled_loss_forward(ctx, True, ignore_index, plan, caps_o, feats, caps, h0, Theta, emb_w, fc_w, fc_b)


def _pooled_loss_forward(ctx, lstm, ignore_index, plan, caps_o, *args):
    logits, sv, dims = _pooled_grouped_forward(plan, lstm, *args)
    B, T, V = logits.shape
    targets = caps_o.reshape(-1).contiguous()
    lossbuf, lse, dhi, dlo = Fn.ce_fwd_for_loss(logits.view(B * T, V), targets, ignore_index, dims[3],
                                                any(ctx.needs_input_grad))
    ctx.save_for_backward(*sv, logits, targets, lse, lossbuf, dhi, dlo)
    ctx.plan, ctx.dims, ctx.lstm, ctx.ignore_index = plan, dims, lstm, ignore_index
    ctx.mark_non_differentiable(logits)
    ctx.set_materialize_grads(False)
    return lossbuf[0].clone(), logits


# ----------------------------------------------------------------------------------------------------------------------
# hypernetwork for many style vectors: X [G, he] -> Theta [G, theta] with the layers as dense tensor-core GEMMs
# ----------------------------------------------------------------------------------------------------------------------
def _sk(M, N, K):
    """Split-K factor for a small exact-fp32 product whose output is one or two 128 x 128 tiles: spread K over CTAs."""
    tiles = ((M + 127) // 128) * ((N + 127) // 128)
    return max(1, min(32, K // 64, 64 // tiles))


def _small_linear(x, W, b, out=None):
    """y = x W^T + b for the hypernet's small layers at G <= a few hundred rows (exact fp32, K split over CTAs)."""
    M, K = x.shape
    N = W.shape[0]
    sk = _sk(M, N, K)
    if sk == 1:
        return ops._gemm(x, x.stride(0), 1, W, W.stride(0), 1, M, N, K, b, False, out)
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=torch.float32)
    out.copy_(b.to(torch.float32).reshape(1, N).expand(M, N))          # bias first, then the K chunks accumulate atomically
    return ops._gemm(x, x.stride(0), 1, W, W.stride(0), 1, M, N, K, None, False, out, splitk=sk, accumulate=True)


class HyperNetThetaManyFn(Function):
    """Same function as functional.HyperNetThetaFn (hypernet_attention.py:111-118), for G > 8 style vectors.

    The weight-streaming kernels read W once per <= 8 (forward) / 4 (backward) groups -- 13 / 25 passes over the 0.58 GB of
    head weights at G = 100.  Here every layer is one GEMM with M = G: theta_i = a_i W_i2^T on the tcgen05 kernel (the head
    weights are split to bf16 hi/lo once per call and that split is reused by the backward, read in place as the MN-major
    operand of da_i = dtheta_i W_i2), dW_i2 = dtheta_i^T a_i as a rank-G tensor-core product.
    params = [base0.W, base0.b, base2.W, base2.b, (head_i.0.W, head_i.0.b, head_i.2.W, head_i.2.b) * n_heads]."""

    @staticmethod
    def forward(ctx, x, *params):
        nh = (len(params) - 4) // 4
        act = lambda y: ops.leaky_relu_(y)
        b0 = act(_small_linear(x.contiguous(), params[0].contiguous(), params[1]))
        b1 = act(_small_linear(b0, params[2].contiguous(), params[3]))
        sizes = [params[4 + 4 * i + 2].shape[0] for i in range(nh)]
        G = x.shape[0]
        theta = torch.empty(G, sum(sizes), device=x.device, dtype=torch.float32)
        mids, splits, off = [], [], 0
        for i in range(nh):
            W1, c1, W2, c2 = params[4 + 4 * i: 8 + 4 * i]
            a = act(_small_linear(b1, W1.contiguous(), c1))
            W2c = W2.contiguous()
            if ops._tc_ok(128, W2c.shape[0], W2c.shape[1]):
                # M = G rows (one partial 128-row tile: TMA zero-fills the missing rows, the epilogue writes only G)
                sW = ops.split_bf16(W2c)
                ops.gemm_tc(ops.split_bf16(a), sW, bias=c2, out=theta[:, off:off + sizes[i]], splitk=1)
                splits.append((sW.hi, sW.lo))
            else:
                _small_linear(a, W2c, c2, out=theta[:, off:off + sizes[i]])
                splits.append((None, None))
            mids.append(a)
            off += sizes[i]
        flat_splits = [t for pair in splits for t in pair]
        ctx.save_for_backward(x, b0, b1, *mids, *params, *flat_splits)
        ctx.nh, ctx.sizes, ctx.np = nh, sizes, len(params)
        return theta

    @staticmethod
    def backward(ctx, dtheta):
        nh, sizes = ctx.nh, ctx.sizes
        sv = ctx.saved_tensors
        x, b0, b1 = sv[0], sv[1], sv[2]
        mids = sv[3:3 + nh]
        params = sv[3 + nh:3 + nh + ctx.np]
        splits = sv[3 + nh + ctx.np:]
        need = ctx.needs_input_grad
        dtheta = dtheta.contiguous()
        G = x.shape[0]
        grads = [None] * len(params)
        db1 = torch.zeros_like(b1)
        off = 0

        def layer_bwd(dy, inp, W, leaky_out):
            """dy [G, N] (already multiplied by the activation derivative) -> dW, db, dinp (small layers: exact-fp32 SIMT
            products, K split over several CTAs)."""
            dy = dy.contiguous()
            Wc = W.contiguous()
            N, K = Wc.shape
            dW = ops._gemm(dy, dy.stride(0), 0, inp, inp.stride(0), 0, N, K, G, splitk=1)                 # dy^T inp
            dinp = ops._gemm(dy, dy.stride(0), 1, Wc, Wc.stride(0), 0, G, K, N, splitk=_sk(G, K, N))      # dy W
            return dW, ops.colsum(dy), dinp

        for i in range(nh):
            W1, c1, W2, c2 = params[4 + 4 * i: 8 + 4 * i]
            pi = 4 + 4 * i
            dth = dtheta[:, off:off + sizes[i]]
            a = mids[i]
            s_hi, s_lo = splits[2 * i], splits[2 * i + 1]
            N, K = W2.shape
            if s_hi is not None and (s_lo is not None) == ops.TC_SPLIT:
                # rank-G weight gradient and the input gradient on the tensor cores; W2's forward split read MN-major
                dsp = ops.split_bf16(dth)                                   # one split of dtheta_i serves both products
                dW2 = ops.gemm_tc(ops.SplitOperand(dsp.hi, dsp.lo, N, G, dsp.ld, True), ops.split_bf16(a, mn=True))   # [N, K], K-dim = G
                W2t = ops.SplitOperand(s_hi, s_lo, K, N, s_hi.shape[1], True)
                da = ops.gemm_tc(dsp, W2t)                                                           # [G, K], K-dim = N
                dc2 = ops.colsum(dth)
            else:
                dW2, dc2, da = layer_bwd(dth, a, W2, False)
            ops.leaky_relu_bwd_(a, da)
            dW1, dc1, db1_i = layer_bwd(da, b1, W1, True)
            db1 += db1_i
            grads[pi], grads[pi + 1], grads[pi + 2], grads[pi + 3] = dW1, dc1, dW2, dc2
            off += sizes[i]
        ops.leaky_relu_bwd_(b1, db1)
        dWb1, dcb1, db0 = layer_bwd(db1, b0, params[2], True)
        ops.leaky_relu_bwd_(b0, db0)
        dWb0, dcb0, dx = layer_bwd(db0, x.contiguous(), params[0], True)
        grads[0], grads[1], grads[2], grads[3] = dWb0, dcb0, dWb1, dcb1
        grads = [g if need[1 + j] else None for j, g in enumerate(grads)]
        from . import parallel
        parallel.join()
        return (dx if need[0] else None, *grads)
