"""Float64 reference of the attention-GRU recurrence kernels (csrc/attgru_step.cu, attgru_step_bwd.cu, attgru_seq.cu):
seeded inputs and every tensor the kernels write, computed on the CPU with autograd.

One step, as the kernels compute it (the keys K = W_a f + b_a and the word half GIw = x_word W_ih[:, :E]^T + b_ih are
hoisted out of the time loop by the caller):

    u = U_a h + b_u;   s_p = v_a . tanh(K_p + u) + b_v;   alpha = softmax_p(s);   ctx = sum_p alpha_p f_p
    h' = GRUCell([GIw_t | ctx], h)   with the input weights [I_3H | W_ih[:, E:]] and no input bias

The attention step is the oracle's Bahdanau attention (oracle/caption_hn_oracle.py bahdanau) with K given; the GRU half
is recurrence_ref._gru_cell, which checks every correct step against the oracle cell.  Rows are independent given the
weights, so the reference runs on row chunks (large batches fit in host memory) and sums the shared-weight gradients.

``mutant`` plants one defect in the reference; the mutation test uses it to show that the tolerances would catch it."""
import torch
import torch.nn.functional as F

import recurrence_ref as R

ATT_MUTANTS = ("f of the next batch row", "last position dropped from the softmax", "u without b_u", "tanh(K) + u",
               "attention reads the new state", "dattn ignored")
GRU_MUTANTS = tuple(m for m in R.GRU_MUTANTS if m != "extra layer fed the step input")   # one layer here
MUTANTS = ATT_MUTANTS + GRU_MUTANTS
E_COLS = 5      # width of the word half of W_ih: arbitrary, the recurrence never reads those columns
CHUNK_ELEMS = 1 << 24


def inputs(B, T, P, H, F, seed, dattn=False):
    """float32 inputs of one case in the kernels' layouts.  Scaled as the step-split tests scale them (K, f, GIw * 0.5,
    W / sqrt(fan-in), biases * 0.1, h0 * 0.5), except v_a: its norm is fixed at 4 so the scores spread over a few units
    and the attention is far from uniform (the median over rows of max alpha / min alpha is about 20 at P = 4 and in
    the hundreds at P = 49), so a mixed-up position or row shows."""
    g = torch.Generator().manual_seed(seed)
    H3 = 3 * H
    va = torch.randn(H, generator=g)
    d = {"K": torch.randn(B, P, H, generator=g) * 0.5,
         "f": torch.randn(B, P, F, generator=g) * 0.5,
         "GIw": torch.randn(T, B, H3, generator=g) * 0.5,
         "W_ih": torch.randn(H3, E_COLS + F, generator=g) / (E_COLS + F) ** 0.5,
         "W_hh": torch.randn(H3, H, generator=g) / H ** 0.5,
         "b_hh": torch.randn(H3, generator=g) * 0.1,
         "U_a": torch.randn(H, H, generator=g) / H ** 0.5,
         "b_u": torch.randn(H, generator=g) * 0.1,
         "v_a": va * (4.0 / va.norm()),
         "b_v": torch.randn(1, generator=g),
         "h0": torch.randn(B, H, generator=g) * 0.5,
         "dHbm": torch.randn(B, T, H, generator=g) * 0.3}
    d["W_ihc"] = d["W_ih"][:, E_COLS:]
    if dattn:
        d["dattn"] = torch.randn(B, T, P, generator=g) * 0.2
    return d


def attention_step(K, f, h, U_a, b_u, v_a, b_v, mutant=None, h_stale=None):
    """One Bahdanau step on precomputed keys: (ctx [B,F], alpha [B,P], u [B,H], s [B,P]).  ``h_stale`` is what the
    mutant "attention reads the new state" reads: the step-split kernels ping-pong h between two buffers, and the one the
    step writes its new state into still holds the state of the step before (h0 at t = 0)."""
    u = F.linear(h_stale if mutant == "attention reads the new state" else h, U_a,
                 None if mutant == "u without b_u" else b_u)
    if mutant == "tanh(K) + u":
        q = torch.tanh(K) + u[:, None, :]
    else:
        q = torch.tanh(K + u[:, None, :])
    s = q @ v_a + b_v
    if mutant == "last position dropped from the softmax":
        alpha = torch.cat([F.softmax(s[:, :-1], dim=1), torch.zeros_like(s[:, -1:])], 1)
    else:
        alpha = F.softmax(s, dim=1)
    fr = torch.roll(f, -1, 0) if mutant == "f of the next batch row" else f
    ctx = (alpha[:, :, None] * fr).sum(1)
    return ctx, alpha, u, s


def _leaf(t):
    return t.double().requires_grad_(True)


def _chunk(d, T, r0, r1, mutant, grad):
    """Forward (+ BPTT when ``grad``) of rows [r0, r1)."""
    rows = slice(r0, r1)
    K, f, h0 = _leaf(d["K"][rows]), _leaf(d["f"][rows]), _leaf(d["h0"][rows])
    GIw = d["GIw"][:, rows].double()
    W_ihc, W_hh, b_hh = _leaf(d["W_ihc"]), _leaf(d["W_hh"]), _leaf(d["b_hh"])
    U_a, b_u, v_a, b_v = _leaf(d["U_a"]), _leaf(d["b_u"]), _leaf(d["v_a"]), _leaf(d["b_v"])
    H3 = W_hh.shape[0]
    W_ih = torch.cat([torch.eye(H3, dtype=torch.float64), W_ihc], 1)
    zero = torch.zeros(H3, dtype=torch.float64)
    h, hs, out = h0, [h0], {k: [] for k in ("attn", "ctx", "u", "s", "gi", "gh", "sv")}
    for t in range(T):
        ctx, alpha, u, s = attention_step(K, f, h, U_a, b_u, v_a, b_v, mutant, hs[max(t - 1, 0)])
        u.retain_grad(); s.retain_grad(); ctx.retain_grad()
        h, sv, gi, gh = R._gru_cell(torch.cat([GIw[t], ctx], 1), h, W_ih, W_hh, zero, b_hh, mutant, t == 0)
        hs.append(h)
        for k, v in zip(("attn", "ctx", "u", "s", "gi", "gh", "sv"), (alpha, ctx, u, s, gi, gh, sv)):
            out[k].append(v)
    attn = torch.stack(out["attn"], 1)                                      # [b,T,P]
    Hs = torch.stack(hs[1:], 1)                                             # [b,T,H]
    r = {"Hall": torch.stack(hs, 0).detach(), "attn": attn.detach(), "ctx": torch.stack(out["ctx"], 0).detach(),
         "saved": torch.stack([torch.stack(out["u"], 0)] +
                              [torch.stack([sv[q] for sv in out["sv"]], 0) for q in range(4)], 0).detach()}
    if not grad:
        return r
    loss = (Hs * d["dHbm"][rows].double()).sum()
    if "dattn" in d and mutant != "dattn ignored":
        loss = loss + (attn * d["dattn"][rows].double()).sum()
    loss.backward()
    st = lambda k: torch.stack([v.grad for v in out[k]], 0)                 # [T,b,...]
    gr = lambda p: p.grad if p.grad is not None else torch.zeros_like(p)   # a mutant may not use the parameter
    r.update(dGI=st("gi"), dGH=st("gh"), dU=st("u"), dCTX=st("ctx"), dK=gr(K), dh0=gr(h0), df_att=gr(f),
             dva=gr(v_a), dbv=gr(b_v), dbv_scale=st("s").abs().sum().reshape(1), dW_ihc=gr(W_ihc),
             dW_hh=gr(W_hh), dU_a=gr(U_a), db_u=gr(b_u), db_hh=gr(b_hh))
    return r


ROW_KEYS = {"Hall": 1, "attn": 0, "ctx": 1, "saved": 2, "dGI": 1, "dGH": 1, "dU": 1, "dCTX": 1, "dK": 0, "dh0": 0,
            "df_att": 0}


def attention_gru(d, mutant=None, grad=True):
    """Forward + BPTT in float64; loss = sum(Hbm * dHbm) (+ sum(attn * dattn) when ``d`` has dattn).  Returns the kernels'
    outputs in their layouts -- Hall [T+1,B,H], attn [B,T,P], ctx [T,B,F], saved [5,T,B,H] = (u, r, z, n, gh_n); dGI,
    dGH [T*B,3H], dU [T*B,H], dCTX [T*B,F], dK [B,P,H], dva [H], dbv [1], dh0 [B,H] -- and the products their callers
    form: dW_ihc = dGI^T ctx, dW_hh = dGH^T Hprev, dU_a = dU^T Hprev, db_u, db_hh, df_att = sum_t alpha_t dctx_t.
    dbv_scale = sum |ds| (dbv is analytically zero: the softmax is shift invariant)."""
    T, B, _ = d["GIw"].shape
    P, H = d["K"].shape[1:]
    step = max(1, CHUNK_ELEMS // (P * max(H, d["f"].shape[2]) * T))
    parts = [_chunk(d, T, r0, min(B, r0 + step), mutant, grad) for r0 in range(0, B, step)]
    r = {}
    for k in parts[0]:
        if k in ROW_KEYS:
            r[k] = torch.cat([p[k] for p in parts], ROW_KEYS[k])
        else:
            r[k] = sum(p[k] for p in parts)
    for k in ("dGI", "dGH", "dU", "dCTX"):
        if k in r:
            r[k] = r[k].reshape(T * B, -1)
    return r
