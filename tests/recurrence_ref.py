"""Float64 references of the GRU / LSTM recurrence kernels (csrc/gru_resident.cu, gru_cluster.cu, gru_seq.cu,
lstm_seq.cu): seeded inputs and every tensor the kernels write, computed on the CPU with autograd.

The cells are the oracle's (oracle/caption_hn_oracle.py gru_cell / lstm_cell), restated so that the gates the kernels
save and the pre-activation gradients they return can be read off; every correct step is checked against the oracle
cell.  Layer 0 receives the kernels' input projection GI through an identity W_ih.  Extra layers are chained as the
oracle chains them: h = layer(h, h) for the GRU (decoder_gru_forward), (h, c) = layer(h, (h, c)) for the LSTM
(decoder_rnn_forward).

``mutant`` plants one defect in the reference; the mutation test uses it to show that the tolerances would catch it."""
import torch
import torch.nn.functional as F

from oracle import caption_hn_oracle as O

GRU_MUTANTS = ("b_hn outside r", "z and 1-z swapped", "r and z blocks swapped", "dh0 without direct term",
               "extra layer fed the step input")
LSTM_MUTANTS = ("i and f swapped", "extra layer fed the step input")


def inputs(B, T, H, NL, gates, seed, c0=False):
    """float32 inputs of one case, scaled so the gates stay unsaturated: GI * 0.5, W / sqrt(H), h0 ~ U(0, 1).  ``gates`` is
    3 (GRU) or 4 (LSTM).  Extra layers carry (W_ih, W_hh, b_ih, b_hh)."""
    g = torch.Generator().manual_seed(seed)
    G = gates * H
    d = {"GI": torch.randn(T, B, G, generator=g) * 0.5,
         "W_hh": torch.randn(G, H, generator=g) / H ** 0.5,
         "b_hh": torch.randn(G, generator=g) * 0.1,
         "h0": torch.rand(B, H, generator=g),
         "extra": [(torch.randn(G, H, generator=g) / H ** 0.5, torch.randn(G, H, generator=g) / H ** 0.5,
                    torch.randn(G, generator=g) * 0.1, torch.randn(G, generator=g) * 0.1) for _ in range(NL - 1)],
         "dH": torch.randn(B, T, H, generator=g)}
    if c0:
        d["c0"] = torch.randn(B, H, generator=g) * 0.5
    return d


def _leaf(t):
    return t.double().requires_grad_(True)


def _gru_cell(x, h, W_ih, W_hh, b_ih, b_hh, mutant, first):
    gi = F.linear(x, W_ih, b_ih)
    gh = F.linear(h, W_hh, b_hh)
    gi.retain_grad()
    gh.retain_grad()
    i_r, i_z, i_n = gi.chunk(3, dim=1)
    h_r, h_z, h_n = gh.chunk(3, dim=1)
    if mutant == "r and z blocks swapped":
        i_r, i_z, h_r, h_z = i_z, i_r, h_z, h_r
    r = torch.sigmoid(i_r + h_r)
    z = torch.sigmoid(i_z + h_z)
    if mutant == "b_hn outside r":
        H = h.shape[1]
        n = torch.tanh(i_n + r * (h_n - b_hh[2 * H:]) + b_hh[2 * H:])
    else:
        n = torch.tanh(i_n + r * h_n)
    hd = h.detach() if (mutant == "dh0 without direct term" and first) else h
    hn = z * n + (1.0 - z) * hd if mutant == "z and 1-z swapped" else (1.0 - z) * n + z * hd
    if mutant is None:
        want = O.gru_cell(x, h, W_ih, W_hh, b_ih, b_hh)
        assert (hn - want).abs().max().item() <= 1e-14, "restated GRU cell differs from the oracle cell"
    return hn, (r, z, n, h_n), gi, gh


def gru(d, mutant=None):
    """Forward + BPTT of the multi-layer GRU on the float64 copies of ``d``; loss = sum(H_bm * dH).  Returns a dict of
    the kernels' outputs: Hall [T+1,B,H], saved [NL,4,T,B,H], Hmid [NL-1,T,B,H], dGI / dGH [T*B,3H] (layer 0),
    xdGI / xdGH [NL-1,T*B,3H], dh0, and the parameter gradients (dW_hh, db_hh, x<l>.dW_ih ...) they must reproduce."""
    T, B, H3 = d["GI"].shape
    H = H3 // 3
    GI, W_hh, b_hh, h0 = _leaf(d["GI"]), _leaf(d["W_hh"]), _leaf(d["b_hh"]), _leaf(d["h0"])
    extra = [tuple(_leaf(t) for t in cell) for cell in d["extra"]]
    NL = 1 + len(extra)
    eye, zero = torch.eye(H3, dtype=torch.float64), torch.zeros(H3, dtype=torch.float64)
    h = h0
    outs, mids = [], [[] for _ in extra]
    saved = [[] for _ in range(NL)]
    gis, ghs = [[] for _ in range(NL)], [[] for _ in range(NL)]
    for t in range(T):
        h_in = h
        h, sv, gi, gh = _gru_cell(GI[t], h, eye, W_hh, zero, b_hh, mutant, t == 0)
        saved[0].append(sv); gis[0].append(gi); ghs[0].append(gh)
        for l, cell in enumerate(extra):
            mids[l].append(h)
            x = h_in if mutant == "extra layer fed the step input" else h
            h, sv, gi, gh = _gru_cell(x, h, *cell, mutant, False)
            saved[l + 1].append(sv); gis[l + 1].append(gi); ghs[l + 1].append(gh)
        outs.append(h)
    Hs = torch.stack(outs, 0)
    (Hs.permute(1, 0, 2) * d["dH"].double()).sum().backward()
    r = {"Hall": torch.cat([h0.detach()[None], Hs.detach()], 0),
         "saved": torch.stack([torch.stack([torch.stack([s[q] for s in saved[l]], 0) for q in range(4)], 0)
                               for l in range(NL)], 0).detach(),
         "dh0": h0.grad, "dW_hh": W_hh.grad, "db_hh": b_hh.grad}
    grads = [(torch.stack([g.grad for g in gis[l]], 0).reshape(T * B, H3),
              torch.stack([g.grad for g in ghs[l]], 0).reshape(T * B, H3)) for l in range(NL)]
    r["dGI"], r["dGH"] = grads[0]
    assert (r["dGI"].view(T, B, H3) - GI.grad).abs().max().item() <= 1e-14
    if NL > 1:
        r["Hmid"] = torch.stack([torch.stack(m, 0) for m in mids], 0).detach()
        r["xdGI"] = torch.stack([g[0] for g in grads[1:]], 0)
        r["xdGH"] = torch.stack([g[1] for g in grads[1:]], 0)
        for l, cell in enumerate(extra):
            for name, p in zip(("dW_ih", "dW_hh", "db_ih", "db_hh"), cell):
                r[f"x{l + 1}.{name}"] = p.grad
    return r


def _lstm_cell(x, h, c, W_ih, W_hh, b_ih, b_hh, mutant):
    g = F.linear(x, W_ih, b_ih) + F.linear(h, W_hh, b_hh)
    g.retain_grad()
    i, f, gg, o = g.chunk(4, dim=1)
    if mutant == "i and f swapped":
        i, f = f, i
    ig, fg, gt, og = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(gg), torch.sigmoid(o)
    c2 = fg * c + ig * gt
    tc = torch.tanh(c2)
    h2 = og * tc
    if mutant is None:
        wh, wc = O.lstm_cell(x, h, c, W_ih, W_hh, b_ih, b_hh)
        assert max((h2 - wh).abs().max().item(), (c2 - wc).abs().max().item()) <= 1e-14, \
            "restated LSTM cell differs from the oracle cell"
    return h2, c2, (ig, fg, gt, og, c, tc), g


def lstm(d, mutant=None):
    """LSTM counterpart of gru(): Hall, saved [NL,6,T,B,H] = (i, f, g, o, c_prev, tanh c), Hmid, cT, dG [NL,T*B,4H], dh0.
    The cell state starts at d["c0"] when present, else at zero."""
    T, B, H4 = d["GI"].shape
    H = H4 // 4
    GI, W_hh, b_hh, h0 = _leaf(d["GI"]), _leaf(d["W_hh"]), _leaf(d["b_hh"]), _leaf(d["h0"])
    extra = [tuple(_leaf(t) for t in cell) for cell in d["extra"]]
    NL = 1 + len(extra)
    eye, zero = torch.eye(H4, dtype=torch.float64), torch.zeros(H4, dtype=torch.float64)
    h = h0
    c = d["c0"].double() if "c0" in d else torch.zeros(B, H, dtype=torch.float64)
    outs, mids = [], [[] for _ in extra]
    saved, gs = [[] for _ in range(NL)], [[] for _ in range(NL)]
    for t in range(T):
        h_in = h
        h, c, sv, g = _lstm_cell(GI[t], h, c, eye, W_hh, zero, b_hh, mutant)
        saved[0].append(sv); gs[0].append(g)
        for l, cell in enumerate(extra):
            mids[l].append(h)
            x = h_in if mutant == "extra layer fed the step input" else h
            h, c, sv, g = _lstm_cell(x, h, c, *cell, mutant)
            saved[l + 1].append(sv); gs[l + 1].append(g)
        outs.append(h)
    Hs = torch.stack(outs, 0)
    (Hs.permute(1, 0, 2) * d["dH"].double()).sum().backward()
    r = {"Hall": torch.cat([h0.detach()[None], Hs.detach()], 0),
         "saved": torch.stack([torch.stack([torch.stack([s[q] for s in saved[l]], 0) for q in range(6)], 0)
                               for l in range(NL)], 0).detach(),
         "cT": c.detach(), "dh0": h0.grad,
         "dG": torch.stack([torch.stack([g.grad for g in gs[l]], 0).reshape(T * B, H4) for l in range(NL)], 0)}
    if NL > 1:
        r["Hmid"] = torch.stack([torch.stack(m, 0) for m in mids], 0).detach()
    return r
