"""Many-style batches on the pooled captioners: the grouped LSTM recurrence kernels, ``forward(groups=)`` of the LSTM
captioner and ``forward_loss(groups=)`` of both captioners.

Kernels: the grouped LSTM forward / BPTT run every row with the same arithmetic as the single-style kernels, so each
group's rows must come out bit for bit equal to ``lstm_seq_fwd`` / ``lstm_seq_bwd`` run on that group alone, and within
the float32 bounds of tests/test_gpu_recurrence_ref.py of the float64 LSTM (tests/recurrence_ref.py).  Modules: against
the oracle run once per group (train_cc.py:90-123 semantics), logits and loss within 1e-4 and every gradient within 1e-3.
The argument checks at the end need no GPU."""
import pytest
import torch
import torch.nn.functional as F

import recurrence_ref as R
from golden_util import rel_err, grad_close
from oracle import caption_hn_oracle as O

gpu = pytest.mark.gpu

FWD, BWD = 5e-6, 2e-5          # float32 bounds of the recurrence against float64 at T <= 5
TOL_LOGITS, TOL_GRAD = 1e-4, 1e-3
# rows per group: empty groups, 1-row tiles, a full 4-row tile, 4 + 1, and 37 = nine full tiles + a 1-row tail
SIZES = {3: (5, 0, 37), 11: (5, 0, 1, 37, 4, 2, 0, 3, 7, 1, 6)}


def _shuffled_groups(sizes, gen):
    groups = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    return groups[torch.randperm(groups.numel(), generator=gen)]


def _lstm_kernel_case(G, H, T=4):
    """Grouped kernels on a batch of groups of SIZES[G] rows (sorted by GroupPlan), and the single-style kernels on each
    group alone.  Returns (per-group float64 inputs, plan, grouped outputs, per-group single-style outputs)."""
    from hypernet_image_captioning_b200 import ops
    from hypernet_image_captioning_b200.grouped import GroupPlan
    sizes = SIZES[G]
    B, H4 = sum(sizes), 4 * H
    assert B % 4
    gen = torch.Generator().manual_seed(100 * G + H)
    plan = GroupPlan.get(_shuffled_groups(sizes, gen), G, T, torch.device("cuda"))
    d = [R.inputs(n, T, H, 1, 4, seed=10_000 * G + 10 * H + g) for g, n in enumerate(sizes)]
    Theta = torch.stack([torch.cat([dg["W_hh"].reshape(-1), dg["b_hh"]]) for dg in d]).cuda()    # [G, 4H*H + 4H]
    GI = torch.cat([dg["GI"] for dg in d], 1).reshape(T * B, H4).cuda()                        # time-major, sorted
    h0 = torch.cat([dg["h0"] for dg in d], 0).cuda()
    dH = torch.cat([dg["dH"] for dg in d], 0).cuda()
    ld4, ldh = ops.round4(H4), ops.round4(H)
    WhhT = ops.transpose_pad_batched(Theta[:, :H4 * H], H4, H, ld4)
    Whh_p = ops.copy_pad_batched(Theta[:, :H4 * H], H4, H, ldh)
    Hall, Hbm, saved, cT = ops.lstm_seq_fwd_grouped(GI, WhhT, Theta[:, H4 * H:], h0, T, plan.tiles4, want_c=True)
    dG, dh0 = ops.lstm_seq_bwd_grouped(dH, saved, Hall, Whh_p, plan.tiles4)
    got = {"Hall": Hall, "Hbm": Hbm, "saved": saved, "cT": cT, "dG": dG.view(T, B, H4), "dh0": dh0}
    single = {}
    for g, (n, dg) in enumerate(zip(sizes, d)):
        W = dg["W_hh"].cuda()
        assert torch.equal(WhhT[g], ops.transpose_pad(W, ld4)) and torch.equal(Whh_p[g], ops.copy_pad(W, ldh))
        if n == 0:
            continue
        Hs, Hbms, svs, _, cTs = ops.lstm_seq_fwd(dg["GI"].reshape(T * n, H4).cuda(), ops.transpose_pad(W, ld4),
                                                 dg["b_hh"].cuda(), dg["h0"].cuda(), T, want_c=True)
        dGs, dh0s = ops.lstm_seq_bwd(dg["dH"].cuda(), svs, Hs, ops.copy_pad(W, ldh))
        single[g] = {"Hall": Hs, "Hbm": Hbms, "saved": svs[0], "cT": cTs, "dG": dGs[0].view(T, n, H4), "dh0": dh0s}
    torch.cuda.synchronize()
    return d, plan, got, single


def _rows(got, r):
    """The outputs of the grouped call restricted to the batch rows r (a slice of the sorted batch)."""
    return {"Hall": got["Hall"][:, r], "Hbm": got["Hbm"][r], "saved": got["saved"][:, :, r], "cT": got["cT"][r],
            "dG": got["dG"][:, r], "dh0": got["dh0"][r]}


@gpu
@pytest.mark.parametrize("G", sorted(SIZES))
@pytest.mark.parametrize("H", [150, 151, 200])
def test_grouped_lstm_kernels_match_single_style_per_group_bit_for_bit(G, H):
    _, plan, got, single = _lstm_kernel_case(G, H)
    tiles = plan.tiles4.cpu()
    assert int(tiles[:, 1].min()) == 1 and int(tiles[:, 1].max()) == 4
    for g, ref in single.items():
        mine = _rows(got, slice(int(plan.goff[g]), int(plan.goff[g + 1])))
        for k in ref:
            assert torch.equal(mine[k], ref[k]), (g, k, (mine[k] - ref[k]).abs().max().item())


@gpu
@pytest.mark.parametrize("G", sorted(SIZES))
@pytest.mark.parametrize("H", [150, 151, 200])
def test_grouped_lstm_kernels_match_float64_lstm_per_group(G, H):
    d, plan, got, _ = _lstm_kernel_case(G, H)
    gates = ("i", "f", "g", "o", "c_prev", "tanh_c")
    for g, dg in enumerate(d):
        if dg["h0"].shape[0] == 0:
            continue
        ref = R.lstm(dg)
        mine = _rows(got, slice(int(plan.goff[g]), int(plan.goff[g + 1])))
        T, n = dg["GI"].shape[:2]
        errs = {"Hall": (rel_err(mine["Hall"][1:], ref["Hall"][1:]), FWD), "cT": (rel_err(mine["cT"], ref["cT"]), FWD),
                "dG": (rel_err(mine["dG"].reshape(T * n, -1), ref["dG"][0]), BWD),
                "dh0": (rel_err(mine["dh0"], ref["dh0"]), BWD)}
        for q, name in enumerate(gates):
            errs["saved." + name] = (rel_err(mine["saved"][q], ref["saved"][0, q]), FWD)
        bad = {k: e for k, (e, b) in errs.items() if not e < b}
        assert not bad, f"G={G} H={H} group {g} ({n} rows): {bad}"


# ----------------------------------------------------------------------------------------------------------------------
# captioners: forward(groups=) / forward_loss(groups=) against the oracle run per group
# ----------------------------------------------------------------------------------------------------------------------
def _oracle(pl, styles, pooled, caps, h0, groups, cell, theta=None):
    """Logits of one oracle call per group, back in batch order.  ``theta`` [G, θ] given: the per-group decoder calls run
    on its rows instead of a hypernet call per group (see the full-size test)."""
    E, H = pl["captioner.embed.weight"].shape[1], pl["captioner.fc_out.weight"].shape[1]
    outs, idxs = [], []
    for g in range(styles.shape[0]):
        idx = (groups == g).nonzero().squeeze(1)
        if idx.numel() == 0:
            continue
        if theta is None:
            lg, _, _ = O.path_pooled(pl, styles[g:g + 1], pooled[idx], caps[idx], h0[idx], cell=cell)
        else:
            cells = O.split_theta_pooled(theta[g], E, H, 1, 4 if cell == "lstm" else 3)
            feats = F.linear(pooled[idx], pl["image_encoder.fc.weight"], pl["image_encoder.fc.bias"])
            lg = (O.decoder_rnn_forward(pl, cells, feats, caps[idx]) if cell == "lstm"
                  else O.decoder_gru_forward(pl, cells, feats, caps[idx], h0[idx]))
        outs.append(lg)
        idxs.append(idx)
    return torch.cat(outs, 0)[torch.argsort(torch.cat(idxs))]


def _model(p, E, H, V, cell):
    import hypernet_image_captioning_b200 as C
    with torch.device("cuda"):
        m = C.HyperNetPooled(E, H, V, None, num_layers=1, type=cell)
    sd = m.state_dict()
    sd.update(p)
    m.load_state_dict(sd)
    return m


def _run(m, styles, pooled, caps, h0, groups, ignore_index, fused):
    """One many-style training step through the public API; returns (loss, logits)."""
    import hypernet_image_captioning_b200 as C
    cap = m.forward_grouped(styles.cuda())
    feats = m.image_encoder(pooled.cuda())
    assert cap._grouped_kernels_ok(feats)
    h0 = None if h0 is None else h0.cuda()
    if fused:
        loss, logits = cap.forward_loss(feats, caps.cuda(), h0=h0, ignore_index=ignore_index, groups=groups)
    else:
        logits = cap(feats, caps.cuda(), True, h0=h0, groups=groups)
        loss = C.cross_entropy(logits, caps.cuda(), ignore_index)
    loss.backward()
    return loss, logits


def _check_against_oracle(m, ref_grads, loss, logits, logits_ref, loss_ref, where):
    assert rel_err(logits, logits_ref.detach()) < TOL_LOGITS, where
    assert abs(loss.item() - loss_ref.item()) <= TOL_LOGITS * abs(loss_ref.item()), where
    worst, checked = 0.0, 0
    for k, v in m.named_parameters():
        if k.startswith("captioner.lstm_cell."):        # generated weights: the gradient flows into the hypernet
            continue
        assert v.grad is not None, (where, k)
        ref = ref_grads[k].cuda()
        d, s = (v.grad - ref).abs().max().item(), ref.abs().max().item()
        assert d <= 1e-7 or d <= TOL_GRAD * s, (where, k, d, s)
        worst = max(worst, d / s if s > 0 else 0.0)
        checked += 1
        del ref
    assert checked == 25      # hypernet base (4) and heads (16), embed, image_encoder.fc (2), fc_out (2)
    print(f"[{where}] logits {rel_err(logits, logits_ref.detach()):.2e} worst grad {worst:.2e}")


SMALL = dict(E=16, H=12, V=97, T=5)
SMALL_SIZES = (5, 0, 1, 15)          # an empty group (zero d(theta) row) and a 1-row group; B = 21


@gpu
@pytest.mark.parametrize("ignore_index", [None, 0])
@pytest.mark.parametrize("cell,fused", [("lstm", False), ("lstm", True), ("gru", True)])
def test_pooled_grouped_matches_per_group_oracle(cell, fused, ignore_index):
    E, H, V, T = SMALL["E"], SMALL["H"], SMALL["V"], SMALL["T"]
    G = len(SMALL_SIZES)
    p = O.init_params_pooled(2048, E, H, V, seed=4, gates=4 if cell == "lstm" else 3)
    gen = torch.Generator().manual_seed(9)
    groups = _shuffled_groups(SMALL_SIZES, gen)
    B = groups.numel()
    pooled = torch.relu(torch.randn(B, 2048, generator=gen))
    caps = O.synth_captions(B, T, V, gen)
    styles = torch.randn(G, E, generator=gen)
    h0 = torch.rand(B, H, generator=gen)
    pl = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    logits_ref = _oracle(pl, styles, pooled, caps, h0, groups, cell)
    loss_ref = O.caption_loss(logits_ref, caps, ignore_index)
    loss_ref.backward()
    m = _model(p, E, H, V, cell)
    loss, logits = _run(m, styles, pooled, caps, h0 if cell == "gru" else None, groups, ignore_index, fused)
    _check_against_oracle(m, {k: v.grad for k, v in pl.items()}, loss, logits, logits_ref, loss_ref,
                          f"{cell} fused={fused} ignore={ignore_index}")


@gpu
@pytest.mark.parametrize("ignore_index", [None, 0])
def test_gru_grouped_forward_loss_matches_forward_plus_cross_entropy(ignore_index):
    E, H, V, T = 48, 56, 500, 6
    p = O.init_params_pooled(2048, E, H, V, seed=2)
    gen = torch.Generator().manual_seed(8)
    groups = _shuffled_groups((9, 0, 1, 24, 16), gen)
    B = groups.numel()
    pooled = torch.relu(torch.randn(B, 2048, generator=gen))
    caps = O.synth_captions(B, T, V, gen)
    styles = torch.randn(5, E, generator=gen)
    h0 = torch.rand(B, H, generator=gen)
    res = []
    for fused in (False, True):
        m = _model(p, E, H, V, "gru")
        loss, logits = _run(m, styles, pooled, caps, h0, groups, ignore_index, fused)
        res.append((loss.item(), logits.detach(), {k: v.grad.clone() for k, v in m.named_parameters() if v.grad is not None}))
    assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[0][0])
    assert torch.equal(res[0][1], res[1][1])
    assert res[0][2].keys() == res[1][2].keys()
    for k, v in res[0][2].items():
        assert grad_close(res[1][2][k], v, 1e-3), k


@gpu
@pytest.mark.parametrize("cell", ["gru", "lstm"])
def test_pooled_grouped_forward_loss_full_size_100_groups(cell):
    """BASELINE configs[1] shapes (B=512, T=20, E=200, H=150, V=9684) with G = 100 domains of random sizes: one-hot domain
    vectors as a dense [G, E] input (the hypernet's dense tensor-core layers), the fused many-style loss with the padding
    index, against one oracle decoder call per group.

    The oracle's hypernet runs once for all G rows (rows are independent) and in float64 on the GPU: in float32 on the CPU
    its backward is the least accurate party here -- d(hidden) = dθ · W2 sums 120 000 terms of the 7.2 GB LSTM W_ih head,
    and its hn_base / first head layer gradients land 1-3e-2 (of max|grad|) away from a float64 backward of the same dθ,
    where the kernels, like the per-group loop, stay within 1e-4."""
    E, H, V, T, B, G = 200, 150, 9684, 20, 512, 100
    p = O.init_params_pooled(2048, E, H, V, L=1, seed=5, gates=4 if cell == "lstm" else 3)
    gen = torch.Generator().manual_seed(100)
    pooled = torch.relu(torch.randn(B, 2048, generator=gen))
    caps = O.synth_captions(B, T, V, gen)
    styles = torch.zeros(G, E)
    styles[torch.arange(G), torch.arange(G)] = 1.0
    h0 = torch.rand(B, H, generator=gen)
    groups = torch.randint(0, G, (B,), generator=gen)
    m = _model(p, E, H, V, cell)
    pl = {k: v.requires_grad_(True) for k, v in p.items() if not k.startswith("hn_")}
    hp = {k: v.double().cuda().requires_grad_(True) for k, v in p.items() if k.startswith("hn_")}
    theta64 = O.hypernet_theta(hp, styles.double().cuda(), 4)
    theta = theta64.detach().float().cpu().requires_grad_(True)
    logits_ref = _oracle(pl, styles, pooled, caps, h0, groups, cell, theta=theta)
    loss_ref = O.caption_loss(logits_ref, caps, 0)
    loss_ref.backward()
    theta64.backward(theta.grad.double().cuda())
    ref_grads = {**{k: v.grad for k, v in pl.items()}, **{k: v.grad for k, v in hp.items()}}
    del theta64
    loss, logits = _run(m, styles, pooled, caps, h0 if cell == "gru" else None, groups, 0, True)
    _check_against_oracle(m, ref_grads, loss, logits, logits_ref, loss_ref, f"{cell} full size G={G}")


# ----------------------------------------------------------------------------------------------------------------------
# argument checks (CPU: they fire before any kernel runs)
# ----------------------------------------------------------------------------------------------------------------------
def _cpu_batch(E, H, V, cell, num_layers=1):
    import hypernet_image_captioning_b200 as C
    m = C.HyperNetPooled(E, H, V, None, num_layers=num_layers, type=cell)
    gen = torch.Generator().manual_seed(0)
    return m, torch.randn(6, E, generator=gen), O.synth_captions(6, 4, V, gen)


@pytest.mark.parametrize("cell", ["gru", "lstm"])
def test_grouped_forward_loss_needs_forward_grouped(cell):
    m, feats, caps = _cpu_batch(8, 6, 30, cell)
    with pytest.raises(ValueError, match="forward_grouped"):
        m.captioner.forward_loss(feats, caps, groups=torch.zeros(6, dtype=torch.long))


@pytest.mark.parametrize("cell", ["gru", "lstm"])
def test_grouped_forward_loss_refuses_extra_layers(cell):
    m, feats, caps = _cpu_batch(8, 6, 30, cell, num_layers=2)
    with pytest.raises(NotImplementedError, match="forward\\(\\.\\.\\., groups=\\.\\.\\.\\) \\+ cross_entropy"):
        m.captioner.forward_loss(feats, caps, groups=torch.zeros(6, dtype=torch.long))


@pytest.mark.parametrize("cell", ["gru", "lstm"])
def test_grouped_forward_loss_refuses_out_of_range_group_ids(cell, monkeypatch):
    m, feats, caps = _cpu_batch(8, 6, 30, cell)
    n = sum(p.numel() for p in m.captioner.lstm_cell.parameters())
    monkeypatch.setattr(m, "generate_theta", lambda x: torch.zeros(x.shape[0], n))   # the hypernet itself needs CUDA
    cap = m.forward_grouped(torch.zeros(3, 8))
    with pytest.raises(ValueError, match="group ids"):
        cap.forward_loss(feats, caps, groups=torch.tensor([0, 1, 2, 3, 0, 1]))
    with pytest.raises(NotImplementedError, match="CUDA tensors"):         # valid ids, but CPU tensors
        cap.forward_loss(feats, caps, groups=torch.tensor([0, 1, 2, 2, 0, 1]))
