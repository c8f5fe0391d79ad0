"""Batched beam search of the pooled GRU captioner (DecoderGRU.beam_search_batched) and the token-fed decode step it runs
on (ops.gru_decode_step_tok): the kernel bit for bit against gather + the GI-fed step, beam_size = 1 against greedy
``infer``, and the search against a CPU restatement of the reference's beam loop with the pooled decoder step."""
import pytest
import torch
import torch.nn.functional as F

from oracle import caption_hn_oracle as O


def pooled_beam_search(p, cells, feature, h0, beam_size=3, end_sentence=2, max_steps=50, pre="captioner."):
    """Beam search of hypernet_attention.py:247-326 for ONE image of the pooled captioner: ``O.attention_beam_search``'s
    loop with two changes only -- the decoder step is ``gru_cell`` with ``cells[0]`` (step 1 feeds ``feature`` [1, E] with
    ``h0`` [1, H], later steps ``F.embedding(prev, emb)``), and no embedding is zeroed.  Returns the best complete sequence
    (leading 0, trailing ``end_sentence``) or None when a beam is still open after ``max_steps`` + 1 steps."""
    emb_w = p[pre + "embed.weight"]
    V = p[pre + "fc_out.weight"].shape[0]
    k = beam_size
    prev = torch.zeros(k, dtype=torch.long)
    seqs = prev.unsqueeze(1)
    top_scores = torch.zeros(k, 1, dtype=emb_w.dtype)
    complete, complete_scores = [], []
    h = h0.expand(k, h0.shape[1])
    step = 1
    while True:
        x = feature.expand(k, feature.shape[1]) if step == 1 else F.embedding(prev, emb_w)
        h = O.gru_cell(x, h, *cells[0])
        scores = F.log_softmax(F.linear(h, p[pre + "fc_out.weight"], p[pre + "fc_out.bias"]), dim=1)
        scores = top_scores.expand_as(scores) + scores
        if step == 1:
            top_scores, top_words = scores[0].topk(k, 0, True, True)
        else:
            top_scores, top_words = scores.reshape(-1).topk(k, 0, True, True)
        prev_inds = torch.div(top_words, V, rounding_mode="floor")
        next_inds = top_words % V
        seqs = torch.cat([seqs[prev_inds], next_inds.unsqueeze(1)], dim=1)
        incomplete = [i for i, w in enumerate(next_inds.tolist()) if w != end_sentence]
        done = [i for i in range(len(next_inds)) if i not in incomplete]
        if done:
            complete.extend(seqs[done].tolist())
            complete_scores.extend(top_scores[done].tolist())
        k -= len(done)
        if k == 0:
            break
        seqs = seqs[incomplete]
        h = h[prev_inds[incomplete]]
        top_scores = top_scores[incomplete].unsqueeze(1)
        prev = next_inds[incomplete]
        if step > max_steps:
            return None
        step += 1
    return complete[complete_scores.index(max(complete_scores))]


def _greedy_caption(tokens, end_sentence=2):
    """Per-step greedy tokens -> the beam result format: leading 0, cut after the first </s>; None without one."""
    tokens = list(tokens)
    if end_sentence not in tokens:
        return None
    return [0] + tokens[:tokens.index(end_sentence) + 1]


def _eos_bias(p):
    p["captioner.fc_out.weight"][2] *= 60.0          # </s> logit swings with h: beams finish at different steps
    p["captioner.fc_out.bias"][2] -= 1.0
    return p


def _oracle_parts(p, style, pooled, E, H):
    cells = O.split_theta_pooled(O.hypernet_theta(p, style, 4), E, H, 1)
    feats = F.linear(pooled, p["image_encoder.fc.weight"], p["image_encoder.fc.bias"])
    return cells, feats


def _model_from(p, E, H, V, L=1, mode="flow", cell="gru"):
    import hypernet_image_captioning_b200 as C
    m = C.HyperNetPooled(E, H, V, None, num_layers=L, type=cell)
    sd = m.state_dict()
    missing = [k for k in p if k not in sd]
    assert not missing, missing
    for k, v in p.items():
        sd[k] = v
    m.load_state_dict(sd)
    m.grad_mode = mode
    return m.cuda()


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the restatement itself, and argument checking
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_beam_size_1_is_greedy(seed):
    """With one beam the search is greedy decoding with an end-of-sentence stop: the tokens of ``decoder_gru_infer``, cut
    after the first </s>.  float64, so no two distinct logits round to one score."""
    D, E, H, V, B, max_steps = 32, 8, 6, 40, 4, 12
    p = {k: v.double() for k, v in _eos_bias(O.init_params_pooled(D, E, H, V, seed=seed)).items()}
    g = torch.Generator().manual_seed(100 + seed)
    style = torch.randn(1, E, generator=g, dtype=torch.float64)
    pooled = torch.randn(B, D, generator=g, dtype=torch.float64)
    h0 = torch.rand(B, H, generator=g, dtype=torch.float64)
    cells, feats = _oracle_parts(p, style, pooled, E, H)
    n_caption = 0
    for bias in (None, -1e4):                       # -1e4: </s> never wins, every image ends without a caption
        if bias is not None:
            p["captioner.fc_out.bias"][2] = bias
        probs = O.decoder_gru_infer(p, cells, feats, max_steps + 1, h0)
        for b in range(B):
            want = _greedy_caption(probs[b].argmax(dim=1).tolist())
            got = pooled_beam_search(p, cells, feats[b:b + 1], h0[b:b + 1], beam_size=1, max_steps=max_steps)
            assert got == want, (seed, bias, b)
            if bias is not None:
                assert got is None
            n_caption += got is not None
    assert n_caption > 0


def test_argument_errors():
    import hypernet_image_captioning_b200 as C
    dec = C.DecoderGRU(8, 6, 5)
    f = torch.zeros(2, 8)
    for k in (0, 9, 6):                             # 6 = V + 1
        with pytest.raises(ValueError):
            dec.beam_search_batched(f, beam_size=k)
    with pytest.raises(ValueError):
        dec.beam_search_batched(torch.zeros(2, 1, 8))
    with pytest.raises(ValueError):
        dec.beam_search_batched(torch.zeros(2, 7))
    with pytest.raises(NotImplementedError):
        C.DecoderRNN(8, 6, 5).beam_search_batched(f)
    att = C.AttentionGru(2048, 8, 6, 6, 5)          # the same checks, before the feature branch runs
    fa = torch.zeros(2, 49, 2048)
    for k in (0, 9, 6):
        with pytest.raises(ValueError):
            att.beam_search_batched(fa, beam_size=k)
    with pytest.raises(ValueError):
        att.beam_search(fa)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the token-fed decode step
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("split", [True, False])
@pytest.mark.parametrize("B", [1, 37, 1536])
@pytest.mark.parametrize("H", [150, 200, 398])
def test_decode_step_tok_matches_gather_then_step(H, B, split):
    """caphn_gru_decode_step_tok == gather_rows(table, tok') + caphn_gru_decode_step(GI) bit for bit, where tok' maps the
    tokens outside [0, V) to 0 (gather_rows itself would give a zero row for a negative index).  H = 398 is the largest H
    the shared-memory bound admits; split = False is bf16 mode (no lo rows)."""
    from hypernet_image_captioning_b200 import ops
    assert ops.gru_decode_step_tok_ok(H) and not ops.gru_decode_step_tok_ok(400)
    V = 1000
    g = torch.Generator().manual_seed(H * 7 + B)
    table = torch.randn(V, 3 * H, generator=g).cuda()
    W_hh = (torch.randn(3 * H, H, generator=g) / H ** 0.5).cuda()
    b_hh = torch.randn(3 * H, generator=g).cuda()
    hprev = torch.rand(B, H, generator=g).cuda()
    tok = torch.randint(0, V, (B,), generator=g, dtype=torch.int32)
    bad = [-1, V, 2 ** 31 - 1]
    tok[:min(B, 3)] = torch.tensor(bad[:min(B, 3)], dtype=torch.int32)
    if B > 3:
        tok[-1] = V - 1
    tok = tok.cuda()
    Kp = ops.round64(H)

    def bufs():
        hi = torch.zeros(B, Kp, device="cuda", dtype=torch.bfloat16)
        lo = torch.zeros(B, Kp, device="cuda", dtype=torch.bfloat16) if split else None
        return torch.full((B, H), 7.0, device="cuda"), hi, lo

    hn, hi, lo = bufs()
    ops.gru_decode_step_tok(tok, table, W_hh, b_hh, hprev, hn, hi, lo)
    hn_r, hi_r, lo_r = bufs()
    tok_r = torch.where((tok >= 0) & (tok < V), tok, torch.zeros_like(tok)).long()
    GI = ops.gather_rows(table, tok_r)
    ops.gru_decode_step(GI, None, None, 0, None, W_hh, b_hh, hprev, hn_r, hi_r, lo_r)
    torch.cuda.synchronize()
    assert torch.isfinite(hn).all()
    assert torch.equal(hn, hn_r)
    assert torch.equal(hi, hi_r)
    if split:
        assert torch.equal(lo, lo_r)
    hn2 = torch.empty_like(hn)                      # without operand rows
    ops.gru_decode_step_tok(tok, table, W_hh, b_hh, hprev, hn2)
    assert torch.equal(hn2, hn_r)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the search
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_beam_size_1_equals_greedy_infer(precision):
    """B = 512, E = 200, H = 150, V = 9684 with hypernet-generated weights: beam_size = 1 reproduces ``infer``'s per-step
    arg-max, cut at the first </s>.  Both run the same GRU kernel and the same GEMM bits; they can only part where the
    score x - lse rounds two distinct logits to one value, so a row whose top-2 gap in ``infer``'s output is below 1e-6 of
    the row maximum at some step before the cut is not compared."""
    from hypernet_image_captioning_b200 import graphs, ops
    B, E, H, V, max_steps = 512, 200, 150, 9684, 20
    p = _eos_bias(O.init_params_pooled(2048, E, H, V, seed=11))
    g = torch.Generator().manual_seed(3)
    style, pooled = torch.randn(1, E, generator=g), torch.randn(B, 2048, generator=g)
    h0 = torch.rand(B, H, generator=g).cuda()
    m = _model_from(p, E, H, V)
    ops.set_precision(precision)
    try:
        graphs.clear()
        with torch.no_grad():
            captioner = m.forward(style.cuda())
            feats = m.image_encoder(pooled.cuda())
            probs = captioner.infer(feats, max_len=max_steps + 1, h0=h0)
            got = captioner.beam_search_batched(feats, beam_size=1, max_steps=max_steps, h0=h0)
    finally:
        ops.set_precision("fp32")
        graphs.clear()
    top2 = probs.topk(2, dim=2).values.cpu()
    close = (top2[..., 0] - top2[..., 1]) < 1e-6 * top2[..., 0]          # [B, T]
    toks = probs.argmax(dim=2).cpu()
    n_checked = n_none = 0
    for b in range(B):
        want = _greedy_caption(toks[b].tolist())
        n = len(want) - 1 if want is not None else max_steps + 1
        if close[b, :n].any():
            continue
        assert got[b] == want, (b, got[b], want)
        n_checked += 1
        n_none += want is None
    print(f"[greedy identity {precision}] {n_checked}/{B} rows checked, {B - n_checked} excluded as near-ties "
          f"({n_none} without a caption)")
    assert n_checked >= 0.95 * B
    assert n_none < n_checked


def _search_vs_oracle(B, V, E, H, k, max_steps, seed, extra_checks=None):
    """Runs the batched search and compares every image with ``pooled_beam_search``.  A beam decision between two
    candidates whose scores differ by less than the 1e-5-class rounding of the GPU products is ambiguous; such images
    are found by re-running the ORACLE with fc_out.weight perturbed at 2e-5 relative and are not compared."""
    p = _eos_bias(O.init_params_pooled(2048, E, H, V, seed=seed))
    g = torch.Generator().manual_seed(seed + 1)
    style, pooled, h0 = torch.randn(1, E, generator=g), torch.randn(B, 2048, generator=g), torch.rand(B, H, generator=g)
    m = _model_from(p, E, H, V)
    with torch.no_grad():
        captioner = m.forward(style.cuda())
        feats = m.image_encoder(pooled.cuda())
    got = captioner.beam_search_batched(feats, beam_size=k, max_steps=max_steps, h0=h0.cuda())
    cells, feats_o = _oracle_parts(p, style, pooled, E, H)
    variants = [p]
    for _ in range(3):
        q = dict(p)
        q["captioner.fc_out.weight"] = p["captioner.fc_out.weight"] * (1 + 2e-5 * torch.randn(V, H, generator=g))
        variants.append(q)
    checked, n_none = [], 0
    for b in range(B):
        wants = [pooled_beam_search(q, cells, feats_o[b:b + 1], h0[b:b + 1], beam_size=k, max_steps=max_steps)
                 for q in variants]
        if any(w != wants[0] for w in wants[1:]):
            continue                                # a near-tie somewhere along this image's search
        assert got[b] == wants[0], (B, V, H, k, b, got[b], wants[0])
        checked.append(b)
        n_none += wants[0] is None
    print(f"[pooled beam B={B} V={V} H={H} k={k}] {len(checked)}/{B} images unambiguous and identical "
          f"({n_none} without a caption), lengths {sorted(len(x) for x in got if x)[::max(1, B // 6)]}")
    assert len(checked) >= max(1, int(0.8 * B))
    return captioner, feats, h0.cuda(), got, checked


@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 5])
def test_beam_search_matches_oracle(k):
    """B = 48, V = 1500, E = 200, H = 150, max_steps = 20: B k >= 128 rows, so the vocabulary projection runs on the tensor
    cores from the operand rows the decode step writes.  Also: the same images in another order give the same results
    bit for bit, a subset (and sync_every = 1) gives the same results for every unambiguous image, and one image with NaN
    features ends without a caption while every other result stays as it was."""
    B, V, E, H = 48, 1500, 200, 150
    captioner, feats, h0, got, checked = _search_vs_oracle(B, V, E, H, k, 20, seed=31)
    assert sum(x is not None for x in got) > B // 4
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(k)).cuda()
    got_p = captioner.beam_search_batched(feats[perm], beam_size=k, max_steps=20, h0=h0[perm], sync_every=1)
    for j, b in enumerate(perm.tolist()):
        assert got_p[j] == got[b], (j, b)
    sub = torch.tensor([5, 0, 17, 5, 40, 23, 11], device="cuda")
    got_s = captioner.beam_search_batched(feats[sub], beam_size=k, max_steps=20, h0=h0[sub], sync_every=1)
    for j, b in enumerate(sub.tolist()):
        if b in checked:
            assert got_s[j] == got[b], (j, b)
    bad = feats.clone()
    bad[7] = float("nan")
    got_n = captioner.beam_search_batched(bad, beam_size=k, max_steps=20, h0=h0)
    assert got_n[7] is None
    for b in range(B):
        if b != 7:
            assert got_n[b] == got[b], b
        if got_n[b] is not None:
            assert all(0 <= t < V for t in got_n[b])


@pytest.mark.gpu
@pytest.mark.parametrize("B,V,H,k", [
    (2, 1500, 150, 3),              # 6 rows: SIMT vocabulary projection
    (48, 1500, 151, 3),             # odd H: table gather + GRU step kernel instead of the fused step
    (16, 16385, 150, 3),            # V above the fused greedy step's partials limit
])
def test_beam_search_matches_oracle_other_paths(B, V, H, k):
    _search_vs_oracle(B, V, 200, H, k, 20, seed=7)
