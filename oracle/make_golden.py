"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED reference modules.

Run in the build container (the only place /root/reference exists):

    python oracle/make_golden.py

Every vector below is produced by the reference's own objects (hypernet_attention.HyperNet, AttentionGru,
hypernet.HyperNet, DecoderGRU) imported through oracle/ref_harness.py -- not by the oracle port.  The port
(oracle/caption_hn_oracle.py) and the CUDA path are then both checked against these files.

Cases
  attn_flickr : Variant B, style vector [1,E] (hypernet_attention.py:139-142), teacher-forced + greedy, literal grads
  attn_cc     : Variant B, cc=True, 1-D one-hot style [he] (cc_train_hypernet.py:141-144), teacher-forced + greedy
  pooled_l1   : Variant A, L=1, DecoderGRU.forward + infer (V must be 9684, later.py:449)
  pooled_l2   : Variant A, L=2 (exercises the offset-0 slicing of utils.py:45,68)
"flow" gradients (hypernet heads receiving gradient) come from the reference with ONE change made here in the
harness, not in the reference: set_all_parameters without the nn.Parameter(...) wrapper of utils.py:57.
"""
import hashlib
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import ref_harness  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _sd(model):
    return {k: v.detach().clone() for k, v in model.state_dict().items()
            if not (k.startswith("image_encoder.") and not k.startswith("image_encoder.fc."))}


def _np(d):
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in d.items()}


# Every file under tests/golden stays below 1 MB.  What makes a case large is stored in a reduced form that
# tests/golden_util.py expands or compares against.  Only the vocabulary sample of the pooled outputs drops values a
# check used to read.
FEATURES_SEED = 1234     # the attention cases draw `features` first from torch.Generator().manual_seed(FEATURES_SEED)
VOCAB_SAMPLE = 1024      # vocabulary entries kept of the pooled cases' [.., V] outputs
VOCAB_SAMPLED = {"tf/logits": 2, "infer/probs": 2, "tf/grad/captioner.fc_out.weight": 0,
                 "tf/grad/captioner.fc_out.bias": 0}


def shrink_attention(out):
    """`features` (0.8 MB of randn) is redrawn from its seed by the tests; its SHA-256 pins the bytes."""
    out = dict(out)
    f = np.ascontiguousarray(out.pop("features"), dtype=np.float32)
    g = torch.Generator().manual_seed(FEATURES_SEED)
    assert np.array_equal(torch.randn(f.shape, generator=g).numpy(), f)
    out["features/seed"] = np.int64(FEATURES_SEED)
    out["features/shape"] = np.array(f.shape, dtype=np.int64)
    out["features/sha256"] = np.array(hashlib.sha256(f.tobytes()).hexdigest())
    return out


def shrink_pooled(out):
    """Embedding rows the case never reads are dropped (the tests see zeros there); the [.., V] outputs keep a fixed
    sample of vocabulary entries -- every caption and greedy token among them -- plus max|x| of the full array, so a
    relative error keeps its full-array scale; the greedy tokens are stored whole."""
    out = dict(out)
    emb = out.pop("sd/captioner.embed.weight")
    tokens = out["infer/probs"].argmax(-1)
    rows = np.union1d(out["captions"].ravel(), tokens.ravel())
    out["sd/captioner.embed.weight/shape"] = np.array(emb.shape, dtype=np.int64)
    out["sd/captioner.embed.weight/rows"] = rows.astype(np.int64)
    out["sd/captioner.embed.weight/values"] = emb[rows]
    V = emb.shape[0]
    keep = np.random.RandomState(0).choice(V, VOCAB_SAMPLE, replace=False)
    sample = np.union1d(keep, rows).astype(np.int64)
    out["infer/tokens"] = tokens.astype(np.int64)
    out["vocab_sample"] = sample
    for k, axis in VOCAB_SAMPLED.items():
        x = out[k]
        out["absmax/" + k] = np.abs(x).max()
        out["vocab_axis/" + k] = np.int64(axis)
        out[k] = np.ascontiguousarray(np.take(x, sample, axis=axis))
    return out


def _flow_set_all_parameters(module, theta):
    """utils.py:44-69 minus the nn.Parameter wrapper at :57 (keeps the autograd graph)."""
    count = 0
    for name in module.registered_parameters_name:
        if name in ("weight", "bias"):
            continue
        a = count
        b = a + getattr(module, name).numel()
        t = torch.reshape(theta[0, a:b], getattr(module, name).shape)
        if name in module._parameters:
            del module._parameters[name]
        object.__setattr__(module, name, t)
        count += t.numel()
    for name in [k for k in module._modules]:
        if name in ("embed", "fc_out"):
            continue
        count += _flow_set_all_parameters(module._modules[name], theta)
    return count


# (tag, step at which the </s> logit crosses zero, its gain, scale of the other fc rows); None: </s> never wins
BEAM_CASES = [("a", 3, 60.0, 8.0), ("b", 3, 200.0, 8.0), ("c", 6, 60.0, 3.0), ("d", 2, 20.0, 8.0), ("noeos", None, 0.0, 1.0)]


def case_attention(ref, name, cc, style, Fo=16, E=12, H=20, V=50, he=10, B=2, T=6):
    torch.manual_seed(0)
    model = ref.HyperNetAttention(Fo, E, H, V, ref.vocab, cc=cc, hyper_emb=he)
    sd = _sd(model)
    g = torch.Generator().manual_seed(1234)
    features = torch.randn(B, 49, 2048, generator=g)
    caps = torch.randint(4, V, (B, T), generator=g)
    caps[:, 0] = 1
    caps[1, T - 2] = 2
    caps[1, T - 1] = 0
    out = {"features": features, "captions": caps, "style": style}
    out.update({"sd/" + k: v for k, v in sd.items() if not k.startswith("captioner.gru.")})

    # literal mode, teacher-forced (cc_train_hypernet.py:150-153)
    np.random.seed(0)
    captioner = model.forward(style)
    logits, att = captioner(features, caps, 0.0)
    loss = F.cross_entropy(logits.view(-1, V), caps.view(-1), ignore_index=0)
    model.zero_grad(set_to_none=True)
    loss.backward()
    out["tf/logits"], out["tf/attn"], out["tf/loss"] = logits, att, loss
    for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
        out["gen/" + k] = getattr(captioner.gru, k).detach().clone()
        out["tf/grad/captioner.gru." + k] = getattr(captioner.gru, k).grad.clone()
    for k, v in model.named_parameters():
        if k.startswith("image_encoder") or k.startswith("captioner.gru."):
            continue
        if v.grad is not None:
            out["tf/grad/" + k] = v.grad.clone()
        else:
            out.setdefault("tf/nograd", []).append(k)
    out["tf/nograd"] = np.array(out.get("tf/nograd", []))

    # greedy, test_hn.py path (cc_train_hypernet.py:228-230)
    np.random.seed(0)
    with torch.no_grad():
        captioner = model.forward(style)
        glogits, gatt = captioner(features, caps, 1.0)
    out["greedy/logits"], out["greedy/attn"] = glogits, gatt

    # B = 1 greedy_search with EOS stop (models/decoderlstm.py:138-175): takes features ALREADY through feature_fc
    with torch.no_grad():
        captioner = model.forward(style)
        for bi in range(B):
            fproj = captioner.feature_fc(features[bi:bi + 1])
            sent, wts = captioner.greedy_search(fproj, end_sentence=2, max_sentence=7)
            out[f"gs/{bi}/tokens"] = torch.tensor(sent)
            out[f"gs/{bi}/weights"] = torch.stack([w.reshape(-1) for w in wts], 0)

    # beam search k = 3: the reference's own test_step (hypernet_attention.py:240-326), unmodified.  Harness-side only:
    # image_encoder is the identity (precomputed features are passed as "imgs"), the metric functions are replaced by a
    # recorder of caps_pred_beam, and the </s> logit bias is shifted so that beams do (eos) / never (noeos) terminate.
    if not cc:
        import hypernet_attention as ref_hna0
        captured = []
        saved = (ref_hna0.metric_score_test, ref_hna0.metric_score, model.image_encoder)
        ref_hna0.metric_score_test = lambda c_, pred, v_, m_: (captured.append(pred.clone()), (0,) * 6)[1]
        ref_hna0.metric_score = lambda *a_, **k_: (0,) * 6
        object.__setattr__(model, "image_encoder", lambda imgs: imgs)
        model._modules.pop("image_encoder", None)
        base_bias = model.captioner.fc.bias.detach().clone()
        base_w = model.captioner.fc.weight.detach().clone()
        # With random weights h_t converges within a few steps, so </s> is either in the top-k at step 1 or never.  To get
        # beams that end after a few words, the </s> row of fc is pointed along the drift of the hidden state: its logit
        # grows with t and crosses the other words' logits around step `cross`.
        with torch.no_grad():
            cap0 = model.forward(model.captioner.embed(torch.tensor([ref.vocab("<unk>")])))
            enc = cap0.feature_fc(features[0:1])
            hs, h = [], cap0.init_hidden(enc)
            x = torch.zeros(1, E)
            for _ in range(12):
                ctx_, _ = cap0.attention(enc, h)
                h = cap0.gru(torch.cat([x, ctx_], 1), h)
                hs.append(h[0].clone())
                x = cap0.embed(cap0.fc(h).argmax(1))
        try:
            for tag, cross, gain, wscale in BEAM_CASES:
                with torch.no_grad():
                    model.captioner.fc.bias.copy_(base_bias)
                    model.captioner.fc.weight.copy_(base_w * wscale)     # sharper word distributions
                    if cross is None:
                        model.captioner.fc.bias[2] = -100.0
                    else:
                        d = hs[-1] - hs[0]
                        d = d / d.dot(d)                                  # d . (h_t - h_1) goes 0 -> 1
                        prog = d.dot(hs[cross] - hs[0])
                        model.captioner.fc.weight[2] = gain * d
                        model.captioner.fc.bias[2] = -gain * (d.dot(hs[0]) + prog)   # logit(</s>) = gain (progress_t - progress_cross)
                out[f"beam/{tag}/fc_bias"] = model.captioner.fc.bias.detach().clone()
                out[f"beam/{tag}/fc_weight"] = model.captioner.fc.weight.detach().clone()
                for bi in range(B):
                    captured.clear()
                    np.random.seed(0)
                    with torch.no_grad():
                        model.test_step((features[bi:bi + 1], ("<unk>", (caps[bi:bi + 1], None))), 0)
                    out[f"beam/{tag}/{bi}"] = captured[0] if captured else torch.tensor([-1])
                    print(name, "beam", tag, bi, out[f"beam/{tag}/{bi}"].tolist())
        finally:
            ref_hna0.metric_score_test, ref_hna0.metric_score = saved[0], saved[1]
            model._modules["image_encoder"] = saved[2]
            with torch.no_grad():
                model.captioner.fc.bias.copy_(base_bias)
                model.captioner.fc.weight.copy_(base_w)
        out["beam/style_id"] = torch.tensor(ref.vocab("<unk>"))

    # flow mode gradients (harness-side patch of set_all_parameters only)
    import hypernet_attention as ref_hna
    orig = ref_hna.set_all_parameters
    ref_hna.set_all_parameters = _flow_set_all_parameters
    try:
        torch.manual_seed(0)
        model2 = ref.HyperNetAttention(Fo, E, H, V, ref.vocab, cc=cc, hyper_emb=he)
        np.random.seed(0)
        captioner = model2.forward(style)
        logits2, _ = captioner(features, caps, 0.0)
        loss2 = F.cross_entropy(logits2.view(-1, V), caps.view(-1), ignore_index=0)
        loss2.backward()
        assert torch.equal(logits2, logits)
        for k, v in model2.named_parameters():
            if k.startswith("hn_") and v.grad is not None:
                out["flow/grad/" + k] = v.grad.clone()
    finally:
        ref_hna.set_all_parameters = orig
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **shrink_attention(_np(out)))
    print(name, "loss", float(loss), "logits", tuple(logits.shape))


def case_pooled(ref, name, L, E=8, H=6, B=2, T=5, max_len=4, kind="gru"):
    V = 9684  # later.py:449 / :311 hard-code it
    torch.manual_seed(0)
    model = ref.HyperNetPooled(E, H, V, ref.vocab, num_layers=L, type=kind)
    sd = _sd(model)
    g = torch.Generator().manual_seed(4321)
    pooled = torch.relu(torch.randn(B, 2048, generator=g))
    caps = torch.randint(7, 3000, (B, T), generator=g)
    caps[:, 0] = 1
    style = torch.randn(1, E, generator=g)
    out = {"pooled": pooled, "captions": caps, "style": style}
    out.update({"sd/" + k: v for k, v in sd.items()
                if not (k.startswith("captioner.lstm_cell.") or k.startswith("captioner.layers."))})

    captioner = model.forward(style)
    feats = model.image_encoder.fc(pooled)  # hypernet.py:46,134
    torch.manual_seed(1)
    h0 = torch.rand(B, H)
    torch.manual_seed(1)  # DecoderGRU.forward draws torch.rand(B,H) first (later.py:393)
    logits = captioner(feats, caps, True)
    loss = F.cross_entropy(logits.view(-1, V), caps.view(-1))  # hypernet.py:145, no ignore_index
    model.zero_grad(set_to_none=True)
    loss.backward()
    out["h0"], out["tf/logits"], out["tf/loss"] = h0, logits, loss
    cells = [captioner.lstm_cell] + (list(captioner.layers) if captioner.layers else [])
    for ci, cell in enumerate(cells):
        for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
            out[f"gen/{ci}/{k}"] = getattr(cell, k).detach().clone()
            out[f"tf/grad/gen/{ci}/{k}"] = getattr(cell, k).grad.clone()
    for k in ("image_encoder.fc.weight", "image_encoder.fc.bias", "captioner.embed.weight",
              "captioner.fc_out.weight", "captioner.fc_out.bias"):
        out["tf/grad/" + k] = dict(model.named_parameters())[k].grad.clone()

    with torch.no_grad():
        captioner = model.forward(style)
        torch.manual_seed(1)
        probs = captioner.infer(model.image_encoder.fc(pooled), max_len=max_len)
    out["infer/probs"] = probs

    import hypernet as ref_hn
    orig = ref_hn.set_all_parameters
    ref_hn.set_all_parameters = _flow_set_all_parameters
    try:
        torch.manual_seed(0)
        model2 = ref.HyperNetPooled(E, H, V, ref.vocab, num_layers=L, type=kind)
        captioner = model2.forward(style)
        torch.manual_seed(1)
        logits2 = captioner(model2.image_encoder.fc(pooled), caps, True)
        loss2 = F.cross_entropy(logits2.view(-1, V), caps.view(-1))
        loss2.backward()
        assert torch.equal(logits2, logits)
        for k, v in model2.named_parameters():
            if k.startswith("hn_") and v.grad is not None:
                out["flow/grad/" + k] = v.grad.clone()
    finally:
        ref_hn.set_all_parameters = orig
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **shrink_pooled(_np(out)))
    print(name, "loss", float(loss), "logits", tuple(logits.shape))


def case_metrics(ref, name="metrics", B=8, T=12):
    """utils.py:161-190 cap_to_text / cap_to_text_gt of the unmodified reference with its own data/vocab.pkl, mapped back
    to token ids (vocab.w2i).  Logits are rebuilt by the tests from `pred_ids` / `tie_ids` exactly as here: zeros, 1.0 at
    pred_ids[b,t] and -- a tie, resolved to the lower index by torch.argmax -- 1.0 at tie_ids[b,t] >= pred_ids[b,t]."""
    voc = ref.vocab
    V = len(voc.i2w)
    g = torch.Generator().manual_seed(11)
    def draw():
        ids = torch.randint(7, V, (B, T), generator=g)
        special = torch.randint(0, 10, (B, T), generator=g)
        ids[special == 0] = 0      # <pad> in the middle of a caption is skipped, not a stop
        ids[special == 1] = 1      # <s>
        ids[special == 2] = 2      # </s>: everything after the first one is dropped
        return ids
    pred_ids, gt_ids = draw(), draw()
    pred_ids[0, :] = torch.randint(7, V, (T,), generator=g)        # no </s> at all: full length
    pred_ids[1, 0] = 2                                             # empty caption
    gt_ids[2, :3] = torch.tensor([1, 0, 2])                        # <s> <pad> </s>: empty reference
    tie_ids = torch.minimum(pred_ids + torch.randint(0, 5, (B, T), generator=g), torch.tensor(V - 1))
    logits = torch.zeros(B, T, V)
    logits.scatter_(2, pred_ids.unsqueeze(-1), 1.0)
    logits.scatter_(2, tie_ids.unsqueeze(-1), 1.0)
    out = {"pred_ids": pred_ids, "tie_ids": tie_ids, "gt_ids": gt_ids}
    hyp = torch.zeros(B, T, dtype=torch.int64)
    refc = torch.zeros(B, T, dtype=torch.int64)
    hl, rl = torch.zeros(B, dtype=torch.int32), torch.zeros(B, dtype=torch.int32)
    for b in range(B):
        words = ref.utils.cap_to_text(logits[b], voc, tokenized=True)
        assert ref.utils.cap_to_text(logits[b], voc, tokenized=False) == " ".join(words)
        gwords = ref.utils.cap_to_text_gt(gt_ids[b], voc, tokenized=True)
        hl[b], rl[b] = len(words), len(gwords)
        hyp[b, :len(words)] = torch.tensor([voc.w2i[w] for w in words], dtype=torch.int64)
        refc[b, :len(gwords)] = torch.tensor([voc.w2i[w] for w in gwords], dtype=torch.int64)
    out.update({"hyp": hyp, "hyp_len": hl, "ref": refc, "ref_len": rl, "V": torch.tensor(V)})
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **_np(out))
    print(name, "hyp_len", hl.tolist(), "ref_len", rl.tolist())


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = ref_harness.load()
    g = torch.Generator().manual_seed(7)
    case_attention(ref, "attn_flickr", cc=False, style=torch.randn(1, 12, generator=g))
    onehot = torch.zeros(10)
    onehot[3] = 1.0
    case_attention(ref, "attn_cc", cc=True, style=onehot, he=10)
    case_pooled(ref, "pooled_l1", L=1)
    case_pooled(ref, "pooled_l2", L=2)
    case_pooled(ref, "pooled_lstm_l1", L=1, kind="lstm")      # hypernet.py:53: DecoderRNN (later.py:227), zero (h, c)
    case_pooled(ref, "pooled_lstm_l2", L=2, kind="lstm")
    case_metrics(ref)


if __name__ == "__main__":
    main()
