"""The oracle port (oracle/caption_hn_oracle.py) against vectors produced by the unmodified reference."""
import numpy as np
import pytest
import torch

from oracle import caption_hn_oracle as O
from golden_util import load_case, params_of, rel_err, grad_close, golden_rel_err, golden_grad_close

TOL = 2e-6  # same torch CPU kernels in the same order; observed <= 1e-6


def _leafify(p):
    return {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in p.items()}


@pytest.mark.parametrize("name", ["attn_flickr", "attn_cc"])
def test_attention_variant_matches_reference(name):
    c = load_case(name)
    p = _leafify(params_of(c))
    rng = np.random.RandomState(0)
    logits, att, theta, gw = O.path_attention(p, c["style"], c["features"], c["captions"], 0.0, rng, flow=False)
    for k, w in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), gw):
        assert rel_err(w, c["gen/" + k]) < TOL, k
    assert rel_err(logits, c["tf/logits"]) < TOL
    assert rel_err(att, c["tf/attn"]) < TOL
    loss = O.caption_loss(logits, c["captions"], 0)
    assert abs(loss.item() - c["tf/loss"].item()) < 1e-6 * abs(c["tf/loss"].item()) + 1e-7
    loss.backward()
    for k, w in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), gw):
        assert grad_close(w.grad, c["tf/grad/captioner.gru." + k], 1e-5), k
    nograd = set(c["tf/nograd"].tolist())
    for k, v in p.items():
        if "tf/grad/" + k in c:
            assert grad_close(v.grad, c["tf/grad/" + k], 1e-5), k
        elif k in nograd:  # reference graph cut: hypernet params get no gradient in literal mode
            assert v.grad is None or float(v.grad.abs().max()) == 0.0, k


@pytest.mark.parametrize("name", ["attn_flickr", "attn_cc"])
def test_attention_variant_flow_grads(name):
    c = load_case(name)
    p = _leafify(params_of(c))
    logits, _, _, _ = O.path_attention(p, c["style"], c["features"], c["captions"], 0.0,
                                       np.random.RandomState(0), flow=True)
    O.caption_loss(logits, c["captions"], 0).backward()
    n = 0
    for k, v in c.items():
        if k.startswith("flow/grad/"):
            assert grad_close(p[k[10:]].grad, v, 1e-5), k
            n += 1
    assert n >= 12


@pytest.mark.parametrize("name", ["attn_flickr", "attn_cc"])
def test_attention_variant_greedy_token_exact(name):
    c = load_case(name)
    p = params_of(c)
    with torch.no_grad():
        logits, att, _, _ = O.path_attention(p, c["style"], c["features"], c["captions"], 1.0,
                                             np.random.RandomState(0))
    assert torch.equal(logits.argmax(-1), c["greedy/logits"].argmax(-1))
    assert rel_err(logits, c["greedy/logits"]) < TOL
    assert rel_err(att, c["greedy/attn"]) < TOL


POOLED_CASES = [("pooled_l1", 1, "gru"), ("pooled_l2", 2, "gru"), ("pooled_lstm_l1", 1, "lstm"), ("pooled_lstm_l2", 2, "lstm")]


@pytest.mark.parametrize("name,L,kind", POOLED_CASES)
def test_pooled_variant_matches_reference(name, L, kind):
    """GRU (DecoderGRU) and LSTM (DecoderRNN, hypernet.py:53) captioners of the pooled hypernet."""
    c = load_case(name)
    p = _leafify(params_of(c))
    logits, theta, cells = O.path_pooled(p, c["style"], c["pooled"], c["captions"], c["h0"], L=L, flow=False, cell=kind)
    for ci, cell in enumerate(cells):
        for k, w in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), cell):
            assert rel_err(w, c[f"gen/{ci}/{k}"]) < TOL, (ci, k)
    assert golden_rel_err(c, "tf/logits", logits) < TOL
    loss = O.caption_loss(logits, c["captions"], None)
    assert abs(loss.item() - c["tf/loss"].item()) < 1e-6 * abs(c["tf/loss"].item())
    loss.backward()
    for ci, cell in enumerate(cells):
        for k, w in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), cell):
            assert grad_close(w.grad, c[f"tf/grad/gen/{ci}/{k}"], 1e-5), (ci, k)
    for k in ("image_encoder.fc.weight", "captioner.embed.weight", "captioner.fc_out.weight", "captioner.fc_out.bias"):
        assert golden_grad_close(c, "tf/grad/" + k, p[k].grad, 1e-5), k
    with torch.no_grad():
        probs, _, _ = O.path_pooled(p, c["style"], c["pooled"], None, c["h0"], L=L, infer_len=c["infer/probs"].shape[1],
                                    cell=kind)
    assert torch.equal(probs.argmax(-1), c["infer/tokens"])
    assert golden_rel_err(c, "infer/probs", probs) < TOL


@pytest.mark.parametrize("name,L,kind", POOLED_CASES)
def test_pooled_variant_flow_grads(name, L, kind):
    c = load_case(name)
    p = _leafify(params_of(c))
    logits, _, _ = O.path_pooled(p, c["style"], c["pooled"], c["captions"], c["h0"], L=L, flow=True, cell=kind)
    O.caption_loss(logits, c["captions"], None).backward()
    n = 0
    for k, v in c.items():
        if k.startswith("flow/grad/"):
            assert grad_close(p[k[10:]].grad, v, 1e-5), k
            n += 1
    assert n >= 12


@pytest.mark.parametrize("name", ["attn_flickr", "attn_cc"])
def test_attention_greedy_search_matches_reference(name):
    c = load_case(name)
    p = params_of(c)
    E, Fo, H = O.dims_attention(p)
    with torch.no_grad():
        gw = O.split_theta_attention(O.hypernet_theta(p, c["style"], 4), E, Fo, H)
        for bi in range(c["features"].shape[0]):
            f = c["features"][bi:bi + 1]
            fproj = torch.nn.functional.linear(torch.relu(torch.nn.functional.linear(
                f, p["captioner.feature_fc.0.weight"], p["captioner.feature_fc.0.bias"])),
                p["captioner.feature_fc.2.weight"], p["captioner.feature_fc.2.bias"])
            toks, wts = O.attention_gru_greedy_search(p, gw, fproj, 2, 7)
            assert toks == c[f"gs/{bi}/tokens"].tolist()
            assert rel_err(wts, c[f"gs/{bi}/weights"]) < TOL


BEAM_TAGS = ["a", "b", "c", "d", "noeos"]


@pytest.mark.parametrize("tag", BEAM_TAGS)
def test_attention_beam_search_matches_reference_test_step(tag):
    """Beam search k = 3 of HyperNet.test_step (hypernet_attention.py:247-326): golden = the caption the unmodified
    reference hands to metric_score_test (or no caption at all when a beam is still open after 51 steps)."""
    c = load_case("attn_flickr")
    p = params_of(c)
    p["captioner.fc.bias"] = c[f"beam/{tag}/fc_bias"]
    p["captioner.fc.weight"] = c[f"beam/{tag}/fc_weight"]
    E, Fo, H = O.dims_attention(p)
    with torch.no_grad():
        style = p["captioner.embed.weight"][int(c["beam/style_id"])].reshape(1, -1)     # :244-246
        gw = O.split_theta_attention(O.hypernet_theta(p, style, 4), E, Fo, H)
        for bi in range(c["features"].shape[0]):
            got = O.attention_beam_search(p, gw, c["features"][bi:bi + 1], 3, 2, 50)
            want = c[f"beam/{tag}/{bi}"].tolist()
            assert (got if got is not None else [-1]) == want, (tag, bi)


# ----------------------------------------------------------------------------------------------------------------------
# caption metrics, token-level part (oracle/metrics_oracle.py)
# ----------------------------------------------------------------------------------------------------------------------
def _metrics_logits(c):
    B, T = c["pred_ids"].shape
    logits = torch.zeros(B, T, int(c["V"]))
    logits.scatter_(2, c["pred_ids"].unsqueeze(-1), 1.0)
    logits.scatter_(2, c["tie_ids"].unsqueeze(-1), 1.0)
    return logits


def test_metrics_oracle_token_filter_matches_reference_cap_to_text():
    """tests/golden/metrics.npz = utils.cap_to_text / cap_to_text_gt of the unmodified reference (with its vocab.pkl)."""
    from golden_util import load_case
    from oracle import metrics_oracle as MO
    c = load_case("metrics")
    logits = _metrics_logits(c)
    for b in range(logits.shape[0]):
        hyp = MO.cap_tokens_from_logits(logits[b])
        assert hyp == c["hyp"][b, :int(c["hyp_len"][b])].tolist(), b
        ref = MO.cap_tokens(c["gt_ids"][b].tolist())
        assert ref == c["ref"][b, :int(c["ref_len"][b])].tolist(), b
    assert int(c["hyp_len"][1]) == 0 and int(c["ref_len"][2]) == 0 and int(c["hyp_len"][0]) == logits.shape[1]


def test_metrics_oracle_bleu_known_answers():
    """compute_bleu (tensorflow/nmt scripts/bleu.py, wrapped by the `datasets` "bleu" metric): hand-computed cases."""
    import math
    from oracle import metrics_oracle as MO
    a = [5, 6, 7, 8, 9, 10]
    assert MO.compute_bleu([a], [a], 4) == pytest.approx(1.0)
    # clipping: "the the the the the the the" vs "the cat is on the mat" -> unigram precision 2/7, longer hypothesis: bp = 1
    hyp, ref = [1] * 7, [1, 2, 3, 4, 1, 5]
    assert MO.compute_bleu([hyp], [ref], 1) == pytest.approx(2.0 / 7.0)
    assert MO.compute_bleu([hyp], [ref], 2) == 0.0                      # no bigram match, no smoothing
    # brevity penalty: hypothesis = first 4 of 6 reference tokens: p1 = p2 = 1, bp = exp(1 - 6/4)
    assert MO.compute_bleu([a[:4]], [a], 2) == pytest.approx(math.exp(1.0 - 6.0 / 4.0))
    # corpus level: statistics are summed over sentence pairs before the ratio is taken
    m, p, hl, rl = MO.bleu_counts([a, hyp], [a, ref], 4)
    assert (m, p, hl, rl) == ([8, 5, 4, 3], [13, 11, 9, 7], 13, 12)
    assert MO.bleu_from_counts(m, p, hl, rl, 4) == pytest.approx(math.exp(sum(math.log(x) for x in
                                                                      (8 / 13, 5 / 11, 4 / 9, 3 / 7)) / 4))
    assert MO.compute_bleu([[]], [a], 4) == 0.0


def test_metrics_host_arithmetic_matches_oracle():
    """hypernet_image_captioning_b200.metrics.bleu_from_counts (the host half of the product path: ten integers ->
    BLEU-n) against the oracle's compute_bleu on random corpora, incl. empty hypotheses and zero-match orders."""
    import random
    from hypernet_image_captioning_b200 import metrics
    from oracle import metrics_oracle as MO
    rng = random.Random(3)
    for trial in range(50):
        B = rng.randint(1, 6)
        hyps = [[rng.randint(3, 8) for _ in range(rng.randint(0, 9))] for _ in range(B)]
        refs = [[rng.randint(3, 8) for _ in range(rng.randint(0, 9))] for _ in range(B)]
        m, p, hl, rl = MO.bleu_counts(hyps, refs, 4)
        counts = m + p + [hl, rl]
        for n in (1, 2, 3, 4):
            assert metrics.bleu_from_counts(counts, n) == pytest.approx(MO.compute_bleu(hyps, refs, n), rel=1e-12, abs=0.0)


def test_projection_table_rule():
    """ops.use_projection_table: the per-call table (V-row GEMM) is chosen once the per-step rows outnumber V / 2."""
    from hypernet_image_captioning_b200 import ops
    assert ops.use_projection_table(512, 20, 9684) and ops.use_projection_table(4096, 16, 9684)
    assert not ops.use_projection_table(1, 20, 9684) and not ops.use_projection_table(64, 20, 9684)
    assert not ops.use_projection_table(512, 1, 9684)
