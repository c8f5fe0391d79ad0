"""Module-level parity of the pooled-feature path (HyperNetPooled + DecoderGRU) through the drop-in API:
against the golden vectors of the unmodified reference (tests/golden/pooled_l1.npz) and against the oracle port
on larger seeded inputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from golden_util import load_case, params_of, rel_err, grad_close, golden_rel_err, golden_grad_close
from oracle import caption_hn_oracle as O

TOL_LOGITS = 1e-4   # BASELINE.json north_star: fp32 mode within 1e-4 relative on logits and loss
TOL_GRAD = 1e-3     # SURVEY 8(d): gradients <= 1e-3 relative


POOLED_CASES = [("pooled_l1", 1, "gru"), ("pooled_l2", 2, "gru"), ("pooled_lstm_l1", 1, "lstm"), ("pooled_lstm_l2", 2, "lstm")]


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


@pytest.mark.parametrize("name,L,kind", POOLED_CASES)
def test_state_dict_layout_matches_reference(name, L, kind):
    c = load_case(name)
    p = params_of(c)
    import hypernet_image_captioning_b200 as C
    m = C.HyperNetPooled(8, 6, 9684, None, num_layers=L, type=kind)
    sd = m.state_dict()
    gen = {"captioner.lstm_cell." + k for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")}
    gen |= {f"captioner.layers.{l}.{k}" for l in range(L - 1) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")}
    assert set(sd.keys()) == set(p.keys()) | gen
    for k, v in p.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k


@pytest.mark.parametrize("name,L,kind", POOLED_CASES)
@pytest.mark.parametrize("mode", ["literal", "flow"])
def test_pooled_golden(name, L, kind, mode):
    """L = 2 exercises the offset-0 aliasing of utils.py:45,68 (layer 2 reads theta[0:...]) and `h = layer(h, h)` /
    `(h, c) = layer(h, (h, c))`; cell = "lstm" is the DecoderRNN captioner of hypernet.py:53 (zero initial state)."""
    c = load_case(name)
    p = params_of(c)
    m = _model_from(p, 8, 6, 9684, L=L, mode=mode, cell=kind)
    import hypernet_image_captioning_b200 as C
    captioner = m.forward(c["style"].cuda())
    cells_mod = [captioner.lstm_cell] + (list(captioner.layers) if captioner.layers else [])
    for ci, cell in enumerate(cells_mod):
        for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
            assert rel_err(getattr(cell, k), c[f"gen/{ci}/{k}"]) < 1e-5, (ci, k)
    feats = m.image_encoder(c["pooled"].cuda())
    h0 = c["h0"].cuda() if kind == "gru" else None        # DecoderRNN starts from zeros (later.py:256-259)
    logits = captioner(feats, c["captions"].cuda(), True, h0=h0)
    assert golden_rel_err(c, "tf/logits", logits) < TOL_LOGITS
    loss = C.cross_entropy(logits, c["captions"].cuda(), None)
    assert abs(loss.item() - c["tf/loss"].item()) < TOL_LOGITS * abs(c["tf/loss"].item())
    loss.backward()
    named = dict(m.named_parameters())
    for k in ("image_encoder.fc.weight", "image_encoder.fc.bias", "captioner.embed.weight",
              "captioner.fc_out.weight", "captioner.fc_out.bias"):
        assert golden_grad_close(c, "tf/grad/" + k, named[k].grad, TOL_GRAD), k
    if mode == "literal":
        for ci, cell in enumerate(cells_mod):
            for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                assert grad_close(getattr(cell, k).grad, c[f"tf/grad/gen/{ci}/{k}"], TOL_GRAD), (ci, k)
        assert all(v.grad is None for k, v in named.items() if k.startswith("hn_"))
    else:
        n = 0
        for k, v in c.items():
            if k.startswith("flow/grad/"):
                assert grad_close(named[k[10:]].grad, v, TOL_GRAD), k
                n += 1
        assert n >= 12


@pytest.mark.parametrize("table", [False, True])
@pytest.mark.parametrize("name,L,kind", POOLED_CASES)
def test_pooled_infer_golden_token_exact(name, L, kind, table, monkeypatch):
    """table = True forces the decode-time projection table (P = Emb W_ih^T + b_ih, one GEMM per call) that large
    batches use instead of a per-step gather + GEMM; both must reproduce the reference's greedy tokens."""
    from hypernet_image_captioning_b200 import graphs, ops
    monkeypatch.setattr(ops, "use_projection_table", lambda B, steps, V: table)
    graphs.clear()
    c = load_case(name)
    m = _model_from(params_of(c), 8, 6, 9684, L=L, cell=kind)
    with torch.no_grad():
        captioner = m.forward(c["style"].cuda())
        probs = captioner.infer(m.image_encoder(c["pooled"].cuda()), max_len=c["infer/probs"].shape[1],
                                h0=c["h0"].cuda() if kind == "gru" else None)
    assert torch.equal(probs.argmax(-1).cpu(), c["infer/tokens"])
    assert golden_rel_err(c, "infer/probs", probs) < TOL_LOGITS


def test_pooled_rng_consumption_matches_reference():
    """DecoderGRU.forward draws torch.rand(B,H) from the global CPU generator (later.py:393)."""
    c = load_case("pooled_l1")
    m = _model_from(params_of(c), 8, 6, 9684)
    captioner = m.forward(c["style"].cuda())
    feats = m.image_encoder(c["pooled"].cuda())
    torch.manual_seed(1)
    logits = captioner(feats, c["captions"].cuda(), True)
    assert golden_rel_err(c, "tf/logits", logits) < TOL_LOGITS


@pytest.mark.parametrize("B,T,E,H,V,L", [(37, 9, 24, 30, 311, 1), (64, 20, 200, 150, 2000, 1), (21, 6, 24, 30, 211, 2),
                                         (10, 5, 16, 12, 97, 3)])
def test_pooled_vs_oracle_medium(B, T, E, H, V, L):
    import hypernet_image_captioning_b200 as C
    p = O.init_params_pooled(2048, E, H, V, L=L, seed=5)
    g = torch.Generator().manual_seed(99)
    pooled = torch.relu(torch.randn(B, 2048, generator=g))
    caps = O.synth_captions(B, T, V, g)
    style = torch.randn(1, E, generator=g)
    h0 = torch.rand(B, H, generator=g)
    pl = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    logits_ref, theta_ref, _ = O.path_pooled(pl, style, pooled, caps, h0, L=L, flow=True)
    loss_ref = O.caption_loss(logits_ref, caps, None)
    loss_ref.backward()

    m = _model_from(p, E, H, V, L=L)
    captioner = m.forward(style.cuda())
    logits = captioner(m.image_encoder(pooled.cuda()), caps.cuda(), True, h0=h0.cuda())
    loss = C.cross_entropy(logits, caps.cuda(), None)
    loss.backward()
    assert rel_err(logits, logits_ref) < TOL_LOGITS
    assert abs(loss.item() - loss_ref.item()) < TOL_LOGITS * abs(loss_ref.item())
    for k, v in m.named_parameters():
        if k.startswith("captioner.lstm_cell.") or k.startswith("captioner.layers."):
            continue
        assert grad_close(v.grad, pl[k].grad, TOL_GRAD), k


@pytest.mark.parametrize("B,T,E,H,V,ignore", [(64, 20, 200, 150, 2000, None), (48, 12, 64, 48, 777, 0), (5, 4, 8, 6, 50, None)])
def test_pooled_fused_loss_matches_unfused(B, T, E, H, V, ignore):
    """forward_loss (decoder + CE in one node, CE gradient emitted as bf16x3 operands) == logits + cross_entropy."""
    import hypernet_image_captioning_b200 as C
    p = O.init_params_pooled(2048, E, H, V, L=1, seed=5)
    g = torch.Generator().manual_seed(99)
    pooled = torch.relu(torch.randn(B, 2048, generator=g)).cuda()
    caps = O.synth_captions(B, T, V, g).cuda()
    style = torch.randn(1, E, generator=g).cuda()
    h0 = torch.rand(B, H, generator=g).cuda()
    grads = []
    for fused in (False, True):
        m = _model_from(p, E, H, V)
        captioner = m.forward(style)
        feats = m.image_encoder(pooled)
        if fused:
            loss, logits = captioner.forward_loss(feats, caps, h0=h0, ignore_index=ignore)
        else:
            logits = captioner(feats, caps, True, h0=h0)
            loss = C.cross_entropy(logits, caps, ignore)
        loss.backward()
        grads.append((loss.item(), logits.detach(), {k: v.grad.clone() for k, v in m.named_parameters() if v.grad is not None}))
    assert abs(grads[0][0] - grads[1][0]) < 1e-6 * abs(grads[0][0])
    assert torch.equal(grads[0][1], grads[1][1])
    for k, v in grads[0][2].items():
        assert grad_close(grads[1][2][k], v, TOL_GRAD), k


@pytest.mark.parametrize("B,T,E,H,V,L", [(37, 9, 24, 30, 311, 1), (64, 20, 200, 150, 2000, 1), (21, 6, 24, 30, 211, 2),
                                         (130, 5, 16, 12, 97, 3)])
@pytest.mark.parametrize("fused", [False, True])
def test_pooled_lstm_vs_oracle_medium(B, T, E, H, V, L, fused):
    """DecoderRNN (LSTM, hypernet.py:53) through the hypernet, flow mode: logits, loss and every gradient against the
    oracle at sizes up to the benchmark's E = 200, H = 150; fused = the decoder + cross-entropy node."""
    import hypernet_image_captioning_b200 as C
    p = O.init_params_pooled(2048, E, H, V, L=L, seed=6, gates=4)
    g = torch.Generator().manual_seed(98)
    pooled = torch.relu(torch.randn(B, 2048, generator=g))
    caps = O.synth_captions(B, T, V, g)
    style = torch.randn(1, E, generator=g)
    pl = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    logits_ref, _, _ = O.path_pooled(pl, style, pooled, caps, None, L=L, flow=True, cell="lstm")
    loss_ref = O.caption_loss(logits_ref, caps, None)
    loss_ref.backward()
    m = _model_from(p, E, H, V, L=L, cell="lstm")
    captioner = m.forward(style.cuda())
    feats = m.image_encoder(pooled.cuda())
    if fused:
        loss, logits = captioner.forward_loss(feats, caps.cuda())
    else:
        logits = captioner(feats, caps.cuda(), True)
        loss = C.cross_entropy(logits, caps.cuda(), None)
    loss.backward()
    assert rel_err(logits, logits_ref) < TOL_LOGITS
    assert abs(loss.item() - loss_ref.item()) < TOL_LOGITS * abs(loss_ref.item())
    for k, v in m.named_parameters():
        if k.startswith("captioner.lstm_cell.") or k.startswith("captioner.layers."):
            continue
        assert grad_close(v.grad, pl[k].grad, TOL_GRAD), k
    with torch.no_grad():
        probs_ref, _, _ = O.path_pooled(p, style, pooled, None, None, L=L, infer_len=6, cell="lstm")
        probs = m.forward(style.cuda()).infer(m.image_encoder(pooled.cuda()), max_len=6)
    assert torch.equal(probs.argmax(-1).cpu(), probs_ref.argmax(-1))


@pytest.mark.parametrize("mode", ["literal", "flow"])
def test_graphed_step_matches_eager(mode):
    """graphs.GraphedStep: the whole fwd+bwd step replayed from one CUDA graph gives the eager step's loss and gradients
    (and, transitively, the reference's: the eager step is pinned by test_pooled_golden), also on fresh inputs."""
    from hypernet_image_captioning_b200 import graphs
    c = load_case("pooled_l1")
    p = params_of(c)
    m = _model_from(p, 8, 6, 9684, L=1, mode=mode)
    pooled, caps, h0 = c["pooled"].cuda(), c["captions"].cuda(), c["h0"].cuda()
    style = c["style"].cuda()

    def step(pooled, caps, h0):
        m.zero_grad(set_to_none=True)
        captioner = m.forward(style)
        loss, _ = captioner.forward_loss(m.image_encoder(pooled), caps, h0=h0, ignore_index=None)
        loss.backward()
        return loss

    def grads():
        named = dict(m.named_parameters())
        return {k: v.grad.detach().clone() for k, v in named.items() if v.grad is not None}

    g = torch.Generator().manual_seed(7)
    pooled2 = torch.relu(torch.randn(pooled.shape, generator=g)).cuda()
    caps2 = caps.flip(0).contiguous()
    h02 = torch.rand(h0.shape, generator=g).cuda()
    eager = []
    for inp in ((pooled, caps, h0), (pooled2, caps2, h02)):
        loss = step(*inp)
        eager.append((loss.item(), grads()))
        del loss        # a live loss keeps the eager autograd graph (and its default-stream AccumulateGrad nodes) alive
    assert abs(eager[0][0] - c["tf/loss"].item()) < TOL_LOGITS * abs(c["tf/loss"].item())

    gstep = graphs.GraphedStep(step, (pooled, caps, h0), params=list(m.parameters()), release=m.release_graph)
    assert gstep.captured and gstep.launches_per_step > 10
    for rep in range(2):
        for inp, (l_ref, g_ref) in zip(((pooled, caps, h0), (pooled2, caps2, h02)), eager):
            loss = gstep(*inp)
            assert abs(loss.item() - l_ref) <= 1e-6 * abs(l_ref)
            got = grads()
            assert set(got) == set(g_ref)
            for k in g_ref:
                assert grad_close(got[k], g_ref[k], 1e-5), (mode, rep, k)
    m.zero_grad(set_to_none=True)          # a user dropping .grad between replays gets them back after the next call
    gstep(pooled, caps, h0)
    assert set(grads()) == set(eager[0][1])


@pytest.mark.parametrize("kind", ["gru", "lstm"])
def test_infer_projection_table_equals_per_step_path_at_bench_size(kind, monkeypatch):
    """B = 512, T = 20, V = 9684 (the size at which the table is chosen automatically): same greedy trajectories as the
    per-step path up to near-ties, probabilities within fp32 rounding."""
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import graphs, ops
    torch.manual_seed(0)
    with torch.device("cuda"):
        m = C.HyperNetPooled(64, 48, 9684, None, type=kind)
    g = torch.Generator().manual_seed(3)
    pooled = torch.relu(torch.randn(512, 2048, generator=g)).cuda()
    h0 = torch.rand(512, 48, generator=g).cuda()
    assert ops.use_projection_table(512, 20, 9684)
    outs = []
    for table in (False, True):
        monkeypatch.setattr(ops, "use_projection_table", lambda B, steps, V, table=table: table)
        graphs.clear()
        with torch.no_grad():
            cap = m.forward(m.captioner.embed.weight[4:5])
            outs.append(cap.infer(m.image_encoder(pooled), max_len=20, h0=h0 if kind == "gru" else None).clone())
    graphs.clear()
    # the per-step GEMM (M = 512) and the table GEMM (M = 9684) may take different kernels (exact-fp32 SIMT vs bf16x3
    # tensor cores, ~1e-6 apart): a random-init model has near-tied scores, so tokens are compared up to the first near-tie
    from golden_util import same_greedy_paths
    ok, why = same_greedy_paths(outs[0], outs[1])
    assert ok, why


def test_pooled_full_size_baseline_config1_matches_oracle():
    """BASELINE configs[1] at its FULL size -- E=200, H=150, V=9684, L=1, B=512, T=20, 1.62 G hypernet parameters -- on
    the kernels the benchmark times (weight-streaming heads, tcgen05 GEMMs, cluster GRU, fused decoder+CE node), against
    the oracle port on the same seeded inputs: logits and loss within 1e-4, gradients within 1e-3 (incl. the 4 GB head
    gradient, compared on the device), and the graphed step (graphs.GraphedStep) reproduces the eager loss."""
    from hypernet_image_captioning_b200 import graphs
    E, H, V, B, T = 200, 150, 9684, 512, 20
    p = O.init_params_pooled(2048, E, H, V, L=1, seed=5)
    g = torch.Generator().manual_seed(99)
    pooled = torch.relu(torch.randn(B, 2048, generator=g))
    caps = O.synth_captions(B, T, V, g)
    style = p["captioner.embed.weight"][4:5].clone()
    h0 = torch.rand(B, H, generator=g)
    import hypernet_image_captioning_b200 as C
    with torch.device("cuda"):                               # (initialising 1.6 G parameters on the CPU takes ~20 s)
        m = C.HyperNetPooled(E, H, V, None, num_layers=1)
    sd = m.state_dict()
    sd.update(p)
    m.load_state_dict(sd)
    del sd
    pl = {k: v.requires_grad_(True) for k, v in p.items()}
    del p
    logits_ref, _, _ = O.path_pooled(pl, style, pooled, caps, h0, L=1, flow=True)
    loss_ref = O.caption_loss(logits_ref, caps, None)
    loss_ref.backward()
    logits_ref = logits_ref.detach()
    pooled_d, caps_d, h0_d, style_d = pooled.cuda(), caps.cuda(), h0.cuda(), style.cuda()

    def step(pooled_, caps_, h0_):
        m.zero_grad(set_to_none=True)
        captioner = m.forward(style_d)
        loss, logits = captioner.forward_loss(m.image_encoder(pooled_), caps_, h0=h0_, ignore_index=None)
        loss.backward()
        return loss, logits

    loss, logits = step(pooled_d, caps_d, h0_d)
    assert rel_err(logits, logits_ref) < TOL_LOGITS
    assert abs(loss.item() - loss_ref.item()) < TOL_LOGITS * abs(loss_ref.item())
    worst = 0.0
    for k, v in m.named_parameters():
        if k.startswith("captioner.lstm_cell."):
            continue                                        # generated, not trained (flow mode)
        ref = pl[k].grad.cuda()                             # compared on the device: hn_heads.0.2.weight is 4 GB
        d = (v.grad - ref).abs().max().item()
        s = ref.abs().max().item()
        assert d <= 1e-7 or d <= TOL_GRAD * s, (k, d, s)
        worst = max(worst, d / s if s > 0 else 0.0)
        del ref
        pl[k].grad = None
    l_eager = loss.item()
    del loss, logits, pl, logits_ref
    m.zero_grad(set_to_none=True)
    torch.cuda.empty_cache()
    gstep = graphs.GraphedStep(step, (pooled_d, caps_d, h0_d), params=list(m.parameters()), release=m.release_graph)
    assert gstep.captured
    l_graph = gstep(pooled_d, caps_d, h0_d)[0].item()
    assert abs(l_graph - l_eager) <= 1e-6 * abs(l_eager)
    assert worst < TOL_GRAD
