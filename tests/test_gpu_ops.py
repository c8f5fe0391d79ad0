"""Kernel-level parity (through the C-ABI) against plain torch fp32/fp64 on the same seeded inputs."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from golden_util import rel_err


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


@pytest.mark.parametrize("G,N,K", [(1, 97, 13), (1, 450, 450), (2, 1000, 1125), (3, 301, 843), (1, 2000, 11250),
                                   (4, 64, 8437), (8, 600, 200), (5, 77, 6), (1, 5, 1)])
@pytest.mark.parametrize("act", [0, 1])
def test_rows_linear_fwd(G, N, K, act):
    ops = _ops()
    g = torch.Generator().manual_seed(G * 1000 + N + K)
    W = torch.randn(N, K, generator=g).cuda()
    b = torch.randn(N, generator=g).cuda()
    A = torch.randn(G, K, generator=g).cuda()
    Y = ops.rows_linear_fwd(W, b, A, act)
    ref = F.linear(A.double(), W.double(), b.double())
    if act:
        ref = F.leaky_relu(ref, 0.01)
    assert rel_err(Y, ref) < 2e-6


@pytest.mark.parametrize("G,N,K", [(1, 97, 13), (1, 450, 450), (2, 1000, 1125), (3, 301, 843), (1, 2000, 11250),
                                   (4, 64, 8437), (6, 600, 200), (5, 77, 6), (1, 5, 1), (1, 130, 4)])
@pytest.mark.parametrize("act", [0, 1])
def test_rows_linear_bwd(G, N, K, act):
    ops = _ops()
    g = torch.Generator().manual_seed(G * 1000 + N + K + 7)
    W = torch.randn(N, K, generator=g).double().requires_grad_(True)
    b = torch.randn(N, generator=g).double().requires_grad_(True)
    A = torch.randn(G, K, generator=g).double().requires_grad_(True)
    Yr = F.linear(A, W, b)
    if act:
        Yr = F.leaky_relu(Yr, 0.01)
    dY = torch.randn(G, N, generator=g).double()
    Yr.backward(dY)
    Wc, Ac = W.detach().float().cuda(), A.detach().float().cuda()
    Y = ops.rows_linear_fwd(Wc, b.detach().float().cuda(), Ac, act)
    dW, db, dA = ops.rows_linear_bwd(Wc, Ac, Y, dY.float().cuda(), act)
    assert rel_err(dW, W.grad) < 2e-6
    assert rel_err(db, b.grad) < 2e-6
    assert rel_err(dA, A.grad) < 1e-5


def test_rows_linear_strided_output_and_accumulate():
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    W = torch.randn(50, 37, generator=g).cuda()
    A = torch.randn(2, 37, generator=g).cuda()
    theta = torch.zeros(2, 120).cuda()
    ops.rows_linear_fwd(W, None, A, 0, out=theta[:, 30:80])
    assert rel_err(theta[:, 30:80], A @ W.t()) < 2e-6
    assert float(theta[:, :30].abs().max()) == 0 and float(theta[:, 80:].abs().max()) == 0
    dY = torch.randn(2, 120, generator=g).cuda()
    acc = torch.ones(2, 37).cuda()
    _, _, dA = ops.rows_linear_bwd(W, A, None, dY[:, 30:80], 0, dA=acc)
    assert rel_err(dA, 1 + dY[:, 30:80] @ W) < 1e-5


@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (130, 70, 33), (257, 129, 150), (1000, 450, 200), (64, 9684, 150)])
def test_gemm_variants(M, N, K):
    ops = _ops()
    g = torch.Generator().manual_seed(M + N + K)
    X = torch.randn(M, K, generator=g).cuda()
    W = torch.randn(N, K, generator=g).cuda()
    b = torch.randn(N, generator=g).cuda()
    ref = F.linear(X.double(), W.double(), b.double())
    # large shapes are routed to the tcgen05 bf16x3 kernel (~1e-5), small ones to the exact-fp32 CUDA-core kernel
    tol = 2e-5 if ops._tc_ok(M, N, K) else 2e-6
    assert rel_err(ops.linear(X, W, b), ref) < tol
    assert rel_err(ops.linear(X, W, b, relu=True), ref.relu()) < tol
    Bm = torch.randn(K, N, generator=g).cuda()
    assert rel_err(ops.matmul_nn(X, Bm), X.double() @ Bm.double()) < tol
    At = torch.randn(K, M, generator=g).cuda()
    assert rel_err(ops.matmul_tn(At, Bm), At.double().t() @ Bm.double()) < tol
    ops.TC_ENABLED = False
    try:
        assert rel_err(ops.linear(X, W, b), ref) < 2e-6
    finally:
        ops.TC_ENABLED = True


def test_gemm_splitk_and_colsum():
    ops = _ops()
    g = torch.Generator().manual_seed(11)
    A = torch.randn(5000, 45, generator=g).cuda()
    Bm = torch.randn(5000, 15, generator=g).cuda()
    assert rel_err(ops.matmul_tn(A, Bm), A.double().t() @ Bm.double()) < 1e-5
    assert rel_err(ops.colsum(A), A.double().sum(0)) < 1e-5


@pytest.mark.parametrize("B,T,H", [(3, 5, 6), (9, 4, 150), (4, 3, 33), (2, 2, 200)])
def test_gru_seq_fwd_bwd(B, T, H):
    """Recurrence kernel vs the oracle cell (oracle/caption_hn_oracle.py gru_cell) run step by step on the CPU."""
    from oracle import caption_hn_oracle as O
    ops = _ops()
    g = torch.Generator().manual_seed(B * 100 + T * 10 + H)
    GI = (torch.randn(T, B, 3 * H, generator=g) * 0.5).double().requires_grad_(True)
    W_hh = (torch.randn(3 * H, H, generator=g) / H ** 0.5).double().requires_grad_(True)
    b_hh = (torch.randn(3 * H, generator=g) * 0.1).double().requires_grad_(True)
    h0 = torch.rand(B, H, generator=g).double().requires_grad_(True)
    E = 3 * H  # trick: feed gi through an identity W_ih so the oracle cell sees it as x W_ih^T
    eye = torch.eye(E).double()
    h = h0
    hs = []
    for t in range(T):
        h = O.gru_cell(GI[t], h, eye, W_hh, torch.zeros(E).double(), b_hh)
        hs.append(h)
    Href = torch.stack(hs, 0)  # [T,B,H]
    dH = torch.randn(B, T, H, generator=g).double()
    (Href.permute(1, 0, 2) * dH).sum().backward()

    GIc = GI.detach().float().cuda().reshape(T * B, 3 * H).contiguous()
    Wc = W_hh.detach().float().cuda()
    WhhT = ops.transpose_pad(Wc, ops.round4(3 * H))
    Hall, Hbm, saved, _ = ops.gru_seq_fwd(GIc, WhhT, b_hh.detach().float().cuda(), h0.detach().float().cuda(), T)
    assert rel_err(Hall[1:], Href) < 5e-6
    assert rel_err(Hbm, Href.permute(1, 0, 2)) < 5e-6
    dGI, dGH, _, _, dh0 = ops.gru_seq_bwd(dH.float().cuda().contiguous(), saved, Hall, None, ops.copy_pad(Wc, ops.round4(H)))
    assert rel_err(dGI.view(T, B, 3 * H), GI.grad) < 2e-5
    assert rel_err(dh0, h0.grad) < 2e-5
    dW = ops.matmul_tn(dGH, Hall[:-1].reshape(T * B, H))
    assert rel_err(dW, W_hh.grad) < 2e-5
    assert rel_err(ops.colsum(dGH), b_hh.grad) < 2e-5


@pytest.mark.parametrize("M,V,ignore", [(7, 50, 0), (33, 9684, 0), (16, 9685, None), (5, 3, 0)])
def test_cross_entropy(M, V, ignore):
    import hypernet_image_captioning_b200 as C
    g = torch.Generator().manual_seed(M + V)
    x = (torch.randn(M, V, generator=g) * 3).double().requires_grad_(True)
    t = torch.randint(0, V, (M,), generator=g)
    t[::3] = 0
    ref = F.cross_entropy(x, t, ignore_index=ignore) if ignore is not None else F.cross_entropy(x, t)
    (ref * 1.7).backward()
    xc = x.detach().float().cuda().requires_grad_(True)
    loss = C.cross_entropy(xc, t.cuda(), ignore)
    (loss * 1.7).backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * abs(ref.item())
    assert rel_err(xc.grad, x.grad) < 1e-5


def test_softmax_argmax_ties_and_gather():
    ops = _ops()
    x = torch.zeros(4, 100).cuda()
    x[0, 7] = 1; x[0, 9] = 1          # tie -> lowest index
    x[1, 99] = 5
    x[2] = torch.randn(100).cuda()
    probs, am = ops.softmax_argmax(x)
    assert am.tolist()[:2] == [7, 99] and am[2].item() == x[2].argmax().item() and am[3].item() == 0
    assert rel_err(probs, torch.softmax(x.double(), 1)) < 2e-6
    table = torch.randn(10, 6).cuda()
    idx = torch.tensor([3, 0, 9]).cuda()
    assert torch.equal(ops.gather_rows(table, idx), table[idx])


@pytest.mark.parametrize("V", [9684, 10240, 10244, 101, 4])
def test_softmax_argmax_vector_and_generic_paths(V):
    """V % 4 == 0 and V <= 10240 takes the register-resident 128-bit kernel, anything else the generic one; strided
    output rows (probs written into outputs[:, t, :]) and ties across threads / vector lanes (lowest index wins)."""
    ops = _ops()
    g = torch.Generator().manual_seed(V)
    M, T = 37, 3
    x = torch.randn(M, V, generator=g).cuda()
    x[0, V - 1] = 9.0; x[0, V // 2] = 9.0          # tie far apart
    x[1, 2 % V] = 9.0; x[1, 3 % V] = 9.0           # tie inside one 128-bit vector
    x[2] = 0.0                                     # all equal -> index 0
    out = torch.zeros(M, T, V).cuda()
    probs, am = ops.softmax_argmax(x, want_probs=True, probs_out=out[:, 1, :])
    ref = torch.softmax(x.double(), 1)
    assert torch.equal(am.cpu(), x.cpu().argmax(1)) and am[0].item() == V // 2 and am[2].item() == 0
    assert rel_err(out[:, 1, :], ref) < 2e-6 and float(out[:, 0].abs().max()) == 0.0 and float(out[:, 2].abs().max()) == 0.0
    _, am2 = ops.softmax_argmax(x, want_probs=False)
    assert torch.equal(am2, am)
    # non-finite rows: the selection contract (NaN counts as -inf, lowest index on ties; all NaN / all -inf -> 0)
    from test_gpu_decode_select import greedy_token
    nan, inf = float("nan"), float("inf")
    y = x.clone()
    y[0] = nan
    y[1] = -inf; y[1, 0] = nan                       # [NaN, -inf, -inf, ...]
    y[2] = -inf
    y[3, V // 3] = inf; y[3, V - 1] = inf            # tied +inf
    y[4, ::3] = nan; y[4, V - 1] = 20.0              # NaN everywhere but a finite maximum
    y[5] = -inf; y[5, 1 % V] = nan; y[5, V - 1] = nan
    y[6, 0] = nan
    _, am3 = ops.softmax_argmax(y, want_probs=True)
    _, am4 = ops.softmax_argmax(y, want_probs=False)
    want = greedy_token(y.cpu())
    assert torch.equal(am3.cpu(), want) and torch.equal(am4.cpu(), want)
    assert am3[:3].tolist() == [0, 0, 0] and am3[3].item() == V // 3 and am3[4].item() == V - 1


@pytest.mark.parametrize("B,T,H", [(3, 5, 6), (9, 4, 150), (21, 3, 33), (16, 6, 200), (5, 2, 301)])
def test_gru_cluster_matches_streaming_kernel(B, T, H):
    """Weights-resident cluster kernels (W_hh in shared memory, DSMEM state exchange) == L2-streaming kernels."""
    ops = _ops()
    assert ops.gru_cluster_size(H) in (2, 4, 8)
    g = torch.Generator().manual_seed(B * 100 + T * 10 + H)
    GI = (torch.randn(T * B, 3 * H, generator=g) * 0.5).cuda()
    W = (torch.randn(3 * H, H, generator=g) / H ** 0.5).cuda()
    b = (torch.randn(3 * H, generator=g) * 0.1).cuda()
    h0 = torch.rand(B, H, generator=g).cuda()
    dH = torch.randn(B, T, H, generator=g).cuda()
    Hall0, Hbm0, sv0, _ = ops.gru_seq_fwd(GI, ops.transpose_pad(W, ops.round4(3 * H)), b, h0, T)
    dGI0, dGH0, _, _, dh00 = ops.gru_seq_bwd(dH, sv0, Hall0, None, ops.copy_pad(W, ops.round4(H)))
    Hall1, Hbm1, sv1, _ = ops.gru_cluster_fwd(GI, W, b, h0, T)
    dGI1, dGH1, _, _, dh01 = ops.gru_cluster_bwd(dH, sv1, Hall1, W)
    assert rel_err(Hall1, Hall0) < 2e-6 and rel_err(Hbm1, Hbm0) < 2e-6 and rel_err(sv1, sv0) < 2e-6
    assert rel_err(dGI1, dGI0) < 1e-5 and rel_err(dGH1, dGH0) < 1e-5 and rel_err(dh01, dh00) < 1e-5


@pytest.mark.parametrize("M,V,ignore", [(1300, 9684, 0), (1300, 9684, None), (257, 1502, 0), (130, 9685, 0)])
def test_ce_forward_with_gradient_operand_in_one_pass(M, V, ignore):
    """caphn_ce_fwd_split (loss + UNSCALED gradient operand from one read of the logits) followed by the scaled products
    (caphn_gemm_tc_scaled: grad_output / #valid rows applied in the epilogue, bias gradient as the ones column) ==
    torch's cross_entropy backward through the vocabulary projection, F.cross_entropy at cc_train_hypernet.py:153."""
    import torch
    import torch.nn.functional as F
    from hypernet_image_captioning_b200 import functional as Fn
    from hypernet_image_captioning_b200 import ops
    g = torch.Generator().manual_seed(1)
    H = 150
    logits = (torch.randn(M, V, generator=g) * 2.0).cuda()
    Hbm = torch.randn(M, H, generator=g).cuda()
    fc_w = (torch.randn(V, H, generator=g) * 0.2).cuda()
    tgt = torch.randint(0, V, (M,), generator=g).cuda()
    if ignore is not None:
        tgt[::5] = ignore
    gscale = torch.tensor([0.37], device="cuda")
    # the separate passes
    lb_ref, lse_ref = ops.ce_fwd(logits, tgt, ignore)
    lb, lse, hi, lo = Fn.ce_fwd_for_loss(logits, tgt, ignore, H, True)
    assert hi is not None, "the one-pass kernel must be selected at this size"
    assert torch.equal(lse, lse_ref) or (lse - lse_ref).abs().max().item() < 2e-6 * lse_ref.abs().max().item()
    assert abs(lb[0].item() - lb_ref[0].item()) < 1e-6 * abs(lb_ref[0].item()) and lb[1].item() == lb_ref[1].item()
    # the operand is softmax - onehot (0 on ignored rows), hi + lo to 2^-16
    u = torch.softmax(logits.double(), dim=1)
    u[torch.arange(M), tgt] -= 1.0
    if ignore is not None:
        u[tgt == ignore] = 0.0
    got = hi[:, :V].double() + lo[:, :V].double()
    assert (got - u).abs().max().item() < 3e-5
    assert hi[:, V:].abs().max().item() == 0 if hi.shape[1] > V else True
    # gradients of gscale * mean CE through logits = Hbm fc_w^T
    Hd, Wd = Hbm.double().requires_grad_(True), fc_w.double().requires_grad_(True)
    bd = torch.zeros(V, device="cuda", dtype=torch.double, requires_grad=True)
    ld = logits.double().requires_grad_(True)
    loss = F.cross_entropy(ld, tgt, ignore_index=-100 if ignore is None else ignore)
    (dl,) = torch.autograd.grad(loss * 0.37, ld)
    dfc_w, dfc_b, dHbm = Fn.vocab_bwd_fused(logits, tgt, ignore, lse, lb, gscale, Hbm, fc_w, hi, lo)
    ref_dH, ref_dW, ref_db = dl @ fc_w.double(), dl.t() @ Hbm.double(), dl.sum(0)
    for got_t, ref_t in ((dHbm, ref_dH), (dfc_w, ref_dW), (dfc_b, ref_db)):
        assert got_t.shape == ref_t.shape and got_t.is_contiguous()
        assert (got_t.double() - ref_t).abs().max().item() < 3e-5 * ref_t.abs().max().item()
    # and it agrees with the two-pass path (ce_fwd + ce_bwd_split + unscaled products)
    dfc_w2, dfc_b2, dHbm2 = Fn.vocab_bwd_fused(logits, tgt, ignore, lse_ref, lb_ref, gscale, Hbm, fc_w)
    for a, b in ((dHbm, dHbm2), (dfc_w, dfc_w2), (dfc_b, dfc_b2)):
        assert (a - b).abs().max().item() < 3e-5 * b.abs().max().item()


@pytest.mark.parametrize("M,N,K", [(10240, 9684, 150), (4096, 9684, 200), (2048, 1100, 64), (5000, 777, 130)])
def test_gemm_tc_a_stationary_schedule_is_bit_identical(M, N, K, monkeypatch):
    """The A-stationary schedule of the tensor-core GEMM (A slab resident per m-tile, contiguous tile runs per CTA; the
    vocabulary projection) only reorders tiles: bit-identical to the round-robin schedule, bias / ragged N / ragged K
    included (CAPHN_TC_ASTAT=0 switches it off)."""
    import torch
    from hypernet_image_captioning_b200 import ops
    g = torch.Generator().manual_seed(2)
    X = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(N, K, generator=g) * 0.3).cuda()
    b = torch.randn(N, generator=g).cuda()
    outs = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("CAPHN_TC_ASTAT", mode)
        outs[mode] = ops.linear(X, W, b).clone()
    ref = X.double() @ W.double().t() + b.double()
    assert (outs["0"].double() - ref).abs().max().item() < 2e-5 * ref.abs().max().item()
    assert torch.equal(outs["0"], outs["1"])


@pytest.mark.parametrize("B,H,V", [(512, 150, 9684), (37, 34, 301), (16, 200, 1000), (5, 6, 40), (300, 256, 500),
                                   (64, 32, 16384)])
def test_fused_decode_step_matches_the_three_launch_chain(B, H, V):
    """caphn_gru_decode_step (arg-max finish + projection-table gather + GRU cell + bf16 operand rows in one launch) ==
    argmax_finish_gather -> gru_seq_fwd(T = 1) -> split_bf16, the chain it replaces in DecoderGRU.infer (later.py:459-490).
    V = 40: one partial slot; V = 16384: all 256 slots the kernel holds, the winner in the last lane's last register.
    Both also take rows of empty (-inf, no column) and NaN partials, whose token is 0."""
    import torch
    from hypernet_image_captioning_b200 import ops
    g = torch.Generator().manual_seed(3)
    nslot, nparts = 2 * ((V + 127) // 128), 2 * ((V + 127) // 128) - 1
    table = torch.randn(V, 3 * H, generator=g).cuda()
    W_hh = (torch.randn(3 * H, H, generator=g) * 0.2).cuda()
    b_hh = torch.randn(3 * H, generator=g).cuda()
    h = torch.rand(B, H, generator=g).cuda()
    pv = torch.randn(B, nslot, generator=g).cuda()
    pi = torch.randint(0, V, (B, nslot), generator=g, dtype=torch.int32).cuda()
    pv[::3, nparts - 1] = pv[::3, 0] = 9.0              # ties: the lower column must win
    WhhT = ops.transpose_pad(W_hh, ops.round4(3 * H))
    # reference chain
    GI = torch.empty(B, 3 * H, device="cuda")
    tok_ref = torch.empty(B, device="cuda", dtype=torch.int64)
    ops.argmax_finish_gather(pv, pi, nparts, table, tok_ref, GI)
    h_ref = ops.gru_seq_fwd(GI, WhhT, b_hh, h, 1, save=False, want_bm=False)[0][1]
    sp = ops.split_bf16(h_ref)
    # fused
    Kp = ops.round64(H)
    hn = torch.empty(B, H, device="cuda")
    hi = torch.zeros(B, Kp, device="cuda", dtype=torch.bfloat16)
    lo = torch.zeros(B, Kp, device="cuda", dtype=torch.bfloat16)
    tok = torch.empty(B, device="cuda", dtype=torch.int64)
    ops.gru_decode_step(None, pv, pi, nparts, table, W_hh, b_hh, h, hn, hi, lo, tok)
    assert torch.equal(tok, tok_ref)
    assert (hn - h_ref).abs().max().item() < 2e-6
    assert (hi[:, :H].float() + lo[:, :H].float() - hn).abs().max().item() < 1e-5 * max(1.0, hn.abs().max().item())
    assert torch.equal(hi[:, :H], hn.to(torch.bfloat16))
    # step 0: the input projection is given
    hn0 = torch.empty(B, H, device="cuda")
    ops.gru_decode_step(GI, None, None, 0, None, W_hh, b_hh, h, hn0)
    assert (hn0 - h_ref).abs().max().item() < 2e-6
    del sp
    # every slot in use, the winner in the last one; empty and NaN rows
    from test_gpu_decode_select import NONE, finish_partials
    pv[1::4, nslot - 1] = 50.0
    pv[2::5], pi[2::5] = float("-inf"), NONE
    pv[3::7] = float("nan")
    tok_ref2 = torch.empty(B, device="cuda", dtype=torch.int64)
    ops.argmax_finish_gather(pv, pi, nslot, table, tok_ref2, GI)
    want = finish_partials(pv, pi, nslot)
    assert torch.equal(tok_ref2.cpu(), want)
    assert bool((want[2::5] == 0).all()) and bool((want[3::7] == 0).all())
    h_ref2 = ops.gru_seq_fwd(GI, WhhT, b_hh, h, 1, save=False, want_bm=False)[0][1]
    ops.gru_decode_step(None, pv, pi, nslot, table, W_hh, b_hh, h, hn, hi, lo, tok)
    assert torch.equal(tok, tok_ref2)
    assert (hn - h_ref2).abs().max().item() < 2e-6


@pytest.mark.parametrize("B,T,H", [(3, 5, 6), (9, 4, 150), (21, 3, 33), (16, 6, 160), (512, 20, 150), (6, 2, 100)])
def test_gru_resident_matches_streaming_kernel(B, T, H):
    """CTA-resident W_hh (csrc/gru_resident.cu: shared memory + registers, no cluster) == the L2-streaming recurrence
    (gru_seq.cu), forward outputs / saved gates and the BPTT gradients (nn.GRUCell + autograd, later.py:411,418)."""
    import torch
    from hypernet_image_captioning_b200 import ops
    from golden_util import rel_err
    if not ops.gru_resident_ok(H):
        pytest.skip("hidden size outside the resident kernels' range")
    g = torch.Generator().manual_seed(5)
    GI = torch.randn(T * B, 3 * H, generator=g).cuda()
    W = (torch.randn(3 * H, H, generator=g) * 0.2).cuda()
    b = torch.randn(3 * H, generator=g).cuda()
    h0 = torch.rand(B, H, generator=g).cuda()
    dH = torch.randn(B, T, H, generator=g).cuda()
    Hall0, Hbm0, sv0, _ = ops.gru_seq_fwd(GI, ops.transpose_pad(W, ops.round4(3 * H)), b, h0, T)
    dGI0, dGH0, _, _, dh00 = ops.gru_seq_bwd(dH, sv0, Hall0, None, ops.copy_pad(W, ops.round4(H)))
    Hall1, Hbm1, sv1, _ = ops.gru_resident_fwd(GI, W, b, h0, T)
    dGI1, dGH1, _, _, dh01 = ops.gru_resident_bwd(dH, sv1, Hall1, W)
    assert rel_err(Hall1, Hall0) < 2e-6 and rel_err(Hbm1, Hbm0) < 2e-6 and rel_err(sv1, sv0) < 2e-6
    assert rel_err(dGI1, dGI0) < 1e-5 and rel_err(dGH1, dGH0) < 1e-5 and rel_err(dh01, dh00) < 1e-5
    # inference form (no saved gates, no batch-major copy)
    Hall2, Hbm2, sv2, _ = ops.gru_resident_fwd(GI, W, b, h0, T, save=False, want_bm=False)
    assert Hbm2 is None and sv2 is None and torch.equal(Hall2, Hall1)
