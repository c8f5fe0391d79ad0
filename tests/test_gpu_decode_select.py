"""Decode token selection against exact references: the arg-max partials of the vocabulary GEMM's epilogue
(caphn_gemm_tc_amax), the finisher that turns them into tokens (caphn_argmax_finish_gather), one beam-search step
(caphn_beam_step) output by output, and the decoders that use them at the edges where selection goes wrong: exact ties
across epilogue warps and tiles, a last tile with one valid column, non-finite logits, vocabularies above 16384.

The selection contract (DESIGN.md §6) is `greedy_token` below.  The tests that only read tokens come first; the ones
that use a token as an address (table gathers, beam bookkeeping, whole decoders) follow."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from golden_util import rel_err, same_greedy_paths
from oracle import caption_hn_oracle as O

NONE = 0x7fffffff          # column of an arg-max partial that saw no candidate


def greedy_token(x):
    """The greedy token of every row of x [..., V]: torch.argmax with NaN counted as -inf, ties to the lowest index.
    (torch.argmax alone returns the first NaN; an all-NaN or all -inf row gives 0.)"""
    return torch.argmax(torch.where(x.isnan(), float("-inf"), x), dim=-1)


def finish_partials(pv, pi, nparts):
    """Token of every row from (value, column) partials [n, >= nparts]: the largest non-NaN value, the lowest column
    among its slots, and 0 where no slot names a column."""
    v, c = pv[:, :nparts].double().cpu(), pi[:, :nparts].long().cpu()
    best = torch.where(v.isnan(), float("-inf"), v).amax(1, keepdim=True)
    tok = torch.where(v == best, c, NONE).amin(1)
    return torch.where(tok == NONE, 0, tok)


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


def _bits(x):
    return x.contiguous().view(torch.int32)


def _tc_bn(M, N, K, split, astat=True):
    """N tile of the tensor-core GEMM for K-major operands (gemm_tc.cu, gemm_tc_impl): one tile for N <= 256; with few
    waves the width of 128..256 that minimises waves x (BN + 32); with many, 128 if the A-stationary schedule fits, else 256."""
    cdiv = lambda a, b: -(-a // b)
    if N <= 256:
        return cdiv(N, 16) * 16
    tm = cdiv(M, 128)
    if tm * cdiv(N, 128) <= 8 * 148:
        return min(range(128, 257, 16), key=lambda bn: (cdiv(tm * cdiv(N, bn), 148) * (bn + 32), bn))
    w = 2 if split else 1
    fits = cdiv(K, 64) * w * 16384 + (32768 + 18 * 8 + 16 + 1024) + 3 * w * 16384 <= 227 * 1024
    return 128 if astat and fits else 256


# ----------------------------------------------------------------------------------------------------------------------
# caphn_gemm_tc_amax: logits and arg-max partials  (reads tokens only)
# ----------------------------------------------------------------------------------------------------------------------
def _planted_case(M, N, K, split, seed):
    """A [M, K], W [N, K], bias [N] with exact ties planted: rows of W and bias entries equal at two columns, and a row of
    A along that W row so the pair is the row's maximum by a wide margin.  Pairs: the two epilogue warp halves (31, 32),
    adjacent tiles (BN - 1, BN), (0, N - 1), three tiles apart.  Row 2 of A is zero (logits = bias) and row M - 1 is NaN."""
    g = torch.Generator().manual_seed(seed)
    A = torch.randn(M, K, generator=g) / K ** 0.5
    W = torch.randn(N, K, generator=g)
    b = torch.randn(N, generator=g)
    bn = _tc_bn(M, N, K, split)
    used, planted = set(), []
    for j, (c1, c2) in enumerate([(31, 32), (bn - 1, bn), (0, N - 1), (5, 5 + 3 * bn)]):
        if c2 >= N or c1 in used or c2 in used:
            continue
        used |= {c1, c2}
        w = torch.randn(K, generator=g)
        W[c1] = W[c2] = w
        b[c2] = b[c1]
        r = 1 + 41 * j
        A[r] = 4.0 * w / w.norm()
        planted.append((r, c1, c2))
    A[2] = 0.0
    A[M - 1] = float("nan")
    return A, W, b, planted


def _bias_variants(b, N, bn):
    inf = float("inf")
    nan_cols = b.clone()
    nan_cols[[1, N // 2, N - 1]] = float("nan")
    few = torch.full_like(b, -inf)                   # all but a few columns -inf (column 0 among the -inf ones)
    keep = sorted({c for c in (N - 1, 31, 32, bn - 1, bn, 7) if 0 < c < N})
    few[keep] = b[keep]
    posinf = b.clone()
    posinf[N // 3] = inf
    return {"finite": b, "const": torch.full_like(b, 0.25), "nan_cols": nan_cols, "few_finite": few, "posinf": posinf,
            "all_neginf": torch.full_like(b, -inf)}


def _amax_run(ops, xs, ws, bias, M, N):
    ld = 2 * ((N + 127) // 128) + 3
    pv = torch.full((M + 3, ld), 12345.0, device="cuda")
    pi = torch.full((M + 3, ld), -77, device="cuda", dtype=torch.int32)
    lg = torch.empty(M, N, device="cuda")
    nparts = ops.gemm_tc_amax(xs, ws, bias, lg, pv, pi)
    tok = torch.empty(M, device="cuda", dtype=torch.int64)
    ops.argmax_finish_gather(pv[:M], pi[:M], nparts, tok=tok)
    torch.cuda.synchronize()
    return lg, pv, pi, nparts, tok


AMAX_POINTS = [  # M, N, K, bf16x3 operands
    (128, 16, 64, True), (129, 32, 150, True), (128, 33, 200, False), (512, 200, 150, True), (129, 256, 64, False),
    (512, 257, 200, True), (2048, 1000, 150, True), (4096, 1000, 64, True), (512, 9684, 150, True),
    (512, 9684, 200, True), (512, 9684, 150, False), (4096, 9684, 150, True), (4096, 9684, 200, True),
    (2048, 9685, 64, True), (128, 16384, 150, True), (128, 16385, 150, True), (129, 16385, 64, False),
    (512, 20000, 150, True), (4096, 20000, 200, False), (2048, 257, 150, False)]


@pytest.mark.parametrize("M,N,K,split", AMAX_POINTS)
def test_gemm_tc_amax_partials_give_the_contract_token(M, N, K, split):
    """For every bias variant: the logits the arg-max GEMM writes are bit-identical to the plain GEMM's (both add bias to
    the same fp32 accumulator once) and match fp64; nparts = 2 ceil(N / BN); no partial slot outside [M, nparts) is
    written; and the finished token of EVERY row is the contract's token of the written logits, exactly."""
    ops = _ops()
    A, W, b, planted = _planted_case(M, N, K, split, seed=M + N + K)
    Ad, Wd = A.cuda(), W.cuda()
    xs, ws = ops.split_bf16(Ad, want_lo=split), ops.split_bf16(Wd, want_lo=split)
    bn = _tc_bn(M, N, K, split)
    for name, bias in _bias_variants(b, N, bn).items():
        bias = bias.cuda()
        lg, pv, pi, nparts, tok = _amax_run(ops, xs, ws, bias, M, N)
        assert nparts == 2 * math.ceil(N / bn) and nparts <= pv.shape[1], (name, nparts, bn)
        ref = ops.gemm_tc(xs, ws, bias=bias, splitk=1)
        assert torch.equal(_bits(lg), _bits(ref)), name
        assert bool((pv[M:] == 12345.0).all()) and bool((pi[M:] == -77).all()), name
        assert bool((pv[:, nparts:] == 12345.0).all()) and bool((pi[:, nparts:] == -77).all()), name
        lg_h = lg.cpu()
        want = greedy_token(lg_h)
        assert torch.equal(tok.cpu(), want), (name, (tok.cpu() != want).nonzero()[:5].flatten().tolist())
        if name == "finite":
            ref64 = Ad[:M - 1].double() @ Wd.double().t() + bias.double()
            assert rel_err(lg[:M - 1], ref64) < (2e-5 if split else 2e-2)
            assert bool(lg_h[M - 1].isnan().all()) and int(tok[M - 1]) == 0
            for r, c1, c2 in planted:           # the planted ties are exact and are the row maximum
                assert lg_h[r, c1] == lg_h[r, c2] == lg_h[r].max(), (r, c1, c2)
                assert int(tok[r]) == c1
        if name == "all_neginf":
            assert bool((tok == 0).all())


@pytest.mark.parametrize("knob,values,M", [("CAPHN_TC_BN_FORCE", [None, "128", "144", "256"], 512),
                                           ("CAPHN_TC_ASTAT", ["0", "1"], 4096)])
def test_gemm_tc_amax_tokens_do_not_depend_on_the_tile_schedule(knob, values, M, monkeypatch):
    """N tile widths (128 / 144 / 256 at the decode shape 512 x 9684 x 150) and the A-stationary schedule on / off
    (4096 x 9684 x 150; off means BN = 256) only regroup the same products: identical tokens, bit-identical logits."""
    ops = _ops()
    N, K = 9684, 150
    A, W, b, _ = _planted_case(M, N, K, True, seed=7)
    xs, ws = ops.split_bf16(A.cuda()), ops.split_bf16(W.cuda())
    bias = b.cuda()
    outs = []
    for v in values:
        if v is None:
            monkeypatch.delenv(knob, raising=False)
        else:
            monkeypatch.setenv(knob, v)
        lg, _, _, nparts, tok = _amax_run(ops, xs, ws, bias, M, N)
        bn = int(v) if knob == "CAPHN_TC_BN_FORCE" and v else _tc_bn(M, N, K, True, astat=v != "0")
        assert nparts == 2 * math.ceil(N / bn), (v, nparts)
        assert torch.equal(tok.cpu(), greedy_token(lg.cpu()))
        outs.append((lg, tok))
    for lg, tok in outs[1:]:
        assert torch.equal(_bits(lg), _bits(outs[0][0])) and torch.equal(tok, outs[0][1])


# ----------------------------------------------------------------------------------------------------------------------
# caphn_argmax_finish_gather on hand-built partials
# ----------------------------------------------------------------------------------------------------------------------
def _hand_partials(nparts, n=40, V=5000, seed=0):
    """[n, nparts + 5] partials (the 5 extra slots hold a value that would win if read).  Row plants: the winner in
    slot 0; in the last slot; a tie won by a slot of a later lane holding a lower column; one real slot among empty
    (-inf, no column) ones; all empty; all NaN; NaN in every third slot; all values equal; +inf in two slots."""
    g = torch.Generator().manual_seed(seed + nparts)
    ld = nparts + 5
    pv = torch.randn(n, ld, generator=g)
    pi = torch.randint(0, V, (n, ld), generator=g, dtype=torch.int32)
    pv[:, nparts:] = 1e30
    pi[:, nparts:] = 1
    last = nparts - 1
    pv[0, 0] = 50.0
    pv[1, last] = 50.0
    a, c = 0, min(last, 37)
    pv[2, a] = pv[2, c] = 50.0
    pi[2, a], pi[2, c] = 4000, 17
    pv[3, :nparts], pi[3, :nparts] = float("-inf"), NONE
    pv[3, nparts // 2], pi[3, nparts // 2] = 0.5, 123
    pv[4, :nparts], pi[4, :nparts] = float("-inf"), NONE
    pv[5, :nparts] = float("nan")
    pv[6, :nparts:3] = float("nan")
    pv[7, :nparts] = 1.0
    pv[8, last] = float("inf")
    pv[8, last // 2] = float("inf")
    return pv.cuda(), pi.cuda()


@pytest.mark.parametrize("nparts", [1, 31, 32, 33, 255, 256, 257, 600])
def test_argmax_finish_from_hand_built_partials(nparts):
    ops = _ops()
    pv, pi = _hand_partials(nparts)
    tok = torch.full((pv.shape[0],), -1, device="cuda", dtype=torch.int64)
    ops.argmax_finish_gather(pv, pi, nparts, tok=tok)
    want = finish_partials(pv, pi, nparts)
    assert torch.equal(tok.cpu(), want)
    assert int(tok[4]) == 0 and int(tok[5]) == 0 and int(tok[3]) == 123
    assert bool(((tok >= 0) & (tok < 5000)).all())


# ---- from here on a token is used as an address -----------------------------------------------------------------------
@pytest.mark.parametrize("nparts", [1, 32, 257, 600])
def test_argmax_finish_gather_copies_the_selected_table_row(nparts):
    ops = _ops()
    pv, pi = _hand_partials(nparts)
    n, E = pv.shape[0], 37
    table = torch.randn(5000, E, device="cuda")
    buf = torch.full((n, E + 9), -3.0, device="cuda")
    out = buf[:, 4:4 + E]
    tok = torch.empty(n, device="cuda", dtype=torch.int64)
    ops.argmax_finish_gather(pv, pi, nparts, table, tok, out)
    assert torch.equal(tok.cpu(), finish_partials(pv, pi, nparts))
    assert torch.equal(out, table[tok])
    assert bool((buf[:, :4] == -3.0).all()) and bool((buf[:, 4 + E:] == -3.0).all())


# ----------------------------------------------------------------------------------------------------------------------
# caphn_beam_step, one call at a time, against a float64 restatement
# ----------------------------------------------------------------------------------------------------------------------
BEAM_OUT = ("h_next", "scores", "live", "prev_tok", "words", "seq_out", "comp_score", "comp_seq", "comp_len", "ncomp",
            "failed")


def beam_step_ref(t, k, V, L, step, end_tok, last):
    """One call of beam_step_kernel (csrc/beam.cu), which restates hypernet_attention.py:268-312 for B images at once
    (oracle.attention_beam_search is the whole loop for one image), with candidate scores in float64.  Returns the
    output tensors; entries the kernel must not write keep their input values."""
    o = {name: t[name].clone() for name in BEAM_OUT}
    B = t["live"].numel()
    for b in range(B):
        n, r0 = int(t["live"][b]), b * k
        if n == 0:
            o["words"][r0:r0 + k] = -1
            continue
        S, I = [], []
        for r in range(1 if step == 1 else n):            # step 1 ranks row 0 only
            x = t["logits"][r0 + r].double()
            lse = torch.logsumexp(x, 0)
            if not bool(torch.isfinite(lse)):             # a NaN / +inf logit, or all -inf: no candidates
                continue
            S.append(t["scores"][r0 + r].double() + (x - lse))
            I.append(torch.arange(V) + r * V)
        s = torch.cat(S) if S else torch.empty(0, dtype=torch.float64)
        idx = torch.cat(I) if I else torch.empty(0, dtype=torch.int64)
        keep = ~s.isnan()
        s, idx = s[keep], idx[keep]
        order = torch.sort(s, descending=True, stable=True).indices    # equal scores: lower flat index first
        s, idx = s[order], idx[order]
        if s.numel() < n:
            o["live"][b], o["failed"][b] = 0, 1
            o["words"][r0:r0 + k] = -1
            continue
        top = s[:n + 1]
        gaps = top[:-1] - top[1:]
        assert bool(((gaps == 0) | (gaps >= 1e-3)).all()), f"image {b}: candidates closer than 1e-3 (test precondition)"
        ln, nc, surv = step, int(t["ncomp"][b]), []
        for j in range(n):
            parent, word = divmod(int(idx[j]), V)
            if word != end_tok:
                surv.append((parent, word, float(s[j])))
                continue
            c = r0 + nc
            o["comp_score"][c] = float(s[j])
            m = min(ln, L)
            o["comp_seq"][c, :m] = t["seq_in"][r0 + parent, :m]
            if ln < L:
                o["comp_seq"][c, ln] = word
            o["comp_len"][c] = min(ln + 1, L)
            nc += 1
        o["ncomp"][b], o["live"][b] = nc, len(surv)
        zero = len(surv) > 0 and surv[0][1] == 0         # :265-266: every embedding zeroed when row 0's word is 0
        if last and surv:
            o["failed"][b] = 1
        for j in range(k):
            if j < len(surv):
                parent, word, sc = surv[j]
                o["scores"][r0 + j] = sc
                o["prev_tok"][r0 + j] = word
                o["words"][r0 + j] = -1 if zero else word
                row = torch.zeros(L, dtype=torch.int32)
                row[:min(ln, L)] = t["seq_in"][r0 + parent, :min(ln, L)]
                if ln < L:
                    row[ln] = word
                o["seq_out"][r0 + j] = row
                o["h_next"][r0 + j] = t["h_out"][r0 + parent]
            else:
                o["words"][r0 + j] = -1
    return o


def beam_step_gpu(t, k, V, L, step, end_tok, last):
    ops = _ops()
    d = {name: x.cuda() for name, x in t.items()}
    ops.beam_step(*[d[n] for n in (
        "logits", "h_out", "h_next", "scores", "live", "prev_tok", "words", "seq_in", "seq_out", "comp_score", "comp_seq",
        "comp_len", "ncomp", "failed")], k, step, end_tok, last)
    torch.cuda.synchronize()
    return {name: d[name].cpu() for name in BEAM_OUT}


def _beam_inputs(kinds, k, V, L, step, seed, H=5):
    """One image per entry of `kinds`.  Every row's logits are a random permutation of 0, 0.05, 0.1, ...; its running
    score is set so that score - lse takes a per-row offset, the offsets of one image 0.0731 apart (0.0061 for
    "all_eos"), so that any two candidates differ by >= 3.8e-3 unless planted equal.  Rows the kernel must not rank carry a
    running score that would win.  kinds: "full" (k live), "fewer" (k - 2 live), "empty" (0 live), "eos" (the best
    candidate is the end token), "all_eos" (every pick is an end token), "zero" (the best candidate is word 0), "tie"
    (rows 0 and 1 identical, equal running scores)."""
    g = torch.Generator().manual_seed(seed)
    B, R, end_tok = len(kinds), len(kinds) * k, 2
    logits = torch.empty(R, V)
    scores = torch.full((R,), 5.0)
    live = torch.zeros(B, dtype=torch.int32)
    for b, kind in enumerate(kinds):
        n = {"empty": 0, "fewer": max(1, k - 2), "all_eos": k if step > 1 else 1}.get(kind, k)
        live[b] = n
        ranked = 1 if step == 1 else n
        for j in range(k):
            x = torch.randperm(V, generator=g).double() * 0.05
            r = b * k + j
            top = int(x.argmax())
            if (kind in ("eos", "all_eos") and j == 0) or (kind == "all_eos" and j < ranked):
                x[[top, end_tok]] = x[[end_tok, top]]
            if kind == "zero" and j == 0:
                x[[top, 0]] = x[[0, top]]
            if kind == "tie" and j == 1 and ranked >= 2:
                x = logits[r - 1].double()
            logits[r] = x.float()
            if j < ranked:
                off = -1.0 - j * (0.0061 if kind == "all_eos" else 0.0731)
                if kind == "tie" and j == 1 and ranked >= 2:
                    scores[r] = scores[r - 1]
                else:
                    scores[r] = float(off + torch.logsumexp(logits[r].double(), 0))
    ncomp = (k - live).to(torch.int32)
    seq_in = torch.randint(0, V, (R, L), generator=g, dtype=torch.int32)
    seq_in[:, 0] = 0
    t = {"logits": logits, "h_out": torch.randn(R, H, generator=g), "h_next": torch.full((R, H), 7.5), "scores": scores,
         "live": live, "prev_tok": torch.full((R,), -5, dtype=torch.int32), "words": torch.full((R,), 99),
         "seq_in": seq_in, "seq_out": torch.full((R, L), -6, dtype=torch.int32), "comp_score": torch.full((R,), -9.5),
         "comp_seq": torch.full((R, L), -4, dtype=torch.int32), "comp_len": torch.full((R,), -3, dtype=torch.int32),
         "ncomp": ncomp, "failed": torch.zeros(B, dtype=torch.int32)}
    return t, end_tok


def _assert_beam_equal(got, want, where):
    for name in ("live", "prev_tok", "words", "seq_out", "comp_seq", "comp_len", "ncomp", "failed", "h_next"):
        assert torch.equal(got[name], want[name]), (where, name, got[name], want[name])
    for name in ("scores", "comp_score"):
        assert torch.allclose(got[name].double(), want[name].double(), rtol=1e-6, atol=0.0), (where, name)


BEAM_KV = [(k, V) for k in (1, 2, 3, 5, 8) for V in (7, 100, 9684) if k <= V]


@pytest.mark.parametrize("k,V", BEAM_KV)
def test_beam_step_matches_float64_restatement(k, V):
    """Step 1 (row 0 ranked), a middle step, and the last permitted step (last = 1, history up to L - 1) over images that
    are full, short of beams, finished, ending some or all beams, feeding word 0, or holding tied rows."""
    L = 12
    kinds = ["full", "fewer", "empty", "eos", "all_eos", "zero", "tie"]
    for step, last in ((1, 0), (4, 0), (L - 1, 1)):
        t, end_tok = _beam_inputs(kinds, k, V, L, step, seed=100 * k + V + step)
        want = beam_step_ref(t, k, V, L, step, end_tok, last)
        got = beam_step_gpu(t, k, V, L, step, end_tok, last)
        _assert_beam_equal(got, want, (k, V, step))
        b = kinds.index("tie")
        if step > 1 and int(want["live"][b]) >= 2:   # the tied rows' best candidates survive side by side
            assert int(got["prev_tok"][b * k]) == int(got["prev_tok"][b * k + 1])
        b = kinds.index("zero")
        if int(want["live"][b]) > 0 and int(want["prev_tok"][b * k]) == 0:
            assert bool((got["words"][b * k:(b + 1) * k] == -1).all())


@pytest.mark.parametrize("step", [1, 4])
def test_beam_step_with_non_finite_rows(step):
    """A row with a NaN or +inf logit (its log-sum-exp is NaN) or with all -inf offers no candidates; an image whose
    ranked rows all do ends at once as failed; no other image notices; and k > V is rejected."""
    ops = _ops()
    k, V, L = 3, 100, 12
    kinds = ["full", "full", "full", "full", "full"]
    t, end_tok = _beam_inputs(kinds, k, V, L, step, seed=11 + step)
    clean = {n: x.clone() for n, x in t.items()}
    t["logits"][0 * k + 1, 17] = float("nan")          # image 0: row 1 (not ranked at step 1)
    t["logits"][1 * k + 0, 40] = float("inf")          # image 1: row 0
    t["logits"][2 * k:3 * k] = float("nan")            # image 2: every row
    t["logits"][4 * k + 0] = float("-inf")             # image 4: row 0
    want = beam_step_ref(t, k, V, L, step, end_tok, 0)
    got = beam_step_gpu(t, k, V, L, step, end_tok, 0)
    _assert_beam_equal(got, want, step)
    assert int(got["failed"][2]) == 1 and int(got["live"][2]) == 0 and bool((got["words"][2 * k:3 * k] == -1).all())
    if step == 1:
        assert int(got["failed"][1]) == 1 and int(got["failed"][4]) == 1
    # image 2 alone made finite again: every other image's outputs are bit-identical
    t2 = {n: x.clone() for n, x in t.items()}
    t2["logits"][2 * k:3 * k] = clean["logits"][2 * k:3 * k]
    got2 = beam_step_gpu(t2, k, V, L, step, end_tok, 0)
    for name in BEAM_OUT:
        per = k if got[name].shape[0] == len(kinds) * k else 1         # per-row outputs vs per-image ones
        a, c = got[name], got2[name]
        if a.is_floating_point():
            a, c = _bits(a), _bits(c)
        for b in (0, 1, 3, 4):
            assert torch.equal(a[b * per:(b + 1) * per], c[b * per:(b + 1) * per]), (name, b)
    from hypernet_image_captioning_b200._cabi import CaphnError
    with pytest.raises(CaphnError):
        beam_step_gpu(_beam_inputs(["full"], 7, 7, L, 1, seed=1)[0], 8, 7, L, 1, end_tok, 0)


# ----------------------------------------------------------------------------------------------------------------------
# decoders end to end
# ----------------------------------------------------------------------------------------------------------------------
def _pooled_model(p, E, H, V):
    import hypernet_image_captioning_b200 as C
    m = C.HyperNetPooled(E, H, V, None)
    sd = m.state_dict()
    sd.update(p)
    m.load_state_dict(sd)
    return m.cuda()


@pytest.mark.parametrize("V,fused", [(16385, False), (16384, True)])
def test_pooled_infer_above_the_fused_step_vocabulary_limit(V, fused, monkeypatch):
    """DecoderGRU.infer at B = 128 (one wave: BN = 128, nparts = 2 ceil(V / 128)).  V = 16385 needs 258 partial slots, more
    than the fused decode step holds: the three-launch branch runs instead.  V = 16384 (256 slots) still takes the fused
    step.  Both against the oracle's greedy decode."""
    from hypernet_image_captioning_b200 import graphs, ops
    B, T, E, H = 128, 66, 16, 32
    assert ops.use_projection_table(B, T, V) and ops._tc_ok(B, V, H)
    p = O.init_params_pooled(2048, E, H, V, L=1, seed=3)    # the oracle's own top-2 margins clear 2e-4 on ~3/4 of steps
    g = torch.Generator().manual_seed(4)
    pooled = torch.relu(torch.randn(B, 2048, generator=g))
    style = torch.randn(1, E, generator=g)
    h0 = torch.rand(B, H, generator=g)
    calls = []
    real = ops.gru_decode_step
    monkeypatch.setattr(ops, "gru_decode_step", lambda *a, **kw: (calls.append(a[3]), real(*a, **kw))[1])
    graphs.clear()
    m = _pooled_model(p, E, H, V)
    with torch.no_grad():
        probs = m.forward(style.cuda()).infer(m.image_encoder(pooled.cuda()), max_len=T, h0=h0.cuda())
    graphs.clear()
    if fused:                                            # (the loop runs more than once: graph warm-up and capture)
        assert calls and max(calls) == 256
    else:
        assert not calls
    ref, _, _ = O.path_pooled(p, style, pooled, None, h0, infer_len=T)
    assert rel_err(probs[:, 0], ref[:, 0]) < 1e-4
    ok, why = same_greedy_paths(probs, ref, tol=1e-4)
    assert ok, why


def test_pooled_infer_with_a_nan_image(monkeypatch):
    """One image's features NaN: no exception, NaN probabilities for it, every other row bit-identical to the run
    without it -- on the fused decode step and on the three-launch branch."""
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import graphs, ops
    B, T, E, H, V = 128, 17, 32, 64, 4000
    assert ops.use_projection_table(B, T, V) and ops._tc_ok(B, V, H)
    torch.manual_seed(2)
    with torch.device("cuda"):
        m = C.HyperNetPooled(E, H, V, None)
    g = torch.Generator().manual_seed(6)
    pooled = torch.relu(torch.randn(B, 2048, generator=g)).cuda()
    h0 = torch.rand(B, H, generator=g).cuda()
    bad = pooled.clone()
    bad[37] = float("nan")
    for fused in (True, False):
        monkeypatch.setattr(ops, "gru_decode_step_ok", lambda H, V, fused=fused: fused)
        outs = []
        for x in (pooled, bad):
            graphs.clear()
            with torch.no_grad():
                outs.append(m.forward(m.captioner.embed.weight[4:5]).infer(m.image_encoder(x), max_len=T, h0=h0).clone())
        graphs.clear()
        keep = torch.arange(B, device="cuda") != 37
        assert bool(outs[1][37].isnan().all()), fused
        assert torch.equal(outs[1][keep], outs[0][keep]), fused


def test_attention_greedy_with_a_nan_image():
    """Attention greedy decode (sample_prob = 1: every step feeds back its arg-max through the fused finisher) with one
    image's features NaN: no exception, every other row bit-identical.  (The feature branch's ReLU is fmaxf(z, 0), which
    maps NaN to 0, so this image's logits stay finite; NaN logits reach the finisher in the tests above.)"""
    import numpy as np
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import graphs, ops
    from hypernet_image_captioning_b200.synth import synth_captions
    B, T, V = 128, 20, 4000
    assert ops.use_projection_table(B, T + 1, V)
    torch.manual_seed(0)
    with torch.device("cuda"):
        m = C.HyperNetAttention(64, 48, 56, V, None)
    g = torch.Generator().manual_seed(3)
    feats = torch.randn(B, 49, 2048, generator=g).cuda()
    caps = synth_captions(B, T, V, g).cuda()
    bad = feats.clone()
    bad[5] = float("nan")
    outs = []
    for x in (feats, bad):
        graphs.clear()
        np.random.seed(0)
        with torch.no_grad():
            logits, _ = m.forward(m.captioner.embed.weight[4:5])(x, caps, 1.0)
        outs.append(logits.clone())
    graphs.clear()
    keep = torch.arange(B, device="cuda") != 5
    assert torch.equal(outs[1][keep], outs[0][keep])


def test_beam_search_with_a_nan_image_and_too_wide_a_beam(monkeypatch):
    """beam_search_batched where one image's logits turn NaN at every step (they are overwritten right after the
    vocabulary projection): that image gets no caption (None) and every other caption is the one the clean run gets.
    The same with that image's features NaN (which the feature branch's ReLU turns into zeros): no other caption moves.
    beam_size > V is rejected before anything runs."""
    import hypernet_image_captioning_b200 as C
    from hypernet_image_captioning_b200 import ops
    B, Fo, E, H, V = 8, 64, 48, 56, 300
    p = O.init_params_attention(2048, Fo, E, H, V, E, seed=31)
    p["captioner.fc.weight"][2] *= 60.0                  # </s> logit swings with h: beams finish at different steps
    p["captioner.fc.bias"][2] -= 1.0
    m = C.HyperNetAttention(Fo, E, H, V, None)
    sd = m.state_dict()
    sd.update(p)
    m.load_state_dict(sd)
    m = m.cuda()
    g = torch.Generator().manual_seed(5)
    feats = torch.randn(B, 49, 2048, generator=g).cuda()
    captioner = m.forward(torch.randn(1, E, generator=g).cuda())
    bad = feats.clone()
    bad[3] = float("nan")
    real = ops.LinearPlan.__call__
    for k in (3, 5):
        ok = captioner.beam_search_batched(feats, beam_size=k, end_sentence=2, max_steps=20)
        assert sum(c is not None for c in ok) >= B // 2
        others = lambda got: [c for i, c in enumerate(got) if i != 3]
        assert others(captioner.beam_search_batched(bad, beam_size=k, end_sentence=2, max_steps=20)) == others(ok)

        def nan_logits(self, x, relu=False, out=None, real=real, k=k):
            y = real(self, x, relu=relu, out=out)
            if y.shape == (B * k, V):                # the vocabulary projection of the beam rows
                y[3 * k:4 * k] = float("nan")
            return y
        monkeypatch.setattr(ops.LinearPlan, "__call__", nan_logits)
        got = captioner.beam_search_batched(feats, beam_size=k, end_sentence=2, max_steps=20)
        monkeypatch.setattr(ops.LinearPlan, "__call__", real)
        assert got[3] is None and others(got) == others(ok)
    small = C.HyperNetAttention(Fo, E, H, 4, None).cuda()
    with pytest.raises(ValueError):
        small.forward(torch.randn(1, E, device="cuda")).beam_search_batched(feats[:2], beam_size=5)
