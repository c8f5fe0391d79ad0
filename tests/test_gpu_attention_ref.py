"""The attention-GRU recurrence kernels against a float64 attention-GRU step (tests/attention_ref.py) at every shape
their plans dispatch on.

Paths and the shapes that select them (confirmed against the host functions named on the right, which the CPU tests
below call through ops._attstep_bytes / ops._attstep_bwd_bytes):

    step-split forward    H % 4 == 0, H, F <= 208 (13 k-tiles = ST_MAXKT),        caphn_attstep_pack_size
      (U / A / Y kernels)  P*F % 4 == 0, P <= 128, K and f tiles of one row in
                           shared memory: P <= 70 at H = F = 200, P <= 128 at H = F = 8
    step-split BPTT       the same, plus the deferred D kernel's shared memory,   caphn_attstep_bwd_size
      (G1 / G2 / A' / D)   which grows with T: T <= 151 at P = 49, T <= 109 at P = 70
                           (H = F = 200); P = 71 is covered (the forward is not)
    attention kernel      two single-buffered CTAs per SM (grid min(B, 296)),     attstep_fwd_impl / attstep_bwd_impl
      (A and A')           else NBUF = 2 with the grid of as_grid / ba_grid:
                           P = 70, H = F = 200: NBUF = 2 at any B, 1184 CTAs (fwd) / 2368 (bwd) at B = 4096;
                           P = 49, H = F = 200: NBUF = 2 from B = 11 841 (fwd) / 5 329 (bwd)
    U / Y / G1 / G2 tiles 16 / 64 / 64 / 32 rows; grouped: 8-row tiles when no      attstep_fwd_impl, GroupPlan
                           style has more than 8 rows, else 64 (fwd) / 32 (bwd)
    streaming forward     every other shape, H <= 1585 at F = 200                 caphn_attgru_seq_fwd
    streaming BPTT        every other shape, H <= 1024                             caphn_attgru_seq_bwd
    caphn_attn_df         T <= 205 at P = 49, F = 200                              caphn_attn_df

Forward and BPTT are chosen independently (AttGruWeights / attgru_bwd), so P = 71 streams forward and runs the BPTT
step-split, and T >= 152 at P = 49 runs the forward step-split and streams the BPTT.

Test per row: step-split forward / BPTT -> test_step_split_sweep; attention kernel plans -> test_attention_kernel_plans;
tiles -> test_step_split_sweep (B = 1, 5, 17, 65, 297), test_grouped_per_style_reference; mixed dispatch ->
test_mixed_dispatch; streaming -> test_streaming_*; attn_df -> test_attn_df*; the one-step decode pattern ->
test_decode_one_step_per_call.

Every output is compared on its own with rel_err = max|kernel - ref| / max|ref|: forward outputs (Hall, attn, ctx, the
saved u / r / z / n / gh_n) within FWD, gradients and the parameter products callers form from them (dW_ihc, dW_hh,
dU_a, db_u, db_hh, df_att) within BWD.  dbv is analytically zero (the softmax is shift invariant): it is compared
absolutely, against DBV * sum|ds| of the reference.  Hall[0] must keep h0, Hbm must be Hall[1:] transposed and the
inference form (no saved tensors, no Hbm) must write the same Hall, attn and ctx, all bit for bit.

Worst rel_err over all cases of this file (drift excepted) on one NVIDIA B200 (1000 W power limit), step-split /
streaming path (mixed-dispatch gradients counted as step-split):
    Hall 6.9e-6 / 5.1e-7, attn 4.4e-6 / 4.9e-7, ctx 4.5e-6 / 7.0e-7, u 7.8e-6 / 1.4e-6, r 3.4e-6 / 5.3e-7,
    z 3.9e-6 / 5.3e-7, n 1.1e-5 / 1.3e-6, gh_n 1.2e-5 / 1.5e-6;
    dGI 3.6e-6 / 4.0e-7, dGH 4.1e-6 / 5.4e-7, dU 1.7e-5 / 2.1e-6, dCTX 1.3e-5 / 6.4e-7, dK 1.2e-5 / 7.4e-7,
    dva 1.2e-5 / 7.8e-7, dh0 4.8e-6 / 4.8e-7, dW_ihc 4.1e-6 / 4.2e-7, dW_hh 6.8e-6 / 4.4e-7, dU_a 2.2e-5 / 1.9e-6,
    db_u 3.2e-5 / 5.6e-6, db_hh 3.9e-6 / 2.9e-7, df_att 1.7e-5 / 5.4e-7; dbv 4.3e-8 / 9.3e-8 of sum|ds|;
    caphn_attn_df alone 3.9e-7.
The largest step-split errors come from the smallest shapes (H = 4 to 8, P <= 4), where few products are summed and
db_u / dU_a sum gradients that cancel.  Each bound is 3 to 4x the worst error of its path."""
import pytest
import torch

import attention_ref as A
from golden_util import rel_err, report

gpu = pytest.mark.gpu

E = A.E_COLS
# rel_err bounds per path (module docstring: the errors they were set from).  The step-split kernels run their products
# as bf16x3 warp MMAs -- hi / lo bf16 halves keep 16 of the 24 mantissa bits of each operand, an error floor of about
# 5e-6 of max|product| (tests/test_bf16x3_numerics.py) -- and tanh_fast / ex2.approx in the attention; the streaming
# kernels are exact-fp32 FMA chains.
FWD = {"step": 4e-5, "seq": 5e-6}
BWD = {"step": 1e-4, "seq": 2e-5}
DBV, DF = 5e-7, 1.5e-6
FWD_KEYS = ("Hall", "attn", "ctx", "saved")
GATES = ("u", "r", "z", "n", "gh_n")

SEQ_FWD_MAX, SEQ_BWD_MAX, ATTN_DF_TMAX = 1585, 1024, 205

# (B, P, H, F) of the step-split sweep: every H % 16 tail and 13 k-tiles, F = 7 with P = 4, P up to 70 at H = F = 200
# and 128 at H = 8, and the row tails of the 16-row U, 64-row Y / G1 and 32-row G2 tiles; B = 297 puts two rows on
# some attention CTAs
SWEEP = [(1, 1, 4, 16), (5, 4, 8, 7), (17, 7, 12, 64), (65, 33, 16, 200), (297, 49, 20, 208), (5, 64, 100, 64),
         (17, 70, 200, 200), (1, 49, 196, 16), (65, 7, 204, 208), (5, 49, 208, 200), (17, 128, 8, 16),
         (297, 33, 200, 200)]


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


def _seed(tag, B, T, P, H, F):
    return {"sweep": 1, "plan": 2, "mixed": 3, "seq": 4, "grouped": 5, "decode": 6, "df": 7, "drift": 8}[tag] * 10 ** 9 \
        + B * 100_000 + T * 1000 + P * 7 + H * 3 + F


def bound(key, bounds=None, fwd="step", bwd="step"):
    """The bound of one output: ``bounds`` overrides; forward outputs take the bound of the forward's path, gradients the
    step-split bound unless both directions stream (a streamed BPTT of a step-split forward inherits its rounding)."""
    if bounds and key in bounds:
        return bounds[key]
    if key == "dbv":
        return DBV
    if key.split(".")[0] in FWD_KEYS:
        return FWD[fwd]
    return BWD["seq" if fwd == bwd == "seq" else "step"]


def flat(r):
    """Result dict (reference or kernel) -> one tensor per compared output."""
    out = {}
    for k, v in r.items():
        if k == "Hall":
            out[k] = v[1:]
        elif k == "saved":
            for q, name in enumerate(GATES):
                out[f"saved.{name}"] = v[q]
        elif k != "dbv_scale":
            out[k] = v
    return out


def errors(got, ref):
    g, r = flat(got), flat(ref)
    return {k: rel_err(g[k], r[k], ref["dbv_scale"].item() if k == "dbv" else None) for k in g}


def compare(got, ref, where, bounds=None, fwd="step", bwd="step"):
    """rel_err of every output of ``got`` against ``ref``; fails listing every output over its bound."""
    errs = errors(got, ref)
    report(f"{where}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    lim = {k: bound(k, bounds, fwd, bwd) for k in errs}
    bad = {k: e for k, e in errs.items() if not e < lim[k]}
    assert not bad, f"{where}: " + ", ".join(f"{k} rel err {e:.3e} (bound {lim[k]:.0e})" for k, e in sorted(bad.items()))
    return errs


def _products(r, T, B, H):
    """The parameter products the backward's callers form from the kernel outputs, in float64 on the host."""
    Hprev = r["Hall"][:-1].reshape(T * B, H).double()
    dGI, dGH, dU = r["dGI"].double(), r["dGH"].double(), r["dU"].double()
    r["dW_ihc"] = dGI.t() @ r["ctx"].reshape(T * B, -1).double()
    r["dW_hh"] = dGH.t() @ Hprev
    r["dU_a"] = dU.t() @ Hprev
    r["db_u"] = dU.sum(0)
    r["db_hh"] = dGH.sum(0)


def _cuda(d):
    return {k: v.cuda() for k, v in d.items()}


def run(d, fwd, bwd, dattns=(False, True), df=True):
    """The module's call pattern on inputs ``d``: ops.attgru_fwd on AttGruWeights, the inference form, ops.attgru_bwd
    (dattn absent and / or present) and ops.attn_df; the plan each direction takes is asserted first ("step" / "seq";
    bwd None: forward only).  Returns the forward outputs and one backward result per dattn setting, on the CPU."""
    ops = _ops()
    T, B, H3 = d["GIw"].shape
    P, H = d["K"].shape[1:]
    Fd = d["f"].shape[2]
    c = _cuda(d)
    GIw = c["GIw"].reshape(T * B, H3)
    lw = ops.AttGruWeights(c["W_ih"], c["W_hh"], c["U_a"], E, P)
    assert (lw.pack is not None) == (fwd == "step"), f"forward plan: expected {fwd}"
    outs = []
    for train in (True, False):
        Hall = torch.empty(T + 1, B, H, device="cuda")
        Hall[0] = c["h0"]
        attn = torch.empty(B, T, P, device="cuda")
        XC = torch.zeros(T * B, E + Fd, device="cuda")
        Hbm = torch.empty(B, T, H, device="cuda") if train else None
        saved = torch.empty(5, T, B, H, device="cuda") if train else None
        ops.attgru_fwd(c["K"], c["f"], GIw, lw, c["b_u"], c["v_a"], c["b_v"], c["b_hh"], Hall, Hbm, attn, XC, E, saved,
                       0, T)
        outs.append((Hall, Hbm, attn, XC, saved))
    torch.cuda.synchronize()
    (Hall, Hbm, attn, XC, saved), (Hinf, _, ainf, XCinf, _) = outs
    assert torch.equal(Hall[0], c["h0"]), "Hall[0] no longer holds h0"
    assert torch.equal(Hbm, Hall[1:].permute(1, 0, 2)), "Hbm is not Hall[1:] transposed"
    assert torch.equal(Hinf, Hall) and torch.equal(ainf, attn) and torch.equal(XCinf[:, E:], XC[:, E:]), \
        "the inference form computes a different Hall / attn / ctx"
    fw = {"Hall": Hall.cpu(), "attn": attn.cpu(), "ctx": XC[:, E:].reshape(T, B, Fd).cpu(), "saved": saved.cpu()}
    if bwd is None:
        return fw, []
    assert (ops._attstep_bwd_bytes(H, Fd, P, B, T)[0] > 0) == (bwd == "step"), f"BPTT plan: expected {bwd}"
    res = []
    for with_dattn in dattns:
        dattn = c["dattn"] if with_dattn else None
        g = ops.attgru_bwd(c["dHbm"], dattn, c["K"], c["f"], attn, saved, Hall, c["U_a"], c["v_a"], c["W_ih"],
                           c["W_hh"], E)
        r = dict(fw)
        r.update({k: v.cpu() for k, v in zip(("dGI", "dGH", "dU", "dCTX", "dK", "dva", "dbv", "dh0"), g)})
        if df:
            r["df_att"] = ops.attn_df(attn, g[3], torch.zeros(B, P, Fd, device="cuda")).cpu()
        torch.cuda.synchronize()
        _products(r, T, B, H)
        res.append(r)
    return fw, res


def reference(d, with_dattn, grad=True):
    dd = dict(d)
    if not with_dattn:
        dd.pop("dattn", None)
    return A.attention_gru(dd, grad=grad)


def check(tag, B, T, P, H, Fd, fwd, bwd, dattns=(False, True), bounds=None):
    d = A.inputs(B, T, P, H, Fd, _seed(tag, B, T, P, H, Fd), dattn=True)
    fw, res = run(d, fwd, bwd, dattns, df=T <= ATTN_DF_TMAX)
    where = f"{tag} B={B} T={T} P={P} H={H} F={Fd} ({fwd} fwd, {bwd} bwd)"
    if bwd is None:
        ref = reference(d, False, grad=False)
        return [compare(fw, ref, where, bounds, fwd, fwd)]
    out = []
    for with_dattn, got in zip(dattns, res):
        ref = reference(d, with_dattn)
        if not T <= ATTN_DF_TMAX:
            del ref["df_att"]
        out.append(compare(got, ref, where + (" dattn" if with_dattn else ""), bounds, fwd, bwd))
    return out


# ----------------------------------------------------------------------------------------------------------------------
# plans (host functions of the library: no device needed)
# ----------------------------------------------------------------------------------------------------------------------
def _fwd_covered(H, Fd, P):
    return _ops()._attstep_bytes(H, Fd, P, 0)[0] > 0


def _bwd_covered(H, Fd, P, T):
    return _ops()._attstep_bwd_bytes(H, Fd, P, 1, T)[0] > 0


def test_step_split_plan_boundaries():
    assert _fwd_covered(200, 200, 70) and not _fwd_covered(200, 200, 71)
    assert _fwd_covered(8, 8, 128) and not _fwd_covered(8, 8, 129)
    assert _bwd_covered(200, 200, 71, 3)
    assert _bwd_covered(200, 200, 49, 151) and not _bwd_covered(200, 200, 49, 152)
    assert _bwd_covered(200, 200, 70, 109) and not _bwd_covered(200, 200, 70, 110)
    for H, Fd, P in ((150, 200, 49), (212, 200, 49), (200, 209, 49), (200, 201, 49), (200, 200, 129)):
        assert not _fwd_covered(H, Fd, P) and not _bwd_covered(H, Fd, P, 3), (H, Fd, P)


def test_swept_shapes_take_the_paths_they_are_listed_under():
    for B, P, H, Fd in SWEEP:
        assert _fwd_covered(H, Fd, P) and _bwd_covered(H, Fd, P, 3), (B, P, H, Fd)
    for H in SEQ_H:
        assert not _fwd_covered(H, 200, 49) and not _bwd_covered(H, 200, 49, 3), H
    for P, Fd in SEQ_PF:
        assert not _fwd_covered(200, Fd, P) and not _bwd_covered(200, Fd, P, 3), (P, Fd)


def test_attention_step_equals_the_oracle():
    """attention_ref.attention_step with K = W_a f + b_a is the oracle's Bahdanau attention."""
    from oracle import caption_hn_oracle as O
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(11)
    B, P, H, Fd = 5, 49, 20, 16
    pre = "captioner.attention."
    p = {pre + "W_a.weight": torch.randn(H, Fd, generator=g, dtype=torch.float64) / Fd ** 0.5,
         pre + "W_a.bias": torch.randn(H, generator=g, dtype=torch.float64) * 0.1,
         pre + "U_a.weight": torch.randn(H, H, generator=g, dtype=torch.float64) / H ** 0.5,
         pre + "U_a.bias": torch.randn(H, generator=g, dtype=torch.float64) * 0.1,
         pre + "v_a.weight": torch.randn(1, H, generator=g, dtype=torch.float64),
         pre + "v_a.bias": torch.randn(1, generator=g, dtype=torch.float64)}
    f = torch.randn(B, P, Fd, generator=g, dtype=torch.float64)
    h = torch.randn(B, H, generator=g, dtype=torch.float64)
    K = F.linear(f, p[pre + "W_a.weight"], p[pre + "W_a.bias"])
    ctx, alpha, _, _ = A.attention_step(K, f, h, p[pre + "U_a.weight"], p[pre + "U_a.bias"],
                                        p[pre + "v_a.weight"].reshape(-1), p[pre + "v_a.bias"])
    want_ctx, want_alpha = O.bahdanau(p, f, h)
    assert (ctx - want_ctx).abs().max().item() <= 1e-14
    assert (alpha - want_alpha).abs().max().item() <= 1e-14


def _mutant_visible(mutant, B, T, P):
    """Shapes on which the defect changes anything at all: a row mix-up needs two rows, a stale state two steps, and
    every defect of the scores or their gradient two positions (at P = 1 alpha == 1 whatever the scores)."""
    if mutant == "f of the next batch row":
        return B > 1
    if mutant == "attention reads the new state":
        return T > 1
    if mutant in ("last position dropped from the softmax", "tanh(K) + u", "dattn ignored"):
        return P > 1
    return True


@pytest.mark.parametrize("mutant", A.MUTANTS)
def test_tolerances_catch_planted_defects(mutant):
    """Each defect planted in the float64 reference moves at least one compared output by more than 10x its bound, on
    the step-split sweep's shapes and seeds (T = 3, dattn present) wherever the defect can show."""
    n = 0
    for B, P, H, Fd in SWEEP:
        T = 3
        if not _mutant_visible(mutant, B, T, P):
            continue
        d = A.inputs(B, T, P, H, Fd, _seed("sweep", B, T, P, H, Fd), dattn=True)
        ref = A.attention_gru(d)
        ratio = max(e / bound(k) for k, e in errors(A.attention_gru(d, mutant), ref).items())
        assert ratio > 10, f"{mutant}: B={B} P={P} H={H} F={Fd} moves the outputs by only {ratio:.1f}x the bound"
        n += 1
    assert n >= 6


# ----------------------------------------------------------------------------------------------------------------------
# step-split sweep and the attention kernel's plans
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("B,P,H,Fd", SWEEP)
def test_step_split_sweep(B, P, H, Fd):
    for T in (1, 3):
        check("sweep", B, T, P, H, Fd, "step", "step")


@gpu
@pytest.mark.parametrize("B,T,P,fwd_only", [
    (5, 2, 70, False),        # NBUF = 2 in both directions, one row per CTA
    (300, 2, 70, False),      # NBUF = 2, 148 CTAs with 3 rows each: the mbarrier parity of reused buffers
    (4096, 1, 70, False),     # NBUF = 2, grid widened to 1184 CTAs (fwd) / 2368 (bwd)
    (12288, 1, 49, True),     # forward NBUF = 2 from B = 11 841 at P = 49 (beam search: 4096 images x k = 3)
    (6144, 1, 49, False),     # BPTT NBUF = 2 from B = 5 329 at P = 49
])
def test_attention_kernel_plans(B, T, P, fwd_only):
    """H = F = 200: the attention kernels of attstep_fwd_impl / attstep_bwd_impl leave the two-CTAs-per-SM plan for one
    double-buffered CTA per SM (NBUF = 2, grid as_grid / ba_grid) when two single-buffered CTAs no longer fit."""
    check("plan", B, T, P, 200, 200, "step", None if fwd_only else "step", dattns=(True,) if B > 300 else (False, True))


@gpu
@pytest.mark.parametrize("B,T,P,fwd,bwd", [(5, 3, 71, "seq", "step"), (2, 151, 49, "step", "step"),
                                           (2, 152, 49, "step", "seq")])
def test_mixed_dispatch(B, T, P, fwd, bwd):
    """Forward and BPTT plans chosen independently, as the module chooses them: P = 71 streams forward and runs the BPTT
    step-split; T = 152 at P = 49 runs the forward step-split and streams the BPTT (the deferred D kernel's shared
    memory grows with T; T = 151 is the last step-split length)."""
    check("mixed", B, T, P, 200, 200, fwd, bwd)


# ----------------------------------------------------------------------------------------------------------------------
# streaming kernels
# ----------------------------------------------------------------------------------------------------------------------
SEQ_H = (1, 5, 150, 202, 212, 256, 512, 1024)
SEQ_PF = ((49, 201), (129, 200), (196, 200))          # P*F % 4 != 0, P > 128


@gpu
@pytest.mark.parametrize("H", SEQ_H)
def test_streaming_hidden_sizes(H):
    for B in (1, 5):
        check("seq", B, 3, 49, H, 200, "seq", "seq")


@gpu
@pytest.mark.parametrize("P,Fd", SEQ_PF)
def test_streaming_positions_and_features(P, Fd):
    for B in (1, 5):
        check("seq", B, 3, P, 200, Fd, "seq", "seq")


@gpu
def test_streaming_forward_at_its_largest_hidden_size():
    """H = 1585 passes the streaming forward's shared-memory check at F = 200, not the BPTT's (H <= 1024)."""
    check("seq", 5, 3, 49, SEQ_FWD_MAX, 200, "seq", None)


@gpu
def test_streaming_refuses_one_above_its_limits():
    ops = _ops()
    from hypernet_image_captioning_b200._cabi import CaphnError
    B, T, P, Fd = 2, 1, 49, 200
    z = lambda *s: torch.zeros(*s, device="cuda")
    for H, direction in ((SEQ_FWD_MAX + 1, "fwd"), (SEQ_BWD_MAX + 1, "bwd")):
        W_ih, W_hh, U_a = z(3 * H, E + Fd), z(3 * H, H), z(H, H)
        K, f, Hall, attn = z(B, P, H), z(B, P, Fd), z(T + 1, B, H), z(B, T, P)
        if direction == "fwd":
            lw = ops.AttGruWeights(W_ih, W_hh, U_a, E, P)
            with pytest.raises(CaphnError):
                ops.attgru_fwd(K, f, z(T * B, 3 * H), lw, z(H), z(H), z(1), z(3 * H), Hall, z(B, T, H), attn,
                               z(T * B, E + Fd), E, z(5, T, B, H), 0, T)
        else:
            with pytest.raises(CaphnError):
                ops.attgru_bwd(z(B, T, H), None, K, f, attn, z(5, T, B, H), Hall, U_a, z(H), W_ih, W_hh, E)


# ----------------------------------------------------------------------------------------------------------------------
# caphn_attn_df
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("T", [1, 20, ATTN_DF_TMAX])
def test_attn_df(T):
    """df = sum_t alpha_t dctx_t from the reference's own alpha and dctx (rounded to float32) against its df_att."""
    ops = _ops()
    B, P, H, Fd = 3, 49, 8, 200
    d = A.inputs(B, T, P, H, Fd, _seed("df", B, T, P, H, Fd), dattn=True)
    ref = A.attention_gru(d)
    df = ops.attn_df(ref["attn"].float().cuda(), ref["dCTX"].float().cuda(), torch.zeros(B, P, Fd, device="cuda"))
    e = rel_err(df, ref["df_att"])
    report(f"attn_df B={B} T={T} P={P} F={Fd}: df_att {e:.2e}")
    assert e < DF, f"attn_df T={T}: rel err {e:.3e} (bound {DF:.0e})"


@gpu
def test_attn_df_refuses_one_above_its_longest_caption():
    ops = _ops()
    from hypernet_image_captioning_b200._cabi import CaphnError
    B, T, P, Fd = 2, ATTN_DF_TMAX + 1, 49, 200
    with pytest.raises(CaphnError):
        ops.attn_df(torch.zeros(B, T, P, device="cuda"), torch.zeros(T * B, Fd, device="cuda"),
                    torch.zeros(B, P, Fd, device="cuda"))


# ----------------------------------------------------------------------------------------------------------------------
# grouped (many-style) recurrence
# ----------------------------------------------------------------------------------------------------------------------
GROUP_SHAPES = [(49, 200, 200), (7, 100, 64)]           # (P, H, F)


@gpu
@pytest.mark.parametrize("counts", [(1, 3, 8), (1, 8, 13, 33, 64, 65)])
@pytest.mark.parametrize("P,H,Fd", GROUP_SHAPES)
def test_grouped_per_style_reference(P, H, Fd, counts):
    """attgru_{fwd,bwd}_grouped called as grouped.py calls them: rows sorted by style, tiles from GroupPlan (8-row tiles
    when no style has more than 8 rows, else 64-row forward / 32-row backward tiles with tails), each style's generated
    W_ih / W_hh / b_ih / b_hh in its own row of Theta.  Each style is compared with its own float64 reference; the
    shared attention weights' gradients (dva, dbv, dU_a, db_u) with the sum over styles."""
    ops = _ops()
    from hypernet_image_captioning_b200.grouped import GroupPlan, _layout
    G, T = len(counts), 3
    B = sum(counts)
    H3, o_hh, o_bi, o_bh, theta = _layout(E, Fd, H)
    styles = [A.inputs(n, T, P, H, Fd, _seed("grouped", n, T, P, H, Fd) + g, dattn=True) for g, n in enumerate(counts)]
    for d in styles[1:]:
        for k in ("U_a", "b_u", "v_a", "b_v"):
            d[k] = styles[0][k]
    groups = torch.cat([torch.full((n,), g, dtype=torch.int64) for g, n in enumerate(counts)])
    plan = GroupPlan.get(groups, G, T, torch.device("cuda"))
    assert plan.tile_rows_fwd == (8 if max(counts) <= 8 else 64)
    Theta = torch.zeros(G, theta)
    for g, d in enumerate(styles):
        Theta[g, :o_hh] = d["W_ih"].reshape(-1)
        Theta[g, o_hh:o_bi] = d["W_hh"].reshape(-1)
        Theta[g, o_bi:o_bh] = torch.randn(H3, generator=torch.Generator().manual_seed(g))   # b_ih: folded into GIw
        Theta[g, o_bh:] = d["b_hh"]
    Theta = Theta.cuda()
    cat = lambda k, dim: torch.cat([d[k] for d in styles], dim).cuda()
    K, f, h0, dHbm, dattn = cat("K", 0), cat("f", 0), cat("h0", 0), cat("dHbm", 0), cat("dattn", 0)
    GIw = cat("GIw", 1).reshape(T * B, H3)
    s0 = _cuda({k: styles[0][k] for k in ("U_a", "b_u", "v_a", "b_v")})
    gw = ops.AttGruGroupWeights(Theta, s0["U_a"], E, Fd, H, P)
    Hall = torch.empty(T + 1, B, H, device="cuda")
    Hall[0] = h0
    Hbm, attn = torch.empty(B, T, H, device="cuda"), torch.empty(B, T, P, device="cuda")
    XC, saved = torch.zeros(T * B, E + Fd, device="cuda"), torch.empty(5, T, B, H, device="cuda")
    ops.attgru_fwd_grouped(K, f, GIw, gw, s0["b_u"], s0["v_a"], s0["b_v"], Theta[:, o_bh:].contiguous(), Hall, Hbm,
                           attn, XC, E, saved, plan.tiles_fwd, plan.tile_rows_fwd)
    g = ops.attgru_bwd_grouped(dHbm, dattn, K, f, attn, saved, Hall, Theta, s0["U_a"], s0["v_a"], E, plan.tiles_bwd,
                               plan.tile_rows_bwd)
    df = ops.attn_df(attn, g[3], torch.zeros(B, P, Fd, device="cuda"))
    torch.cuda.synchronize()
    assert torch.equal(Hall[0], h0) and torch.equal(Hbm, Hall[1:].permute(1, 0, 2))
    dGI, dGH, dU, dCTX, dK, dva, dbv, dh0 = [t.cpu() for t in g]
    Hall, attn, ctx, saved, df = Hall.cpu(), attn.cpu(), XC[:, E:].reshape(T, B, Fd).cpu(), saved.cpu(), df.cpu()
    tb = lambda x: x.view(T, B, -1)
    shared = {"dva": 0, "dbv": 0, "dbv_scale": 0, "dU_a": 0, "db_u": 0}
    r0 = 0
    for gi, d in enumerate(styles):
        rows = slice(r0, r0 + counts[gi])
        ref = A.attention_gru(d)
        got = {"Hall": Hall[:, rows], "attn": attn[rows], "ctx": ctx[:, rows], "saved": saved[:, :, rows],
               "dGI": tb(dGI)[:, rows].reshape(-1, H3), "dGH": tb(dGH)[:, rows].reshape(-1, H3),
               "dU": tb(dU)[:, rows].reshape(-1, H), "dCTX": tb(dCTX)[:, rows].reshape(-1, Fd), "dK": dK[rows],
               "dh0": dh0[rows], "df_att": df[rows]}
        _products(got, T, counts[gi], H)
        for k in shared:
            shared[k] = shared[k] + ref.pop(k)
        got.pop("dU_a"), got.pop("db_u")
        compare(got, ref, f"grouped P={P} H={H} F={Fd} style {gi} ({counts[gi]} rows of {counts})")
        r0 += counts[gi]
    Hprev = Hall[:-1].reshape(T * B, H).double()
    got = {"dva": dva, "dbv": dbv, "dU_a": dU.double().t() @ Hprev, "db_u": dU.double().sum(0)}
    compare(got, shared, f"grouped P={P} H={H} F={Fd} shared attention weights ({counts})")


# ----------------------------------------------------------------------------------------------------------------------
# one step per call (greedy decode / beam search) and the bf16 operand rows of h
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("B,P,H,Fd", [(65, 49, 200, 200), (5, 7, 100, 64)])
def test_decode_one_step_per_call(B, P, H, Fd):
    """attgru_fwd(t, t + 1) step by step, the workspace resumed between calls (no saved tensors, no Hbm), against the
    reference; after each step the hi / lo bf16 rows of h the gates kernel wrote for the next step (the vocabulary
    projection's A operand, ops.attstep_h_operand) must be h rounded to bf16 plus a remainder good to 2^-16 max|h|."""
    ops = _ops()
    T = 4
    d = A.inputs(B, T, P, H, Fd, _seed("decode", B, T, P, H, Fd))
    ref = A.attention_gru(d, grad=False)
    c = _cuda(d)
    lw = ops.AttGruWeights(c["W_ih"], c["W_hh"], c["U_a"], E, P)
    assert lw.pack is not None
    GIw = c["GIw"].reshape(T * B, 3 * H)
    Hall = torch.empty(T + 1, B, H, device="cuda")
    Hall[0] = c["h0"]
    attn, XC = torch.empty(B, T, P, device="cuda"), torch.zeros(T * B, E + Fd, device="cuda")
    for t in range(T):
        assert (lw._resume == (Hall.data_ptr(), t)) == (t > 0), "the one-step calls do not resume the workspace"
        ops.attgru_fwd(c["K"], c["f"], GIw, lw, c["b_u"], c["v_a"], c["b_v"], c["b_hh"], Hall, None, attn, XC, E, None,
                       t, t + 1)
        op = ops.attstep_h_operand(lw, B, H, Fd, t)
        h = Hall[t + 1]
        assert torch.equal(op.hi[:, :H], h.to(torch.bfloat16)), f"step {t}: hi is not h rounded to bf16"
        if op.lo is not None:
            e = (op.hi[:, :H].float() + op.lo[:, :H].float() - h).abs().max().item()
            assert e <= 2.0 ** -16 * h.abs().max().item(), f"step {t}: hi + lo misses h by {e:.3e}"
    torch.cuda.synchronize()
    got = {"Hall": Hall.cpu(), "attn": attn.cpu(), "ctx": XC[:, E:].reshape(T, B, Fd).cpu()}
    compare(got, {k: ref[k] for k in got}, f"decode B={B} P={P} H={H} F={Fd} one step per call")


# ----------------------------------------------------------------------------------------------------------------------
# drift at the benchmark's shape
# ----------------------------------------------------------------------------------------------------------------------
DRIFT_BOUNDS = {"Hall": 1.5e-5, "attn": 6e-6, "ctx": 8e-6, "saved.u": 1.9e-5, "saved.r": 1.2e-5, "saved.z": 1.1e-5,
                "saved.n": 3.5e-5, "saved.gh_n": 2e-5, "dGI": 1.2e-5, "dGH": 1.1e-5, "dU": 2.8e-5, "dCTX": 2.2e-5,
                "dK": 1.4e-5, "dva": 1.6e-5, "dbv": 1.5e-9, "dh0": 1.2e-5, "df_att": 1.8e-5, "dW_ihc": 8e-6,
                "dW_hh": 1.2e-5, "dU_a": 2.5e-5, "db_u": 2.8e-5, "db_hh": 7e-6}


@gpu
@pytest.mark.parametrize("B,T", [(512, 20), (64, 64)])
def test_drift_at_the_benchmark_shape(B, T):
    """P = 49, F = E = H = 200 (step-split both ways), dattn present: the benchmark's batch and caption length, and a
    long caption.

    rel_err measured on one NVIDIA B200 (1000 W power limit), B = 512, T = 20 / B = 64, T = 64:
        Hall 3.65e-6 / 3.91e-6, attn 1.59e-6 / 1.50e-6, ctx 2.06e-6 / 1.70e-6, u 4.98e-6 / 4.70e-6,
        r 3.03e-6 / 2.82e-6, z 2.82e-6 / 3.00e-6, n 9.55e-6 / 7.01e-6, gh_n 5.32e-6 / 4.55e-6, dGI 3.45e-6 / 1.96e-6,
        dGH 2.90e-6 / 2.70e-6, dU 7.25e-6 / 7.33e-6, dCTX 5.50e-6 / 5.88e-6, dK 3.54e-6 / 3.54e-6, dva 4.33e-6 / 3.58e-6,
        dbv 4.3e-10 / 1.4e-10 of sum|ds|, dh0 3.09e-6 / 2.87e-6, df_att 4.68e-6 / 4.74e-6, dW_ihc 1.80e-6 / 2.12e-6,
        dW_hh 2.75e-6 / 3.15e-6, dU_a 4.95e-6 / 6.53e-6, db_u 4.06e-6 / 7.02e-6, db_hh 1.58e-6 / 1.79e-6.
    Each bound in DRIFT_BOUNDS is at most 4x the larger of the two.  Relative to max|ref| the error does not grow over
    64 steps: it stays below the T <= 5 bounds of the sweep."""
    errs = check("drift", B, T, 49, 200, 200, "step", "step", dattns=(True,), bounds=DRIFT_BOUNDS)[0]
    assert set(errs) == set(DRIFT_BOUNDS)
