"""The cross-entropy kernels, the loss nodes' path selection and the decoder's gather / scatter / reduction kernels
(csrc/ce_misc.cu, csrc/grouped.cu, csrc/gru_seq.cu) against float64 (tests/loss_ref.py) at every path they dispatch on.

Dispatch table (host code -> the test that reaches each cell; every swept shape is asserted to land in its cell):

    kernel / entry point        cells                                              host code               test
    ce_fwd_kernel               vec: ld % 4, V % 4, X 16-B aligned; else scalar.   ce_misc.cu:53           test_ce_sweep
                                One 256-thread CTA per row: V tails against
                                1024 (vec) and 256 (scalar)
    ce_finish_kernel            M < 1024, M = 1024, M > 1024 (per-thread loop);    caphn_ce_fwd            test_ce_sweep,
                                every row ignored -> NaN, count 0                                          test_ce_all_rows_ignored
    ce_fwd_split_kernel         vec (one cp.async.bulk of the row) or scalar       ce_misc.cu:244, 626-629 test_ce_sweep,
                                staging of round4(V) floats; V = 50000 accepted,                           test_ce_refusals
                                50001 refused; [V, Vp) zero; lo == NULL;
                                misaligned hi / lo refused
    ce_bwd_kernel               vec: ld, lddx, V % 4, X and dX aligned; scalar     ce_misc.cu:110          test_ce_sweep
    ce_bwd_split_kernel         64 x 64 tiles, vecx per thread (v0 + c4 + 3 < V);  ce_misc.cu:148, 653-655 test_ce_sweep
                                M % 64 and V % 64 tails; lo, hiT / loT, dbias
                                each NULL or not; m-tiles on gridDim.x             test_ce_bwd_split_past_old_grid_limit
    ce_fwd_for_loss /           (a) one-pass (b) two-pass, V > 50000 only          functional.py:264,      test_loss_node_paths,
    vocab_bwd_fused /           (c) fp32 dlogits (M < 128; 32 <= V < 128);         278-279, 332-338        test_loss_path_boundaries
    VocabPrep                   fp32 and bf16 precision; VocabPrep on / off
    gather_rows                 vec (E, ldo % 4, both aligned) or scalar;          ce_misc.cu gather_rows  test_gather_rows
                                negative index -> zero row
    build_inputs                mode 0 / 1, T = 1 and 2                            build_inputs_kernel     test_build_inputs
    embed_scatter_add /         red.global.add.v4 or atomicAdd; t0 = 1, 2;         embed_scatter_add,      test_embed_scatter_add,
    scatter_add_rows            T <= t0 launches nothing; negative idx skipped     scatter_add_rows        test_scatter_add_rows
                                (scatter_add_rows); duplicate tokens
    colsum                      rows_per_block 256 .. 16; 8-row unroll tail;       ce_misc.cu:713-715      test_colsum,
                                out accumulates; ceil(M / rpb) <= 65535                                    test_colsum_past_old_grid_limit
    group_colsum                empty groups, odd sizes, T > 1, ldo pitch          grouped.cu:69-81        test_group_colsum
    mean_pos / mean_pos_bwd     P = 1, 49, 70; Fd tails against 128 / 256;         ce_misc.cu mean_pos*    test_mean_pos
                                extra or NULL; += semantics
    relu_mask, leaky_relu(_bwd) NaN, +-0, subnormals, n tails                      ce_misc.cu, grouped.cu  test_masks
    transpose_pad / copy_pad    R, C tails against 32, ldd > R / C, nb = 1 and     gru_seq.cu:199-264      test_pad_builders,
    (+ _batched)                65535; nb = 65536 and small dstride refused                                test_pad_batched_limits_and_refusals

The float64 reference against torch's float64 cross_entropy -> test_reference_*; the restated plans' boundaries ->
test_loss_path_boundaries, test_colsum_rows_per_block_steps; planted defects (tests/loss_ref.py CE_MUTANTS, GLUE_MUTANTS)
-> test_planted_ce_defects_exceed_the_tolerance (the sweep's shapes up to 2^22 logits) and
test_planted_glue_defects_exceed_the_tolerance; each prints its smallest margin over the tolerance (13.8x for the
missing lo term, 951x for the lost dbias tile, 6e4x or more for the others).

Target contract (DESIGN.md §6): the ignore index may be any value (-100 included); any other target outside [0, V) is a
counted row with a NaN loss and a zero gradient row, and no logit outside the row is read
(test_out_of_range_targets_*: the targets sit in the row pitch [V, V + 8) and at -1 on rows >= 1, so the unfixed kernels
read inside the buffer and fail with a finite wrong loss and a missing -1 rather than a fault).

Bounds: 3-4x the worst error measured on one NVIDIA B200 (1000 W power limit) over the sweep, with the analytic
expectation in brackets.
    quantity                   bound                              measured                  [expected]
    lse, per row               LSE_ULPS = 5 ulp of max(|lse|, 1)  1.32 ulp (M 10240, V 4)   [a few ulp: expf / logf <= 2
                                                                                              ulp each, no fast-math]
    loss, per row              LOSS_ULPS = 16 ulp, same unit      4.34 ulp (M 1023, V 3)    [lse's error plus the rounding
                                                                                              of lse - x[t]]
    mean loss                  MEAN_REL = 4e-7 of mean max(|lse|, 1)    9.9e-8              [log2(M) ulp of the sum]
    u = softmax - onehot       U_ABS = 4e-6 absolute (|u| <= 1)   1.09e-6 (M 1024, V 9684)  [~2^-20: x - max rounded in
                                                                                              fp32 at |x - max| <= 32]
    hi + lo                    U_ABS + 2^-16 |u| (bf16 mode       0.986 of the bound        [the bound itself: each bf16
                               U_ABS + 2^-8 |u|); analytic                                   rounding reaches half an ulp]
    dbias (ce_bwd_split)       DBIAS_REL = 5e-6 of sum_m |d|      1.41e-6 (M 1, V 9685)     [64-row partials: a few 2^-24
                                                                                              of sum |d| per atomic add]
    loss-node gradients        NODE_TOL = 3.5e-5 (fp32 mode),     1.05e-5, 3.9e-3           [test_gpu_gemm_ref.py bounds
                               1.5e-2 (bf16 mode) of max |ref|                               of the products]
    float-data accumulations   ACC_REL = 6e-7 of the sum of |x|   1.72e-7 (embed_scatter)   [n 2^-24 worst case; far less
    (scatter, colsum, groups)                                                                 with random signs]
    mean_pos                   (P + 1) 2^-24 of mean |x|          1.78e-7 (P 70)            [analytic]
    mean_pos_bwd               4 roundings of 2^-24, elementwise  within                    [analytic]
The split's errors reach its bound because the bound is the rounding itself, not a measurement.  On the old kernels the
out-of-range-target tests fail with a finite mean (6.84 and 8.35 where NaN is due) and non-zero gradient rows (0.139),
the grid-limit tests with CaphnError status 9 (cudaErrorInvalidConfiguration), and test_ce_refusals with the Vp / 64 >
65535 call not refused (its launch captured in a graph, never run).  The file's GPU tests take about 8 s
on the B200.
Exact data (integers: every partial sum an fp32 number whatever the atomic order) must come out equal to float64."""
import math
import warnings

import numpy as np
import pytest
import torch

import loss_ref as R
from golden_util import report

gpu = pytest.mark.gpu

# bounds (module docstring)
LSE_ULPS = 5.0
LOSS_ULPS = 16.0
MEAN_REL = 4e-7
U_ABS = 4e-6
DBIAS_REL = 5e-6
ACC_REL = 6e-7
NODE_TOL = {"fp32": 3.5e-5, "bf16": 1.5e-2}
SPLIT_REL = {True: 2.0 ** -16, False: 2.0 ** -8}

GSCALES = (1.7, 0.0, -0.9)
# (M, V, ignore): V over {1, 3, 4, 255, 256, 257, 1023, 1024, 1025, 9684, 9685, 10240, 50000}, M over {1, 63, 64, 65,
# 1023, 1024, 1025, 10240}, crossed sparsely; ignore None, an in-range column, or -100
SWEEP = [
    (1, 1, None), (63, 3, 0), (64, 4, None), (65, 255, R.IGNORE_NEG), (1023, 256, None), (1024, 257, 0),
    (1025, 1023, None), (10240, 1024, 5), (63, 1025, None), (1024, 9684, R.IGNORE_NEG), (65, 9685, None),
    (1025, 10240, 0), (64, 50000, None), (1, 50000, R.IGNORE_NEG), (10240, 4, 0), (1, 9685, None), (1023, 3, R.IGNORE_NEG),
    (65, 257, None),
]
LAYOUTS = ("pitch", "offset")      # ld = round4(V) + 4 at an aligned base (vec iff V % 4 == 0) / one float in (scalar)


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


def _cabi():
    from hypernet_image_captioning_b200 import _cabi
    return _cabi


def ulp32(x):
    """ulp of fp32 numbers of magnitude |x| (float64 tensor in, float64 out)."""
    a = x.abs().clamp_min(2.0 ** -126)
    return torch.pow(2.0, torch.floor(torch.log2(a)) - 23)


def _layout(M, V, seed, layout, device="cuda", gap=float("nan")):
    ld = R.round4(V) + 4
    return R.logits(M, V, seed, ld=ld, off=0 if layout == "pitch" else 1, gap=gap, device=device)


# ----------------------------------------------------------------------------------------------------------------------
# direct C-ABI calls (own output buffers: pitches, alignments and NULL operands chosen by the test)
# ----------------------------------------------------------------------------------------------------------------------
def _st():
    return torch.cuda.current_stream().cuda_stream


def _ign(ignore):
    return (0, 0) if ignore is None else (1, int(ignore))


def c_ce_fwd(x, t, ignore):
    M, V = x.shape
    lse = torch.empty(M, device="cuda")
    scratch = torch.empty(2 * M, device="cuda")
    lb = torch.empty(2, device="cuda")
    _cabi().call("caphn_ce_fwd", x.data_ptr(), x.stride(0), t.data_ptr(), M, V, *_ign(ignore), lse.data_ptr(),
                 scratch.data_ptr(), lb.data_ptr(), _st())
    return lse, scratch[:M], scratch[M:], lb


def _bf16_buf(rows, cols):
    """bf16 [rows, cols] in a buffer with one sentinel row (NaN bits) after it."""
    b = torch.full((rows + 1, cols), float("nan"), device="cuda", dtype=torch.bfloat16)
    return b[:rows], b


def c_ce_fwd_split(x, t, ignore, Vp, with_lo=True):
    M, V = x.shape
    lse = torch.empty(M, device="cuda")
    scratch = torch.empty(2 * M, device="cuda")
    lb = torch.empty(2, device="cuda")
    hi, hib = _bf16_buf(M, Vp)
    lo, lob = _bf16_buf(M, Vp) if with_lo else (None, None)
    _cabi().call("caphn_ce_fwd_split", x.data_ptr(), x.stride(0), t.data_ptr(), M, V, *_ign(ignore), lse.data_ptr(),
                 scratch.data_ptr(), lb.data_ptr(), hi.data_ptr(), None if lo is None else lo.data_ptr(), Vp, _st())
    return lse, scratch[:M], scratch[M:], lb, hi, lo, (hib, lob)


def c_ce_bwd(x, t, ignore, lse, lb, g, lddx, off):
    M, V = x.shape
    buf = torch.full((off + M * lddx + 1,), float("nan"), device="cuda")
    dX = buf.as_strided((M, V), (lddx, 1), off)
    _cabi().call("caphn_ce_bwd", x.data_ptr(), x.stride(0), t.data_ptr(), M, V, *_ign(ignore), lse.data_ptr(),
                 g.data_ptr(), lb.data_ptr(), dX.data_ptr(), lddx, _st())
    return dX, buf


def c_ce_bwd_split(x, t, ignore, lse, lb, g, lo=True, hiT=False, loT=False, dbias=True, Vp=None, Mp=None):
    M, V = x.shape
    Vp = R.round64(V) if Vp is None else Vp
    Mp = R.round64(M) if Mp is None else Mp
    h, hb = _bf16_buf(M, Vp)
    l, lb_ = _bf16_buf(M, Vp) if lo else (None, None)
    hT, hTb = _bf16_buf(V, Mp) if hiT else (None, None)
    lT, lTb = _bf16_buf(V, Mp) if loT else (None, None)
    db = torch.zeros(V, device="cuda") if dbias else None
    p = lambda a: None if a is None else a.data_ptr()
    _cabi().call("caphn_ce_bwd_split", x.data_ptr(), x.stride(0), t.data_ptr(), M, V, *_ign(ignore), lse.data_ptr(),
                 g.data_ptr(), lb.data_ptr(), h.data_ptr(), p(l), Vp, p(hT), p(lT), Mp, p(db), _st())
    return h, l, hT, lT, db, (hb, lb_, hTb, lTb)


def _sentinel_row_intact(buf):
    return buf is None or bool(torch.isnan(buf[-1].float()).all())


def _split_err(hi, lo, u, sc=1.0):
    """max over elements of |(hi + lo) / sc - u| / (U_ABS + rel |u|); elements where sc == 0 must be exactly 0."""
    got = hi.double() + (lo.double() if lo is not None else 0.0)
    if sc == 0.0:
        return 0.0 if float(got.abs().max()) == 0.0 else math.inf
    err = (got / sc - u).abs() / (U_ABS + SPLIT_REL[lo is not None] * u.abs())
    return float(err.max())


def _split_invariant(hi, lo):
    """|lo| <= ulp(hi) / 2 (bf16: 8 significant bits) and hi == rn_bf16(hi + lo), except where |lo| is exactly
    ulp(hi) / 2: rounding u - hi to bf16 can land on the tie, and ties go to the even neighbour."""
    h, l = hi.double(), lo.double()
    _, e = torch.frexp(h)                                      # |h| = m 2^e, m in [0.5, 1): ulp(h) / 2 = 2^(e - 9)
    half_ulp = torch.where(h != 0, torch.ldexp(torch.ones_like(h), e - 9), torch.zeros_like(h))
    if not bool((l.abs() <= half_ulp).all()):
        return False
    return bool(((R.bf16_rn(h + l) == h) | (l.abs() == half_ulp)).all())


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the reference, the plans' boundaries, the planted defects
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ignore", [None, 0, R.IGNORE_NEG])
def test_reference_matches_torch_cross_entropy(ignore):
    import torch.nn.functional as F
    x, _ = R.logits(37, 257, 3)
    x = x.contiguous()
    t = R.targets(37, 257, 3, ignore)
    r = R.ce_ref(x, t, ignore)
    xd = x.double().requires_grad_(True)
    loss = F.cross_entropy(xd, t, ignore_index=R.IGNORE_NEG if ignore is None else ignore)
    (dl,) = torch.autograd.grad(loss * 1.7, xd)
    assert abs(r["mean"] - loss.item()) <= 1e-14 * abs(loss.item())
    d = r["u"] * R.grad_scale(1.7, r["count"])
    assert float((d - dl).abs().max()) <= 1e-14
    rows = F.cross_entropy(xd.detach(), t, ignore_index=R.IGNORE_NEG if ignore is None else ignore, reduction="none")
    assert float((r["loss"] - rows).abs().max()) <= 1e-14 * float(rows.abs().max())
    assert float((r["lse"] - torch.logsumexp(xd.detach(), 1)).abs().max()) <= 1e-14 * 8
    Hm = torch.randn(37, 20, generator=R._gen(1), dtype=torch.float64)
    W = torch.randn(257, 20, generator=R._gen(2), dtype=torch.float64)
    dH, dW, db = R.vocab_ref(x, t, ignore, 1.7, Hm, W)
    assert float((dH - dl @ W).abs().max()) <= 1e-14 and float((dW - dl.t() @ Hm).abs().max()) <= 1e-14
    assert float((db - dl.sum(0)).abs().max()) <= 1e-14


def test_reference_out_of_range_and_all_ignored():
    x, _ = R.logits(4, 5, 1)
    x = x.contiguous()
    t = torch.tensor([2, 5, -1, R.IGNORE_NEG])
    r = R.ce_ref(x, t, R.IGNORE_NEG)
    assert r["count"] == 3 and math.isnan(r["mean"]) and math.isnan(r["loss"][1]) and math.isnan(r["loss"][2])
    assert float(r["u"][1:].abs().max()) == 0.0 and r["loss"][3] == 0.0
    r = R.ce_ref(x, torch.full((4,), 7), 7)
    assert r["count"] == 0 and math.isnan(r["mean"]) and float(r["u"].abs().max()) == 0.0


def test_loss_path_boundaries():
    P = R.loss_path
    # M = 127 / 128 (tensor-core rows), V = 31 / 32 (K of dH), V = 127 / 128 (rows of the dW product)
    assert P(127, 1000, 150) == "fp32-dlogits" and P(128, 1000, 150) == "one-pass"
    assert P(4096, 31, 150) == "fp32-dlogits" and P(4096, 32, 150) == "fp32-dlogits"
    assert P(2048, 127, 150) == "fp32-dlogits" and P(2048, 128, 150) == "one-pass"
    # V = 50000 / 50001: the one-pass kernel's shared-memory row; above it the two-pass operands
    assert P(256, 50000, 150) == "one-pass" and P(256, 50001, 150) == "two-pass"
    assert R.fwd_split_smem(50000) == 200000 and R.fwd_split_smem(50001) is None and R.fwd_split_smem(3) == 16
    assert not R.tc_ok(4096, 150, 31) and R.tc_ok(4096, 150, 32)
    # M H V = 2^24 - 1 / 2^24, the tensor-core work threshold (2^24 - 1 = 4097 * 21 * 195)
    assert 4097 * 21 * 195 == 2 ** 24 - 1 and P(4097, 195, 21) == "fp32-dlogits" and P(4096, 256, 16) == "one-pass"
    # without gradients the one-pass kernel is never picked
    assert P(4096, 256, 16, need_grad=False) == "two-pass" and not R.vocab_prep_on(4096, 256, 64, need_grad=False)
    # VocabPrep also needs the logits product (K = H >= 32) on the tensor cores
    assert R.vocab_prep_on(1024, 1000, 64) and not R.vocab_prep_on(1024, 1000, 20) and P(1024, 1000, 20) == "one-pass"
    assert not R.vocab_prep_on(256, 50001, 150)
    # vec conditions
    assert R.fwd_vec(1028, 1024, 0) and not R.fwd_vec(1028, 1024, 4) and not R.fwd_vec(1030, 1024, 0)
    assert not R.fwd_vec(1028, 1025, 0)
    assert R.bwd_vec(8, 8, 4, 16, 32) and not R.bwd_vec(8, 9, 4, 16, 32) and not R.bwd_vec(8, 8, 4, 16, 36)
    assert R.split_vec_threads(68, 65, 0) == (16, 16) and R.split_vec_threads(68, 64, 4) == (0, 16)


def test_colsum_rows_per_block_steps():
    C = R.colsum_rpb
    assert C(65536, 1200) == (256, 256)                          # 10 x 256 blocks: enough at 256 rows
    assert C(160003, 100) == (128, 1251) and C(80001, 100) == (64, 1251) and C(38005, 100) == (32, 1188)
    assert C(37000, 100) == (16, 2313) and C(10240, 150) == (16, 640) and C(1, 1) == (16, 1)
    assert C(16776960, 3) == (256, 65535)                        # the last M the old plan could launch
    assert C(16776961, 3) == (257, 65281)                        # raised so that gridDim.y <= 65535
    assert R.cdiv(16776961, 256) == 65536


def _mutant_margin(mutant, M, V, ignore, i):
    """Error of the mutant / its tolerance, in the metric the GPU sweep uses (inf: NaN or an infinite error)."""
    x, _ = _layout(M, V, 100 + i, "pitch", device="cpu")
    t = R.targets(M, V, 100 + i, ignore)
    ok = R.ce_ref(x, t, ignore)
    g = 1.7
    if mutant != "last vector dropped from max / sum exp" and float(ok["u"].abs().max()) == 0.0:
        return None                                                       # V = 1: u is 0 whatever the kernel does
    if mutant == "last vector dropped from max / sum exp":
        mu = R.ce_ref(x, t, ignore, mutant)
        e = ((mu["lse"] - ok["lse"]).abs() / ulp32(ok["lse"].abs().clamp_min(1.0))).max() / LSE_ULPS
    elif mutant == "target column off by one":
        if V < 2:
            return None
        mu = R.ce_ref(x, t, ignore, mutant)
        e = ((mu["u"] - ok["u"]).abs().max() / U_ABS)
    elif mutant == "ignored rows counted in the denominator":
        if ignore is None or ok["count"] == M:
            return None
        mu = R.ce_ref(x, t, ignore, mutant)
        e = abs(mu["mean"] - ok["mean"]) / (MEAN_REL * float(ok["lse"].abs().clamp_min(1.0).mean()))
    elif mutant == "scale by M instead of the count":
        if ignore is None or ok["count"] == M:
            return None
        sc, sm = R.grad_scale(g, ok["count"]), R.grad_scale(g, ok["count"], M, mutant)
        e = (ok["u"] * sm / sc - ok["u"]).abs().max() / U_ABS
    elif mutant == "dbias missing the last partial 64-row tile":
        if M % 64 == 0:
            return None
        d = ok["u"] * R.grad_scale(g, ok["count"])
        e = ((R.dbias_ref(d, mutant) - d.sum(0)).abs() / (DBIAS_REL * d.abs().sum(0) + 1e-300)).max()
    else:
        mu = R.split_ref(ok["u"].float(), True, mutant)
        e = ((mu - ok["u"]).abs() / (U_ABS + SPLIT_REL[True] * ok["u"].abs())).max()
    e = float(e)
    return math.inf if math.isnan(e) else e


@pytest.mark.parametrize("mutant", R.CE_MUTANTS)
def test_planted_ce_defects_exceed_the_tolerance(mutant):
    ratios = [r for i, (M, V, ig) in enumerate(SWEEP) if M * V <= 1 << 22
              for r in [_mutant_margin(mutant, M, V, ig, i)] if r is not None]
    assert ratios, mutant
    report(f"ce mutant {mutant!r}: smallest margin {min(ratios):.3g}x the tolerance over {len(ratios)} shapes")
    assert min(ratios) > 10, f"{mutant}: moves the result by only {min(ratios):.2f}x the tolerance"


def test_planted_glue_defects_exceed_the_tolerance():
    g = R._gen(5)
    ratios = {}
    for B, T, sizes in GROUP_CASES:
        goff = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32)
        X = torch.randn(T * B, 37, generator=g)
        ok = R.group_colsum_ref(X, goff, B, T)
        mu = R.group_colsum_ref(X, goff, B, T, "odd last row of a group dropped")
        den = ACC_REL * (_group_abs(X, goff, B, T) + 1e-300)
        if any(s % 2 for s in sizes):
            ratios.setdefault("odd last row of a group dropped", []).append(float(((mu - ok).abs() / den).max()))
    for Bm, P, Fd in MEAN_CASES:
        dX0, gg, ex = torch.randn(Bm, P, Fd, generator=g), torch.randn(Bm, Fd, generator=g), torch.randn(Bm, P, Fd, generator=g)
        ok = R.mean_pos_bwd_ref(gg, dX0, ex)
        mu = R.mean_pos_bwd_ref(gg, dX0, ex, "mean_pos_bwd ignores extra")
        ratios.setdefault("mean_pos_bwd ignores extra", []).append(float(((mu - ok).abs() / (ACC_REL * ok.abs().clamp_min(1e-30))).max()))
    for n, E, rows in SCATTER_CASES:
        idx = _scatter_idx(n, rows, 3)
        dX = torch.randn(n, E, generator=g)
        tb = torch.zeros(rows, E)
        ok = R.scatter_ref(tb, idx, dX)
        mu = R.scatter_ref(tb, idx, dX, "one duplicate contribution lost")
        absum = R.scatter_ref(tb, idx, dX.abs())
        ratios.setdefault("one duplicate contribution lost", []).append(float(((mu - ok).abs() / (ACC_REL * absum + 1e-300)).max()))
    assert set(ratios) == set(R.GLUE_MUTANTS)
    for k, v in ratios.items():
        report(f"glue mutant {k!r}: smallest margin {min(v):.3g}x the tolerance over {len(v)} shapes")
        assert min(v) > 10, k


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the cross-entropy kernel sweep
# ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def fp32_precision():
    ops = _ops()
    yield ops
    ops.set_precision("fp32")


@gpu
@pytest.mark.parametrize("i", range(len(SWEEP)), ids=[f"M{M}-V{V}-ign{ig}" for M, V, ig in SWEEP])
def test_ce_sweep(i):
    M, V, ignore = SWEEP[i]
    t = R.targets(M, V, 100 + i, ignore, device="cuda")
    g = torch.tensor([GSCALES[i % 3]], device="cuda")
    worst = dict(lse=0.0, loss=0.0, mean=0.0, u=0.0, split=0.0, db=0.0)
    invariant = True
    cells = set()
    for li, layout in enumerate(LAYOUTS):
        x, xbuf = _layout(M, V, 100 + i, layout)
        xaddr = x.data_ptr()
        ref = R.ce_ref(x, t, ignore)
        vec = R.fwd_vec(x.stride(0), V, xaddr)
        assert vec == (layout == "pitch" and V % 4 == 0)
        cells.add(("fwd", vec))
        u = ref["u"]
        lscale = ulp32(ref["lse"].abs().clamp_min(1.0))
        mean_scale = float(ref["lse"].abs().clamp_min(1.0).mean())
        # ce_fwd and ce_fwd_split: lse, row loss, row validity, mean and count
        Vp = R.round64(V)
        fwd = c_ce_fwd(x, t, ignore)
        one = c_ce_fwd_split(x, t, ignore, Vp, with_lo=(i + li) % 2 == 0)
        hi, lo, sent = one[4:]
        for lse, rl, rv, lb in (fwd, one[:4]):
            worst["lse"] = max(worst["lse"], float(((lse.double() - ref["lse"]).abs() / lscale).max()))
            worst["loss"] = max(worst["loss"], float(((rl.double() - ref["loss"]).abs() / lscale).max()))
            assert torch.equal(rv.bool(), ref["valid"]) and lb[1].item() == ref["count"]
            if ref["count"]:
                worst["mean"] = max(worst["mean"], abs(lb[0].item() - ref["mean"]) / mean_scale)
            assert float(rl[~ref["valid"]].abs().max()) == 0.0 if (~ref["valid"]).any() else True
        # the unscaled operand of ce_fwd_split: within the split's bound of u, the split invariant, [V, Vp) zero
        worst["split"] = max(worst["split"], _split_err(hi[:, :V], None if lo is None else lo[:, :V], u))
        if lo is not None:
            invariant &= _split_invariant(hi[:, :V], lo[:, :V])
        if Vp > V:
            assert float(hi[:, V:].float().abs().max()) == 0.0 and (lo is None or float(lo[:, V:].float().abs().max()) == 0.0)
        assert all(_sentinel_row_intact(b) for b in sent)
        # ce_bwd: per element against u * sc, dX's pitch gaps untouched; vec or scalar per the restated condition
        lse, _, _, lb = fwd
        sc = R.grad_scale(g.item(), ref["count"])
        lddx = R.round4(V) + 4 if li == 0 else V
        dX, dbuf = c_ce_bwd(x, t, ignore, lse, lb, g, lddx, 0 if li == 0 else 1)
        cells.add(("bwd", R.bwd_vec(x.stride(0), lddx, V, xaddr, dX.data_ptr())))
        if sc == 0.0:
            assert float(dX.abs().max()) == 0.0
        else:
            worst["u"] = max(worst["u"], float((dX.double() / sc - u).abs().max()))
        inside = torch.zeros_like(dbuf, dtype=torch.bool)
        inside.as_strided((M, V), (lddx, 1), 0 if li == 0 else 1).fill_(True)
        assert bool(torch.isnan(dbuf[~inside]).all())
        # ce_bwd_split: the four NULL / non-NULL combinations rotate with the shape and the layout
        var = (i + 2 * li) % 4
        opt = [dict(lo=True, hiT=True, loT=True, dbias=True), dict(lo=False, hiT=True, loT=False, dbias=True),
               dict(lo=True, hiT=False, loT=False, dbias=False), dict(lo=False, hiT=False, loT=False, dbias=True)][var]
        h, l, hT, lT, db, sent = c_ce_bwd_split(x, t, ignore, lse, lb, g, **opt)
        nv, ns = R.split_vec_threads(x.stride(0), V, xaddr)
        cells.add(("split", nv > 0, ns > 0))
        worst["split"] = max(worst["split"], _split_err(h[:, :V], None if l is None else l[:, :V], u, sc))
        if R.round64(V) > V:
            assert float(h[:, V:].float().abs().max()) == 0.0
        if hT is not None:       # the transposed copy is the same numbers, [M, Mp) zero
            assert torch.equal(hT[:, :M], h[:, :V].t()) and float(hT[:, M:].float().abs().max() if hT.shape[1] > M else 0) == 0.0
            if lT is not None:
                assert torch.equal(lT[:, :M], l[:, :V].t())
        if db is not None:
            d = u * sc
            if sc == 0.0:
                assert float(db.abs().max()) == 0.0
            else:
                worst["db"] = max(worst["db"], float(((db.double() - d.sum(0)).abs() / (d.abs().sum(0) + 1e-30)).max()))
        assert all(_sentinel_row_intact(b) for b in sent)
        del xbuf
    report(f"ce sweep M={M} V={V} ignore={ignore} g={g.item()}: lse {worst['lse']:.2f} ulp, loss {worst['loss']:.2f} ulp, "
           f"mean {worst['mean']:.2e}, u {worst['u']:.2e}, split {worst['split']:.3f} of bound, dbias {worst['db']:.2e} "
           f"cells {sorted(cells)}")
    assert invariant
    assert worst["lse"] <= LSE_ULPS and worst["loss"] <= LOSS_ULPS and worst["mean"] <= MEAN_REL
    assert worst["u"] <= U_ABS and worst["split"] <= 1.0 and worst["db"] <= DBIAS_REL
    # every shape lands where the restated plan puts it: vec only with V % 4 == 0 on the aligned layout, a per-thread
    # mix in ce_bwd_split exactly when V % 64 is not 0 (or V % 4 is not 0) on the aligned layout
    assert ("fwd", True) in cells if V % 4 == 0 else ("fwd", True) not in cells
    assert ("fwd", False) in cells
    assert ("split", True, V % 64 != 0) in cells if V >= 4 else ("split", False, True) in cells


def test_sweep_covers_every_cell():
    """The swept (M, V) land in every cell of the table: ce_fwd's V tails against 1024 / 256, ce_finish's three M
    regimes, ce_bwd_split's M % 64 and V % 64 tails."""
    Vs = {V for _, V, _ in SWEEP}
    Ms = {M for M, _, _ in SWEEP}
    assert {V % 1024 for V in Vs if V % 4 == 0} >= {0, 4, 256} and {V % 256 for V in Vs if V % 4} >= {1, 3, 255}
    assert min(Ms) < 1024 and 1024 in Ms and max(Ms) > 1024
    assert {M % 64 for M in Ms} >= {0, 1, 63} and {V % 64 for V in Vs} >= {0, 1, 63}
    assert {ig for _, _, ig in SWEEP} == {None, 0, 5, R.IGNORE_NEG}
    assert any(R.fwd_split_smem(V) == 200000 for V in Vs)


@gpu
def test_ce_all_rows_ignored():
    x, _ = _layout(70, 33, 1, "pitch")
    t = torch.full((70,), 4, device="cuda")
    for out in (c_ce_fwd(x, t, 4), c_ce_fwd_split(x, t, 4, 64)):
        lb = out[3]
        assert math.isnan(lb[0].item()) and lb[1].item() == 0.0
    hi = c_ce_fwd_split(x, t, 4, 64)[4]
    assert float(hi.float().abs().max()) == 0.0


def _refuses(call):
    """True when call() raises CaphnError.  It runs while a CUDA graph is captured on a side stream, so a kernel that a
    missing argument check would let through is recorded in a graph that is never replayed, not executed."""
    C = _cabi()
    g = torch.cuda.CUDAGraph()
    refused = False
    with warnings.catch_warnings():
        warnings.filterwarnings("ignore", "The CUDA Graph is empty")     # what a refused call leaves: nothing captured
        with torch.cuda.graph(g, capture_error_mode="relaxed"):
            try:
                call()
            except C.CaphnError:
                refused = True
    g.reset()
    return refused


@gpu
def test_ce_refusals():
    C = _cabi()
    x = torch.zeros(2, 50001, device="cuda")
    t = torch.zeros(2, dtype=torch.int64, device="cuda")
    ok = c_ce_fwd_split(x[:, :50000], t, None, R.round64(50000))          # 200 KB of dynamic shared memory
    assert abs(ok[3][0].item() - math.log(50000)) < 1e-5
    with pytest.raises(C.CaphnError):
        c_ce_fwd_split(x, t, None, R.round64(50001))
    # Every buffer below is sized for what the call would touch if it launched, and the calls run under _refuses (graph
    # capture): were a check lost, the launch would be recorded, never run, and the test would fail with "not refused".
    lse, scratch = torch.zeros(1, device="cuda"), torch.zeros(2, device="cuda")
    lossbuf, gscale = torch.tensor([1.0, 1.0], device="cuda"), torch.ones(1, device="cuda")
    hb = torch.zeros(2 * 64 + 8, device="cuda", dtype=torch.bfloat16)   # hi [1, 64] and lo [1, 64] at offsets 0..65
    for hi_off, lo_off in ((1, 0), (0, 1)):                               # 2-byte offsets: not 8-byte aligned
        assert _refuses(lambda: C.call("caphn_ce_fwd_split", x.data_ptr(), x.stride(0), t.data_ptr(), 1, 33, 0, 0,
                                       lse.data_ptr(), scratch.data_ptr(), lossbuf.data_ptr(), hb[hi_off:].data_ptr(),
                                       hb[64 + lo_off:].data_ptr(), 64, _st())), (hi_off, lo_off)
    # the capture itself: a call that passes its checks is not counted as refused (and its launch is not run)
    assert not _refuses(lambda: C.call("caphn_ce_bwd_split", x.data_ptr(), x.stride(0), t.data_ptr(), 1, 33, 0, 0,
                                       lse.data_ptr(), gscale.data_ptr(), lossbuf.data_ptr(), hb.data_ptr(), None, 64,
                                       None, None, 64, None, _st()))
    Vp = 64 * 65536                                                       # Vp / 64 > 65535 v-tiles
    hi = torch.zeros(1, Vp, device="cuda", dtype=torch.bfloat16)          # row 0 of hi: all a launch would write
    assert _refuses(lambda: C.call("caphn_ce_bwd_split", x.data_ptr(), x.stride(0), t.data_ptr(), 1, 50001, 0, 0,
                                   lse.data_ptr(), gscale.data_ptr(), lossbuf.data_ptr(), hi.data_ptr(), None, Vp, None,
                                   None, 64, None, _st()))


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the loss nodes' three paths
# ----------------------------------------------------------------------------------------------------------------------
# (path, M, V, H): (a) one-pass with / without VocabPrep (K = H < 32: the logits product is not on the tensor cores),
# (b) two-pass above the shared-memory row, (c) fp32 dlogits for M < 128 and for 32 <= V < 128
NODE_CASES = [("one-pass", 512, 1000, 64), ("one-pass", 1024, 1000, 20), ("two-pass", 128, 50001, 16),
              ("fp32-dlogits", 127, 1000, 150), ("fp32-dlogits", 2048, 100, 150)]


# VocabPrep on and off where the plan turns it on, off only elsewhere (test_loss_path_boundaries pins the plan)
NODE_PARAMS = [pytest.param(c, prep, id=f"{c[0]}-M{c[1]}-V{c[2]}-H{c[3]}-{'prep' if prep else 'noprep'}")
               for c in NODE_CASES for prep in ((True, False) if R.vocab_prep_on(*c[1:]) else (False,))]


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("case,prep", NODE_PARAMS)
def test_loss_node_paths(case, prep, prec, monkeypatch, fp32_precision):
    import torch.nn.functional as F
    from hypernet_image_captioning_b200 import functional as Fn
    ops = fp32_precision
    path, M, V, H = case
    assert R.loss_path(M, V, H) == path
    ops.set_precision(prec)
    g = R._gen(M + V + H)
    Hbm = torch.randn(M, H, generator=g).cuda()
    fc_w = (torch.randn(V, H, generator=g) * (2.0 / H ** 0.5)).cuda()
    fc_b = (torch.randn(V, generator=g) * 0.1).cuda()
    ignore = 0 if V % 2 else None
    tgt = R.targets(M, V, 9, ignore, device="cuda")
    gscale = torch.tensor([1.7], device="cuda")
    ran = []
    for name in ("ce_fwd", "ce_fwd_split", "ce_bwd", "ce_bwd_split"):
        fn = getattr(ops, name)
        monkeypatch.setattr(ops, name, lambda *a, _fn=fn, _n=name, **k: (ran.append(_n), _fn(*a, **k))[1])
    vp = Fn.VocabPrep(M, V, H, True, Hbm)
    assert vp.on == R.vocab_prep_on(M, V, H) and (vp.on or not prep)
    use_prep = prep
    if use_prep:
        vp.start(fc_w)
        logits = vp.logits(Hbm, fc_b)
        vp.finish()
        pre = vp.saved()
    else:
        logits = ops.linear(Hbm, fc_w, fc_b)
        pre = None
    lb, lse, hi, lo = Fn.ce_fwd_for_loss(logits, tgt, ignore, H, True)
    dfc_w, dfc_b, dHbm = Fn.vocab_bwd_fused(logits, tgt, ignore, lse, lb, gscale, Hbm, fc_w, hi, lo, pre)
    torch.cuda.synchronize()
    want = {"one-pass": ["ce_fwd_split"], "two-pass": ["ce_fwd", "ce_bwd_split"], "fp32-dlogits": ["ce_fwd", "ce_bwd"]}[path]
    assert ran == want, (path, ran)
    assert (hi is not None) == (path == "one-pass") and (lo is not None) == (path == "one-pass" and prec == "fp32")
    xd = logits.double().requires_grad_(True)
    loss = F.cross_entropy(xd, tgt, ignore_index=R.IGNORE_NEG if ignore is None else ignore)
    (dl,) = torch.autograd.grad(loss * 1.7, xd)
    assert abs(lb[0].item() - loss.item()) <= 1e-5 * abs(loss.item())
    errs = []
    for got, ref in ((dHbm, dl @ fc_w.double()), (dfc_w, dl.t() @ Hbm.double()), (dfc_b, dl.sum(0))):
        assert got.shape == ref.shape
        errs.append(float((got.double() - ref).abs().max()) / float(ref.abs().max()))
    report(f"loss node {path} M={M} V={V} H={H} {prec} prep={use_prep}: dH {errs[0]:.2e} dW {errs[1]:.2e} "
           f"db {errs[2]:.2e} of max|ref|")
    assert max(errs) <= NODE_TOL[prec]


# ----------------------------------------------------------------------------------------------------------------------
# GPU: out-of-range targets and the grid limits (fixed in this change; the unfixed kernels fail without a fault)
# ----------------------------------------------------------------------------------------------------------------------
def _oor_case(V, layout):
    """Logits with pitch V + 8 whose gaps hold 0.5 (finite: an unfixed kernel reads them and returns a finite loss),
    targets in [V, V + 8) and -1 (rows >= 1 only), the ignore index -100 and in-range targets."""
    M = 12
    x, buf = R.logits(M, V, 4, ld=V + 8, off=0 if layout == "pitch" else 1, gap=0.5, device="cuda")
    t = torch.tensor([V - 1, V, -1, 0, R.IGNORE_NEG, V + 7, 1 % V, -1, V + 3, 0, R.IGNORE_NEG, V - 1], device="cuda")
    bad = torch.tensor([False, True, True, False, False, True, False, True, True, False, False, False], device="cuda")
    return x, buf, t, bad


@gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("V", [64, 257])
def test_out_of_range_targets_forward(V, layout):
    x, _, t, bad = _oor_case(V, layout)
    ref = R.ce_ref(x, t, R.IGNORE_NEG)
    assert ref["count"] == 10
    outs = {"ce_fwd": c_ce_fwd(x, t, R.IGNORE_NEG), "ce_fwd_split": c_ce_fwd_split(x, t, R.IGNORE_NEG, R.round64(V))}
    for name, (lse, rl, rv, lb, *rest) in outs.items():
        assert lb[1].item() == 10, name                                      # out-of-range rows are counted
        assert math.isnan(lb[0].item()), f"{name}: the mean must be NaN, got {lb[0].item()}"
        assert bool(torch.isnan(rl[bad]).all()), f"{name}: row losses {rl[bad].tolist()}"
        good = ~bad
        assert float((rl[good].double() - ref["loss"][good]).abs().max()) < 1e-4
        if rest:                                                            # the operand: zero rows, others u
            hi, lo = rest[0], rest[1]
            assert float(hi[bad].float().abs().max()) == 0.0 and float(lo[bad].float().abs().max()) == 0.0, name
            assert _split_err(hi[good][:, :V], lo[good][:, :V], ref["u"][good]) <= 1.0


@gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("V", [64, 257])
def test_out_of_range_targets_backward(V, layout):
    x, _, t, bad = _oor_case(V, layout)
    ref = R.ce_ref(x, t, R.IGNORE_NEG)
    lse, _, _, lb = c_ce_fwd(x, t, R.IGNORE_NEG)
    g = torch.tensor([1.7], device="cuda")
    sc = R.grad_scale(1.7, 10)
    dX, _ = c_ce_bwd(x, t, R.IGNORE_NEG, lse, lb, g, V, 0)
    h, l, hT, lT, db, _ = c_ce_bwd_split(x, t, R.IGNORE_NEG, lse, lb, g, hiT=True, loT=True)
    assert float(dX[bad].abs().max()) == 0.0, "ce_bwd: gradient rows of out-of-range targets must be zero"
    assert float(h[bad].float().abs().max()) == 0.0 and float(l[bad].float().abs().max()) == 0.0, "ce_bwd_split"
    assert float((dX.double() / sc - ref["u"]).abs().max()) <= U_ABS
    assert _split_err(h[:, :V], l[:, :V], ref["u"], sc) <= 1.0
    d = ref["u"] * sc
    assert float(((db.double() - d.sum(0)).abs() / (d.abs().sum(0) + 1e-30)).max()) <= DBIAS_REL
    # and through the drop-in cross_entropy
    import hypernet_image_captioning_b200 as C
    xc = x.detach().clone().requires_grad_(True)
    loss = C.cross_entropy(xc, t, R.IGNORE_NEG)
    loss.backward()
    assert math.isnan(loss.item()) and float(xc.grad[bad].abs().max()) == 0.0


@gpu
def test_ce_bwd_split_past_old_grid_limit():
    """M = 4 194 305 rows: 65 537 m-tiles, one more than gridDim.y allowed when the m-tiles were on y."""
    M, V = 4194305, 64
    x = (torch.randn(M, V, device="cuda", generator=torch.Generator("cuda").manual_seed(3)) * 3.0)
    t = torch.randint(0, V, (M,), device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    lse, _, _, lb = c_ce_fwd(x, t, None)
    g = torch.tensor([float(M)], device="cuda")                            # sc = 1: d = u
    h, l, _, _, db, _ = c_ce_bwd_split(x, t, None, lse, lb, g)
    tail = slice(M - 129, M)                                               # the rows past the old limit and before it
    ref = R.ce_ref(x[tail], t[tail])
    assert _split_err(h[tail], l[tail], ref["u"]) <= 1.0
    d_sum = torch.zeros(V, dtype=torch.float64, device="cuda")
    d_abs = torch.zeros(V, dtype=torch.float64, device="cuda")
    for m0 in range(0, M, 1 << 20):
        u = R.ce_ref(x[m0:m0 + (1 << 20)], t[m0:m0 + (1 << 20)])["u"]
        d_sum += u.sum(0)
        d_abs += u.abs().sum(0)
    e = float(((db.double() - d_sum).abs() / d_abs).max())
    report(f"ce_bwd_split M={M}: dbias {e:.2e} of sum |d|")
    assert e <= DBIAS_REL


@gpu
def test_colsum_past_old_grid_limit():
    """M = 16 776 961 rows, N = 3: 65 536 row blocks of 256, one more than gridDim.y allows; values in {-1, 0, 1} keep
    every partial sum exact (|sum| <= M < 2^24)."""
    M, N = 16776961, 3
    X = torch.randint(-1, 2, (M, N), device="cuda", generator=torch.Generator("cuda").manual_seed(5)).float()
    out = _ops().colsum(X)
    assert torch.equal(out.double(), X.double().sum(0))


# ----------------------------------------------------------------------------------------------------------------------
# GPU: gather / scatter / reduction kernels
# ----------------------------------------------------------------------------------------------------------------------
def _int_data(shape, seed, lo=-4, hi=5, device="cuda"):
    return torch.randint(lo, hi, shape, generator=R._gen(seed)).float().to(device)


def _misaligned(rows, cols, seed, ints=True):
    """[rows, cols] view one float into a buffer (not 16-byte aligned)."""
    b = torch.empty(rows * cols + 1, device="cuda")
    v = b[1:].view(rows, cols)
    v.copy_(_int_data((rows, cols), seed) if ints else torch.randn(rows, cols, generator=R._gen(seed)).cuda())
    return v


@gpu
@pytest.mark.parametrize("E,aligned", [(64, True), (150, True), (64, False), (1, True), (513, True)])
def test_gather_rows(E, aligned):
    ops = _ops()
    table = torch.randn(40, E, generator=R._gen(E)).cuda()
    idx = torch.tensor([3, -1, 39, 0, 3, -7, 17], device="cuda")
    ldo = E + (4 if aligned else 1)
    buf = torch.full((len(idx) * ldo + (0 if aligned else 1),), float("nan"), device="cuda")
    out = buf[(0 if aligned else 1):].as_strided((len(idx), E), (ldo, 1))
    if not aligned:
        table = _misaligned(40, E, 7, ints=False)
    vec = E % 4 == 0 and ldo % 4 == 0 and table.data_ptr() % 16 == 0 and out.data_ptr() % 16 == 0
    assert vec == (E % 4 == 0 and aligned)
    _cabi().call("caphn_gather_rows", table.data_ptr(), idx.data_ptr(), len(idx), E, out.data_ptr(), ldo, _st())
    want = torch.where((idx >= 0)[:, None], table[idx.clamp_min(0)], torch.zeros(1, device="cuda"))
    assert torch.equal(out, want)
    gaps = torch.ones_like(buf, dtype=torch.bool)
    gaps[(0 if aligned else 1):].as_strided((len(idx), E), (ldo, 1)).fill_(False)
    assert bool(torch.isnan(buf[gaps]).all())


@gpu
@pytest.mark.parametrize("T", [1, 2, 5])
@pytest.mark.parametrize("mode", [0, 1])
def test_build_inputs(mode, T):
    ops = _ops()
    B, E, Vv = 6, 37, 20
    emb = torch.randn(Vv, E, generator=R._gen(1)).cuda()
    feat = torch.randn(B, E, generator=R._gen(2)).cuda() if mode == 0 else None
    caps = torch.randint(0, Vv, (B, T), generator=R._gen(3)).cuda()
    caps[:, 0] = Vv - 1
    X = ops.build_inputs(feat, emb, caps, mode).view(T, B, E)
    want = torch.zeros(T, B, E, device="cuda")
    for tt in range(T):
        if mode == 0:
            want[tt] = feat if tt == 0 else emb[caps[:, tt - 1]]
        elif tt >= 2:
            want[tt] = emb[caps[:, tt - 1]]
    assert torch.equal(X, want)
    if mode == 1 and T <= 2:
        assert float(X.abs().max()) == 0.0


def _scatter_idx(n, rows, seed):
    """Indices with duplicates (rows 0 and rows - 1 several times) and a few negatives."""
    idx = torch.randint(0, rows, (n,), generator=R._gen(seed))
    idx[::4] = 0
    idx[1::7] = rows - 1
    idx[2::9] = -1
    return idx


SCATTER_CASES = [(50, 64, 9), (33, 150, 5), (7, 3, 2), (300, 512, 40)]


@gpu
@pytest.mark.parametrize("case", SCATTER_CASES)
@pytest.mark.parametrize("aligned", [True, False])
def test_scatter_add_rows(case, aligned):
    ops = _ops()
    n, E, rows = case
    idx = _scatter_idx(n, rows, 3)
    ldx = E + (4 if aligned else 3)
    for data in ("int", "float"):
        src = (_int_data((n, ldx), 4) if data == "int" else torch.randn(n, ldx, generator=R._gen(4)).cuda())[:, :E]
        tb0 = _int_data((rows, E), 6) if data == "int" else torch.randn(rows, E, generator=R._gen(6)).cuda()
        tbuf = torch.empty(rows * E + 1, device="cuda")
        table = tbuf[(0 if aligned else 1):][:rows * E].view(rows, E)
        table.copy_(tb0)
        vec = E % 4 == 0 and src.data_ptr() % 16 == 0 and table.data_ptr() % 16 == 0
        assert vec == (E % 4 == 0 and aligned)
        ops.scatter_add_rows(src, idx.cuda(), table)
        ref = R.scatter_ref(tb0, idx.cuda(), src)
        if data == "int":
            assert torch.equal(table.double(), ref)
        else:
            absum = R.scatter_ref(tb0.abs(), idx.cuda(), src.abs())
            e = float(((table.double() - ref).abs() / absum.clamp_min(1e-30)).max())
            report(f"scatter_add_rows n={n} E={E} aligned={aligned}: {e:.2e} of the sum of |terms|")
            assert e <= ACC_REL


@gpu
@pytest.mark.parametrize("E", [64, 150, 3])
@pytest.mark.parametrize("t0", [1, 2])
@pytest.mark.parametrize("T", [1, 2, 3, 7])
def test_embed_scatter_add(T, t0, E):
    ops = _ops()
    B, Vv = 9, 11
    caps = torch.randint(0, Vv, (B, T), generator=R._gen(T + E)).cuda()
    caps[::2] = 4                                                         # duplicate tokens across the batch
    for data in ("int", "float"):
        dX = _int_data((T * B, E), 8) if data == "int" else torch.randn(T * B, E, generator=R._gen(8)).cuda()
        dEmb0 = _int_data((Vv, E), 9) if data == "int" else torch.randn(Vv, E, generator=R._gen(9)).cuda()
        dEmb = dEmb0.clone()
        ops.embed_scatter_add(dX, caps, dEmb, t0)
        ref, absum = dEmb0.double().clone(), dEmb0.double().abs()
        for tt in range(t0, T):
            ref.index_add_(0, caps[:, tt - 1], dX.view(T, B, E)[tt].double())
            absum.index_add_(0, caps[:, tt - 1], dX.view(T, B, E)[tt].double().abs())
        if T <= t0:
            assert torch.equal(dEmb, dEmb0)
        if data == "int":
            assert torch.equal(dEmb.double(), ref)
        else:
            e = float(((dEmb.double() - ref).abs() / absum.clamp_min(1e-30)).max())
            report(f"embed_scatter_add T={T} t0={t0} E={E}: {e:.2e} of the sum of |terms|")
            assert e <= ACC_REL


COLSUM_CASES = [(1, 1), (7, 129), (38005, 100), (80001, 100), (160003, 3), (65536, 1200), (10240, 150), (300, 257),
                (37000, 100)]


@gpu
@pytest.mark.parametrize("case", COLSUM_CASES, ids=[f"M{M}-N{N}" for M, N in COLSUM_CASES])
def test_colsum(case):
    ops = _ops()
    M, N = case
    rpb, gy = R.colsum_rpb(M, N)
    assert rpb in (16, 32, 64, 128, 256) and gy <= 65535
    ld = N + 3
    for data in ("int", "float"):
        Xb = _int_data((M, ld), M + N) if data == "int" else torch.randn(M, ld, generator=R._gen(M + N)).cuda()
        X = Xb[:, :N]
        out0 = _int_data((N,), 1) if data == "int" else torch.randn(N, generator=R._gen(1)).cuda()
        out = ops.colsum(X, out0.clone())                                 # accumulates into out
        ref = out0.double() + X.double().sum(0)
        if data == "int":
            assert torch.equal(out.double(), ref)
        else:
            e = float(((out.double() - ref).abs() / (X.double().abs().sum(0) + out0.double().abs())).max())
            report(f"colsum M={M} N={N} rpb={rpb}: {e:.2e} of the sum of |x|")
            assert e <= ACC_REL


GROUP_CASES = [(10, 1, [3, 0, 5, 2]), (9, 3, [0, 9]), (20, 4, [1, 1, 7, 0, 11]), (130, 2, [65, 64, 1])]


def _group_abs(X, goff, B, T):
    return R.group_colsum_ref(X.abs(), goff, B, T)


@gpu
@pytest.mark.parametrize("case", GROUP_CASES)
def test_group_colsum(case):
    ops = _ops()
    B, T, sizes = case
    G, N = len(sizes), 300
    goff = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32)
    ldx, ldo = N + 5, N + 9
    for data in ("int", "float"):
        Xb = _int_data((T * B, ldx), B) if data == "int" else torch.randn(T * B, ldx, generator=R._gen(B)).cuda()
        X = Xb[:, :N]
        obuf = torch.full((G, ldo), float("nan"), device="cuda")
        obuf[:, :N] = 0
        ops.group_colsum(X, goff.cuda(), G, B, T, obuf[:, :N])
        ref = R.group_colsum_ref(X, goff, B, T)
        assert bool(torch.isnan(obuf[:, N:]).all())
        if data == "int":
            assert torch.equal(obuf[:, :N].double(), ref)
        else:
            e = float(((obuf[:, :N].double() - ref).abs() / (_group_abs(X, goff, B, T) + 1e-30)).max())
            report(f"group_colsum B={B} T={T} sizes={sizes}: {e:.2e} of the sum of |x|")
            assert e <= ACC_REL


MEAN_CASES = [(3, 1, 129), (2, 49, 2048), (4, 70, 257), (5, 49, 1), (2, 70, 255)]


@gpu
@pytest.mark.parametrize("case", MEAN_CASES)
@pytest.mark.parametrize("with_extra", [True, False])
def test_mean_pos(case, with_extra):
    ops = _ops()
    Bm, P, Fd = case
    g = R._gen(P * Fd)
    X = torch.randn(Bm, P, Fd, generator=g).cuda()
    m = ops.mean_pos(X)
    # P - 1 adds and one division in fp32: at most (P + 1) 2^-24 of mean |x|
    e = float(((m.double() - X.double().mean(1)).abs() / (X.double().abs().mean(1) + 1e-30)).max())
    report(f"mean_pos B={Bm} P={P} F={Fd}: {e:.2e} of mean |x|")
    assert e <= (P + 1) * 2.0 ** -24
    gg = torch.randn(Bm, Fd, generator=g).cuda()
    dX0 = torch.randn(Bm, P, Fd, generator=g).cuda()
    ex = torch.randn(Bm, P, Fd, generator=g).cuda() if with_extra else None
    dX = ops.mean_pos_bwd(gg, dX0.clone(), ex)                            # += into dX
    ref = R.mean_pos_bwd_ref(gg, dX0, ex)
    # the roundings of 1 / P, of g * (1 / P) and of the two adds
    bound = 4 * 2.0 ** -24 * (dX0.double().abs() + (gg.double().abs() / P)[:, None] + (ex.double().abs() if ex is not None else 0))
    assert bool(((dX.double() - ref).abs() <= bound).all())


@gpu
@pytest.mark.parametrize("n", [1, 255, 256, 257, 1000])
def test_masks(n):
    ops = _ops()
    specials = torch.tensor([float("nan"), 0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, float("inf"), -float("inf"), 1.0, -2.5],
                            device="cuda")
    y = torch.randn(n, generator=R._gen(n)).cuda()
    y[:min(n, len(specials))] = specials[:n]
    ref = torch.randn(n, generator=R._gen(n + 1)).cuda()
    ref[-min(n, len(specials)):] = specials[:n]
    slope = torch.tensor(0.01, dtype=torch.float32, device="cuda")

    def same(a, b):
        return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a[~torch.isnan(a)].view(torch.int32),
                                                                           b[~torch.isnan(b)].view(torch.int32))
    buf = torch.full((n + 1,), 7.0, device="cuda")                        # one element past the end: must stay 7
    buf[:n] = y
    ops.relu_mask_(ref, buf[:n])
    assert same(buf[:n], torch.where(ref > 0, y, torch.zeros(1, device="cuda"))) and buf[n].item() == 7.0
    buf[:n] = y
    ops.leaky_relu_(buf[:n])
    assert same(buf[:n], torch.where(y > 0, y, y * slope)) and buf[n].item() == 7.0
    dy = torch.randn(n, generator=R._gen(n + 2)).cuda()
    buf[:n] = dy
    ops.leaky_relu_bwd_(y, buf[:n])
    assert same(buf[:n], torch.where(y > 0, dy, dy * slope)) and buf[n].item() == 7.0


PAD_CASES = [(1, 1, 4, 4), (31, 33, 32, 36), (32, 32, 32, 32), (33, 65, 64, 68), (70, 3, 72, 4), (5, 150, 8, 152)]


@gpu
@pytest.mark.parametrize("case", PAD_CASES, ids=[f"R{a}-C{b}" for a, b, _, _ in PAD_CASES])
def test_pad_builders(case):
    ops = _ops()
    Rr, C, ldt, ldc = case                       # ldt >= R (transpose pitch), ldc >= C (copy pitch)
    srcb = torch.randn(Rr, C + 3, generator=R._gen(Rr * C)).cuda()
    src = srcb[:, :C]                            # row pitch C + 3
    t = ops.transpose_pad(src, ldt)
    want = torch.zeros(C, ldt, device="cuda")
    want[:, :Rr] = src.t()
    assert torch.equal(t, want)
    c = ops.copy_pad(src, ldc)
    want = torch.zeros(Rr, ldc, device="cuda")
    want[:, :C] = src
    assert torch.equal(c, want)
    for nb in (1, 3):
        S = torch.randn(nb, Rr * C, generator=R._gen(nb)).cuda()
        Sv = S.view(nb, Rr, C)
        want_t = torch.zeros(nb, C, ldt, device="cuda")
        want_t[:, :, :Rr] = Sv.transpose(1, 2)
        want_c = torch.zeros(nb, Rr, ldc, device="cuda")
        want_c[:, :, :C] = Sv
        assert torch.equal(ops.transpose_pad_batched(S, Rr, C, ldt), want_t)
        assert torch.equal(ops.copy_pad_batched(S, Rr, C, ldc), want_c)


@gpu
def test_pad_batched_limits_and_refusals():
    ops = _ops()
    C_ = _cabi()
    S = torch.randn(65535, 6, generator=R._gen(1)).cuda()
    tb = ops.transpose_pad_batched(S, 2, 3, 4)
    cb = ops.copy_pad_batched(S, 2, 3, 4)
    V = S.view(65535, 2, 3)
    want_t = torch.zeros(65535, 3, 4, device="cuda")
    want_t[:, :, :2] = V.transpose(1, 2)
    want_c = torch.zeros(65535, 2, 4, device="cuda")
    want_c[:, :, :3] = V
    assert torch.equal(tb, want_t) and torch.equal(cb, want_c)
    S2 = torch.zeros(65536, 6, device="cuda")
    with pytest.raises(C_.CaphnError):
        ops.transpose_pad_batched(S2, 2, 3, 4)
    with pytest.raises(C_.CaphnError):
        ops.copy_pad_batched(S2, 2, 3, 4)
    d = torch.zeros(2 * 3 * 4, device="cuda")
    with pytest.raises(C_.CaphnError):                                     # dstride < C * ldd
        C_.call("caphn_transpose_pad_batched", S.data_ptr(), 6, 3, d.data_ptr(), 11, 4, 2, 2, 3, _st())
    with pytest.raises(C_.CaphnError):                                     # dstride < R * ldd
        C_.call("caphn_copy_pad_batched", S.data_ptr(), 6, 3, d.data_ptr(), 7, 4, 2, 2, 3, _st())
