"""The two GEMMs -- tcgen05 tensor-core kernel (csrc/gemm_tc.cu) and exact-fp32 SIMT kernel (csrc/gemm_simt.cu) -- and the
bf16x3 operand builders against float64 (tests/gemm_ref.py) at every cell their host plans dispatch on.

Dispatch table of caphn_gemm_tc_ex / _scaled / _amax (gemm_tc_impl; restated as gemm_ref.tc_plan, pinned by the CPU
tests below; tm = ceil(M / 128), "waves" counted at BN = 128 against 8 x 148 tiles):

    row            condition                                             BN / schedule                 host code
    one-tile-16    N <= 256, B K-major                                   round16(N)                    N <= 256 branch
    one-tile-64    N <= 256, B MN-major                                  round64(N)                    N <= 256 branch
    few-waves      N > 256, tm ceil(N/128) <= 1184                       argmin over 128..256 (step    few_waves loop
                                                                         16, 64 for MN-major B) of
                                                                         ceil(tiles/148) (BN + 32):
                                                                         M = 512, N = 9684: 144 with
                                                                         TMEM 512 and TMA-store /
                                                                         register chunks mixed;
                                                                         M = 1000: 192; M = 1920: 256
    many-256       N > 256, > 1184 tiles, A slab + 3 B stages do not     256 (2 stages at K = 193)     !few_waves, !astat_fits
                   fit (K > 192 bf16x3 / 576 bf16), an MN-major
                   operand, or CAPHN_TC_ASTAT=0
    many-128       N > 256, > 1184 tiles, slab fits, < 4 n-tiles         128, round robin              astat_shape false
    astat          K-major operands, splitk 1, >= 4 n-tiles,             A slab resident, B ring;      astat_shape
                   >= 592 tiles, slab + fixed + 3 B stages fit           (also in the few-waves row:   + smem check
                   (bf16 mode: up to 6 stages)                           bf16, M = 1024, N = 18944)
    split-K auto   not ReLU, tiles < 444: smallest s (<= 32,             kb_per = ceil(kb / s),        splitk <= 0 loop
                   <= kb / 4) filling >= 90 % of 148 SMs, else the       splits of kb_per k-blocks
                   best by > 2 %: dH (10240, 150, 9684) 5,
                   [dW | db] (9684, 151, 10240) 9
    split-K given  requested s > num_kb collapses to num_kb;             ceil(kb / ceil(kb / s))       kb_per / splitk
                   s = 3 at kb = 10: 4 / 4 / 2
    epilogue       splitk 1, ldc % 4 = 0, N % 4 = 0, C 16-B aligned:     TMA store of full 32-column   tma_store
                   TMA store (chunks narrower than 32 tile columns:     chunks, else vector / scalar
                   registers); else ldc % 4 = 0 and C aligned: float4   register stores, or red.v4 /
                   stores; else scalar; split-K: red.v4 / red.v2 /      .v2 / scalar atomics per row
                   scalar atomics by row address alignment; memset of   alignment
                   C, 2-D when ldc != N
    K tail         the last k-block issues ceil(rem / 16) k-steps        ksteps                        MMA issuer
    TMEM           256 columns when 2 BN <= 256, else 512                tmem_cols
    stages         min(6, (227 KiB - fixed [- slab]) / stage bytes)      stages

Grouped mode (caphn_gemm_tc_grouped) takes every tile from a 12-word unit record (a_row, b_row, ka0, kb0, nkb, m_valid,
n_valid, bias_off, map0, c_lo, c_hi); GroupPlan builds them (units_xproj / units_dx / units_dw) and _dev_units packs the
64-bit C offset as a signed low word and a high word.  caphn_gemm_f32 runs ceil(K / kchunk) K slices,
kchunk = round16(ceil(K / splitk)), with atomics under split-K or accumulate.

Which test reaches each cell: every row -> test_exact_sweep (placement and lo-term data, both precisions, bias / ReLU /
scale rotated, CAPHN_TC_ASTAT=0 and CAPHN_TC_TMA_STORE=0 where those paths differ) and test_swept_shapes_land_in_their_cells
(plan pinned on the CPU) + test_library_picks_the_planned_n_tile (BN read back through caphn_gemm_tc_amax's nparts);
boundaries -> test_plan_boundaries; K residues 1..15 in the last k-block x all four majorness pairs, pitch padding that
holds NaN -> test_k_edges_all_majorness; ldc = 0 / 1 / 2 / 3 (mod 4), unaligned C, 1-D and 2-D memset, den = 0 ->
test_strided_outputs; accuracy on float data -> test_accuracy_float_data, test_accuracy_vocabulary_chain; grouped ->
test_grouped_plan_units, test_grouped_hand_built_units, test_grouped_large_c_offset; builders -> test_split_bf16*;
SIMT -> test_gemm_f32; refusals -> test_refusals; planted defects -> test_planted_defects_*.

Exact data (gemm_ref docstring) must come out bit for bit, and every element of the output buffer outside [M, N] must
still hold the NaN sentinel.  Float data is checked per element against |A| |B|^T (gemm_ref.elem_err): TOL is set per
precision and K band; gemm_ref.bound_tc is the analytic ceiling (3 2^-16 + (3 ceil(K/16) + 2) 2^-23 in bf16x3).

Worst elem_err measured on one NVIDIA B200 (1000 W power limit), with the analytic bound in brackets:
    bf16x3  K <= 256     5.3e-6 (M = 300, N = 150, K = 150; the logits product 4.0e-6)           [5.0e-5]
            K <= 2048    8.8e-7 (M = 2000, N = 150, K = 2048, MN-major A)                         [9.2e-5]
            K <= 10240   3.1e-6 ([dW | db], K = 10240; dH 1.6e-6 at K = 9684)                     [2.8e-4]
    bf16    K <= 256     1.6e-3 (M = 1000, N = 9684, K = 150)                                     [7.8e-3]
            K <= 2048    3.7e-4 (M = 700, N = 150, K = 1536, both MN-major)                       [7.9e-3]
The errors stay an order of magnitude or more below the bound because the truncation errors of the accumulator adds
are not all of one sign.  The longest-K band is worse than the middle one only on the vocabulary chain, whose
gradient operand has rows of very different magnitude.  The new tests found no kernel defect.  A copy of the kernel
that skips the last k-step of the K tail fails the exact sweep and every majorness pair of test_k_edges_all_majorness.
The file's GPU tests take about 5 s on the B200."""
import numpy as np
import pytest
import torch

import gemm_ref as R
from golden_util import report

gpu = pytest.mark.gpu
ENV = ("CAPHN_TC_BN_FORCE", "CAPHN_TC_ASTAT", "CAPHN_TC_TMA_STORE")

# per-element tolerance per (precision, largest K of the band), 3-4x the worst error measured (module docstring)
TOL = {("bf16x3", 256): 2e-5, ("bf16x3", 2048): 3e-6, ("bf16x3", 10240): 1.2e-5, ("bf16", 256): 6e-3, ("bf16", 2048): 1.5e-3}


def tol(K, split=True):
    mode = "bf16x3" if split else "bf16"
    return TOL[(mode, min(k for (m, k) in TOL if m == mode and k >= K))]


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


# ----------------------------------------------------------------------------------------------------------------------
# the swept shapes and the cell each lands in
# ----------------------------------------------------------------------------------------------------------------------
# (row, M, N, K, options, plan fields).  options: a_mn, b_mn, split (default True), splitk (default 0 = auto), env
# ("astat0" / "tma0").  Each entry runs with placement data, and with lo-term data when K <= 4095.
SWEEP = [
    ("one-tile-16", 300, 150, 150, {}, dict(BN=160, splitk=1, epi="scalar", tmem_cols=512, ksteps_last=2)),
    ("one-tile-16", 129, 1, 17, {}, dict(BN=16, splitk=1, epi="scalar", tmem_cols=256, ksteps_last=2)),
    ("one-tile-16", 127, 17, 1, {"split": False}, dict(BN=32, splitk=1, epi="scalar", ksteps_last=1)),
    ("one-tile-16", 255, 48, 65, {}, dict(BN=48, splitk=1, epi="tma+reg", ksteps_last=1)),
    ("one-tile-64", 200, 130, 100, {"b_mn": True}, dict(BN=192, splitk=1, epi="scalar", tmem_cols=512)),
    ("one-tile-64", 130, 64, 129, {"a_mn": True, "b_mn": True, "split": False}, dict(BN=64, splitk=1, epi="tma")),
    ("few-waves", 512, 9684, 150, {}, dict(BN=144, few_waves=True, splitk=1, astat=False, epi="tma+reg", tmem_cols=512)),
    ("few-waves", 512, 9684, 150, {"env": "tma0"}, dict(BN=144, splitk=1, epi="vec")),
    ("few-waves", 1000, 9684, 150, {}, dict(BN=192, few_waves=True, splitk=1, units_per_cta=3)),
    ("few-waves", 1000, 9684, 150, {"b_mn": True}, dict(BN=192, few_waves=True, splitk=1)),
    ("few-waves", 1920, 9684, 150, {}, dict(BN=256, few_waves=True, astat=False, stages=2, units_per_cta=4)),
    ("few-waves", 1024, 18944, 64, {"split": False}, dict(BN=256, few_waves=True, astat=True, stages=5, tiles=592)),
    ("few-waves", 1024, 18688, 64, {"split": False}, dict(BN=256, few_waves=True, astat=False, tiles=584)),
    ("few-waves", 1024, 18944, 64, {"split": False, "env": "astat0"}, dict(BN=256, astat=False)),
    ("many-256", 1921, 9684, 193, {}, dict(BN=256, few_waves=False, astat=False, stages=2, ksteps_last=1)),
    ("many-256", 1921, 9684, 150, {"a_mn": True}, dict(BN=256, few_waves=False, astat=False)),
    ("many-256", 1921, 9684, 577, {"split": False}, dict(BN=256, astat=False, stages=4)),
    ("many-256", 1921, 9684, 150, {"env": "astat0"}, dict(BN=256, astat=False)),
    ("many-128", 50433, 384, 64, {}, dict(BN=128, few_waves=False, astat=False, tiles=1185)),
    ("astat", 1921, 9684, 150, {}, dict(BN=128, few_waves=False, astat=True, stages=3, units_per_cta=9)),
    ("astat", 1921, 9684, 192, {}, dict(BN=128, astat=True, stages=3, ksteps_last=4)),
    ("astat", 1921, 9684, 576, {"split": False}, dict(BN=128, astat=True, stages=3)),
    ("astat", 1921, 9684, 150, {"split": False}, dict(BN=128, astat=True, stages=6)),
    ("astat", 1921, 9684, 150, {"env": "tma0"}, dict(BN=128, astat=True, epi="vec")),
    ("astat", 50433, 385, 64, {}, dict(BN=128, astat=True, epi="scalar", tiles=1580)),
    ("split-K auto", 10240, 150, 9684, {}, dict(BN=160, splitk=5, splits=[31] * 4 + [28], epi="atomic", memset="1d")),
    ("split-K auto", 512, 150, 9684, {"split": False}, dict(BN=160, epi="atomic")),
    ("split-K auto", 256, 150, 2048, {}, dict(BN=160, splitk=8, epi="atomic")),
    ("split-K given", 640, 100, 600, {"splitk": 3}, dict(BN=112, splitk=3, splits=[4, 4, 2], ksteps_last=2)),
    ("split-K given", 128, 100, 150, {"splitk": 50}, dict(splitk=3, splits=[1, 1, 1])),
]


def _plan_of(M, N, K, o, ldc=None, c_align=16, relu=False):
    env = o.get("env")
    return R.tc_plan(M, N, K, o.get("a_mn", False), o.get("b_mn", False), o.get("split", True),
                     1 if relu else o.get("splitk", 0), relu, ldc, c_align, astat_on=env != "astat0",
                     tma_on=env != "tma0")


def _sweep_id(e):
    row, M, N, K, o, _ = e
    tags = [k if v is True else f"{k}{v}" for k, v in sorted(o.items()) if v is not False]
    return f"{row}-{M}x{N}x{K}" + ("-" + "-".join(tags) if tags else "") + ("" if o.get("split", True) else "-bf16")


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the plan's boundaries and the swept shapes' cells
# ----------------------------------------------------------------------------------------------------------------------
def test_plan_boundaries():
    P = R.tc_plan
    # few / many waves flips at tm ceil(N / 128) = 1184 / 1185
    a, b = P(1920, 9684, 150), P(1921, 9684, 150)
    assert (a["few_waves"], a["BN"], a["astat"]) == (True, 256, False)
    assert (b["few_waves"], b["BN"], b["astat"]) == (False, 128, True)
    # the A slab: bf16x3 up to K = 192, then BN 256 with 2 stages; bf16 up to K = 576
    assert P(1921, 9684, 192)["astat"] and not P(1921, 9684, 193)["astat"]
    assert (P(1921, 9684, 193)["BN"], P(1921, 9684, 193)["stages"]) == (256, 2)
    assert P(1921, 9684, 576, split=False)["astat"] and not P(1921, 9684, 577, split=False)["astat"]
    assert P(1921, 9684, 577, split=False)["BN"] == 256
    # astat needs >= 4 n-tiles (N = 385 vs 384 at 395 m-tiles) and >= 592 tiles (bf16 few-waves, BN 256: 592 vs 584)
    assert P(50433, 385, 64)["astat"] and not P(50433, 384, 64)["astat"]
    assert P(50433, 384, 64)["BN"] == 128 and not P(50433, 384, 64)["few_waves"]
    assert P(1024, 18944, 64, split=False)["astat"] and not P(1024, 18688, 64, split=False)["astat"]
    assert not P(1921, 9684, 150, a_mn=True)["astat"] and P(1921, 9684, 150, a_mn=True)["BN"] == 256
    assert not P(1921, 9684, 150, astat_on=False)["astat"] and P(1921, 9684, 150, astat_on=False)["BN"] == 256
    # the decode product and M = 1000
    d = P(512, 9684, 150)
    assert (d["BN"], d["tmem_cols"], d["tiles"], d["epi"]) == (144, 512, 272, "tma+reg")
    assert P(1000, 9684, 150)["BN"] == 192 and P(1000, 9684, 150, b_mn=True)["BN"] == 192
    assert P(128, 130, 64, b_mn=True)["BN"] == 192 and P(128, 130, 64)["BN"] == 144
    # the vocabulary chain of the benchmark
    assert P(10240, 9684, 150)["astat"] and P(10240, 9684, 150)["epi"] == "tma"
    dh = P(10240, 150, 9684)
    assert (dh["BN"], dh["splitk"], dh["kb_per"], dh["memset"]) == (160, 5, 31, "1d")
    dw = P(9684, 151, 10240, a_mn=True, ldc=152)
    assert (dw["BN"], dw["splitk"], dw["memset"], dw["epi"]) == (160, 9, "2d", "atomic")
    # requested split-K: collapse to num_kb, uneven splits, ReLU refused
    assert P(128, 100, 150, splitk=50)["splits"] == [1, 1, 1]
    assert P(640, 100, 600, splitk=3)["splits"] == [4, 4, 2]
    assert P(640, 100, 600, splitk=2, relu=True) is None
    assert P(640, 100, 600, relu=True)["splitk"] == 1
    # TMA store: splitk 1, ldc % 4 == 0, N % 4 == 0, 16-byte aligned C
    assert P(300, 160, 150)["epi"] == "tma"
    assert P(300, 160, 150, ldc=162)["epi"] == "scalar" and P(300, 160, 150, ldc=164)["epi"] == "tma"
    assert P(300, 158, 150, ldc=160)["epi"] == "vec" and P(300, 160, 150, c_align=4)["epi"] == "scalar"
    assert P(300, 160, 150, splitk=2)["epi"] == "atomic" and P(300, 160, 150, tma_on=False)["epi"] == "vec"
    # K tail: k-steps of the last k-block
    assert [P(128, 16, K)["ksteps_last"] for K in (1, 15, 16, 17, 63, 64, 65, 129)] == [1, 1, 1, 2, 4, 4, 1, 1]
    # grid and units per CTA
    assert P(10240, 9684, 150)["grid"] == 148 and P(1000, 9684, 150)["units_per_cta"] == 3


@pytest.mark.parametrize("entry", SWEEP, ids=_sweep_id)
def test_swept_shapes_land_in_their_cells(entry):
    row, M, N, K, o, fields = entry
    p = _plan_of(M, N, K, o)
    assert {k: p[k] for k in fields} == fields, (row, p)
    if "splitk" in o:
        cell = "split-K given"
    elif p["splitk"] > 1:
        cell = "split-K auto"
    elif p["few_waves"] is None:
        cell = "one-tile-64" if o.get("b_mn") else "one-tile-16"
    elif p["few_waves"]:
        cell = "few-waves"
    elif p["astat"]:
        cell = "astat"
    else:
        cell = "many-256" if p["BN"] == 256 else "many-128"
    assert cell == row, (row, cell, p)


def test_f32_plan():
    assert R.f32_plan(100, 6) == (32, 4) and R.f32_plan(100, 7) == (16, 7) and R.f32_plan(17, 1) == (32, 1)
    assert R.f32_plan(1, 0) == (16, 1) and R.f32_plan(256, 3) == (96, 3)


# ----------------------------------------------------------------------------------------------------------------------
# CPU: planted defects
# ----------------------------------------------------------------------------------------------------------------------
MUTANT_SHAPES = [(300, 150, 150, {}), (300, 40, 65, {}), (256, 150, 2048, {}), (640, 100, 600, {"splitk": 3})]


def _mutant_cases(mutant, data):
    for M, N, K, o in MUTANT_SHAPES:
        p = _plan_of(M, N, K, o)
        need = R.mutant_needs(mutant)
        if need == "splitk" and p["splitk"] < 2 or need == "two m-tiles" and M <= R.BM:
            continue
        if need == "split" and data == "placement":
            continue
        mk = {"placement": R.placement_operand, "lo-term": R.loterm_operand, "float": R.float_operand}[data]
        a, b = mk(M, K, 11), mk(N, K, 12)
        bias = R.int_bias(N, 3) if data != "float" else torch.randn(N, generator=torch.Generator().manual_seed(3))
        num = 3.0 if data == "placement" else 2.0
        scale = (num, 4.0) if need in ("den", "splitk") or mutant == "last K-tail step dropped" else None
        yield a, b, p, bias, scale, K


@pytest.mark.parametrize("mutant", R.MUTANTS)
def test_planted_defects_fail_the_exact_comparison(mutant):
    n = 0
    for data in ("placement", "lo-term"):
        for a, b, p, bias, scale, K in _mutant_cases(mutant, data):
            ref = R.epilogue(R.product(a, b), bias, scale)
            mut = R.mutate(mutant, a, b, p, True, bias, scale)
            M, N = ref.shape
            buf, _ = R.out_buffer(M, N, N + 1, device="cpu")          # column N lies outside the output: sentinel
            exp = R.expected_buffer(buf, N + 1, 0, ref)
            got = exp.clone()
            got[N + 1:].as_strided(mut.shape, (N + 1, 1)).copy_(mut.float())
            assert R.mismatches(got, exp) > 0, (mutant, data, M, N, K)
            n += 1
    assert n >= 2, mutant


@pytest.mark.parametrize("mutant", [m for m in R.MUTANTS if m != "write one column past n_valid"])
def test_planted_defects_exceed_the_float_tolerance(mutant):
    ratios = []
    for a, b, p, bias, scale, K in _mutant_cases(mutant, "float"):
        ref = R.epilogue(R.product(a, b), bias, scale)
        exact = R.epilogue(a.double() @ b.double().t(), bias, scale)
        mut = R.mutate(mutant, a, b, p, True, bias, scale)
        ratios.append(R.elem_err(mut, exact, a, b, bias, scale) / tol(K))
        assert R.elem_err(ref, exact, a, b, bias, scale) <= R.bound_tc(K)
    assert ratios, mutant
    report(f"gemm mutant {mutant!r}: smallest margin {min(ratios):.0f}x the tolerance over {len(ratios)} shapes")
    assert min(ratios) > 10, f"{mutant}: moves the output by only {min(ratios):.1f}x the tolerance"


def test_exact_data_is_exact():
    """The premise of the exact sweep: the split of lo-term data is (h, l) exactly, and hh + hl + lh of K = 4095 is an
    fp32 number."""
    x = R.loterm_operand(64, 4095, 1)
    hi, lo = R.split_ref(x)
    assert torch.equal(hi.double() + lo.double(), x.double())
    assert bool(hi.float().abs().log2().frac().eq(0).all())
    c = R.product(x[:8], x[8:16])
    assert torch.equal(c.float().double(), c)
    p = R.placement_operand(4, 10240, 2)
    assert float(p.abs().max()) <= 8 and bool((p[:, -1] != 0).all())


# ----------------------------------------------------------------------------------------------------------------------
# GPU: exact sweep
# ----------------------------------------------------------------------------------------------------------------------
EPIS = [dict(), dict(bias=True), dict(bias=True, relu=True), dict(scale=(3.0, 4.0)), dict(bias=True, scale=(3.0, 0.0)),
        dict(scale=(3.0, None))]
EPIS_P2 = [dict(), dict(bias=True), dict(bias=True, relu=True), dict(scale=(2.0, 4.0)), dict(bias=True, scale=(2.0, 0.0)),
           dict(scale=(0.5, None))]


def run_exact(M, N, K, a_mn=False, b_mn=False, split=True, splitk=0, data="placement", bias=False, relu=False,
              scale=None, ldc=None, col0=0, pad_ld=False, seed=0):
    """One tensor-core GEMM on exact data into a sentinel-filled buffer; returns (mismatching elements, output view,
    float64 reference)."""
    ops = _ops()
    dev = "cuda"
    mk = R.placement_operand if data == "placement" else R.loterm_operand
    a, b = mk(M, K, seed, dev), mk(N, K, seed + 1, dev)
    lda = R.round64(M if a_mn else K) + 8 if pad_ld else None
    ldb = R.round64(N if b_mn else K) + 8 if pad_ld else None
    A, B = R.place(a, a_mn, split, lda, pad=R.NAN_BF16), R.place(b, b_mn, split, ldb, pad=R.NAN_BF16)
    bias_t = R.int_bias(N, seed, dev) if bias else None
    ldc = ldc or N
    buf, view = R.out_buffer(M, N, ldc, col0)
    sc = None
    if scale is not None:
        sc = (torch.tensor([scale[0]], device=dev), None if scale[1] is None else torch.tensor([scale[1]], device=dev))
    ops.gemm_tc(A, B, bias=bias_t, relu=relu, out=view, splitk=splitk, scale=sc)
    torch.cuda.synchronize()
    ref = R.epilogue(R.product(a, b, split), bias_t, scale, relu)
    exp = R.expected_buffer(buf, ldc, col0, ref)
    return R.mismatches(buf, exp), view, ref


@gpu
@pytest.mark.parametrize("data", ["placement", "lo-term"])
@pytest.mark.parametrize("i", range(len(SWEEP)), ids=[_sweep_id(e) for e in SWEEP])
def test_exact_sweep(i, data, monkeypatch):
    row, M, N, K, o, _ = SWEEP[i]
    if data == "lo-term" and K > 4095:
        pytest.skip("lo-term data is exact for K <= 4095 only")
    if o.get("env") == "astat0":
        monkeypatch.setenv("CAPHN_TC_ASTAT", "0")
    if o.get("env") == "tma0":
        monkeypatch.setenv("CAPHN_TC_TMA_STORE", "0")
    epi = dict((EPIS if data == "placement" else EPIS_P2)[(i + (data == "lo-term")) % len(EPIS)])
    plan = _plan_of(M, N, K, o, relu=epi.get("relu", False))
    assert plan is not None
    bad, _, _ = run_exact(M, N, K, o.get("a_mn", False), o.get("b_mn", False), o.get("split", True), o.get("splitk", 0),
                          data, seed=i, **epi)
    assert bad == 0, f"{row}: {bad} elements differ ({epi}, plan {plan})"


@gpu
@pytest.mark.parametrize("split", [True, False], ids=["bf16x3", "bf16"])
@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (True, False), (False, True), (True, True)])
def test_k_edges_all_majorness(a_mn, b_mn, split):
    """K residues 1..15 of the last k-block (and K < 64, K = 64 + 1, 2 k-blocks + 1), two m-tiles with a 2-row tail,
    operand pitches round64 + 8 whose padding holds NaN; bias and scale alternate."""
    for j, K in enumerate((1, 15, 16, 17, 63, 64, 65, 129)):
        for data in ("placement", "lo-term"):
            epi = [dict(bias=True), dict(scale=(2.0, 4.0))][j % 2]
            bad, _, _ = run_exact(130, 40, K, a_mn, b_mn, split, data=data, pad_ld=True, seed=K, **epi)
            assert bad == 0, (K, data, epi)


@gpu
@pytest.mark.parametrize("M,N,K,splitk", [(256, 150, 2048, 0), (300, 150, 150, 1), (640, 100, 600, 3)])
def test_strided_outputs(M, N, K, splitk):
    """Row pitches 0 / 1 / 2 / 3 (mod 4) and a C offset by one float: TMA store, vector and scalar register stores, and
    under split-K red.v4 / red.v2 / scalar atomics and the 1-D / 2-D memset; den = 0 scales by num."""
    for ldc in (N, R.round16(N), R.round16(N) + 1, R.round16(N) + 2, R.round16(N) + 3):
        for col0 in (0, 1):
            p = R.tc_plan(M, N, K, splitk=splitk, ldc=ldc, c_align=4 if col0 else 16)
            scale = (3.0, 0.0) if col0 else (3.0, 4.0)
            for data in ("placement", "lo-term"):
                bad, _, _ = run_exact(M, N, K, splitk=splitk, data=data, bias=True, scale=scale if data == "placement"
                                      else (2.0, 0.0), ldc=ldc, col0=col0, seed=ldc + col0)
                assert bad == 0, (ldc, col0, data, p["epi"], p["memset"])


@gpu
def test_library_picks_the_planned_n_tile():
    """caphn_gemm_tc_amax returns nparts = 2 ceil(N / BN): the library's BN for every swept shape whose candidate widths
    give different tile counts (amax runs without split-K; BN does not depend on it)."""
    import ctypes
    from hypernet_image_captioning_b200 import _cabi
    ops = _ops()
    seen = set()
    for row, M, N, K, o, _ in SWEEP:
        key = (M, N, K, o.get("a_mn", False), o.get("b_mn", False), o.get("split", True), o.get("env"))
        if key in seen:
            continue
        seen.add(key)
        p = _plan_of(M, N, K, o)
        a_mn, b_mn, split = key[3:6]
        A = R.place(torch.zeros(M, K, device="cuda"), a_mn, split)
        B = R.place(torch.zeros(N, K, device="cuda"), b_mn, split)
        out = torch.empty(M, N, device="cuda")
        ld = 2 * R.cdiv(N, 16)
        pv = torch.empty(M, ld, device="cuda")
        pi = torch.empty(M, ld, device="cuda", dtype=torch.int32)
        env = {"astat0": ("CAPHN_TC_ASTAT", "0"), "tma0": ("CAPHN_TC_TMA_STORE", "0")}.get(o.get("env"))
        mp = pytest.MonkeyPatch()
        if env:
            mp.setenv(*env)
        n = ctypes.c_int(0)
        try:
            _cabi.call("caphn_gemm_tc_amax", A.hi.data_ptr(), None if A.lo is None else A.lo.data_ptr(), A.ld, int(a_mn),
                       B.hi.data_ptr(), None if B.lo is None else B.lo.data_ptr(), B.ld, int(b_mn), K, out.data_ptr(), N,
                       None, M, N, pv.data_ptr(), pi.data_ptr(), ld, ctypes.byref(n), torch.cuda.current_stream().cuda_stream)
        finally:
            mp.undo()
        torch.cuda.synchronize()
        assert n.value == 2 * R.cdiv(N, p["BN"]), (row, M, N, K, o, p["BN"], n.value)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: float data, per-element error
# ----------------------------------------------------------------------------------------------------------------------
ACC_SHAPES = [(300, 150, 150, False, False, True), (1000, 9684, 150, False, False, True),
              (1921, 9684, 150, False, False, True), (1921, 9684, 193, False, False, True),
              (700, 150, 1536, True, True, True), (2000, 150, 2048, True, False, True),
              (512, 150, 9684, False, False, True), (450, 200, 10240, False, True, True),
              (300, 150, 150, False, False, False), (1000, 9684, 150, False, False, False),
              (700, 150, 1536, True, True, False)]


@gpu
@pytest.mark.parametrize("M,N,K,a_mn,b_mn,split", ACC_SHAPES)
def test_accuracy_float_data(M, N, K, a_mn, b_mn, split):
    a, b = R.float_operand(M, K, M + K, "cuda"), R.float_operand(N, K, N + 2 * K, "cuda")
    bias = torch.randn(N, device="cuda", generator=torch.Generator("cuda").manual_seed(N))
    out = _ops().gemm_tc(R.place(a, a_mn, split), R.place(b, b_mn, split), bias=bias)
    torch.cuda.synchronize()
    exact = a.double() @ b.double().t() + bias.double()
    e = R.elem_err(out, exact, a, b, bias)
    report(f"gemm accuracy {'bf16x3' if split else 'bf16'} M={M} N={N} K={K} a_mn={a_mn} b_mn={b_mn}: elem_err {e:.3e} "
           f"(tolerance {tol(K, split):.2e}, bound {R.bound_tc(K, split):.2e})")
    assert e <= tol(K, split) and e <= R.bound_tc(K, split)


@gpu
def test_accuracy_vocabulary_chain():
    """The benchmark's vocabulary products at full size, with the operand layout of functional.vocab_bwd_fused: logits
    (10240, 9684, 150) + bias; dH (10240, 150, 9684) and [dW | db] (9684, 151, 10240) from the unscaled gradient operand
    read K-major and MN-major, scaled by num / max(den, 1) with den = lossbuf[1:]."""
    ops = _ops()
    M, V, H = 10240, 9684, 150
    dev = "cuda"
    Hbm, fc_w, d = R.float_operand(M, H, 1, dev), R.float_operand(V, H, 2, dev), R.float_operand(M, V, 3, dev)
    fc_b = torch.randn(V, device=dev, generator=torch.Generator(dev).manual_seed(4))
    logits = ops.gemm_tc(ops.split_bf16(Hbm), ops.split_bf16(fc_w), bias=fc_b)
    gscale, lossbuf = torch.tensor([1.0], device=dev), torch.tensor([2.5, 7.0], device=dev)
    sp = ops.split_bf16(d)
    dop, dT = ops.SplitOperand(sp.hi, sp.lo, M, V, sp.ld), ops.SplitOperand(sp.hi, sp.lo, V, M, sp.ld, True)
    scale = (gscale, lossbuf[1:])
    dH = ops.gemm_tc(dop, ops.split_bf16_t(fc_w), scale=scale)
    wb = torch.empty(V, ops.round4(H + 1), device=dev)[:, :H + 1]
    ops.gemm_tc(dT, ops.split_bf16_t(Hbm, ones_row=True), scale=scale, out=wb)
    torch.cuda.synchronize()
    sc = (1.0, 7.0)
    H1 = torch.cat([Hbm, torch.ones(M, 1, device=dev)], 1)
    errs = {"logits": R.elem_err(logits, Hbm.double() @ fc_w.double().t() + fc_b.double(), Hbm, fc_w, fc_b),
            "dH": R.elem_err(dH, (d.double() @ fc_w.double()) / 7.0, d, fc_w.t(), scale=sc),
            "dW|db": R.elem_err(wb, (d.double().t() @ H1.double()) / 7.0, d.t(), H1.t(), scale=sc)}
    for name, K in (("logits", H), ("dH", V), ("dW|db", M)):
        report(f"gemm accuracy vocabulary chain {name} (K = {K}): elem_err {errs[name]:.3e} (tolerance {tol(K):.2e}, "
               f"bound {R.bound_tc(K):.2e})")
        assert errs[name] <= tol(K) and errs[name] <= R.bound_tc(K), name


# ----------------------------------------------------------------------------------------------------------------------
# GPU: grouped mode
# ----------------------------------------------------------------------------------------------------------------------
def _gather_rows(x, gm2tm):
    out = torch.zeros(gm2tm.numel(), x.shape[1], device=x.device)
    ok = gm2tm >= 0
    out[ok] = x[gm2tm[ok].long()]
    return out


@gpu
@pytest.mark.parametrize("split", [True, False], ids=["bf16x3", "bf16"])
@pytest.mark.parametrize("data", ["placement", "lo-term"])
@pytest.mark.parametrize("T,cnt", [(1, [0, 1, 63, 64, 65, 0, 129]), (3, [1, 21, 0, 43])], ids=["T1", "T3"])
def test_grouped_plan_units(T, cnt, data, split):
    """x-projection, dX and dW through GroupPlan's unit tables against per-group float64 products: groups of 0 and 1
    rows, T cnt = 63 / 64 / 65 / 129, 3H = 150 (a K range that ends inside a k-block), E + F = 70."""
    from hypernet_image_captioning_b200.grouped import GroupPlan
    ops = _ops()
    dev = "cuda"
    G, E, Fd, H3 = len(cnt), 40, 30, 150
    EF = E + Fd
    g_host = np.random.default_rng(T).permutation(np.repeat(np.arange(G), cnt))
    plan = GroupPlan(g_host, G, T, dev)
    B = len(g_host)
    # lo-term data without the per-row 2^s: the dW products sum over time-major rows, where a row scale would lie along
    # K and take the partial sums past 24 bits
    mk = R.placement_operand if data == "placement" else lambda r, k, s, d: R.loterm_operand(r, k, s, d, exps=False)
    W = mk(G * H3, EF, 1, dev)                       # W_ih of every group, [G * 3H, E + F]
    bg = R.int_bias(G * H3, 2, dev)
    X = mk(T * B, EF, 3, dev)                        # [x | ctx] per time-major row (t * B + b, b in the sorted batch)
    dGI = mk(T * B, H3, 4, dev)
    gm2tm = plan.gm2tm
    g_of_row = torch.from_numpy(np.tile(np.sort(g_host), T)).to(dev)      # group of each time-major row
    Wsp = R.place(W, False, split)
    prod = lambda x, w: R.product(x, w, split)

    # x-projection: GIw[row] = X[row, :E] W[g][:, :E]^T + b[g], rows scattered through gm2tm
    Xgm = R.place(_gather_rows(X[:, :E].contiguous(), gm2tm), False, split)
    buf, GIw = R.out_buffer(T * B, H3, H3, device=dev)
    ops.gemm_tc_grouped(Xgm, False, Wsp, False, GIw, H3, plan.units_xproj(H3, E, 128), 128, bias=bg, rowmap=gm2tm)
    # dX[row] = dGI[row] W[g][:, :E]   (B read MN-major from the same split, k rows g 3H ..)
    dGIgm = R.place(_gather_rows(dGI, gm2tm), False, split)
    Wmn = ops.SplitOperand(Wsp.hi, Wsp.lo, EF, G * H3, Wsp.ld, True)
    buf2, dX = R.out_buffer(T * B, E, E, device=dev)
    ops.gemm_tc_grouped(dGIgm, False, Wmn, True, dX, E, plan.units_dx(H3, E, 128), 128, rowmap=gm2tm)
    # dW[g] = dGI_g^T X_g over the group's padded K range, written at dTheta[g, 0:]
    theta = H3 * EF + 16
    XCgm = R.place(_gather_rows(X, gm2tm), False, split)
    mn = lambda op: ops.SplitOperand(op.hi, op.lo, op.K, op.rows, op.ld, True)
    buf3, dTheta = R.out_buffer(G, theta, theta, device=dev)
    ops.gemm_tc_grouped(mn(dGIgm), True, mn(XCgm), True, dTheta, EF, plan.units_dw(H3, EF, 128, theta, 0, EF), 128)
    torch.cuda.synchronize()

    ref1 = torch.empty(T * B, H3, dtype=torch.float64, device=dev)
    ref2 = torch.empty(T * B, E, dtype=torch.float64, device=dev)
    ref3 = torch.full((G, theta), float("nan"), dtype=torch.float64, device=dev)
    for g in range(G):
        rows = (g_of_row == g).nonzero().flatten()
        Wg = W[g * H3:(g + 1) * H3]
        if rows.numel() == 0:
            continue
        ref1[rows] = prod(X[rows, :E], Wg[:, :E].contiguous()) + bg[g * H3:(g + 1) * H3].double()
        ref2[rows] = prod(dGI[rows], Wg[:, :E].t().contiguous())
        ref3[g, :H3 * EF] = prod(dGI[rows].t().contiguous(), X[rows].t().contiguous()).reshape(-1)
    assert R.mismatches(buf, R.expected_buffer(buf, H3, 0, ref1)) == 0
    assert R.mismatches(buf2, R.expected_buffer(buf2, E, 0, ref2)) == 0
    exp3 = R.expected_buffer(buf3, theta, 0, ref3)          # absent groups and the tail of each row: sentinel (NaN ref)
    exp3.view(torch.int32)[exp3 != exp3] = R.SENTINEL
    assert R.mismatches(buf3, exp3) == 0


@gpu
@pytest.mark.parametrize("split", [True, False], ids=["bf16x3", "bf16"])
@pytest.mark.parametrize("data", ["placement", "lo-term"])
def test_grouped_hand_built_units(data, split):
    """Unit records the planners do not make: m_valid = 1, n_valid = 1, nkb = 1, ka0 != kb0, a rowmap with negative
    entries (those rows keep the sentinel), bias_off not a multiple of BN; against the record semantics in float64."""
    from hypernet_image_captioning_b200.grouped import GroupPlan
    ops = _ops()
    dev = "cuda"
    mk = R.placement_operand if data == "placement" else R.loterm_operand
    A = R.place(mk(300, 200, 5, dev), False, split)
    Bop = R.place(mk(100, 200, 6, dev), False, split)
    BN, ldc = 112, 130
    bias = R.int_bias(256, 7, dev)
    rowmap = torch.tensor([400 + r if r % 3 else -1 for r in range(128)], dtype=torch.int32, device=dev)
    rows = [(0, 0, 0, 0, 4, 128, 100, 0, 0, 0, 0, 0),                         # a full tile, K through a zero-padded block
            (128, 10, 0, 0, 1, 1, 50, 5, 0, 130 * ldc + 3, 0, 0),             # m_valid 1, nkb 1, bias_off 5
            (200, 40, 64, 128, 1, 100, 1, 17, 0, 140 * ldc + 120, 0, 0),      # n_valid 1, ka0 != kb0
            (64, 0, 0, 0, 4, 128, 112, 131, 0, 10, 0, 0)]                     # through the rowmap (added below)
    plan = GroupPlan(np.zeros(1, np.int64), 1, 1, dev)
    units = plan._dev_units(("hand", data, split), rows[:3])
    umap = plan._dev_units(("hand-map", data, split), rows[3:])
    C = torch.empty(600 * ldc, dtype=torch.int32, device=dev).fill_(R.SENTINEL).view(torch.float32)
    ops.gemm_tc_grouped(A, False, Bop, False, C, ldc, units, BN, bias=bias)
    ops.gemm_tc_grouped(A, False, Bop, False, C, ldc, umap, BN, bias=bias, rowmap=rowmap)
    torch.cuda.synchronize()
    ref = torch.full((600 * ldc,), float("nan"), dtype=torch.float64, device=dev)
    ref = R.grouped_ref(A, False, Bop, False, ref, ldc, units, BN, bias)
    ref = R.grouped_ref(A, False, Bop, False, ref, ldc, umap, BN, bias, rowmap.cpu())
    exp = ref.float()
    exp.view(torch.int32)[exp != exp] = R.SENTINEL
    assert R.mismatches(C, exp) == 0


@gpu
@pytest.mark.parametrize("off", [2 ** 31 + 4099, 2 ** 32 + 4099], ids=["2^31", "2^32"])
def test_grouped_large_c_offset(off):
    """One unit whose C offset does not fit 31 bits (8.6 GB / 17 GB output): _dev_units packs it as a signed low word and
    a high word, the kernel must write exactly the 5 x 16 tile there."""
    from hypernet_image_captioning_b200.grouped import GroupPlan
    ops = _ops()
    ldc, n = 64, off + 8 * 64
    if torch.cuda.mem_get_info()[0] < 2 * 4 * n:
        pytest.skip(f"needs {2 * 4 * n / 1e9:.1f} GB of free device memory")
    A = R.place(R.placement_operand(128, 64, 1, "cuda"), False, True)
    Bop = R.place(R.placement_operand(16, 64, 2, "cuda"), False, True)
    plan = GroupPlan(np.zeros(1, np.int64), 1, 1, "cuda")
    units = plan._dev_units(("big", off), [(0, 0, 0, 0, 1, 5, 16, 0, 0, off, 0, 0)])
    assert int(units[0, 9]) == (off & 0xFFFFFFFF) - (2 ** 32 if off & 0x80000000 else 0) and int(units[0, 10]) == off >> 32
    C = torch.empty(n, dtype=torch.int32, device="cuda").fill_(R.SENTINEL).view(torch.float32)
    ops.gemm_tc_grouped(A, False, Bop, False, C, ldc, units, 16)
    torch.cuda.synchronize()
    ref = R.product(R.placement_operand(128, 64, 1, "cuda")[:5], R.placement_operand(16, 64, 2, "cuda"))
    got = C[off:off + 5 * ldc].view(5, ldc)
    assert torch.equal(got[:, :16].double(), ref)
    assert bool((got[:, 16:].view(torch.int32) == R.SENTINEL).all())
    written = sum(int((C[i:i + (1 << 28)].view(torch.int32) != R.SENTINEL).sum()) for i in range(0, n, 1 << 28))
    assert written == 5 * 16
    del C
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------------------------------------------------
# GPU: operand builders, bit for bit
# ----------------------------------------------------------------------------------------------------------------------
def _special(R_, C, seed):
    """Gaussian values of many magnitudes plus RNE ties, subnormals, +-0 and values near the bf16 overflow."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(R_, C, generator=g) * 2.0 ** torch.randint(-30, 30, (R_, C), generator=g).float()
    bits = torch.from_numpy(np.array([0x3F808000, 0x3F818000, 0xBF808000, 0x00000001, 0x80000003, 0x007FFFFF, 0x00800000,
                                      0x00000000, 0x80000000, 0x7F7F7FFF, 0x7F7F8000, 0x7F7FFFFF, 0xFF7FFFFF, 0x3F80FFFF,
                                      0x3F807FFF, 0x00018000], dtype=np.uint32).view(np.int32))
    flat = x.view(-1)
    idx = torch.randperm(flat.numel(), generator=g)[:min(flat.numel(), 4 * bits.numel())]
    flat[idx] = bits.repeat(4)[:idx.numel()].view(torch.float32)
    return x


def _same_bits(a, b):
    return torch.equal(a.cpu().view(torch.int16), b.cpu().view(torch.int16))


def _check_split(hi, lo, x, C):
    rh, rl = R.split_ref(x)
    assert _same_bits(hi[:, :C], rh) and _same_bits(lo[:, :C], rl)
    assert int((hi[:, C:].view(torch.int16) != 0).sum()) == 0 and int((lo[:, C:].view(torch.int16) != 0).sum()) == 0


@gpu
@pytest.mark.parametrize("C,extra,shift", [(150, 0, 0), (150, 3, 0), (151, 1, 1), (64, 0, 1), (7, 2, 0)])
def test_split_bf16(C, extra, shift):
    """caphn_split_bf16: the 16-byte-aligned vector path and the scalar path (row pitch % 4 != 0, source one float off)."""
    ops = _ops()
    x = _special(37, C, C + extra)
    big = torch.zeros(37 * (C + extra) + 4, device="cuda")
    src = big[shift:shift + 37 * (C + extra)].view(37, C + extra)[:, :C]
    src.copy_(x.cuda())
    op = ops.split_bf16(src, want_lo=True)
    torch.cuda.synchronize()
    _check_split(op.hi, op.lo, x, C)
    assert ops.split_bf16(src, want_lo=False).lo is None


@gpu
@pytest.mark.parametrize("R_,C", [(70, 45), (33, 1), (128, 64)])
def test_split_bf16_t(R_, C):
    """caphn_split_bf16_t: hi / lo [C, round64(R)] = split(src^T), tails of 32 x 32 tiles, ones_row."""
    ops = _ops()
    x = _special(R_, C, R_ * C)
    op = ops.split_bf16_t(x.cuda(), want_lo=True, ones_row=True)
    torch.cuda.synchronize()
    _check_split(op.hi[:C], op.lo[:C], x.t().contiguous(), R_)
    assert bool((op.hi[C].float() == 1).all()) and int((op.lo[C].view(torch.int16) != 0).sum()) == 0


@gpu
def test_split_bf16_gather_and_batched():
    ops = _ops()
    x = _special(50, 77, 9)
    rowmap = torch.tensor([3, -1, 49, 0, -5, 7, 7, 20], dtype=torch.int32)
    op = ops.split_bf16_gather(x.cuda(), rowmap.cuda(), 8, want_lo=True)
    torch.cuda.synchronize()
    gx = torch.zeros(8, 77)
    gx[rowmap >= 0] = x[rowmap[rowmap >= 0].long()]
    _check_split(op.hi, op.lo, gx, 77)
    # batched: 3 matrices [5, 70] at a stride of 500 floats, rows 90 floats apart
    src = _special(1, 1600, 10).view(-1)
    op = ops.split_bf16_batched(src.cuda(), 500, 90, 3, 5, 70, want_lo=True)
    torch.cuda.synchronize()
    ref = torch.cat([src[b * 500: b * 500 + 5 * 90].view(5, 90)[:, :70] for b in range(3)])
    _check_split(op.hi, op.lo, ref, 70)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the SIMT GEMM
# ----------------------------------------------------------------------------------------------------------------------
F32_CASES = [(130, 129, 17, 1, False, True), (1, 1, 1, 1, False, True), (257, 200, 33, 1, True, False),
             (129, 130, 100, 6, False, True), (300, 45, 100, 7, False, True), (200, 260, 512, 3, True, True)]


def _f32_layout(x, kmajor, extra):
    """x [rows, K] stored K-major ([rows, K + extra]) or MN-major ([K, rows + extra]); returns (tensor, ld)."""
    rows, K = x.shape
    if kmajor:
        buf = torch.zeros(rows, K + extra, device=x.device)
        buf[:, :K] = x
    else:
        buf = torch.zeros(K, rows + extra, device=x.device)
        buf[:, :rows] = x.t()
    return buf, buf.stride(0)


@gpu
@pytest.mark.parametrize("a_k,b_k", [(1, 1), (1, 0), (0, 1), (0, 0)])
@pytest.mark.parametrize("data", ["placement", "float"])
def test_gemm_f32(a_k, b_k, data):
    """caphn_gemm_f32: ragged M / N / K against 128 / 128 / 16, split-K whose kchunk rounding changes the split count
    (K = 100: 6 -> 4), accumulate into a nonzero C, the bias added once under split-K, ReLU; exact data bit for bit,
    float data within the fp32-FMA bound per element."""
    ops = _ops()
    dev = "cuda"
    for j, (M, N, K, sk, acc, relu) in enumerate(F32_CASES):
        mk = R.placement_operand if data == "placement" else R.float_operand
        a, b = mk(M, K, j, dev), mk(N, K, j + 50, dev)
        bias = R.int_bias(N, j, dev) if data == "placement" else torch.randn(N, device=dev)
        A, lda = _f32_layout(a, a_k, 3)
        B, ldb = _f32_layout(b, b_k, 5)
        ldc = N + 3
        buf, out = R.out_buffer(M, N, ldc, device=dev)
        c0 = (R.int_bias(M * N, j + 9, dev) if data == "placement" else torch.randn(M * N, device=dev)).view(M, N)
        relu = relu and not acc and R.f32_plan(K, sk)[1] == 1
        out.copy_(c0 if acc else torch.zeros_like(c0))
        ops._gemm(A, lda, a_k, B, ldb, b_k, M, N, K, bias=bias, relu=relu, out=out, splitk=sk, accumulate=acc)
        torch.cuda.synchronize()
        exact = a.double() @ b.double().t() + bias.double() + (c0.double() if acc else 0)
        if relu:
            exact = exact.clamp_min(0)
        if data == "placement":
            assert R.mismatches(buf, R.expected_buffer(buf, ldc, 0, exact)) == 0, (M, N, K, sk, acc)
        else:
            den = a.double().abs() @ b.double().abs().t() + bias.double().abs() + (c0.double().abs() if acc else 0)
            e = float(((out.double() - exact).abs() / den).max())
            assert e <= R.bound_f32(K, R.f32_plan(K, sk)[1] + acc), (M, N, K, sk, acc, e)
            assert bool((buf.view(torch.int32)[:ldc] == R.SENTINEL).all())


# ----------------------------------------------------------------------------------------------------------------------
# GPU: refusals (each rejected by the host before any launch)
# ----------------------------------------------------------------------------------------------------------------------
@gpu
def test_refusals():
    from hypernet_image_captioning_b200 import _cabi
    ops = _ops()
    st = torch.cuda.current_stream().cuda_stream
    a = R.place(torch.ones(256, 640, device="cuda"), False, True)
    b = R.place(torch.ones(128, 640, device="cuda"), False, True)
    bm = R.place(torch.ones(128, 640, device="cuda"), True, True)
    C = torch.empty(256, 128, device="cuda")
    num = torch.ones(1, device="cuda")

    def ex(*over, **kw):
        args = dict(ah=a.hi.data_ptr(), al=a.lo.data_ptr(), ald=a.ld, bh=b.hi.data_ptr(), bl=b.lo.data_ptr(), relu=0, sk=0)
        args.update(kw)
        return ("caphn_gemm_tc_ex", args["ah"], args["al"], args["ald"], 0, args["bh"], args["bl"], b.ld, 0, 640,
                C.data_ptr(), 128, None, 256, 128, args["relu"], args["sk"], st)

    refused = {
        "ReLU with split-K": ex(relu=1, sk=2),
        "misaligned A hi": ex(ah=a.hi.data_ptr() + 2),
        "misaligned B lo": ex(bl=b.lo.data_ptr() + 8),
        "a_ld % 8 != 0": ex(ald=a.ld - 4),
        "lo of one operand only": ex(al=None),
        "scale_den without scale_num": ("caphn_gemm_tc_scaled", a.hi.data_ptr(), a.lo.data_ptr(), a.ld, 0, b.hi.data_ptr(),
                                        b.lo.data_ptr(), b.ld, 0, 640, C.data_ptr(), 128, None, 256, 128, 0, None,
                                        num.data_ptr(), st),
        "amax_ld below 2 ceil(N / BN)": ("caphn_gemm_tc_amax", a.hi.data_ptr(), a.lo.data_ptr(), a.ld, 0, b.hi.data_ptr(),
                                         b.lo.data_ptr(), b.ld, 0, 640, C.data_ptr(), 128, None, 256, 128, C.data_ptr(),
                                         C.data_ptr(), 1, None, st),
    }
    units = torch.zeros(1, 12, dtype=torch.int32, device="cuda")
    for BN, op, mnb in ((100, b, 0), (8, b, 0), (272, b, 0), (80, bm, 1)):
        refused[f"grouped BN {BN} (B {'MN' if mnb else 'K'}-major)"] = (
            "caphn_gemm_tc_grouped", a.hi.data_ptr(), a.lo.data_ptr(), a.ld, 256, a.ld, 0, op.hi.data_ptr(),
            op.lo.data_ptr(), op.ld, op.hi.shape[0], op.ld, mnb, C.data_ptr(), 128, None, None, units.data_ptr(), 1, BN, st)
    for name, call in refused.items():
        with pytest.raises(_cabi.CaphnError, match="invalid argument"):
            _cabi.call(*call)
    torch.cuda.synchronize()
    # the same arguments, corrected, run
    _cabi.call(*ex(relu=1, sk=1))
    ops.gemm_tc(a, b, out=C)
    torch.cuda.synchronize()
    assert float(C.min()) == 640.0 and float(C.max()) == 640.0
