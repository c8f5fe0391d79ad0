"""The hypernetwork parameter path -- weight-streaming layers (csrc/hn_rows.cu), gradient norm and Adam (csrc/optim.cu)
-- against a float64 reference (tests/hypernet_ref.py) at every shape their plans dispatch on.

Dispatch table (V = 4 fp32 / 8 bf16 elements per 128-bit vector; the functions on the right are restated below as
fwd_plan / bwd_plan / *_grid, and the CPU tests pin their thresholds):

    forward G-chunks     ops.rows_linear_fwd splits G into calls of <= 8; each call   rows_linear_fwd_t
                         runs chunks of 8 / 4 / 2 / 1, each halved while
                         gc * V * (ceil(K/V) + 2) * 4 B > 200 KB:
                           fp32  gc = 8 up to K = 6392, 4 to 12792, 2 to 25592
                           bf16  gc = 8 up to K = 6384, 4 to 12784, 2 to 25584
    forward K limit      gc = 1 needs V * (ceil(K/V) + 2) * 4 B <= 227 KB:            launch_rows_fwd
                         K <= 58104 (fp32) / 58096 (bf16), above: CaphnError
    forward fetch        NQ = ceil((K + m) / V) vectors per row, 128 per batch:       rows_fwd_kernel
                         NQ > 128 runs the pipelined second fetch; N > 16 x grid
                         (grid min(ceil(N/16), 148 occ)) wraps rows over the grid
    backward G-chunks    4 / 2 / 1 in that order, chunks after the first              rows_linear_bwd_t
                         accumulate into dW; G <= 64, G = 65 refused
    backward (QPL, RU)   fp32 gc 4 / 2 / 1: (1,4) (2,2) (4,2);                        rows_linear_bwd_t
                         bf16 gc 4 / 2 / 1: (1,2) (1,4) (2,4)
    backward regime      S = ceil(((K + 2(V-1)) div V) / (32 QPL)) strips;            launch_rows_bwd
                         "tiny" when N K < 2^22, else "many" when S >= 8, else "few"
                         (the benchmark's K = 1600 at G = 1 is few-strips: S = 4)
    misalignment classes ncls = V / gcd(K mod V, V): fp32 1 / 2 / 4, bf16 1 / 2 / 4 / 8 rows_bwd_kernel
    sumsq                float4 loop unrolled x4 once n/4 > 3 x stride,               caphn_sumsq / opt_grid
                         stride = 256 min(ceil(n/4 / 512), 2368): from n = 7 274 500;
                         n % 4 tail apart; bf16: 8 per vector, n % 8 tail apart
    dense Adam           pairs (i, i + stride), `two` false on the last half-pass;    caphn_adam_step / opt_grid
                         grid-stride wrap once n/4 > 2 x 256 x 2368 (from n = 4 849 668)
    bf16 Adam            one 8-vector per iteration, stride 256 min(ceil(n/8 / 512),  caphn_adam_step_bf16 / opt_grid
                         2368): a second iteration per thread once n/8 > 256
                         (from n = 2056), a third once n/8 > 2 x 256 x 2368
                         (from n = 9 699 336); n % 8 tail apart
    lowrank Adam         grid min(n4 / 1024 + 1, 1184) x 256 threads, 4 float4 per   caphn_adam_step_lowrank
                         thread: wraps once N K > 4 x 4 x 256 x 1184 = 4 849 664;
                         float4s straddle rows when K % 4 != 0; total % 4 tail apart

Which test reaches each cell: forward G-chunks and K limit -> test_forward_g_chunks, test_forward_refuses_k_above_limit;
fetch / residues / wrap / strided -> test_forward_shapes, test_forward_rows_wrap_the_grid; backward regimes x classes x
(QPL, RU) -> test_backward_regimes_and_classes; G-chunks and mixed regimes -> test_backward_g_chunks,
test_backward_refuses_g_65; dA-only / no dA / accumulate / strided -> test_backward_options; sumsq / gram / clip ->
test_sumsq*, test_gram_and_lowrank_norm, test_clip_coef; dense / bf16 Adam -> test_adam_dense, test_adam_bf16;
lowrank Adam -> test_adam_lowrank; the benchmark's head shapes -> test_drift_*.

Outputs are compared one by one with rel_err = max|kernel - ref| / max|ref| (elementwise against one scale), except the
bf16 dW, which is checked per element against the rounding bound of its chunks (bf16_dw_ratio), and p == bf16(master)
of the bf16 Adam step, which is bit for bit.

Worst rel_err over all cases of this file on one NVIDIA B200 (1000 W power limit), drift tests included; each bound in
BOUNDS is 3 to 4x the worst error of its output:
    Y 1.05e-6 (bf16, K = 58096; 3.5e-7 at N = 90000, K = 11250), dP 1.0e-9, dbias 2.2e-7, dW (fp32) 1.4e-7 (G = 64),
    dA 5.2e-7 (1.41e-6 at N = 90000, K = 11250), bf16 dW 0.995 of its rounding bound (G = 1: one rounding, the bound
    is reached); sumsq 4.4e-8, sumsq_bf16 3.2e-8, gram 2.8e-8, ||dP^T A||^2 4.0e-8, clip coefficient 6.9e-8, norm 4.5e-8;
    dense Adam p 4.8e-8, m 1.6e-7, v 9.2e-8; bf16 Adam master 4.9e-8, m 9.4e-8, v 8.7e-8; lowrank Adam p 5.1e-8,
    m 1.3e-7, v 9.8e-8 (one step at N = 90000, K = 11250: 3.9e-8, 1.0e-7, 7.5e-8)."""
import math
import zlib

import pytest
import torch

import hypernet_ref as R
from golden_util import report

gpu = pytest.mark.gpu

# rel_err bounds (module docstring).  Forward / backward are fp32 FMA chains against float64; Adam is a handful of fp32
# operations per element.
BOUNDS = {"Y": 4e-6, "dP": 4e-9, "dbias": 8e-7, "dW": 5e-7, "dA": 5e-6, "sumsq": 1.5e-7, "gram": 1e-7, "frob": 1.5e-7,
          "coef": 2.5e-7, "p": 2e-7, "m": 6e-7, "v": 4e-7, "master": 2e-7}

FWD_CAP, FWD_SMEM = 200 * 1024, 227 * 1024
NUM_SMS, BWD_WARPS = 148, 8
BWD_QPL_RU = {(torch.float32, 4): (1, 4), (torch.float32, 2): (2, 2), (torch.float32, 1): (4, 2),
              (torch.bfloat16, 4): (1, 2), (torch.bfloat16, 2): (1, 4), (torch.bfloat16, 1): (2, 4)}
DTYPES = (torch.float32, torch.bfloat16)
DNAME = {torch.float32: "fp32", torch.bfloat16: "bf16"}


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ----------------------------------------------------------------------------------------------------------------------
# the host plans, restated
# ----------------------------------------------------------------------------------------------------------------------
def fwd_plan(dtype, G, K):
    """gc of every chunk of one caphn_rows_linear_fwd call (G <= 8), or None when the call is refused."""
    V = R.vec_width(dtype)
    per_g = V * ((K + V - 1) // V + 2) * 4
    out, g0 = [], 0
    while g0 < G:
        gc = 8 if G - g0 >= 8 else (4 if G - g0 >= 4 else (2 if G - g0 >= 2 else 1))
        while gc > 1 and gc * per_g > FWD_CAP:
            gc >>= 1
        if gc * per_g > FWD_SMEM:
            return None
        out.append(gc)
        g0 += gc
    return out


def fwd_k_limits(dtype):
    """The largest K of each gc (8, 4, 2, 1)."""
    return [_largest(lambda K: fwd_plan(dtype, gc, K) == [gc]) for gc in (8, 4, 2, 1)]


def _largest(ok, lo=1, hi=1 << 20):
    """Largest K in [lo, hi) with ok(K), for a predicate true up to some K and false above."""
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if ok(mid) else (lo, mid)
    return lo


def ncls(dtype, K):
    V = R.vec_width(dtype)
    return V // math.gcd(K % V, V)


def bwd_plan(dtype, G, N, K):
    """[(gc, regime)] of one caphn_rows_linear_bwd call: regime "tiny" / "many" / "few" (launch_rows_bwd)."""
    V = R.vec_width(dtype)
    out = []
    for _, gc in R.bwd_chunks(G):
        qpl, _ = BWD_QPL_RU[(dtype, gc)]
        S = (((K + 2 * (V - 1)) // V) + 32 * qpl - 1) // (32 * qpl)
        out.append((gc, "tiny" if N * K < (1 << 22) else ("many" if S >= 8 else "few")))
    return out


def opt_grid(n4):
    return max(1, min((n4 + 511) // 512, NUM_SMS * 16))


def dense_adam_wraps(n):
    return n // 4 > 2 * 256 * opt_grid(n // 4)


def bf16_adam_iterations(n):
    """Loop iterations of the busiest thread of adam_bf16_kernel (one 8-vector each)."""
    n8 = n // 8
    return -(-n8 // (256 * opt_grid(n8))) if n8 else 0


def sumsq_unrolled(n):
    return n // 4 > 3 * 256 * opt_grid(n // 4)


def lowrank_wraps(N, K):
    n4 = N * K // 4
    return n4 > 4 * 256 * min(n4 // 1024 + 1, NUM_SMS * 8)


# ----------------------------------------------------------------------------------------------------------------------
# comparison
# ----------------------------------------------------------------------------------------------------------------------
def rel(got, ref):
    """rel_err on the device, in row chunks (the large outputs stay on the GPU)."""
    got, ref = got.reshape(got.shape[0], -1) if got.dim() > 1 else got[None], \
        ref.reshape(ref.shape[0], -1) if ref.dim() > 1 else ref[None]
    ref = ref.to(got.device)
    d = s = 0.0
    step = max(1, R.CHUNK_ELEMS // max(1, got.shape[1]))
    for r0 in range(0, got.shape[0], step):
        rr = ref[r0:r0 + step].double()
        d = max(d, (got[r0:r0 + step].double() - rr).abs().max().item())
        s = max(s, rr.abs().max().item())
    return d / s if s > 0 else d


def bf16_dw_ratio(got, ref, dP, A):
    """bf16 dW per element against its rounding bound: every G-chunk rounds the running sum to bf16 (half an ulp,
    <= 2^-8 of sum_g |dP_g A_g|), plus the fp32 accumulation.  Returns max |got - ref| / bound (must be < 1)."""
    nch = len(R.bwd_chunks(dP.shape[0]))
    worst = 0.0
    step = max(1, R.CHUNK_ELEMS // A.shape[1])
    for r0 in range(0, got.shape[0], step):
        S = dP[:, r0:r0 + step].double().abs().t() @ A.double().abs()
        lim = nch * 2.0 ** -8 * S + 1e-6 * S.max()
        worst = max(worst, ((got[r0:r0 + step].double() - ref[r0:r0 + step]).abs() / lim).max().item())
    return worst


def compare(errs, where, bounds=None):
    bounds = bounds or BOUNDS
    report(f"{where}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    bad = {k: e for k, e in errs.items() if not e < (1.0 if k == "dW_bf16" else bounds[k])}
    assert not bad, f"{where}: " + ", ".join(f"{k} {e:.3e}" for k, e in sorted(bad.items()))


def _seed(*xs):
    return zlib.crc32(repr(xs).encode()) & 0x7fffffff


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the plans' thresholds
# ----------------------------------------------------------------------------------------------------------------------
def test_forward_chunk_limits():
    assert fwd_k_limits(torch.float32) == [6392, 12792, 25592, 58104]
    assert fwd_k_limits(torch.bfloat16) == [6384, 12784, 25584, 58096]
    assert fwd_plan(torch.float32, 7, 1600) == [4, 2, 1]
    assert fwd_plan(torch.float32, 8, 6393) == [4, 4]
    assert fwd_plan(torch.float32, 8, 25593) == [1] * 8
    assert fwd_plan(torch.float32, 1, 58105) is None and fwd_plan(torch.bfloat16, 1, 58097) is None


def test_backward_regime_thresholds():
    f, b = torch.float32, torch.bfloat16
    assert bwd_plan(f, 1, 11250, 1600) == [(1, "few")]            # the benchmark's first head layers (E = 200)
    assert bwd_plan(f, 1, 90000, 11250) == [(1, "many")]
    assert bwd_plan(f, 1, 2621, 1600) == [(1, "tiny")] and bwd_plan(f, 1, 2622, 1600) == [(1, "few")]
    assert bwd_plan(f, 5, 2700, 1600) == [(4, "many"), (1, "few")]
    assert bwd_plan(b, 5, 2700, 2001) == [(4, "many"), (1, "few")]
    assert [gc for gc, _ in bwd_plan(f, 7, 1, 1)] == [4, 2, 1] and len(bwd_plan(f, 64, 1, 1)) == 16
    assert [ncls(f, K) for K in (8, 6, 5, 7)] == [1, 2, 4, 4]
    assert [ncls(b, K) for K in (16, 12, 10, 9, 11250, 8437)] == [1, 2, 4, 8, 4, 8]


def test_optimizer_grid_thresholds():
    assert not dense_adam_wraps(4_849_664) and dense_adam_wraps(4_849_668)
    assert not sumsq_unrolled(7_274_496) and sumsq_unrolled(7_274_500)
    assert [bf16_adam_iterations(n) for n in (2055, 2056, 4099, 4_849_671, 9_699_335, 9_699_337)] == [1, 2, 2, 2, 2, 3]
    assert not lowrank_wraps(4_849_664, 1) and lowrank_wraps(4_849_668, 1)
    assert lowrank_wraps(90000, 11250) and not lowrank_wraps(300, 11250) and lowrank_wraps(600, 8437)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: forward
# ----------------------------------------------------------------------------------------------------------------------
def _fwd_check(d, G, N, K, dtype, act, where, bias=True, out=None, lda=None):
    """``lda``: the row stride A must reach the kernel with (inputs built on the device: a copy would be dense)."""
    ops = _ops()
    W, A = d["W"].cuda(), d["A"].cuda()
    assert A.stride(0) == (lda or K), f"{where}: A has row stride {A.stride(0)}"
    b = d["b"].cuda() if bias else None
    Y = ops.rows_linear_fwd(W, b, A, act, out=out)
    torch.cuda.synchronize()
    ref = R.rows_fwd(W, b, A, act)
    compare({"Y": rel(Y, ref)}, where)
    return Y


FWD_LIMIT_K = {torch.float32: [6392, 6393, 12792, 12793, 25592, 25593, 58104],
               torch.bfloat16: [6384, 6385, 12784, 12785, 25584, 25585, 58096]}


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DNAME.get)
@pytest.mark.parametrize("ki", range(7))
def test_forward_g_chunks(dtype, ki):
    """G = 1..8 on both sides of every gc boundary and at the largest accepted K."""
    K, N = FWD_LIMIT_K[dtype][ki], 37
    d = R.rows_inputs(8, N, K, dtype, _seed("fwd-g", K))
    for G in range(1, 9):
        dd = dict(d, A=d["A"][:G])
        _fwd_check(dd, G, N, K, dtype, 1, f"fwd {DNAME[dtype]} G={G} K={K} chunks {fwd_plan(dtype, G, K)}")


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DNAME.get)
def test_forward_refuses_k_above_limit(dtype):
    from hypernet_image_captioning_b200._cabi import CaphnError
    K = FWD_LIMIT_K[dtype][-1] + 1
    assert fwd_plan(dtype, 1, K) is None
    with pytest.raises(CaphnError):
        _ops().rows_linear_fwd(torch.zeros(3, K, device="cuda", dtype=dtype), None, torch.zeros(1, K, device="cuda"))
    torch.cuda.synchronize()


def _fwd_shapes(dtype):
    V = R.vec_width(dtype)
    return [1] + list(range(2, V + 2)) + [V * 130 + r for r in range(V)]       # K < V, K = 1, NQ > 128, every residue


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DNAME.get)
def test_forward_shapes(dtype):
    """Every K mod V, K < V, K = 1 and NQ > 128; act 0 / 1, bias None, A with lda > K, and Y written into a
    sentinel-filled theta buffer at an odd column offset: nothing outside the slice may change."""
    G, N = 3, 50
    for K in _fwd_shapes(dtype):
        d = R.rows_inputs(G, N, K, dtype, _seed("fwd-shape", K), "cuda", lda=K + 3)
        _fwd_check(d, G, N, K, dtype, 1, f"fwd {DNAME[dtype]} K={K} lda={K + 3} act=1", lda=K + 3)
        theta = torch.full((G, N + 20), 7.25, device="cuda")
        Y = _fwd_check(d, G, N, K, dtype, 0, f"fwd {DNAME[dtype]} K={K} lda={K + 3} act=0 no bias, theta[:, 7:]",
                       bias=False, out=theta[:, 7:7 + N], lda=K + 3)
        assert Y.data_ptr() == theta[:, 7:].data_ptr()
        assert bool((theta[:, :7] == 7.25).all()) and bool((theta[:, 7 + N:] == 7.25).all()), \
            f"K={K}: the forward wrote outside its slice of theta"


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DNAME.get)
def test_forward_rows_wrap_the_grid(dtype):
    """N = 20011 rows at K = 37: more rows than warps in the grid (592 CTAs x 16 warps)."""
    G, N, K = 2, 20011, 37
    d = R.rows_inputs(G, N, K, dtype, _seed("fwd-wrap", N))
    _fwd_check(d, G, N, K, dtype, 1, f"fwd {DNAME[dtype]} N={N} K={K}")


# ----------------------------------------------------------------------------------------------------------------------
# GPU: backward
# ----------------------------------------------------------------------------------------------------------------------
def bwd_errors(got, ref, dtype, dP_in, A):
    errs = {"dP": rel(got["dP"], ref["dP"]), "dbias": rel(got["dbias"], ref["dbias"])}
    if got.get("dW") is not None:
        if dtype == torch.bfloat16:
            errs["dW_bf16"] = bf16_dw_ratio(got["dW"], ref["dW"], ref["dP"], A)
        else:
            errs["dW"] = rel(got["dW"], ref["dW"])
    if got.get("dA") is not None:
        errs["dA"] = rel(got["dA"], ref["dA"])
    return errs


def _bwd_check(d, dtype, act, where, need_dW=True, need_dA=True, dA0=True, bounds=None):
    ops = _ops()
    W, A, Y, dY = d["W"].cuda(), d["A"].cuda(), d["Y"].cuda(), d["dY"].cuda()
    dA = d["dA0"].cuda().clone() if (dA0 and need_dA) else None
    dW, db, dA, dP = ops.rows_linear_bwd(W, A, Y if act else None, dY, act, need_dW=need_dW, need_dA=need_dA, dA=dA,
                                         return_dP=True)
    torch.cuda.synchronize()
    ref = R.rows_bwd(W, A, Y, dY, act, dA0=d["dA0"].cuda() if (dA0 and need_dA) else None, need_dW=need_dW)
    got = {"dP": dP, "dbias": db, "dW": dW, "dA": dA}
    compare(bwd_errors(got, ref, dtype, dY, A), where, bounds)


def regime_shape(dtype, gc, regime, r):
    """(N, K) with K % V == r that puts a gc-chunk in ``regime``."""
    V = R.vec_width(dtype)
    qpl, _ = BWD_QPL_RU[(dtype, gc)]
    if regime == "tiny":
        K = 200 + r
        return 300, K
    K = (256 * qpl * V + r) if regime == "many" else (1600 + r if bwd_plan(dtype, gc, 1 << 22, 1600)[0][1] == "few"
                                                      else 640 + r)
    return (1 << 22) // K + 5, K


def class_residues(dtype):
    """One K mod V per misalignment class count: fp32 0, 2, 1 (ncls 1, 2, 4); bf16 0, 4, 2, 1 (1, 2, 4, 8)."""
    return (0, 2, 1) if dtype == torch.float32 else (0, 4, 2, 1)


BWD_SWEEP = [(dt, gc, rg, r) for dt in DTYPES for gc in (1, 2, 4) for rg in ("tiny", "many", "few")
             for r in class_residues(dt)]


@gpu
@pytest.mark.parametrize("dtype,gc,regime,r", BWD_SWEEP,
                         ids=[f"{DNAME[a]}-G{b}-{c}-r{d}" for a, b, c, d in BWD_SWEEP])
def test_backward_regimes_and_classes(dtype, gc, regime, r):
    """Each (dtype, gc) template in each regime at each misalignment class (G = gc: one chunk), LeakyReLU, dA onto a
    nonzero initial value."""
    N, K = regime_shape(dtype, gc, regime, r)
    assert bwd_plan(dtype, gc, N, K) == [(gc, regime)]
    d = R.rows_inputs(gc, N, K, dtype, _seed("bwd", gc, N, K))
    _bwd_check(d, dtype, 1, f"bwd {DNAME[dtype]} G={gc} N={N} K={K} {regime} ncls={ncls(dtype, K)}")


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DNAME.get)
@pytest.mark.parametrize("G", [1, 2, 3, 4, 5, 7, 8, 13, 64])
def test_backward_g_chunks(dtype, G):
    """G split 4 / 2 / 1, the later chunks accumulating into dW, at a tiny shape with ncls = V; G = 5 also at a shape
    where the gc = 4 chunk runs many strips and the gc = 1 chunk few strips."""
    V = R.vec_width(dtype)
    N, K = 64, 16 * V + 1
    d = R.rows_inputs(G, N, K, dtype, _seed("bwd-g", G, K))
    _bwd_check(d, dtype, 1, f"bwd {DNAME[dtype]} G={G} N={N} K={K} chunks {bwd_plan(dtype, G, N, K)}")
    if G == 5:
        N, K = (2700, 1601) if dtype == torch.float32 else (2700, 2001)
        assert bwd_plan(dtype, G, N, K) == [(4, "many"), (1, "few")]
        d = R.rows_inputs(G, N, K, dtype, _seed("bwd-mixed", G, K))
        _bwd_check(d, dtype, 1, f"bwd {DNAME[dtype]} G={G} N={N} K={K} chunks {bwd_plan(dtype, G, N, K)}")


@gpu
def test_backward_refuses_g_65():
    from hypernet_image_captioning_b200._cabi import CaphnError
    z = lambda *s: torch.zeros(*s, device="cuda")
    with pytest.raises(CaphnError):
        _ops().rows_linear_bwd(z(10, 12), z(65, 12), None, z(65, 10))
    torch.cuda.synchronize()


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DNAME.get)
@pytest.mark.parametrize("regime", ["tiny", "many", "few"])
def test_backward_options(dtype, regime):
    """The dA-only pass (need_dW=False, lowrank mode), need_dA=False, dA accumulated onto a nonzero value, and
    dY / Y slices of theta at odd column offsets with dA a strided view whose sentinel columns beyond K stay."""
    ops = _ops()
    G = 3
    N, K = regime_shape(dtype, 1, regime, 3)
    d = R.rows_inputs(G, N, K, dtype, _seed("bwd-opt", N, K))
    tag = f"bwd {DNAME[dtype]} G={G} N={N} K={K} {bwd_plan(dtype, G, N, K)}"
    _bwd_check(d, dtype, 1, tag + " dA only", need_dW=False)
    _bwd_check(d, dtype, 0, tag + " no dA", need_dA=False)
    _bwd_check(d, dtype, 0, tag + " dA from zero", dA0=False)
    W, A = d["W"].cuda(), d["A"].cuda()
    theta = torch.randn(G, N + 40, device="cuda")
    Yt, dYt = theta[:, 3:3 + N], theta[:, 21:21 + N]
    dAbuf = torch.full((G, K + 5), -3.5, device="cuda")
    dAbuf[:, :K] = d["dA0"].cuda()
    dW, db, dA, dP = ops.rows_linear_bwd(W, A, Yt, dYt, 1, dA=dAbuf[:, :K], return_dP=True)
    torch.cuda.synchronize()
    assert dA.data_ptr() == dAbuf.data_ptr() and bool((dAbuf[:, K:] == -3.5).all()), "dA written beyond column K"
    ref = R.rows_bwd(W, A, Yt, dYt, 1, dA0=d["dA0"].cuda())
    compare(bwd_errors({"dP": dP, "dbias": db, "dW": dW, "dA": dA}, ref, dtype, dYt, A), tag + " strided Y / dY / dA")


# ----------------------------------------------------------------------------------------------------------------------
# GPU: gradient norm
# ----------------------------------------------------------------------------------------------------------------------
def _tail_heavy(n, vec, seed, dtype=torch.float32):
    """x ~ N(0,1) with the last n % vec entries scaled so the tail carries ~1 % of sum x^2 at any n."""
    x = torch.randn(n, generator=torch.Generator(device="cuda").manual_seed(seed), device="cuda")
    t = n % vec
    if t:
        x[n - t:] *= math.sqrt(0.01 * n / t) + 1.0
    return x.to(dtype)


def _sumsq(x, bf16=False):
    from hypernet_image_captioning_b200 import _cabi
    out = torch.zeros(1, device="cuda", dtype=torch.float64)
    _cabi.call("caphn_sumsq_bf16" if bf16 else "caphn_sumsq", x.data_ptr(), x.numel(), out.data_ptr(), _stream())
    return out


SUMSQ_N = [1, 2, 3, 4, 5, 6, 7, 1000, 1001, 1002, 1003, 7_274_500, 8_000_003]


@gpu
@pytest.mark.parametrize("n", SUMSQ_N)
def test_sumsq(n):
    """n % 4 in 0..3, n < 4, and n past the unrolled grid-stride threshold."""
    x = _tail_heavy(n, 4, _seed("sumsq", n))
    compare({"sumsq": rel(_sumsq(x), R.sumsq(x)[None])}, f"sumsq n={n} unrolled={sumsq_unrolled(n)}")


@gpu
@pytest.mark.parametrize("n", list(range(1, 17)) + [1 << 20, 5_000_005])
def test_sumsq_bf16(n):
    x = _tail_heavy(n, 8, _seed("sumsq-bf16", n), torch.bfloat16)
    compare({"sumsq": rel(_sumsq(x, True), R.sumsq(x)[None])}, f"sumsq_bf16 n={n}")


@gpu
@pytest.mark.parametrize("G", [1, 2, 3, 4])
def test_gram_and_lowrank_norm(G):
    """caphn_gram of dP [G, N] and A [G, K] with row strides beyond the row, and caphn_sumsq_lowrank from them
    against ||dP^T A||_F^2 in float64."""
    from hypernet_image_captioning_b200 import _cabi
    for N, K in ((11250, 1600), (90000, 8437), (7, 3)):
        d = R.lowrank_inputs(G, N, K, _seed("gram", G, N, K), "cuda", ldp=N + 5, lda=K + 3)
        gram = torch.zeros(2, G * G, device="cuda", dtype=torch.float64)
        s = torch.zeros(1, device="cuda", dtype=torch.float64)
        _cabi.call("caphn_gram", d["dP"].data_ptr(), d["dP"].stride(0), G, N, gram[0].data_ptr(), _stream())
        _cabi.call("caphn_gram", d["A"].data_ptr(), d["A"].stride(0), G, K, gram[1].data_ptr(), _stream())
        _cabi.call("caphn_sumsq_lowrank", gram[0].data_ptr(), gram[1].data_ptr(), G, s.data_ptr(), _stream())
        torch.cuda.synchronize()
        P64, A64 = d["dP"].double(), d["A"].double()
        errs = {"gram": max(rel(gram[0], (P64 @ P64.t()).reshape(-1)), rel(gram[1], (A64 @ A64.t()).reshape(-1))),
                "frob": rel(s, R.lowrank_frob2(d["dP"], d["A"])[None])}
        compare(errs, f"gram / sumsq_lowrank G={G} N={N} K={K}")


@gpu
def test_clip_coef():
    """Both sides of max_norm: the coefficient is 1 below it and max_norm / (norm + 1e-6) above."""
    from hypernet_image_captioning_b200 import _cabi
    for s in (0.0, 1.0, 24.9, 25.0001, 400.0, 1e12):
        ss = torch.tensor([s], device="cuda", dtype=torch.float64)
        coef, norm = torch.zeros(1, device="cuda"), torch.zeros(1, device="cuda")
        _cabi.call("caphn_clip_coef", ss.data_ptr(), 5.0, coef.data_ptr(), norm.data_ptr(), _stream())
        want_c, want_n = R.clip_coef(s, 5.0)
        errs = {"coef": abs(coef.item() - want_c) / want_c, "coef_norm": abs(norm.item() - want_n) / max(want_n, 1e-30)}
        report(f"clip_coef sumsq={s}: coef {errs['coef']:.2e}, norm {errs['coef_norm']:.2e}")
        assert errs["coef"] < BOUNDS["coef"] and errs["coef_norm"] < BOUNDS["coef"], (s, coef.item(), norm.item())
        assert (coef.item() == 1.0) == (want_c == 1.0)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: Adam
# ----------------------------------------------------------------------------------------------------------------------
ADAM_CASES = [(None, 0.0), (0.37, 0.0), (None, 0.05), (0.37, 0.05)]       # (gscale, weight decay)
ADAM_N = [1, 2, 3, 4, 5, 6, 7, 1029, 1030, 1031, 1032, 4_849_667, 6_000_001]


def _gs(gscale):
    return None if gscale is None else torch.tensor([gscale], device="cuda")


def _adam_errs(got, ref, keys):
    return {k: rel(got[k], r) for k, r in zip(keys, ref)}


@gpu
@pytest.mark.parametrize("n", ADAM_N)
def test_adam_dense(n):
    """caphn_adam_step from a random state at step 3, one call per case, with and without gscale and weight decay:
    n % 4 tails, n < 4, the half-pass `two` branch and the grid-stride wrap (n > 4 849 664)."""
    from hypernet_image_captioning_b200 import _cabi
    for gscale, wd in ADAM_CASES:
        d = {k: v.cuda() for k, v in R.adam_inputs(n, _seed("adam", n, wd)).items()}
        ref = R.adam_step(d["p"], d["g"], d["m"], d["v"], 3, wd=wd, gscale=gscale)
        gs = _gs(gscale)
        _cabi.call("caphn_adam_step", d["p"].data_ptr(), d["g"].data_ptr(), d["m"].data_ptr(), d["v"].data_ptr(), n,
                   1e-2, 0.9, 0.999, 1e-8, wd, 3, None if gs is None else gs.data_ptr(), _stream())
        torch.cuda.synchronize()
        compare(_adam_errs(d, ref, ("p", "m", "v")),
                f"adam n={n} gscale={gscale} wd={wd} wraps={dense_adam_wraps(n)}")


@gpu
@pytest.mark.parametrize("n", list(range(1, 17)) + [4096 + 3, 4_849_671, 9_699_337])
def test_adam_bf16(n):
    """caphn_adam_step_bf16: master, m and v against the reference, p == bf16(master) bit for bit, n % 8 tails, and
    one, two and three loop iterations per thread (bf16_adam_iterations)."""
    from hypernet_image_captioning_b200 import _cabi
    for gscale, wd in ADAM_CASES:
        d = {k: v.cuda() for k, v in R.adam_inputs(n, _seed("adam-bf16", n, wd), bf16=True).items()}
        ref = R.adam_step(d["master"], d["g"], d["m"], d["v"], 3, wd=wd, gscale=gscale)
        gs = _gs(gscale)
        _cabi.call("caphn_adam_step_bf16", d["p"].data_ptr(), d["g"].data_ptr(), d["master"].data_ptr(),
                   d["m"].data_ptr(), d["v"].data_ptr(), n, 1e-2, 0.9, 0.999, 1e-8, wd, 3,
                   None if gs is None else gs.data_ptr(), _stream())
        torch.cuda.synchronize()
        compare(_adam_errs(d, ref, ("master", "m", "v")), f"adam_bf16 n={n} gscale={gscale} wd={wd}")
        assert torch.equal(d["p"], d["master"].to(torch.bfloat16)), f"n={n}: p is not bf16(master)"


LOWRANK_K = [1, 2, 3, 4, 5, 1600, 8437, 11250]


def lowrank_shapes(K):
    """N below and above the grid-stride wrap of N K, with N K % 4 != 0 where K allows it."""
    lo = max(1, 1_000_000 // K) | 1
    hi = (4_849_664 // K + 7) | 1
    return [(lo, K), (hi, K)]


def _lowrank_case(G, N, K, gscale, wd, ldp, lda, bounds=None, tag="lowrank"):
    from hypernet_image_captioning_b200 import _cabi
    d = R.lowrank_inputs(G, N, K, _seed(tag, G, N, K), "cuda", ldp=ldp, lda=lda)
    p0, m0, v0 = d["p"].clone(), d["m"].clone(), d["v"].clone()
    gs = _gs(gscale)
    _cabi.call("caphn_adam_step_lowrank", d["p"].data_ptr(), d["m"].data_ptr(), d["v"].data_ptr(), d["dP"].data_ptr(),
               d["dP"].stride(0), d["A"].data_ptr(), d["A"].stride(0), G, N, K, 1e-2, 0.9, 0.999, 1e-8, wd, 3,
               None if gs is None else gs.data_ptr(), _stream())
    torch.cuda.synchronize()
    errs = {"p": 0.0, "m": 0.0, "v": 0.0}
    scale = {"p": 0.0, "m": 0.0, "v": 0.0}
    step = max(1, R.CHUNK_ELEMS // (4 * K))
    for r0 in range(0, N, step):
        rows = slice(r0, r0 + step)
        g = d["dP"][:, rows].double().t() @ d["A"].double()
        ref = R.adam_step(p0[rows], g, m0[rows], v0[rows], 3, wd=wd, gscale=gscale)
        for k, r in zip(("p", "m", "v"), ref):
            errs[k] = max(errs[k], (d[k][rows].double() - r).abs().max().item())
            scale[k] = max(scale[k], r.abs().max().item())
    errs = {k: errs[k] / scale[k] for k in errs}
    compare(errs, f"{tag} G={G} N={N} K={K} ldp={ldp} lda={lda} gscale={gscale} wd={wd} "
                  f"wraps={lowrank_wraps(N, K)} tail={N * K % 4}", bounds)


@gpu
@pytest.mark.parametrize("K", LOWRANK_K)
@pytest.mark.parametrize("G", [1, 2, 3, 4])
def test_adam_lowrank(G, K):
    """caphn_adam_step_lowrank against the dense float64 step fed with g = dP^T A: float4s straddling rows (K % 4 != 0),
    N K below and above the grid-stride wrap and total % 4 tails, ldp > N and lda > K.  m = beta-update(m0, gscale g)
    per element names the g each element used."""
    for i, (N, KK) in enumerate(lowrank_shapes(K)):
        gscale, wd = ADAM_CASES[(G + i) % 4]
        _lowrank_case(G, N, KK, gscale, wd, N + 3, KK + 1)


# ----------------------------------------------------------------------------------------------------------------------
# drift at the benchmark's head shapes
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("N,K", [(90000, 11250), (11250, 1600)])
def test_drift_rows_at_the_head_shape(N, K):
    """fp32, G = 1: the second head layer of the pooled benchmark (many strips) and its first layer (few strips)."""
    d = R.rows_inputs(1, N, K, torch.float32, _seed("drift", N, K), "cuda")
    tag = f"drift fp32 G=1 N={N} K={K} {bwd_plan(torch.float32, 1, N, K)}"
    _fwd_check(d, 1, N, K, torch.float32, 0, tag + " fwd")
    _bwd_check(d, torch.float32, 0, tag + " bwd")


@gpu
def test_drift_lowrank_at_the_head_shape():
    """One lowrank step at N = 90000, K = 11250 (G = 1, clip coefficient applied), the reference chunked on the GPU."""
    _lowrank_case(1, 90000, 11250, 0.37, 0.0, 90000, 11250, tag="drift lowrank")


# ----------------------------------------------------------------------------------------------------------------------
# CPU: planted defects
# ----------------------------------------------------------------------------------------------------------------------
def _rows_mutant_shapes(mutant):
    out = []
    for dt, gc, rg, r in BWD_SWEEP:
        if rg != "tiny":
            continue
        N, K = regime_shape(dt, gc, rg, r)
        G = 3 if mutant == "later G-chunk overwrites dW" else gc
        if mutant == "misalignment m of the next row" and ncls(dt, K) == 1:
            continue
        out.append((dt, G, N, K))
    return out


def _rows_ratio(mutant, dt, G, N, K):
    d = R.rows_inputs(G, N, K, dt, _seed("bwd", G, N, K))
    W, A = d["W"], d["A"]
    errs = {"Y": rel(R.rows_fwd(W, d["b"], A, 1, mutant=mutant), R.rows_fwd(W, d["b"], A, 1))}
    ref = R.rows_bwd(W, A, d["Y"], d["dY"], 1, dA0=d["dA0"])
    mut = R.rows_bwd(W, A, d["Y"], d["dY"], 1, dA0=d["dA0"], mutant=mutant)
    errs.update(bwd_errors(mut, ref, dt, d["dY"], A))
    return max(e / (1.0 if k == "dW_bf16" else BOUNDS[k]) for k, e in errs.items())


@pytest.mark.parametrize("mutant", R.MUTANTS)
def test_tolerances_catch_planted_defects(mutant):
    """Each defect planted in the float64 reference moves at least one compared output by more than 10x its bound, on
    the sweep's shapes wherever the defect can show (CPU inputs of the same shapes).  The smallest margin is 128x
    ("later G-chunk overwrites dW"); every other defect moves an output by more than 150x."""
    ratios = []
    if mutant in R.ROW_MUTANTS:
        for dt, G, N, K in _rows_mutant_shapes(mutant):
            ratios.append(_rows_ratio(mutant, dt, G, N, K))
    elif mutant in R.ADAM_MUTANTS:
        for n in ADAM_N[:11]:
            for gscale, wd in ADAM_CASES:
                if mutant == "gscale after weight decay" and not (gscale and wd):
                    continue
                d = R.adam_inputs(n, _seed("adam", n, wd))
                ref = R.adam_step(d["p"], d["g"], d["m"], d["v"], 3, wd=wd, gscale=gscale)
                mut = R.adam_step(d["p"], d["g"], d["m"], d["v"], 3, wd=wd, gscale=gscale, mutant=mutant)
                ratios.append(max(rel(a, b) / BOUNDS[k] for k, a, b in zip("pmv", mut, ref)))
    elif mutant in R.LOWRANK_MUTANTS:
        for G in (1, 2, 3, 4):
            for K in LOWRANK_K:
                for i, (N, _) in enumerate(lowrank_shapes(K)):     # test_adam_lowrank's shapes and hyper-parameters
                    if mutant == "k-carry wraps to 1" and K % 4 == 0 or mutant == "tail reads the previous row" and \
                            N * K % 4 == 0:
                        continue
                    gscale, wd = ADAM_CASES[(G + i) % 4]
                    d = R.lowrank_inputs(G, N, K, _seed("lowrank", G, N, K))
                    step = lambda g: R.adam_step(d["p"], g, d["m"], d["v"], 3, wd=wd, gscale=gscale)
                    ref, mut = step(R.lowrank_grad(d["dP"], d["A"])), step(R.lowrank_grad(d["dP"], d["A"], mutant))
                    ratios.append(max(rel(a, b) / BOUNDS[k] for k, a, b in zip("pmv", mut, ref)))
    else:
        for n in SUMSQ_N[:11]:
            if n % 4 == 0:
                continue
            g = torch.Generator().manual_seed(n)
            x = torch.randn(n, generator=g)
            t = n % 4
            x[n - t:] *= math.sqrt(0.01 * n / t) + 1.0
            ratios.append(rel(R.sumsq(x, mutant=mutant)[None], R.sumsq(x)[None]) / BOUNDS["sumsq"])
    assert len(ratios) >= 3, mutant
    report(f"mutant {mutant!r}: smallest margin {min(ratios):.1f}x the bound over {len(ratios)} shapes")
    assert min(ratios) > 10, f"{mutant}: moves the outputs by only {min(ratios):.1f}x the bound"
