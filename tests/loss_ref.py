"""Float64 reference of the cross-entropy kernels (csrc/ce_misc.cu: ce_fwd, ce_finish, ce_bwd, ce_bwd_split,
ce_fwd_split) and of the vocabulary backward of the fused loss nodes (functional.ce_fwd_for_loss / vocab_bwd_fused /
VocabPrep), with their host plans restated, seeded inputs in the kernels' layouts, and planted defects.

    lse[m]   = log sum_{v < V} exp(x[m, v])
    valid[m] = not (has_ignore and t[m] == ignore)                 count = sum_m valid[m]
    live[m]  = valid[m] and 0 <= t[m] < V
    loss[m]  = valid ? (live ? lse[m] - x[m, t[m]] : NaN) : 0       mean = sum_m loss[m] / count   (0 / 0 = NaN)
    u[m, v]  = live ? softmax(x[m])[v] - [v == t[m]] : 0            ce_fwd_split writes u (unscaled)
    d        = u * g / max(count, 1)                                ce_bwd, ce_bwd_split (g = gscale[0])
    dbias    = sum_m d[m, :]      dH = d W      dW = d^T H          (logits = H W^T + b)
    split    hi = rn_bf16(u),  lo = rn_bf16(u - hi)                 (lo absent in bf16 mode)

Everything is float64 torch on the device of its inputs (the large shapes on the GPU: torch's float64 ops, not the code
under test)."""
import math

import torch

IGNORE_NEG = -100             # torch's default ignore_index, the negative value the kernels must take as is

# ----------------------------------------------------------------------------------------------------------------------
# the host plans, restated
# ----------------------------------------------------------------------------------------------------------------------
CE_THREADS = 256
CE_FWD_SPLIT_MAX_V = 50000    # ops.CE_FWD_SPLIT_MAX_V; caphn_ce_fwd_split refuses V > 50000 (ce_misc.cu:626)
NUM_SMS = 148
TC_MIN_WORK = 1 << 24


def cdiv(a, b):
    return -(-a // b)


def round4(n):
    return cdiv(n, 4) * 4


def round64(n):
    return cdiv(n, 64) * 64


def fwd_vec(ld, V, x_addr):
    """ce_fwd_kernel (ce_misc.cu:53) and ce_fwd_split_kernel (ce_misc.cu:244; the vec path is the one cp.async.bulk)."""
    return ld % 4 == 0 and V % 4 == 0 and x_addr % 16 == 0


def bwd_vec(ld, lddx, V, x_addr, dx_addr):
    """ce_bwd_kernel (ce_misc.cu:110)."""
    return ld % 4 == 0 and lddx % 4 == 0 and V % 4 == 0 and x_addr % 16 == 0 and dx_addr % 16 == 0


def split_vec_threads(ld, V, x_addr):
    """ce_bwd_split_kernel (ce_misc.cu:148): how many of the row's 4-column groups v0 + c4 < round64(V) load a float4 and
    how many load scalars (c4 = 4 * (tid & 15)), as (vector, scalar)."""
    ok = ld % 4 == 0 and x_addr % 16 == 0
    groups = [v for v in range(0, round64(V), 4)]
    vec = sum(1 for v in groups if ok and v + 3 < V)
    return vec, len(groups) - vec


def fwd_split_smem(V):
    """Dynamic shared memory of ce_fwd_split_kernel: round4(V) floats (ce_misc.cu:629); None where the call refuses V."""
    return None if V > CE_FWD_SPLIT_MAX_V else cdiv(V, 4) * 16


def colsum_rpb(M, N):
    """caphn_colsum (ce_misc.cu:713-715): rows per block and gridDim.y."""
    xb = cdiv(N, 128)
    rpb = 256
    while rpb > 16 and xb * cdiv(M, rpb) < 8 * NUM_SMS:
        rpb >>= 1
    if cdiv(M, rpb) > 65535:
        rpb = cdiv(M, 65535)
    return rpb, cdiv(M, rpb)


def tc_ok(M, N, K):
    """ops._tc_ok (ops.py:123)."""
    return M >= 128 and N >= 16 and K >= 32 and M * N * K >= TC_MIN_WORK


def loss_path(M, V, H, need_grad=True):
    """Which path the fused loss nodes take: "one-pass" (ce_fwd_for_loss, functional.py:264: ce_fwd_split, then the two
    scaled products), "two-pass" (vocab_bwd_fused, functional.py:332-338: ce_fwd, ce_bwd_split, two TC products) or
    "fp32-dlogits" (functional.py:332-334: ce_fwd, ce_bwd, matmul_* and colsum)."""
    if need_grad and V <= CE_FWD_SPLIT_MAX_V and tc_ok(M, H, V) and tc_ok(V, H + 1, M):
        return "one-pass"
    if tc_ok(M, H, V) and tc_ok(V, H, M):
        return "two-pass"
    return "fp32-dlogits"


def vocab_prep_on(M, V, H, need_grad=True):
    """VocabPrep.on (functional.py:278-279): the one-pass path and the logits product on the tensor cores."""
    return loss_path(M, V, H, need_grad) == "one-pass" and tc_ok(M, V, H)


# ----------------------------------------------------------------------------------------------------------------------
# seeded inputs in the kernels' layouts
# ----------------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def logits(M, V, seed, ld=None, off=0, scale=3.0, gap=float("nan"), device="cpu"):
    """Logits [M, V] as a view with row pitch ld (default V) starting ``off`` floats into a buffer whose every other
    element (the pitch gaps, the first ``off`` floats, one float past the end) holds ``gap``.  off = 1 misaligns the base
    by 4 bytes, so the scalar paths are taken whatever ld and V are.  The row maximum sits in the last column on even rows
    and in the first column on rows 3 (mod 4), so the row tails carry weight in the max and the sum.  Returns (view,
    buffer)."""
    ld = V if ld is None else ld
    x = torch.randn(M, V, generator=_gen(seed)) * scale
    x[0::2, V - 1] = x[0::2].max(1).values + 2.0
    x[3::4, 0] = x[3::4].max(1).values + 2.0
    buf = torch.full((off + M * ld + 1,), gap, dtype=torch.float32)
    view = buf.as_strided((M, V), (ld, 1), off)
    view.copy_(x)
    buf = buf.to(device)
    return buf.as_strided((M, V), (ld, 1), off), buf


def targets(M, V, seed, ignore=None, device="cpu"):
    """Targets in [0, V) that include the first and the last column, and the ignore index on every 5th row (from row 2)
    when one is set."""
    t = torch.randint(0, V, (M,), generator=_gen(seed + 7))
    t[0::3] = 0
    t[1::3] = V - 1
    if ignore is not None:
        t[2::5] = ignore
    return t.to(device)


# ----------------------------------------------------------------------------------------------------------------------
# float64 references
# ----------------------------------------------------------------------------------------------------------------------
def ce_ref(x, t, ignore=None, mutant=None):
    """dict(lse, loss, valid, count, mean, u) in float64 for logits x [M, V] and targets t (int64)."""
    x = x.double()
    M, V = x.shape
    lse_cols = V
    if mutant == "last vector dropped from max / sum exp":
        lse_cols = V - (V % 4 or 4)                    # the last (partial) 4-column vector of the row never enters
    if lse_cols > 0:
        lse = torch.logsumexp(x[:, :lse_cols], dim=1)
    else:
        lse = torch.full((M,), -math.inf, dtype=torch.float64, device=x.device)
    if mutant == "target column off by one":
        t = torch.where(t + 1 < V, t + 1, t - 1)
    valid = torch.ones(M, dtype=torch.bool, device=x.device) if ignore is None else t != ignore
    live = valid & (t >= 0) & (t < V)
    tc = torch.where(live, t, torch.zeros_like(t))
    xt = x.gather(1, tc[:, None])[:, 0]
    loss = torch.where(live, lse - xt, torch.full_like(lse, math.nan))
    loss = torch.where(valid, loss, torch.zeros_like(lse))
    count = int(valid.sum())
    den = M if mutant == "ignored rows counted in the denominator" else count
    mean = loss.sum() / den if den else torch.tensor(math.nan, dtype=torch.float64)
    u = torch.exp(x - lse[:, None])
    u[torch.arange(M, device=x.device)[live], t[live]] -= 1.0
    u[~live] = 0.0
    return dict(lse=lse, loss=loss, valid=valid, count=den, mean=float(mean), u=u)


def grad_scale(g, count, M=None, mutant=None):
    """gscale / max(count, 1) as the backward kernels (and the scaled products' epilogues) apply it."""
    den = M if mutant == "scale by M instead of the count" else count
    return g / max(den, 1)


def dbias_ref(d, mutant=None):
    """sum_m d[m, :]; the mutant loses the last partial 64-row tile of ce_bwd_split's grid."""
    M = d.shape[0]
    if mutant == "dbias missing the last partial 64-row tile" and M % 64:
        d = d[:M - M % 64]
    return d.sum(0)


def bf16_rn(x):
    return x.float().to(torch.bfloat16).double()


def split_ref(u32, split=True, mutant=None):
    """hi + lo of the bf16 split of an fp32 tensor, as float64; hi only in bf16 mode or for the planted 'lo term missing'."""
    hi = bf16_rn(u32)
    if not split or mutant == "lo term missing from the split":
        return hi
    return hi + bf16_rn(u32.double() - hi)


def vocab_ref(x, t, ignore, g, Hm, W):
    """(dH, dW_out, db) of g * CE(H W^T + b) in float64 (x = the logits the kernels saw)."""
    r = ce_ref(x, t, ignore)
    d = r["u"] * grad_scale(g, r["count"])
    return d @ W.double(), d.t() @ Hm.double(), d.sum(0)


# ----------------------------------------------------------------------------------------------------------------------
# glue kernels (group_colsum, mean_pos_bwd, scatter): float64 references with their planted defects
# ----------------------------------------------------------------------------------------------------------------------
def group_colsum_ref(X, goff, B, T, mutant=None):
    """out[g, :] = sum over t < T and goff[g] <= b < goff[g+1] of X[t*B + b, :] (X [T*B, N])."""
    X = X.double().reshape(T, B, -1)
    G = len(goff) - 1
    out = torch.zeros(G, X.shape[2], dtype=torch.float64, device=X.device)
    for gi in range(G):
        b0, b1 = int(goff[gi]), int(goff[gi + 1])
        if mutant == "odd last row of a group dropped" and (b1 - b0) % 2:
            b1 -= 1
        if b1 > b0:
            out[gi] = X[:, b0:b1].sum((0, 1))
    return out


def mean_pos_bwd_ref(g, dX0, extra=None, mutant=None):
    """dX0 + g / P broadcast over positions (+ extra)."""
    P = dX0.shape[1]
    out = dX0.double() + (g.double() / P)[:, None, :]
    if extra is not None and mutant != "mean_pos_bwd ignores extra":
        out = out + extra.double()
    return out


def scatter_ref(table0, idx, dX, mutant=None):
    """table0[idx[i], :] += dX[i, :] for idx[i] >= 0; the mutant loses the last contribution to a repeated row."""
    out = table0.double().clone()
    keep = idx >= 0
    if mutant == "one duplicate contribution lost":
        seen, last = set(), None
        for i, r in enumerate(idx.tolist()):
            if r >= 0 and r in seen:
                last = i
            seen.add(r)
        if last is not None:
            keep = keep.clone()
            keep[last] = False
    out.index_add_(0, idx[keep], dX.double()[keep])
    return out


CE_MUTANTS = ("last vector dropped from max / sum exp", "target column off by one",
              "ignored rows counted in the denominator", "scale by M instead of the count",
              "dbias missing the last partial 64-row tile", "lo term missing from the split")
GLUE_MUTANTS = ("odd last row of a group dropped", "mean_pos_bwd ignores extra", "one duplicate contribution lost")
