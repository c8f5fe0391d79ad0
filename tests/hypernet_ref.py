"""Float64 reference of the hypernetwork parameter path: the weight-streaming layers (csrc/hn_rows.cu), the gradient norm
and the Adam updates (csrc/optim.cu), and seeded inputs in the kernels' layouts.

    forward     Y[g,n] = act(sum_k A[g,k] W[n,k] + b[n])                      rows_fwd_kernel
    backward    dP = dY * act'(Y);  db = sum_g dP;  dW = dP^T A;  dA += dP W  rows_bwd_prep_kernel + rows_bwd_kernel
    norm        sum x^2;  ||dP^T A||_F^2 = sum_{q,r} (dP_q . dP_r)(A_q . A_r)   sumsq / gram / sumsq_lowrank
    update      torch.optim.Adam (amsgrad off) with the clip coefficient       adam_* kernels
                multiplied into the gradient first

Everything runs in float64 on whatever device its inputs are on: the large shapes are computed on the GPU in row chunks
(torch float64 matrix products, not the code under test), so host memory stays bounded.

``mutant`` plants one defect, modelled on the kernels' own data flow; the mutation tests use them to show that the
tolerances would catch each one."""
import math

import torch

LEAKY = 0.01
ROW_MUTANTS = ("misalignment m of the next row", "last vector of a row dropped", "later G-chunk overwrites dW")
ADAM_MUTANTS = ("bias correction at step - 1", "gscale after weight decay")
LOWRANK_MUTANTS = ("k-carry wraps to 1", "tail reads the previous row")
NORM_MUTANTS = ("sumsq tail dropped",)
MUTANTS = ROW_MUTANTS + ADAM_MUTANTS + LOWRANK_MUTANTS + NORM_MUTANTS
CHUNK_ELEMS = 1 << 26


def vec_width(dtype):
    """Elements per 128-bit vector of a weight row: 4 fp32, 8 bf16."""
    return 8 if dtype == torch.bfloat16 else 4


def bwd_chunks(G):
    """rows_linear_bwd_t: G split into chunks of 4, 2 and 1, in that order."""
    out, g0 = [], 0
    while g0 < G:
        gc = 4 if G - g0 >= 4 else (2 if G - g0 >= 2 else 1)
        out.append((g0, gc))
        g0 += gc
    return out


# ----------------------------------------------------------------------------------------------------------------------
# inputs
# ----------------------------------------------------------------------------------------------------------------------
def _gen(seed, device):
    return torch.Generator(device=device).manual_seed(seed)


def rows_inputs(G, N, K, dtype, seed, device="cpu", lda=None, ldy=None, ldda=None):
    """One layer: W [N,K] (fp32 or bf16, its values exact in float64), b [N], A [G,K] with row stride lda, Y and dY
    [G,N] with row strides ldy (the values a forward would have left; Y half negative so LeakyReLU matters), and a
    nonzero initial dA0 [G,K] with row stride ldda.  Strided operands are views of wider buffers."""
    g = _gen(seed, device)
    r = lambda *s: torch.randn(*s, generator=g, device=device)
    lda, ldy, ldda = lda or K, ldy or N, ldda or K
    d = {"W": (r(N, K) / math.sqrt(K)).to(dtype), "b": r(N) * 0.1,
         "A": r(G, lda)[:, :K], "Y": r(G, ldy)[:, :N], "dY": r(G, ldy)[:, :N] * 0.3, "dA0": r(G, ldda)[:, :K] * 0.2}
    return d


def adam_inputs(n, seed, device="cpu", bf16=False):
    """A random optimizer state away from zero: p, g ~ N(0, 1), m ~ 0.1 N(0, 1), v = (0.3 N(0,1))^2 + 1e-3 (so sqrt(v)
    dominates eps and the update depends on |g|).  bf16: g holds bf16 values and p = bf16(master)."""
    gen = _gen(seed, device)
    r = lambda: torch.randn(n, generator=gen, device=device)
    d = {"p": r(), "g": r(), "m": r() * 0.1, "v": (r() * 0.3) ** 2 + 1e-3}
    if bf16:
        d["master"] = d.pop("p")
        d["p"] = d["master"].to(torch.bfloat16)
        d["g"] = d["g"].to(torch.bfloat16)
    return d


def lowrank_inputs(G, N, K, seed, device="cpu", ldp=None, lda=None):
    """p, m, v [N,K] as adam_inputs, dP [G,N] (row stride ldp) and A [G,K] (row stride lda) scaled so g ~ N(0, 1)."""
    d = {k: v.reshape(N, K) for k, v in adam_inputs(N * K, seed, device).items() if k != "g"}
    gen = _gen(seed + 1, device)
    d["dP"] = torch.randn(G, ldp or N, generator=gen, device=device)[:, :N] / math.sqrt(G)
    d["A"] = torch.randn(G, lda or K, generator=gen, device=device)[:, :K]
    return d


# ----------------------------------------------------------------------------------------------------------------------
# weight-streaming layers
# ----------------------------------------------------------------------------------------------------------------------
def _shift_cols(A, d):
    """A[:, k + d] with zeros outside [0, K)."""
    out = torch.zeros_like(A)
    K = A.shape[1]
    if d >= 0:
        out[:, :K - d] = A[:, d:]
    else:
        out[:, -d:] = A[:, :K + d]
    return out


def _rowwise(W, A, mutant, V, r0):
    """The rows r0.. of a chunk as the kernels pair them with the activation: (W64 [n,K], [(row mask or None, A64)]).
    Row n's vectors start m = (n K) mod V elements before the row; the kernels index the activation by m."""
    n, K = W.shape
    W64, A64 = W.double(), A.double()
    m = (torch.arange(r0, r0 + n, device=W.device, dtype=torch.int64) * K) % V
    if mutant == "last vector of a row dropped":
        start = V * ((K + m + V - 1) // V - 1) - m                    # first k of the last vector of each row
        W64 = torch.where(torch.arange(K, device=W.device)[None, :] >= start[:, None], 0.0, W64)
    if mutant == "misalignment m of the next row":
        d = m - ((m + K) % V)                                         # activation offset by the next row's m
        return W64, [(d == s, _shift_cols(A64, s)) for s in range(-V + 1, V)]
    return W64, [(None, A64)]


def _chunks(N, K):
    step = max(1, CHUNK_ELEMS // max(K, 1))
    return [(r0, min(N, r0 + step)) for r0 in range(0, N, step)]


def rows_fwd(W, b, A, act, slope=LEAKY, mutant=None):
    """Y [G,N] float64 of rows_linear_fwd."""
    G, K = A.shape
    N = W.shape[0]
    V = vec_width(W.dtype)
    Y = torch.empty(G, N, dtype=torch.float64, device=W.device)
    for r0, r1 in _chunks(N, K):
        W64, parts = _rowwise(W[r0:r1], A, mutant, V, r0)
        y = torch.zeros(G, r1 - r0, dtype=torch.float64, device=W.device)
        for mask, Ash in parts:
            t = Ash @ W64.t()
            y = t if mask is None else torch.where(mask[None, :], t, y)
        Y[:, r0:r1] = y
    if b is not None:
        Y += b.double()[None, :]
    if act:
        Y = torch.where(Y > 0, Y, Y * slope)
    return Y


def rows_bwd(W, A, Y, dY, act, slope=LEAKY, dA0=None, mutant=None, need_dW=True):
    """dP, dbias, dW (None unless need_dW), dA (+ dA0) of rows_linear_bwd, float64.  Y is the forward output the
    kernel is given (its sign selects the LeakyReLU branch)."""
    G, K = A.shape
    N = W.shape[0]
    V = vec_width(W.dtype)
    dP = dY.double()
    if act:
        dP = torch.where(Y > 0, dP, dP * slope)
    dA = torch.zeros(G, K, dtype=torch.float64, device=W.device) if dA0 is None else dA0.double().clone()
    dW = torch.empty(N, K, dtype=torch.float64, device=W.device) if need_dW else None
    last = bwd_chunks(G)[-1][0]
    for r0, r1 in _chunks(N, K):
        W64, parts = _rowwise(W[r0:r1], A, mutant, V, r0)
        dPc = dP[:, r0:r1]
        for mask, Ash in parts:
            dPm = dPc if mask is None else dPc * mask[None, :]
            dA += dPm @ W64
            if need_dW:
                src = slice(last, G) if mutant == "later G-chunk overwrites dW" else slice(0, G)
                t = dPm[src].t() @ Ash[src]
                dW[r0:r1] = t if mask is None else torch.where(mask[:, None], t, dW[r0:r1])
    return {"dP": dP, "dbias": dP.sum(0), "dW": dW, "dA": dA}


# ----------------------------------------------------------------------------------------------------------------------
# gradient norm and Adam
# ----------------------------------------------------------------------------------------------------------------------
def sumsq(x, vec=4, mutant=None):
    """sum x^2 in float64; the mutant drops the n % vec tail the kernels handle apart from the vector loop."""
    x = x.double().reshape(-1)
    if mutant == "sumsq tail dropped":
        x = x[:x.numel() - x.numel() % vec]
    return (x * x).sum()


def lowrank_frob2(dP, A):
    """||dP^T A||_F^2 without forming the product: trace((dP dP^T)(A A^T))."""
    dP, A = dP.double(), A.double()
    return ((dP @ dP.t()) * (A @ A.t())).sum()


def clip_coef(s, max_norm):
    """torch.nn.utils.clip_grad_norm_: min(1, max_norm / (||g|| + 1e-6)) and ||g||, from the float64 sum of squares."""
    norm = math.sqrt(s)
    return min(1.0, max_norm / (norm + 1e-6)), norm


def hyper(lr, betas, eps, wd, step, mutant=None):
    """The fp32 hyper-parameters the host functions derive in double and round once (caphn_adam_step*)."""
    f32 = lambda x: float(torch.tensor(x, dtype=torch.float32))
    t = step - 1 if mutant == "bias correction at step - 1" else step
    bc1, bc2 = 1.0 - betas[0] ** t, 1.0 - betas[1] ** t
    return {"beta2": f32(betas[1]), "omb1": f32(1.0 - betas[0]), "omb2": f32(1.0 - betas[1]), "eps": f32(eps),
            "wd": f32(wd), "step_size": f32(lr / bc1), "bc2_sqrt": f32(math.sqrt(bc2))}


def adam_step(p, g, m, v, step, lr=1e-2, betas=(0.9, 0.999), eps=1e-8, wd=0.0, gscale=None, mutant=None):
    """One torch.optim.Adam step in float64 -> (p, m, v).  gscale (a float, the clip coefficient as fp32) multiplies
    the gradient before weight decay is added."""
    h = hyper(lr, betas, eps, wd, step, mutant)
    p, g, m, v = p.double(), g.double(), m.double(), v.double()
    gs = 1.0 if gscale is None else gscale
    if mutant == "gscale after weight decay":
        g = (g + h["wd"] * p) * gs if h["wd"] else g * gs
    else:
        g = g * gs
        if h["wd"]:
            g = g + h["wd"] * p
    m = m + h["omb1"] * (g - m)
    v = v * h["beta2"] + h["omb2"] * g * g
    denom = v.sqrt() / h["bc2_sqrt"] + h["eps"]
    return p - h["step_size"] * (m / denom), m, v


def lowrank_grad(dP, A, mutant=None):
    """g [N,K] = dP^T A in float64, walked as adam_lowrank_kernel walks it: the flat index e = n K + k in float4 steps
    with an incremental (n, k) carry, the last total % 4 elements apart.  The mutants break the carry or the tail."""
    G, N = dP.shape
    K = A.shape[1]
    g = dP.double().t() @ A.double()
    if mutant is None:
        return g
    total = N * K
    flat = g.reshape(-1).clone()
    dP64, A64 = dP.double(), A.double()
    val = lambda n, k: torch.where((n < N) & (k < K), (dP64[:, n.clamp(max=N - 1)] * A64[:, k.clamp(max=K - 1)]).sum(0),
                                   torch.zeros((), dtype=torch.float64, device=g.device))
    n4 = total // 4
    if mutant == "k-carry wraps to 1":
        e0 = torch.arange(n4, device=g.device, dtype=torch.int64) * 4
        n, k = e0 // K, e0 % K
        for c in range(4):
            flat[e0 + c] = val(n, k)
            k = k + 1
            wrap = k == K
            k = torch.where(wrap, 1, k)
            n = n + wrap.long()
    elif mutant == "tail reads the previous row":
        e = torch.arange(4 * n4, total, device=g.device, dtype=torch.int64)
        flat[e] = val((e // K - 1) % N, e % K)
    return flat.reshape(N, K)
