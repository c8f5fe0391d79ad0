"""Float64 reference of the two GEMMs -- the tensor-core kernel (csrc/gemm_tc.cu, bf16x3 or bf16 operands, fp32 TMEM
accumulator) and the exact-fp32 SIMT kernel (csrc/gemm_simt.cu) -- with the host plan of the tensor-core kernel restated,
seeded data builders in the kernels' operand layouts, and planted defects.

    C = alpha * (A_hi B_hi^T + A_hi B_lo^T + A_lo B_hi^T) + bias     (ReLU)      gemm_tc_kernel, bf16x3
    C = alpha * (A_hi B_hi^T) + bias                                  (ReLU)      gemm_tc_kernel, bf16 mode
    alpha = num / max(den, 1)  (den None: 1; no scale: 1)
    hi = rn_bf16(x),  lo = rn_bf16(x - hi)                                        caphn_split_bf16* builders

Two kinds of data make the comparison exact (every partial sum is an fp32 number, so the result does not depend on the
order of accumulation, the accumulator's truncation or the split-K atomics):
    placement  integers in [-8, 8]: hi = x, lo = 0.  |C| <= 64 K < 2^24 up to K = 10240 (and 3 x that with alpha = 3).
    lo-term    x = h + l, h in {+-1, +-2}, l in {-1, 0, 1} 2^-10 (times 2^s per row / column): hi = h, lo = l exactly.
               hh + hl + lh is a multiple of 2^-10 below 2^12 in magnitude for K <= 4095, so it is exact; the lo.lo
               term the kernel must NOT issue would add multiples of 2^-20, and a missing hl / lh term moves it by >= 2^-10.
Float data (``float_operand``) has rows scaled by 2^s, s in [-8, 8], so rows of very different magnitude are checked
per element (``elem_err``) instead of against max|C|.

Everything is computed with torch float64 on the device of its inputs (the large shapes on the GPU: torch's float64
matrix product, not the code under test)."""
import math

import torch

# ----------------------------------------------------------------------------------------------------------------------
# the host plan of gemm_tc_impl (csrc/gemm_tc.cu), restated line for line
# ----------------------------------------------------------------------------------------------------------------------
BM, BK, NUM_SMS = 128, 64, 148
TILE_BYTES = BM * BK * 2
STG_BYTES = 8 * 32 * 32 * 4            # one 32 x 32 fp32 staging tile per epilogue warp
MAX_STAGES = 6
SMEM_BUDGET = 227 * 1024
BAR_BYTES = (2 * MAX_STAGES + 6) * 8 + 16 + 1024


def cdiv(a, b):
    return -(-a // b)


def round16(n):
    return cdiv(n, 16) * 16


def round64(n):
    return cdiv(n, 64) * 64


def tc_plan(M, N, K, a_mn=False, b_mn=False, split=True, splitk=0, relu=False, ldc=None, c_align=16, astat_on=True,
            tma_on=True, bn_force=None):
    """The launch gemm_tc_impl makes for one caphn_gemm_tc_ex / _scaled call, or None where it returns CAPHN_EINVAL.
    c_align: byte alignment of C (16 or less); astat_on / tma_on: CAPHN_TC_ASTAT / CAPHN_TC_TMA_STORE not set to 0."""
    ldc = N if ldc is None else ldc
    np_ = 2 if split else 1
    num_kb = cdiv(K, BK)
    few = None
    if N <= 256:
        BN = round64(N) if b_mn else round16(N)
    else:
        step = 64 if b_mn else 16
        tm = cdiv(M, BM)
        few = tm * cdiv(N, 128) <= 8 * NUM_SMS
        best, BN = -1, 128
        if few:
            for bn in range(128, 257, step):
                cost = cdiv(tm * cdiv(N, bn), NUM_SMS) * (bn + 32)
                if best < 0 or cost < best:
                    best, BN = cost, bn
        else:
            slab0 = num_kb * np_ * TILE_BYTES
            fits = astat_on and not a_mn and not b_mn and slab0 + STG_BYTES + BAR_BYTES + 3 * np_ * 128 * BK * 2 <= SMEM_BUDGET
            if not fits:
                BN = 256
        if bn_force is not None and 128 <= bn_force <= 256 and bn_force % step == 0:
            BN = bn_force
    tiles = cdiv(M, BM) * cdiv(N, BN)
    if splitk <= 0:
        splitk = 1
        if not relu and tiles < 3 * NUM_SMS:
            best = 0.0
            smax = min(32, max(1, num_kb // 4))
            for s in range(1, smax + 1):
                units = tiles * s
                eff = units / (cdiv(units, NUM_SMS) * NUM_SMS)
                if eff > best + 0.02:
                    best, splitk = eff, s
                if eff >= 0.9:
                    break
    if splitk > 1 and relu:
        return None
    kb_per = cdiv(num_kb, splitk)
    splitk = cdiv(num_kb, kb_per)
    b_bytes = BN * BK * 2
    stage_bytes = np_ * (TILE_BYTES + b_bytes)
    tma = tma_on and splitk == 1 and ldc % 4 == 0 and N % 4 == 0 and c_align % 16 == 0
    slab = num_kb * np_ * TILE_BYTES
    bstage = np_ * b_bytes
    astat_shape = astat_on and not a_mn and not b_mn and splitk == 1 and cdiv(N, BN) >= 4 and tiles >= 4 * NUM_SMS
    fixed = (0 if splitk > 1 else STG_BYTES) + BAR_BYTES
    if astat_shape and slab + fixed + 3 * bstage <= SMEM_BUDGET:
        astat, stages = True, (SMEM_BUDGET - fixed - slab) // bstage
    else:
        if fixed + 2 * stage_bytes > SMEM_BUDGET:
            return None
        astat, stages = False, (SMEM_BUDGET - fixed) // stage_bytes
    stages = min(stages, MAX_STAGES)
    if stages < 2:
        return None
    units = tiles * splitk
    grid = min(units, NUM_SMS)
    if splitk > 1:
        epi = "atomic"
    elif tma:
        epi = "tma" if BN % 32 == 0 else "tma+reg"      # chunks of fewer than 32 tile columns leave by registers
    elif ldc % 4 == 0 and c_align % 16 == 0:
        epi = "vec"
    else:
        epi = "scalar"
    return {"BN": BN, "few_waves": few, "splitk": splitk, "kb_per": kb_per, "num_kb": num_kb,
            "splits": [min(num_kb, (s + 1) * kb_per) - s * kb_per for s in range(splitk)], "astat": astat,
            "stages": stages, "epi": epi, "tmem_cols": 256 if 2 * BN <= 256 else 512, "tiles": tiles, "grid": grid,
            "units_per_cta": cdiv(units, grid), "ksteps_last": cdiv(K - (num_kb - 1) * BK, 16),
            "memset": None if splitk == 1 else ("1d" if ldc == N else "2d")}


def f32_plan(K, splitk):
    """caphn_gemm_f32: (kchunk, effective split count)."""
    splitk = max(1, splitk)
    kchunk = cdiv(cdiv(K, splitk), 16) * 16
    return kchunk, cdiv(K, kchunk)


# ----------------------------------------------------------------------------------------------------------------------
# operand format
# ----------------------------------------------------------------------------------------------------------------------
def split_ref(x):
    """The bf16x3 operand format of a float32 tensor: (hi, lo) = (rn_bf16(x), rn_bf16(x - hi))."""
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


NAN_BF16 = -0x0053          # 0xFFAD as int16: a NaN bf16 pattern for padding no kernel may read
SENTINEL = 0x7FBADBAD       # a NaN fp32 pattern no kernel writes


def place(x, mn, split, ld=None, pad=None):
    """A K-major ([rows, K]) or MN-major ([K, rows]) operand holding x [rows, K] in bf16x3 format (lo None in bf16 mode)
    with row pitch ld (default round64 of the inner extent).  The pitch padding holds ``pad`` (an int16 bit pattern;
    default zero): the kernel's TMA boxes clip at the inner extent, so a NaN there must never reach C."""
    from hypernet_image_captioning_b200 import ops
    rows, K = x.shape
    src = x.t() if mn else x
    outer, inner = src.shape
    ld = ld or round64(inner)
    hi, lo = split_ref(src.contiguous())
    out = []
    for p in (hi, lo) if split else (hi,):
        buf = torch.zeros(outer, ld, dtype=torch.bfloat16, device=x.device)
        if pad is not None:
            buf.view(torch.int16).fill_(pad)
        buf[:, :inner] = p
        out.append(buf)
    return ops.SplitOperand(out[0], out[1] if split else None, rows, K, ld, mn)


# ----------------------------------------------------------------------------------------------------------------------
# data
# ----------------------------------------------------------------------------------------------------------------------
def _gen(seed, device):
    return torch.Generator(device=device).manual_seed(seed)


def placement_operand(rows, K, seed, device="cpu"):
    """Integers in [-8, 8]; the last column is nonzero, so a dropped K-tail step changes every row."""
    g = _gen(seed, device)
    x = torch.randint(-8, 9, (rows, K), generator=g, device=device).float()
    x[:, -1] = torch.randint(1, 9, (rows,), generator=g, device=device).float() * (1 - 2 * (torch.arange(
        rows, device=device) % 2)).float()
    return x


def loterm_operand(rows, K, seed, device="cpu", exps=True):
    """x = (h + l) 2^s: h in {+-1, +-2}, l in {-1, 0, 1} 2^-10, s in [-3, 3] per row (0 with exps=False).  hi = h 2^s and
    lo = l 2^s exactly; the last column has l != 0."""
    g = _gen(seed, device)
    h = torch.tensor([-2.0, -1.0, 1.0, 2.0], device=device)[torch.randint(0, 4, (rows, K), generator=g, device=device)]
    l = torch.randint(-1, 2, (rows, K), generator=g, device=device).float()
    l[:, -1] = 1.0
    x = h + l * 2.0 ** -10
    if exps:
        x = x * 2.0 ** torch.randint(-3, 4, (rows, 1), generator=g, device=device).float()
    return x


def float_operand(rows, K, seed, device="cpu", smin=-8, smax=8):
    """Gaussian rows scaled by 2^s, s uniform in [smin, smax] per row (power-of-two scaling commutes with the split)."""
    g = _gen(seed, device)
    s = torch.randint(smin, smax + 1, (rows, 1), generator=g, device=device).float()
    return torch.randn(rows, K, generator=g, device=device) * 2.0 ** s


def int_bias(N, seed, device="cpu"):
    g = _gen(seed + 7, device)
    return torch.randint(-20, 21, (N,), generator=g, device=device).float()


def alpha_of(scale):
    """scale = None or (num, den) host floats (den None allowed): the epilogue's num / max(den, 1)."""
    if scale is None:
        return 1.0
    num, den = scale
    return num / max(1.0 if den is None else den, 1.0)


# ----------------------------------------------------------------------------------------------------------------------
# references
# ----------------------------------------------------------------------------------------------------------------------
def terms(a, b, split=True, k0=0, k1=None):
    """(hh, hl, lh) in float64 over k in [k0, k1) for fp32 operands a [M, K], b [N, K] (hl = lh = None in bf16 mode)."""
    k1 = a.shape[1] if k1 is None else k1
    ah, al = (t.double() for t in split_ref(a[:, k0:k1].contiguous()))
    bh, bl = (t.double() for t in split_ref(b[:, k0:k1].contiguous()))
    if not split:
        return ah @ bh.t(), None, None
    return ah @ bh.t(), ah @ bl.t(), al @ bh.t()


def product(a, b, split=True, k0=0, k1=None):
    hh, hl, lh = terms(a, b, split, k0, k1)
    return hh if not split else hh + hl + lh


def epilogue(acc, bias=None, scale=None, relu=False):
    out = acc * alpha_of(scale)
    if bias is not None:
        out = out + bias.double()
    return out.clamp_min(0.0) if relu else out


def elem_err(got, ref, a, b, bias=None, scale=None):
    """Largest |got - ref| / (|alpha| |A| |B|^T + |bias|) over the elements: the error of each element relative to the
    magnitudes that entered it, so rows of small magnitude count as much as the largest."""
    den = a.double().abs() @ b.double().abs().t() * abs(alpha_of(scale))
    if bias is not None:
        den = den + bias.double().abs()
    return float(((got.double() - ref.double()).abs() / den.clamp_min(1e-300)).max())


def bound_tc(K, split=True):
    """Analytic per-element bound of elem_err for the tensor-core GEMM.  Format: |x - hi| <= 2^-8 |x| and
    |x - hi - lo| <= 2^-16 |x|, so one bf16x3 product misses at most 3 2^-16 |a b| (lo.lo and the two residuals; bf16 mode:
    2 2^-8 + 2^-16).  Accumulation: 3 ceil(K/16) MMA adds into fp32 with truncation (at most 2^-23 each relative to the
    running sum of |a b|; 1 add per k-step in bf16 mode), plus the scale product and the bias add (2^-23 each)."""
    adds = (3 if split else 1) * cdiv(K, 16) + 2
    fmt = 3 * 2.0 ** -16 if split else 2 * 2.0 ** -8 + 2.0 ** -16
    return (fmt + adds * 2.0 ** -23) * (1 + 1e-3)


def bound_f32(K, splitk=1):
    """caphn_gemm_f32: K fp32 FMAs rounded to nearest, splitk atomic adds and the bias add: gamma_n = n 2^-24 / (1 - n 2^-24)
    relative to |A| |B|^T + |bias|."""
    n = K + splitk + 2
    return n * 2.0 ** -24 / (1 - n * 2.0 ** -24)


# ----------------------------------------------------------------------------------------------------------------------
# output buffers: [M, N] views of a sentinel-filled buffer, with the row pitch and alignment under test
# ----------------------------------------------------------------------------------------------------------------------
def out_buffer(M, N, ldc, col0=0, device="cuda"):
    """(buffer, view): buffer of (M + 2) rows x ldc + 8 floats filled with SENTINEL, view = [M, N] with row pitch ldc
    starting one row + col0 floats in (col0 = 1 gives a C that is 4- but not 16-byte aligned)."""
    total = (M + 2) * ldc + 8
    buf = torch.empty(total, dtype=torch.int32, device=device).fill_(SENTINEL).view(torch.float32)
    view = buf[ldc + col0:].as_strided((M, N), (ldc, 1))
    return buf, view


def expected_buffer(buf, ldc, col0, ref):
    exp = torch.empty_like(buf).view(torch.int32).fill_(SENTINEL).view(torch.float32)
    M, N = ref.shape
    exp[ldc + col0:].as_strided((M, N), (ldc, 1)).copy_(ref.to(exp.device, torch.float32))
    return exp


def mismatches(got, exp):
    """Elements whose bits differ, where the values are not equal either (+0 and -0 count as equal; a NaN sentinel only
    matches itself bit for bit)."""
    gb, eb = got.view(torch.int32), exp.view(torch.int32)
    return int(((gb != eb) & ~(got == exp)).sum())


# ----------------------------------------------------------------------------------------------------------------------
# grouped mode: the unit record semantics (caphn_gemm_tc_grouped), interpreted in float64
# ----------------------------------------------------------------------------------------------------------------------
def grouped_ref(Aop, a_mn, Bop, b_mn, C, ldc, units, BN, bias=None, rowmap=None):
    """Apply every unit record of ``units`` (int32 [n, 12]) to the float64 copy C (flat) and return it.  Aop / Bop are the
    SplitOperand arrays the kernel reads: K-major [rows, ld] (k = column) or MN-major [K rows, ld] (mn = column); what
    lies past the array reads as zero."""
    def tile(op, mn, r0, k0, nrows, nk):
        planes = [op.hi.double()] + ([op.lo.double()] if op.lo is not None else [])
        out = []
        for p in planes:
            if mn:
                p = p.t()                                  # [mn, K]
            t = torch.zeros(nrows, nk, dtype=torch.float64, device=p.device)
            rr, kk = min(nrows, max(0, p.shape[0] - r0)), min(nk, max(0, p.shape[1] - k0))
            t[:rr, :kk] = p[r0:r0 + rr, k0:k0 + kk]
            out.append(t)
        return out
    C = C.double().clone()
    for u in units.cpu().tolist():
        a_row, b_row, ka0, kb0, nkb, mv, nv, boff, map0, c_lo, c_hi, _ = u
        c_off = (c_hi << 32) | (c_lo & 0xFFFFFFFF)
        A = tile(Aop, a_mn, a_row, ka0, BM, nkb * BK)
        B = tile(Bop, b_mn, b_row, kb0, BN, nkb * BK)
        acc = A[0] @ B[0].t()
        if len(A) == 2:
            acc = acc + A[0] @ B[1].t() + A[1] @ B[0].t()
        for r in range(mv):
            orow = r if rowmap is None else int(rowmap[map0 + r])
            if orow < 0:
                continue
            v = acc[r, :nv]
            if bias is not None:
                v = v + bias.double()[boff:boff + nv]
            C[c_off + orow * ldc: c_off + orow * ldc + nv] = v
    return C


# ----------------------------------------------------------------------------------------------------------------------
# planted defects: the reference output as a plausible kernel bug would leave it
# ----------------------------------------------------------------------------------------------------------------------
MUTANTS = ("last K-tail step dropped", "lo.hi missing on one tile", "bias shifted one column", "scale without den",
           "scale applied twice on split-K partials", "one split-K partial lost", "rows of two m-tiles swapped",
           "write one column past n_valid")


def mutant_needs(mutant):
    """What a shape needs for the defect to exist: split-K, two m-tiles, a bias, a den, the lo terms."""
    return {"scale applied twice on split-K partials": "splitk", "one split-K partial lost": "splitk",
            "rows of two m-tiles swapped": "two m-tiles", "bias shifted one column": "bias",
            "scale without den": "den", "lo.hi missing on one tile": "split"}.get(mutant)


def mutate(mutant, a, b, plan, split=True, bias=None, scale=None):
    """The [M, N] output (float64) with one planted defect, for operands a [M, K], b [N, K] and the launch ``plan``.
    "write one column past n_valid" returns the correct [M, N] block plus the extra column ([M, N + 1])."""
    K = a.shape[1]
    acc = product(a, b, split)
    if mutant == "last K-tail step dropped":
        acc = acc - product(a, b, split, 16 * (cdiv(K, 16) - 1), K)
    elif mutant == "lo.hi missing on one tile":
        _, _, lh = terms(a[:BM], b[:plan["BN"]], split)
        acc = acc.clone()
        acc[:BM, :plan["BN"]] -= lh
    elif mutant == "one split-K partial lost":
        k0 = plan["kb_per"] * BK
        acc = acc - product(a, b, split, k0, min(K, 2 * k0))
    elif mutant == "scale applied twice on split-K partials":
        return epilogue(acc * alpha_of(scale), bias, scale)
    elif mutant == "scale without den":
        return epilogue(acc * scale[0] / alpha_of(scale), bias, scale)
    elif mutant == "bias shifted one column":
        sh = torch.zeros_like(bias)
        sh[:-1] = bias[1:]
        return epilogue(acc, sh, scale)
    out = epilogue(acc, bias, scale)
    if mutant == "rows of two m-tiles swapped":
        n = min(BM, out.shape[0] - BM)
        out = out.clone()
        out[:n], out[BM:BM + n] = out[BM:BM + n].clone(), out[:n].clone()
    elif mutant == "write one column past n_valid":
        out = torch.cat([out, torch.zeros_like(out[:, :1])], 1)
    return out
