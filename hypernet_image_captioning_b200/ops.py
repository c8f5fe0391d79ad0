"""Tensor-level wrappers over the C-ABI (device pointers in, nothing computed on the host).

torch is used here for memory (allocation, views) and the current CUDA stream only.
"""
from typing import Optional

import torch

from . import _cabi

LEAKY_SLOPE = 0.01
ACT_NONE, ACT_LEAKY = 0, 1


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _chk(t: torch.Tensor, dtype=torch.float32):
    if not t.is_cuda:
        raise _cabi.CaphnError("caphn ops need CUDA tensors (there is no CPU fallback)")
    if t.dtype != dtype:
        raise _cabi.CaphnError(f"expected {dtype}, got {t.dtype}")
    return t


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


# ----------------------------------------------------------------------------------------------------------------------
# hypernet linear layers (weight streaming)
# ----------------------------------------------------------------------------------------------------------------------
def rows_linear_fwd(W, bias, A, act=ACT_NONE, out=None, slope=LEAKY_SLOPE):
    """Y[g,n] = act(A[g,:] . W[n,:] + bias[n]).  A [G,K] (row stride may exceed K), W [N,K] contiguous.
    ``out`` may be a column slice of a wider matrix (e.g. theta[:, a:b])."""
    _chk(W, W.dtype if W.dtype == torch.bfloat16 else torch.float32), _chk(A)
    W = _aligned16(W)
    N, K = W.shape
    G = A.shape[0]
    assert A.shape[1] == K and A.stride(1) == 1
    if bias is not None and bias.dtype != torch.float32:
        bias = bias.float()
    if out is None:
        out = torch.empty(G, N, device=W.device, dtype=torch.float32)
    assert out.shape == (G, N) and out.stride(1) == 1
    fn = "caphn_rows_linear_fwd_bf16" if W.dtype == torch.bfloat16 else "caphn_rows_linear_fwd"
    for g0 in range(0, G, 8):
        g1 = min(G, g0 + 8)
        _cabi.call(fn, W.data_ptr(), _p(bias), A[g0:g1].data_ptr(), A.stride(0),
                   out[g0:g1].data_ptr(), out.stride(0), g1 - g0, N, K, act, slope, _stream())
    return out


def rows_linear_bwd(W, A, Y, dY, act=ACT_NONE, need_dW=True, need_dA=True, dA=None, slope=LEAKY_SLOPE, return_dP=False):
    """Backward of rows_linear_fwd.  Returns (dW [N,K] or None, dbias [N], dA [G,K] or None).
    When ``dA`` is given the input gradient is accumulated into it (atomics)."""
    _chk(W, W.dtype if W.dtype == torch.bfloat16 else torch.float32), _chk(A), _chk(dY)
    W = _aligned16(W)
    N, K = W.shape
    G = A.shape[0]
    assert dY.shape == (G, N) and dY.stride(1) == 1 and A.stride(1) == 1
    if act != ACT_NONE:
        assert Y is not None and Y.shape == (G, N) and Y.stride(1) == 1
    dev = W.device
    dP = torch.empty(G, N, device=dev, dtype=torch.float32)
    dbias = torch.empty(N, device=dev, dtype=torch.float32)
    dW = torch.empty(N, K, device=dev, dtype=W.dtype) if need_dW else None   # bf16 weights -> bf16 gradient; None: dA-only pass
    if need_dA and dA is None:
        dA = torch.zeros(G, K, device=dev, dtype=torch.float32)
    if not need_dA:
        dA = None
    _cabi.call("caphn_rows_linear_bwd_bf16" if W.dtype == torch.bfloat16 else "caphn_rows_linear_bwd", W.data_ptr(), A.data_ptr(), A.stride(0), _p(Y), Y.stride(0) if Y is not None else 0,
               dY.data_ptr(), dY.stride(0), dP.data_ptr(), _p(dW), dbias.data_ptr(), _p(dA),
               dA.stride(0) if dA is not None else 0, G, N, K, act, slope, _stream())
    if return_dP:
        return dW, dbias, dA, dP
    return dW, dbias, dA


# ----------------------------------------------------------------------------------------------------------------------
# dense fp32 GEMMs
# ----------------------------------------------------------------------------------------------------------------------
def _gemm(A, lda, a_k, Bm, ldb, b_k, M, N, K, bias=None, relu=False, out=None, splitk=1, accumulate=False):
    if out is None:
        if splitk > 1 or accumulate:
            out = torch.zeros(M, N, device=A.device, dtype=torch.float32)
        else:
            out = torch.empty(M, N, device=A.device, dtype=torch.float32)
    assert out.stride(-1) == 1
    _cabi.call("caphn_gemm_f32", A.data_ptr(), lda, int(a_k), Bm.data_ptr(), ldb, int(b_k), out.data_ptr(),
               out.stride(0), _p(bias), M, N, K, int(relu), splitk, int(accumulate), _stream())
    return out


def _auto_splitk(M, N, K):
    tiles = ((M + 127) // 128) * ((N + 127) // 128)
    if tiles >= 148 or K <= 512:
        return 1
    return max(1, min((K + 255) // 256, (2 * 148 + tiles - 1) // tiles))


TC_ENABLED = True   # route the large dense contractions to the tcgen05 kernel (bf16x3, fp32-class accuracy)
TC_SPLIT = True     # True: bf16x3 (hi/lo split, fp32-class accuracy); False: single bf16 MMA per k-slice ("bf16 mode")


def set_precision(mode: str):
    """"fp32": tensor-core products use the bf16x3 split (1e-5-class).  "bf16": plain bf16 operands, fp32 accumulate."""
    global TC_SPLIT
    if mode not in ("fp32", "bf16"):
        raise ValueError(mode)
    TC_SPLIT = mode == "fp32"
TC_MIN_WORK = 1 << 24


def _tc_ok(M, N, K, accumulate=False):
    return TC_ENABLED and not accumulate and M >= 128 and N >= 16 and K >= 32 and M * N * K >= TC_MIN_WORK


def _operand_of_transpose(Bm):
    """B operand ([N, K]) of a product with Bm = [K, N] stored row-major.  Large matrices are read in place (MN-major; the
    N tile is then a multiple of 64); small ones go through the transposing split so the N tile can hug N (e.g. 160)."""
    if Bm.numel() >= (1 << 22) and (Bm.shape[1] > 256 or Bm.shape[1] % 64 == 0):
        return split_bf16(Bm, mn=True)
    return split_bf16_t(Bm)


def linear(X, W, bias=None, relu=False, out=None):
    """out[M,N] = X[M,K] @ W[N,K]^T + bias (optional ReLU)."""
    _chk(X), _chk(W)
    assert X.dim() == 2 and X.stride(1) == 1 and W.stride(1) == 1 and X.shape[1] == W.shape[1]
    if _tc_ok(X.shape[0], W.shape[0], X.shape[1]):
        return gemm_tc(split_bf16(X), split_bf16(W), bias=bias, relu=relu, out=out)
    return _gemm(X, X.stride(0), 1, W, W.stride(0), 1, X.shape[0], W.shape[0], X.shape[1], bias, relu, out)


def matmul_nn(A, Bm, out=None, accumulate=False):
    """out[M,N] = A[M,K] @ B[K,N]."""
    _chk(A), _chk(Bm)
    assert A.stride(1) == 1 and Bm.stride(1) == 1 and A.shape[1] == Bm.shape[0]
    if _tc_ok(A.shape[0], Bm.shape[1], A.shape[1], accumulate):
        return gemm_tc(split_bf16(A), _operand_of_transpose(Bm), out=out)
    return _gemm(A, A.stride(0), 1, Bm, Bm.stride(0), 0, A.shape[0], Bm.shape[1], A.shape[1], out=out,
                 accumulate=accumulate)


def matmul_tn(A, Bm, out=None, accumulate=False):
    """out[M,N] = A[K,M]^T @ B[K,N]   (weight gradients: dW = dY^T X); split-K when the output is small."""
    _chk(A), _chk(Bm)
    assert A.stride(1) == 1 and Bm.stride(1) == 1 and A.shape[0] == Bm.shape[0]
    K, M = A.shape
    N = Bm.shape[1]
    if _tc_ok(M, N, K, accumulate):
        return gemm_tc(split_bf16(A, mn=True), _operand_of_transpose(Bm), out=out)
    sk = _auto_splitk(M, N, K)
    if out is not None and sk > 1 and not accumulate:
        out.zero_()
    return _gemm(A, A.stride(0), 0, Bm, Bm.stride(0), 0, M, N, K, out=out, splitk=sk, accumulate=accumulate)


def colsum(X, out=None):
    """out[n] (+)= sum_m X[m,n]."""
    _chk(X)
    assert X.dim() == 2 and X.stride(1) == 1
    if out is None:
        out = torch.zeros(X.shape[1], device=X.device, dtype=torch.float32)
    _cabi.call("caphn_colsum", X.data_ptr(), X.stride(0), X.shape[0], X.shape[1], out.data_ptr(), _stream())
    return out


def transpose_pad(src, ldd):
    """dst [C, ldd] with dst[c, r] = src[r, c], zero padded."""
    _chk(src)
    R, C = src.shape
    assert src.stride(1) == 1
    dst = torch.empty(C, ldd, device=src.device, dtype=torch.float32)
    _cabi.call("caphn_transpose_pad", src.data_ptr(), src.stride(0), dst.data_ptr(), ldd, R, C, _stream())
    return dst


def copy_pad(src, ldd):
    _chk(src)
    R, C = src.shape
    assert src.stride(1) == 1
    if ldd == C and src.is_contiguous() and src.stride(0) == C and src.data_ptr() % 16 == 0:
        return src
    dst = torch.empty(R, ldd, device=src.device, dtype=torch.float32)
    _cabi.call("caphn_copy_pad", src.data_ptr(), src.stride(0), dst.data_ptr(), ldd, R, C, _stream())
    return dst


def transpose_pad_batched(src, R, C, ldd):
    """src [nb, R*C]: row z holds a matrix [R, C] (e.g. the W_hh block of every row of Theta, a column slice).  Returns
    dst [nb, C, ldd] with dst[z, c, r] = src_z[r, c], zero padded; one launch for all nb."""
    _chk(src)
    nb = src.shape[0]
    assert src.dim() == 2 and src.stride(1) == 1 and src.shape[1] == R * C
    dst = torch.empty(nb, C, ldd, device=src.device, dtype=torch.float32)
    _cabi.call("caphn_transpose_pad_batched", src.data_ptr(), src.stride(0), C, dst.data_ptr(), C * ldd, ldd, nb, R, C,
               _stream())
    return dst


def copy_pad_batched(src, R, C, ldd):
    """src [nb, R*C] as in transpose_pad_batched -> dst [nb, R, ldd] with dst[z, r, c] = src_z[r, c], zero padded."""
    _chk(src)
    nb = src.shape[0]
    assert src.dim() == 2 and src.stride(1) == 1 and src.shape[1] == R * C
    dst = torch.empty(nb, R, ldd, device=src.device, dtype=torch.float32)
    _cabi.call("caphn_copy_pad_batched", src.data_ptr(), src.stride(0), C, dst.data_ptr(), R * ldd, ldd, nb, R, C,
               _stream())
    return dst


def round4(n):
    return (n + 3) // 4 * 4


# ----------------------------------------------------------------------------------------------------------------------
# recurrences
# ----------------------------------------------------------------------------------------------------------------------
def _ptr_array(tensors):
    import ctypes
    arr = (ctypes.c_void_p * max(1, len(tensors)))(*[t.data_ptr() for t in tensors])
    return arr


def gru_seq_fwd(GI, WhhT, bhh, h0, T, save=True, want_bm=True, extra=()):
    """GI [T*B,3H] time-major, WhhT [H,ld3]; ``extra`` = [(WihT_l, WhhT_l, bih_l, bhh_l), ...] for layers 1..NL-1.
    Returns Hall [T+1,B,H], Hbm [B,T,H] | None, saved [NL,4,T,B,H] | None, Hmid [NL-1,T,B,H] | None."""
    B, H = h0.shape
    NL = 1 + len(extra)
    dev = GI.device
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32) if want_bm else None
    saved = torch.empty(NL, 4, T, B, H, device=dev, dtype=torch.float32) if save else None
    Hmid = torch.empty(NL - 1, T, B, H, device=dev, dtype=torch.float32) if (save and NL > 1) else None
    flat = [t for cell in extra for t in cell]
    arr = _ptr_array(flat)
    _cabi.call("caphn_gru_seq_fwd", GI.data_ptr(), WhhT.data_ptr(), WhhT.stride(0), bhh.data_ptr(), Hall.data_ptr(),
               _p(Hbm), _p(saved), _p(Hmid), arr if NL > 1 else None, NL, B, T, H, _stream())
    return Hall, Hbm, saved, Hmid


def lstm_seq_fwd(GI, WhhT, bhh, h0, T, save=True, want_bm=True, extra=(), c0=None, want_c=False):
    """LSTM analogue of gru_seq_fwd: GI [T*B,4H], WhhT [H,ld4]; saved [NL,6,T,B,H] = (i, f, g, o, c_prev, tanh c)."""
    B, H = h0.shape
    NL = 1 + len(extra)
    dev = GI.device
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32) if want_bm else None
    saved = torch.empty(NL, 6, T, B, H, device=dev, dtype=torch.float32) if save else None
    Hmid = torch.empty(NL - 1, T, B, H, device=dev, dtype=torch.float32) if (save and NL > 1) else None
    arr = _ptr_array([t for cell in extra for t in cell])
    cT = torch.empty(B, H, device=dev, dtype=torch.float32) if want_c else None
    _cabi.call("caphn_lstm_seq_fwd", GI.data_ptr(), WhhT.data_ptr(), WhhT.stride(0), bhh.data_ptr(), Hall.data_ptr(),
               _p(Hbm), _p(saved), _p(Hmid), arr if NL > 1 else None, _p(c0), _p(cT), NL, B, T, H, _stream())
    if want_c:
        return Hall, Hbm, saved, Hmid, cT
    return Hall, Hbm, saved, Hmid


def lstm_seq_bwd(dHbm, saved, Hall, Whh_p, extra=()):
    """``extra`` = [(Wih_l, Whh_l) padded [4H,ldh], ...].  Returns dG [NL, T*B, 4H], dh0 [B,H]."""
    Tp1, B, H = Hall.shape
    T = Tp1 - 1
    NL = 1 + len(extra)
    dev = Hall.device
    dG = torch.empty(NL, T * B, 4 * H, device=dev, dtype=torch.float32)
    dh0 = torch.empty(B, H, device=dev, dtype=torch.float32)
    assert dHbm.is_contiguous()
    arr = _ptr_array([t for cell in extra for t in cell])
    _cabi.call("caphn_lstm_seq_bwd", dHbm.data_ptr(), saved.data_ptr(), Whh_p.data_ptr(), Whh_p.stride(0),
               arr if NL > 1 else None, dG.data_ptr(), dh0.data_ptr(), NL, B, T, H, _stream())
    return dG, dh0


def _at_cqt(ld):
    return min(512, max(32, 1 << max(0, (ld // 4 - 1).bit_length())))


def lstm_seq_fits(H):
    """Whether the single-layer LSTM recurrence (forward and BPTT) fits the 227 KB of shared memory of one CTA at hidden
    size H: the same sizes the entry points of csrc/lstm_seq.cu check."""
    ld4, ldh = round4(4 * H), round4(H)
    fwd = H * 4 + round4(4 * H) + 2 * (512 // _at_cqt(ld4)) * 4 * ld4
    bwd = 16 * H + 2 * round4(4 * H) + 2 * (512 // _at_cqt(ldh)) * 4 * ldh
    return 4 * max(fwd, bwd) <= 227 * 1024


def lstm_seq_fwd_grouped(GI, WhhT, bhh, h0, T, tiles, want_c=False):
    """Single-layer LSTM recurrence of a batch sorted by style group.  GI [T*B, 4H]; WhhT [G, H, ld4] (one W_hh^T per
    group); bhh [G, 4H] (row stride free, e.g. a column slice of Theta); tiles int32 [n, 4] = (first row, rows <= 4,
    group, 0).  Returns Hall [T+1,B,H], Hbm [B,T,H], saved [6,T,B,H] (+ cT [B,H] with ``want_c``)."""
    B, H = h0.shape
    dev = GI.device
    _chk(GI), _chk(WhhT), _chk(bhh), _chk(tiles, torch.int32)
    assert WhhT.is_contiguous() and WhhT.shape[1] == H and bhh.stride(1) == 1 and tiles.is_contiguous()
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32)
    saved = torch.empty(6, T, B, H, device=dev, dtype=torch.float32)
    cT = torch.empty(B, H, device=dev, dtype=torch.float32) if want_c else None
    _cabi.call("caphn_lstm_seq_fwd_grouped", GI.data_ptr(), WhhT.data_ptr(), WhhT.shape[2], bhh.data_ptr(), bhh.stride(0),
               Hall.data_ptr(), Hbm.data_ptr(), saved.data_ptr(), _p(cT), B, T, H, tiles.data_ptr(), tiles.shape[0],
               _stream())
    if want_c:
        return Hall, Hbm, saved, cT
    return Hall, Hbm, saved


def lstm_seq_bwd_grouped(dHbm, saved, Hall, Whh_p, tiles):
    """BPTT of lstm_seq_fwd_grouped; Whh_p [G, 4H, ldh] (one padded W_hh per group).  Returns dG [T*B, 4H], dh0 [B, H]."""
    Tp1, B, H = Hall.shape
    T = Tp1 - 1
    dev = Hall.device
    _chk(dHbm), _chk(saved), _chk(Whh_p), _chk(tiles, torch.int32)
    assert dHbm.is_contiguous() and saved.is_contiguous() and Whh_p.is_contiguous() and tiles.is_contiguous()
    dG = torch.empty(T * B, 4 * H, device=dev, dtype=torch.float32)
    dh0 = torch.empty(B, H, device=dev, dtype=torch.float32)
    _cabi.call("caphn_lstm_seq_bwd_grouped", dHbm.data_ptr(), saved.data_ptr(), Whh_p.data_ptr(), Whh_p.shape[2],
               dG.data_ptr(), dh0.data_ptr(), B, T, H, tiles.data_ptr(), tiles.shape[0], _stream())
    return dG, dh0


_cluster_plan_cache = {}


def gru_cluster_size(H):
    """Cluster size of the weights-resident GRU kernels for hidden size H (0 = not applicable)."""
    if H not in _cluster_plan_cache:
        import ctypes
        cs = ctypes.c_int(0)
        _cabi.call("caphn_gru_cluster_plan", H, ctypes.byref(cs))
        _cluster_plan_cache[H] = int(cs.value)
    return _cluster_plan_cache[H]


_resident_plan_cache = {}


def gru_resident_ok(H):
    """True when the CTA-resident GRU kernels (csrc/gru_resident.cu) apply to hidden size H."""
    if H not in _resident_plan_cache:
        import ctypes
        ok = ctypes.c_int(0)
        _cabi.call("caphn_gru_resident_plan", H, ctypes.byref(ok))
        _resident_plan_cache[H] = bool(ok.value)
    return _resident_plan_cache[H]


def gru_resident_fwd(GI, W_hh, bhh, h0, T, save=True, want_bm=True):
    """Single-layer recurrence with the whole W_hh resident in one CTA per 4 rows.  Same returns as gru_seq_fwd."""
    B, H = h0.shape
    dev = GI.device
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32) if want_bm else None
    saved = torch.empty(1, 4, T, B, H, device=dev, dtype=torch.float32) if save else None
    _cabi.call("caphn_gru_resident_fwd", GI.data_ptr(), W_hh.data_ptr(), bhh.data_ptr(), Hall.data_ptr(), _p(Hbm),
               _p(saved), B, T, H, _stream())
    return Hall, Hbm, saved, None


def gru_resident_bwd(dHbm, saved, Hall, W_hh):
    Tp1, B, H = Hall.shape
    T = Tp1 - 1
    dev = Hall.device
    dGI = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
    dGH = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
    dh0 = torch.empty(B, H, device=dev, dtype=torch.float32)
    assert dHbm.is_contiguous()
    _cabi.call("caphn_gru_resident_bwd", dHbm.data_ptr(), saved.data_ptr(), Hall.data_ptr(), W_hh.data_ptr(),
               dGI.data_ptr(), dGH.data_ptr(), dh0.data_ptr(), B, T, H, _stream())
    return dGI, dGH, None, None, dh0


def gru_cluster_fwd(GI, W_hh, bhh, h0, T, save=True, want_bm=True):
    """Single-layer recurrence with W_hh resident in shared memory (cluster + DSMEM).  Same returns as gru_seq_fwd."""
    B, H = h0.shape
    dev = GI.device
    Hall = torch.empty(T + 1, B, H, device=dev, dtype=torch.float32)
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device=dev, dtype=torch.float32) if want_bm else None
    saved = torch.empty(1, 4, T, B, H, device=dev, dtype=torch.float32) if save else None
    _cabi.call("caphn_gru_cluster_fwd", GI.data_ptr(), W_hh.data_ptr(), bhh.data_ptr(), Hall.data_ptr(), _p(Hbm),
               _p(saved), B, T, H, _stream())
    return Hall, Hbm, saved, None


def gru_cluster_bwd(dHbm, saved, Hall, W_hh):
    Tp1, B, H = Hall.shape
    T = Tp1 - 1
    dev = Hall.device
    dGI = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
    dGH = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
    dh0 = torch.empty(B, H, device=dev, dtype=torch.float32)
    assert dHbm.is_contiguous()
    _cabi.call("caphn_gru_cluster_bwd", dHbm.data_ptr(), saved.data_ptr(), Hall.data_ptr(), W_hh.data_ptr(),
               dGI.data_ptr(), dGH.data_ptr(), dh0.data_ptr(), B, T, H, _stream())
    return dGI, dGH, None, None, dh0


def gru_seq_bwd(dHbm, saved, Hall, Hmid, Whh_p, extra=()):
    """``extra`` = [(Wih_l, Whh_l) padded [3H,ldh], ...].  Returns dGI, dGH [T*B,3H], xdGI, xdGH [NL-1,T*B,3H] | None, dh0."""
    Tp1, B, H = Hall.shape
    T = Tp1 - 1
    NL = 1 + len(extra)
    dev = Hall.device
    dGI = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
    dGH = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
    xdGI = torch.empty(NL - 1, T * B, 3 * H, device=dev, dtype=torch.float32) if NL > 1 else None
    xdGH = torch.empty(NL - 1, T * B, 3 * H, device=dev, dtype=torch.float32) if NL > 1 else None
    dh0 = torch.empty(B, H, device=dev, dtype=torch.float32)
    assert dHbm.is_contiguous()
    flat = [t for cell in extra for t in cell]
    arr = _ptr_array(flat)
    _cabi.call("caphn_gru_seq_bwd", dHbm.data_ptr(), saved.data_ptr(), Hall.data_ptr(), _p(Hmid), Whh_p.data_ptr(),
               Whh_p.stride(0), arr if NL > 1 else None, dGI.data_ptr(), dGH.data_ptr(), _p(xdGI), _p(xdGH),
               dh0.data_ptr(), NL, B, T, H, _stream())
    return dGI, dGH, xdGI, xdGH, dh0


# ----------------------------------------------------------------------------------------------------------------------
# cross-entropy, softmax/argmax, embedding
# ----------------------------------------------------------------------------------------------------------------------
def ce_fwd(logits2d, targets, ignore_index):
    """Returns (lossbuf [2] = (mean loss, #valid rows), lse [M])."""
    _chk(logits2d), _chk(targets, torch.int64)
    M, V = logits2d.shape
    assert logits2d.stride(1) == 1 and targets.is_contiguous() and targets.numel() == M
    dev = logits2d.device
    lse = torch.empty(M, device=dev, dtype=torch.float32)
    scratch = torch.empty(2 * M, device=dev, dtype=torch.float32)
    lossbuf = torch.empty(2, device=dev, dtype=torch.float32)
    has = ignore_index is not None
    _cabi.call("caphn_ce_fwd", logits2d.data_ptr(), logits2d.stride(0), targets.data_ptr(), M, V, int(has),
               int(ignore_index) if has else 0, lse.data_ptr(), scratch.data_ptr(), lossbuf.data_ptr(), _stream())
    return lossbuf, lse


def ce_bwd(logits2d, targets, ignore_index, lse, lossbuf, gscale):
    M, V = logits2d.shape
    dX = torch.empty(M, V, device=logits2d.device, dtype=torch.float32)
    has = ignore_index is not None
    _cabi.call("caphn_ce_bwd", logits2d.data_ptr(), logits2d.stride(0), targets.data_ptr(), M, V, int(has),
               int(ignore_index) if has else 0, lse.data_ptr(), gscale.data_ptr(), lossbuf.data_ptr(), dX.data_ptr(),
               dX.stride(0), _stream())
    return dX


def ce_bwd_split(logits2d, targets, ignore_index, lse, lossbuf, gscale):
    """CE gradient d [M,V] as tensor-core operands, written once: returns (d as K-major operand [M rows, K=V],
    the SAME buffers viewed as the MN-major operand of d^T [V rows, K=M], dbias [V])."""
    M, V = logits2d.shape
    dev = logits2d.device
    Vp, Mp = round64(V), round64(M)
    hi = torch.empty(M, Vp, device=dev, dtype=torch.bfloat16)
    lo = torch.empty(M, Vp, device=dev, dtype=torch.bfloat16) if TC_SPLIT else None
    hiT = loT = None
    dbias = torch.zeros(V, device=dev, dtype=torch.float32)
    has = ignore_index is not None
    _cabi.call("caphn_ce_bwd_split", logits2d.data_ptr(), logits2d.stride(0), targets.data_ptr(), M, V, int(has),
               int(ignore_index) if has else 0, lse.data_ptr(), gscale.data_ptr(), lossbuf.data_ptr(), hi.data_ptr(),
               _p(lo), Vp, _p(hiT), _p(loT), Mp, dbias.data_ptr(), _stream())
    return SplitOperand(hi, lo, M, V, Vp), SplitOperand(hi, lo, V, M, Vp, True), dbias


CE_FWD_SPLIT_MAX_V = 50000   # the fused kernel stages one row of logits in shared memory


def ce_fwd_split(logits2d, targets, ignore_index):
    """ce_fwd + the UNSCALED CE gradient u = softmax - onehot (0 on ignored rows) as a tensor-core operand, from one read of
    the logits.  Returns (lossbuf, lse, hi, lo): hi / lo [M, round64(V)] bf16 (lo None in bf16 mode), to be viewed as the
    K-major operand of u or the MN-major operand of u^T.  The products that consume them apply grad_output / #valid rows
    (``gemm_tc(..., scale=...)``)."""
    _chk(logits2d), _chk(targets, torch.int64)
    M, V = logits2d.shape
    assert logits2d.stride(1) == 1 and targets.is_contiguous() and targets.numel() == M and V <= CE_FWD_SPLIT_MAX_V
    dev = logits2d.device
    Vp = round64(V)
    lse = torch.empty(M, device=dev, dtype=torch.float32)
    scratch = torch.empty(2 * M, device=dev, dtype=torch.float32)
    lossbuf = torch.empty(2, device=dev, dtype=torch.float32)
    hi = torch.empty(M, Vp, device=dev, dtype=torch.bfloat16)
    lo = torch.empty(M, Vp, device=dev, dtype=torch.bfloat16) if TC_SPLIT else None
    has = ignore_index is not None
    _cabi.call("caphn_ce_fwd_split", logits2d.data_ptr(), logits2d.stride(0), targets.data_ptr(), M, V, int(has),
               int(ignore_index) if has else 0, lse.data_ptr(), scratch.data_ptr(), lossbuf.data_ptr(), hi.data_ptr(),
               _p(lo), Vp, _stream())
    return lossbuf, lse, hi, lo


def softmax_argmax(X, want_probs=True, probs_out=None, want_argmax=True):
    _chk(X)
    M, V = X.shape
    assert X.stride(1) == 1
    Y = None
    if want_probs:
        Y = probs_out if probs_out is not None else torch.empty(M, V, device=X.device, dtype=torch.float32)
        assert Y.stride(1) == 1
    am = torch.empty(M, device=X.device, dtype=torch.int64) if want_argmax else None
    _cabi.call("caphn_softmax_argmax", X.data_ptr(), X.stride(0), M, V, _p(Y), Y.stride(0) if Y is not None else 0,
               _p(am), _stream())
    return Y, am


def gather_rows(table, idx, out=None):
    _chk(table), _chk(idx, torch.int64)
    assert table.is_contiguous()
    idx = idx.contiguous()
    n, E = idx.numel(), table.shape[1]
    if out is None:
        out = torch.empty(n, E, device=table.device, dtype=torch.float32)
    assert out.shape == (n, E) and out.stride(1) == 1
    _cabi.call("caphn_gather_rows", table.data_ptr(), idx.data_ptr(), n, E, out.data_ptr(), out.stride(0), _stream())
    return out


def build_inputs(feat, emb, caps, mode):
    """Time-major decoder inputs X [T*B, E]; mode 0 = pooled decoder (x_0 = feat), 1 = attention decoder (x_0 = x_1 = 0)."""
    _chk(emb), _chk(caps, torch.int64)
    B, T = caps.shape
    E = emb.shape[1]
    X = torch.empty(T * B, E, device=emb.device, dtype=torch.float32)
    _cabi.call("caphn_build_inputs", _p(feat), emb.data_ptr(), caps.data_ptr(), B, T, E, mode, X.data_ptr(), _stream())
    return X


def embed_scatter_add(dX, caps, dEmb, t0):
    B, T = caps.shape
    E = dEmb.shape[1]
    _cabi.call("caphn_embed_scatter_add", dX.data_ptr(), caps.data_ptr(), B, T, E, t0, dEmb.data_ptr(), _stream())
    return dEmb


def scatter_add_rows(dX, idx, table):
    """table[idx[i], :] += dX[i, :] for idx[i] >= 0."""
    _chk(dX), _chk(idx, torch.int64)
    idx = idx.contiguous()
    assert dX.stride(1) == 1 and dX.shape[0] == idx.numel()
    _cabi.call("caphn_scatter_add_rows", dX.data_ptr(), dX.stride(0), idx.data_ptr(), idx.numel(), table.shape[1],
               table.data_ptr(), _stream())
    return table


def mean_pos(X):
    """X [B,P,F] -> mean over P."""
    B, P, Fd = X.shape
    out = torch.empty(B, Fd, device=X.device, dtype=torch.float32)
    _cabi.call("caphn_mean_pos", X.data_ptr(), B, P, Fd, out.data_ptr(), _stream())
    return out


def mean_pos_bwd(g, dX, extra=None):
    """dX[b,p,:] += g[b,:] / P (+ extra[b,p,:])."""
    B, P, Fd = dX.shape
    if extra is not None:
        assert extra.is_contiguous() and extra.numel() == dX.numel()
    _cabi.call("caphn_mean_pos_bwd", g.data_ptr(), _p(extra), B, P, Fd, dX.data_ptr(), _stream())
    return dX


def relu_mask_(ref, y):
    _cabi.call("caphn_relu_mask", ref.data_ptr(), y.data_ptr(), y.numel(), _stream())
    return y


ATT_STEP = True   # two batch-wide kernels per step (attention | tensor-core gates) instead of the persistent streaming kernel


_attstep_sizes = {}


def _attstep_bytes(H, Fd, P, B):
    """(pack bytes, workspace bytes) of the step-split recurrence; pack bytes == 0: shape not covered."""
    key = (H, Fd, P, B)
    if key not in _attstep_sizes:
        import ctypes
        n, w = ctypes.c_long(0), ctypes.c_long(0)
        _cabi.call("caphn_attstep_pack_size", H, Fd, P, B, ctypes.byref(n), ctypes.byref(w))
        _attstep_sizes[key] = (int(n.value), int(w.value))
    return _attstep_sizes[key]


class AttGruWeights:
    """Generated / attention weights laid out for the recurrence kernels: the mma-fragment pack of W_ih[:, E:], W_hh and
    U_a (step-split path, needs the number of positions P), or their k-major transposes with 16-byte rows (persistent
    streaming path)."""

    def __init__(self, W_ih, W_hh, U_a, E, P=None, step=None):
        H = W_hh.shape[1]
        Fd = W_ih.shape[1] - E
        self.ldh, self.ld3, self.ldf = round4(H), round4(3 * H), round4(Fd)
        use_step = (ATT_STEP if step is None else step) and P is not None
        n = _attstep_bytes(H, Fd, P, 0)[0] if use_step else 0
        self.pack = self.UaT = self.WhhT = self.WihcT = self.work = self._resume = None
        if n > 0:
            W_ih, W_hh, U_a = W_ih.contiguous(), W_hh.contiguous(), U_a.contiguous()
            self.pack = torch.empty(n, device=W_hh.device, dtype=torch.uint8)
            _cabi.call("caphn_attstep_pack", W_ih.data_ptr(), W_hh.data_ptr(), U_a.data_ptr(), E, Fd, H,
                       self.pack.data_ptr(), _stream())
        else:
            self.UaT = transpose_pad(U_a, self.ldh)
            self.WhhT = transpose_pad(W_hh, self.ld3)
            self.WihcT = transpose_pad(W_ih[:, E:], self.ld3)


def attgru_fwd(Kp, f, GIw, lw, bu, va, bv, bhh, Hall, Hbm, attn, XC, E, saved, t0, t1):
    """Steps [t0,t1) of the attention-GRU recurrence on whichever layout `lw` was prepared for."""
    if lw.pack is None:
        return attgru_seq_fwd(Kp, f, GIw, lw, bu, va, bv, bhh, Hall, Hbm, attn, XC, E, saved, t0, t1)
    B, P, H = Kp.shape
    Fd = f.shape[2]
    T = Hall.shape[0] - 1
    sp = [saved[i].data_ptr() for i in range(5)] if saved is not None else [None] * 5
    ctx_ptr = XC.data_ptr() + 4 * E
    wbytes = _attstep_bytes(H, Fd, P, B)[1]
    if lw.work is None or lw.work.numel() < wbytes:
        lw.work = torch.empty(wbytes, device=Kp.device, dtype=torch.uint8)
        lw._resume = None
    # one-step-per-call decode: the workspace still holds the operand rows of Hall[t0] from the previous call
    resume = 1 if lw._resume == (Hall.data_ptr(), t0) else 0
    _cabi.call("caphn_attstep_fwd", Kp.data_ptr(), f.data_ptr(), GIw.data_ptr(), bu.data_ptr(), va.data_ptr(),
               bv.data_ptr(), lw.pack.data_ptr(), lw.work.data_ptr(), bhh.data_ptr(), Hall.data_ptr(), _p(Hbm),
               attn.data_ptr(), ctx_ptr, XC.stride(0), sp[0], sp[1], sp[2], sp[3], sp[4], B, T, P, H, Fd, t0, t1, resume,
               _stream())
    lw._resume = (Hall.data_ptr(), t1)


def attgru_seq_fwd(Kp, f, GIw, lw, bu, va, bv, bhh, Hall, Hbm, attn, XC, E, saved, t0, t1):
    """Runs steps [t0,t1).  Kp [B,P,H], f [B,P,F], GIw [T*B,3H], XC [T*B,E+F] (ctx written into columns E:),
    saved = tensor [5,T,B,H] (Upre,R,Z,Nn,GHN) or None."""
    B, P, H = Kp.shape
    Fd = f.shape[2]
    T = Hall.shape[0] - 1
    sp = [saved[i].data_ptr() for i in range(5)] if saved is not None else [None] * 5
    ctx_ptr = XC.data_ptr() + 4 * E
    _cabi.call("caphn_attgru_seq_fwd", Kp.data_ptr(), f.data_ptr(), GIw.data_ptr(), lw.UaT.data_ptr(), bu.data_ptr(),
               va.data_ptr(), bv.data_ptr(), lw.WihcT.data_ptr(), lw.WhhT.data_ptr(), bhh.data_ptr(), Hall.data_ptr(),
               _p(Hbm), attn.data_ptr(), ctx_ptr, XC.stride(0), sp[0], sp[1], sp[2], sp[3], sp[4],
               B, T, P, H, Fd, lw.ldh, lw.ld3, t0, t1, _stream())


def attgru_seq_bwd(dHbm, dattn, Kp, f, attn, saved, Hall, U_a, va, W_ih, W_hh, E):
    B, P, H = Kp.shape
    Fd = f.shape[2]
    T = Hall.shape[0] - 1
    dev = Kp.device
    ldh, ldf = round4(H), round4(Fd)
    Ua_p = copy_pad(U_a, ldh)
    Whh_p = copy_pad(W_hh, ldh)
    Wihc_p = copy_pad(W_ih[:, E:], ldf)
    if Wihc_p.data_ptr() % 16 or Wihc_p.stride(0) != ldf:
        Wihc_p = Wihc_p.contiguous().clone()
    z = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
    e = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    dGI, dGH, dU, dCTX = e(T * B, 3 * H), e(T * B, 3 * H), e(T * B, H), e(T * B, Fd)
    dK, dva, dbv, dh0 = z(B, P, H), z(H), z(1), e(B, H)
    _cabi.call("caphn_attgru_seq_bwd", dHbm.data_ptr(), _p(dattn), Kp.data_ptr(), f.data_ptr(), attn.data_ptr(),
               saved[0].data_ptr(), saved[1].data_ptr(), saved[2].data_ptr(), saved[3].data_ptr(), saved[4].data_ptr(),
               Hall.data_ptr(), Ua_p.data_ptr(), va.data_ptr(), Wihc_p.data_ptr(), Whh_p.data_ptr(), dGI.data_ptr(),
               dGH.data_ptr(), dU.data_ptr(), dCTX.data_ptr(), dK.data_ptr(), dva.data_ptr(), dbv.data_ptr(),
               dh0.data_ptr(), B, T, P, H, Fd, ldh, ldf, _stream())
    return dGI, dGH, dU, dCTX, dK, dva, dbv, dh0


_attstep_bwd_sizes = {}


def _attstep_bwd_bytes(H, Fd, P, B, T):
    key = (H, Fd, P, B, T)
    if key not in _attstep_bwd_sizes:
        import ctypes
        n, w = ctypes.c_long(0), ctypes.c_long(0)
        _cabi.call("caphn_attstep_bwd_size", H, Fd, P, B, T, ctypes.byref(n), ctypes.byref(w))
        _attstep_bwd_sizes[key] = (int(n.value), int(w.value))
    return _attstep_bwd_sizes[key]


def attgru_bwd(dHbm, dattn, Kp, f, attn, saved, Hall, U_a, va, W_ih, W_hh, E, step=None):
    """BPTT of the attention-GRU recurrence: step-split kernels when the shape is covered, else the persistent kernel.
    Returns dGI, dGH [T*B,3H], dU [T*B,H], dCTX [T*B,F], dK [B,P,H], dva [H], dbv [1], dh0 [B,H]."""
    B, P, H = Kp.shape
    Fd = f.shape[2]
    T = Hall.shape[0] - 1
    nbytes, wbytes = _attstep_bwd_bytes(H, Fd, P, B, T) if (ATT_STEP if step is None else step) else (0, 0)
    if nbytes == 0:
        return attgru_seq_bwd(dHbm, dattn, Kp, f, attn, saved, Hall, U_a, va, W_ih, W_hh, E)
    dev = Kp.device
    W_ih, W_hh, U_a = W_ih.contiguous(), W_hh.contiguous(), U_a.contiguous()
    pack = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    work = torch.empty(wbytes, device=dev, dtype=torch.uint8)
    _cabi.call("caphn_attstep_bwd_pack", W_ih.data_ptr(), W_hh.data_ptr(), U_a.data_ptr(), E, Fd, H, pack.data_ptr(),
               _stream())
    e = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    dGI, dGH, dU, dCTX = e(T * B, 3 * H), e(T * B, 3 * H), e(T * B, H), e(T * B, Fd)
    dK, dva, dbv, dh0 = e(B, P, H), e(H), e(1), e(B, H)
    _cabi.call("caphn_attstep_bwd", dHbm.data_ptr(), _p(dattn), Kp.data_ptr(), f.data_ptr(), attn.data_ptr(),
               saved[0].data_ptr(), saved[1].data_ptr(), saved[2].data_ptr(), saved[3].data_ptr(), saved[4].data_ptr(),
               Hall.data_ptr(), va.data_ptr(), pack.data_ptr(), work.data_ptr(), dGI.data_ptr(), dGH.data_ptr(),
               dU.data_ptr(), dCTX.data_ptr(), dK.data_ptr(), dva.data_ptr(), dbv.data_ptr(), dh0.data_ptr(),
               B, T, P, H, Fd, _stream())
    return dGI, dGH, dU, dCTX, dK, dva, dbv, dh0


def attn_df(attn, dCTX, df):
    B, T, P = attn.shape
    Fd = df.shape[-1]
    _cabi.call("caphn_attn_df", attn.data_ptr(), dCTX.data_ptr(), df.data_ptr(), B, T, P, Fd, _stream())
    return df


# ----------------------------------------------------------------------------------------------------------------------
# tensor-core GEMM (tcgen05/TMEM/TMA) on bf16x3-split operands
# ----------------------------------------------------------------------------------------------------------------------
def round64(n):
    return (n + 63) // 64 * 64


class SplitOperand:
    """fp32 matrix in the bf16x3 operand format: hi, lo bf16 (lo None in plain-bf16 mode).
    K-major  (mn=False): source [rows, K]  -> hi/lo [rows, ld], operand rows = source rows.
    MN-major (mn=True):  source [K, rows]  -> hi/lo [K, ld]: the operand of a transposed product, read in place."""
    __slots__ = ("hi", "lo", "rows", "K", "ld", "mn")

    def __init__(self, hi, lo, rows, K, ld, mn=False):
        self.hi, self.lo, self.rows, self.K, self.ld, self.mn = hi, lo, rows, K, ld, mn

    @property
    def Kp(self):   # kept for the K-major call sites
        return self.ld


def split_bf16(src, want_lo=None, mn=False):
    """mn=False: operand rows = src rows (K-major).  mn=True: operand = src^T without a transposed copy (MN-major)."""
    want_lo = TC_SPLIT if want_lo is None else want_lo
    _chk(src)
    assert src.dim() == 2 and src.stride(1) == 1
    R, C = src.shape
    Kp = round64(C)
    hi = torch.empty(R, Kp, device=src.device, dtype=torch.bfloat16)
    lo = torch.empty(R, Kp, device=src.device, dtype=torch.bfloat16) if want_lo else None
    _cabi.call("caphn_split_bf16", src.data_ptr(), src.stride(0), R, C, hi.data_ptr(), _p(lo), Kp, _stream())
    if mn:
        return SplitOperand(hi, lo, C, R, Kp, True)
    return SplitOperand(hi, lo, R, C, Kp, False)


def split_bf16_t(src, want_lo=None, ones_row=False):
    """src [R, C] -> operand for src^T: hi, lo [C, Rp].  ones_row: one more operand row of ones (hi = 1, lo = 0), so that
    a product X^T [src | 1] also delivers the column sums of X (the bias gradient) from the tensor cores."""
    want_lo = TC_SPLIT if want_lo is None else want_lo
    _chk(src)
    assert src.dim() == 2 and src.stride(1) == 1
    R, C = src.shape
    Rp = round64(R)
    Cx = C + (1 if ones_row else 0)
    hi = torch.empty(Cx, Rp, device=src.device, dtype=torch.bfloat16)
    lo = torch.empty(Cx, Rp, device=src.device, dtype=torch.bfloat16) if want_lo else None
    _cabi.call("caphn_split_bf16_t", src.data_ptr(), src.stride(0), R, C, hi.data_ptr(), _p(lo), Rp, _stream())
    if ones_row:
        hi[C].fill_(1.0)
        if lo is not None:
            lo[C].zero_()
    return SplitOperand(hi, lo, Cx, R, Rp, False)


def gemm_tc(A: SplitOperand, Bm: SplitOperand, bias=None, relu=False, out=None, splitk=0, scale=None):
    """out[M,N] = A B^T (+bias) on the tensor cores; operands K-major or MN-major (see SplitOperand), equal K.
    scale = (num, den): device scalars, the product is multiplied by num[0] / max(den[0], 1) in the epilogue (den may be
    None)."""
    assert A.K == Bm.K and (A.lo is None) == (Bm.lo is None)
    M, N = A.rows, Bm.rows
    if out is None:
        out = torch.empty(M, N, device=A.hi.device, dtype=torch.float32)
    assert out.stride(1) == 1
    if scale is not None:
        assert not relu
        num, den = scale
        _cabi.call("caphn_gemm_tc_scaled", A.hi.data_ptr(), _p(A.lo), A.ld, int(A.mn), Bm.hi.data_ptr(), _p(Bm.lo),
                   Bm.ld, int(Bm.mn), A.K, out.data_ptr(), out.stride(0), _p(bias), M, N, splitk, num.data_ptr(), _p(den),
                   _stream())
        return out
    _cabi.call("caphn_gemm_tc_ex", A.hi.data_ptr(), _p(A.lo), A.ld, int(A.mn), Bm.hi.data_ptr(), _p(Bm.lo), Bm.ld,
               int(Bm.mn), A.K, out.data_ptr(), out.stride(0), _p(bias), M, N, int(relu), 1 if relu else splitk,
               _stream())
    return out


def gemm_tc_amax(A: SplitOperand, Bm: SplitOperand, bias, out, pval, pidx):
    """out[M,N] = A B^T + bias on the tensor cores, and per-row arg-max partials of the result written by the epilogue into
    pval (fp32) / pidx (int32) [M, ld]; returns the number of partial slots per row (finish with argmax_finish_gather)."""
    import ctypes
    assert A.K == Bm.K and (A.lo is None) == (Bm.lo is None) and out.stride(1) == 1
    assert pval.dtype == torch.float32 and pidx.dtype == torch.int32 and pval.stride(0) == pidx.stride(0)
    M, N = A.rows, Bm.rows
    n = ctypes.c_int(0)
    _cabi.call("caphn_gemm_tc_amax", A.hi.data_ptr(), _p(A.lo), A.ld, int(A.mn), Bm.hi.data_ptr(), _p(Bm.lo), Bm.ld,
               int(Bm.mn), A.K, out.data_ptr(), out.stride(0), _p(bias), M, N, pval.data_ptr(), pidx.data_ptr(),
               pval.stride(0), ctypes.byref(n), _stream())
    return int(n.value)


def argmax_finish_gather(pval, pidx, nparts, table=None, tok=None, out=None):
    """tok[i] = arg-max of row i from its ``nparts`` partials (lowest column on ties); out[i] = table[tok[i]] if given."""
    n = pval.shape[0]
    E = table.shape[1] if table is not None else 0
    if table is not None:
        assert table.is_contiguous() and out is not None and out.stride(1) == 1
    _cabi.call("caphn_argmax_finish_gather", pval.data_ptr(), pidx.data_ptr(), pval.stride(0), nparts, n, _p(table), E,
               _p(tok), _p(out), out.stride(0) if out is not None else 0, _stream())


def gru_decode_step_ok(H, V):
    """The fused decode-step kernel keeps 96 rows of W_hh and up to 32 states in shared memory as float2: H even, <= ~390;
    and each lane holds 8 arg-max partial slots: at most 256 = 2 ceil(V / BN) per row, bounded here with the narrowest N
    tile the GEMM picks for V > 256 (BN = 128), i.e. V <= 16384."""
    return H % 2 == 0 and (96 * (H + 2) + 32 * H) * 4 <= 200 * 1024 and 2 * ((V + 127) // 128) <= 256


def gru_decode_step(GI, pval, pidx, nparts, table, W_hh, b_hh, hprev, hnew, hi=None, lo=None, tok=None):
    """One greedy-decode step of the pooled captioner in one launch (csrc/gru_decode.cu): arg-max finish + projection-table
    gather (GI None) or the given input projection, GRU cell, new state as fp32 and as bf16 hi / lo operand rows."""
    B, H = hprev.shape
    assert W_hh.is_contiguous() and hprev.is_contiguous() and hnew.is_contiguous() and hnew.data_ptr() != hprev.data_ptr()
    if GI is not None:
        assert GI.is_contiguous() and GI.shape == (B, 3 * H)
    else:
        assert table.is_contiguous() and table.shape[1] == 3 * H and pval.stride(0) == pidx.stride(0)
    _cabi.call("caphn_gru_decode_step", _p(GI), _p(pval), _p(pidx), pval.stride(0) if pval is not None else 0, nparts,
               _p(table), W_hh.data_ptr(), b_hh.data_ptr(), hprev.data_ptr(), hnew.data_ptr(), _p(hi), _p(lo),
               hi.stride(0) if hi is not None else 0, _p(tok), B, H, _stream())
    return hnew


def gru_decode_step_tok_ok(H):
    """The token-fed decode step reads no arg-max partials: only the shared-memory bound of gru_decode_step_ok (H even,
    <= 398) applies, for any V."""
    return H % 2 == 0 and (96 * (H + 2) + 32 * H) * 4 <= 200 * 1024


def gru_decode_step_tok(tok, table, W_hh, b_hh, hprev, hnew, hi=None, lo=None):
    """gru_decode_step with the input token given (csrc/gru_decode.cu, caphn_gru_decode_step_tok): row b's input projection
    is table[tok[b]] (int32 tokens; one outside [0, V) reads row 0), then the GRU cell and the operand rows as there."""
    _chk(tok, torch.int32)
    B, H = hprev.shape
    assert W_hh.is_contiguous() and hprev.is_contiguous() and hnew.is_contiguous() and hnew.data_ptr() != hprev.data_ptr()
    assert table.is_contiguous() and table.shape[1] == 3 * H and tok.is_contiguous() and tok.numel() == B
    _cabi.call("caphn_gru_decode_step_tok", tok.data_ptr(), table.shape[0], table.data_ptr(), W_hh.data_ptr(),
               b_hh.data_ptr(), hprev.data_ptr(), hnew.data_ptr(), _p(hi), _p(lo), hi.stride(0) if hi is not None else 0, B,
               H, _stream())
    return hnew


def beam_step(logits, h_out, h_next, scores, live, prev_tok, words, seq_in, seq_out, comp_score, comp_seq, comp_len, ncomp,
              failed, k, step, end_tok, last):
    """One bookkeeping step of the batched beam search (csrc/beam.cu, caphn_beam_step) for B = live.numel() images x k
    beams: log-softmax + running scores, top-k of the live rows' candidates, completed beams to the complete list,
    survivors compacted (history, score, hidden state h_out -> h_next), next input words.  logits [B*k, V], h_out /
    h_next [B*k, H], token histories seq_in / seq_out / comp_seq [B*k, L]; step is 1-based, ``last`` marks the final one."""
    for t in (logits, h_out, h_next, scores, comp_score):
        _chk(t)
    for t in (live, prev_tok, seq_in, seq_out, comp_seq, comp_len, ncomp, failed):
        _chk(t, torch.int32)
    _chk(words, torch.int64)
    assert all(t.is_contiguous() for t in (logits, h_out, h_next, scores, live, prev_tok, words, seq_in, seq_out,
                                           comp_score, comp_seq, comp_len, ncomp, failed))
    _cabi.call("caphn_beam_step", logits.data_ptr(), h_out.data_ptr(), h_next.data_ptr(), scores.data_ptr(),
               live.data_ptr(), prev_tok.data_ptr(), words.data_ptr(), seq_in.data_ptr(), seq_out.data_ptr(),
               comp_score.data_ptr(), comp_seq.data_ptr(), comp_len.data_ptr(), ncomp.data_ptr(), failed.data_ptr(),
               live.numel(), k, logits.shape[1], h_out.shape[1], seq_in.shape[1], step, end_tok, int(last), _stream())


def attstep_h_operand(lw, B, H, Fd, t_done):
    """The hidden state h_{t_done} as the bf16 hi/lo operand rows the step-split gates kernel has just written into its
    workspace for the next step's U kernel (attgru_step.cu: hsp buffers) -- the A operand of the vocabulary projection,
    with no separate split pass.  Only for the step-split path (``lw.pack`` set), after ``attgru_fwd(..., t_done, t_done+1)``."""
    KP = ((max(H, Fd) + 15) // 16) * 16 + 8
    a256 = lambda v: (v + 255) & ~255
    plane2 = a256(B * KP * 2)
    base = a256(B * H * 4) + 2 * plane2 + (2 * plane2 if ((t_done + 1) & 1) else 0)      # hbuf(t_done + 1)
    w = lw.work
    hi = w[base: base + B * KP * 2].view(torch.bfloat16).view(B, KP)
    lo = w[base + B * KP * 2: base + 2 * B * KP * 2].view(torch.bfloat16).view(B, KP) if TC_SPLIT else None
    return SplitOperand(hi, lo, B, H, KP, False)


def use_projection_table(B, steps, V):
    """Greedy decode feeds back word embeddings, so  x_t W^T + b  is a row of the table  Emb W^T + b  [V, N].  Building
    the table costs one V-row GEMM per decode call (the generated W changes with every style); it replaces a gather, an
    operand split and a B-row GEMM in each of the remaining steps, and pays off once those rows outnumber V / 2."""
    return (steps - 1) * B >= V // 2


class LinearPlan:
    """y = x W^T + b for a weight that is reused many times (greedy decode: one projection per time step).  The bf16x3
    split of W is made once; every call only splits the (small) activation."""

    def __init__(self, W, bias=None):
        _chk(W)
        assert W.stride(1) == 1
        self.W, self.bias = W, bias
        self.N, self.K = W.shape
        self._split = None

    def operand(self):
        """The cached bf16 hi/lo split of W (the B operand of the tensor-core path)."""
        if self._split is None or (self._split.lo is None) == TC_SPLIT:
            self._split = split_bf16(self.W)
        return self._split

    def __call__(self, X, relu=False, out=None):
        M = X.shape[0]
        if _tc_ok(M, self.N, self.K):
            return gemm_tc(split_bf16(X), self.operand(), bias=self.bias, relu=relu, out=out)
        return _gemm(X, X.stride(0), 1, self.W, self.W.stride(0), 1, M, self.N, self.K, self.bias, relu, out)


# ----------------------------------------------------------------------------------------------------------------------
# many-style ("grouped") path: operand builders, grouped tensor-core GEMM, per-group recurrence tiles
# ----------------------------------------------------------------------------------------------------------------------
def split_bf16_gather(src, rowmap, R, want_lo=None):
    """K-major operand [R, round64(C)] whose row i is src[rowmap[i]] (zero when rowmap[i] < 0); rowmap int32 [R]."""
    want_lo = TC_SPLIT if want_lo is None else want_lo
    _chk(src), _chk(rowmap, torch.int32)
    assert src.dim() == 2 and src.stride(1) == 1 and rowmap.numel() == R
    C = src.shape[1]
    Kp = round64(C)
    hi = torch.empty(R, Kp, device=src.device, dtype=torch.bfloat16)
    lo = torch.empty(R, Kp, device=src.device, dtype=torch.bfloat16) if want_lo else None
    _cabi.call("caphn_split_bf16_gather", src.data_ptr(), src.stride(0), rowmap.data_ptr(), R, C, hi.data_ptr(), _p(lo),
               Kp, _stream())
    return SplitOperand(hi, lo, R, C, Kp, False)


def split_bf16_batched(src, sstride, lds, nb, R, C, want_lo=None):
    """nb matrices [R, C] taken from ``src`` (a tensor whose data pointer is matrix 0; matrix b starts sstride floats later,
    rows lds floats apart) -> one K-major operand [nb*R, round64(C)]."""
    want_lo = TC_SPLIT if want_lo is None else want_lo
    _chk(src)
    Kp = round64(C)
    hi = torch.empty(nb * R, Kp, device=src.device, dtype=torch.bfloat16)
    lo = torch.empty(nb * R, Kp, device=src.device, dtype=torch.bfloat16) if want_lo else None
    _cabi.call("caphn_split_bf16_batched", src.data_ptr(), sstride, lds, nb, R, C, hi.data_ptr(), _p(lo), Kp, _stream())
    return SplitOperand(hi, lo, nb * R, C, Kp, False)


def gemm_tc_grouped(A: SplitOperand, a_mn, Bm: SplitOperand, b_mn, C, ldc, units, BN, bias=None, rowmap=None):
    """One launch for all the tiles listed in ``units`` (int32 [n, 12], see include/caphn_b200.h).  The operands are the
    raw 2-D bf16 arrays of ``A`` / ``Bm`` ([rows, ld]); which rows / k range a tile uses is in its unit record."""
    assert (A.lo is None) == (Bm.lo is None) and units.dtype == torch.int32 and units.is_contiguous()
    a_outer, b_outer = A.hi.shape[0], Bm.hi.shape[0]
    _cabi.call("caphn_gemm_tc_grouped", A.hi.data_ptr(), _p(A.lo), A.ld, a_outer, A.ld, int(a_mn), Bm.hi.data_ptr(),
               _p(Bm.lo), Bm.ld, b_outer, Bm.ld, int(b_mn), C.data_ptr(), ldc, _p(bias), _p(rowmap), units.data_ptr(),
               units.shape[0], BN, _stream())
    return C


def group_colsum(X, goff, G, B, T, out):
    """out[g, :] += sum over the rows of group g (time-major X [T*B, N], batch sorted by group, goff int32 [G+1])."""
    _chk(X), _chk(goff, torch.int32)
    assert X.stride(1) == 1 and out.stride(1) == 1
    _cabi.call("caphn_group_colsum", X.data_ptr(), X.stride(0), goff.data_ptr(), G, B, T, X.shape[1], out.data_ptr(),
               out.stride(0), _stream())
    return out


def leaky_relu_(y, slope=LEAKY_SLOPE):
    assert y.is_contiguous()
    _cabi.call("caphn_leaky_relu", y.data_ptr(), y.numel(), slope, _stream())
    return y


def leaky_relu_bwd_(y, dy, slope=LEAKY_SLOPE):
    assert y.is_contiguous() and dy.is_contiguous() and y.numel() == dy.numel()
    _cabi.call("caphn_leaky_relu_bwd", y.data_ptr(), dy.data_ptr(), y.numel(), slope, _stream())
    return dy


class AttGruGroupWeights:
    """Per-group mma-fragment packs of the generated W_ih[:, E:], W_hh (+ the shared U_a) for the step-split kernels.
    ``Theta`` [G, theta] holds (W_ih [3H, E+F], W_hh [3H, H], b_ih, b_hh) per row."""

    def __init__(self, Theta, U_a, E, Fd, H, P):
        G, theta = Theta.shape
        assert Theta.is_contiguous()
        n = _attstep_bytes(H, Fd, P, 0)[0]
        if n == 0:
            raise _cabi.CaphnError(f"the grouped recurrence needs the step-split kernels (H={H}, F={Fd}, P={P} not covered)")
        self.G, self.pack_bytes = G, n
        self.pack = torch.empty(G * n, device=Theta.device, dtype=torch.uint8)
        whh_off = 3 * H * (E + Fd)
        _cabi.call("caphn_attstep_pack_grouped", Theta.data_ptr(), Theta.data_ptr() + 4 * whh_off, U_a.data_ptr(), E, Fd,
                   H, G, theta, self.pack.data_ptr(), _stream())
        self.work = None


def attgru_fwd_grouped(Kp, f, GIw, gw: AttGruGroupWeights, bu, va, bv, bhh_g, Hall, Hbm, attn, XC, E, saved, tiles,
                       tile_rows=64):
    """All T steps; rows sorted by group; tiles int32 [n, 4] = (first row, rows <= tile_rows <= 64, group, 0); bhh_g [G, 3H]."""
    B, P, H = Kp.shape
    Fd = f.shape[2]
    T = Hall.shape[0] - 1
    sp = [saved[i].data_ptr() for i in range(5)] if saved is not None else [None] * 5
    ctx_ptr = XC.data_ptr() + 4 * E
    wbytes = _attstep_bytes(H, Fd, P, B)[1]
    if gw.work is None or gw.work.numel() < wbytes:
        gw.work = torch.empty(wbytes, device=Kp.device, dtype=torch.uint8)
    assert tiles.dtype == torch.int32 and tiles.is_contiguous() and bhh_g.is_contiguous()
    _cabi.call("caphn_attstep_fwd_grouped", Kp.data_ptr(), f.data_ptr(), GIw.data_ptr(), bu.data_ptr(), va.data_ptr(),
               bv.data_ptr(), gw.pack.data_ptr(), gw.work.data_ptr(), bhh_g.data_ptr(), Hall.data_ptr(), _p(Hbm),
               attn.data_ptr(), ctx_ptr, XC.stride(0), sp[0], sp[1], sp[2], sp[3], sp[4], B, T, P, H, Fd, 0, T, 0,
               tiles.data_ptr(), tiles.shape[0], int(tile_rows), _stream())


def attgru_bwd_grouped(dHbm, dattn, Kp, f, attn, saved, Hall, Theta, U_a, va, E, tiles, tile_rows=32):
    """BPTT of attgru_fwd_grouped.  tiles int32 [n, 4] with <= tile_rows <= 32 rows each.  Returns dGI, dGH, dU, dCTX, dK, dva,
    dbv, dh0."""
    B, P, H = Kp.shape
    Fd = f.shape[2]
    T = Hall.shape[0] - 1
    G, theta = Theta.shape
    nbytes, wbytes = _attstep_bwd_bytes(H, Fd, P, B, T)
    if nbytes == 0:
        raise _cabi.CaphnError("the grouped BPTT needs the step-split kernels (shape not covered)")
    dev = Kp.device
    pack = torch.empty(G * nbytes, device=dev, dtype=torch.uint8)
    work = torch.empty(wbytes, device=dev, dtype=torch.uint8)
    whh_off = 3 * H * (E + Fd)
    _cabi.call("caphn_attstep_bwd_pack_grouped", Theta.data_ptr(), Theta.data_ptr() + 4 * whh_off, U_a.data_ptr(), E, Fd,
               H, G, theta, pack.data_ptr(), _stream())
    e = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    dGI, dGH, dU, dCTX = e(T * B, 3 * H), e(T * B, 3 * H), e(T * B, H), e(T * B, Fd)
    dK, dva, dbv, dh0 = e(B, P, H), e(H), e(1), e(B, H)
    assert tiles.dtype == torch.int32 and tiles.is_contiguous()
    _cabi.call("caphn_attstep_bwd_grouped", dHbm.data_ptr(), _p(dattn), Kp.data_ptr(), f.data_ptr(), attn.data_ptr(),
               saved[0].data_ptr(), saved[1].data_ptr(), saved[2].data_ptr(), saved[3].data_ptr(), saved[4].data_ptr(),
               Hall.data_ptr(), va.data_ptr(), pack.data_ptr(), work.data_ptr(), dGI.data_ptr(), dGH.data_ptr(),
               dU.data_ptr(), dCTX.data_ptr(), dK.data_ptr(), dva.data_ptr(), dbv.data_ptr(), dh0.data_ptr(),
               B, T, P, H, Fd, tiles.data_ptr(), tiles.shape[0], int(tile_rows), _stream())
    return dGI, dGH, dU, dCTX, dK, dva, dbv, dh0
