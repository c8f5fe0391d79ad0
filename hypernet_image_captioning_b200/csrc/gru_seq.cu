// Persistent GRU recurrence (pooled-feature decoder, "Variant A"): all T time steps in one launch.
//
// Replaces the per-step nn.GRUCell calls of DecoderGRU.forward / infer (reference later.py:411,418,471-477; cell
// formula = torch GRUCell, gates r,z,n) and their autograd backward (BPTT).  The input projection
// gi = x W_ih^T + b_ih does not depend on the recurrence in teacher-forced mode and arrives precomputed for all steps
// (time-major [T,B,3H]); this kernel does gh = h W_hh^T + b_hh, the gate non-linearities and the state update.
//
// Round-1 decomposition: one CTA owns BT batch rows for the whole sequence and keeps h on-chip (shared memory); the
// generated W_hh (transposed + padded to 16-byte rows by caphn_transpose_pad) is re-read from L2 every step.
// (A cluster version that keeps W_hh slices resident in shared memory is the next step; see DESIGN.md.)
//
// Sequence tensors are time-major: row index = t*B + b.  Hall is [T+1, B, H] with Hall[0] = h0, so that
// Hall[1:] = h_t and Hall[:-1] = h_{t-1} are both plain [T*B, H] matrices for the dW_hh GEMM.
#include "seq_common.cuh"

namespace caphn {

constexpr int GRU_MAX_EXTRA = 3;  // DecoderGRU(num_layers <= 4)

struct GruFwdArgs {
    const float* GI;     // [T,B,3H] layer-0 input projection (+ b_ih)
    const float* WhhT;   // [H, ld3] layer 0
    const float* bhh;    // [3H]
    float* Hall;         // [T+1,B,H]: Hall[0] = h0, Hall[t+1] = output of the LAST layer at step t
    float* Hbm;          // [B,T,H] or null
    float* saved;        // [NL][4][T,B,H] (R,Z,N,GHN per layer) or null
    float* Hmid;         // [NL-1][T,B,H] outputs of layers 0..NL-2 (needed for NL > 1 when saving)
    const float* xWihT[GRU_MAX_EXTRA];  // extra layers: [H, ld3] each (input = state = previous layer's output)
    const float* xWhhT[GRU_MAX_EXTRA];
    const float* xbih[GRU_MAX_EXTRA];
    const float* xbhh[GRU_MAX_EXTRA];
    int NL, B, T, H, ld3;
};

__global__ void __launch_bounds__(AT_THREADS) gru_seq_fwd_kernel(const GruFwdArgs a) {
    constexpr int BT = AT_BT;
    extern __shared__ __align__(16) float smem[];
    const int H = a.H, B = a.B, T = a.T, ld3 = a.ld3, H3 = 3 * a.H;
    const int CQT3 = at_cqt(ld3), KG3 = AT_THREADS / CQT3;
    float* hs = smem;                           // [H][BT]
    float* part_gh = smem + H * BT;             // [KG3][BT][ld3]
    float* part_gi = part_gh + KG3 * BT * ld3;  // [KG3][BT][ld3]   (extra layers only)
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * BT;
    const long TBH = (long)T * B * H;

    for (int i = tid; i < H * BT; i += AT_THREADS) {
        const int k = i / BT, b = i - k * BT;
        hs[i] = (b0 + b < B) ? a.Hall[(long)(b0 + b) * H + k] : 0.f;
    }
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        for (int l = 0; l < a.NL; ++l) {
            const bool last = (l == a.NL - 1);
            if (l == 0) {
                block_matvec<BT, false>(a.WhhT, ld3, H, hs, part_gh, CQT3, tid);
            } else {
                block_matvec<BT, false>(a.xWihT[l - 1], ld3, H, hs, part_gi, CQT3, tid);
                block_matvec<BT, false>(a.xWhhT[l - 1], ld3, H, hs, part_gh, CQT3, tid);
            }
            __syncthreads();
            const float* bhh = (l == 0) ? a.bhh : a.xbhh[l - 1];
            for (int i = tid; i < BT * H; i += AT_THREADS) {
                const int b = i / H, j = i - b * H;
                const int gb = b0 + b;
                if (gb < B) {
                    const float ghr = bhh[j] + part_sum(part_gh, KG3, BT, ld3, b, j);
                    const float ghz = bhh[H + j] + part_sum(part_gh, KG3, BT, ld3, b, H + j);
                    const float ghn = bhh[2 * H + j] + part_sum(part_gh, KG3, BT, ld3, b, 2 * H + j);
                    float gir, giz, gin;
                    if (l == 0) {
                        const float* gi = a.GI + ((long)t * B + gb) * H3;
                        gir = gi[j]; giz = gi[H + j]; gin = gi[2 * H + j];
                    } else {
                        const float* bih = a.xbih[l - 1];
                        gir = bih[j] + part_sum(part_gi, KG3, BT, ld3, b, j);
                        giz = bih[H + j] + part_sum(part_gi, KG3, BT, ld3, b, H + j);
                        gin = bih[2 * H + j] + part_sum(part_gi, KG3, BT, ld3, b, 2 * H + j);
                    }
                    const float r = sigmoidf_acc(gir + ghr);
                    const float z = sigmoidf_acc(giz + ghz);
                    const float n = tanhf(gin + r * ghn);
                    const float hp = hs[j * BT + b];
                    const float hn = (1.f - z) * n + z * hp;
                    hs[j * BT + b] = hn;
                    const long o = ((long)t * B + gb) * H + j;
                    if (last) {
                        a.Hall[o + (long)B * H] = hn;
                        if (a.Hbm) a.Hbm[((long)gb * T + t) * H + j] = hn;
                    } else if (a.Hmid) {
                        a.Hmid[(long)l * TBH + o] = hn;
                    }
                    if (a.saved) {
                        float* sv = a.saved + (long)l * 4 * TBH + o;
                        sv[0] = r; sv[TBH] = z; sv[2 * TBH] = n; sv[3 * TBH] = ghn;
                    }
                }
            }
            __syncthreads();
        }
    }
}

struct GruBwdArgs {
    const float* dHbm;   // [B,T,H] gradient w.r.t. the last layer's output at every step
    const float* saved;  // [NL][4][T,B,H]
    const float* Hall;   // [T+1,B,H]
    const float* Hmid;   // [NL-1][T,B,H]
    const float* Whh;    // [3H, ldh] layer 0
    const float* xWih[GRU_MAX_EXTRA];  // [3H, ldh]
    const float* xWhh[GRU_MAX_EXTRA];
    float* dGI;          // [T,B,3H] layer 0
    float* dGH;          // [T,B,3H] layer 0
    float* xdGI;         // [NL-1][T,B,3H]
    float* xdGH;         // [NL-1][T,B,3H]
    float* dh0;          // [B,H]
    int NL, B, T, H, ldh;
};

// One GRU cell backward for the (row, unit) items of this CTA.  dht = total gradient w.r.t. the cell output.
__device__ __forceinline__ void gru_gate_bwd(float dht, float r, float z, float n, float ghn, float hp, float& dar,
                                             float& daz, float& dan, float& danr, float& keep) {
    const float dn = dht * (1.f - z);
    const float dz = dht * (hp - n);
    dan = dn * (1.f - n * n);
    dar = dan * ghn * r * (1.f - r);
    daz = dz * z * (1.f - z);
    danr = dan * r;
    keep = dht * z;
}

__global__ void __launch_bounds__(AT_THREADS) gru_seq_bwd_kernel(const GruBwdArgs a) {
    constexpr int BT = AT_BT;
    extern __shared__ __align__(16) float smem[];
    const int H = a.H, B = a.B, T = a.T, ldh = a.ldh, H3 = 3 * a.H;
    const int CQTh = at_cqt(ldh), KGh = AT_THREADS / CQTh;
    float* dgi = smem;                               // [3H][BT]
    float* dgh = dgi + H3 * BT;                      // [3H][BT]
    float* dhd = dgh + H3 * BT;                      // [BT][H] carried direct term (layer 0: dh_t * z)
    float* dhin = dhd + ((BT * H + 3) & ~3);         // [BT][H] gradient handed from layer l to layer l-1
    float* part_dh = dhin + ((BT * H + 3) & ~3);     // [KGh][BT][ldh]  dgh . W_hh
    float* part_di = part_dh + KGh * BT * ldh;       // [KGh][BT][ldh]  dgi . W_ih (extra layers)
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * BT;
    const long TBH = (long)T * B * H, TB3 = (long)T * B * H3;

    for (int i = tid; i < BT * H; i += AT_THREADS) dhd[i] = 0.f;
    for (int i = tid; i < KGh * BT * ldh; i += AT_THREADS) part_dh[i] = 0.f;
    __syncthreads();

    for (int t = T - 1; t >= 0; --t) {
        for (int l = a.NL - 1; l >= 0; --l) {
            const bool top = (l == a.NL - 1);
            for (int i = tid; i < BT * H; i += AT_THREADS) {
                const int b = i / H, j = i - b * H;
                const int gb = b0 + b;
                float dar = 0.f, daz = 0.f, dan = 0.f, danr = 0.f, keep = 0.f;
                if (gb < B) {
                    float dht;
                    if (top) dht = dhd[i] + a.dHbm[((long)gb * T + t) * H + j] + part_sum(part_dh, KGh, BT, ldh, b, j);
                    else dht = dhin[i];
                    const long o = ((long)t * B + gb) * H + j;
                    const float* sv = a.saved + (long)l * 4 * TBH + o;
                    const float hp = (l == 0) ? a.Hall[o] : a.Hmid[(long)(l - 1) * TBH + o];
                    gru_gate_bwd(dht, sv[0], sv[TBH], sv[2 * TBH], sv[3 * TBH], hp, dar, daz, dan, danr, keep);
                    float* gi = ((l == 0) ? a.dGI : a.xdGI + (long)(l - 1) * TB3) + ((long)t * B + gb) * H3;
                    float* gh = ((l == 0) ? a.dGH : a.xdGH + (long)(l - 1) * TB3) + ((long)t * B + gb) * H3;
                    gi[j] = dar; gi[H + j] = daz; gi[2 * H + j] = dan;
                    gh[j] = dar; gh[H + j] = daz; gh[2 * H + j] = danr;
                }
                if (l == 0) dhd[i] = keep; else dhin[i] = keep;
                dgh[j * BT + b] = dar; dgh[(H + j) * BT + b] = daz; dgh[(2 * H + j) * BT + b] = danr;
                if (l > 0) { dgi[j * BT + b] = dar; dgi[(H + j) * BT + b] = daz; dgi[(2 * H + j) * BT + b] = dan; }
            }
            __syncthreads();
            if (l == 0) {
                block_matvec<BT, false>(a.Whh, ldh, H3, dgh, part_dh, CQTh, tid);
                __syncthreads();
            } else {
                // input and state of an extra layer are the same vector: both paths flow into the layer below
                block_matvec<BT, false>(a.xWhh[l - 1], ldh, H3, dgh, part_di, CQTh, tid);
                block_matvec<BT, true>(a.xWih[l - 1], ldh, H3, dgi, part_di, CQTh, tid);
                __syncthreads();
                for (int i = tid; i < BT * H; i += AT_THREADS) {
                    const int b = i / H, j = i - b * H;
                    dhin[i] += part_sum(part_di, KGh, BT, ldh, b, j);
                }
                __syncthreads();
            }
        }
    }
    for (int i = tid; i < BT * H; i += AT_THREADS) {
        const int b = i / H, j = i - b * H;
        if (b0 + b < B) a.dh0[(long)(b0 + b) * H + j] = dhd[i] + part_sum(part_dh, KGh, BT, ldh, b, j);
    }
}

// dst[c*ldd + r] = src[r*lds + c]  (r < R, c < C); pad columns [R, ldd) of dst are zeroed.  blockIdx.z = matrix z of a
// batch: src + z * sstride -> dst + z * dstride.
__global__ void transpose_pad_kernel(const float* __restrict__ src, long lds, float* __restrict__ dst, long ldd, int R,
                                     int C, long sstride, long dstride) {
    __shared__ float tile[32][33];
    src += blockIdx.z * sstride;
    dst += blockIdx.z * dstride;
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (r < R && c < C) ? src[(long)r * lds + c] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i, r = r0 + threadIdx.x;
        if (c < C && r < ldd) dst[(long)c * ldd + r] = tile[threadIdx.x][i];
    }
}

// dst[r*ldd + c] = c < C ? src[r*lds + c] : 0;  blockIdx.y = matrix y of a batch (src + y * sstride -> dst + y * dstride)
__global__ void copy_pad_kernel(const float* __restrict__ src, long lds, float* __restrict__ dst, long ldd, long R,
                                int C, long sstride, long dstride) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * ldd) return;
    src += blockIdx.y * sstride;
    dst += blockIdx.y * dstride;
    const long r = i / ldd;
    const int c = (int)(i - r * ldd);
    dst[i] = c < C ? src[r * lds + c] : 0.f;
}

}  // namespace caphn

using namespace caphn;

extern "C" {

int caphn_transpose_pad(const float* src, long lds, float* dst, long ldd, int R, int C, void* stream) {
    if (R <= 0 || C <= 0 || ldd < R) return CAPHN_EINVAL;
    dim3 grid(ceil_div(C, 32), ceil_div(ldd, 32));
    transpose_pad_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, R, C, 0, 0);
    CAPHN_RETURN_LAST();
}

int caphn_copy_pad(const float* src, long lds, float* dst, long ldd, long R, int C, void* stream) {
    if (R <= 0 || C <= 0 || ldd < C) return CAPHN_EINVAL;
    copy_pad_kernel<<<ceil_div(R * ldd, 256), 256, 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, R, C, 0, 0);
    CAPHN_RETURN_LAST();
}

// nb matrices in one launch: matrix z at src + z * sstride -> dst + z * dstride (floats); dst pitch ldd as above.
int caphn_transpose_pad_batched(const float* src, long sstride, long lds, float* dst, long dstride, long ldd, int nb,
                                int R, int C, void* stream) {
    if (nb <= 0 || nb > 65535 || R <= 0 || C <= 0 || ldd < R || dstride < (long)C * ldd) return CAPHN_EINVAL;
    dim3 grid(ceil_div(C, 32), ceil_div(ldd, 32), nb);
    transpose_pad_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, R, C, sstride, dstride);
    CAPHN_RETURN_LAST();
}

int caphn_copy_pad_batched(const float* src, long sstride, long lds, float* dst, long dstride, long ldd, int nb, long R,
                           int C, void* stream) {
    if (nb <= 0 || nb > 65535 || R <= 0 || C <= 0 || ldd < C || dstride < R * ldd) return CAPHN_EINVAL;
    copy_pad_kernel<<<dim3(ceil_div(R * ldd, 256), nb), 256, 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, R, C, sstride,
                                                                                       dstride);
    CAPHN_RETURN_LAST();
}

// GRU recurrence over T steps (all layers).  GI [T,B,3H] (layer-0 x-projection incl. b_ih); WhhT [H, ld3] (ld3 % 4 == 0,
// 16B aligned); Hall [T+1,B,H] with Hall[0] = h0 filled by the caller; optional Hbm [B,T,H].  Extra layers (DecoderGRU
// num_layers > 1, later.py:413-414: h = layer(h, h)): `extra` is a HOST array of 4*(NL-1) device pointers
// {WihT_l, WhhT_l, bih_l, bhh_l}.  saved [NL][4][T,B,H] and Hmid [NL-1][T,B,H] are needed for the backward (or NULL).
int caphn_gru_seq_fwd(const float* GI, const float* WhhT, int ld3, const float* bhh, float* Hall, float* Hbm,
                      float* saved, float* Hmid, const void* const* extra, int NL, int B, int T, int H, void* stream) {
    if (B <= 0 || T <= 0 || H <= 0 || (ld3 & 3) || ld3 < 3 * H || ((uintptr_t)WhhT & 15)) return CAPHN_EINVAL;
    if (NL < 1 || NL > 1 + GRU_MAX_EXTRA || (NL > 1 && !extra) || (NL > 1 && saved && !Hmid)) return CAPHN_EINVAL;
    GruFwdArgs a{};
    a.GI = GI; a.WhhT = WhhT; a.bhh = bhh; a.Hall = Hall; a.Hbm = Hbm; a.saved = saved; a.Hmid = Hmid;
    a.NL = NL; a.B = B; a.T = T; a.H = H; a.ld3 = ld3;
    for (int l = 0; l < NL - 1; ++l) {
        a.xWihT[l] = (const float*)extra[4 * l]; a.xWhhT[l] = (const float*)extra[4 * l + 1];
        a.xbih[l] = (const float*)extra[4 * l + 2]; a.xbhh[l] = (const float*)extra[4 * l + 3];
        if (((uintptr_t)a.xWihT[l] & 15) || ((uintptr_t)a.xWhhT[l] & 15)) return CAPHN_EINVAL;
    }
    const int KG3 = AT_THREADS / at_cqt(ld3);
    const size_t smem = ((size_t)H * AT_BT + 2 * (size_t)KG3 * AT_BT * ld3) * sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(gru_seq_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gru_seq_fwd_kernel<<<ceil_div(B, AT_BT), AT_THREADS, smem, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

// BPTT of caphn_gru_seq_fwd.  Whh [3H, ldh] (ldh % 4 == 0); `extra` = HOST array of 2*(NL-1) device pointers
// {Wih_l, Whh_l} ([3H, ldh] each).  Outputs: dGI, dGH [T,B,3H] (layer 0), xdGI, xdGH [NL-1][T,B,3H], dh0 [B,H].
int caphn_gru_seq_bwd(const float* dHbm, const float* saved, const float* Hall, const float* Hmid, const float* Whh,
                      int ldh, const void* const* extra, float* dGI, float* dGH, float* xdGI, float* xdGH, float* dh0,
                      int NL, int B, int T, int H, void* stream) {
    if (B <= 0 || T <= 0 || H <= 0 || (ldh & 3) || ldh < H || ((uintptr_t)Whh & 15)) return CAPHN_EINVAL;
    if (NL < 1 || NL > 1 + GRU_MAX_EXTRA || (NL > 1 && !(extra && Hmid && xdGI && xdGH))) return CAPHN_EINVAL;
    GruBwdArgs a{};
    a.dHbm = dHbm; a.saved = saved; a.Hall = Hall; a.Hmid = Hmid; a.Whh = Whh; a.dGI = dGI; a.dGH = dGH;
    a.xdGI = xdGI; a.xdGH = xdGH; a.dh0 = dh0; a.NL = NL; a.B = B; a.T = T; a.H = H; a.ldh = ldh;
    for (int l = 0; l < NL - 1; ++l) {
        a.xWih[l] = (const float*)extra[2 * l]; a.xWhh[l] = (const float*)extra[2 * l + 1];
        if (((uintptr_t)a.xWih[l] & 15) || ((uintptr_t)a.xWhh[l] & 15)) return CAPHN_EINVAL;
    }
    const int KGh = AT_THREADS / at_cqt(ldh);
    const size_t smem = (2 * (size_t)3 * H * AT_BT + 2 * (size_t)((AT_BT * H + 3) & ~3) +
                         2 * (size_t)KGh * AT_BT * ldh) * sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(gru_seq_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gru_seq_bwd_kernel<<<ceil_div(B, AT_BT), AT_THREADS, smem, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

}  // extern "C"
