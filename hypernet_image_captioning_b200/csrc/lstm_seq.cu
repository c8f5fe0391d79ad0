// Persistent LSTM recurrence: the hypernet-generated DecoderRNN of the pooled variant (hypernet.py:53 with type != 'gru',
// later.py:227-360), all T time steps in one launch, forward and BPTT.
//
// Replaces the per-step nn.LSTMCell calls of DecoderRNN.forward / infer (later.py:277-291, 344-351; torch LSTMCell,
// gate order i, f, g, o:  c' = f c + i g,  h' = o tanh(c')) and their autograd.  As in the GRU kernels the layer-0
// input projection gi = x W_ih^T + b_ih arrives precomputed for all steps (time-major [T,B,4H]).  Extra layers are
// applied as  (h, c) = layer(h, (h, c))  (later.py:279-281): ONE (h, c) pair is threaded through all cells of a step and
// on to the next step, so the cells form a single chain  (t,0) -> (t,1) -> ... -> (t,L-1) -> (t+1,0).
// The pre-activation is a plain sum gi + gh, so one gate-gradient array dG serves both weight-gradient products.
//
// Same decomposition as gru_seq.cu: a CTA owns 4 batch rows and keeps (h, c) in shared memory; the generated weights
// (k-major, 16-byte rows) stream from L2 every step.  The grouped kernels run the same rows code for a many-style batch:
// each CTA takes a tile of <= 4 rows of one style group and that group's slice of a per-group weight pack.
#include "seq_common.cuh"

namespace caphn {

constexpr int LSTM_MAX_EXTRA = 3;

struct LstmFwdArgs {
    const float* GI;     // [T,B,4H] layer-0 input projection (+ b_ih)
    const float* WhhT;   // [H, ld4] layer 0
    const float* bhh;    // [4H]
    float* Hall;         // [T+1,B,H]: Hall[0] = h0 (zeros), Hall[t+1] = h after the LAST cell of step t
    float* Hbm;          // [B,T,H] or null
    float* saved;        // [NL][6][T,B,H]  (i, f, g, o, c_prev, tanh(c')) or null
    float* Hmid;         // [NL-1][T,B,H] outputs of cells 0..NL-2
    const float* xWihT[LSTM_MAX_EXTRA];
    const float* xWhhT[LSTM_MAX_EXTRA];
    const float* xbih[LSTM_MAX_EXTRA];
    const float* xbhh[LSTM_MAX_EXTRA];
    const float* c0;     // [B,H] initial cell state, or null = zeros (later.py:258-259)
    float* cT;           // [B,H] cell state after the last step, or null (one-step-per-call decode)
    int NL, B, T, H, ld4;
};

// Batch rows [b0, b0 + nb) (nb <= AT_BT) of the whole recurrence; cell 0 uses WhhT / bhh.  The single-style kernel passes
// the CTA's 4 rows and the call's weights, the grouped kernel a tile of one style group and that group's weights.
__device__ __forceinline__ void lstm_fwd_rows(const LstmFwdArgs& a, const float* __restrict__ WhhT,
                                              const float* __restrict__ bhh0, int b0, int nb) {
    constexpr int BT = AT_BT;
    extern __shared__ __align__(16) float smem[];
    const int H = a.H, B = a.B, T = a.T, ld4 = a.ld4, H4 = 4 * a.H;
    const int CQT = at_cqt(ld4), KG = AT_THREADS / CQT;
    float* hs = smem;                           // [H][BT]
    float* cs = hs + H * BT;                    // [BT][H]
    float* part_gh = cs + ((BT * H + 3) & ~3);  // [KG][BT][ld4]
    float* part_gi = part_gh + KG * BT * ld4;   // [KG][BT][ld4]   (extra layers only)
    const int tid = threadIdx.x;
    const long TBH = (long)T * B * H;

    for (int i = tid; i < H * BT; i += AT_THREADS) {
        const int k = i / BT, b = i - k * BT;
        hs[i] = (b < nb) ? a.Hall[(long)(b0 + b) * H + k] : 0.f;
    }
    for (int i = tid; i < BT * H; i += AT_THREADS) {
        const int b = i / H, j = i - b * H;
        cs[i] = (a.c0 && b < nb) ? a.c0[(long)(b0 + b) * H + j] : 0.f;
    }
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        for (int l = 0; l < a.NL; ++l) {
            const bool last = (l == a.NL - 1);
            if (l == 0) {
                block_matvec<BT, false>(WhhT, ld4, H, hs, part_gh, CQT, tid);
            } else {
                block_matvec<BT, false>(a.xWihT[l - 1], ld4, H, hs, part_gi, CQT, tid);
                block_matvec<BT, false>(a.xWhhT[l - 1], ld4, H, hs, part_gh, CQT, tid);
            }
            __syncthreads();
            const float* bhh = (l == 0) ? bhh0 : a.xbhh[l - 1];
            for (int i = tid; i < BT * H; i += AT_THREADS) {
                const int b = i / H, j = i - b * H;
                const int gb = b0 + b;
                if (b < nb) {
                    float g4[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float v = bhh[q * H + j] + part_sum(part_gh, KG, BT, ld4, b, q * H + j);
                        if (l == 0) v += a.GI[((long)t * B + gb) * H4 + q * H + j];
                        else v += a.xbih[l - 1][q * H + j] + part_sum(part_gi, KG, BT, ld4, b, q * H + j);
                        g4[q] = v;
                    }
                    const float ig = sigmoidf_acc(g4[0]), fg = sigmoidf_acc(g4[1]), gg = tanhf(g4[2]), og = sigmoidf_acc(g4[3]);
                    const float cp = cs[i];
                    const float cn = fg * cp + ig * gg;
                    const float tc = tanhf(cn);
                    const float hn = og * tc;
                    cs[i] = cn;
                    hs[j * BT + b] = hn;
                    const long o = ((long)t * B + gb) * H + j;
                    if (last) {
                        a.Hall[o + (long)B * H] = hn;
                        if (a.Hbm) a.Hbm[((long)gb * T + t) * H + j] = hn;
                    } else if (a.Hmid) {
                        a.Hmid[(long)l * TBH + o] = hn;
                    }
                    if (a.saved) {
                        float* sv = a.saved + (long)l * 6 * TBH + o;
                        sv[0] = ig; sv[TBH] = fg; sv[2 * TBH] = gg; sv[3 * TBH] = og; sv[4 * TBH] = cp; sv[5 * TBH] = tc;
                    }
                }
            }
            __syncthreads();
        }
    }
    if (a.cT)
        for (int i = tid; i < BT * H; i += AT_THREADS) {
            const int b = i / H, j = i - b * H;
            if (b < nb) a.cT[(long)(b0 + b) * H + j] = cs[i];
        }
}

__global__ void __launch_bounds__(AT_THREADS) lstm_seq_fwd_kernel(const LstmFwdArgs a) {
    const int b0 = blockIdx.x * AT_BT;
    lstm_fwd_rows(a, a.WhhT, a.bhh, b0, min(AT_BT, a.B - b0));
}

// Many-style batch (rows sorted by group, one layer): CTA i runs tile i = {first row, rows <= AT_BT, group, 0} with its
// group's slice [H][ld4] of the W_hh^T pack and b_hh at bhh + group * bstride.
__global__ void __launch_bounds__(AT_THREADS) lstm_seq_fwd_grouped_kernel(const LstmFwdArgs a, const int4* __restrict__ tiles,
                                                                          long bstride) {
    const int4 tl = tiles[blockIdx.x];
    lstm_fwd_rows(a, a.WhhT + (long)tl.z * a.H * a.ld4, a.bhh + (long)tl.z * bstride, tl.x, tl.y);
}

struct LstmBwdArgs {
    const float* dHbm;   // [B,T,H] gradient w.r.t. the last cell's h at every step
    const float* saved;  // [NL][6][T,B,H]
    const float* Whh;    // [4H, ldh] layer 0
    const float* xWih[LSTM_MAX_EXTRA];  // [4H, ldh]
    const float* xWhh[LSTM_MAX_EXTRA];
    float* dG;           // [NL][T,B,4H] gate pre-activation gradients
    float* dh0;          // [B,H]
    int NL, B, T, H, ldh;
};

// Batch rows [b0, b0 + nb) (nb <= AT_BT) of the BPTT; cell 0 uses Whh.
__device__ __forceinline__ void lstm_bwd_rows(const LstmBwdArgs& a, const float* __restrict__ Whh, int b0, int nb) {
    constexpr int BT = AT_BT;
    extern __shared__ __align__(16) float smem[];
    const int H = a.H, B = a.B, T = a.T, ldh = a.ldh, H4 = 4 * a.H;
    const int CQTh = at_cqt(ldh), KGh = AT_THREADS / CQTh;
    float* dg = smem;                                // [4H][BT]
    float* dcs = dg + H4 * BT;                       // [BT][H] carried d c
    float* dhin = dcs + ((BT * H + 3) & ~3);         // [BT][H] gradient handed from cell l to cell l-1
    float* part_dh = dhin + ((BT * H + 3) & ~3);     // [KGh][BT][ldh]  dG . W_hh of layer 0 (for the previous step)
    float* part_di = part_dh + KGh * BT * ldh;       // [KGh][BT][ldh]  dG . (W_hh + W_ih) of an extra layer
    const int tid = threadIdx.x;
    const long TBH = (long)T * B * H, TB4 = (long)T * B * H4;

    for (int i = tid; i < BT * H; i += AT_THREADS) dcs[i] = 0.f;
    for (int i = tid; i < KGh * BT * ldh; i += AT_THREADS) part_dh[i] = 0.f;
    __syncthreads();

    for (int t = T - 1; t >= 0; --t) {
        for (int l = a.NL - 1; l >= 0; --l) {
            const bool top = (l == a.NL - 1);
            for (int i = tid; i < BT * H; i += AT_THREADS) {
                const int b = i / H, j = i - b * H;
                const int gb = b0 + b;
                float da[4] = {0.f, 0.f, 0.f, 0.f};
                float dcp = 0.f;
                if (b < nb) {
                    float dh;
                    if (top) dh = a.dHbm[((long)gb * T + t) * H + j] + part_sum(part_dh, KGh, BT, ldh, b, j);
                    else dh = dhin[i];
                    const long o = ((long)t * B + gb) * H + j;
                    const float* sv = a.saved + (long)l * 6 * TBH + o;
                    const float ig = sv[0], fg = sv[TBH], gg = sv[2 * TBH], og = sv[3 * TBH], cp = sv[4 * TBH], tc = sv[5 * TBH];
                    const float dct = dcs[i] + dh * og * (1.f - tc * tc);
                    da[0] = dct * gg * ig * (1.f - ig);
                    da[1] = dct * cp * fg * (1.f - fg);
                    da[2] = dct * ig * (1.f - gg * gg);
                    da[3] = dh * tc * og * (1.f - og);
                    dcp = dct * fg;
                    float* g = a.dG + (long)l * TB4 + ((long)t * B + gb) * H4;
                    g[j] = da[0]; g[H + j] = da[1]; g[2 * H + j] = da[2]; g[3 * H + j] = da[3];
                }
                dcs[i] = dcp;
#pragma unroll
                for (int q = 0; q < 4; ++q) dg[(q * H + j) * BT + b] = da[q];
            }
            __syncthreads();
            if (l == 0) {
                block_matvec<BT, false>(Whh, ldh, H4, dg, part_dh, CQTh, tid);
                __syncthreads();
            } else {
                // input and state of an extra cell are the same vector: both products flow into the cell below
                block_matvec<BT, false>(a.xWhh[l - 1], ldh, H4, dg, part_di, CQTh, tid);
                block_matvec<BT, true>(a.xWih[l - 1], ldh, H4, dg, part_di, CQTh, tid);
                __syncthreads();
                for (int i = tid; i < BT * H; i += AT_THREADS) {
                    const int b = i / H, j = i - b * H;
                    dhin[i] = part_sum(part_di, KGh, BT, ldh, b, j);
                }
                __syncthreads();
            }
        }
    }
    for (int i = tid; i < BT * H; i += AT_THREADS) {
        const int b = i / H, j = i - b * H;
        if (b < nb) a.dh0[(long)(b0 + b) * H + j] = part_sum(part_dh, KGh, BT, ldh, b, j);
    }
}

__global__ void __launch_bounds__(AT_THREADS) lstm_seq_bwd_kernel(const LstmBwdArgs a) {
    const int b0 = blockIdx.x * AT_BT;
    lstm_bwd_rows(a, a.Whh, b0, min(AT_BT, a.B - b0));
}

// BPTT of lstm_seq_fwd_grouped_kernel: tile i with its group's slice [4H][ldh] of the W_hh pack.
__global__ void __launch_bounds__(AT_THREADS) lstm_seq_bwd_grouped_kernel(const LstmBwdArgs a, const int4* __restrict__ tiles) {
    const int4 tl = tiles[blockIdx.x];
    lstm_bwd_rows(a, a.Whh + (long)tl.z * 4 * a.H * a.ldh, tl.x, tl.y);
}

}  // namespace caphn

using namespace caphn;

extern "C" {

// LSTM recurrence over T steps (all cells).  GI [T,B,4H] (layer-0 x-projection incl. b_ih); WhhT [H, ld4] (ld4 % 4 == 0,
// 16 B aligned, gate order i,f,g,o); Hall [T+1,B,H] with Hall[0] = h0 (zeros in the reference) filled by the caller; the
// cell state starts at c0 (NULL = zeros) and is returned in cT (or NULL).  `extra`: HOST array of 4*(NL-1) device pointers {WihT_l, WhhT_l, bih_l, bhh_l}.
// saved [NL][6][T,B,H] and Hmid [NL-1][T,B,H] are needed for the backward (or NULL).
int caphn_lstm_seq_fwd(const float* GI, const float* WhhT, int ld4, const float* bhh, float* Hall, float* Hbm,
                       float* saved, float* Hmid, const void* const* extra, const float* c0, float* cT, int NL, int B,
                       int T, int H, void* stream) {
    if (B <= 0 || T <= 0 || H <= 0 || (ld4 & 3) || ld4 < 4 * H || ((uintptr_t)WhhT & 15)) return CAPHN_EINVAL;
    if (NL < 1 || NL > 1 + LSTM_MAX_EXTRA || (NL > 1 && !extra) || (NL > 1 && saved && !Hmid)) return CAPHN_EINVAL;
    LstmFwdArgs a{};
    a.GI = GI; a.WhhT = WhhT; a.bhh = bhh; a.Hall = Hall; a.Hbm = Hbm; a.saved = saved; a.Hmid = Hmid;
    a.c0 = c0; a.cT = cT; a.NL = NL; a.B = B; a.T = T; a.H = H; a.ld4 = ld4;
    for (int l = 0; l < NL - 1; ++l) {
        a.xWihT[l] = (const float*)extra[4 * l]; a.xWhhT[l] = (const float*)extra[4 * l + 1];
        a.xbih[l] = (const float*)extra[4 * l + 2]; a.xbhh[l] = (const float*)extra[4 * l + 3];
        if (((uintptr_t)a.xWihT[l] & 15) || ((uintptr_t)a.xWhhT[l] & 15)) return CAPHN_EINVAL;
    }
    const int KG = AT_THREADS / at_cqt(ld4);
    const size_t smem = ((size_t)H * AT_BT + (size_t)((AT_BT * H + 3) & ~3) + 2 * (size_t)KG * AT_BT * ld4) * sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(lstm_seq_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lstm_seq_fwd_kernel<<<ceil_div(B, AT_BT), AT_THREADS, smem, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

// BPTT of caphn_lstm_seq_fwd.  Whh [4H, ldh] (ldh % 4 == 0); `extra` = HOST array of 2*(NL-1) device pointers
// {Wih_l, Whh_l} ([4H, ldh] each).  Outputs: dG [NL][T,B,4H] (gate pre-activation gradients: dW_ih = dG^T x,
// dW_hh = dG^T h_prev, db_ih = db_hh = colsum dG), dh0 [B,H].
int caphn_lstm_seq_bwd(const float* dHbm, const float* saved, const float* Whh, int ldh, const void* const* extra,
                       float* dG, float* dh0, int NL, int B, int T, int H, void* stream) {
    if (B <= 0 || T <= 0 || H <= 0 || (ldh & 3) || ldh < H || ((uintptr_t)Whh & 15)) return CAPHN_EINVAL;
    if (NL < 1 || NL > 1 + LSTM_MAX_EXTRA || (NL > 1 && !extra)) return CAPHN_EINVAL;
    LstmBwdArgs a{};
    a.dHbm = dHbm; a.saved = saved; a.Whh = Whh; a.dG = dG; a.dh0 = dh0; a.NL = NL; a.B = B; a.T = T; a.H = H; a.ldh = ldh;
    for (int l = 0; l < NL - 1; ++l) {
        a.xWih[l] = (const float*)extra[2 * l]; a.xWhh[l] = (const float*)extra[2 * l + 1];
        if (((uintptr_t)a.xWih[l] & 15) || ((uintptr_t)a.xWhh[l] & 15)) return CAPHN_EINVAL;
    }
    const int KGh = AT_THREADS / at_cqt(ldh);
    const size_t smem = ((size_t)4 * H * AT_BT + 2 * (size_t)((AT_BT * H + 3) & ~3) + 2 * (size_t)KGh * AT_BT * ldh) *
                        sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(lstm_seq_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lstm_seq_bwd_kernel<<<ceil_div(B, AT_BT), AT_THREADS, smem, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

// Single-layer LSTM recurrence of a many-style batch (rows sorted by style group; h0 = Hall[0], c0 = zeros).  CTA i runs
// tiles[i] = {first row, rows (1..4), group, 0} (16-byte aligned int4 table, no tile straddles two groups) with the group's
// W_hh^T from the pack WhhT [G][H][ld4] and b_hh = bhh + group * bstride (floats).  GI, Hall, Hbm, saved [6][T,B,H] and
// cT (or NULL) as in caphn_lstm_seq_fwd; every row computes exactly what the single-style kernel computes for it.
int caphn_lstm_seq_fwd_grouped(const float* GI, const float* WhhT, int ld4, const float* bhh, long bstride, float* Hall,
                               float* Hbm, float* saved, float* cT, int B, int T, int H, const int* tiles, int ntiles,
                               void* stream) {
    if (B <= 0 || T <= 0 || H <= 0 || (ld4 & 3) || ld4 < 4 * H || ((uintptr_t)WhhT & 15)) return CAPHN_EINVAL;
    if (!tiles || ntiles < 1 || ((uintptr_t)tiles & 15) || bstride < 0) return CAPHN_EINVAL;
    LstmFwdArgs a{};
    a.GI = GI; a.WhhT = WhhT; a.bhh = bhh; a.Hall = Hall; a.Hbm = Hbm; a.saved = saved; a.cT = cT;
    a.NL = 1; a.B = B; a.T = T; a.H = H; a.ld4 = ld4;
    const int KG = AT_THREADS / at_cqt(ld4);
    const size_t smem = ((size_t)H * AT_BT + (size_t)((AT_BT * H + 3) & ~3) + 2 * (size_t)KG * AT_BT * ld4) * sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(lstm_seq_fwd_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lstm_seq_fwd_grouped_kernel<<<ntiles, AT_THREADS, smem, (cudaStream_t)stream>>>(a, (const int4*)tiles, bstride);
    CAPHN_RETURN_LAST();
}

// BPTT of caphn_lstm_seq_fwd_grouped: the group's W_hh from the pack Whh [G][4H][ldh]; dG [T,B,4H], dh0 [B,H].
int caphn_lstm_seq_bwd_grouped(const float* dHbm, const float* saved, const float* Whh, int ldh, float* dG, float* dh0,
                               int B, int T, int H, const int* tiles, int ntiles, void* stream) {
    if (B <= 0 || T <= 0 || H <= 0 || (ldh & 3) || ldh < H || ((uintptr_t)Whh & 15)) return CAPHN_EINVAL;
    if (!tiles || ntiles < 1 || ((uintptr_t)tiles & 15)) return CAPHN_EINVAL;
    LstmBwdArgs a{};
    a.dHbm = dHbm; a.saved = saved; a.Whh = Whh; a.dG = dG; a.dh0 = dh0; a.NL = 1; a.B = B; a.T = T; a.H = H; a.ldh = ldh;
    const int KGh = AT_THREADS / at_cqt(ldh);
    const size_t smem = ((size_t)4 * H * AT_BT + 2 * (size_t)((AT_BT * H + 3) & ~3) + 2 * (size_t)KGh * AT_BT * ldh) *
                        sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(lstm_seq_bwd_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lstm_seq_bwd_grouped_kernel<<<ntiles, AT_THREADS, smem, (cudaStream_t)stream>>>(a, (const int4*)tiles);
    CAPHN_RETURN_LAST();
}

}  // extern "C"
