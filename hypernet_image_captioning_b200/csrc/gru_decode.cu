// One greedy-decode step of the pooled captioner as ONE launch (reference later.py:459-490: argmax feedback -> embedding ->
// nn.GRUCell -> fc_out): finishes the arg-max of the previous step's vocabulary projection from the partials its GEMM epilogue
// left (caphn_gemm_tc_amax), takes the next input's projection  P[tok] = Emb[tok] W_ih^T + b_ih  from the projection table,
// runs the GRU cell against the generated W_hh and writes the new state both as fp32 and as the bf16 hi/lo operand rows of the
// next vocabulary projection.  Replaces argmax_finish_gather + gru_seq_fwd(T = 1) + split_bf16 -- three dependent launches
// (5 + 16 + 3 us at B = 512, H = 150) on the 20-step dependency chain of DecoderGRU.infer.  The token-fed variant
// (caphn_gru_decode_step_tok) takes the token from an array instead: DecoderGRU.beam_search_batched feeds it the words the
// beam bookkeeping kernel chose.
//
// Grid: (ceil(H / 32) unit blocks, row blocks), sized to at most one CTA per SM (one wave, no SM with two CTAs' worth of
// shared-memory reads): a CTA of W warps owns 2 W batch rows x 32 hidden units.  The 3 x 32 rows of W_hh it needs sit in shared
// memory (row stride = 2 x odd floats: the float2 reads of a warp, lane = unit, are conflict-free) next to its rows' previous
// states (k-major pairs: one 8-byte broadcast per row pair and k); warp w owns rows 2w, 2w + 1, lane = hidden unit; fp32 FMA
// throughout (the same precision class as gru_seq.cu, whose T = 1 launch this replaces; k ascending per output).  H even.
#include "common.cuh"
#include <cuda_bf16.h>
#include <math.h>

namespace caphn {

constexpr int GD_UNITS = 32;
constexpr int GD_MAXW = 16;

__device__ __forceinline__ void gd_cp_async8(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// Where a step's input projection comes from (template parameter of the kernel).  GD_SRC_GREEDY: GI if given, else row tok
// of the table with tok finished from the arg-max partials -- one instantiation, so greedy decode runs the same machine code
// for both.  GD_SRC_TOK: row tokin[b] of the table (an entry outside [0, V): row 0).  tokin / V are kernel parameters of
// their own, not GruDecArgs fields, so the greedy instantiation's parameter block and machine code stay as they were.
enum GruDecSrc { GD_SRC_GREEDY = 0, GD_SRC_TOK = 1 };

struct GruDecArgs {
    const float* GI;        // [B, 3H] input projection incl. b_ih (step 0), or NULL: gather table[tok] with tok from the partials
    const float* pval; const int* pidx; int ldp, nparts;   // arg-max partials of the previous step [B, ldp]
    const float* table;     // [V, 3H]
    const float* Whh;       // [3H, H]
    const float* bhh;       // [3H]
    const float* hprev;     // [B, H]
    float* hnew;            // [B, H]
    __nv_bfloat16* hi; __nv_bfloat16* lo; long Kp;   // operand rows [B, Kp] (lo may be NULL)
    long long* tok;         // [B] or NULL
    int B, H, ldw, nw;      // ldw: shared row stride of the weight slice; nw: warps per CTA (rows per CTA = 2 nw)
};

template <int SRC>
__global__ void __launch_bounds__(GD_MAXW * 32) gru_decode_step_kernel(const GruDecArgs a, const int* tokin, int V) {
    extern __shared__ float2 gd_smem2[];
    float* gd_smem = reinterpret_cast<float*>(gd_smem2);
    const int H = a.H, B = a.B, H3 = 3 * a.H, ldw = a.ldw, nw = a.nw, H2 = a.H >> 1;
    const int hstr = 2 * nw;                               // floats per k in the state tile
    float* Ws = gd_smem;                                   // [3 * 32][ldw]
    float* hs = Ws + 3 * GD_UNITS * ldw;                   // [H][2 nw]  k-major
    __shared__ int s_tok[2 * GD_MAXW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int j0 = blockIdx.x * GD_UNITS, b0 = blockIdx.y * 2 * nw;

    // Everything this CTA needs from global memory is requested up front, so the launch pays ~2 dependent round trips
    // (the gathered projection rows need the token) instead of one per loop iteration.
    // (1) W_hh rows {r, z, n} of this CTA's units: asynchronous 8-byte copies straight into shared memory (rows are H even
    //     floats, 8-byte aligned); warp w copies slice rows w, w + nw, ...
    for (int lr = warp; lr < 3 * GD_UNITS; lr += nw) {
        const int g = lr >> 5, j = j0 + (lr & 31);
        float* dst = Ws + lr * ldw;
        if (j < H) {
            const float* src = a.Whh + ((long)g * H + j) * H;
            for (int c = lane; c < H2; c += 32) gd_cp_async8(dst + 2 * c, src + 2 * c);
        } else {
            for (int c = lane; c < H2; c += 32) *reinterpret_cast<float2*>(dst + 2 * c) = make_float2(0.f, 0.f);
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    // (2) arg-max partials and previous states of this warp's two rows: independent loads, all in flight together
    constexpr int PMAX = 8;                                // partial slots per lane (nparts <= 256)
    constexpr int KMAX = 13;                               // state elements per lane (H <= 416)
    float pvr[2][PMAX];
    int pir[2][PMAX];
    float hreg[2][KMAX];
    int tin[2] = {0, 0};
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        const int b = b0 + 2 * warp + rr;
        if (SRC == GD_SRC_TOK && b < B) tin[rr] = tokin[b];
        if (SRC == GD_SRC_GREEDY && !a.GI) {
#pragma unroll
            for (int it = 0; it < PMAX; ++it) {
                const int q = lane + 32 * it;
                const bool ok = b < B && q < a.nparts;
                pvr[rr][it] = ok ? a.pval[(long)b * a.ldp + q] : -INFINITY;
                pir[rr][it] = ok ? a.pidx[(long)b * a.ldp + q] : 0x7fffffff;
            }
        }
#pragma unroll
        for (int it = 0; it < KMAX; ++it) {
            const int k = lane + 32 * it;
            hreg[rr][it] = (b < B && k < H) ? a.hprev[(long)b * H + k] : 0.f;
        }
    }
    // (3) finish the arg-max of the previous step for this warp's rows (lowest column on ties)
    if (SRC == GD_SRC_GREEDY && !a.GI) {
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int b = b0 + 2 * warp + rr;
            float bv = -INFINITY;
            int bi = 0x7fffffff;
#pragma unroll
            for (int it = 0; it < PMAX; ++it) {            // ascending columns per lane
                const float v = pvr[rr][it];
                const int c = pir[rr][it];
                if (v > bv || (v == bv && c < bi)) { bv = v; bi = c; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (bi == 0x7fffffff) bi = 0;                  // all partials empty (logits all NaN / -inf): token 0
            if (lane == 0 && b < B) {
                s_tok[2 * warp + rr] = bi;
                if (a.tok && blockIdx.x == 0) a.tok[b] = bi;
            }
        }
        __syncwarp();
    }
    // (4) gate inputs of this thread's (rows, unit): the loads fly while the weight slice lands and the product runs
    const int j = j0 + lane;
    float gir[2] = {0.f, 0.f}, giz[2] = {0.f, 0.f}, gin[2] = {0.f, 0.f};
    float bhr = 0.f, bhz = 0.f, bhn = 0.f;
    if (j < H) {
        bhr = a.bhh[j]; bhz = a.bhh[H + j]; bhn = a.bhh[2 * H + j];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int r = 2 * warp + rr, b = b0 + r;
            if (b < B) {
                const float* gi = SRC == GD_SRC_TOK ? a.table + (long)((unsigned)tin[rr] < (unsigned)V ? tin[rr] : 0) * H3
                                : a.GI ? a.GI + (long)b * H3 : a.table + (long)s_tok[r] * H3;
                gir[rr] = gi[j]; giz[rr] = gi[H + j]; gin[rr] = gi[2 * H + j];
            }
        }
    }
#pragma unroll
    for (int rr = 0; rr < 2; ++rr)
#pragma unroll
        for (int it = 0; it < KMAX; ++it) {
            const int k = lane + 32 * it;
            if (k < H) hs[k * hstr + 2 * warp + rr] = hreg[rr][it];
        }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    // (5) gh[row][gate] = sum_k W[gate][unit][k] h[row][k], two k per iteration
    float acc[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    const float2* w0 = reinterpret_cast<const float2*>(Ws + lane * ldw);
    const float2* w1 = reinterpret_cast<const float2*>(Ws + (GD_UNITS + lane) * ldw);
    const float2* w2 = reinterpret_cast<const float2*>(Ws + (2 * GD_UNITS + lane) * ldw);
    const float* hp = hs + 2 * warp;
#pragma unroll 5
    for (int c = 0; c < H2; ++c) {
        const float2 ha = *reinterpret_cast<const float2*>(hp + (2 * c) * hstr);        // (row 0, row 1) at k = 2c
        const float2 hb = *reinterpret_cast<const float2*>(hp + (2 * c + 1) * hstr);    // at k = 2c + 1
        const float2 wr = w0[c], wz = w1[c], wn = w2[c];
        acc[0][0] = fmaf(wr.x, ha.x, acc[0][0]); acc[1][0] = fmaf(wr.x, ha.y, acc[1][0]);
        acc[0][1] = fmaf(wz.x, ha.x, acc[0][1]); acc[1][1] = fmaf(wz.x, ha.y, acc[1][1]);
        acc[0][2] = fmaf(wn.x, ha.x, acc[0][2]); acc[1][2] = fmaf(wn.x, ha.y, acc[1][2]);
        acc[0][0] = fmaf(wr.y, hb.x, acc[0][0]); acc[1][0] = fmaf(wr.y, hb.y, acc[1][0]);
        acc[0][1] = fmaf(wz.y, hb.x, acc[0][1]); acc[1][1] = fmaf(wz.y, hb.y, acc[1][1]);
        acc[0][2] = fmaf(wn.y, hb.x, acc[0][2]); acc[1][2] = fmaf(wn.y, hb.y, acc[1][2]);
    }
    // (6) gates, new state, operand rows
    if (j < H) {
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int r = 2 * warp + rr, b = b0 + r;
            if (b < B) {
                const float ghr = bhr + acc[rr][0], ghz = bhz + acc[rr][1], ghn = bhn + acc[rr][2];
                const float rg = sigmoidf_acc(gir[rr] + ghr);
                const float zg = sigmoidf_acc(giz[rr] + ghz);
                const float ng = tanhf(gin[rr] + rg * ghn);
                const float hn = (1.f - zg) * ng + zg * hs[j * hstr + r];
                a.hnew[(long)b * H + j] = hn;
                if (a.hi) {
                    const __nv_bfloat16 h = __float2bfloat16_rn(hn);
                    a.hi[(long)b * a.Kp + j] = h;
                    if (a.lo) a.lo[(long)b * a.Kp + j] = __float2bfloat16_rn(hn - __bfloat162float(h));
                }
            }
        }
    }
}

}  // namespace caphn

using namespace caphn;

// Sizes the grid and launches the instantiation for SRC; the caller has checked the source-specific arguments.
template <int SRC>
static int gd_launch(const GruDecArgs& args, const int* tokin, int V, void* stream) {
    GruDecArgs a = args;
    const int B = a.B, H = a.H;
    if (B <= 0 || H <= 0 || (H & 1) || !a.Whh || !a.bhh || !a.hprev || !a.hnew || a.hnew == a.hprev) return CAPHN_EINVAL;
    if (((uintptr_t)a.Whh & 7)) return CAPHN_EINVAL;
    if (a.hi && a.Kp < H) return CAPHN_EINVAL;
    // row blocks: as many as keep the grid within one CTA per SM, at most 32 rows (16 warps) per CTA
    const int ub = ceil_div(H, GD_UNITS);
    int rb = kNumSMs / ub;
    if (rb < 1) rb = 1;
    int nw = ceil_div(ceil_div(B, rb), 2);
    if (nw > GD_MAXW) nw = GD_MAXW;
    if (nw < 1) nw = 1;
    a.ldw = ((H >> 1) & 1) ? H : H + 2;                    // (ldw / 2) odd
    a.nw = nw;
    const size_t smem = ((size_t)3 * GD_UNITS * a.ldw + (size_t)2 * nw * H) * sizeof(float);
    if (smem > 200 * 1024 || H > 416) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(gru_decode_step_kernel<SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)ub, (unsigned)ceil_div(B, 2 * nw));
    gru_decode_step_kernel<SRC><<<grid, nw * 32, smem, (cudaStream_t)stream>>>(a, tokin, V);
    CAPHN_RETURN_LAST();
}

extern "C" {

// One greedy-decode step of DecoderGRU.infer (single layer).  GI != NULL: the input projection [B, 3H] (incl. b_ih) is given
// (step 0: the image feature).  GI == NULL: the previous step's token is the arg-max of the nparts (value, column) partials
// per row in pval / pidx [B, ldp] (caphn_gemm_tc_amax; lowest column on ties; written to tok if non-NULL) and the projection
// is row tok of table [V, 3H].  Outputs: hnew [B, H] and, if hi != NULL, its bf16 hi / lo split [B, Kp] (lo may be NULL).
// hnew must not alias hprev.
int caphn_gru_decode_step(const float* GI, const float* pval, const int* pidx, int ldp, int nparts, const float* table,
                          const float* Whh, const float* bhh, const float* hprev, float* hnew, void* hi, void* lo, long Kp,
                          long long* tok, int B, int H, void* stream) {
    if (!GI && (!pval || !pidx || !table || nparts <= 0 || nparts > ldp)) return CAPHN_EINVAL;
    if (nparts > 256) return CAPHN_EINVAL;
    const GruDecArgs a{GI, pval, pidx, ldp, nparts, table, Whh, bhh, hprev, hnew, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, Kp,
                       tok, B, H, 0, 0};
    return gd_launch<GD_SRC_GREEDY>(a, nullptr, 0, stream);
}

// The same step with the input token given: row b's input projection is table[tok[b]] (an entry outside [0, V) reads row 0).
// Beam search feeds the tokens its bookkeeping kernel chose (caphn_beam_step's prev_tok).  No partials, so no limit on V.
int caphn_gru_decode_step_tok(const int* tok, int V, const float* table, const float* Whh, const float* bhh,
                              const float* hprev, float* hnew, void* hi, void* lo, long Kp, int B, int H, void* stream) {
    if (!tok || !table || V <= 0) return CAPHN_EINVAL;
    const GruDecArgs a{nullptr, nullptr, nullptr, 0, 0, table, Whh, bhh, hprev, hnew, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo,
                       Kp, nullptr, B, H, 0, 0};
    return gd_launch<GD_SRC_TOK>(a, tok, V, stream);
}

}  // extern "C"
