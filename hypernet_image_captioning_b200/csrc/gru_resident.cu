// Weights-resident GRU recurrence, one CTA per 4 batch rows, NO cluster: the whole generated W_hh ([3H, H] fp32, 270 KB at
// H = 150 -- more than one SM's shared memory) is held by a single CTA as THREAD-PRIVATE weight vectors, the first KS
// elements of each in shared memory (odd row stride: conflict-free) and the last KR in registers (512 threads x KR floats).
// Every step is then CTA-local -- two __syncthreads instead of the DSMEM exchange + cluster barrier of gru_cluster.cu, whose
// per-step cost (7.4 us at B = 512, T = 20, H = 150, of which ~1.7 us is the product itself) was dominated by that
// exchange.  This is the north-star design of BASELINE.json ("persistent kernel that keeps each style group's generated W_hh
// resident ... across timesteps, gates / state update / BPTT gate gradients fused in") for the single-style, single-layer
// case; gru_cluster.cu keeps the many-style (per-group weights) variant, gru_seq.cu the multi-layer / large-H fallback.
//
// Replaces nn.GRUCell per step + autograd BPTT (later.py:411,418) like gru_seq.cu.  Same buffers: GI [T,B,3H] (input
// projection incl. b_ih), Hall [T+1,B,H], Hbm [B,T,H], saved [4][T,B,H] = (r, z, n, gh_n).
//   forward : thread j < 3H owns weight row j;          gh[row][j]  = sum_k  W[j][k] h[row][k]       (k ascending)
//   backward: thread (g, k) owns column k of gate block g; part[g][row][k] = sum_jj dgh[row][gH + jj] W[gH + jj][k]
#include "common.cuh"
#include <math.h>
#include <stdlib.h>

namespace caphn {

constexpr int GR_THREADS = 512;
constexpr int GR_RB = 4;          // batch rows per CTA

__device__ __forceinline__ void gr_cp_async4(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
                 : "memory");
}
__device__ __forceinline__ void gr_cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

struct GruResArgs {
    const float* GI; const float* Whh; const float* bhh;
    float* Hall; float* Hbm; float* saved;
    const float* dHbm; float* dGI; float* dGH; float* dh0;     // backward only
    int B, T, H, KS, ldw;                                      // KS = H - KR (elements of a weight vector kept in smem)
};

// Forward.  Thread (ks, u) = (k third, hidden unit) -- warp w: ks = w / UB, u = (w % UB) * 32 + lane, UB = ceil(H / 32) --
// owns the three gate rows {r, z, n} of unit u over k in [ks KC, (ks + 1) KC), KC = ceil(H / 3): a private vector of 3 KC
// weights ordered (kk, gate), the first KS (multiple of 3) in shared memory, the last KR in registers.  Per k it reads three
// private weights and ONE broadcast float4 of the state (4 batch rows) for 12 FMAs -- the broadcast reads were the bottleneck
// of the one-row-per-thread layout (4 FMAs per broadcast).  The three k-partials per gate meet in shared memory.
template <int KR>
__global__ void __launch_bounds__(GR_THREADS, 1) gru_res_fwd_kernel(const GruResArgs a) {
    extern __shared__ __align__(16) float gr_smem[];
    const int H = a.H, H3 = 3 * a.H, KS = a.KS, ldw = a.ldw, B = a.B, T = a.T;
    const int KC = (H + 2) / 3, HP = 3 * KC;               // k per third; padded state length
    const int UB = (H + 31) >> 5;                          // warps per k third
    float* Ws = gr_smem;                                   // [3 (ks)][H (u)][ldw]   thread-private vectors
    float* hs = Ws + (((long)H3 * ldw + 3) & ~3L);         // [2][HP][4]  state, k-major, 4 rows contiguous; tail zero
    float* gps = hs + 2 * HP * GR_RB;                      // [3 (ks)][3H][4]  partial gh
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b0 = blockIdx.x * GR_RB, nb = min(GR_RB, B - b0);
    const long TBH = (long)T * B * H;
    const int ks = warp / UB, u_own = (warp - ks * UB) * 32 + lane;
    const bool owner = ks < 3 && u_own < H;
    const int vrow = ks * H + u_own;                       // row of this thread's vector in Ws

    // ---- weights: W[g H + u][k] -> vector (ks = k / KC, u), element e = (k % KC) * 3 + g.  Warp w copies rows w, w + 16, ...
    //      of W_hh with its lanes along k (coalesced, asynchronous 4-byte copies, no divisions in the loop: the lane's k
    //      positions are decoded once); the register part (e >= KS) is staged through the still empty Ws area first ----
    constexpr int KIT = 6;                                 // k positions per lane: H <= 192 (3H <= 512 anyway)
    const int KSK = KS / 3;                                // k steps (per third) whose weights are in shared memory
    const int sst = KR | 1;
    int dR[KIT], dS[KIT];                                  // destination offsets of k = lane + 32 it (-1: not in this part)
#pragma unroll
    for (int it = 0; it < KIT; ++it) {
        const int k = lane + 32 * it;
        const int kq = k / KC, kk = k - kq * KC;
        dR[it] = (k < H && kk >= KSK) ? kq * H * sst + (kk - KSK) * 3 : -1;
        dS[it] = (k < H && kk < KSK) ? kq * H * ldw + kk * 3 : -1;
    }
    float wr[KR > 0 ? KR : 1];
    if (KR > 0) {
        for (int j = warp; j < H3; j += GR_THREADS / 32) {
            const int g = j / H, u = j - g * H;
            const float* src = a.Whh + (long)j * H + lane;
            float* dst = Ws + u * sst + g;
#pragma unroll
            for (int it = 0; it < KIT; ++it)
                if (dR[it] >= 0) gr_cp_async4(dst + dR[it], src + 32 * it);
        }
        gr_cp_async_wait_all();
        __syncthreads();
#pragma unroll
        for (int q = 0; q < KR; ++q) {
            const int kk = (KS + q) / 3;                   // weights of k >= H (padding of the last third) are zero
            wr[q] = (owner && ks * KC + kk < H) ? Ws[(long)vrow * sst + q] : 0.f;
        }
        __syncthreads();
    }
    if (3 * KC != H) {                                     // padding elements of the last third must read as zero
        for (int i = tid; i < H3 * ldw; i += GR_THREADS) Ws[i] = 0.f;
        __syncthreads();
    }
    for (int j = warp; j < H3; j += GR_THREADS / 32) {
        const int g = j / H, u = j - g * H;
        const float* src = a.Whh + (long)j * H + lane;
        float* dst = Ws + u * ldw + g;
#pragma unroll
        for (int it = 0; it < KIT; ++it)
            if (dS[it] >= 0) gr_cp_async4(dst + dS[it], src + 32 * it);
    }
    for (int i = tid; i < 2 * HP * GR_RB; i += GR_THREADS) {
        const int k = (i / GR_RB) % HP, r = i % GR_RB;
        hs[i] = (i < HP * GR_RB && k < H && r < nb) ? a.Hall[(long)(b0 + r) * H + k] : 0.f;
    }
    gr_cp_async_wait_all();
    __syncthreads();

    // gate items of this thread: (unit u, row r) = (i >> 2, i & 3) for i = tid, tid + 512
    constexpr int MAXI = 2;
    float bh[MAXI][3], gi_next[MAXI][3];
    bool live[MAXI];
#pragma unroll
    for (int q = 0; q < MAXI; ++q) {
        const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
        live[q] = (u < H) && (r < nb);
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            bh[q][g] = live[q] ? a.bhh[g * H + u] : 0.f;
            gi_next[q][g] = live[q] ? a.GI[((long)0 * B + b0 + r) * H3 + g * H + u] : 0.f;
        }
    }
    const float* wv = Ws + (long)(owner ? vrow : 0) * ldw;
    for (int t = 0; t < T; ++t) {
        const float* hc = hs + (t & 1) * HP * GR_RB;
        float* hn = hs + ((t + 1) & 1) * HP * GR_RB;
        float gi_cur[MAXI][3];
#pragma unroll
        for (int q = 0; q < MAXI; ++q) {
            const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
#pragma unroll
            for (int g = 0; g < 3; ++g) {
                gi_cur[q][g] = gi_next[q][g];
                if (live[q] && t + 1 < T) gi_next[q][g] = a.GI[((long)(t + 1) * B + b0 + r) * H3 + g * H + u];
            }
        }
        if (owner) {
            float ar[4] = {0.f, 0.f, 0.f, 0.f}, az[4] = {0.f, 0.f, 0.f, 0.f}, an[4] = {0.f, 0.f, 0.f, 0.f};
            const float* hk = hc + (long)ks * KC * GR_RB;
#pragma unroll 4
            for (int kk = 0; kk < KSK; ++kk) {
                const float w0 = wv[3 * kk], w1 = wv[3 * kk + 1], w2 = wv[3 * kk + 2];
                const float4 h4 = *reinterpret_cast<const float4*>(hk + kk * GR_RB);
                ar[0] = fmaf(w0, h4.x, ar[0]); ar[1] = fmaf(w0, h4.y, ar[1]); ar[2] = fmaf(w0, h4.z, ar[2]); ar[3] = fmaf(w0, h4.w, ar[3]);
                az[0] = fmaf(w1, h4.x, az[0]); az[1] = fmaf(w1, h4.y, az[1]); az[2] = fmaf(w1, h4.z, az[2]); az[3] = fmaf(w1, h4.w, az[3]);
                an[0] = fmaf(w2, h4.x, an[0]); an[1] = fmaf(w2, h4.y, an[1]); an[2] = fmaf(w2, h4.z, an[2]); an[3] = fmaf(w2, h4.w, an[3]);
            }
#pragma unroll
            for (int q = 0; q < KR / 3; ++q) {
                const float4 h4 = *reinterpret_cast<const float4*>(hk + (KSK + q) * GR_RB);
                const float w0 = wr[3 * q], w1 = wr[3 * q + 1], w2 = wr[3 * q + 2];
                ar[0] = fmaf(w0, h4.x, ar[0]); ar[1] = fmaf(w0, h4.y, ar[1]); ar[2] = fmaf(w0, h4.z, ar[2]); ar[3] = fmaf(w0, h4.w, ar[3]);
                az[0] = fmaf(w1, h4.x, az[0]); az[1] = fmaf(w1, h4.y, az[1]); az[2] = fmaf(w1, h4.z, az[2]); az[3] = fmaf(w1, h4.w, az[3]);
                an[0] = fmaf(w2, h4.x, an[0]); an[1] = fmaf(w2, h4.y, an[1]); an[2] = fmaf(w2, h4.z, an[2]); an[3] = fmaf(w2, h4.w, an[3]);
            }
            float* gp = gps + (long)ks * H3 * GR_RB;
            *reinterpret_cast<float4*>(gp + u_own * GR_RB) = make_float4(ar[0], ar[1], ar[2], ar[3]);
            *reinterpret_cast<float4*>(gp + (H + u_own) * GR_RB) = make_float4(az[0], az[1], az[2], az[3]);
            *reinterpret_cast<float4*>(gp + (2 * H + u_own) * GR_RB) = make_float4(an[0], an[1], an[2], an[3]);
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < MAXI; ++q) {
            const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
            if (u < H) {
                float hnew = 0.f;
                if (live[q]) {
                    const float* g0 = gps + u * GR_RB + r;
                    const float* g1 = g0 + (long)H3 * GR_RB;
                    const float* g2 = g1 + (long)H3 * GR_RB;
                    const int oz = H * GR_RB, on = 2 * H * GR_RB;
                    const float ghr = bh[q][0] + ((g0[0] + g1[0]) + g2[0]);
                    const float ghz = bh[q][1] + ((g0[oz] + g1[oz]) + g2[oz]);
                    const float ghn = bh[q][2] + ((g0[on] + g1[on]) + g2[on]);
                    const float rg = sigmoidf_acc(gi_cur[q][0] + ghr);
                    const float zg = sigmoidf_acc(gi_cur[q][1] + ghz);
                    const float ng = tanhf(gi_cur[q][2] + rg * ghn);
                    hnew = (1.f - zg) * ng + zg * hc[u * GR_RB + r];
                    const int gb = b0 + r;
                    const long o = ((long)t * B + gb) * H + u;
                    a.Hall[o + (long)B * H] = hnew;
                    if (a.Hbm) a.Hbm[((long)gb * T + t) * H + u] = hnew;
                    if (a.saved) {
                        a.saved[o] = rg; a.saved[TBH + o] = zg; a.saved[2 * TBH + o] = ng; a.saved[3 * TBH + o] = ghn;
                    }
                }
                hn[u * GR_RB + r] = hnew;
            }
        }
        __syncthreads();
    }
}

template <int KR>
__global__ void __launch_bounds__(GR_THREADS, 1) gru_res_bwd_kernel(const GruResArgs a) {
    extern __shared__ __align__(16) float gr_smem[];
    const int H = a.H, H3 = 3 * a.H, KS = a.KS, ldw = a.ldw, B = a.B, T = a.T;
    float* Ws = gr_smem;                                   // [3H][ldw]  thread (g, k): W[gH + jj][k], jj < KS
    float* dgs = Ws + (((long)H3 * ldw + 3) & ~3L);        // [3][H + KR][4]  dgh, gate-block major; tails zero
    float* dhz = dgs + 3 * (H + KR) * GR_RB;               // [H][4]   direct term dh_t * z
    float* part = dhz + H * GR_RB;                         // [3H][4]  partial dh per gate block
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * GR_RB, nb = min(GR_RB, B - b0);
    const long TBH = (long)T * B * H;
    const int g = tid / H, k = tid - g * H;                // (gate block, column) of this thread's weight vector

    // column k of gate block g: consecutive threads read consecutive addresses -- no staging needed
    float wr[KR > 0 ? KR : 1];
    if (tid < H3) {
        const float* src = a.Whh + (long)g * H * H + k;
        float* dst = Ws + (long)tid * ldw;
        for (int jj = 0; jj < KS; ++jj) gr_cp_async4(dst + jj, src + (long)jj * H);
#pragma unroll
        for (int q = 0; q < KR; ++q) wr[q] = (KS + q < H) ? src[(long)(KS + q) * H] : 0.f;
    } else {
#pragma unroll
        for (int q = 0; q < KR; ++q) wr[q] = 0.f;
    }
    for (int i = tid; i < 3 * (H + KR) * GR_RB + H * GR_RB + H3 * GR_RB; i += GR_THREADS) dgs[i] = 0.f;   // dgs, dhz, part
    gr_cp_async_wait_all();
    __syncthreads();

    constexpr int MAXI = 2;
    bool live[MAXI];
    float nx[MAXI][6];   // prefetched r, z, n, gh_n, h_prev, dHbm of the step about to be processed
#pragma unroll
    for (int q = 0; q < MAXI; ++q) {
        const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
        live[q] = (u < H) && (r < nb);
        if (live[q]) {
            const long o = ((long)(T - 1) * B + b0 + r) * H + u;
            nx[q][0] = a.saved[o]; nx[q][1] = a.saved[TBH + o]; nx[q][2] = a.saved[2 * TBH + o];
            nx[q][3] = a.saved[3 * TBH + o]; nx[q][4] = a.Hall[o];
            nx[q][5] = a.dHbm[((long)(b0 + r) * T + (T - 1)) * H + u];
        }
    }
    const float* wcol = Ws + (long)tid * ldw;
    const float* dg = dgs + (long)(g < 3 ? g : 0) * (H + KR) * GR_RB;
    for (int t = T - 1; t >= 0; --t) {
        // ---- gate gradients of (unit u, row r) ----
#pragma unroll
        for (int q = 0; q < MAXI; ++q) {
            const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
            if (u < H) {
                float dar = 0.f, daz = 0.f, danr = 0.f, keep = 0.f;
                if (live[q]) {
                    const float dht = dhz[i] + nx[q][5] + part[u * GR_RB + r] + part[(H + u) * GR_RB + r] +
                                      part[(2 * H + u) * GR_RB + r];
                    const float rg = nx[q][0], z = nx[q][1], n = nx[q][2], ghn = nx[q][3], hp = nx[q][4];
                    const float dn = dht * (1.f - z);
                    const float dz = dht * (hp - n);
                    const float dan = dn * (1.f - n * n);
                    dar = dan * ghn * rg * (1.f - rg);
                    daz = dz * z * (1.f - z);
                    danr = dan * rg;
                    keep = dht * z;
                    const int gb = b0 + r;
                    float* gi = a.dGI + ((long)t * B + gb) * H3;
                    float* gh = a.dGH + ((long)t * B + gb) * H3;
                    gi[u] = dar; gi[H + u] = daz; gi[2 * H + u] = dan;
                    gh[u] = dar; gh[H + u] = daz; gh[2 * H + u] = danr;
                    if (t > 0) {   // prefetch the next (earlier) step while the product below runs
                        const long o = ((long)(t - 1) * B + gb) * H + u;
                        nx[q][0] = a.saved[o]; nx[q][1] = a.saved[TBH + o]; nx[q][2] = a.saved[2 * TBH + o];
                        nx[q][3] = a.saved[3 * TBH + o]; nx[q][4] = a.Hall[o];
                        nx[q][5] = a.dHbm[((long)gb * T + (t - 1)) * H + u];
                    }
                }
                dhz[i] = keep;
                dgs[u * GR_RB + r] = dar;
                dgs[((H + KR) + u) * GR_RB + r] = daz;
                dgs[(2 * (H + KR) + u) * GR_RB + r] = danr;
            }
        }
        __syncthreads();
        // ---- part[g][k][row] = sum_jj dgh[row][gH + jj] * W[gH + jj][k] ----
        if (tid < H3) {
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
            for (int jj = 0; jj < KS; ++jj) {
                const float w = wcol[jj];
                const float4 d4 = *reinterpret_cast<const float4*>(dg + jj * GR_RB);
                a0 = fmaf(w, d4.x, a0); a1 = fmaf(w, d4.y, a1); a2 = fmaf(w, d4.z, a2); a3 = fmaf(w, d4.w, a3);
            }
#pragma unroll
            for (int q = 0; q < KR; ++q) {                 // (dgs entries beyond H are zero)
                const float4 d4 = *reinterpret_cast<const float4*>(dg + (KS + q) * GR_RB);
                a0 = fmaf(wr[q], d4.x, a0); a1 = fmaf(wr[q], d4.y, a1); a2 = fmaf(wr[q], d4.z, a2); a3 = fmaf(wr[q], d4.w, a3);
            }
            *reinterpret_cast<float4*>(part + tid * GR_RB) = make_float4(a0, a1, a2, a3);
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < MAXI; ++q) {
        const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
        if (live[q])
            a.dh0[(long)(b0 + r) * H + u] = dhz[i] + part[u * GR_RB + r] + part[(H + u) * GR_RB + r] + part[(2 * H + u) * GR_RB + r];
    }
}

// Backward, column-blocked (H >= ~100): warp jg owns the RJ = ceil(3H / 15) rows [jg RJ, (jg + 1) RJ) of W_hh, lane kc the C columns
// 5 kc .. 5 kc + C - 1 -- a private vector of RJ x C weights (row-major), the last 60 in registers.  Per row it reads C private
// weights and ONE broadcast float4 of dgh (4 batch rows) for 4 C FMAs (the one-column-per-thread kernel above does 4 FMAs per
// broadcast and is bound by those reads); the 15 row-group partials per (column, batch row) are summed by the next step's
// gate-gradient items.
constexpr int GB_KR = 60;
constexpr int GB_JG = 15;
template <int C>
__global__ void __launch_bounds__(GR_THREADS, 1) gru_res_bwdc_kernel(const GruResArgs a) {
    extern __shared__ __align__(16) float gr_smem[];
    const int H = a.H, H3 = 3 * a.H, KS = a.KS, ldw = a.ldw, B = a.B, T = a.T;
    const int RJ = (H3 + GB_JG - 1) / GB_JG;               // rows per warp
    const int LN = (H + C - 1) / C;                        // lanes in use
    const int KSR = KS / C, RR = GB_KR / C;                // rows of a vector in shared memory / in registers (KSR + RR = RJ)
    float* Ws = gr_smem;                                   // [15][LN][ldw]
    float* dgs = Ws + (((long)GB_JG * LN * ldw + 3) & ~3L);   // [15 RJ][4]  dgh (rows >= 3H zero)
    float* dhz = dgs + GB_JG * RJ * GR_RB;                 // [H][4]   direct term dh_t * z
    float* part = dhz + H * GR_RB;                         // [15][H][4]  partial dh per row group
    const int tid = threadIdx.x, lane = tid & 31, jg = tid >> 5;
    const int b0 = blockIdx.x * GR_RB, nb = min(GR_RB, B - b0);
    const long TBH = (long)T * B * H;
    const bool owner = jg < GB_JG && lane < LN;
    const int k0 = lane * C;

    float wr[GB_KR];
    {
        float* dst = Ws + (long)(jg * LN + lane) * ldw;
        if (owner) {
            for (int jl = 0; jl < KSR; ++jl) {
                const int j = jg * RJ + jl;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    if (j < H3 && k0 + c < H) gr_cp_async4(dst + jl * C + c, a.Whh + (long)j * H + k0 + c);
                    else dst[jl * C + c] = 0.f;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < GB_KR; ++q) {
            const int jl = KSR + q / C, c = q % C, j = jg * RJ + jl;
            wr[q] = (owner && jl < RJ && j < H3 && k0 + c < H) ? a.Whh[(long)j * H + k0 + c] : 0.f;
        }
    }
    for (int i = tid; i < GB_JG * RJ * GR_RB + H * GR_RB + GB_JG * H * GR_RB; i += GR_THREADS) dgs[i] = 0.f;   // dgs, dhz, part
    gr_cp_async_wait_all();
    __syncthreads();

    constexpr int MAXI = 2;
    bool live[MAXI];
    float nx[MAXI][6];   // prefetched r, z, n, gh_n, h_prev, dHbm of the step about to be processed
#pragma unroll
    for (int q = 0; q < MAXI; ++q) {
        const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
        live[q] = (u < H) && (r < nb);
        if (live[q]) {
            const long o = ((long)(T - 1) * B + b0 + r) * H + u;
            nx[q][0] = a.saved[o]; nx[q][1] = a.saved[TBH + o]; nx[q][2] = a.saved[2 * TBH + o];
            nx[q][3] = a.saved[3 * TBH + o]; nx[q][4] = a.Hall[o];
            nx[q][5] = a.dHbm[((long)(b0 + r) * T + (T - 1)) * H + u];
        }
    }
    const float* wv = Ws + (long)(owner ? jg * LN + lane : 0) * ldw;
    const float* dg = dgs + (long)(jg < GB_JG ? jg : 0) * RJ * GR_RB;
    for (int t = T - 1; t >= 0; --t) {
        // ---- gate gradients of (unit u, row r) ----
#pragma unroll
        for (int q = 0; q < MAXI; ++q) {
            const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
            if (u < H) {
                float dar = 0.f, daz = 0.f, danr = 0.f, keep = 0.f;
                if (live[q]) {
                    float ps = 0.f;
#pragma unroll
                    for (int w = 0; w < GB_JG; ++w) ps += part[(w * H + u) * GR_RB + r];
                    const float dht = dhz[i] + nx[q][5] + ps;
                    const float rg = nx[q][0], z = nx[q][1], n = nx[q][2], ghn = nx[q][3], hp = nx[q][4];
                    const float dn = dht * (1.f - z);
                    const float dz = dht * (hp - n);
                    const float dan = dn * (1.f - n * n);
                    dar = dan * ghn * rg * (1.f - rg);
                    daz = dz * z * (1.f - z);
                    danr = dan * rg;
                    keep = dht * z;
                    const int gb = b0 + r;
                    float* gi = a.dGI + ((long)t * B + gb) * H3;
                    float* gh = a.dGH + ((long)t * B + gb) * H3;
                    gi[u] = dar; gi[H + u] = daz; gi[2 * H + u] = dan;
                    gh[u] = dar; gh[H + u] = daz; gh[2 * H + u] = danr;
                    if (t > 0) {   // prefetch the next (earlier) step while the product below runs
                        const long o = ((long)(t - 1) * B + gb) * H + u;
                        nx[q][0] = a.saved[o]; nx[q][1] = a.saved[TBH + o]; nx[q][2] = a.saved[2 * TBH + o];
                        nx[q][3] = a.saved[3 * TBH + o]; nx[q][4] = a.Hall[o];
                        nx[q][5] = a.dHbm[((long)gb * T + (t - 1)) * H + u];
                    }
                }
                dhz[i] = keep;
                dgs[u * GR_RB + r] = dar;
                dgs[(H + u) * GR_RB + r] = daz;
                dgs[(2 * H + u) * GR_RB + r] = danr;
            }
        }
        __syncthreads();
        // ---- part[jg][k][row] = sum over this warp's rows j of dgh[row][j] * W[j][k] ----
        if (owner) {
            float acc[C][4];
#pragma unroll
            for (int c = 0; c < C; ++c) { acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0.f; }
#pragma unroll 2
            for (int jl = 0; jl < KSR; ++jl) {
                const float4 d4 = *reinterpret_cast<const float4*>(dg + jl * GR_RB);
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float w = wv[jl * C + c];
                    acc[c][0] = fmaf(w, d4.x, acc[c][0]); acc[c][1] = fmaf(w, d4.y, acc[c][1]);
                    acc[c][2] = fmaf(w, d4.z, acc[c][2]); acc[c][3] = fmaf(w, d4.w, acc[c][3]);
                }
            }
#pragma unroll
            for (int q = 0; q < GB_KR / C; ++q) {
                if (KSR + q < RJ) {
                    const float4 d4 = *reinterpret_cast<const float4*>(dg + (KSR + q) * GR_RB);
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const float w = wr[q * C + c];
                        acc[c][0] = fmaf(w, d4.x, acc[c][0]); acc[c][1] = fmaf(w, d4.y, acc[c][1]);
                        acc[c][2] = fmaf(w, d4.z, acc[c][2]); acc[c][3] = fmaf(w, d4.w, acc[c][3]);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c)
                if (k0 + c < H)
                    *reinterpret_cast<float4*>(part + ((long)jg * H + k0 + c) * GR_RB) =
                        make_float4(acc[c][0], acc[c][1], acc[c][2], acc[c][3]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < MAXI; ++q) {
        const int i = tid + q * GR_THREADS, u = i >> 2, r = i & 3;
        if (live[q]) {
            float ps = 0.f;
#pragma unroll
            for (int w = 0; w < GB_JG; ++w) ps += part[(w * H + u) * GR_RB + r];
            a.dh0[(long)(b0 + r) * H + u] = dhz[i] + ps;
        }
    }
}

// plan of the column-blocked backward: C columns per lane, 60 register weights; 0 when it does not apply
static int gr_plan_bwdc(int H, int* C, int* KS, int* ldw, size_t* smem) {
    if (H <= 0 || 3 * H > GR_THREADS) return 0;
    const int c = (H + 31) / 32;                           // columns per lane
    if (c < 1 || c > 5 || GB_KR % c) return 0;
    const int RJ = (3 * H + GB_JG - 1) / GB_JG, LN = (H + c - 1) / c, VL = RJ * c;
    const int ks = VL - GB_KR;
    if (ks < 0 || (ks % c)) return 0;
    const int l = ks | 1;
    const size_t w = (((size_t)GB_JG * LN * l + 3) & ~(size_t)3);
    const size_t tot = (w + (size_t)GB_JG * RJ * GR_RB + (size_t)H * GR_RB + (size_t)GB_JG * H * GR_RB) * sizeof(float);
    if (tot > 226 * 1024) return 0;
    *C = c; *KS = ks; *ldw = l; *smem = tot;
    return 1;
}

// Registers per private weight vector: the largest multiple of 12 (<= 60, no spills at 512 threads) with which the rest fits
// in shared memory.
//   forward : 3H vectors of 3 ceil(H/3) weights (+ 2 x padded state + 3 x partial gh)
//   backward: 3H vectors of H weights (+ dgh, direct term, partial dh)
static int gr_plan(int H, bool bwd, int* KR, int* ldw, size_t* smem) {
    if (H <= 0 || H > 192 || 3 * H > GR_THREADS || ((H + 31) / 32) * 3 * 32 > GR_THREADS) return 0;
    const int KC = (H + 2) / 3, VL = bwd ? H : 3 * KC;
    for (int kr = 60; kr >= 0; kr -= 12) {      // as many weights in registers as the 128-register budget allows
        const int ks = VL - kr;
        if (ks <= 0 || kr > ks) continue;       // (the register part is staged through the smem rows: KR <= KS)
        const int l = ks | 1;
        const size_t w = (((size_t)3 * H * l + 3) & ~(size_t)3);
        const size_t extra = bwd ? 3 * (size_t)(H + kr) * GR_RB + (size_t)H * GR_RB + (size_t)3 * H * GR_RB
                                 : 2 * (size_t)3 * KC * GR_RB + 3 * (size_t)3 * H * GR_RB;
        const size_t tot = (w + extra) * sizeof(float);
        if (tot <= 226 * 1024) {
            *KR = kr; *ldw = l; *smem = tot;
            return 1;
        }
    }
    return 0;
}

template <int KR>
static int gr_launch(bool bwd, const GruResArgs& a, size_t smem, cudaStream_t st) {
    const unsigned grid = (unsigned)ceil_div(a.B, GR_RB);
    if (bwd) {
        CAPHN_CHECK(cudaFuncSetAttribute(gru_res_bwd_kernel<KR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gru_res_bwd_kernel<KR><<<grid, GR_THREADS, smem, st>>>(a);
    } else {
        CAPHN_CHECK(cudaFuncSetAttribute(gru_res_fwd_kernel<KR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gru_res_fwd_kernel<KR><<<grid, GR_THREADS, smem, st>>>(a);
    }
    CAPHN_RETURN_LAST();
}

template <int C>
static int gr_launch_bwdc(const GruResArgs& a, size_t smem, cudaStream_t st) {
    CAPHN_CHECK(cudaFuncSetAttribute(gru_res_bwdc_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gru_res_bwdc_kernel<C><<<(unsigned)ceil_div(a.B, GR_RB), GR_THREADS, smem, st>>>(a);
    CAPHN_RETURN_LAST();
}

static int gr_dispatch(bool bwd, GruResArgs& a, cudaStream_t st) {
    int KR = 0, ldw = 0;
    size_t smem = 0;
    if (bwd) {
        int C = 0, KS = 0;
        if (gr_plan_bwdc(a.H, &C, &KS, &ldw, &smem)) {
            a.KS = KS; a.ldw = ldw;
            switch (C) {
                case 1: return gr_launch_bwdc<1>(a, smem, st);
                case 2: return gr_launch_bwdc<2>(a, smem, st);
                case 3: return gr_launch_bwdc<3>(a, smem, st);
                case 4: return gr_launch_bwdc<4>(a, smem, st);
                default: return gr_launch_bwdc<5>(a, smem, st);
            }
        }
    }
    if (!gr_plan(a.H, bwd, &KR, &ldw, &smem)) return CAPHN_EINVAL;
    a.KS = (bwd ? a.H : 3 * ((a.H + 2) / 3)) - KR; a.ldw = ldw;
    switch (KR) {
        case 0: return gr_launch<0>(bwd, a, smem, st);
        case 12: return gr_launch<12>(bwd, a, smem, st);
        case 24: return gr_launch<24>(bwd, a, smem, st);
        case 36: return gr_launch<36>(bwd, a, smem, st);
        case 48: return gr_launch<48>(bwd, a, smem, st);
        default: return gr_launch<60>(bwd, a, smem, st);
    }
}

}  // namespace caphn

using namespace caphn;

extern "C" {

// *ok = 1 when the CTA-resident GRU kernels apply to hidden size H (3H <= 512 threads and W_hh fits in one CTA's shared
// memory + registers), else 0.
int caphn_gru_resident_plan(int H, int* ok) {
    if (!ok) return CAPHN_EINVAL;
    int KR, ldw;
    size_t sm;
    *ok = gr_plan(H, false, &KR, &ldw, &sm) && gr_plan(H, true, &KR, &ldw, &sm);
    return CAPHN_OK;
}

// Single-layer GRU recurrence over T steps with W_hh resident in one CTA (see the header comment).  Same arguments and
// outputs as caphn_gru_cluster_fwd: GI [T,B,3H], Whh [3H,H], bhh [3H], Hall [T+1,B,H] with Hall[0] = h0 on entry, Hbm
// [B,T,H] (may be NULL), saved [4][T,B,H] (may be NULL).
int caphn_gru_resident_fwd(const float* GI, const float* Whh, const float* bhh, float* Hall, float* Hbm, float* saved, int B,
                           int T, int H, void* stream) {
    if (B <= 0 || T <= 0 || !GI || !Whh || !bhh || !Hall) return CAPHN_EINVAL;
    GruResArgs a{};
    a.GI = GI; a.Whh = Whh; a.bhh = bhh; a.Hall = Hall; a.Hbm = Hbm; a.saved = saved; a.B = B; a.T = T; a.H = H;
    return gr_dispatch(false, a, (cudaStream_t)stream);
}

// BPTT of caphn_gru_resident_fwd: dHbm [B,T,H] -> dGI, dGH [T,B,3H], dh0 [B,H]  (same contract as caphn_gru_cluster_bwd).
int caphn_gru_resident_bwd(const float* dHbm, const float* saved, const float* Hall, const float* Whh, float* dGI,
                           float* dGH, float* dh0, int B, int T, int H, void* stream) {
    if (B <= 0 || T <= 0 || !dHbm || !saved || !Hall || !Whh || !dGI || !dGH || !dh0) return CAPHN_EINVAL;
    GruResArgs a{};
    a.dHbm = dHbm; a.saved = const_cast<float*>(saved); a.Hall = const_cast<float*>(Hall); a.Whh = Whh; a.dGI = dGI;
    a.dGH = dGH; a.dh0 = dh0; a.B = B; a.T = T; a.H = H;
    return gr_dispatch(true, a, (cudaStream_t)stream);
}

}  // extern "C"
