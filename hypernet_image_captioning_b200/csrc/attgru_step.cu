// Attention-GRU recurrence, forward, as THREE batch-wide kernels per time step ("step-split" path), chained with
// programmatic dependent launch so that each kernel's loop-invariant prefetch overlaps its predecessor.
//
// Same arithmetic as attgru_seq.cu (reference models/decoderlstm.py:97-100 + models/attention.py:33-45), different
// decomposition.  The persistent kernel of attgru_seq.cu keeps 4 rows per CTA for all steps and therefore re-streams the
// whole generated W_hh / W_ih[:, E:] / U_a (1.1 MB) per CTA per step from L2 -- 143 MB per step at B = 512 -- in
// dependent phases that each expose an L2 round trip.  Here every step is
//
//   U  attstep_u_kernel      u = U_a h_{t-1} + b_u for all rows on the warp tensor cores (mma.sync m16n8k16, bf16 hi/lo
//                            split, fp32 accumulate -- see mma_common.cuh).
//   A  attstep_attn_kernel   one CTA per batch row: K_b and f_b (2 x 39 KB) are pulled into shared memory by two bulk TMA
//                            copies issued BEFORE the grid dependency is awaited, so they fly while U runs; then
//                            scores -> softmax over P -> ctx from shared memory.
//   Y  attstep_gates_kernel  CTA = (16 hidden units) x (32 batch rows): gi_ctx = ctx W_ih[:,E:]^T and gh = h W_hh^T on
//                            the warp tensor cores, r/z/n gates and h' in the epilogue.  The weight fragments
//                            (register-resident, 26 x 16 B per lane) are requested before the dependency wait.
//
// Weights come from a fragment-ordered bf16 hi/lo pack built once per generated theta (caphn_attstep_pack): they are
// read once per 16/32 rows instead of once per 4.  The activations move between the kernels as bf16 hi/lo rows
// (workspace), written by the producer's epilogue and fetched with 16-byte cp.async.
#include "step_common.cuh"

namespace caphn {

// ------------------------------------------------------------------------------------------------------------------
// weight pack:  A fragments of mma.m16n8k16 for tile m = (src, gate, unit tile), k-tile kt, as uint4 {a0,a1,a2,a3} per lane
//   out[((m * NKT + kt) * 2 + hl) * 32 + lane],   src 0: W_ih[:, E:E+F] (input ctx), src 1: W_hh (input h); after the
//   6 * NUT gate tiles come NUT tiles of U_a (input h)
// ------------------------------------------------------------------------------------------------------------------
// blockIdx.y = style group g: the generated W_ih / W_hh of group g start gstride floats after those of group g - 1 (rows
// of Theta [G, theta]); U_a is shared.  Pack g starts pstride uint4 after pack g - 1.
__global__ void attstep_pack_kernel(const float* __restrict__ Wih, const float* __restrict__ Whh,
                                    const float* __restrict__ Ua, int E, int F, int H, int NUT, int NKT,
                                    uint4* __restrict__ out, long gstride, long pstride) {
    const long total = (long)7 * NUT * NKT * 32;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    Wih += (long)blockIdx.y * gstride;
    Whh += (long)blockIdx.y * gstride;
    out += (long)blockIdx.y * pstride;
    const int lane = (int)(idx & 31);
    long r = idx >> 5;
    const int kt = (int)(r % NKT);
    r /= NKT;
    const int ut = (int)(r % NUT);
    const int grp = (int)(r / NUT);                  // 0..2: W_ih[:,E:] r,z,n   3..5: W_hh r,z,n   6: U_a
    const int K = grp < 3 ? F : H;
    const int ja = ut * 16 + (lane >> 2), jb = ja + 8;
    const int k0 = kt * 16 + (lane & 3) * 2;
    auto w = [&](int j, int k) -> float {
        if (j >= H || k >= K) return 0.f;
        if (grp < 3) return Wih[((long)grp * H + j) * (E + F) + E + k];
        if (grp < 6) return Whh[((long)(grp - 3) * H + j) * H + k];
        return Ua[(long)j * H + k];
    };
    uint4 hi, lo;
    split2(w(ja, k0), w(ja, k0 + 1), hi.x, lo.x);
    split2(w(jb, k0), w(jb, k0 + 1), hi.y, lo.y);
    split2(w(ja, k0 + 8), w(ja, k0 + 9), hi.z, lo.z);
    split2(w(jb, k0 + 8), w(jb, k0 + 9), hi.w, lo.w);
    const long m = (long)grp * NUT + ut;
    out[((m * NKT + kt) * 2 + 0) * 32 + lane] = hi;
    out[((m * NKT + kt) * 2 + 1) * 32 + lane] = lo;
}

#ifdef CAPHN_ATTCL_TIMING
__device__ long long g_attst_ts[32];
#define XTS(i) do { if (blockIdx.x == 1 && blockIdx.y == 0 && threadIdx.x == 0) g_attst_ts[i] = clock64(); } while (0)
#else
#define XTS(i)
#endif


// Workspace layout (bf16 unless noted), KP = padded operand row length:
//   u    [B][H] fp32 | csp [2][B][KP] ctx hi, lo | hsp [2 buffers][2][B][KP] h hi, lo (buffer t & 1 holds h_{t-1})
struct StepWork {
    float* u;
    __nv_bfloat16* csp;
    __nv_bfloat16* hsp;
};

// fp32 rows -> bf16 hi/lo operand rows (h of the first step), and zero the padding columns of the other h buffer
__global__ void attstep_split_kernel(const float* __restrict__ h, int B, int H, int KP, __nv_bfloat16* __restrict__ dst,
                                     __nv_bfloat16* __restrict__ other) {
    const int KP2 = KP >> 1;
    const long plane = (long)B * KP;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < (long)B * KP2; i += (long)gridDim.x * blockDim.x) {
        const long b = i / KP2;
        const int k = (int)(i - b * KP2) * 2;
        uint32_t hi, lo;
        split2(k < H ? h[b * H + k] : 0.f, k + 1 < H ? h[b * H + k + 1] : 0.f, hi, lo);
        *reinterpret_cast<uint32_t*>(dst + b * KP + k) = hi;
        *reinterpret_cast<uint32_t*>(dst + plane + b * KP + k) = lo;
        if (k + 1 >= H) {     // pair touches the padding: keep it finite (zero) in the buffer the gates kernel fills
            if (k >= H) {
                *reinterpret_cast<uint32_t*>(other + b * KP + k) = 0u;
                *reinterpret_cast<uint32_t*>(other + plane + b * KP + k) = 0u;
            } else {
                other[b * KP + k + 1] = __float2bfloat16_rn(0.f);
                other[plane + b * KP + k + 1] = __float2bfloat16_rn(0.f);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// U: u = U_a h_{t-1} + b_u          CTA = 2 unit tiles (2 warps) x 16 batch rows
// ------------------------------------------------------------------------------------------------------------------
constexpr int US_NB = 16, US_NT = US_NB / 8, US_WARPS = 2, US_THREADS = US_WARPS * 32;

struct AttStepU {
    const uint4* Wp;            // pack; U_a tiles start at tile 6 * NUT
    const float* bu;
    const __nv_bfloat16* hsp;   // [2][B][KP] h_{t-1} hi, lo
    float* u;                   // [B,H]
    int B, H, NUT, NKT, KP;
};

__global__ void __launch_bounds__(US_THREADS) attstep_u_kernel(const AttStepU a) {
    extern __shared__ __align__(16) uint8_t usm[];
    __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(usm);   // [2][NB][KP]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(act + 2 * US_NB * a.KP);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ut = blockIdx.x * US_WARPS + warp, r0 = blockIdx.y * US_NB;
    if (tid == 0) st_mbar_init(mbar, 1);
    const int B = a.B, H = a.H, KP = a.KP, NKT = a.NKT;
    const bool has_tile = ut < a.NUT;
    uint4 ah[ST_MAXKT], al[ST_MAXKT];
    {
        const uint4* wp = a.Wp + (((long)6 * a.NUT + (has_tile ? ut : 0)) * NKT) * 64 + lane;
#pragma unroll
        for (int kt = 0; kt < ST_MAXKT; ++kt)
            if (kt < NKT) { ah[kt] = st_ldg_u4(wp + (long)kt * 64); al[kt] = st_ldg_u4(wp + (long)kt * 64 + 32); }
    }
    const int ja = ut * 16 + (lane >> 2);
    const float bua = (has_tile && ja < H) ? a.bu[ja] : 0.f, bub = (has_tile && ja + 8 < H) ? a.bu[ja + 8] : 0.f;
    pdl_launch_dependents();
    pdl_wait();                                   // h_{t-1} rows come from the previous step's gates kernel
    stage_rows_bulk<US_NB, US_THREADS>(a.hsp, (long)B * KP, r0, min(US_NB, B - r0), KP, 2, act, mbar, tid);
    __syncthreads();                              // zero-filled tail rows + the barrier initialisation are visible
    st_mbar_wait(mbar, 0);
    if (!has_tile) return;
    float acc[US_NT][4];
#pragma unroll
    for (int nt = 0; nt < US_NT; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
    warp_mma_rows<US_NT>(ah, al, NKT, act, act + US_NB * KP, KP, lane, acc);
#pragma unroll
    for (int nt = 0; nt < US_NT; ++nt) {
        const int b = r0 + nt * 8 + (lane & 3) * 2;
        if (ja < H) {
            if (b < B) a.u[(long)b * H + ja] = acc[nt][0] + bua;
            if (b + 1 < B) a.u[(long)(b + 1) * H + ja] = acc[nt][1] + bua;
        }
        if (ja + 8 < H) {
            if (b < B) a.u[(long)b * H + ja + 8] = acc[nt][2] + bub;
            if (b + 1 < B) a.u[(long)(b + 1) * H + ja + 8] = acc[nt][3] + bub;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// A: attention for step t.  Persistent over the batch: CTA c handles rows c, c + grid, c + 2 grid, ...; the K_b / f_b
//    tiles are double-buffered in shared memory (2 x 78 KB) and fetched by bulk TMA copies, the first two before the
//    grid dependency is awaited (they fly while U runs), the next ones while the previous row is being processed.
// ------------------------------------------------------------------------------------------------------------------
constexpr int AS_THREADS = 512, AS_WARPS = AS_THREADS / 32;
constexpr int AS_PSPL = AS_THREADS / 128;     // position groups of the context phase (needs KP / 2 <= 128)
constexpr int AS_SMAX = 4;                    // softmax elements per lane: P <= 128

struct AttStepA {
    const float* Kp;     // [B,P,H]
    const float* f;      // [B,P,F]
    const float* va; const float* bv;
    const float* u;      // [B,H]   u of step t
    float* attn;         // [B,T,P]
    float* ctx;          // row b of step t at ctx + b*ldctx
    long ldctx;
    __nv_bfloat16* csp;  // [2][B][KP] ctx hi, lo
    int B, T, t, P, H, F, KP, RPC;   // RPC = rows per CTA = ceil(B / grid)
    int NBUF;                        // tile buffers per CTA: 1 (two co-resident CTAs per SM overlap each other) or 2
};

__global__ void __launch_bounds__(AS_THREADS, 2) attstep_attn_kernel(const AttStepA a) {
    extern __shared__ __align__(16) float asmem[];
    const int H = a.H, F = a.F, P = a.P, KP = a.KP, B = a.B;
    const int PS = (P + 3) & ~3, H4 = (H + 3) & ~3;
    const int tile = P * H + P * F;                      // floats per buffer: K_b then f_b
    float* bufs = asmem;                                 // [2][tile]
    const int NBUF = a.NBUF;
    float* us = bufs + NBUF * tile;                      // [RPC][H4]
    float* vs = us + a.RPC * H4;                         // [H4]
    float* sc = vs + H4;                                 // [PS]
    float* cpart = sc + PS;                              // [PSPL][KP]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(cpart + AS_PSPL * KP + (KP & 1));   // [2]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nrows = (B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // rows of this CTA
    const uint32_t kb = (uint32_t)P * H * 4, fb = (uint32_t)P * F * 4;
    XTS(0);
    if (tid == 0) {
        st_mbar_init(&mbar[0], 1);
        st_mbar_init(&mbar[1], 1);
        for (int i = 0; i < NBUF && i < nrows; ++i) {
            const long b = blockIdx.x + (long)i * gridDim.x;
            st_mbar_expect_tx(&mbar[i], kb + fb);
            st_bulk_g2s(bufs + i * tile, a.Kp + b * P * H, kb, &mbar[i]);
            st_bulk_g2s(bufs + i * tile + P * H, a.f + b * P * F, fb, &mbar[i]);
        }
    }
    for (int j = tid; j < H; j += AS_THREADS) vs[j] = a.va[j];
    const float bv = a.bv[0];
    pdl_launch_dependents();
    pdl_wait();                                          // u comes from the U kernel of this step
    XTS(1);
    for (int i = tid; i < nrows * H; i += AS_THREADS) {
        const int r = i / H, j = i - r * H;
        us[r * H4 + j] = ldg_stream1(a.u + (blockIdx.x + (long)r * gridDim.x) * H + j);
    }
    __syncthreads();
    XTS(2);
    const long plane = (long)B * KP;
    for (int i = 0; i < nrows; ++i) {
        const long b = blockIdx.x + (long)i * gridDim.x;
        const int bi = NBUF == 2 ? (i & 1) : 0, ph = NBUF == 2 ? ((i >> 1) & 1) : (i & 1);
        const float* Ks = bufs + bi * tile;
        const float* fs = Ks + P * H;
        const float* ur = us + i * H4;
        st_mbar_wait(&mbar[bi], ph);
        if (i == 0) XTS(3);
        // scores: one warp per group of 4 positions; v_a and u are reused across the 4 positions
        {
            const int PG = (P + 3) >> 2;
            for (int task = warp; task < PG; task += AS_WARPS) {
                const int p0 = task * 4;
                const int np = min(4, P - p0);
                const float* kp = Ks + (long)p0 * H;
                float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
                for (int j = lane; j < H; j += 32) {
                    const float vj = vs[j], uj = ur[j];
                    float kv[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) kv[q] = kp[(q < np ? q : 0) * H + j];
#pragma unroll
                    for (int q = 0; q < 4; ++q) s4[q] = fmaf(vj, tanh_fast(kv[q] + uj), s4[q]);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float s = warp_sum(s4[q]);
                    if (lane == 0 && q < np) sc[p0 + q] = s + bv;
                }
            }
        }
        __syncthreads();
        if (i == 0) XTS(4);
        if (warp == 0) {       // softmax over P positions, AS_SMAX elements per lane held in registers
            float x[AS_SMAX];
            float mx = -INFINITY;
#pragma unroll
            for (int e = 0; e < AS_SMAX; ++e) {
                const int p = lane + 32 * e;
                x[e] = p < P ? sc[p] : -INFINITY;
                mx = fmaxf(mx, x[e]);
            }
            mx = warp_max(mx);
            float sum = 0.f;
#pragma unroll
            for (int e = 0; e < AS_SMAX; ++e) { x[e] = expf(x[e] - mx); sum += x[e]; }   // exp(-inf) = 0 for the padding
            const float inv = 1.f / warp_sum(sum);
#pragma unroll
            for (int e = 0; e < AS_SMAX; ++e) {
                const int p = lane + 32 * e;
                if (p < P) {
                    const float al = x[e] * inv;
                    sc[p] = al;
                    a.attn[(b * a.T + a.t) * P + p] = al;
                }
            }
        }
        __syncthreads();
        if (i == 0) XTS(5);
        // context from shared memory: thread = (feature pair, position group); partials reduced through smem
        {
            const int q = tid & 127, ps = tid >> 7;
            const int k = q * 2;
            if (k < KP) {
                const int pchunk = (P + AS_PSPL - 1) / AS_PSPL;
                const int pa = ps * pchunk, pb = min(P, pa + pchunk);
                float c0 = 0.f, c1 = 0.f;
                if (k + 1 < F) {
                    float d0 = 0.f, d1 = 0.f;
                    int p = pa;
#pragma unroll 4
                    for (; p + 1 < pb; p += 2) {
                        const float w0 = sc[p], w1 = sc[p + 1];
                        c0 = fmaf(w0, fs[p * F + k], c0);
                        c1 = fmaf(w0, fs[p * F + k + 1], c1);
                        d0 = fmaf(w1, fs[(p + 1) * F + k], d0);
                        d1 = fmaf(w1, fs[(p + 1) * F + k + 1], d1);
                    }
                    if (p < pb) { c0 = fmaf(sc[p], fs[p * F + k], c0); c1 = fmaf(sc[p], fs[p * F + k + 1], c1); }
                    c0 += d0; c1 += d1;
                } else if (k < F) {
                    for (int p = pa; p < pb; ++p) c0 = fmaf(sc[p], fs[p * F + k], c0);
                }
                cpart[ps * KP + k] = c0;
                cpart[ps * KP + k + 1] = c1;
            }
        }
        __syncthreads();
        // both tiles of this buffer are dead now: fetch the row after next into it
        if (tid == 0 && i + NBUF < nrows) {
            const long bn = blockIdx.x + (long)(i + NBUF) * gridDim.x;
            float* dst = bufs + bi * tile;
            st_mbar_expect_tx(&mbar[bi], kb + fb);
            st_bulk_g2s(dst, a.Kp + bn * P * H, kb, &mbar[bi]);
            st_bulk_g2s(dst + P * H, a.f + bn * P * F, fb, &mbar[bi]);
        }
        if (tid < 128 && tid * 2 < KP) {
            const int k = tid * 2;
            float c0 = 0.f, c1 = 0.f;
#pragma unroll
            for (int ps = 0; ps < AS_PSPL; ++ps) { c0 += cpart[ps * KP + k]; c1 += cpart[ps * KP + k + 1]; }
            float* cp = a.ctx + b * a.ldctx;
            if (k < F) cp[k] = c0;
            if (k + 1 < F) cp[k + 1] = c1;
            uint32_t hi, lo;
            split2(c0, c1, hi, lo);
            *reinterpret_cast<uint32_t*>(a.csp + b * KP + k) = hi;
            *reinterpret_cast<uint32_t*>(a.csp + plane + b * KP + k) = lo;
        }
        if (i == 0) XTS(6);
        // (sc / cpart are rewritten only after the next row's first __syncthreads)
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Y: gi_ctx, gh on the warp tensor cores + gates for step t     CTA = 16 units (6 gate tiles, one warp each) x 64 rows
// ------------------------------------------------------------------------------------------------------------------
constexpr int YS_NB = 64;                 // batch rows per CTA (8 n-tiles of 8): the weight tiles are read once per 64 rows
constexpr int YS_NB_SMALL = 8;            // many-style batches with <= 8 rows per group: one n-tile, 14 KB of operand rows, many CTAs per SM
constexpr int YS_WARPS = 6;               // one warp per (source, gate) m-tile of 16 hidden units
constexpr int YS_THREADS = YS_WARPS * 32;

struct AttStepY {
    const __nv_bfloat16* csp;   // [2][B][KP] ctx hi, lo        (written by A of this step)
    const __nv_bfloat16* hsp;   // [2][B][KP] h_{t-1} hi, lo
    __nv_bfloat16* hsp_next;    // [2][B][KP] h_t hi, lo        (the other buffer)
    const float* hprev;  // [B,H]
    const float* GIw;    // [B,3H] of step t
    const uint4* Wp;     // fragment pack
    const float* bhh;    // [3H]
    float* hnext;        // [B,H]
    float* Hbm;          // [B,T,H] or null
    float* R; float* Z; float* Nn; float* GHN;   // [B,H] of step t, or null
    int B, T, t, H, NUT, NKT, KP;
    // many-style batch (rows sorted by style group): tile blockIdx.y covers rows [tiles[y].x, +tiles[y].y) of group
    // tiles[y].z, whose weight pack / b_hh start pstride uint4 / 3H floats after the previous group's.  null: one group.
    const int4* tiles;
    long pstride;
};

template <int YS_NB>
__global__ void __launch_bounds__(YS_THREADS, YS_NB >= 64 ? 1 : 4) attstep_gates_kernel(const AttStepY a) {
    constexpr int YS_NT = YS_NB / 8;
    constexpr int YS_RP = YS_NB + 1;          // pitch of the result exchange array
    extern __shared__ __align__(16) uint8_t ysm[];
    const int H = a.H, B = a.B, KP = a.KP, NKT = a.NKT, H3 = 3 * a.H;
    __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(ysm);   // [4][NB][KP]: ctx hi | ctx lo | h hi | h lo
    float* res = reinterpret_cast<float*>(act + 4 * YS_NB * KP);  // [6][16][RP]
    float* gis = res + 6 * 16 * YS_RP;                            // [NB][3][16]  GIw tile (word half of the input projection)
    float* hps = gis + YS_NB * 48;                                // [NB][16]     h_{t-1} tile, fp32
    float* bhs = hps + YS_NB * 16;                                // [3][16]      b_hh tile
    uint64_t* mbar = reinterpret_cast<uint64_t*>(bhs + 48);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ut = blockIdx.x;
    int r0 = blockIdx.y * YS_NB, rows_valid = min(YS_NB, B - r0), grp = 0;
    if (a.tiles) { const int4 tl = a.tiles[blockIdx.y]; r0 = tl.x; rows_valid = tl.y; grp = tl.z; }
    if (tid == 0) st_mbar_init(mbar, 1);
    if (tid < 48) {
        const int j = ut * 16 + (tid & 15);
        bhs[tid] = j < H ? a.bhh[(long)grp * H3 + (tid >> 4) * H + j] : 0.f;
    }
    const int src = warp / 3;                         // warp tile: gate (warp % 3) of W_ih[:,E:] (src 0) / W_hh (src 1)
    XTS(16);
    // loop-invariant inputs first (they do not depend on the previous kernels): weight fragments, GIw tile
    uint4 ah[ST_MAXKT], al[ST_MAXKT];
    {
        const uint4* wp = a.Wp + (long)grp * a.pstride + (((long)warp * a.NUT + ut) * NKT) * 64 + lane;
#pragma unroll
        for (int kt = 0; kt < ST_MAXKT; ++kt)
            if (kt < NKT) { ah[kt] = st_ldg_u4(wp + (long)kt * 64); al[kt] = st_ldg_u4(wp + (long)kt * 64 + 32); }
    }
    for (int i = tid; i < YS_NB * 12; i += YS_THREADS) {          // (row, gate, 4-unit chunk): H % 4 == 0
        const int row = i / 12, r = i - row * 12, e = r >> 2, c = r & 3;
        float* d = gis + row * 48 + e * 16 + c * 4;
        const int j = ut * 16 + c * 4;
        if (row < rows_valid && j < H) st_cp_async16(d, a.GIw + (long)(r0 + row) * H3 + e * H + j);
        else *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    pdl_launch_dependents();
    pdl_wait();                                       // ctx rows: A of this step; h rows: gates kernel of the previous step
    XTS(17);
    if (tid == 0) {       // one barrier, four bulk copies: ctx hi, ctx lo, h hi, h lo (rows of a plane are contiguous)
        const uint32_t bytes = (uint32_t)rows_valid * KP * 2;
        const long plane = (long)B * KP;
        st_mbar_expect_tx(mbar, 4 * bytes);
        st_bulk_g2s(act, a.csp + (long)r0 * KP, bytes, mbar);
        st_bulk_g2s(act + YS_NB * KP, a.csp + plane + (long)r0 * KP, bytes, mbar);
        st_bulk_g2s(act + 2 * YS_NB * KP, a.hsp + (long)r0 * KP, bytes, mbar);
        st_bulk_g2s(act + 3 * YS_NB * KP, a.hsp + plane + (long)r0 * KP, bytes, mbar);
    }
    if (rows_valid < YS_NB) {
        const int CPR = KP >> 3, nz = (YS_NB - rows_valid) * CPR;
        for (int i = tid; i < 4 * nz; i += YS_THREADS) {
            const int pl = i / nz, r = i - pl * nz;
            *reinterpret_cast<uint4*>(act + ((long)pl * YS_NB + rows_valid) * KP + r * 8) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    for (int i = tid; i < YS_NB * 4; i += YS_THREADS) {
        const int row = i >> 2, c = i & 3;
        float* d = hps + row * 16 + c * 4;
        const int j = ut * 16 + c * 4;
        if (row < rows_valid && j < H) st_cp_async16(d, a.hprev + (long)(r0 + row) * H + j);
        else *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    st_cp_async_wait_all();
    __syncthreads();
    st_mbar_wait(mbar, 0);
    XTS(18);
    {
        float acc[YS_NT][4];
#pragma unroll
        for (int nt = 0; nt < YS_NT; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        warp_mma_rows<YS_NT>(ah, al, NKT, act + (src * 2) * YS_NB * KP, act + (src * 2 + 1) * YS_NB * KP, KP, lane, acc);
        float* rw = res + warp * 16 * YS_RP;
        const int ra = lane >> 2, col = (lane & 3) * 2;
#pragma unroll
        for (int nt = 0; nt < YS_NT; ++nt) {
            rw[ra * YS_RP + nt * 8 + col] = acc[nt][0];
            rw[ra * YS_RP + nt * 8 + col + 1] = acc[nt][1];
            rw[(ra + 8) * YS_RP + nt * 8 + col] = acc[nt][2];
            rw[(ra + 8) * YS_RP + nt * 8 + col + 1] = acc[nt][3];
        }
    }
    XTS(19);
    __syncthreads();
    const long plane = (long)B * KP;
    for (int i = tid; i < 16 * rows_valid; i += YS_THREADS) {    // unit jl fastest -> 64-byte row segments
        const int jl = i & 15, bl = i >> 4;
        const int j = ut * 16 + jl, gb = r0 + bl;
        if (j < H) {
            const float* gi = gis + bl * 48 + jl;
            const float gir = gi[0] + res[(0 * 16 + jl) * YS_RP + bl];
            const float giz = gi[16] + res[(1 * 16 + jl) * YS_RP + bl];
            const float gin = gi[32] + res[(2 * 16 + jl) * YS_RP + bl];
            const float ghr = bhs[jl] + res[(3 * 16 + jl) * YS_RP + bl];
            const float ghz = bhs[16 + jl] + res[(4 * 16 + jl) * YS_RP + bl];
            const float ghn = bhs[32 + jl] + res[(5 * 16 + jl) * YS_RP + bl];
            // sigmoid(x) = (1 + tanh(x/2)) / 2 and tanh through ex2.approx / rcp.approx: ~1e-7 absolute error
            const float r = 0.5f + 0.5f * tanh_fast(0.5f * (gir + ghr));
            const float z = 0.5f + 0.5f * tanh_fast(0.5f * (giz + ghz));
            const float n = tanh_fast(gin + r * ghn);
            const float hn = (1.f - z) * n + z * hps[bl * 16 + jl];
            const long o = (long)gb * H + j;
            a.hnext[o] = hn;
            const __nv_bfloat16 hh = __float2bfloat16_rn(hn);
            a.hsp_next[(long)gb * KP + j] = hh;
            a.hsp_next[plane + (long)gb * KP + j] = __float2bfloat16_rn(hn - __bfloat162float(hh));
            if (a.Hbm) a.Hbm[((long)gb * a.T + a.t) * H + j] = hn;
            if (a.R) { a.R[o] = r; a.Z[o] = z; a.Nn[o] = n; a.GHN[o] = ghn; }
        }
    }
    XTS(20);
}

static inline int ys_kp(int H, int F) { return ((((H > F ? H : F) + 15) >> 4) << 4) + 8; }
static inline size_t ys_smem(int KP, int NB = YS_NB) {
    return (size_t)4 * NB * KP * 2 + ((size_t)6 * 16 * (NB + 1) + (size_t)NB * 64 + 48) * sizeof(float) + 16;
}
static inline size_t as_smem(int P, int H, int F, int rpc, int nbuf = 2) {
    const int KP = ys_kp(H, F);
    return (nbuf * ((size_t)P * H + (size_t)P * F) + (size_t)(rpc + 1) * ((H + 3) & ~3) + (size_t)((P + 3) & ~3) +
            (size_t)AS_PSPL * KP + (KP & 1)) * sizeof(float) + 16;
}
// persistent grid of the attention kernel: one CTA per SM, more only when a CTA's u rows would not fit in shared memory
static inline int as_grid(int B, int P, int H, int F) {
    int grid = B < kNumSMs ? B : kNumSMs;
    while (as_smem(P, H, F, (B + grid - 1) / grid) > 227 * 1024 && grid < B) grid *= 2;
    return grid < B ? grid : B;
}
static long pack_elems(int H, int F) {
    if (H < 1 || F < 1 || H > ST_MAXKT * 16 || F > ST_MAXKT * 16) return 0;
    const long NUT = (H + 15) / 16, NKT = ((H > F ? H : F) + 15) / 16;
    return 7 * NUT * NKT * 64;
}
}  // namespace caphn

using namespace caphn;

extern "C" {

// *pack_bytes = size of the weight pack for (H, F, P) (0: the step-split path does not cover the shape -- use
// caphn_attgru_seq_fwd); *work_bytes = size of the per-call workspace for batch B.
int caphn_attstep_pack_size(int H, int F, int P, int B, long* pack_bytes, long* work_bytes) {
    if (!pack_bytes || !work_bytes || B < 0 || P < 1) return CAPHN_EINVAL;
    long n = pack_elems(H, F);
    // the attention kernel keeps K_b and f_b in shared memory and fetches them with bulk copies (16-byte granules)
    if (n && (as_smem(P, H, F, 1) > 227 * 1024 || ys_kp(H, F) > 256 || (H & 3) || P > 32 * AS_SMAX || ((long)P * H) % 4 != 0 || ((long)P * F) % 4 != 0)) n = 0;
    *pack_bytes = n * 16;
    const int KP = ys_kp(H, F);
    *work_bytes = n ? (long)(align256((size_t)B * H * 4) + 6 * align256((size_t)B * KP * 2)) : 0;
    return CAPHN_OK;
}

// Build the fragment-ordered bf16 hi/lo pack of W_ih[:, E:E+F], W_hh (plain row-major [3H, E+F], [3H, H]) and U_a [H, H].
int caphn_attstep_pack(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, void* pack, void* stream) {
    if (pack_elems(H, F) == 0 || E < 0 || !pack || ((uintptr_t)pack & 15)) return CAPHN_EINVAL;
    const int NUT = (H + 15) / 16, NKT = ((H > F ? H : F) + 15) / 16;
    const long total = (long)7 * NUT * NKT * 32;
    attstep_pack_kernel<<<(unsigned)ceil_div(total, 256L), 256, 0, (cudaStream_t)stream>>>(Wih, Whh, Ua, E, F, H, NUT, NKT,
                                                                                         (uint4*)pack, 0, 0);
    CAPHN_RETURN_LAST();
}

// Many-style batch: one pack per style group.  Wih / Whh point at group 0's generated weights inside Theta [G, theta];
// group g's start gstride floats later (gstride = theta).  pack holds G packs of caphn_attstep_pack_size bytes each.
int caphn_attstep_pack_grouped(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, int G,
                               long gstride, void* pack, void* stream) {
    if (pack_elems(H, F) == 0 || E < 0 || G < 1 || !pack || ((uintptr_t)pack & 15)) return CAPHN_EINVAL;
    const int NUT = (H + 15) / 16, NKT = ((H > F ? H : F) + 15) / 16;
    const long total = (long)7 * NUT * NKT * 32;
    attstep_pack_kernel<<<dim3((unsigned)ceil_div(total, 256L), G), 256, 0, (cudaStream_t)stream>>>(
        Wih, Whh, Ua, E, F, H, NUT, NKT, (uint4*)pack, gstride, pack_elems(H, F));
    CAPHN_RETURN_LAST();
}

// Steps [t0, t1) of the attention-GRU recurrence, three launches per step.  Tensors as in caphn_attgru_seq_fwd (Hall[t0]
// holds h_{t0-1}); pack from caphn_attstep_pack, work a scratch buffer of *work_bytes (256-byte aligned).
// resume != 0: the workspace still holds the operand rows of Hall[t0] written by the previous call (which ran up to step
// t0 on the same buffers), so the initial conversion is skipped -- the one-step-per-call decode pattern.
static int attstep_fwd_impl(const float* Kp, const float* f, const float* GIw, const float* bu, const float* va,
                            const float* bv, const void* pack, void* work, const float* bhh, float* Hall, float* Hbm,
                            float* attn, float* ctx, long ldctx, float* Upre, float* R, float* Z, float* Nn, float* GHN,
                            int B, int T, int P, int H, int F, int t0, int t1, int resume, const int* tiles, int ntiles,
                            int tile_rows, void* stream) {
    long pb = 0, wb = 0;
    if (B <= 0 || T <= 0 || caphn_attstep_pack_size(H, F, P, B, &pb, &wb) != CAPHN_OK || pb == 0 || t0 < 0 || t1 > T ||
        t0 >= t1 || ((uintptr_t)pack & 15) || !work || ((uintptr_t)work & 255) || ((uintptr_t)Kp & 15) ||
        ((uintptr_t)f & 15))
        return CAPHN_EINVAL;
    if (R && !(Z && Nn && GHN && Upre)) return CAPHN_EINVAL;
    const int KP = ys_kp(H, F);
    const int NUT = (H + 15) / 16, NKT = ((H > F ? H : F) + 15) / 16;
    const long BH = (long)B * H;
    const size_t plane2 = align256((size_t)B * KP * 2);     // one bf16 plane; hi and lo planes are B*KP apart inside a pair
    uint8_t* w8 = (uint8_t*)work;
    float* ubuf = (float*)w8;
    __nv_bfloat16* csp = (__nv_bfloat16*)(w8 + align256((size_t)BH * 4));
    __nv_bfloat16* hsp0 = (__nv_bfloat16*)((uint8_t*)csp + 2 * plane2);
    __nv_bfloat16* hsp1 = (__nv_bfloat16*)((uint8_t*)hsp0 + 2 * plane2);
    auto hbuf = [&](int t) { return (t & 1) ? hsp1 : hsp0; };
    cudaStream_t st = (cudaStream_t)stream;
    // attention kernel: two single-buffered CTAs per SM when they fit (their phases overlap each other), else one
    // double-buffered CTA per SM
    int agrid = B < 2 * kNumSMs ? B : 2 * kNumSMs, nbuf = 1;
    int rpc = (B + agrid - 1) / agrid;
    if (2 * (as_smem(P, H, F, rpc, 1) + 1024) > 227 * 1024) {
        agrid = as_grid(B, P, H, F); rpc = (B + agrid - 1) / agrid; nbuf = 2;
    }
    const bool small_tiles = tiles && tile_rows <= YS_NB_SMALL;
    const size_t usmem = (size_t)2 * US_NB * KP * 2 + 16, asmem = as_smem(P, H, F, rpc, nbuf),
                 ysmem = ys_smem(KP, small_tiles ? YS_NB_SMALL : YS_NB);
    if (asmem > 227 * 1024 || (tiles && tile_rows > YS_NB)) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(attstep_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)asmem));
    CAPHN_CHECK(cudaFuncSetAttribute(attstep_gates_kernel<YS_NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ys_smem(KP)));
    CAPHN_CHECK(cudaFuncSetAttribute(attstep_gates_kernel<YS_NB_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)ys_smem(KP, YS_NB_SMALL)));
    if (!resume) {
        attstep_split_kernel<<<ceil_div(B * (KP / 2), 256), 256, 0, st>>>(Hall + t0 * BH, B, H, KP, hbuf(t0), hbuf(t0 + 1));
        CAPHN_LAUNCH_CHECK();
    }
    for (int t = t0; t < t1; ++t) {
        float* ut = Upre ? Upre + t * BH : ubuf;
        AttStepU u{(const uint4*)pack, bu, hbuf(t), ut, B, H, NUT, NKT, KP};
        CAPHN_CHECK(launch_pdl(attstep_u_kernel, dim3(ceil_div(NUT, US_WARPS), ceil_div(B, US_NB)), dim3(US_THREADS), usmem,
                               st, !(t == t0 && resume), u));
        ++caphn_launch_counter;
        AttStepA x{Kp, f, va, bv, ut, attn, ctx + (long)t * B * ldctx, ldctx, csp, B, T, t, P, H, F, KP, rpc, nbuf};
        CAPHN_CHECK(launch_pdl(attstep_attn_kernel, dim3(agrid), dim3(AS_THREADS), asmem, st, true, x));
        ++caphn_launch_counter;
        AttStepY y{csp, hbuf(t), hbuf(t + 1), Hall + t * BH, GIw + (long)t * B * 3 * H, (const uint4*)pack, bhh,
                   Hall + (t + 1) * BH, Hbm, R ? R + t * BH : nullptr, Z ? Z + t * BH : nullptr,
                   Nn ? Nn + t * BH : nullptr, GHN ? GHN + t * BH : nullptr, B, T, t, H, NUT, NKT, KP,
                   (const int4*)tiles, pack_elems(H, F)};
        if (small_tiles) {
            CAPHN_CHECK(launch_pdl(attstep_gates_kernel<YS_NB_SMALL>, dim3(NUT, ntiles), dim3(YS_THREADS), ysmem, st, true, y));
        } else {
            CAPHN_CHECK(launch_pdl(attstep_gates_kernel<YS_NB>, dim3(NUT, tiles ? ntiles : ceil_div(B, YS_NB)),
                                   dim3(YS_THREADS), ysmem, st, true, y));
        }
        ++caphn_launch_counter;
    }
    return (int)cudaGetLastError();
}

int caphn_attstep_fwd(const float* Kp, const float* f, const float* GIw, const float* bu, const float* va,
                      const float* bv, const void* pack, void* work, const float* bhh, float* Hall, float* Hbm,
                      float* attn, float* ctx, long ldctx, float* Upre, float* R, float* Z, float* Nn, float* GHN, int B,
                      int T, int P, int H, int F, int t0, int t1, int resume, void* stream) {
    return attstep_fwd_impl(Kp, f, GIw, bu, va, bv, pack, work, bhh, Hall, Hbm, attn, ctx, ldctx, Upre, R, Z, Nn, GHN, B, T,
                            P, H, F, t0, t1, resume, nullptr, 0, 0, stream);
}

// Many-style batch: rows sorted by style group; `tiles` = ntiles records {first row, rows (<= 64), group, 0} that never
// straddle a group (tile_rows = the largest row count in the table: <= 8 selects the small-tile gates kernel);
// `pack` = the G packs of caphn_attstep_pack_grouped, bhh = [G, 3H].  The U and attention kernels use
// no generated weights and run exactly as in the single-group call (U_a is read from group 0's pack).
int caphn_attstep_fwd_grouped(const float* Kp, const float* f, const float* GIw, const float* bu, const float* va,
                              const float* bv, const void* pack, void* work, const float* bhh, float* Hall, float* Hbm,
                              float* attn, float* ctx, long ldctx, float* Upre, float* R, float* Z, float* Nn, float* GHN,
                              int B, int T, int P, int H, int F, int t0, int t1, int resume, const int* tiles, int ntiles,
                              int tile_rows, void* stream) {
    if (!tiles || ntiles < 1 || tile_rows < 1 || ((uintptr_t)tiles & 15)) return CAPHN_EINVAL;
    return attstep_fwd_impl(Kp, f, GIw, bu, va, bv, pack, work, bhh, Hall, Hbm, attn, ctx, ldctx, Upre, R, Z, Nn, GHN, B, T,
                            P, H, F, t0, t1, resume, tiles, ntiles, tile_rows, stream);
}

#ifdef CAPHN_ATTCL_TIMING
int caphn_attst_timestamps(long long* out) {
    return (int)cudaMemcpyFromSymbol(out, caphn::g_attst_ts, sizeof(long long) * 32);
}
#endif

}  // extern "C"
