// Attention-GRU recurrence, BPTT, as three batch-wide kernels per time step (the backward of attgru_step.cu), chained with
// programmatic dependent launch, plus one deferred kernel for the gradients that do not feed the recurrence.
//
// Same arithmetic as attgru_seq_bwd_kernel (autograd of reference models/decoderlstm.py:97-100 and
// models/attention.py:33-45; SURVEY.md Appendix B.2-B.4).  Per step t = T-1 .. 0:
//
//   G1 attbwd_gate_kernel   dh_t = keep_{t+1} + dgh_{t+1} W_hh + du_{t+1} U_a + dL/dh_t   (the U_a product on the warp
//                           tensor cores, bf16 hi/lo split), then the GRU gate gradients dgi_t, dgh_t, keep_t in the
//                           epilogue.  CTA = 16 hidden units x 64 rows.
//   G2 attbwd_gemm_kernel   dctx_t = dgi_t W_ih[:,E:]   and   dgh_t W_hh   (contraction over the 3H gate axis) on the warp
//                           tensor cores; the transposed-weight fragments stream from an L2-resident pack.
//   A' attbwd_attn_kernel   persistent over rows, K_b / f_b tiles double-buffered by bulk TMA:  dalpha = <dctx, f_p>,
//                           softmax backward -> ds,  du_j = v_j sum_p ds_p (1 - tanh^2(K_pj + u_j)).
//
// Deferred (they are sums over t that nothing in the loop consumes):
//   D  attbwd_dk_kernel     dK[b,p,j] = v_j sum_t ds[b,t,p] (1 - q^2),  dv_a[j] = sum_{b,t,p} ds q,  q = tanh(K + u_t) --
//                           instead of a read-modify-write of the 20 MB dK tensor in every step.
//   (df = sum_t alpha_t dctx_t is caphn_attn_df, as before.)
#include "step_common.cuh"

namespace caphn {

// ------------------------------------------------------------------------------------------------------------------
// transposed-weight pack (A fragments, uint4 {a0,a1,a2,a3} per lane, hi then lo):
//   group 0: U_a^T      NUT tiles x NKT   (rows = output unit j, K = k over H)      A[j][k]  = Ua[k][j]
//   group 1: W_ih[:,E:]^T NFT tiles x NKT3 (rows = feature fi,   K = q over 3H)     A[fi][q] = Wih[q][E+fi]
//   group 2: W_hh^T     NUT tiles x NKT3  (rows = unit k,        K = q over 3H)     A[k][q]  = Whh[q][k]
// ------------------------------------------------------------------------------------------------------------------
// blockIdx.y = style group (see attstep_pack_kernel): W_ih / W_hh advance gstride floats, the pack pstride uint4 per group.
__global__ void attbwd_pack_kernel(const float* __restrict__ Wih, const float* __restrict__ Whh,
                                   const float* __restrict__ Ua, int E, int F, int H, int NUT, int NFT, int NKT, int NKT3,
                                   uint4* __restrict__ out, long gstride, long pstride) {
    const long n0 = (long)NUT * NKT, n1 = (long)NFT * NKT3, n2 = (long)NUT * NKT3;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (n0 + n1 + n2) * 32) return;
    Wih += (long)blockIdx.y * gstride;
    Whh += (long)blockIdx.y * gstride;
    out += (long)blockIdx.y * pstride;
    const int lane = (int)(idx & 31);
    const long r = idx >> 5;
    int grp, tile, kt;
    if (r < n0) { grp = 0; tile = (int)(r / NKT); kt = (int)(r % NKT); }
    else if (r < n0 + n1) { grp = 1; tile = (int)((r - n0) / NKT3); kt = (int)((r - n0) % NKT3); }
    else { grp = 2; tile = (int)((r - n0 - n1) / NKT3); kt = (int)((r - n0 - n1) % NKT3); }
    const int ma = tile * 16 + (lane >> 2), mb = ma + 8;
    const int k0 = kt * 16 + (lane & 3) * 2;
    const int H3 = 3 * H;
    auto w = [&](int m, int k) -> float {
        if (grp == 0) return (m < H && k < H) ? Ua[(long)k * H + m] : 0.f;
        if (grp == 1) return (m < F && k < H3) ? Wih[(long)k * (E + F) + E + m] : 0.f;
        return (m < H && k < H3) ? Whh[(long)k * H + m] : 0.f;
    };
    uint4 hi, lo;
    split2(w(ma, k0), w(ma, k0 + 1), hi.x, lo.x);
    split2(w(mb, k0), w(mb, k0 + 1), hi.y, lo.y);
    split2(w(ma, k0 + 8), w(ma, k0 + 9), hi.z, lo.z);
    split2(w(mb, k0 + 8), w(mb, k0 + 9), hi.w, lo.w);
    out[(r * 2 + 0) * 32 + lane] = hi;
    out[(r * 2 + 1) * 32 + lane] = lo;
}

// ------------------------------------------------------------------------------------------------------------------
// G1: dh_t and the gate gradients.      CTA = 16 units x 64 rows, 4 warps (each 16 rows = 2 n-tiles)
// ------------------------------------------------------------------------------------------------------------------
constexpr int G1_NB = 64, G1_WARPS = 4, G1_THREADS = G1_WARPS * 32, G1_RP = G1_NB + 1;

struct BwdG1 {
    const uint4* Wp;             // group 0 (U_a^T) tiles
    const __nv_bfloat16* dusp;   // [2][B][KP]  du_{t+1} hi, lo
    const float* dhp;            // [B,H]   dgh_{t+1} W_hh
    float* keep;                 // [B,H]   dh_{t+1} * z_{t+1} on entry, dh_t * z_t on exit
    const float* dHbm;           // [B,T,H]
    const float* R; const float* Z; const float* Nn; const float* GHN; const float* Hprev;   // [B,H] of step t
    float* dGI; float* dGH;      // [B,3H] of step t
    __nv_bfloat16* gisp;         // [2][B][KP3] dgi_t hi, lo
    __nv_bfloat16* ghsp;         // [2][B][KP3] dgh_t hi, lo
    float* dh0;                  // [B,H]  (mode 2)
    int B, T, t, H, NUT, NKT, KP, KP3;
    int mode;                    // 0: last time step (no carry)   1: inner step   2: after step 0 -> dh0 only
};

__global__ void __launch_bounds__(G1_THREADS) attbwd_gate_kernel(const BwdG1 a) {
    extern __shared__ __align__(16) uint8_t gsm[];
    const int H = a.H, B = a.B, KP = a.KP, NKT = a.NKT, H3 = 3 * a.H;
    __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(gsm);      // [2][NB][KP]  du rows
    float* res = reinterpret_cast<float*>(act + 2 * G1_NB * KP);      // [16][RP]     (du U_a) tile
    float* sv = res + 16 * G1_RP;                                     // [6][NB][16]  R Z N GHN Hprev dHbm tiles (16 x 65 floats: 16-byte aligned)
    float* cr = sv + 6 * G1_NB * 16;                                  // [2][NB][16]  keep, dhp tiles
    uint64_t* mbar = reinterpret_cast<uint64_t*>(cr + 2 * G1_NB * 16);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ut = blockIdx.x, r0 = blockIdx.y * G1_NB;
    const int rows_valid = min(G1_NB, B - r0);
    if (tid == 0) st_mbar_init(mbar, 1);
    // ---- inputs that do not depend on the previous kernels: weight fragments, saved forward tiles, dL/dh_t ----
    uint4 ah[ST_MAXKT], al[ST_MAXKT];
    if (a.mode != 0) {
        const uint4* wp = a.Wp + ((long)ut * NKT) * 64 + lane;
#pragma unroll
        for (int kt = 0; kt < ST_MAXKT; ++kt)
            if (kt < NKT) { ah[kt] = st_ldg_u4(wp + (long)kt * 64); al[kt] = st_ldg_u4(wp + (long)kt * 64 + 32); }
    }
    if (a.mode != 2) {
        for (int i = tid; i < 6 * G1_NB * 4; i += G1_THREADS) {     // (array, row, 4-unit chunk); H % 4 == 0
            const int arr = i / (G1_NB * 4), r = i - arr * (G1_NB * 4);
            const int row = r >> 2, c = r & 3;
            float* d = sv + (arr * G1_NB + row) * 16 + c * 4;
            const int j = ut * 16 + c * 4;
            if (row < rows_valid && j < H) {
                const long gb = r0 + row;
                const float* src = arr == 0 ? a.R : arr == 1 ? a.Z : arr == 2 ? a.Nn : arr == 3 ? a.GHN : a.Hprev;
                st_cp_async16(d, arr < 5 ? src + gb * H + j : a.dHbm + (gb * a.T + a.t) * H + j);
            } else {
                *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    }
    pdl_launch_dependents();
    pdl_wait();
    if (a.mode != 0) {
        stage_rows_bulk<G1_NB, G1_THREADS>(a.dusp, (long)B * KP, r0, rows_valid, KP, 2, act, mbar, tid);
        for (int i = tid; i < 2 * G1_NB * 4; i += G1_THREADS) {
            const int arr = i / (G1_NB * 4), r = i - arr * (G1_NB * 4);
            const int row = r >> 2, c = r & 3;
            float* d = cr + (arr * G1_NB + row) * 16 + c * 4;
            const int j = ut * 16 + c * 4;
            if (row < rows_valid && j < H) st_cp_async16(d, (arr == 0 ? a.keep : a.dhp) + (long)(r0 + row) * H + j);
            else *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    st_cp_async_wait_all();
    __syncthreads();
    if (a.mode != 0) {
        st_mbar_wait(mbar, 0);
        float acc[2][4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        warp_mma_rows<2>(ah, al, NKT, act + (warp * 16) * KP, act + (G1_NB + warp * 16) * KP, KP, lane, acc);
        const int ra = lane >> 2, col = warp * 16 + (lane & 3) * 2;
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            res[ra * G1_RP + nt * 8 + col] = acc[nt][0];
            res[ra * G1_RP + nt * 8 + col + 1] = acc[nt][1];
            res[(ra + 8) * G1_RP + nt * 8 + col] = acc[nt][2];
            res[(ra + 8) * G1_RP + nt * 8 + col + 1] = acc[nt][3];
        }
        __syncthreads();
    }
    const long plane3 = (long)B * a.KP3;
    for (int i = tid; i < 16 * rows_valid; i += G1_THREADS) {        // unit jl fastest -> 64-byte row segments
        const int jl = i & 15, bl = i >> 4;
        const int j = ut * 16 + jl;
        if (j >= H) continue;
        const long gb = r0 + bl;
        float dh = 0.f;
        if (a.mode != 0) dh = cr[bl * 16 + jl] + cr[(G1_NB + bl) * 16 + jl] + res[jl * G1_RP + bl];
        if (a.mode == 2) { a.dh0[gb * H + j] = dh; continue; }
        const float r = sv[(0 * G1_NB + bl) * 16 + jl], z = sv[(1 * G1_NB + bl) * 16 + jl];
        const float n = sv[(2 * G1_NB + bl) * 16 + jl], ghn = sv[(3 * G1_NB + bl) * 16 + jl];
        const float hp = sv[(4 * G1_NB + bl) * 16 + jl];
        dh += sv[(5 * G1_NB + bl) * 16 + jl];
        const float dn = dh * (1.f - z);
        const float dz = dh * (hp - n);
        const float dan = dn * (1.f - n * n);
        const float dar = dan * ghn * r * (1.f - r);
        const float daz = dz * z * (1.f - z);
        const float danr = dan * r;
        a.keep[gb * H + j] = dh * z;
        float* gi = a.dGI + gb * H3;
        float* gh = a.dGH + gb * H3;
        gi[j] = dar; gi[H + j] = daz; gi[2 * H + j] = dan;
        gh[j] = dar; gh[H + j] = daz; gh[2 * H + j] = danr;
        const float v[4] = {dar, daz, dan, danr};
        __nv_bfloat16 vh[4], vl[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            vh[e] = __float2bfloat16_rn(v[e]);
            vl[e] = __float2bfloat16_rn(v[e] - __bfloat162float(vh[e]));
        }
        __nv_bfloat16* gi_h = a.gisp + gb * a.KP3;
        __nv_bfloat16* gh_h = a.ghsp + gb * a.KP3;
        gi_h[j] = vh[0]; gi_h[H + j] = vh[1]; gi_h[2 * H + j] = vh[2];
        gi_h[plane3 + j] = vl[0]; gi_h[plane3 + H + j] = vl[1]; gi_h[plane3 + 2 * H + j] = vl[2];
        gh_h[j] = vh[0]; gh_h[H + j] = vh[1]; gh_h[2 * H + j] = vh[3];
        gh_h[plane3 + j] = vl[0]; gh_h[plane3 + H + j] = vl[1]; gh_h[plane3 + 2 * H + j] = vl[3];
    }
}

// ------------------------------------------------------------------------------------------------------------------
// G2: dctx_t = dgi_t W_ih[:,E:],  dhp = dgh_t W_hh        CTA = 4 output tiles of one kind (4 warps) x 32 rows
// ------------------------------------------------------------------------------------------------------------------
constexpr int G2_NB = 32, G2_NB_SMALL = 8, G2_WARPS = 4, G2_THREADS = G2_WARPS * 32;
constexpr int G2_PF_BIG = 19;     // register prefetch depth (uint4 pairs) of the weight fragments: 32-row tiles, 2 CTAs per SM
constexpr int G2_PF_SMALL = 8;    // 8-row tiles of a many-domain batch: shallow prefetch, ~100 registers, 4-5 CTAs per SM hide the loads

struct BwdG2 {
    const uint4* Wc;             // group 1 tiles (NFT x NKT3)
    const uint4* Wh;             // group 2 tiles (NUT x NKT3)
    const __nv_bfloat16* gisp;   // [2][B][KP3]
    const __nv_bfloat16* ghsp;   // [2][B][KP3]
    float* dctx;                 // [B,F] of step t
    float* dhp;                  // [B,H]
    int B, H, F, NUT, NFT, NKT3, KP3, NG1;   // NG1 = number of dctx tile groups (blockIdx.x < NG1)
    // many-style batch: row tile blockIdx.y = rows [tiles[y].x, +tiles[y].y) of style group tiles[y].z, whose transposed-weight
    // pack starts pstride uint4 after the previous group's.  null: one group, tiles of G2_NB consecutive rows.
    const int4* tiles;
    long pstride;
};

template <int G2_NB, int G2_PF>
__global__ void __launch_bounds__(G2_THREADS, G2_NB >= 32 ? 2 : 4) attbwd_gemm_kernel(const BwdG2 a) {
    constexpr int G2_NT = G2_NB / 8, G2_RP = G2_NB + 1;
    extern __shared__ __align__(16) uint8_t g2sm[];
    const int B = a.B, KP3 = a.KP3, NKT3 = a.NKT3;
    __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(g2sm);          // [2][NB][KP3]
    float* res = reinterpret_cast<float*>(act + 2 * G2_NB * KP3);          // [4][16][RP]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(res + 4 * 16 * G2_RP + ((4 * 16 * G2_RP) & 1));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool is_ctx = (int)blockIdx.x < a.NG1;
    const int tile = (is_ctx ? blockIdx.x : blockIdx.x - a.NG1) * G2_WARPS + warp;
    const int ntiles = is_ctx ? a.NFT : a.NUT;
    int r0 = blockIdx.y * G2_NB, rows_valid = min(G2_NB, B - r0), grp = 0;
    if (a.tiles) { const int4 tl = a.tiles[blockIdx.y]; r0 = tl.x; rows_valid = tl.y; grp = tl.z; }
    const bool has_tile = tile < ntiles;
    if (tid == 0) st_mbar_init(mbar, 1);
    const uint4* wp = (is_ctx ? a.Wc : a.Wh) + (long)grp * a.pstride + ((long)(has_tile ? tile : 0) * NKT3) * 64 + lane;
    uint4 ah[G2_PF], al[G2_PF];
#pragma unroll
    for (int i = 0; i < G2_PF; ++i)
        if (i < NKT3) { ah[i] = st_ldg_u4(wp + (long)i * 64); al[i] = st_ldg_u4(wp + (long)i * 64 + 32); }
    pdl_launch_dependents();
    pdl_wait();                                   // the split gate-gradient rows come from G1 of this step
    stage_rows_bulk<G2_NB, G2_THREADS>(is_ctx ? a.gisp : a.ghsp, (long)B * KP3, r0, rows_valid, KP3, 2, act, mbar, tid);
    __syncthreads();
    st_mbar_wait(mbar, 0);
    float acc[G2_NT][4];
#pragma unroll
    for (int nt = 0; nt < G2_NT; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
    if (has_tile) {
        const __nv_bfloat16* bhi = act;
        const __nv_bfloat16* blo = act + G2_NB * KP3;
        const int nrow = lane >> 2, kc = (lane & 3) * 2;
        for (int kt0 = 0; kt0 < NKT3; kt0 += G2_PF) {
#pragma unroll
            for (int i = 0; i < G2_PF; ++i) {
                const int kt = kt0 + i;
                if (kt < NKT3) {
                    const uint32_t fh[4] = {ah[i].x, ah[i].y, ah[i].z, ah[i].w};
                    const uint32_t fl[4] = {al[i].x, al[i].y, al[i].z, al[i].w};
                    if (kt + G2_PF < NKT3) {
                        ah[i] = st_ldg_u4(wp + (long)(kt + G2_PF) * 64);
                        al[i] = st_ldg_u4(wp + (long)(kt + G2_PF) * 64 + 32);
                    }
#pragma unroll
                    for (int nt = 0; nt < G2_NT; ++nt) {
                        const uint32_t* ph = reinterpret_cast<const uint32_t*>(bhi + (nt * 8 + nrow) * KP3 + kt * 16 + kc);
                        const uint32_t* pl = reinterpret_cast<const uint32_t*>(blo + (nt * 8 + nrow) * KP3 + kt * 16 + kc);
                        const uint32_t h0 = ph[0], h1 = ph[4], l0 = pl[0], l1 = pl[4];
                        mma_bf16(acc[nt], fh, h0, h1);
                        mma_bf16(acc[nt], fh, l0, l1);
                        mma_bf16(acc[nt], fl, h0, h1);
                    }
                }
            }
        }
    }
    {
        float* rw = res + warp * 16 * G2_RP;
        const int ra = lane >> 2, col = (lane & 3) * 2;
#pragma unroll
        for (int nt = 0; nt < G2_NT; ++nt) {
            rw[ra * G2_RP + nt * 8 + col] = acc[nt][0];
            rw[ra * G2_RP + nt * 8 + col + 1] = acc[nt][1];
            rw[(ra + 8) * G2_RP + nt * 8 + col] = acc[nt][2];
            rw[(ra + 8) * G2_RP + nt * 8 + col + 1] = acc[nt][3];
        }
    }
    __syncthreads();
    const int ncol = is_ctx ? a.F : a.H;
    float* out = is_ctx ? a.dctx : a.dhp;
    const int m0 = (is_ctx ? blockIdx.x : blockIdx.x - a.NG1) * G2_WARPS * 16;
    for (int i = tid; i < G2_WARPS * 16 * rows_valid; i += G2_THREADS) {   // 64 consecutive outputs of a row per pass
        const int ml = i & (G2_WARPS * 16 - 1), bl = i / (G2_WARPS * 16);
        const int m = m0 + ml;
        if (m < ncol) out[(long)(r0 + bl) * ncol + m] = res[ml * G2_RP + bl];
    }
}

// ------------------------------------------------------------------------------------------------------------------
// A': attention backward for step t, persistent over rows (same tile pipeline as the forward attention kernel)
// ------------------------------------------------------------------------------------------------------------------
constexpr int BA_THREADS = 512, BA_WARPS = BA_THREADS / 32, BA_SMAX = 4;

struct BwdA {
    const float* Kp; const float* f; const float* va;
    const float* dctx;           // [B,F] of step t
    const float* attn;           // [B,T,P]
    const float* dattn;          // [B,T,P] or null
    const float* Upre;           // [B,H] of step t
    float* dS;                   // [B,T,P]  d score
    float* dU;                   // [B,H] of step t
    __nv_bfloat16* dusp;         // [2][B][KP]
    float* dbv;                  // [1] atomically accumulated
    int B, T, t, P, H, F, KP, RPC;
    int NBUF;                    // tile buffers per CTA (see attstep_attn_kernel)
};

__global__ void __launch_bounds__(BA_THREADS, 2) attbwd_attn_kernel(const BwdA a) {
    extern __shared__ __align__(16) float basm[];
    const int H = a.H, F = a.F, P = a.P, KP = a.KP, B = a.B;
    const int PS = (P + 3) & ~3, H4 = (H + 3) & ~3, F4 = (F + 3) & ~3;
    const int tile = P * H + P * F;
    float* bufs = basm;                                  // [2][tile]
    const int NBUF = a.NBUF;
    float* us = bufs + NBUF * tile;                      // [RPC][H4]
    float* dcs = us + a.RPC * H4;                        // [RPC][F4]
    float* als = dcs + a.RPC * F4;                       // [RPC][PS]
    float* vs = als + a.RPC * PS;                        // [H4]
    float* dal = vs + H4;                                // [PS]
    float* dup = dal + PS;                               // [2][H4]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(dup + 2 * H4);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nrows = (B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const uint32_t kb = (uint32_t)P * H * 4, fb = (uint32_t)P * F * 4;
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
    for (int j = tid; j < H; j += BA_THREADS) vs[j] = a.va[j];
    for (int i = tid; i < nrows * H; i += BA_THREADS) {                 // saved by the forward: not a dependency
        const int r = i / H, j = i - r * H;
        us[r * H4 + j] = ldg_stream1(a.Upre + (blockIdx.x + (long)r * gridDim.x) * H + j);
    }
    for (int i = tid; i < nrows * P; i += BA_THREADS) {
        const int r = i / P, p = i - r * P;
        als[r * PS + p] = ldg_stream1(a.attn + ((blockIdx.x + (long)r * gridDim.x) * a.T + a.t) * P + p);
    }
    pdl_launch_dependents();
    pdl_wait();                                          // dctx comes from G2 of this step
    for (int i = tid; i < nrows * F; i += BA_THREADS) {
        const int r = i / F, k = i - r * F;
        dcs[r * F4 + k] = ldg_stream1(a.dctx + (blockIdx.x + (long)r * gridDim.x) * F + k);
    }
    __syncthreads();
    const long plane = (long)B * KP;
    float dbv_acc = 0.f;
    for (int i = 0; i < nrows; ++i) {
        const long b = blockIdx.x + (long)i * gridDim.x;
        const int bi = NBUF == 2 ? (i & 1) : 0, ph = NBUF == 2 ? ((i >> 1) & 1) : (i & 1);
        const float* Ks = bufs + bi * tile;
        const float* fs = Ks + P * H;
        const float* ur = us + i * H4;
        const float* dc = dcs + i * F4;
        const float* alr = als + i * PS;
        st_mbar_wait(&mbar[bi], ph);
        // d alpha_p = <dctx, f_p> (+ external gradient of the returned attention weights)
        for (int p = warp; p < P; p += BA_WARPS) {
            float s = 0.f;
            for (int k = lane; k < F; k += 32) s = fmaf(dc[k], fs[p * F + k], s);
            s = warp_sum(s);
            if (lane == 0) dal[p] = s + (a.dattn ? a.dattn[(b * a.T + a.t) * P + p] : 0.f);
        }
        __syncthreads();
        if (warp == 0) {       // softmax backward: ds_p = alpha_p (dalpha_p - sum_q alpha_q dalpha_q)
            float x[BA_SMAX], al[BA_SMAX];
            float c = 0.f;
#pragma unroll
            for (int e = 0; e < BA_SMAX; ++e) {
                const int p = lane + 32 * e;
                x[e] = p < P ? dal[p] : 0.f;
                al[e] = p < P ? alr[p] : 0.f;
                c = fmaf(al[e], x[e], c);
            }
            c = warp_sum(c);
#pragma unroll
            for (int e = 0; e < BA_SMAX; ++e) {
                const int p = lane + 32 * e;
                if (p < P) {
                    const float ds = al[e] * (x[e] - c);
                    dal[p] = ds;
                    a.dS[(b * a.T + a.t) * P + p] = ds;
                    dbv_acc += ds;
                }
            }
        }
        __syncthreads();
        {   // du_j = v_j sum_p ds_p (1 - q^2), q = tanh(K_pj + u_j); the positions split over two thread groups
            const int j = tid & 255, half = tid >> 8;
            if (j < H) {
                const int ph = (P + 1) >> 1;
                const int pa = half * ph, pb = min(P, pa + ph);
                const float uj = ur[j];
                float acc0 = 0.f, acc1 = 0.f;
                int p = pa;
                for (; p + 1 < pb; p += 2) {
                    const float q0 = tanh_fast(Ks[p * H + j] + uj), q1 = tanh_fast(Ks[(p + 1) * H + j] + uj);
                    acc0 = fmaf(dal[p], 1.f - q0 * q0, acc0);
                    acc1 = fmaf(dal[p + 1], 1.f - q1 * q1, acc1);
                }
                if (p < pb) {
                    const float q0 = tanh_fast(Ks[p * H + j] + uj);
                    acc0 = fmaf(dal[p], 1.f - q0 * q0, acc0);
                }
                dup[half * H4 + j] = acc0 + acc1;
            }
        }
        __syncthreads();
        if (tid == 0 && i + NBUF < nrows) {   // both tiles of this buffer are dead: fetch this CTA's next row for it
            const long bn = blockIdx.x + (long)(i + NBUF) * gridDim.x;
            float* dst = bufs + bi * tile;
            st_mbar_expect_tx(&mbar[bi], kb + fb);
            st_bulk_g2s(dst, a.Kp + bn * P * H, kb, &mbar[bi]);
            st_bulk_g2s(dst + P * H, a.f + bn * P * F, fb, &mbar[bi]);
        }
        if (tid < 128 && tid * 2 < KP) {
            const int k = tid * 2;
            const float d0 = k < H ? vs[k] * (dup[k] + dup[H4 + k]) : 0.f;
            const float d1 = k + 1 < H ? vs[k + 1] * (dup[k + 1] + dup[H4 + k + 1]) : 0.f;
            if (k < H) a.dU[b * H + k] = d0;
            if (k + 1 < H) a.dU[b * H + k + 1] = d1;
            uint32_t hi, lo;
            split2(d0, d1, hi, lo);
            *reinterpret_cast<uint32_t*>(a.dusp + b * KP + k) = hi;
            *reinterpret_cast<uint32_t*>(a.dusp + plane + b * KP + k) = lo;
        }
        // (dal / dup are rewritten only after the next row's first __syncthreads)
    }
    if (warp == 0) {
        dbv_acc = warp_sum(dbv_acc);
        if (lane == 0 && dbv_acc != 0.f) atomicAdd(a.dbv, dbv_acc);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// D: deferred dK and dv_a
// ------------------------------------------------------------------------------------------------------------------
constexpr int BD_THREADS = 512;

struct BwdD {
    const float* Kp; const float* va;
    const float* Upre;           // [T,B,H]
    const float* dS;             // [B,T,P]
    float* dK;                   // [B,P,H]
    float* dva;                  // [H] atomically accumulated
    int B, T, P, H;
};

__global__ void __launch_bounds__(BD_THREADS, 1) attbwd_dk_kernel(const BwdD a) {
    extern __shared__ __align__(16) float bdsm[];
    const int H = a.H, P = a.P, B = a.B, T = a.T;
    const int PS = (P + 3) & ~3, H4 = (H + 3) & ~3;
    float* Kt = bdsm;                                    // [2][P*H]
    float* us = Kt + 2 * P * H;                          // [T][H4]
    float* dss = us + T * H4;                            // [T][PS]
    float* red = dss + T * PS;                           // [2][H4]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(red + 2 * H4);
    const int tid = threadIdx.x;
    const int nrows = (B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const uint32_t kb = (uint32_t)P * H * 4;
    if (tid == 0) {
        st_mbar_init(&mbar[0], 1);
        st_mbar_init(&mbar[1], 1);
        for (int i = 0; i < 2 && i < nrows; ++i) {
            st_mbar_expect_tx(&mbar[i], kb);
            st_bulk_g2s(Kt + i * P * H, a.Kp + (blockIdx.x + (long)i * gridDim.x) * P * H, kb, &mbar[i]);
        }
    }
    const int j = tid & 255, half = tid >> 8;
    const float vj = j < H ? a.va[j] : 0.f;
    float dva_acc = 0.f, dva_acc2 = 0.f;
    pdl_launch_dependents();
    pdl_wait();                                          // ds of every step
    __syncthreads();
    for (int i = 0; i < nrows; ++i) {
        const long b = blockIdx.x + (long)i * gridDim.x;
        for (int e = tid; e < T * H; e += BD_THREADS) {
            const int t = e / H, k = e - t * H;
            us[t * H4 + k] = ldg_stream1(a.Upre + ((long)t * B + b) * H + k);
        }
        for (int e = tid; e < T * P; e += BD_THREADS) {
            const int t = e / P, p = e - t * P;
            dss[t * PS + p] = ldg_stream1(a.dS + (b * T + t) * P + p);
        }
        __syncthreads();
        st_mbar_wait(&mbar[i & 1], (i >> 1) & 1);
        const float* Ks = Kt + (i & 1) * P * H;
        if (j < H) {
            const int ph = (P + 1) >> 1;
            const int pa = half * ph, pb = min(P, pa + ph);
            int p = pa;
            for (; p + 1 < pb; p += 2) {          // two positions x two time steps: four independent tanh chains
                const float kv0 = Ks[p * H + j], kv1 = Ks[(p + 1) * H + j];
                float a00 = 0.f, a01 = 0.f, a10 = 0.f, a11 = 0.f;
                int t = 0;
                for (; t + 1 < T; t += 2) {
                    const float u0 = us[t * H4 + j], u1 = us[(t + 1) * H4 + j];
                    const float q00 = tanh_fast(kv0 + u0), q01 = tanh_fast(kv0 + u1);
                    const float q10 = tanh_fast(kv1 + u0), q11 = tanh_fast(kv1 + u1);
                    const float d00 = dss[t * PS + p], d01 = dss[(t + 1) * PS + p];
                    const float d10 = dss[t * PS + p + 1], d11 = dss[(t + 1) * PS + p + 1];
                    a00 = fmaf(d00, 1.f - q00 * q00, a00); a01 = fmaf(d01, 1.f - q01 * q01, a01);
                    a10 = fmaf(d10, 1.f - q10 * q10, a10); a11 = fmaf(d11, 1.f - q11 * q11, a11);
                    dva_acc = fmaf(d00, q00, dva_acc); dva_acc2 = fmaf(d01, q01, dva_acc2);
                    dva_acc = fmaf(d10, q10, dva_acc); dva_acc2 = fmaf(d11, q11, dva_acc2);
                }
                if (t < T) {
                    const float u0 = us[t * H4 + j];
                    const float q00 = tanh_fast(kv0 + u0), q10 = tanh_fast(kv1 + u0);
                    const float d00 = dss[t * PS + p], d10 = dss[t * PS + p + 1];
                    a00 = fmaf(d00, 1.f - q00 * q00, a00); a10 = fmaf(d10, 1.f - q10 * q10, a10);
                    dva_acc = fmaf(d00, q00, dva_acc); dva_acc2 = fmaf(d10, q10, dva_acc2);
                }
                a.dK[(b * P + p) * H + j] = vj * (a00 + a01);
                a.dK[(b * P + p + 1) * H + j] = vj * (a10 + a11);
            }
            if (p < pb) {
                const float kv = Ks[p * H + j];
                float acc0 = 0.f;
                for (int t = 0; t < T; ++t) {
                    const float q0 = tanh_fast(kv + us[t * H4 + j]);
                    const float d0 = dss[t * PS + p];
                    acc0 = fmaf(d0, 1.f - q0 * q0, acc0);
                    dva_acc = fmaf(d0, q0, dva_acc);
                }
                a.dK[(b * P + p) * H + j] = vj * acc0;
            }
        }
        __syncthreads();
        if (tid == 0 && i + 2 < nrows) {
            st_mbar_expect_tx(&mbar[i & 1], kb);
            st_bulk_g2s(Kt + (i & 1) * P * H, a.Kp + (blockIdx.x + (long)(i + 2) * gridDim.x) * P * H, kb, &mbar[i & 1]);
        }
    }
    if (j < H) red[half * H4 + j] = dva_acc + dva_acc2;
    __syncthreads();
    if (tid < H) {
        const float s = red[tid] + red[H4 + tid];
        if (s != 0.f) atomicAdd(a.dva + tid, s);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// host-side sizing
// ------------------------------------------------------------------------------------------------------------------
static inline int bw_kp(int H, int F) { return ((((H > F ? H : F) + 15) >> 4) << 4) + 8; }
static inline int bw_kp3(int H) { return (((3 * H + 15) >> 4) << 4) + 8; }
static inline size_t g1_smem(int KP) {
    return (size_t)2 * G1_NB * KP * 2 + ((size_t)16 * G1_RP + (size_t)8 * G1_NB * 16) * sizeof(float) + 16;
}
static inline size_t g2_smem(int KP3, int NB = G2_NB) {
    return (size_t)2 * NB * KP3 * 2 + ((size_t)4 * 16 * (NB + 1) + 2) * sizeof(float) + 16;
}
static inline size_t ba_smem(int P, int H, int F, int rpc, int nbuf = 2) {
    const int PS = (P + 3) & ~3, H4 = (H + 3) & ~3, F4 = (F + 3) & ~3;
    return (nbuf * ((size_t)P * H + (size_t)P * F) + (size_t)rpc * (H4 + F4 + PS) + 3 * (size_t)H4 + PS) * sizeof(float) + 16;
}
static inline size_t bd_smem(int P, int H, int T) {
    const int PS = (P + 3) & ~3, H4 = (H + 3) & ~3;
    return (2 * (size_t)P * H + (size_t)T * (H4 + PS) + 2 * (size_t)H4) * sizeof(float) + 16;
}
static inline int ba_grid(int B, int P, int H, int F) {
    int grid = B < kNumSMs ? B : kNumSMs;
    while (ba_smem(P, H, F, (B + grid - 1) / grid) > 227 * 1024 && grid < B) grid *= 2;
    return grid < B ? grid : B;
}
static long bw_pack_elems(int H, int F, int P, int T) {
    if (H < 4 || F < 1 || P < 1 || T < 1 || H > ST_MAXKT * 16 || F > ST_MAXKT * 16 || (H & 3) || ((long)P * F) % 4 != 0 ||
        P > 32 * BA_SMAX || bw_kp(H, F) > 256 || ba_smem(P, H, F, 1) > 227 * 1024 || bd_smem(P, H, T) > 227 * 1024 ||
        g2_smem(bw_kp3(H)) > 227 * 1024)
        return 0;
    const long NUT = (H + 15) / 16, NFT = (F + 15) / 16, NKT = (H + 15) / 16, NKT3 = (3 * H + 15) / 16;
    return (NUT * NKT + (NFT + NUT) * NKT3) * 64;
}

}  // namespace caphn

using namespace caphn;

extern "C" {

// *pack_bytes = size of the transposed-weight pack (0: shape not covered -- use caphn_attgru_seq_bwd);
// *work_bytes = size of the scratch buffer for (B, T).
int caphn_attstep_bwd_size(int H, int F, int P, int B, int T, long* pack_bytes, long* work_bytes) {
    if (!pack_bytes || !work_bytes || B < 0) return CAPHN_EINVAL;
    const long n = bw_pack_elems(H, F, P, T < 1 ? 1 : T);
    *pack_bytes = n * 16;
    const int KP = bw_kp(H, F), KP3 = bw_kp3(H);
    *work_bytes = n ? (long)(2 * align256((size_t)B * H * 4) + align256((size_t)2 * B * KP * 2) +
                             2 * align256((size_t)2 * B * KP3 * 2) + align256((size_t)B * T * P * 4))
                    : 0;
    return CAPHN_OK;
}

int caphn_attstep_bwd_pack(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, void* pack,
                           void* stream) {
    if (H < 1 || F < 1 || H > ST_MAXKT * 16 || F > ST_MAXKT * 16 || E < 0 || !pack || ((uintptr_t)pack & 15))
        return CAPHN_EINVAL;
    const int NUT = (H + 15) / 16, NFT = (F + 15) / 16, NKT = (H + 15) / 16, NKT3 = (3 * H + 15) / 16;
    const long total = ((long)NUT * NKT + (long)(NFT + NUT) * NKT3) * 32;
    attbwd_pack_kernel<<<(unsigned)ceil_div(total, 256L), 256, 0, (cudaStream_t)stream>>>(Wih, Whh, Ua, E, F, H, NUT, NFT,
                                                                                         NKT, NKT3, (uint4*)pack, 0, 0);
    CAPHN_RETURN_LAST();
}

// Many-style batch: G transposed-weight packs (each caphn_attstep_bwd_size bytes); group g's W_ih / W_hh start gstride
// floats after group g - 1's.
int caphn_attstep_bwd_pack_grouped(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, int G,
                                   long gstride, void* pack, void* stream) {
    if (H < 1 || F < 1 || H > ST_MAXKT * 16 || F > ST_MAXKT * 16 || E < 0 || G < 1 || !pack || ((uintptr_t)pack & 15))
        return CAPHN_EINVAL;
    const int NUT = (H + 15) / 16, NFT = (F + 15) / 16, NKT = (H + 15) / 16, NKT3 = (3 * H + 15) / 16;
    const long per = ((long)NUT * NKT + (long)(NFT + NUT) * NKT3) * 64;
    attbwd_pack_kernel<<<dim3((unsigned)ceil_div(per / 2, 256L), G), 256, 0, (cudaStream_t)stream>>>(
        Wih, Whh, Ua, E, F, H, NUT, NFT, NKT, NKT3, (uint4*)pack, gstride, per);
    CAPHN_RETURN_LAST();
}

// BPTT of the attention-GRU recurrence over all T steps; same tensors and results as caphn_attgru_seq_bwd, except that
// dK, dva, dbv need not be zero-initialised by the caller (dK is overwritten, dva / dbv are zeroed here).
static int attstep_bwd_impl(const float* dHbm, const float* dattn, const float* Kp, const float* f, const float* attn,
                            const float* Upre, const float* R, const float* Z, const float* Nn, const float* GHN,
                            const float* Hall, const float* va, const void* pack, void* work, float* dGI, float* dGH,
                            float* dU, float* dCTX, float* dK, float* dva, float* dbv, float* dh0, int B, int T, int P,
                            int H, int F, const int* tiles, int ntiles, int tile_rows, void* stream) {
    if (B <= 0 || T <= 0 || bw_pack_elems(H, F, P, T) == 0 || !pack || ((uintptr_t)pack & 15) || !work ||
        ((uintptr_t)work & 255) || ((uintptr_t)Kp & 15) || ((uintptr_t)f & 15))
        return CAPHN_EINVAL;
    const int KP = bw_kp(H, F), KP3 = bw_kp3(H);
    const int NUT = (H + 15) / 16, NFT = (F + 15) / 16, NKT = (H + 15) / 16, NKT3 = (3 * H + 15) / 16;
    const long BH = (long)B * H;
    cudaStream_t st = (cudaStream_t)stream;
    long pb = 0, wb = 0;
    caphn_attstep_bwd_size(H, F, P, B, T, &pb, &wb);
    uint8_t* w8 = (uint8_t*)work;
    float* keep = (float*)w8;                      w8 += align256((size_t)BH * 4);
    float* dhp = (float*)w8;                       w8 += align256((size_t)BH * 4);
    __nv_bfloat16* dusp = (__nv_bfloat16*)w8;      w8 += align256((size_t)2 * B * KP * 2);
    __nv_bfloat16* gisp = (__nv_bfloat16*)w8;      w8 += align256((size_t)2 * B * KP3 * 2);
    __nv_bfloat16* ghsp = (__nv_bfloat16*)w8;      w8 += align256((size_t)2 * B * KP3 * 2);
    float* dS = (float*)w8;
    CAPHN_CHECK(cudaMemsetAsync(work, 0, (size_t)wb, st));       // padding columns of the operand rows must be finite
    CAPHN_CHECK(cudaMemsetAsync(dva, 0, (size_t)H * 4, st));
    CAPHN_CHECK(cudaMemsetAsync(dbv, 0, 4, st));
    const uint4* p0 = (const uint4*)pack;
    const uint4* p1 = p0 + (long)NUT * NKT * 64;
    const uint4* p2 = p1 + (long)NFT * NKT3 * 64;
    int agrid = B < 2 * kNumSMs ? B : 2 * kNumSMs, nbuf = 1;
    int rpc = (B + agrid - 1) / agrid;
    if (2 * (ba_smem(P, H, F, rpc, 1) + 1024) > 227 * 1024) {
        agrid = ba_grid(B, P, H, F); rpc = (B + agrid - 1) / agrid; nbuf = 2;
    }
    const size_t s1 = g1_smem(KP), s2 = g2_smem(KP3), sa = ba_smem(P, H, F, rpc, nbuf), sd = bd_smem(P, H, T);
    if (sa > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(attbwd_gate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1));
    const bool small_tiles = tiles && tile_rows <= G2_NB_SMALL;
    if (tiles && tile_rows > G2_NB) return CAPHN_EINVAL;
    const size_t s2s = g2_smem(KP3, G2_NB_SMALL);
    CAPHN_CHECK(cudaFuncSetAttribute(attbwd_gemm_kernel<G2_NB, G2_PF_BIG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2));
    CAPHN_CHECK(cudaFuncSetAttribute(attbwd_gemm_kernel<G2_NB_SMALL, G2_PF_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2s));
    CAPHN_CHECK(cudaFuncSetAttribute(attbwd_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sa));
    CAPHN_CHECK(cudaFuncSetAttribute(attbwd_dk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sd));
    const int NG1 = ceil_div(NFT, G2_WARPS), NG2 = ceil_div(NUT, G2_WARPS);
    for (int t = T - 1; t >= 0; --t) {
        BwdG1 g1{p0, dusp, dhp, keep, dHbm, R + t * BH, Z + t * BH, Nn + t * BH, GHN + t * BH, Hall + t * BH,
                 dGI + (long)t * B * 3 * H, dGH + (long)t * B * 3 * H, gisp, ghsp, nullptr, B, T, t, H, NUT, NKT, KP, KP3,
                 t == T - 1 ? 0 : 1};
        CAPHN_CHECK(launch_pdl(attbwd_gate_kernel, dim3(NUT, ceil_div(B, G1_NB)), dim3(G1_THREADS), s1, st,
                               t != T - 1, g1));
        ++caphn_launch_counter;
        BwdG2 g2{p1, p2, gisp, ghsp, dCTX + (long)t * B * F, dhp, B, H, F, NUT, NFT, NKT3, KP3, NG1, (const int4*)tiles,
                 pb / 16};
        if (small_tiles) {
            CAPHN_CHECK(launch_pdl(attbwd_gemm_kernel<G2_NB_SMALL, G2_PF_SMALL>, dim3(NG1 + NG2, ntiles), dim3(G2_THREADS), s2s, st, true, g2));
        } else {
            CAPHN_CHECK(launch_pdl(attbwd_gemm_kernel<G2_NB, G2_PF_BIG>, dim3(NG1 + NG2, tiles ? ntiles : ceil_div(B, G2_NB)),
                                   dim3(G2_THREADS), s2, st, true, g2));
        }
        ++caphn_launch_counter;
        BwdA ba{Kp, f, va, dCTX + (long)t * B * F, attn, dattn, Upre + t * BH, dS, dU + t * BH, dusp, dbv,
                B, T, t, P, H, F, KP, rpc, nbuf};
        CAPHN_CHECK(launch_pdl(attbwd_attn_kernel, dim3(agrid), dim3(BA_THREADS), sa, st, true, ba));
        ++caphn_launch_counter;
    }
    BwdG1 g1{p0, dusp, dhp, keep, dHbm, R, Z, Nn, GHN, Hall, dGI, dGH, gisp, ghsp, dh0, B, T, 0, H, NUT, NKT, KP, KP3, 2};
    CAPHN_CHECK(launch_pdl(attbwd_gate_kernel, dim3(NUT, ceil_div(B, G1_NB)), dim3(G1_THREADS), s1, st, true, g1));
    ++caphn_launch_counter;
    BwdD bd{Kp, va, Upre, dS, dK, dva, B, T, P, H};
    const int dgrid = B < kNumSMs ? B : kNumSMs;
    CAPHN_CHECK(launch_pdl(attbwd_dk_kernel, dim3(dgrid), dim3(BD_THREADS), sd, st, true, bd));
    ++caphn_launch_counter;
    return (int)cudaGetLastError();
}

int caphn_attstep_bwd(const float* dHbm, const float* dattn, const float* Kp, const float* f, const float* attn,
                      const float* Upre, const float* R, const float* Z, const float* Nn, const float* GHN,
                      const float* Hall, const float* va, const void* pack, void* work, float* dGI, float* dGH,
                      float* dU, float* dCTX, float* dK, float* dva, float* dbv, float* dh0, int B, int T, int P, int H,
                      int F, void* stream) {
    return attstep_bwd_impl(dHbm, dattn, Kp, f, attn, Upre, R, Z, Nn, GHN, Hall, va, pack, work, dGI, dGH, dU, dCTX, dK, dva,
                            dbv, dh0, B, T, P, H, F, nullptr, 0, 0, stream);
}

// Many-style batch (rows sorted by style group): `tiles` = ntiles records {first row, rows (<= 32), group, 0} for the
// transposed-weight GEMM kernel (the only backward kernel that reads generated weights); pack = the G packs of
// caphn_attstep_bwd_pack_grouped (U_a^T is read from group 0's).
int caphn_attstep_bwd_grouped(const float* dHbm, const float* dattn, const float* Kp, const float* f, const float* attn,
                              const float* Upre, const float* R, const float* Z, const float* Nn, const float* GHN,
                              const float* Hall, const float* va, const void* pack, void* work, float* dGI, float* dGH,
                              float* dU, float* dCTX, float* dK, float* dva, float* dbv, float* dh0, int B, int T, int P,
                              int H, int F, const int* tiles, int ntiles, int tile_rows, void* stream) {
    if (!tiles || ntiles < 1 || tile_rows < 1 || ((uintptr_t)tiles & 15)) return CAPHN_EINVAL;
    return attstep_bwd_impl(dHbm, dattn, Kp, f, attn, Upre, R, Z, Nn, GHN, Hall, va, pack, work, dGI, dGH, dU, dCTX, dK, dva,
                            dbv, dh0, B, T, P, H, F, tiles, ntiles, tile_rows, stream);
}

}  // extern "C"
