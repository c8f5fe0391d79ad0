// Hypernetwork linear layers for a handful of style groups: weight-streaming kernels (HBM-bound).
//
// Replaces the nn.Linear / nn.LeakyReLU calls of HyperNet.forward (reference hypernet_attention.py:111-118,
// hypernet.py:104-111) and their autograd backward.  The layers are y = act(A W^T + b) with A = [G, K] (G = number of
// style groups in flight, 1 in every reference call site) and W = [N, K] with N*K up to ~1e9: the arithmetic intensity
// is 2G flop per weight, so the only thing that matters is streaming W exactly once at HBM speed.
//
// Layout problem solved here: W rows are K elements long and K is rarely a multiple of the 128-bit vector width V
// (4 floats / 8 bf16): K = 11250, 8437, 450 ... so rows are not 16-byte aligned.  Each warp walks a row in
// *address-aligned* vectors; vector q of row n covers k = V*q - m .. V*q - m + V-1 with m = (n*K) mod V.  The activation
// vector is kept in shared memory split into V residue planes (plane r holds a[k] for k mod V == r) so that the V scalar
// reads a lane needs are bank-conflict free for every m.  Edge vectors (first/last of a row) use predicated scalar
// accesses.  Templated on the weight type: float (fp32 mode) or __nv_bfloat16 (bf16 mode: half the bytes; fp32
// activations / accumulation, gradients rounded to bf16 on store).
#include "common.cuh"
#include <stdlib.h>
#include <cuda_bf16.h>

namespace caphn {

constexpr int ROWS_FWD_THREADS = 512;
constexpr int ROWS_BWD_THREADS = 256;

template <typename T> struct WT;
template <> struct WT<float> {
    static constexpr int V = 4;
    static __device__ __forceinline__ void load(const float* p, float* o) {
        const float4 t = ldg_stream4(p);
        o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
    }
    static __device__ __forceinline__ float load1(const float* p) { return ldg_stream1(p); }
    // raw 128-bit vector in registers (unpacked lazily so that more loads can be kept in flight)
    static __device__ __forceinline__ uint4 load_raw(const float* p) {
        const float4 t = ldg_stream4(p);
        return make_uint4(__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w));
    }
    static __device__ __forceinline__ void put_raw(uint4& r, int c, float v) {
        const uint32_t b = __float_as_uint(v);
        if (c == 0) r.x = b; else if (c == 1) r.y = b; else if (c == 2) r.z = b; else r.w = b;
    }
    static __device__ __forceinline__ void unpack(const uint4& t, float* o) {
        o[0] = __uint_as_float(t.x); o[1] = __uint_as_float(t.y); o[2] = __uint_as_float(t.z); o[3] = __uint_as_float(t.w);
    }
    static __device__ __forceinline__ void load_rw(const float* p, float* o) {
        const float4 t = *reinterpret_cast<const float4*>(p);
        o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
    }
    static __device__ __forceinline__ float load1_rw(const float* p) { return *p; }
    static __device__ __forceinline__ void store(float* p, const float* v) {
        stg_stream4(p, make_float4(v[0], v[1], v[2], v[3]));
    }
    static __device__ __forceinline__ void store1(float* p, float v) { *p = v; }
};
template <> struct WT<__nv_bfloat16> {
    static constexpr int V = 8;
    static __device__ __forceinline__ void unpack(const uint4& t, float* o) {
        o[0] = __uint_as_float(t.x << 16); o[1] = __uint_as_float(t.x & 0xffff0000u);
        o[2] = __uint_as_float(t.y << 16); o[3] = __uint_as_float(t.y & 0xffff0000u);
        o[4] = __uint_as_float(t.z << 16); o[5] = __uint_as_float(t.z & 0xffff0000u);
        o[6] = __uint_as_float(t.w << 16); o[7] = __uint_as_float(t.w & 0xffff0000u);
    }
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float* o) {
        uint4 t;
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(t.x), "=r"(t.y), "=r"(t.z), "=r"(t.w) : "l"(p));
        unpack(t, o);
    }
    static __device__ __forceinline__ float load1(const __nv_bfloat16* p) {
        unsigned short u;
        asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(u) : "l"(p));
        return __uint_as_float((uint32_t)u << 16);
    }
    static __device__ __forceinline__ uint4 load_raw(const __nv_bfloat16* p) {
        uint4 t;
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(t.x), "=r"(t.y), "=r"(t.z), "=r"(t.w) : "l"(p));
        return t;
    }
    static __device__ __forceinline__ void put_raw(uint4& r, int c, float v) {   // v is exactly representable in bf16
        const uint32_t b = __float_as_uint(v) >> 16;
        uint32_t& w = (c >> 1) == 0 ? r.x : ((c >> 1) == 1 ? r.y : ((c >> 1) == 2 ? r.z : r.w));
        w = (c & 1) ? ((w & 0x0000ffffu) | (b << 16)) : ((w & 0xffff0000u) | b);
    }
    static __device__ __forceinline__ void load_rw(const __nv_bfloat16* p, float* o) {
        unpack(*reinterpret_cast<const uint4*>(p), o);
    }
    static __device__ __forceinline__ float load1_rw(const __nv_bfloat16* p) { return __bfloat162float(*p); }
    static __device__ __forceinline__ uint32_t pk(float a, float b) {
        uint32_t r;                                        // one cvt.rn.bf16x2.f32: low half = a, high half = b
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
        return r;
    }
    static __device__ __forceinline__ void store(__nv_bfloat16* p, const float* v) {
        const uint32_t a = pk(v[0], v[1]), b = pk(v[2], v[3]), c = pk(v[4], v[5]), d = pk(v[6], v[7]);
        asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d)
                     : "memory");
    }
    static __device__ __forceinline__ void store1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

template <typename T, int GC>
__global__ void __launch_bounds__(ROWS_FWD_THREADS) rows_fwd_kernel(
    const T* __restrict__ W, const float* __restrict__ bias, const float* __restrict__ A, long lda,
    float* __restrict__ Y, long ldy, long N, int K, int KQ, int act, float slope) {
    constexpr int V = WT<T>::V;
    extern __shared__ float As[];  // [GC][V][KQ], plane entries shifted by +1 so index -1 is a readable zero
    const int tid = threadIdx.x;
    for (int i = tid; i < GC * V * KQ; i += ROWS_FWD_THREADS) As[i] = 0.f;
    __syncthreads();
    for (int i = tid; i < GC * K; i += ROWS_FWD_THREADS) {
        const int g = i / K, k = i - g * K;
        As[(g * V + (k % V)) * KQ + 1 + (k / V)] = A[(long)g * lda + k];
    }
    __syncthreads();

    const int lane = tid & 31;
    const long warps_total = (long)gridDim.x * (ROWS_FWD_THREADS / 32);
    for (long n = (long)blockIdx.x * (ROWS_FWD_THREADS / 32) + (tid >> 5); n < N; n += warps_total) {
        const long rowoff = n * (long)K;
        const int m = (int)(rowoff % V);
        const T* wq = W + (rowoff - m);
        const int NQ = (K + m + V - 1) / V;
        int aoff[V];
#pragma unroll
        for (int c = 0; c < V; ++c) {
            const int d = c - m;                           // in (-V, V)
            aoff[c] = ((d + V) % V) * KQ + 1 + (d < 0 ? -1 : 0);
        }
        float acc[GC];
#pragma unroll
        for (int g = 0; g < GC; ++g) acc[g] = 0.f;

        // software pipeline: the raw vectors of the next batch are in flight while the current batch is consumed
        auto fetch = [&](int qb, uint4* raw) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int q = qb + u * 32 + lane;
                raw[u] = make_uint4(0u, 0u, 0u, 0u);
                if (q < NQ) {
                    const int k0 = V * q - m;
                    if (k0 >= 0 && k0 + V - 1 < K) {
                        raw[u] = WT<T>::load_raw(wq + (long)V * q);
                    } else {
#pragma unroll
                        for (int c = 0; c < V; ++c)
                            if (k0 + c >= 0 && k0 + c < K) WT<T>::put_raw(raw[u], c, WT<T>::load1(W + rowoff + k0 + c));
                    }
                }
            }
        };
        uint4 cur[4], nxt[4];
        fetch(0, cur);
        for (int qb = 0; qb < NQ; qb += 128) {
            if (qb + 128 < NQ) fetch(qb + 128, nxt);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int q = qb + u * 32 + lane;
                if (q < NQ) {
                    float w[V];
                    WT<T>::unpack(cur[u], w);
#pragma unroll
                    for (int g = 0; g < GC; ++g) {
                        const float* ag = As + g * V * KQ + q;
#pragma unroll
                        for (int c = 0; c < V; ++c) acc[g] = fmaf(w[c], ag[aoff[c]], acc[g]);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) cur[u] = nxt[u];
        }
#pragma unroll
        for (int g = 0; g < GC; ++g) acc[g] = warp_sum(acc[g]);
        if (lane == 0) {
            const float b = bias ? bias[n] : 0.f;
#pragma unroll
            for (int g = 0; g < GC; ++g) {
                float v = acc[g] + b;
                if (act == 1) v = v > 0.f ? v : v * slope;
                Y[(long)g * ldy + n] = v;
            }
        }
    }
}

// dP[g,n] = dY[g,n] * act'(Y[g,n]);  dbias[n] (+)= sum_g dP[g,n]
__global__ void rows_bwd_prep_kernel(const float* __restrict__ Y, long ldy, const float* __restrict__ dY, long lddy,
                                     float* __restrict__ dP, long ldp, float* __restrict__ dbias, int G, long N,
                                     int act, float slope, int accum_bias) {
    const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float s = 0.f;
    for (int g = 0; g < G; ++g) {
        float d = dY[(long)g * lddy + n];
        if (act == 1) d = Y[(long)g * ldy + n] > 0.f ? d : d * slope;
        dP[(long)g * ldp + n] = d;
        s += d;
    }
    if (dbias) dbias[n] = accum_bias ? dbias[n] + s : s;
}

// One pass over W: dW[n,k] (=|+=) sum_g dP[g,n] A[g,k]   and   dA[g,k] += sum_n dP[g,n] W[n,k]  (dA pre-zeroed).
// A warp owns (block of RB rows) x (strip of 32*QPL aligned vectors): QPL*512 contiguous bytes of a row per access batch
// (the shape that reaches ~95 % of copy bandwidth in the forward kernel).  Rows are visited class by class
// (n mod V == cls) so that a lane sees the same k for every row of the class and keeps its dA partial sums in
// registers; RU rows are in flight per lane (RU*QPL 128-bit loads).
//   SMEM_REDUCE = false ("many strips", large K): adjacent warps take adjacent strips of the same rows (16 KB contiguous
//                 per row across a CTA); every lane flushes its dA partials with global atomics (few per address).
//   SMEM_REDUCE = true  ("few strips", small K => many row blocks): a CTA owns one strip and 8 consecutive row blocks;
//                 the 8 warps' partials are combined in shared memory and leave as ONE atomic per (g,k) per class.
template <typename T, int GC, int QPL, int RU, bool SMEM_REDUCE>
__global__ void __launch_bounds__(ROWS_BWD_THREADS) rows_bwd_kernel(
    const T* __restrict__ W, const float* __restrict__ A, long lda, const float* __restrict__ dP, long ldp,
    T* __restrict__ dW, float* __restrict__ dA, long ldda, long N, int K, int RB, int S, long items, int accum_dw,
    int need_da) {
    constexpr int V = WT<T>::V;
    __shared__ float red[SMEM_REDUCE ? GC * QPL * 32 * V : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // rows n and n' have the same misalignment m = (n*K) mod V iff n == n' (mod V / gcd(K mod V, V))
    int gdiv = K % V;
    { int y = V; while (y) { const int t = gdiv % y; gdiv = y; y = t; } }     // gcd(K mod V, V)  (gcd(0, V) = V)
    const int ncls = V / gdiv;
    const long warps_total = (long)gridDim.x * (ROWS_BWD_THREADS / 32);
    long item = SMEM_REDUCE ? 0 : (long)blockIdx.x * (ROWS_BWD_THREADS / 32) + warp;
    const long item_end = SMEM_REDUCE ? 1 : items;
    for (; item < item_end; item += warps_total) {
        long rb; int s;
        if (SMEM_REDUCE) { s = blockIdx.x % S; rb = (long)(blockIdx.x / S) * (ROWS_BWD_THREADS / 32) + warp; }
        else { rb = item / S; s = (int)(item - rb * S); }
        const long row0 = rb * RB;
        const long row1 = (row0 + RB < N) ? row0 + RB : N;
        for (int cls = 0; cls < ncls; ++cls) {
            const int m = (cls * (K % V)) % V;
            int k0[QPL];
            bool full[QPL];
            float a[GC][QPL][V], acc[GC][QPL][V];
#pragma unroll
            for (int u = 0; u < QPL; ++u) {
                k0[u] = V * ((s * QPL + u) * 32 + lane) - m;
                full[u] = (k0[u] >= 0) && (k0[u] + V - 1 < K);
#pragma unroll
                for (int g = 0; g < GC; ++g)
#pragma unroll
                    for (int c = 0; c < V; ++c) {
                        const int k = k0[u] + c;
                        a[g][u][c] = (k >= 0 && k < K) ? A[(long)g * lda + k] : 0.f;
                        acc[g][u][c] = 0.f;
                    }
            }
            for (long nb = row0 + cls; nb < row1; nb += (long)RU * ncls) {
                uint4 raw[RU][QPL];   // raw 128-bit vectors: RU*QPL loads in flight per lane, unpacked when consumed
#pragma unroll
                for (int r = 0; r < RU; ++r) {
                    const long n = nb + (long)r * ncls;
#pragma unroll
                    for (int u = 0; u < QPL; ++u) {
                        raw[r][u] = make_uint4(0u, 0u, 0u, 0u);
                        if (n < row1) {
                            const T* p = W + n * (long)K + k0[u];
                            if (full[u]) {
                                raw[r][u] = WT<T>::load_raw(p);
                            } else {
#pragma unroll
                                for (int c = 0; c < V; ++c)
                                    if (k0[u] + c >= 0 && k0[u] + c < K) WT<T>::put_raw(raw[r][u], c, WT<T>::load1(p + c));
                            }
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < RU; ++r) {
                    const long n = nb + (long)r * ncls;
                    if (n < row1) {
                        float dp[GC];
#pragma unroll
                        for (int g = 0; g < GC; ++g) dp[g] = __ldg(dP + (long)g * ldp + n);
#pragma unroll
                        for (int u = 0; u < QPL; ++u) {
                            float dw[V], wv[V];
                            WT<T>::unpack(raw[r][u], wv);
#pragma unroll
                            for (int c = 0; c < V; ++c) dw[c] = 0.f;
#pragma unroll
                            for (int g = 0; g < GC; ++g)
#pragma unroll
                                for (int c = 0; c < V; ++c) {
                                    acc[g][u][c] = fmaf(dp[g], wv[c], acc[g][u][c]);
                                    dw[c] = fmaf(dp[g], a[g][u][c], dw[c]);
                                }
                            if (!dW) continue;       // dA-only pass (the weight gradient stays in its rank-G form)
                            T* o = dW + n * (long)K + k0[u];
                            if (full[u]) {
                                if (accum_dw) {
                                    float old[V];
                                    WT<T>::load_rw(o, old);
#pragma unroll
                                    for (int c = 0; c < V; ++c) dw[c] += old[c];
                                }
                                WT<T>::store(o, dw);
                            } else {
#pragma unroll
                                for (int c = 0; c < V; ++c)
                                    if (k0[u] + c >= 0 && k0[u] + c < K)
                                        WT<T>::store1(o + c, accum_dw ? WT<T>::load1_rw(o + c) + dw[c] : dw[c]);
                            }
                        }
                    }
                }
            }
            if (need_da) {
                if (SMEM_REDUCE) {   // (uniform across the CTA: safe to synchronise)
                    for (int i = threadIdx.x; i < GC * QPL * 32 * V; i += ROWS_BWD_THREADS) red[i] = 0.f;
                    __syncthreads();
#pragma unroll
                    for (int g = 0; g < GC; ++g)
#pragma unroll
                        for (int u = 0; u < QPL; ++u)
#pragma unroll
                            for (int c = 0; c < V; ++c)
                                if (acc[g][u][c] != 0.f) atomicAdd(&red[((g * QPL + u) * 32 + lane) * V + c], acc[g][u][c]);
                    __syncthreads();
                    for (int i = threadIdx.x; i < GC * QPL * 32 * V; i += ROWS_BWD_THREADS) {
                        const int c = i % V, ln = (i / V) & 31, u = (i / (V * 32)) % QPL, g = i / (QPL * 32 * V);
                        const int k = V * ((s * QPL + u) * 32 + ln) - m + c;
                        const float v = red[i];
                        if (k >= 0 && k < K && v != 0.f) atomicAdd(dA + (long)g * ldda + k, v);
                    }
                    __syncthreads();
                } else {
#pragma unroll
                    for (int g = 0; g < GC; ++g)
#pragma unroll
                        for (int u = 0; u < QPL; ++u)
#pragma unroll
                            for (int c = 0; c < V; ++c) {
                                const int k = k0[u] + c;
                                if (k >= 0 && k < K && acc[g][u][c] != 0.f) atomicAdd(dA + (long)g * ldda + k, acc[g][u][c]);
                            }
                }
            }
        }
    }
}

template <typename T, int GC>
static int launch_rows_fwd(const T* W, const float* bias, const float* A, long lda, float* Y, long ldy, long N,
                           int K, int act, float slope, cudaStream_t st) {
    constexpr int V = WT<T>::V;
    const int KQ = (K + V - 1) / V + 2;
    const size_t smem = (size_t)GC * V * KQ * sizeof(float);
    if (smem > 227 * 1024) return CAPHN_EINVAL;
    CAPHN_CHECK(cudaFuncSetAttribute(rows_fwd_kernel<T, GC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = (int)((227 * 1024) / (smem + 1024));
    if (occ > 4) occ = 4;
    if (occ < 1) occ = 1;
    long blocks = (N + 15) / 16;
    if (blocks > (long)kNumSMs * occ) blocks = (long)kNumSMs * occ;
    if (blocks < 1) blocks = 1;
    rows_fwd_kernel<T, GC><<<(unsigned)blocks, ROWS_FWD_THREADS, smem, st>>>(W, bias, A, lda, Y, ldy, N, K, KQ, act,
                                                                            slope);
    CAPHN_RETURN_LAST();
}

template <typename T, int GC, int QPL, int RU>
static int launch_rows_bwd(const T* W, const float* A, long lda, const float* dP, long ldp, T* dW, float* dA,
                           long ldda, long N, int K, int accum_dw, int need_da, cudaStream_t st) {
    constexpr int V = WT<T>::V;
    constexpr int WPB = ROWS_BWD_THREADS / 32;
    const int S = ((K + 2 * (V - 1)) / V + 32 * QPL - 1) / (32 * QPL);
    int gdiv = K % V;
    { int y = V; while (y) { const int t = gdiv % y; gdiv = y; y = t; } }
    const int ncls = V / gdiv;
    if ((long)N * K < (1L << 22)) {
        // tiny matrices (hn_base, the bias heads): a chain of dependent HBM round trips, not bandwidth.  One batch of
        // RU rows per misalignment class per warp (every load of a warp is issued at once), as many warps as that
        // gives, and the CTA-level reduction so the dA atomics stay at N/(8 RU ncls) per address.
        const int RB = RU * ncls;
        const long groups = (N + (long)RB * WPB - 1) / ((long)RB * WPB);
        rows_bwd_kernel<T, GC, QPL, RU, true><<<(unsigned)(groups * S), ROWS_BWD_THREADS, 0, st>>>(
            W, A, lda, dP, ldp, dW, dA, ldda, N, K, RB, S, 0, accum_dw, need_da);
    } else if (S >= 8) {
        // many strips: warp-granular work items
        // >= 32 rows per misalignment class per work item keeps the dA atomics <= ~10 % of the memory instructions
        int RB = 128 * (ncls > 4 ? ncls / 4 : 1);
        const int rb_min = 32 * ncls;
        while (RB > rb_min && RB > 16 && ((N + RB - 1) / RB) * S < 8L * kNumSMs * WPB) RB >>= 1;
        const long items = ((N + RB - 1) / RB) * S;
        long blocks = (items + WPB - 1) / WPB;
        const long cap = (long)kNumSMs * 64;
        if (blocks > cap) blocks = cap;
        rows_bwd_kernel<T, GC, QPL, RU, false><<<(unsigned)blocks, ROWS_BWD_THREADS, 0, st>>>(
            W, A, lda, dP, ldp, dW, dA, ldda, N, K, RB, S, items, accum_dw, need_da);
    } else {
        // few strips: rows per warp as large as possible (fewer atomics) while still giving every SM a few CTAs
        int RB = 256;
        while (RB > 32 && ((N + (long)RB * WPB - 1) / ((long)RB * WPB)) * S < 4L * kNumSMs) RB >>= 1;
        const long groups = (N + (long)RB * WPB - 1) / ((long)RB * WPB);
        const long blocks = groups * S;
        if (blocks > 0x7fffffffL) return CAPHN_EINVAL;
        rows_bwd_kernel<T, GC, QPL, RU, true><<<(unsigned)blocks, ROWS_BWD_THREADS, 0, st>>>(
            W, A, lda, dP, ldp, dW, dA, ldda, N, K, RB, S, 0, accum_dw, need_da);
    }
    CAPHN_RETURN_LAST();
}

template <typename T>
static int rows_linear_fwd_t(const T* W, const float* bias, const float* A, long lda, float* Y, long ldy, int G,
                             long N, long K, int act, float slope, cudaStream_t st) {
    constexpr int V = WT<T>::V;
    if (N <= 0 || K <= 0 || G <= 0 || G > 8 || ((uintptr_t)W & 15) || K > (1 << 28)) return CAPHN_EINVAL;
    const size_t per_g = (size_t)V * ((K + V - 1) / V + 2) * sizeof(float);
    int g0 = 0;
    while (g0 < G) {
        int gc = G - g0 >= 8 ? 8 : (G - g0 >= 4 ? 4 : (G - g0 >= 2 ? 2 : 1));
        while (gc > 1 && gc * per_g > 200 * 1024) gc >>= 1;
        int rc;
        const float* Ag = A + (long)g0 * lda;
        float* Yg = Y + (long)g0 * ldy;
        switch (gc) {
            case 8: rc = launch_rows_fwd<T, 8>(W, bias, Ag, lda, Yg, ldy, N, (int)K, act, slope, st); break;
            case 4: rc = launch_rows_fwd<T, 4>(W, bias, Ag, lda, Yg, ldy, N, (int)K, act, slope, st); break;
            case 2: rc = launch_rows_fwd<T, 2>(W, bias, Ag, lda, Yg, ldy, N, (int)K, act, slope, st); break;
            default: rc = launch_rows_fwd<T, 1>(W, bias, Ag, lda, Yg, ldy, N, (int)K, act, slope, st); break;
        }
        if (rc) return rc;
        g0 += gc;
    }
    return CAPHN_OK;
}

template <typename T>
static int rows_linear_bwd_t(const T* W, const float* A, long lda, const float* Y, long ldy, const float* dY,
                             long lddy, float* dP, T* dW, float* dbias, float* dA, long ldda, int G, long N, long K,
                             int act, float slope, cudaStream_t st) {
    if (N <= 0 || K <= 0 || G <= 0 || G > 64 || ((uintptr_t)W & 15) || (dW && ((uintptr_t)dW & 15)) || K > (1 << 28))
        return CAPHN_EINVAL;
    rows_bwd_prep_kernel<<<ceil_div(N, 256), 256, 0, st>>>(Y, ldy, dY, lddy, dP, N, dbias, G, N, act, slope, 0);
    CAPHN_LAUNCH_CHECK();
    if (!dW && !dA) return CAPHN_OK;
    constexpr bool F32 = (WT<T>::V == 4);
    int g0 = 0;
    while (g0 < G) {
        const int gc = G - g0 >= 4 ? 4 : (G - g0 >= 2 ? 2 : 1);
        const float* Ag = A + (long)g0 * lda;
        const float* dPg = dP + (long)g0 * N;
        float* dAg = dA ? dA + (long)g0 * ldda : nullptr;
        const int acc = g0 > 0, nda = dA != nullptr;
        int rc;
        // vectors per lane / rows in flight chosen so that the register tile stays <= 128 registers
        if constexpr (F32) {
            switch (gc) {
                case 4: rc = launch_rows_bwd<T, 4, 1, 4>(W, Ag, lda, dPg, N, dW, dAg, ldda, N, (int)K, acc, nda, st); break;
                case 2: rc = launch_rows_bwd<T, 2, 2, 2>(W, Ag, lda, dPg, N, dW, dAg, ldda, N, (int)K, acc, nda, st); break;
                default: rc = launch_rows_bwd<T, 1, 4, 2>(W, Ag, lda, dPg, N, dW, dAg, ldda, N, (int)K, acc, nda, st); break;
            }
        } else {
            switch (gc) {
                case 4: rc = launch_rows_bwd<T, 4, 1, 2>(W, Ag, lda, dPg, N, dW, dAg, ldda, N, (int)K, acc, nda, st); break;
                case 2: rc = launch_rows_bwd<T, 2, 1, 4>(W, Ag, lda, dPg, N, dW, dAg, ldda, N, (int)K, acc, nda, st); break;
                default: rc = launch_rows_bwd<T, 1, 2, 4>(W, Ag, lda, dPg, N, dW, dAg, ldda, N, (int)K, acc, nda, st); break;
            }
        }
        if (rc) return rc;
        g0 += gc;
    }
    return CAPHN_OK;
}

}  // namespace caphn

using namespace caphn;

extern "C" {

// Y[g, n] = act(sum_k A[g*lda + k] * W[n*K + k] + bias[n]),  g < G <= 8, act: 0 none, 1 LeakyReLU(slope).
// W must be 16-byte aligned.  Streams W once.
int caphn_rows_linear_fwd(const float* W, const float* bias, const float* A, long lda, float* Y, long ldy, int G,
                          long N, long K, int act, float slope, void* stream) {
    return rows_linear_fwd_t<float>(W, bias, A, lda, Y, ldy, G, N, K, act, slope, (cudaStream_t)stream);
}

// Backward of caphn_rows_linear_fwd.  Y is the forward output (needed only for act == 1), dY its gradient.
//   dP (scratch, [G, N] dense) <- dY * act'(Y);  dbias[n] = sum_g dP;  dW[n,k] = sum_g dP[g,n] A[g,k];
//   dA[g,k] += sum_n dP[g,n] W[n,k]   (dA must be zero-initialised by the caller; pass NULL to skip).
// dW / dbias may be NULL.  dW == NULL with dA != NULL is the dA-only pass (W streamed once, nothing W-sized written):
// the caller keeps the weight gradient in its rank-G form (dP, A) -- see caphn_adam_step_lowrank.
int caphn_rows_linear_bwd(const float* W, const float* A, long lda, const float* Y, long ldy, const float* dY,
                          long lddy, float* dP, float* dW, float* dbias, float* dA, long ldda, int G, long N, long K,
                          int act, float slope, void* stream) {
    return rows_linear_bwd_t<float>(W, A, lda, Y, ldy, dY, lddy, dP, dW, dbias, dA, ldda, G, N, K, act, slope,
                                    (cudaStream_t)stream);
}

// bf16-weight variants (bf16 mode): W, dW are __nv_bfloat16 [N,K]; bias, A, Y, dY, dP, dbias, dA stay fp32;
// accumulation in fp32, dW rounded to bf16 (round-to-nearest-even) on store.  Half the HBM bytes of the fp32 kernels.
int caphn_rows_linear_fwd_bf16(const void* W, const float* bias, const float* A, long lda, float* Y, long ldy, int G,
                               long N, long K, int act, float slope, void* stream) {
    return rows_linear_fwd_t<__nv_bfloat16>((const __nv_bfloat16*)W, bias, A, lda, Y, ldy, G, N, K, act, slope,
                                            (cudaStream_t)stream);
}
int caphn_rows_linear_bwd_bf16(const void* W, const float* A, long lda, const float* Y, long ldy, const float* dY,
                               long lddy, float* dP, void* dW, float* dbias, float* dA, long ldda, int G, long N,
                               long K, int act, float slope, void* stream) {
    return rows_linear_bwd_t<__nv_bfloat16>((const __nv_bfloat16*)W, A, lda, Y, ldy, dY, lddy, dP, (__nv_bfloat16*)dW,
                                            dbias, dA, ldda, G, N, K, act, slope, (cudaStream_t)stream);
}

}  // extern "C"
