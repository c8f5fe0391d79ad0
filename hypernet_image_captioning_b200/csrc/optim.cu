// Optimizer step for the hypernet parameters (SURVEY.md §8(f) rank 1): torch.optim.Adam as configured by the reference
// (cc_train_hypernet.py:110-122, hypernet.py:116-123: Adam(params, lr), default betas/eps, no weight decay) together
// with Lightning's gradient_clip_val=5. (cc_train_hypernet.py:405: torch.nn.utils.clip_grad_norm_ over all parameters).
//
// The head parameters are 6.46 GB (pooled) / 0.58 GB (attention) in fp32, so the step is pure HBM streaming: per
// element 16 bytes read (p, g, m, v) + 12 written (p, m, v).  One pass, 128-bit vectors, the clip coefficient applied
// to the gradient on the fly (read from a device scalar: no host synchronisation, the gradients themselves are left
// untouched), the global norm accumulated in double by a separate read-only pass over the gradients.
#include "common.cuh"
#include <cuda_bf16.h>
#include <math.h>

namespace caphn {

// p, m, v are rewritten by the same kernel: a coherent (non-.nc) streaming load
__device__ __forceinline__ float4 ld_rw4(const float4* p) {
    float4 r;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

constexpr int OPT_THREADS = 256;
constexpr int OPT_UNROLL = 4;      // float4 per thread in flight

__global__ void __launch_bounds__(OPT_THREADS) sumsq_kernel(const float* __restrict__ x, long n, double* __restrict__ out) {
    const long n4 = n >> 2;
    const float4* x4 = reinterpret_cast<const float4*>(x);
    float acc[OPT_UNROLL] = {0.f, 0.f, 0.f, 0.f};
    const long stride = (long)gridDim.x * OPT_THREADS;
    long i = (long)blockIdx.x * OPT_THREADS + threadIdx.x;
    for (; i + (OPT_UNROLL - 1) * stride < n4; i += OPT_UNROLL * stride) {
        float4 v[OPT_UNROLL];
#pragma unroll
        for (int e = 0; e < OPT_UNROLL; ++e) v[e] = ldg_stream4(reinterpret_cast<const float*>(x4 + i + e * stride));
#pragma unroll
        for (int e = 0; e < OPT_UNROLL; ++e)
            acc[e] += v[e].x * v[e].x + v[e].y * v[e].y + v[e].z * v[e].z + v[e].w * v[e].w;
    }
    for (; i < n4; i += stride) {
        const float4 v = ldg_stream4(reinterpret_cast<const float*>(x4 + i));
        acc[0] += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) { const float t = x[(n4 << 2) + threadIdx.x]; acc[1] += t * t; }
    double s = (double)acc[0] + (double)acc[1] + (double)acc[2] + (double)acc[3];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double ws[OPT_THREADS / 32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < OPT_THREADS / 32; ++w) t += ws[w];
        atomicAdd(out, t);
    }
}

// coef = min(1, max_norm / (||g|| + 1e-6))    (torch.nn.utils.clip_grad_norm_)
__global__ void clip_coef_kernel(const double* __restrict__ sumsq, float max_norm, float* __restrict__ coef,
                                 float* __restrict__ norm_out) {
    const float norm = (float)sqrt(*sumsq);
    const float c = max_norm / (norm + 1e-6f);
    *coef = c < 1.f ? c : 1.f;
    if (norm_out) *norm_out = norm;
}

struct AdamArgs {
    float* p; const float* g; float* m; float* v;
    long n;
    float beta2, omb1, omb2, eps, weight_decay, step_size, bc2_sqrt;   // omb = 1 - beta, rounded from double like torch does
    const float* gscale;     // device scalar multiplied into the gradient (clip coefficient), or null
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamArgs& a, float gs) {
    g *= gs;
    if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
    m = fmaf(a.omb1, g - m, m);                              // exp_avg.lerp_(grad, 1 - beta1)
    v = fmaf(a.omb2, g * g, v * a.beta2);                    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
    p -= a.step_size * (m / denom);                          // param.addcdiv_(exp_avg, denom, value=-lr / bias_correction1)
}

__global__ void __launch_bounds__(OPT_THREADS) adam_kernel(const AdamArgs a) {
    const float gs = a.gscale ? *a.gscale : 1.f;
    const long n4 = a.n >> 2;
    float4* p4 = reinterpret_cast<float4*>(a.p);
    float4* m4 = reinterpret_cast<float4*>(a.m);
    float4* v4 = reinterpret_cast<float4*>(a.v);
    const float4* g4 = reinterpret_cast<const float4*>(a.g);
    const long stride = (long)gridDim.x * OPT_THREADS;
    for (long i = (long)blockIdx.x * OPT_THREADS + threadIdx.x; i < n4; i += 2 * stride) {
        const bool two = i + stride < n4;
        const long i2 = two ? i + stride : i;
        // 8 independent 128-bit loads in flight per thread
        float4 p0 = ld_rw4(p4 + i), g0 = ldg_stream4(reinterpret_cast<const float*>(g4 + i));
        float4 m0 = ld_rw4(m4 + i), v0 = ld_rw4(v4 + i);
        float4 p1 = ld_rw4(p4 + i2), g1 = ldg_stream4(reinterpret_cast<const float*>(g4 + i2));
        float4 m1 = ld_rw4(m4 + i2), v1 = ld_rw4(v4 + i2);
        adam_one(p0.x, g0.x, m0.x, v0.x, a, gs); adam_one(p0.y, g0.y, m0.y, v0.y, a, gs);
        adam_one(p0.z, g0.z, m0.z, v0.z, a, gs); adam_one(p0.w, g0.w, m0.w, v0.w, a, gs);
        stg_stream4(reinterpret_cast<float*>(p4 + i), p0);
        stg_stream4(reinterpret_cast<float*>(m4 + i), m0);
        stg_stream4(reinterpret_cast<float*>(v4 + i), v0);
        if (two) {
            adam_one(p1.x, g1.x, m1.x, v1.x, a, gs); adam_one(p1.y, g1.y, m1.y, v1.y, a, gs);
            adam_one(p1.z, g1.z, m1.z, v1.z, a, gs); adam_one(p1.w, g1.w, m1.w, v1.w, a, gs);
            stg_stream4(reinterpret_cast<float*>(p4 + i2), p1);
            stg_stream4(reinterpret_cast<float*>(m4 + i2), m1);
            stg_stream4(reinterpret_cast<float*>(v4 + i2), v1);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (a.n & 3)) {
        const long i = (n4 << 2) + threadIdx.x;
        float p = a.p[i], m = a.m[i], v = a.v[i];
        adam_one(p, a.g[i], m, v, a, gs);
        a.p[i] = p; a.m[i] = m; a.v[i] = v;
    }
}

// ---- rank-G weight gradient: g[n,k] = sum_q dP[q,n] A[q,k] formed on the fly (never materialised) ----------------------
// The hypernet head layer y = a W^T has dW = dP^T a with G = #style groups rows (1 at every reference call site), so the
// 6.46 GB gradient of the benchmark model is a 0.4 MB pair (dP, a).  The update reads p, m, v and writes p, m, v: 24
// bytes per parameter instead of 8 (backward writes dW, norm pass reads it) + 28 (Adam).
constexpr int LR_MAXG = 4;

struct AdamLrArgs {
    float* p; float* m; float* v;
    const float* dP; long ldp; const float* A; long lda;
    int G; long N; int K;
    float beta2, omb1, omb2, eps, weight_decay, step_size, bc2_sqrt;
    const float* gscale;
};

template <int G>
__device__ __forceinline__ float lowrank_g(const AdamLrArgs& a, long n, int k) {
    float g = 0.f;
#pragma unroll
    for (int q = 0; q < G; ++q) g = fmaf(__ldg(a.dP + q * a.ldp + n), __ldg(a.A + q * a.lda + k), g);
    return g;
}

constexpr int LR_UNR = 4;     // float4 triples (p, m, v) in flight per thread: 12 x 16 B

template <int G>
__global__ void __launch_bounds__(OPT_THREADS) adam_lowrank_kernel(const AdamLrArgs a) {
    const float gs = a.gscale ? *a.gscale : 1.f;
    const long total = a.N * a.K;
    const long n4 = total >> 2;
    float4* p4 = reinterpret_cast<float4*>(a.p);
    float4* m4 = reinterpret_cast<float4*>(a.m);
    float4* v4 = reinterpret_cast<float4*>(a.v);
    AdamArgs h{nullptr, nullptr, nullptr, nullptr, 0, a.beta2, a.omb1, a.omb2, a.eps, a.weight_decay, a.step_size, a.bc2_sqrt,
               nullptr};
    const long stride = (long)gridDim.x * OPT_THREADS;
    // (row, column) of this thread's float4s, advanced incrementally: 64-bit divisions only once per thread
    const long i0 = (long)blockIdx.x * OPT_THREADS + threadIdx.x;
    long nn[LR_UNR];
    int kk[LR_UNR];
#pragma unroll
    for (int u = 0; u < LR_UNR; ++u) {
        const long e = (i0 + u * stride) << 2;
        nn[u] = e / a.K;
        kk[u] = (int)(e - nn[u] * a.K);
    }
    const long step4 = (stride * LR_UNR) << 2;
    const long dq = step4 / a.K;
    const int dr = (int)(step4 - dq * a.K);
    for (long i = i0; i < n4; i += LR_UNR * stride) {
        float4 pv[LR_UNR], mv[LR_UNR], vv[LR_UNR];
        long idx[LR_UNR];
#pragma unroll
        for (int u = 0; u < LR_UNR; ++u) {
            idx[u] = i + u * stride < n4 ? i + u * stride : i;     // clamped duplicates are loaded but not stored
            pv[u] = ld_rw4(p4 + idx[u]); mv[u] = ld_rw4(m4 + idx[u]); vv[u] = ld_rw4(v4 + idx[u]);
        }
#pragma unroll
        for (int u = 0; u < LR_UNR; ++u) {
            const long n0 = nn[u]; const int k0 = kk[u];
            nn[u] += dq; kk[u] += dr; if (kk[u] >= a.K) { kk[u] -= a.K; ++nn[u]; }
            // a slot past the end has (n0, k0) beyond row N - 1: dP must not be read there
            if (u == 0 || i + u * stride < n4) {
                float g[4];
                long n = n0; int k = k0;
#pragma unroll
                for (int c = 0; c < 4; ++c) { g[c] = lowrank_g<G>(a, n, k); if (++k == a.K) { k = 0; ++n; } }
                adam_one(pv[u].x, g[0], mv[u].x, vv[u].x, h, gs); adam_one(pv[u].y, g[1], mv[u].y, vv[u].y, h, gs);
                adam_one(pv[u].z, g[2], mv[u].z, vv[u].z, h, gs); adam_one(pv[u].w, g[3], mv[u].w, vv[u].w, h, gs);
                stg_stream4(reinterpret_cast<float*>(p4 + idx[u]), pv[u]);
                stg_stream4(reinterpret_cast<float*>(m4 + idx[u]), mv[u]);
                stg_stream4(reinterpret_cast<float*>(v4 + idx[u]), vv[u]);
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (total & 3)) {
        const long e = (n4 << 2) + threadIdx.x;
        const long n = e / a.K;
        float p = a.p[e], m = a.m[e], v = a.v[e];
        adam_one(p, lowrank_g<G>(a, n, (int)(e - n * a.K)), m, v, h, gs);
        a.p[e] = p; a.m[e] = m; a.v[e] = v;
    }
}

// out[q*G + r] += sum_i X[q*ld + i] X[r*ld + i]     (G <= LR_MAXG)
__global__ void __launch_bounds__(OPT_THREADS) gram_kernel(const float* __restrict__ X, long ld, int G, long L,
                                                           double* __restrict__ out) {
    float acc[LR_MAXG][LR_MAXG];
#pragma unroll
    for (int q = 0; q < LR_MAXG; ++q)
#pragma unroll
        for (int r = 0; r < LR_MAXG; ++r) acc[q][r] = 0.f;
    for (long i = (long)blockIdx.x * OPT_THREADS + threadIdx.x; i < L; i += (long)gridDim.x * OPT_THREADS) {
        float x[LR_MAXG];
#pragma unroll
        for (int q = 0; q < LR_MAXG; ++q) x[q] = q < G ? X[q * ld + i] : 0.f;
#pragma unroll
        for (int q = 0; q < LR_MAXG; ++q)
#pragma unroll
            for (int r = 0; r < LR_MAXG; ++r) acc[q][r] = fmaf(x[q], x[r], acc[q][r]);
    }
    __shared__ double ws[OPT_THREADS / 32];
#pragma unroll
    for (int q = 0; q < LR_MAXG; ++q)
#pragma unroll
        for (int r = 0; r < LR_MAXG; ++r) {
            if (q >= G || r >= G) continue;                 // uniform
            double s = (double)acc[q][r];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
            __syncthreads();
            if (threadIdx.x == 0) {
                double t = 0.0;
                for (int w = 0; w < OPT_THREADS / 32; ++w) t += ws[w];
                atomicAdd(out + q * G + r, t);
            }
            __syncthreads();
        }
}

// *sumsq += || sum_q dP_q (x) A_q ||_F^2 = sum_{q,r} (dP_q . dP_r)(A_q . A_r)
__global__ void sumsq_lowrank_kernel(const double* __restrict__ gp, const double* __restrict__ ga, int G,
                                     double* __restrict__ sumsq) {
    double s = 0.0;
    for (int i = 0; i < G * G; ++i) s += gp[i] * ga[i];
    atomicAdd(sumsq, s);
}

static inline int opt_grid(long n4) {
    long blocks = (n4 + (long)OPT_THREADS * 2 - 1) / ((long)OPT_THREADS * 2);
    const long cap = (long)kNumSMs * 16;            // 16 resident CTAs of 256 threads per SM x 148: grid-stride beyond that
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace caphn

using namespace caphn;

// ---- bf16 parameters with fp32 master weights (bf16 mode: hypernet.set_precision("bf16")) ------------------------------
// The streaming kernels read bf16 head weights and write bf16 gradients; the optimizer keeps the fp32 master copy and the
// Adam moments (fp32), reads the bf16 gradient (8 values per 128-bit load) and writes the master weight and its bf16
// rounding.  30 bytes per parameter: g 2 + master/m/v 12 read, master/m/v 12 + p 2 written (+ 2 for the norm pass).
__global__ void __launch_bounds__(OPT_THREADS) sumsq_bf16_kernel(const __nv_bfloat16* __restrict__ x, long n,
                                                                  double* __restrict__ out) {
    const long n8 = n >> 3;
    const uint4* x8 = reinterpret_cast<const uint4*>(x);
    float acc = 0.f;
    const long stride = (long)gridDim.x * OPT_THREADS;
    for (long i = (long)blockIdx.x * OPT_THREADS + threadIdx.x; i < n8; i += stride) {
        const uint4 u = x8[i];
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float a = __uint_as_float(w[e] << 16), b = __uint_as_float(w[e] & 0xffff0000u);
            acc += a * a + b * b;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 7)) { const float t = __bfloat162float(x[(n8 << 3) + threadIdx.x]); acc += t * t; }
    double s = (double)acc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double ws[OPT_THREADS / 32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < OPT_THREADS / 32; ++w) t += ws[w];
        atomicAdd(out, t);
    }
}

struct AdamBf16Args {
    __nv_bfloat16* p; const __nv_bfloat16* g; float* master; float* m; float* v;
    long n;
    AdamArgs h;     // hyper-parameters (pointer fields unused)
};

__global__ void __launch_bounds__(OPT_THREADS) adam_bf16_kernel(const AdamBf16Args a) {
    const float gs = a.h.gscale ? *a.h.gscale : 1.f;
    const long n8 = a.n >> 3;
    const long stride = (long)gridDim.x * OPT_THREADS;
    for (long i = (long)blockIdx.x * OPT_THREADS + threadIdx.x; i < n8; i += stride) {
        const uint4 gu = *reinterpret_cast<const uint4*>(a.g + i * 8);
        float4 w0 = ld_rw4(reinterpret_cast<float4*>(a.master) + 2 * i), w1 = ld_rw4(reinterpret_cast<float4*>(a.master) + 2 * i + 1);
        float4 m0 = ld_rw4(reinterpret_cast<float4*>(a.m) + 2 * i), m1 = ld_rw4(reinterpret_cast<float4*>(a.m) + 2 * i + 1);
        float4 v0 = ld_rw4(reinterpret_cast<float4*>(a.v) + 2 * i), v1 = ld_rw4(reinterpret_cast<float4*>(a.v) + 2 * i + 1);
        const uint32_t gw[4] = {gu.x, gu.y, gu.z, gu.w};
        float g[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) { g[2 * e] = __uint_as_float(gw[e] << 16); g[2 * e + 1] = __uint_as_float(gw[e] & 0xffff0000u); }
        adam_one(w0.x, g[0], m0.x, v0.x, a.h, gs); adam_one(w0.y, g[1], m0.y, v0.y, a.h, gs);
        adam_one(w0.z, g[2], m0.z, v0.z, a.h, gs); adam_one(w0.w, g[3], m0.w, v0.w, a.h, gs);
        adam_one(w1.x, g[4], m1.x, v1.x, a.h, gs); adam_one(w1.y, g[5], m1.y, v1.y, a.h, gs);
        adam_one(w1.z, g[6], m1.z, v1.z, a.h, gs); adam_one(w1.w, g[7], m1.w, v1.w, a.h, gs);
        stg_stream4(a.master + 8 * i, w0); stg_stream4(a.master + 8 * i + 4, w1);
        stg_stream4(a.m + 8 * i, m0); stg_stream4(a.m + 8 * i + 4, m1);
        stg_stream4(a.v + 8 * i, v0); stg_stream4(a.v + 8 * i + 4, v1);
        const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        uint4 pu;
        uint32_t* pw = reinterpret_cast<uint32_t*>(&pu);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const __nv_bfloat16 lo = __float2bfloat16_rn(w[2 * e]), hi = __float2bfloat16_rn(w[2 * e + 1]);
            pw[e] = (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
        }
        *reinterpret_cast<uint4*>(a.p + i * 8) = pu;
    }
    if (blockIdx.x == 0 && threadIdx.x < (a.n & 7)) {
        const long i = (n8 << 3) + threadIdx.x;
        float w = a.master[i], m = a.m[i], v = a.v[i];
        adam_one(w, __bfloat162float(a.g[i]), m, v, a.h, gs);
        a.master[i] = w; a.m[i] = m; a.v[i] = v;
        a.p[i] = __float2bfloat16_rn(w);
    }
}

extern "C" {

// *sumsq (double, device) += sum_i x[i]^2.  x must be 16-byte aligned.
int caphn_sumsq(const float* x, long n, double* sumsq, void* stream) {
    if (n < 0 || !sumsq || ((uintptr_t)x & 15)) return CAPHN_EINVAL;
    if (n == 0) return CAPHN_OK;
    sumsq_kernel<<<opt_grid(n >> 2), OPT_THREADS, 0, (cudaStream_t)stream>>>(x, n, sumsq);
    CAPHN_RETURN_LAST();
}

// *coef = min(1, max_norm / (sqrt(*sumsq) + 1e-6)); *norm (optional) = sqrt(*sumsq).   torch.nn.utils.clip_grad_norm_.
int caphn_clip_coef(const double* sumsq, float max_norm, float* coef, float* norm, void* stream) {
    if (!sumsq || !coef) return CAPHN_EINVAL;
    clip_coef_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sumsq, max_norm, coef, norm);
    CAPHN_RETURN_LAST();
}

// One Adam step (torch.optim.Adam semantics, amsgrad=False, maximize=False) on a flat fp32 tensor; `step` is the 1-based
// step count; gscale (device scalar or NULL) multiplies the gradient first (the clip coefficient).  Hyper-parameters are
// doubles because torch derives 1 - beta, lr / (1 - beta1^t) and sqrt(1 - beta2^t) in double before rounding to fp32.
int caphn_adam_step(float* p, const float* g, float* m, float* v, long n, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int step, const float* gscale, void* stream) {
    if (n < 0 || step < 1 || (((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15)) return CAPHN_EINVAL;
    if (n == 0) return CAPHN_OK;
    const double bc1 = 1.0 - pow(beta1, step), bc2 = 1.0 - pow(beta2, step);
    AdamArgs a{p, g, m, v, n, (float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps, (float)weight_decay,
               (float)(lr / bc1), (float)sqrt(bc2), gscale};
    adam_kernel<<<opt_grid(n >> 2), OPT_THREADS, 0, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

// out[G*G] (device double, caller-zeroed) += X X^T for X [G, L] (row stride ld), G <= 4.
int caphn_gram(const float* X, long ld, int G, long L, double* out, void* stream) {
    if (G < 1 || G > LR_MAXG || L < 0 || !out) return CAPHN_EINVAL;
    if (L == 0) return CAPHN_OK;
    long blocks = (L + OPT_THREADS * 4 - 1) / (OPT_THREADS * 4);
    if (blocks > 4L * kNumSMs) blocks = 4L * kNumSMs;
    gram_kernel<<<(unsigned)(blocks < 1 ? 1 : blocks), OPT_THREADS, 0, (cudaStream_t)stream>>>(X, ld, G, L, out);
    CAPHN_RETURN_LAST();
}

// *sumsq += ||dP^T A||_F^2 from the two Gram matrices (the norm of a rank-G gradient without forming it).
int caphn_sumsq_lowrank(const double* gram_dp, const double* gram_a, int G, double* sumsq, void* stream) {
    if (G < 1 || G > LR_MAXG || !gram_dp || !gram_a || !sumsq) return CAPHN_EINVAL;
    sumsq_lowrank_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(gram_dp, gram_a, G, sumsq);
    CAPHN_RETURN_LAST();
}

// caphn_adam_step with the gradient given in rank-G form: g[n,k] = sum_q dP[q*ldp + n] * A[q*lda + k], p/m/v [N,K].
int caphn_adam_step_lowrank(float* p, float* m, float* v, const float* dP, long ldp, const float* A, long lda, int G,
                            long N, long K, double lr, double beta1, double beta2, double eps, double weight_decay,
                            int step, const float* gscale, void* stream) {
    if (N <= 0 || K <= 0 || K > (1L << 30) || G < 1 || G > LR_MAXG || step < 1 ||
        (((uintptr_t)p | (uintptr_t)m | (uintptr_t)v) & 15))
        return CAPHN_EINVAL;
    const double bc1 = 1.0 - pow(beta1, step), bc2 = 1.0 - pow(beta2, step);
    AdamLrArgs a{p, m, v, dP, ldp, A, lda, G, N, (int)K, (float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps,
                 (float)weight_decay, (float)(lr / bc1), (float)sqrt(bc2), gscale};
    long blocks = ((N * K) >> 2) / ((long)OPT_THREADS * LR_UNR) + 1;
    if (blocks > (long)kNumSMs * 8) blocks = (long)kNumSMs * 8;
    const unsigned grid = (unsigned)blocks;
    cudaStream_t st = (cudaStream_t)stream;
    switch (G) {
        case 1: adam_lowrank_kernel<1><<<grid, OPT_THREADS, 0, st>>>(a); break;
        case 2: adam_lowrank_kernel<2><<<grid, OPT_THREADS, 0, st>>>(a); break;
        case 3: adam_lowrank_kernel<3><<<grid, OPT_THREADS, 0, st>>>(a); break;
        default: adam_lowrank_kernel<4><<<grid, OPT_THREADS, 0, st>>>(a); break;
    }
    CAPHN_RETURN_LAST();
}

// bf16 variants (see adam_bf16_kernel): *sumsq += sum x^2 over a bf16 tensor; Adam step on fp32 master / moments with a
// bf16 gradient, writing the bf16 parameter as the rounding of the updated master weight.
int caphn_sumsq_bf16(const void* x, long n, double* sumsq, void* stream) {
    if (n < 0 || !sumsq || ((uintptr_t)x & 15)) return CAPHN_EINVAL;
    if (n == 0) return CAPHN_OK;
    sumsq_bf16_kernel<<<opt_grid(n >> 3), OPT_THREADS, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, n, sumsq);
    CAPHN_RETURN_LAST();
}

int caphn_adam_step_bf16(void* p, const void* g, float* master, float* m, float* v, long n, double lr, double beta1,
                         double beta2, double eps, double weight_decay, int step, const float* gscale, void* stream) {
    if (n < 0 || step < 1 ||
        (((uintptr_t)p | (uintptr_t)g | (uintptr_t)master | (uintptr_t)m | (uintptr_t)v) & 15))
        return CAPHN_EINVAL;
    if (n == 0) return CAPHN_OK;
    const double bc1 = 1.0 - pow(beta1, step), bc2 = 1.0 - pow(beta2, step);
    AdamBf16Args a{(__nv_bfloat16*)p, (const __nv_bfloat16*)g, master, m, v, n,
                   AdamArgs{nullptr, nullptr, nullptr, nullptr, n, (float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2),
                            (float)eps, (float)weight_decay, (float)(lr / bc1), (float)sqrt(bc2), gscale}};
    adam_bf16_kernel<<<opt_grid(n >> 3), OPT_THREADS, 0, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

}  // extern "C"
