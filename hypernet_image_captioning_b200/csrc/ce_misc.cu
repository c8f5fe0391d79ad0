// Memory-bound pieces of the decoder: softmax cross-entropy over the vocabulary (forward + backward), row softmax /
// argmax for greedy decode, embedding gather / scatter-add, column sums (bias gradients), mean over image positions.
//
// Reference call sites: F.cross_entropy(..., ignore_index=<pad>) cc_train_hypernet.py:153 / hypernet.py:145;
// nn.Embedding lookups models/decoderlstm.py:62,96, later.py:400,473; softmax+argmax later.py:472,479 and
// log_softmax+topk models/decoderlstm.py:94-95; torch.mean(features, dim=1) models/decoderlstm.py:133.
#include "common.cuh"
#include <cuda_bf16.h>
#include <math.h>

namespace caphn {

constexpr int CE_THREADS = 256;

__device__ __forceinline__ float block_reduce_sum(float v, float* sh) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    float r = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.f;
    if (w == 0) r = warp_sum(r);
    if (threadIdx.x == 0) sh[0] = r;
    __syncthreads();
    return sh[0];
}
__device__ __forceinline__ float block_reduce_max(float v, float* sh) {
    v = warp_max(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    float r = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : -INFINITY;
    if (w == 0) r = warp_max(r);
    if (threadIdx.x == 0) sh[0] = r;
    __syncthreads();
    return sh[0];
}

// Target contract of every kernel below (DESIGN.md §6): a row whose target equals the ignore index is ignored (loss 0, not
// counted, zero gradient); any other target outside [0, V) still counts as a row, its loss is NaN (so the mean is NaN and
// the error shows without a host sync) and its gradient row is zero.  x[t] is read only for t in [0, V).
__device__ __forceinline__ bool ce_in_range(long long t, int V) { return (unsigned long long)t < (unsigned long long)V; }

// One CTA per row: lse[m], row_loss[m] = valid ? lse - x[target] : 0, row_valid[m].
__global__ void __launch_bounds__(CE_THREADS) ce_fwd_kernel(const float* __restrict__ X, long ld,
                                                            const long long* __restrict__ tgt, int V, int has_ignore,
                                                            long long ignore, float* __restrict__ lse,
                                                            float* __restrict__ row_loss, float* __restrict__ row_valid) {
    __shared__ float sh[32];
    const long m = blockIdx.x;
    const float* x = X + m * ld;
    const bool vec = ((ld & 3) == 0) && ((V & 3) == 0) && (((uintptr_t)X & 15) == 0);
    float mx = -INFINITY;
    if (vec) {
        for (int i = threadIdx.x * 4; i < V; i += CE_THREADS * 4) {
            const float4 v = *reinterpret_cast<const float4*>(x + i);
            mx = fmaxf(mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
        }
    } else {
        for (int i = threadIdx.x; i < V; i += CE_THREADS) mx = fmaxf(mx, x[i]);
    }
    mx = block_reduce_max(mx, sh);
    float s = 0.f;
    if (vec) {
        for (int i = threadIdx.x * 4; i < V; i += CE_THREADS * 4) {
            const float4 v = *reinterpret_cast<const float4*>(x + i);
            s += expf(v.x - mx) + expf(v.y - mx) + expf(v.z - mx) + expf(v.w - mx);
        }
    } else {
        for (int i = threadIdx.x; i < V; i += CE_THREADS) s += expf(x[i] - mx);
    }
    s = block_reduce_sum(s, sh);
    if (threadIdx.x == 0) {
        const float l = mx + logf(s);
        lse[m] = l;
        const long long t = tgt[m];
        const bool valid = !(has_ignore && t == ignore);
        row_valid[m] = valid ? 1.f : 0.f;
        row_loss[m] = valid ? (ce_in_range(t, V) ? l - x[t] : __int_as_float(0x7fc00000)) : 0.f;
    }
}

// out[0] = sum(row_loss) / sum(row_valid)   out[1] = sum(row_valid)        (single CTA; deterministic)
__global__ void __launch_bounds__(1024) ce_finish_kernel(const float* __restrict__ row_loss,
                                                         const float* __restrict__ row_valid, long M,
                                                         float* __restrict__ out) {
    __shared__ float sh[32];
    float a = 0.f, c = 0.f;
    for (long i = threadIdx.x; i < M; i += 1024) { a += row_loss[i]; c += row_valid[i]; }
    a = block_reduce_sum(a, sh);
    c = block_reduce_sum(c, sh);
    if (threadIdx.x == 0) { out[0] = a / c; out[1] = c; }   // 0/0 = NaN when every row is ignored, like F.cross_entropy
}

// dX[m,v] = (exp(x - lse[m]) - [v == tgt[m]]) * gscale[0] / count   for valid rows, 0 otherwise.
__global__ void __launch_bounds__(CE_THREADS) ce_bwd_kernel(const float* __restrict__ X, long ld,
                                                            const long long* __restrict__ tgt, int V, int has_ignore,
                                                            long long ignore, const float* __restrict__ lse,
                                                            const float* __restrict__ gscale,
                                                            const float* __restrict__ lossbuf, float* __restrict__ dX,
                                                            long lddx) {
    const long m = blockIdx.x;
    const float* x = X + m * ld;
    float* dx = dX + m * lddx;
    const long long t = tgt[m];
    const bool valid = !(has_ignore && t == ignore) && ce_in_range(t, V);     // a zero row for an out-of-range target
    const float sc = valid ? gscale[0] / fmaxf(lossbuf[1], 1.f) : 0.f;
    const float l = lse[m];
    const bool vec = ((ld & 3) == 0) && ((lddx & 3) == 0) && ((V & 3) == 0) && (((uintptr_t)X & 15) == 0) &&
                     (((uintptr_t)dX & 15) == 0);
    if (vec) {
        for (int i = threadIdx.x * 4; i < V; i += CE_THREADS * 4) {
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) {
                const float4 v = *reinterpret_cast<const float4*>(x + i);
                o.x = (expf(v.x - l) - (i == t ? 1.f : 0.f)) * sc;
                o.y = (expf(v.y - l) - (i + 1 == t ? 1.f : 0.f)) * sc;
                o.z = (expf(v.z - l) - (i + 2 == t ? 1.f : 0.f)) * sc;
                o.w = (expf(v.w - l) - (i + 3 == t ? 1.f : 0.f)) * sc;
            }
            *reinterpret_cast<float4*>(dx + i) = o;
        }
    } else {
        for (int i = threadIdx.x; i < V; i += CE_THREADS)
            dx[i] = valid ? (expf(x[i] - l) - (i == t ? 1.f : 0.f)) * sc : 0.f;
    }
}

// Cross-entropy backward emitted directly in the tensor-core operand format (no fp32 dlogits round trip):
//   d[m,v] = (exp(x - lse[m]) - [v == tgt[m]]) * gscale / count   (0 for ignored rows)
//   hi/lo  [M, Vp]  bf16 split of d        (operand of dH  = d  . W_out,  K = V)
//   hiT/loT [V, Mp] bf16 split of d^T      (operand of dW  = d^T . H,     K = M)
//   dbias[v] += sum_m d[m,v]
// One CTA per 64 x 64 tile: coalesced row-major writes, shared-memory transpose for the [V, Mp] copy.
// (256, 8): 32 registers, 8 CTAs per SM -- without the bound ptxas takes 36 once the m-tiles are on blockIdx.x
__global__ void __launch_bounds__(256, 8) ce_bwd_split_kernel(
    const float* __restrict__ X, long ld, const long long* __restrict__ tgt, int M, int V, int has_ignore,
    long long ignore, const float* __restrict__ lse, const float* __restrict__ gscale,
    const float* __restrict__ lossbuf, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, long Vp,
    __nv_bfloat16* __restrict__ hiT, __nv_bfloat16* __restrict__ loT, long Mp, float* __restrict__ dbias) {
    __shared__ float tile[64][65];
    __shared__ float csum[16][64];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * 64, v0 = blockIdx.y * 64;      // m-tiles on x: up to 2^24 of them
    const float sc0 = gscale[0] / fmaxf(lossbuf[1], 1.f);
    const int c4 = (tid & 15) * 4;
    const bool vecx = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && (v0 + c4 + 3 < V);
    float cs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = (tid >> 4) + 16 * i;
        const int m = m0 + r;
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        if (m < M) {
            const long long t = tgt[m];
            const bool valid = !(has_ignore && t == ignore) && ce_in_range(t, V);
            if (valid) {
                const float l = lse[m];
                const float* xp = X + (long)m * ld + v0 + c4;
                float x[4] = {0.f, 0.f, 0.f, 0.f};
                if (vecx) {
                    const float4 xv = *reinterpret_cast<const float4*>(xp);
                    x[0] = xv.x; x[1] = xv.y; x[2] = xv.z; x[3] = xv.w;
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (v0 + c4 + c < V) x[c] = xp[c];
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int v = v0 + c4 + c;
                    if (v < V) d[c] = (expf(x[c] - l) - (v == t ? 1.f : 0.f)) * sc0;
                }
            }
            __nv_bfloat16 h[4], lw[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                h[c] = __float2bfloat16_rn(d[c]);
                lw[c] = __float2bfloat16_rn(d[c] - __bfloat162float(h[c]));
            }
            // 4 bf16 = one 8-byte store per array (row offsets are multiples of 4 elements: Vp % 64 == 0)
            uint2 ph, pl;
            ph.x = (uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16);
            ph.y = (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16);
            pl.x = (uint32_t)__bfloat16_as_ushort(lw[0]) | ((uint32_t)__bfloat16_as_ushort(lw[1]) << 16);
            pl.y = (uint32_t)__bfloat16_as_ushort(lw[2]) | ((uint32_t)__bfloat16_as_ushort(lw[3]) << 16);
            *reinterpret_cast<uint2*>(hi + (long)m * Vp + v0 + c4) = ph;
            if (lo) *reinterpret_cast<uint2*>(lo + (long)m * Vp + v0 + c4) = pl;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) { tile[r][c4 + c] = d[c]; cs[c] += d[c]; }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) csum[tid >> 4][c4 + c] = cs[c];
    __syncthreads();
    if (tid < 64 && dbias != nullptr && v0 + tid < V) {
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) s += csum[g][tid];
        atomicAdd(dbias + v0 + tid, s);
    }
    // transposed copy: item = (column c, group of 8 rows); 8 consecutive lanes cover the 64 rows of one column = 128 B
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        const int item = tid + it * 256;
        const int c = item >> 3, r8 = (item & 7) * 8;
        const int v = v0 + c;
        if (hiT != nullptr && v < V) {
            uint32_t wh[4], wl[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float x0 = tile[r8 + 2 * k][c], x1 = tile[r8 + 2 * k + 1][c];
                const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
                const __nv_bfloat16 l0 = __float2bfloat16_rn(x0 - __bfloat162float(h0));
                const __nv_bfloat16 l1 = __float2bfloat16_rn(x1 - __bfloat162float(h1));
                wh[k] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                wl[k] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
            }
            *reinterpret_cast<uint4*>(hiT + (long)v * Mp + m0 + r8) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
            if (loT) *reinterpret_cast<uint4*>(loT + (long)v * Mp + m0 + r8) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
        }
    }
}

// Cross-entropy forward AND the gradient operand in one pass over the logits (fused loss nodes): one CTA per row, the row
// is read from HBM once into shared memory; out come lse / row_loss / row_valid exactly as from ce_fwd_kernel plus the
// bf16 hi/lo split of the UNSCALED gradient  u[m,v] = softmax(x_m)[v] - [v == tgt[m]]  (0 for ignored rows), columns
// [V, Vp) zeroed.  The scalar the true gradient carries -- grad_output / #valid rows, unknown until backward -- is applied by
// the epilogues of the two products that consume u (caphn_gemm_tc_scaled); the bias gradient is a column of one of them.
// Traffic: logits read once + operand written once (0.8 GB at [10240, 9684]) instead of ce_fwd's extra 0.4 GB read.
__global__ void __launch_bounds__(CE_THREADS) ce_fwd_split_kernel(const float* __restrict__ X, long ld,
                                                                  const long long* __restrict__ tgt, int V, int has_ignore,
                                                                  long long ignore, float* __restrict__ lse,
                                                                  float* __restrict__ row_loss, float* __restrict__ row_valid,
                                                                  __nv_bfloat16* __restrict__ hi,
                                                                  __nv_bfloat16* __restrict__ lo, long Vp) {
    extern __shared__ float4 ce_row4[];
    float* row = reinterpret_cast<float*>(ce_row4);
    __shared__ float sh[32];
    __shared__ uint64_t bar;
    const long m = blockIdx.x;
    const float* x = X + m * ld;
    const bool vec = ((ld & 3) == 0) && ((V & 3) == 0) && (((uintptr_t)X & 15) == 0);
    float mx = -INFINITY;
    if (vec) {
        // the whole row arrives through ONE bulk async copy (no per-thread load chains, nothing held in registers)
        const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
        const uint32_t bytes = (uint32_t)V * 4u;
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"((uint32_t)__cvta_generic_to_shared(row)), "l"(__cvta_generic_to_global(x)), "r"(bytes), "r"(bar_a)
                         : "memory");
        }
        __syncthreads();                        // the barrier is initialised before anyone polls it
        uint32_t done = 0;
        const long long t0 = clock64();
        while (!done) {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(bar_a), "r"(0u)
                : "memory");
            if (!done && clock64() - t0 > 4000000000LL) __trap();     // a protocol bug traps instead of hanging the GPU
        }
        for (int i = threadIdx.x * 4; i < V; i += CE_THREADS * 4) {
            const float4 v = *reinterpret_cast<const float4*>(row + i);
            mx = fmaxf(mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
        }
    } else {
        for (int i = threadIdx.x; i < V; i += CE_THREADS) {
            const float v = x[i];
            row[i] = v;
            mx = fmaxf(mx, v);
        }
    }
    mx = block_reduce_max(mx, sh);
    float s = 0.f;
    if (vec) {          // every thread revisits the elements it wrote itself
        for (int i = threadIdx.x * 4; i < V; i += CE_THREADS * 4) {
            float4 v = *reinterpret_cast<const float4*>(row + i);
            v.x = expf(v.x - mx); v.y = expf(v.y - mx); v.z = expf(v.z - mx); v.w = expf(v.w - mx);
            *reinterpret_cast<float4*>(row + i) = v;
            s += (v.x + v.y) + (v.z + v.w);
        }
    } else {
        for (int i = threadIdx.x; i < V; i += CE_THREADS) {
            const float e = expf(row[i] - mx);
            row[i] = e;
            s += e;
        }
    }
    s = block_reduce_sum(s, sh);          // its barriers also publish the exponentials to the whole CTA
    const long long t = tgt[m];
    const bool valid = !(has_ignore && t == ignore);
    const bool live = valid && ce_in_range(t, V);       // counted, but an out-of-range target gets NaN and a zero row
    if (threadIdx.x == 0) {
        const float l = mx + logf(s);
        lse[m] = l;
        row_valid[m] = valid ? 1.f : 0.f;
        row_loss[m] = valid ? (live ? l - x[t] : __int_as_float(0x7fc00000)) : 0.f;
    }
    const float inv = live ? 1.f / s : 0.f;
    __nv_bfloat16* hrow = hi + m * Vp;
    __nv_bfloat16* lrow = lo ? lo + m * Vp : nullptr;
    const int tcol = live ? (int)t : -1;
    for (int i = threadIdx.x * 4; i < Vp; i += CE_THREADS * 4) {      // Vp % 64 == 0; shared row holds round4(V) floats
        float u[4] = {0.f, 0.f, 0.f, 0.f};
        if (i < V) {
            const float4 e = *reinterpret_cast<const float4*>(row + i);
            u[0] = e.x * inv; u[1] = e.y * inv; u[2] = e.z * inv; u[3] = e.w * inv;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (i + c == tcol) u[c] -= 1.f;
                if (i + c >= V) u[c] = 0.f;
            }
        }
        uint2 ph, pl;
        {
            const __nv_bfloat16 h0 = __float2bfloat16_rn(u[0]), h1 = __float2bfloat16_rn(u[1]);
            const __nv_bfloat16 h2 = __float2bfloat16_rn(u[2]), h3 = __float2bfloat16_rn(u[3]);
            ph.x = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
            ph.y = (uint32_t)__bfloat16_as_ushort(h2) | ((uint32_t)__bfloat16_as_ushort(h3) << 16);
            const __nv_bfloat16 l0 = __float2bfloat16_rn(u[0] - __bfloat162float(h0));
            const __nv_bfloat16 l1 = __float2bfloat16_rn(u[1] - __bfloat162float(h1));
            const __nv_bfloat16 l2 = __float2bfloat16_rn(u[2] - __bfloat162float(h2));
            const __nv_bfloat16 l3 = __float2bfloat16_rn(u[3] - __bfloat162float(h3));
            pl.x = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
            pl.y = (uint32_t)__bfloat16_as_ushort(l2) | ((uint32_t)__bfloat16_as_ushort(l3) << 16);
        }
        *reinterpret_cast<uint2*>(hrow + i) = ph;
        if (lrow) *reinterpret_cast<uint2*>(lrow + i) = pl;
    }
}

// Row softmax (optional, Y may be null) and first-max argmax (matches torch.argmax / topk(1) tie-breaking: lowest index;
// NaN counts as -inf, DESIGN.md §6).
__global__ void __launch_bounds__(CE_THREADS) softmax_argmax_kernel(const float* __restrict__ X, long ld, int V,
                                                                    float* __restrict__ Y, long ldy,
                                                                    long long* __restrict__ amax) {
    __shared__ float sh[32];
    __shared__ int shi[32];
    const long m = blockIdx.x;
    const float* x = X + m * ld;
    float mx = -INFINITY;
    int mi = 0x7fffffff;
    for (int i = threadIdx.x; i < V; i += CE_THREADS) {
        const float v = isnan(x[i]) ? -INFINITY : x[i];     // else [NaN, -inf, ..] would tie to index 1, not 0
        if (v > mx || (v == mx && i < mi)) { mx = v; mi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, mx, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (ov > mx || (ov == mx && oi < mi)) { mx = ov; mi = oi; }
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { sh[w] = mx; shi[w] = mi; }
    __syncthreads();
    if (w == 0) {
        float v = l < (CE_THREADS >> 5) ? sh[l] : -INFINITY;
        int vi = l < (CE_THREADS >> 5) ? shi[l] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, vi, o);
            if (ov > v || (ov == v && oi < vi)) { v = ov; vi = oi; }
        }
        if (l == 0) { sh[0] = v; shi[0] = vi; }
    }
    __syncthreads();
    mx = sh[0];
    if (threadIdx.x == 0 && amax) amax[m] = shi[0] == 0x7fffffff ? 0 : shi[0];   // all-NaN row: stay in range
    if (!Y) return;
    float s = 0.f;
    for (int i = threadIdx.x; i < V; i += CE_THREADS) s += expf(x[i] - mx);
    s = block_reduce_sum(s, sh);
    const float inv = 1.f / s;
    float* y = Y + m * ldy;
    for (int i = threadIdx.x; i < V; i += CE_THREADS) y[i] = expf(x[i] - mx) * inv;
}

// Same, for rows that fit in registers (V % 4 == 0, V <= 256 * 4 * SMAX_RV, 16-byte aligned rows): the row is read ONCE
// with 128-bit loads and kept in registers for the max / argmax, the exp-sum and the normalised write (the generic
// kernel reads it three times with scalar loads).  One per decode step on [B, 9684] logits.
constexpr int SMAX_RV = 10;
__global__ void __launch_bounds__(CE_THREADS) softmax_argmax_vec_kernel(const float* __restrict__ X, long ld, int V,
                                                                        float* __restrict__ Y, long ldy,
                                                                        long long* __restrict__ amax) {
    __shared__ float sh[32];
    __shared__ int shi[32];
    const long m = blockIdx.x;
    const float4* x4 = reinterpret_cast<const float4*>(X + m * ld);
    const int V4 = V >> 2;
    float4 r[SMAX_RV];
    float mx = -INFINITY;
    int mi = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < SMAX_RV; ++j) {
        const int q = j * CE_THREADS + threadIdx.x;
        r[j] = q < V4 ? x4[q] : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
#pragma unroll
    for (int j = 0; j < SMAX_RV; ++j) {      // ascending index within a thread: '>' keeps the lowest index on ties
        const int i0 = (j * CE_THREADS + threadIdx.x) * 4;
        if (r[j].x > mx) { mx = r[j].x; mi = i0; }
        if (r[j].y > mx) { mx = r[j].y; mi = i0 + 1; }
        if (r[j].z > mx) { mx = r[j].z; mi = i0 + 2; }
        if (r[j].w > mx) { mx = r[j].w; mi = i0 + 3; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, mx, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (ov > mx || (ov == mx && oi < mi)) { mx = ov; mi = oi; }
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { sh[w] = mx; shi[w] = mi; }
    __syncthreads();
    if (w == 0) {
        float v = l < (CE_THREADS >> 5) ? sh[l] : -INFINITY;
        int vi = l < (CE_THREADS >> 5) ? shi[l] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, vi, o);
            if (ov > v || (ov == v && oi < vi)) { v = ov; vi = oi; }
        }
        if (l == 0) { sh[0] = v; shi[0] = vi; }
    }
    __syncthreads();
    mx = sh[0];
    if (threadIdx.x == 0 && amax) amax[m] = shi[0] == 0x7fffffff ? 0 : shi[0];   // all-NaN row: stay in range
    if (!Y) return;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < SMAX_RV; ++j) {      // exp(-inf) = 0 for the padding lanes
        r[j].x = expf(r[j].x - mx); r[j].y = expf(r[j].y - mx); r[j].z = expf(r[j].z - mx); r[j].w = expf(r[j].w - mx);
        s += (r[j].x + r[j].y) + (r[j].z + r[j].w);
    }
    s = block_reduce_sum(s, sh);
    const float inv = 1.f / s;
    float4* y4 = reinterpret_cast<float4*>(Y + m * ldy);
#pragma unroll
    for (int j = 0; j < SMAX_RV; ++j) {
        const int q = j * CE_THREADS + threadIdx.x;
        if (q < V4) y4[q] = make_float4(r[j].x * inv, r[j].y * inv, r[j].z * inv, r[j].w * inv);
    }
}

// out[i,:] = idx[i] >= 0 ? table[idx[i],:] : 0      (i < n, row length E)
__global__ void gather_rows_kernel(const float* __restrict__ table, const long long* __restrict__ idx, long n, int E,
                                   float* __restrict__ out, long ldo) {
    const long i = blockIdx.x;
    const long long r = idx[i];
    if (((E | ldo) & 3) == 0 && ((reinterpret_cast<uintptr_t>(table) | reinterpret_cast<uintptr_t>(out)) & 15) == 0) {
        // 128-bit path (rows of 39 KB when whole [P, F] feature blocks are permuted for a many-style batch)
        const float4* src = reinterpret_cast<const float4*>(table + (r >= 0 ? r : 0) * E);
        float4* dst = reinterpret_cast<float4*>(out + i * ldo);
        for (int e = threadIdx.x; e < (E >> 2); e += blockDim.x)
            dst[e] = r >= 0 ? src[e] : make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    for (int e = threadIdx.x; e < E; e += blockDim.x) out[i * ldo + e] = r >= 0 ? table[r * E + e] : 0.f;
}

// Greedy feedback after caphn_gemm_tc_amax: finish the row arg-max from the epilogue's partials (ties: lowest column, like
// torch.argmax / topk(1)), write the token, and gather the row of `table` it selects (the embedding, or the pre-multiplied
// input projection Emb W_ih^T + b_ih) -- one launch between the vocabulary projection of step t and the recurrence of t+1.
// A row whose partials are all empty (its logits all NaN / -inf) gets token 0, never the empty slot's column.
__global__ void __launch_bounds__(128) argmax_finish_gather_kernel(const float* __restrict__ pval, const int* __restrict__ pidx,
                                                                    int ld, int nparts, const float* __restrict__ table,
                                                                    int E, long long* __restrict__ tok,
                                                                    float* __restrict__ out, long ldo) {
    __shared__ int s_tok;
    const long i = blockIdx.x;
    if (threadIdx.x < 32) {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int q = threadIdx.x; q < nparts; q += 32) {
            const float v = pval[i * ld + q];
            const int c = pidx[i * ld + q];
            if (v > bv || (v == bv && c < bi)) { bv = v; bi = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if (bi == 0x7fffffff) bi = 0;
        if (threadIdx.x == 0) { s_tok = bi; if (tok) tok[i] = bi; }
    }
    __syncthreads();
    if (table) {
        const long r = s_tok;
        for (int e = threadIdx.x; e < E; e += blockDim.x) out[i * ldo + e] = table[r * E + e];
    }
}

// Decoder inputs, time-major X[t,b,:]:  mode 0 (DecoderGRU, later.py:411,418): X[0,b] = feat[b], X[t,b] = Emb[caps[b,t-1]]
//                                       mode 1 (AttentionGru, decoderlstm.py:82-88): X[0] = X[1] = 0, X[t] = Emb[caps[b,t-1]]
__global__ void build_inputs_kernel(const float* __restrict__ feat, const float* __restrict__ emb,
                                    const long long* __restrict__ caps, int B, int T, int E, int mode,
                                    float* __restrict__ X) {
    const int t = blockIdx.x / B, b = blockIdx.x - t * B;
    float* x = X + ((long)t * B + b) * E;
    const float* src = nullptr;
    if (mode == 0) src = (t == 0) ? feat + (long)b * E : emb + caps[(long)b * T + t - 1] * E;
    else if (t >= 2) src = emb + caps[(long)b * T + t - 1] * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) x[e] = src ? src[e] : 0.f;
}

// dEmb[caps[b,t-1],:] += dX[t,b,:]  for t >= t0 (t0 = 1 pooled, 2 attention).
__global__ void embed_scatter_add_kernel(const float* __restrict__ dX, const long long* __restrict__ caps, int B, int T,
                                         int E, int t0, float* __restrict__ dEmb) {
    const int t = t0 + blockIdx.x / B, b = blockIdx.x % B;
    if (t >= T) return;
    const long long r = caps[(long)b * T + t - 1];
    const float* d = dX + ((long)t * B + b) * E;
    float* o = dEmb + r * E;
    if ((E & 3) == 0 && (((uintptr_t)d | (uintptr_t)o) & 15) == 0) {      // 16-byte vector reductions: a quarter of the atomics
        for (int e = threadIdx.x * 4; e < E; e += blockDim.x * 4) {
            const float4 v = *reinterpret_cast<const float4*>(d + e);
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + e), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                         : "memory");
        }
    } else {
        for (int e = threadIdx.x; e < E; e += blockDim.x) atomicAdd(o + e, d[e]);
    }
}

// table[idx[i],:] += dX[i,:]   (rows with idx < 0 are skipped)
__global__ void scatter_add_rows_kernel(const float* __restrict__ dX, long ldx, const long long* __restrict__ idx,
                                        int E, float* __restrict__ table) {
    const long i = blockIdx.x;
    const long long r = idx[i];
    if (r < 0) return;
    const float* d = dX + i * ldx;
    float* o = table + r * E;
    if ((E & 3) == 0 && (((uintptr_t)d | (uintptr_t)o) & 15) == 0) {
        for (int e = threadIdx.x * 4; e < E; e += blockDim.x * 4) {
            const float4 v = *reinterpret_cast<const float4*>(d + e);
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + e), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                         : "memory");
        }
    } else {
        for (int e = threadIdx.x; e < E; e += blockDim.x) atomicAdd(o + e, d[e]);
    }
}

// out[n] (+)= sum_m X[m*ld + n]
__global__ void colsum_kernel(const float* __restrict__ X, long ld, long M, int N, long rows_per_block,
                              float* __restrict__ out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const long m0 = (long)blockIdx.y * rows_per_block;
    const long m1 = min(M, m0 + rows_per_block);
    if (n >= N) return;
    float s = 0.f;
    long m = m0;
    for (; m + 8 <= m1; m += 8) {          // 8 independent loads in flight per thread
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldg(X + (m + u) * ld + n);
#pragma unroll
        for (int u = 0; u < 8; ++u) s += v[u];
    }
    for (; m < m1; ++m) s += __ldg(X + m * ld + n);
    atomicAdd(out + n, s);
}

// out[b,f] = mean_p X[b,p,f]
__global__ void mean_pos_kernel(const float* __restrict__ X, int P, int Fd, float* __restrict__ out) {
    const long b = blockIdx.x;
    for (int f = threadIdx.x; f < Fd; f += blockDim.x) {
        float s = 0.f;
        for (int p = 0; p < P; ++p) s += X[(b * P + p) * Fd + f];
        out[b * Fd + f] = s / (float)P;
    }
}
// dX[b,p,f] += g[b,f] / P (+ extra[b,p,f])
__global__ void mean_pos_bwd_kernel(const float* __restrict__ g, const float* __restrict__ extra, int P, int Fd,
                                    float* __restrict__ dX) {
    const long b = blockIdx.x;
    const float inv = 1.f / (float)P;
    for (int i = threadIdx.x; i < P * Fd; i += blockDim.x) {
        const long o = b * P * Fd + i;
        dX[o] += g[b * Fd + (i % Fd)] * inv + (extra ? extra[o] : 0.f);
    }
}

// y = relu'(ref) * y   (in place on y): y[i] = ref[i] > 0 ? y[i] : 0
__global__ void relu_mask_kernel(const float* __restrict__ ref, float* __restrict__ y, long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !(ref[i] > 0.f)) y[i] = 0.f;
}

}  // namespace caphn

using namespace caphn;

extern "C" {

// Cross-entropy over rows of X [M,V] (row stride ld).  ignore_index is honoured when has_ignore != 0.
// Outputs: lse [M]; scratch [2*M]; lossbuf[0] = mean loss over valid rows, lossbuf[1] = number of valid rows.
int caphn_ce_fwd(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                 float* lse, float* scratch, float* lossbuf, void* stream) {
    if (M <= 0 || V <= 0) return CAPHN_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    ce_fwd_kernel<<<(unsigned)M, CE_THREADS, 0, st>>>(X, ld, tgt, V, has_ignore, ignore, lse, scratch, scratch + M);
    CAPHN_LAUNCH_CHECK();
    ce_finish_kernel<<<1, 1024, 0, st>>>(scratch, scratch + M, M, lossbuf);
    CAPHN_RETURN_LAST();
}

// caphn_ce_fwd + the unscaled gradient u = softmax(X) - onehot(tgt) (0 on ignored rows) as the bf16 hi/lo operand
// [M, Vp] (Vp % 64 == 0, Vp >= V; lo may be NULL), from ONE read of X (see ce_fwd_split_kernel).  The consumer applies
// gscale / max(lossbuf[1], 1) (caphn_gemm_tc_scaled).  V is limited by the row having to fit in shared memory (V <= 50000).
int caphn_ce_fwd_split(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                       float* lse, float* scratch, float* lossbuf, void* hi, void* lo, long Vp, void* stream) {
    if (M <= 0 || V <= 0 || V > 50000 || Vp < V || (Vp & 63) || !hi) return CAPHN_EINVAL;
    if (((uintptr_t)hi & 7) || ((uintptr_t)lo & 7)) return CAPHN_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)((V + 3) / 4) * 16;
    CAPHN_CHECK(cudaFuncSetAttribute(ce_fwd_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ce_fwd_split_kernel<<<(unsigned)M, CE_THREADS, smem, st>>>(X, ld, tgt, V, has_ignore, ignore, lse, scratch, scratch + M,
                                                               (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, Vp);
    CAPHN_LAUNCH_CHECK();
    ce_finish_kernel<<<1, 1024, 0, st>>>(scratch, scratch + M, M, lossbuf);
    CAPHN_RETURN_LAST();
}

// dX = d(mean loss)/dX * gscale[0];  lossbuf as produced by caphn_ce_fwd (valid-row count read on device: no sync).
int caphn_ce_bwd(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                 const float* lse, const float* gscale, const float* lossbuf, float* dX, long lddx, void* stream) {
    if (M <= 0 || V <= 0) return CAPHN_EINVAL;
    ce_bwd_kernel<<<(unsigned)M, CE_THREADS, 0, (cudaStream_t)stream>>>(X, ld, tgt, V, has_ignore, ignore, lse, gscale,
                                                                        lossbuf, dX, lddx);
    CAPHN_RETURN_LAST();
}

// Cross-entropy backward written straight into the bf16x3 operand formats of caphn_gemm_tc (see kernel comment):
// hi/lo [M, Vp], hiT/loT [V, Mp] (Vp, Mp multiples of 64, >= V, M), dbias [V] accumulated (zero-initialised by caller).
// lo / loT may be NULL (plain bf16 mode); hiT == NULL skips the transposed copy (the GEMM reads d MN-major in place).
int caphn_ce_bwd_split(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                       const float* lse, const float* gscale, const float* lossbuf, void* hi, void* lo, long Vp,
                       void* hiT, void* loT, long Mp, float* dbias, void* stream) {
    if (M <= 0 || V <= 0 || Vp < V || (Vp & 63) || Mp < M || (Mp & 63) || M > (1L << 30)) return CAPHN_EINVAL;
    if (Vp / 64 > 65535) return CAPHN_EINVAL;               // v-tiles on gridDim.y
    dim3 grid((unsigned)(Mp / 64), (unsigned)(Vp / 64));
    ce_bwd_split_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
        X, ld, tgt, (int)M, V, has_ignore, ignore, lse, gscale, lossbuf, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, Vp,
        (__nv_bfloat16*)hiT, (__nv_bfloat16*)loT, Mp, dbias);
    CAPHN_RETURN_LAST();
}

// Y (optional) = softmax rows of X; amax (optional) = argmax per row (lowest index on ties).
int caphn_softmax_argmax(const float* X, long ld, long M, int V, float* Y, long ldy, long long* amax, void* stream) {
    if (M <= 0 || V <= 0) return CAPHN_EINVAL;
    const bool vec = (V % 4 == 0) && V <= CE_THREADS * 4 * SMAX_RV && (ld % 4 == 0) && ((uintptr_t)X % 16 == 0) &&
                     (!Y || ((ldy % 4 == 0) && ((uintptr_t)Y % 16 == 0)));
    if (vec) softmax_argmax_vec_kernel<<<(unsigned)M, CE_THREADS, 0, (cudaStream_t)stream>>>(X, ld, V, Y, ldy, amax);
    else softmax_argmax_kernel<<<(unsigned)M, CE_THREADS, 0, (cudaStream_t)stream>>>(X, ld, V, Y, ldy, amax);
    CAPHN_RETURN_LAST();
}

int caphn_gather_rows(const float* table, const long long* idx, long n, int E, float* out, long ldo, void* stream) {
    if (n <= 0 || E <= 0) return CAPHN_EINVAL;
    gather_rows_kernel<<<(unsigned)n, 128, 0, (cudaStream_t)stream>>>(table, idx, n, E, out, ldo);
    CAPHN_RETURN_LAST();
}

// tok[i] = arg-max over the nparts (value, column) partials of row i (pval / pidx [n, ld], from caphn_gemm_tc_amax);
// out[i, :] = table[tok[i], :E] when table != NULL.  tok may be NULL.
int caphn_argmax_finish_gather(const float* pval, const int* pidx, int ld, int nparts, long n, const float* table, int E,
                               long long* tok, float* out, long ldo, void* stream) {
    if (n <= 0 || nparts <= 0 || nparts > ld || (table && (E <= 0 || !out))) return CAPHN_EINVAL;
    argmax_finish_gather_kernel<<<(unsigned)n, 128, 0, (cudaStream_t)stream>>>(pval, pidx, ld, nparts, table, E, tok, out, ldo);
    CAPHN_RETURN_LAST();
}

int caphn_build_inputs(const float* feat, const float* emb, const long long* caps, int B, int T, int E, int mode,
                       float* X, void* stream) {
    if (B <= 0 || T <= 0 || E <= 0) return CAPHN_EINVAL;
    build_inputs_kernel<<<(unsigned)(B * T), 128, 0, (cudaStream_t)stream>>>(feat, emb, caps, B, T, E, mode, X);
    CAPHN_RETURN_LAST();
}

int caphn_embed_scatter_add(const float* dX, const long long* caps, int B, int T, int E, int t0, float* dEmb,
                            void* stream) {
    if (B <= 0 || T <= 0 || E <= 0 || t0 < 1) return CAPHN_EINVAL;
    if (T - t0 <= 0) return CAPHN_OK;
    embed_scatter_add_kernel<<<(unsigned)(B * (T - t0)), 128, 0, (cudaStream_t)stream>>>(dX, caps, B, T, E, t0, dEmb);
    CAPHN_RETURN_LAST();
}

int caphn_scatter_add_rows(const float* dX, long ldx, const long long* idx, long n, int E, float* table, void* stream) {
    if (n <= 0 || E <= 0) return CAPHN_EINVAL;
    scatter_add_rows_kernel<<<(unsigned)n, 128, 0, (cudaStream_t)stream>>>(dX, ldx, idx, E, table);
    CAPHN_RETURN_LAST();
}

// out[n] += sum_m X[m,n]   (caller zeroes out for a plain sum)
int caphn_colsum(const float* X, long ld, long M, int N, float* out, void* stream) {
    if (M <= 0 || N <= 0) return CAPHN_EINVAL;
    // enough row blocks for ~8 CTAs per SM (the kernel is a latency chain of loads otherwise), >= 16 rows each
    const long xb = ceil_div(N, 128);
    long rpb = 256;
    while (rpb > 16 && xb * ceil_div(M, rpb) < 8L * kNumSMs) rpb >>= 1;
    if (ceil_div(M, rpb) > 65535) rpb = (M + 65534) / 65535;     // the row blocks are on gridDim.y, which stops at 65535
    dim3 grid(xb, ceil_div(M, rpb));
    colsum_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(X, ld, M, N, rpb, out);
    CAPHN_RETURN_LAST();
}

int caphn_mean_pos(const float* X, int B, int P, int Fd, float* out, void* stream) {
    if (B <= 0 || P <= 0 || Fd <= 0) return CAPHN_EINVAL;
    mean_pos_kernel<<<(unsigned)B, 128, 0, (cudaStream_t)stream>>>(X, P, Fd, out);
    CAPHN_RETURN_LAST();
}

int caphn_mean_pos_bwd(const float* g, const float* extra, int B, int P, int Fd, float* dX, void* stream) {
    if (B <= 0 || P <= 0 || Fd <= 0) return CAPHN_EINVAL;
    mean_pos_bwd_kernel<<<(unsigned)B, 256, 0, (cudaStream_t)stream>>>(g, extra, P, Fd, dX);
    CAPHN_RETURN_LAST();
}

int caphn_relu_mask(const float* ref, float* y, long n, void* stream) {
    if (n <= 0) return CAPHN_EINVAL;
    relu_mask_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(ref, y, n);
    CAPHN_RETURN_LAST();
}

}  // extern "C"
