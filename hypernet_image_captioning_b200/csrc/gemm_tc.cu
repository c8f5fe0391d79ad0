// Tensor-core GEMM for sm_100a: C[M,N] (fp32) = A[M,K] B[N,K]^T (+bias) (ReLU), tcgen05.mma with the accumulator in
// TMEM, operands staged by TMA (cp.async.bulk.tensor, 128-byte swizzle), mbarrier pipelines, persistent CTAs.
//
// fp32-accurate mode ("bf16x3"): every fp32 operand is pre-split (caphn_split_bf16*) into bf16 hi = rn(x) and
// lo = rn(x - hi); the kernel issues three MMAs per k-slice, hi*hi + hi*lo + lo*hi, accumulating in fp32.  The dropped
// lo*lo term and the residual of the split are ~2^-17 relative, i.e. ~1e-5 on the result -- inside the 1e-4 parity
// budget of BASELINE.json (plain TF32 would be ~1e-3).  With lo == NULL the same kernel runs a plain bf16 GEMM.
//
// Replaces the large addmm calls behind nn.Linear in the reference: vocabulary projection self.fc / fc_out
// (models/decoderlstm.py:105, later.py:442) forward and both backward products, feature_fc (models/decoderlstm.py:61).
//
// Warp roles (384 threads, 1 CTA/SM): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warp 2 = TMEM
// allocator, warps 4-11 = epilogue (tcgen05.ld -> swizzled smem transpose -> 128-bit coalesced global stores, or fp32
// atomics under split-K).  Two TMEM accumulator stages (2 x BN columns) let the MMAs of work unit i+1 overlap the
// epilogue of unit i.  The N tile is chosen at run time (one tile of N rounded to 16 when N <= 256, e.g. 160 for
// H = 150), and long-K / few-tile products are split along K so that ~148 CTAs are busy.
#include "common.cuh"
#include <cuda.h>
#include <stdlib.h>
#include <cuda_bf16.h>

namespace caphn {
namespace tc {

constexpr int BM = 128, BK = 64;
constexpr int TILE_BYTES = BM * BK * 2;  // 16 KiB: one 128 x 64 bf16 operand tile (128-byte rows, SWIZZLE_128B)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int x, int y) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
}
// One elected lane of a fully converged warp.  The single-thread roles (TMA producer, MMA issuer, bulk stores) run their loops
// with all 32 lanes converged and only issue under this predicate: the operands of UTMALDG / UTCHMMA / UTMASTG must sit in
// uniform registers, and a loop under `if (lane == 0)` is divergent code where ptxas cannot use the uniform datapath -- it
// wrapped EVERY such instruction in an ELECT / 5 x R2UR.BROADCAST / BRA.U.ANY waterfall loop, which made the MMA thread the
// bottleneck of the kernel (~160 cycles per 128x128x16 MMA issued, against ~64-100 of tensor-pipe time).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout): start address >> 4 in
// bits [0,14), LBO = 1 (16-byte units; fixed for swizzled K-major), SBO = 1024 B (8 rows x 128 B) in bits [32,46),
// version = 1 (Blackwell) in bits [46,48), layout type 2 (SWIZZLE_128B) in bits [61,64).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, bool mn_major = false) {
    // K-major : canonical ((8,n),2):((8,SBO),1)        -> LBO = 1 (unused), SBO = 1024 B (8 rows x 128 B)
    // MN-major: canonical ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units: 64 MN elements (128 B) contiguous, k rows 128 B
    //           apart, groups of 8 k rows SBO = 1024 B apart, next 64 MN elements LBO = 8192 B apart (= one 64x64 TMA box)
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(mn_major ? (8192 >> 4) : 1) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// Instruction descriptor for kind::f16: D = F32 (bits [4,6) = 1), A = B = BF16 (bits [7,10) = [10,13) = 1), both K-major,
// N >> 3 in bits [17,23), M >> 4 in bits [24,29).
__device__ __forceinline__ uint32_t make_idesc(int m, int n, bool a_mn = false, bool b_mn = false) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// TMA store of one [32 rows x 32 fp32] SWIZZLE_128B box from shared memory (TMA_STORE = true epilogue)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, const void* smem_src, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(x), "r"(y)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void red_add_v2(float* p, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Shared-memory plan (dynamic, 1024-byte aligned): [stage 0 | stage 1 | ...][epilogue staging][mbarriers][tmem slot].
// A stage holds A_hi, (A_lo), B_hi, (B_lo); A tiles are 128 x 64 bf16 (16 KiB), B tiles BN x 64 bf16 (BN * 128 B).
constexpr int EPI_WARPS = 8;
constexpr int STG_STRIDE = 32;                              // floats per staged row; float4 slots XOR-swizzled by (row & 7)
constexpr int STG_FLOATS_V2 = EPI_WARPS * 32 * STG_STRIDE;  // 32 KiB
constexpr int THREADS_V2 = 128 + EPI_WARPS * 32;            // warps 0-3: TMA / MMA / TMEM alloc / idle; 4-11: epilogue
constexpr int MAX_STAGES = 6;
constexpr size_t SMEM_BUDGET = 227 * 1024;

// Grouped mode (caphn_gemm_tc_grouped): every work unit is described by one record instead of being derived from the unit
// index -- a tile of group g reads A rows / B rows / a K range that belong to that group and writes into that group's
// slice of C (optionally through a row map).  Ten 32-bit words per unit, built on the host once per batch composition.
struct GUnit {
    int a_row;      // first operand row of the A tile (K-major: row index; MN-major: MN column)
    int b_row;      // same for B
    int ka0;        // first k index of the A operand: column offset (K-major) / row offset (MN-major)
    int kb0;        // first k index of the B operand (the two operands may keep a group's K range at different places)
    int nkb;        // 64-wide k blocks to accumulate (>= 1)
    int m_valid;    // rows of the tile that exist (1..128)
    int n_valid;    // columns of the tile that exist (1..BN)
    int bias_off;   // bias[bias_off + col] is added (ignored when bias == NULL)
    int map0;       // rowmap != NULL: tile row r is written to C row rowmap[map0 + r] (skipped when negative)
    unsigned c_lo;  // element offset of the tile's (0, 0) inside C (rowmap: column offset only), low / high word
    int c_hi;
    int pad;        // 12 words = 48 bytes per record
};

struct UnitInfo {
    int a0, b0, ka0, kb0, nkb, m_valid, n_valid, bias_off, map0, ks;   // ka0 / kb0 in elements
    long c_off;
};

struct TcParams {
    float* C; long ldc; const float* bias;
    const GUnit* units;   // grouped mode when non-null (num_units records)
    const int* rowmap;
    int num_units;
    // optional row arg-max partials (greedy decode, SURVEY K9: the arg-max of step t feeds step t+1): every epilogue warp
    // reduces the columns it reads of every row to (max, column) and writes them to amax_val / amax_idx [M, amax_ld],
    // slot 2 * n-tile + warp half; a tiny kernel finishes the reduction (and gathers the next input row).  null: off.
    float* amax_val; int* amax_idx; int amax_ld;
    int M, N, num_kb, relu;
    int BN;          // N tile (multiple of 16, <= 256)
    int splitk;      // K split factor; > 1 => epilogue adds atomically into a zero-initialised C
    int kb_per;      // k-blocks per split
    int stages, stage_bytes, b_bytes;
    uint32_t tmem_cols;
    int a_mn, b_mn;  // operand stored MN-major ([K rows, MN cols] row-major) instead of K-major ([MN rows, K cols])
    // optional scalar applied to the accumulators before the bias: scale_num[0] / max(scale_den[0], 1) (den NULL = 1).
    // The fused cross-entropy nodes hand the UNSCALED gradient operand to the two backward products and let their
    // epilogues apply grad_output / #valid rows (both device scalars: no host synchronisation).
    const float* scale_num; const float* scale_den;
    int K;           // true K (0 in grouped mode): the MMAs of the zero-filled tail of the last k-block are skipped
    // A-stationary schedule (short K, many N tiles: the vocabulary projection): every CTA owns a contiguous run of tiles in
    // (m-tile major, n-tile minor) order and keeps the whole [128, K] A slab of its m-tile in shared memory (loaded once per
    // m-tile, i.e. once or twice per CTA); only B tiles stream through the stage ring.  Halves the L2 -> SM operand traffic
    // of a product that was bound by it (1.17 GB for 0.4 GB of output at M=10240, N=9684, K=150).
    int astat;
    int a_slab_bytes;
};

__device__ __forceinline__ UnitInfo decode_unit(const TcParams& p, int unit, int tiles_m, int BN) {
    UnitInfo u;
    if (p.units) {
        const GUnit g = p.units[unit];
        u.a0 = g.a_row; u.b0 = g.b_row; u.ka0 = g.ka0; u.kb0 = g.kb0; u.nkb = g.nkb; u.m_valid = g.m_valid; u.n_valid = g.n_valid;
        u.bias_off = g.bias_off; u.map0 = g.map0; u.ks = 0;
        u.c_off = ((long)g.c_hi << 32) | (long)g.c_lo;
    } else {
        const int ks = unit % p.splitk, tile = unit / p.splitk;
        int mb, nb;
        if (p.astat) {                      // n-tile fastest: consecutive units of a CTA share their A slab
            const int tiles_n = (p.N + BN - 1) / BN;
            mb = tile / tiles_n; nb = tile - mb * tiles_n;
        } else {
            mb = tile % tiles_m; nb = tile / tiles_m;
        }
        const int kblk0 = ks * p.kb_per;
        u.a0 = mb * BM; u.b0 = nb * BN; u.ka0 = u.kb0 = kblk0 * BK; u.nkb = min(p.num_kb, kblk0 + p.kb_per) - kblk0;
        u.m_valid = min(BM, p.M - mb * BM); u.n_valid = min(BN, p.N - nb * BN);
        u.bias_off = nb * BN; u.map0 = 0; u.ks = ks;
        u.c_off = (long)mb * BM * p.ldc + (long)nb * BN;
    }
    return u;
}

// TMA_STORE (the default epilogue for N % 4 == 0 without split-K since round 2; CAPHN_TC_TMA_STORE=0 switches it off): full
// 32-column chunks leave through one cp.async.bulk.tensor store per warp from the swizzled staging tile instead of
// 8 x (ld.shared + st.global) per lane.  Bit-identical to the register-store epilogue (tests/test_gpu_gemm_tc.py) and 2-9 %
// faster on the logits products (profiles/r02_gemm_tma_store.txt); ragged N keeps the register-store epilogue.
template <bool SPLIT, bool TMA_STORE = false>
__global__ void __launch_bounds__(THREADS_V2, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
               const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
               const __grid_constant__ CUtensorMap tmC, const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* tiles = smem;
    float* stg = reinterpret_cast<float*>(smem + (size_t)p.a_slab_bytes + (size_t)p.stages * p.stage_bytes);
    uint64_t* full = reinterpret_cast<uint64_t*>(stg + (p.splitk > 1 ? 0 : STG_FLOATS_V2));   // split-K: no staging
    uint64_t* empty = full + MAX_STAGES;
    uint64_t* tfull = empty + MAX_STAGES;
    uint64_t* tempty = tfull + 2;
    uint64_t* afull = tempty + 2;            // A-stationary schedule: slab loaded / slab free
    uint64_t* aempty = afull + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty + 1);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // provably warp-uniform
    const int lane = threadIdx.x & 31;
    const int BN = p.BN;
    const int tiles_m = (p.M + BM - 1) / BM, tiles_n = (p.N + BN - 1) / BN;
    const int num_units = p.units ? p.num_units : tiles_m * tiles_n * p.splitk;
    // this CTA's units: round-robin over the grid, or (A-stationary) one contiguous, balanced run
    int u_first, u_step, u_count;
    if (p.astat) {
        const int q = num_units / (int)gridDim.x, r = num_units % (int)gridDim.x;
        u_first = (int)blockIdx.x * q + min((int)blockIdx.x, r);
        u_count = q + ((int)blockIdx.x < r ? 1 : 0);
        u_step = 1;
    } else {
        u_first = blockIdx.x;
        u_step = gridDim.x;
        u_count = (int)blockIdx.x < num_units ? (num_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    }
    // operand offsets inside a stage (A-stationary: the slab comes first, a stage holds only B_hi, (B_lo))
    const int offAh = 0, offBh = p.astat ? 0 : TILE_BYTES;
    const int offAl = TILE_BYTES + p.b_bytes, offBl = p.astat ? p.b_bytes : 2 * TILE_BYTES + p.b_bytes;
    const int ablk = (SPLIT ? 2 : 1) * TILE_BYTES;       // slab bytes per k-block: A_hi, (A_lo)
    uint8_t* slab = smem;
    if (p.astat) tiles = smem + p.a_slab_bytes;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull + s, 1); mbar_init(tempty + s, EPI_WARPS); }
        mbar_init(afull, 1); mbar_init(aempty, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        // TMA producer: all 32 lanes run the loop (converged), one elected lane issues
        int stage = 0;
        uint32_t phase = 0;
        int cur_a0 = -1;
        uint32_t a_it = 0;
        for (int ui = 0, unit = u_first; ui < u_count; ++ui, unit += u_step) {
            const UnitInfo u = decode_unit(p, unit, tiles_m, BN);
            if (p.astat && u.a0 != cur_a0) {       // new m-tile: (re)load the A slab once the MMAs reading the old one are done
                mbar_wait(aempty, (a_it & 1) ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(afull, (uint32_t)p.a_slab_bytes);
                    for (int i = 0; i < u.nkb; ++i) {
                        tma_load_2d(slab + (size_t)i * ablk, &tmAh, afull, u.ka0 + i * BK, u.a0);
                        if (SPLIT) tma_load_2d(slab + (size_t)i * ablk + TILE_BYTES, &tmAl, afull, u.ka0 + i * BK, u.a0);
                    }
                }
                __syncwarp();
                cur_a0 = u.a0;
                ++a_it;
            }
            for (int i = 0; i < u.nkb; ++i) {
                const int ka = u.ka0 + i * BK, kbk = u.kb0 + i * BK;
                mbar_wait(empty + stage, phase ^ 1);
                uint8_t* st = tiles + (size_t)stage * p.stage_bytes;
                if (elect_one()) {
                    mbar_expect_tx(full + stage, (uint32_t)p.stage_bytes);
                    // K-major operand: one box [64 k x rows].  MN-major operand: boxes of [64 mn x 64 k] (8 KiB each).
                    if (p.astat) {
                        // A is resident in the slab
                    } else if (!p.a_mn) {
                        tma_load_2d(st + offAh, &tmAh, full + stage, ka, u.a0);
                        if (SPLIT) tma_load_2d(st + offAl, &tmAl, full + stage, ka, u.a0);
                    } else {
                        for (int h = 0; h < BM / 64; ++h) {
                            tma_load_2d(st + offAh + h * 8192, &tmAh, full + stage, u.a0 + h * 64, ka);
                            if (SPLIT) tma_load_2d(st + offAl + h * 8192, &tmAl, full + stage, u.a0 + h * 64, ka);
                        }
                    }
                    if (!p.b_mn) {
                        tma_load_2d(st + offBh, &tmBh, full + stage, kbk, u.b0);
                        if (SPLIT) tma_load_2d(st + offBl, &tmBl, full + stage, kbk, u.b0);
                    } else {
                        for (int h = 0; h < BN / 64; ++h) {
                            tma_load_2d(st + offBh + h * 8192, &tmBh, full + stage, u.b0 + h * 64, kbk);
                            if (SPLIT) tma_load_2d(st + offBl + h * 8192, &tmBl, full + stage, u.b0 + h * 64, kbk);
                        }
                    }
                }
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // MMA issuer: converged warp, one elected lane issues the tcgen05.mma / tcgen05.commit instructions
        const uint32_t idesc = make_idesc(BM, BN, p.a_mn != 0, p.b_mn != 0);
        // advance per 16-wide k step: 32 B inside the 128 B swizzle row (K-major) / two 8-row k groups (MN-major)
        const uint64_t stepA = p.a_mn ? (uint64_t)(2048 >> 4) : (uint64_t)(32 >> 4);
        const uint64_t stepB = p.b_mn ? (uint64_t)(2048 >> 4) : (uint64_t)(32 >> 4);
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        int cur_a0 = -1;
        uint32_t a_it = 0;
        const uint32_t slab_base = smem_u32(slab);
        for (int ui = 0, unit = u_first; ui < u_count; ++ui, unit += u_step, ++it) {
            const UnitInfo u = decode_unit(p, unit, tiles_m, BN);
            const int kb0 = 0, kb1 = u.nkb;
            const int as = it & 1;
            const uint32_t aph = (it >> 1) & 1;
            mbar_wait(tempty + as, aph ^ 1);
            tcgen05_fence_after();
            if (p.astat && u.a0 != cur_a0) {
                mbar_wait(afull, a_it & 1);
                tcgen05_fence_after();
                cur_a0 = u.a0;
                ++a_it;
            }
            const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(full + stage, phase);
                tcgen05_fence_after();
                const uint32_t sbase = smem_u32(tiles + (size_t)stage * p.stage_bytes);
                const uint32_t abase = p.astat ? slab_base + (uint32_t)(kb * ablk) : sbase;
                const uint64_t dAh = make_desc(abase + offAh, p.a_mn), dBh = make_desc(sbase + offBh, p.b_mn);
                const uint64_t dAl = make_desc(abase + (p.astat ? TILE_BYTES : offAl), p.a_mn);
                const uint64_t dBl = make_desc(sbase + offBl, p.b_mn);
                // last k-block: only the 16-wide steps that hold real columns (TMA zero-filled the rest)
                int ksteps = BK / 16;
                if (p.K > 0 && kb == kb1 - 1) {
                    const int rem = p.K - (u.ka0 + kb * BK);
                    ksteps = rem >= BK ? BK / 16 : (rem <= 0 ? 1 : (rem + 15) / 16);
                }
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        if (k < ksteps) {
                            const uint64_t ka = stepA * k, kbo = stepB * k;
                            umma_f16(tmem_d, dAh + ka, dBh + kbo, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                            if (SPLIT) {
                                umma_f16(tmem_d, dAh + ka, dBl + kbo, idesc, 1u);
                                umma_f16(tmem_d, dAl + ka, dBh + kbo, idesc, 1u);
                            }
                        }
                    }
                    umma_commit(empty + stage);   // frees this smem stage once the MMAs above have read it
                }
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            bool last_on_slab = false;
            if (p.astat) {                    // last unit on this A slab: it may be overwritten once these MMAs are done
                last_on_slab = ui + 1 == u_count;
                if (!last_on_slab) last_on_slab = decode_unit(p, unit + u_step, tiles_m, BN).a0 != u.a0;
            }
            if (elect_one()) {
                if (last_on_slab) umma_commit(aempty);   // (committed before tfull so that it never outlives the CTA)
                umma_commit(tfull + as);                 // accumulator complete -> epilogue
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        const int ew = warp - 4;
        const int q = warp & 3;                   // TMEM lane quadrant this warp may access (warp id % 4)
        const int half = ew >> 2;                 // two warps per quadrant split the 32-column chunks
        float* const st = stg + ew * (32 * STG_STRIDE);
        const int nchunks = (BN + 31) / 32;
        const bool atomic = p.splitk > 1;
        const bool vec = !atomic && ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
        int it = 0;
        const float alpha = p.scale_num ? p.scale_num[0] / fmaxf(p.scale_den ? p.scale_den[0] : 1.f, 1.f) : 1.f;
        for (int ui = 0, unit = u_first; ui < u_count; ++ui, unit += u_step, ++it) {
            const UnitInfo u = decode_unit(p, unit, tiles_m, BN);
            const int as = it & 1;
            const uint32_t aph = (it >> 1) & 1;
            mbar_wait(tfull + as, aph);
            tcgen05_fence_after();
            const int row0 = u.a0 + q * 32;           // (non-grouped TMA-store path only: global row of this warp's first row)
            const int rl0 = q * 32;                   // first tile-local row of this warp
            const bool add_bias = p.bias != nullptr && u.ks == 0;
            const float* biasp = p.bias ? p.bias + u.bias_off : nullptr;
            float* Ct = p.C + u.c_off;
            const int* rmap = p.rowmap ? p.rowmap + u.map0 : nullptr;
            int last_c = half;
            while (last_c + 2 < nchunks) last_c += 2;
            float am_best = -INFINITY;            // arg-max partial of row (rl0 + lane) over this warp's chunks
            int am_idx = 0x7fffffff;
            if (half >= nchunks) {                 // nothing to read for this warp: release the stage immediately
                tcgen05_fence_before();
                if (lane == 0) mbar_arrive(tempty + as);
            }
#pragma unroll 1
            for (int c = half; c < nchunks; c += 2) {
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + c * 32), r);
                tmem_ld_wait();
                if (c == last_c) {
                    tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty + as);   // this warp no longer needs the TMEM stage
                }
                if (p.scale_num) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * alpha);
                }
                const int colbase = u.b0 + c * 32;            // (TMA-store path: global column)
                const int cl0 = c * 32;                       // tile-local column of this chunk
                const int cvalid = min(32, u.n_valid - cl0);  // valid columns of this chunk (may be <= 0)
                bool bias_done = false;
                if (atomic) {
                    // split-K: partial tiles are added into a zero-initialised C straight from the registers -- lane = row,
                    // its 32 consecutive columns leave as vector reductions (red.global.add.v4 / .v2.f32 by row alignment: the same
                    // four 32-byte sectors per row as a coalesced warp-wide atomicAdd, a quarter / half the instructions of the scalar
                    // form) -- so this mode needs no staging tile and the 32 KiB go to a third operand stage.
                    const int rl = rl0 + lane;
                    long orow = rl;
                    if (rmap && rl < u.m_valid) orow = rmap[rl];
                    if (rl < u.m_valid && orow >= 0 && cvalid > 0) {
                        float* o = Ct + orow * p.ldc + cl0;
                        if (add_bias) {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < cvalid) r[j] = __float_as_uint(__uint_as_float(r[j]) + biasp[cl0 + j]);
                        }
                        if ((reinterpret_cast<uintptr_t>(o) & 15) == 0) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                if (j + 3 < cvalid) {
                                    red_add_v4(o + j, __uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                               __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                                } else {
#pragma unroll
                                    for (int e = 0; e < 4; ++e)
                                        if (j + e < cvalid) atomicAdd(o + j + e, __uint_as_float(r[j + e]));
                                }
                            }
                        } else if ((reinterpret_cast<uintptr_t>(o) & 7) == 0) {
#pragma unroll
                            for (int j = 0; j < 32; j += 2) {
                                if (j + 1 < cvalid) red_add_v2(o + j, __uint_as_float(r[j]), __uint_as_float(r[j + 1]));
                                else if (j < cvalid) atomicAdd(o + j, __uint_as_float(r[j]));
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < cvalid) atomicAdd(o + j, __uint_as_float(r[j]));
                        }
                    }
                    continue;
                }
                if (p.amax_val) {                             // lane = row: 32 consecutive columns of it are in r[]
                    const float bl = (add_bias && lane < cvalid) ? biasp[cl0 + lane] : 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j)              // the bias is in: the store paths below must not add it again
                        r[j] = __float_as_uint(__uint_as_float(r[j]) + __shfl_sync(0xffffffffu, bl, j));
                    // a separate scan: fused into the loop above, the kernel compiled to 18-24 more registers
#pragma unroll
                    for (int j = 0; j < 32; ++j) {            // ascending columns: first max wins
                        const float v = __uint_as_float(r[j]);
                        if (j < cvalid && v > am_best) { am_best = v; am_idx = colbase + j; }
                    }
                    bias_done = true;
                }
                if constexpr (TMA_STORE) {
                    // chunks that lie fully inside the N tile (TMA clips at the matrix edge, not at the tile edge)
                    if (!atomic && BN - c * 32 >= 32) {
                        if (lane == 0) tma_store_wait_read();          // the previous store has finished reading `st`
                        __syncwarp();
                        const float bl = (add_bias && !bias_done && lane < cvalid) ? biasp[cl0 + lane] : 0.f;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {                 // lane = row: it needs the bias of all 32 columns
                            float v = __uint_as_float(r[j]) + __shfl_sync(0xffffffffu, bl, j);
                            if (p.relu) v = fmaxf(v, 0.f);
                            r[j] = __float_as_uint(v);
                        }
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4)                 // same swizzle as SWIZZLE_128B of a 128-byte-row box
                            *reinterpret_cast<float4*>(st + lane * STG_STRIDE + ((j4 ^ (lane & 7)) << 2)) =
                                make_float4(__uint_as_float(r[4 * j4]), __uint_as_float(r[4 * j4 + 1]),
                                            __uint_as_float(r[4 * j4 + 2]), __uint_as_float(r[4 * j4 + 3]));
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(&tmC, st, colbase, row0);
                            tma_store_commit();
                        }
                        continue;
                    }
                    if (lane == 0) tma_store_wait_read();              // legacy path below reuses the staging tile
                    __syncwarp();
                }
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4)   // row = lane; float4 slot j4 lives at (j4 ^ (row & 7)): conflict-free
                    *reinterpret_cast<float4*>(st + lane * STG_STRIDE + ((j4 ^ (lane & 7)) << 2)) =
                        make_float4(__uint_as_float(r[4 * j4]), __uint_as_float(r[4 * j4 + 1]),
                                    __uint_as_float(r[4 * j4 + 2]), __uint_as_float(r[4 * j4 + 3]));
                __syncwarp();
                if (vec && ((u.c_off & 3) == 0)) {
                    const int cl = (lane & 7) * 4;             // 4 consecutive columns per lane, 8 lanes per row
                    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (add_bias && !bias_done) {
                        if (cl + 0 < cvalid) bv.x = biasp[cl0 + cl + 0];
                        if (cl + 1 < cvalid) bv.y = biasp[cl0 + cl + 1];
                        if (cl + 2 < cvalid) bv.z = biasp[cl0 + cl + 2];
                        if (cl + 3 < cvalid) bv.w = biasp[cl0 + cl + 3];
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int rr = (lane >> 3) + 4 * i;
                        const int rl = rl0 + rr;
                        float4 v = *reinterpret_cast<const float4*>(st + rr * STG_STRIDE + (((lane & 7) ^ (rr & 7)) << 2));
                        v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
                        if (p.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                        long orow = rl;
                        if (rmap && rl < u.m_valid) orow = rmap[rl];
                        if (rl < u.m_valid && orow >= 0) {
                            float* o = Ct + orow * p.ldc + cl0 + cl;
                            if (cl + 3 < cvalid) {
                                *reinterpret_cast<float4*>(o) = v;
                            } else {
                                if (cl + 0 < cvalid) o[0] = v.x;
                                if (cl + 1 < cvalid) o[1] = v.y;
                                if (cl + 2 < cvalid) o[2] = v.z;
                            }
                        }
                    }
                } else {
                    const bool colok = lane < cvalid;
                    const float bv = (add_bias && !bias_done && colok) ? biasp[cl0 + lane] : 0.f;
#pragma unroll 8
                    for (int rr = 0; rr < 32; ++rr) {
                        const int rl = rl0 + rr;
                        long orow = rl;
                        if (rmap && rl < u.m_valid) orow = rmap[rl];
                        if (rl < u.m_valid && orow >= 0 && colok) {
                            float v = st[rr * STG_STRIDE + ((((lane >> 2) ^ (rr & 7)) << 2) | (lane & 3))] + bv;
                            float* o = Ct + orow * p.ldc + cl0 + lane;
                            if (atomic) {
                                atomicAdd(o, v);
                            } else {
                                if (p.relu) v = fmaxf(v, 0.f);
                                *o = v;
                            }
                        }
                    }
                }
                __syncwarp();
            }
            if (p.amax_val && rl0 + lane < u.m_valid) {
                const long o = (long)(u.a0 + rl0 + lane) * p.amax_ld + 2 * (u.b0 / BN) + half;
                p.amax_val[o] = am_best;
                p.amax_idx[o] = am_idx;
            }
        }
        if constexpr (TMA_STORE) {
            if (lane == 0) tma_store_wait_all();       // shared memory must outlive the bulk stores that read it
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
    }
}

// hi[r, c] = bf16(src[r, c]);  lo[r, c] = bf16(src - hi);  columns [C, Kp) are zeroed.   (lo may be null)
// One thread per 8 columns: two 128-bit loads when the source is 16-byte aligned there, one 128-bit store per plane.
__global__ void split_bf16_kernel(const float* __restrict__ src, long lds, long R, int C, __nv_bfloat16* __restrict__ hi,
                                  __nv_bfloat16* __restrict__ lo, long Kp) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long oct = Kp >> 3;
    if (i >= R * oct) return;
    const long r = i / oct;
    const int c = (int)(i - r * oct) * 8;
    float x[8];
    const float* p = src + r * lds + c;
    if (c + 8 <= C && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
        const float4 a = ldg_stream4(p), b = ldg_stream4(p + 4);
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
    } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = (c + e < C) ? p[e] : 0.f;
    }
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * e]), h1 = __float2bfloat16_rn(x[2 * e + 1]);
        hw[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        const __nv_bfloat16 l0 = __float2bfloat16_rn(x[2 * e] - __bfloat162float(h0));
        const __nv_bfloat16 l1 = __float2bfloat16_rn(x[2 * e + 1] - __bfloat162float(h1));
        lw[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
    }
    *reinterpret_cast<uint4*>(hi + r * Kp + c) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    if (lo) *reinterpret_cast<uint4*>(lo + r * Kp + c) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
}

// Transposing split: hi/lo [C, Rp] with hi[c, r] = bf16(src[r, c]); columns [R, Rp) zeroed.
__global__ void split_bf16_t_kernel(const float* __restrict__ src, long lds, int R, int C, __nv_bfloat16* __restrict__ hi,
                                    __nv_bfloat16* __restrict__ lo, long Rp) {
    __shared__ float tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (r < R && c < C) ? src[(long)r * lds + c] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i, r = r0 + threadIdx.x;
        if (c < C && r < Rp) {
            const float x = tile[threadIdx.x][i];
            const __nv_bfloat16 h = __float2bfloat16_rn(x);
            hi[(long)c * Rp + r] = h;
            if (lo) lo[(long)c * Rp + r] = __float2bfloat16_rn(x - __bfloat162float(h));
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D map over a row-major bf16 matrix [rows, Kp]: box = 64 (K) x box_rows, 128-byte swizzle, zero fill out of bounds.
static int make_map(CUtensorMap* m, const void* base, long rows, long Kp, int box_rows, long pitch = 0) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return CAPHN_EINVAL;
    if (pitch == 0) pitch = Kp;
    cuuint64_t dims[2] = {(cuuint64_t)Kp, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)pitch * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? CAPHN_OK : 1000 + (int)r;
}

// 2-D map over the fp32 output [M, N] (row pitch ldc): box = 32 columns (128 bytes) x 32 rows, 128-byte swizzle -- the
// layout of one epilogue warp's staging tile.  Only used by the TMA_STORE epilogue.
static int make_map_c(CUtensorMap* m, const float* C, long M, long N, long ldc) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return CAPHN_EINVAL;
    cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)ldc * 4};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(C), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? CAPHN_OK : 1000 + (int)r;
}

}  // namespace tc
}  // namespace caphn

using namespace caphn;

extern "C" {

// hi/lo [R, Kp] bf16 (Kp % 64 == 0, Kp >= C): the bf16x3 operand format of caphn_gemm_tc.  lo may be NULL (bf16 mode).
int caphn_split_bf16(const float* src, long lds, long R, int C, void* hi, void* lo, long Kp, void* stream) {
    if (R <= 0 || C <= 0 || Kp < C || (Kp & 63)) return CAPHN_EINVAL;
    if (((uintptr_t)hi & 15) || ((uintptr_t)lo & 15)) return CAPHN_EINVAL;
    const long n = R * (Kp >> 3);
    tc::split_bf16_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(
        src, lds, R, C, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, Kp);
    CAPHN_RETURN_LAST();
}

// Transposing variant: src [R, C] fp32 -> hi/lo [C, Rp] bf16 (Rp % 64 == 0, Rp >= R).
int caphn_split_bf16_t(const float* src, long lds, int R, int C, void* hi, void* lo, long Rp, void* stream) {
    if (R <= 0 || C <= 0 || Rp < R || (Rp & 63)) return CAPHN_EINVAL;
    dim3 grid(ceil_div(C, 32), ceil_div(Rp, 32));
    tc::split_bf16_t_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(src, lds, R, C, (__nv_bfloat16*)hi,
                                                                            (__nv_bfloat16*)lo, Rp);
    CAPHN_RETURN_LAST();
}

// C[M,N] (fp32, row stride ldc) = A B^T (+bias[n]) (ReLU) on the tensor cores, general operand layouts.
//   K-major operand  (x_mn = 0): hi/lo [rows = M or N, K cols], row pitch x_ld elements (x_ld % 8 == 0), zero padded to x_ld
//                                when K % 64 != 0 is irrelevant: TMA zero-fills out-of-range columns.
//   MN-major operand (x_mn = 1): hi/lo [K rows, M or N cols], row pitch x_ld -- i.e. the operand of a TRANSPOSED product
//                                (dW = dY^T X) read in place, no transposed copy.
// Alo == Blo == NULL selects plain bf16.  splitk: 0 = automatic, 1 = none, > 1 = split K, partial tiles added atomically.
static int gemm_tc_impl(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                        int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, int relu, int splitk,
                        float* amax_val, int* amax_idx, int amax_ld, void* stream, int* bn_used = nullptr,
                        const float* scale_num = nullptr, const float* scale_den = nullptr) {
    if (M <= 0 || N <= 0 || K <= 0 || ((Alo == nullptr) != (Blo == nullptr))) return CAPHN_EINVAL;
    if (scale_den && !scale_num) return CAPHN_EINVAL;
    if (amax_val && (!amax_idx || splitk > 1 || relu)) return CAPHN_EINVAL;
    if (amax_val) splitk = 1;
    if (((uintptr_t)Ahi & 15) || ((uintptr_t)Bhi & 15) || ((uintptr_t)Alo & 15) || ((uintptr_t)Blo & 15) ||
        (a_ld & 7) || (b_ld & 7))
        return CAPHN_EINVAL;
    const bool split = Alo != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    tc::TcParams p{};
    p.C = C; p.ldc = ldc; p.bias = bias; p.M = M; p.N = N; p.relu = relu; p.a_mn = a_mn ? 1 : 0; p.b_mn = b_mn ? 1 : 0;
    p.num_kb = (int)((K + tc::BK - 1) / tc::BK);
    p.K = (int)K;
    p.scale_num = scale_num; p.scale_den = scale_den;
    // A-stationary schedule (see TcParams::astat), used where the shape allows it; CAPHN_TC_ASTAT=0 switches it off
    const char* ae = getenv("CAPHN_TC_ASTAT");
    const bool astat_on = !(ae && atoi(ae) == 0);
    // N tile: one tile when N <= 256 (rounded up to 16, or to 64 for an MN-major B whose boxes are 64 wide), else 128
    if (N <= 256) {
        p.BN = b_mn ? ((N + 63) / 64) * 64 : ((N + 15) / 16) * 16;
    } else {
        // wide N: the tile width that minimises (waves over the 148 SMs) x (per-tile cost ~ BN + fixed part).  Matters when
        // there are only a few waves: the decode-step vocabulary projection (M = 512, N = 9684) is 304 tiles = 3 waves at
        // BN = 128 but 272 tiles = 2 waves at BN = 144.
        // With many waves the quantisation loss is small and BN = 128 keeps 3 operand stages in flight: left alone.
        const int step = b_mn ? 64 : 16;
        const long tm = ceil_div(M, tc::BM);
        const bool few_waves = tm * ceil_div(N, 128) <= 8L * kNumSMs;
        long best_cost = -1;
        p.BN = 128;
        for (int bn = 128; few_waves && bn <= 256; bn += step) {
            const long t = tm * ceil_div(N, bn);
            const long cost = ((t + kNumSMs - 1) / kNumSMs) * (bn + 32);
            if (best_cost < 0 || cost < best_cost) { best_cost = cost; p.BN = bn; }
        }
        if (!few_waves) {
            // many waves: the kernel is bound by the MMA's operand fetch from shared memory (a cta_group::1 MMA reads
            // 4 KB of A + 32 BN bytes of B per 64 BN / 128 cycles of math), so either A stays resident and BN = 128 keeps three
            // B stages (A-stationary schedule, short K), or the tile is as wide as it gets: BN = 256 moves 25 % fewer operand
            // bytes per flop (K = 200: 159 -> 144 us at M = 10240, N = 9684, with two 96 KB stages).
            const size_t slab0 = (size_t)p.num_kb * (split ? 2 : 1) * tc::TILE_BYTES;
            const size_t fixed0 = (size_t)tc::STG_FLOATS_V2 * 4 + (2 * tc::MAX_STAGES + 6) * 8 + 16 + 1024;
            const size_t bst0 = (size_t)(split ? 2 : 1) * 128 * tc::BK * 2;
            const bool astat_fits = astat_on && !a_mn && !b_mn && slab0 + fixed0 + 3 * bst0 <= tc::SMEM_BUDGET;
            if (!astat_fits) p.BN = 256;
        }
        // tuning knob (tools/bench_gemm.py): CAPHN_TC_BN_FORCE=<multiple of 16 (64 for an MN-major B) in 128..256>
        if (const char* f = getenv("CAPHN_TC_BN_FORCE")) {
            const int bn = atoi(f);
            if (bn >= 128 && bn <= 256 && bn % step == 0) p.BN = bn;
        }
    }
    const int tiles = ceil_div(M, tc::BM) * ceil_div(N, p.BN);
    if (splitk <= 0) {
        // smallest split whose unit count fills the 148 SMs to >= 90 % (or the best available), >= 4 k-blocks per unit
        splitk = 1;
        if (!relu && tiles < 3 * kNumSMs) {
            double best = 0.0;
            const int smax = p.num_kb / 4 > 32 ? 32 : (p.num_kb / 4 < 1 ? 1 : p.num_kb / 4);
            for (int s = 1; s <= smax; ++s) {
                const long units = (long)tiles * s;
                const double eff = (double)units / (double)(((units + kNumSMs - 1) / kNumSMs) * kNumSMs);
                if (eff > best + 0.02) { best = eff; splitk = s; }
                if (eff >= 0.9) break;
            }
        }
    }
    if (splitk > 1 && relu) return CAPHN_EINVAL;
    p.kb_per = (p.num_kb + splitk - 1) / splitk;
    p.splitk = (p.num_kb + p.kb_per - 1) / p.kb_per;
    p.b_bytes = p.BN * tc::BK * 2;
    p.stage_bytes = (split ? 2 : 1) * (tc::TILE_BYTES + p.b_bytes);
    bool tma_store = false;
    {   // TMA-store epilogue: full 32-column chunks leave through cp.async.bulk.tensor stores.  Bit-identical to the default
        // epilogue and 2-9 % faster on the logits products (profiles/r02_gemm_tma_store.txt); N % 4 == 0 only (a clipped
        // edge box of a ragged N did not match in round 1 -- those shapes keep the default epilogue).  CAPHN_TC_TMA_STORE=0
        // switches it off.
        const char* e = getenv("CAPHN_TC_TMA_STORE");
        tma_store = !(e && e[0] == '0') && p.splitk == 1 && (ldc % 4 == 0) && (N % 4 == 0) && ((uintptr_t)C % 16 == 0);
    }
    const size_t slab = (size_t)p.num_kb * (split ? 2 : 1) * tc::TILE_BYTES;
    const size_t bstage = (size_t)(split ? 2 : 1) * p.b_bytes;
    // A-stationary schedule: K-major operands, no split-K, >= 4 tiles per CTA, >= 4 n-tiles, the A slab and three B stages
    // fit in shared memory.
    const bool astat_shape = astat_on && !a_mn && !b_mn && p.splitk == 1 && ceil_div(N, p.BN) >= 4 && tiles >= 4 * kNumSMs;
    // one staging tile per epilogue warp; none under split-K, where the epilogue adds from registers
    const size_t fixed = (size_t)(p.splitk > 1 ? 0 : tc::STG_FLOATS_V2 * 4) + (2 * tc::MAX_STAGES + 6) * 8 + 16 + 1024;
    int stages;
    if (astat_shape && slab + fixed + 3 * bstage <= tc::SMEM_BUDGET) {
        p.astat = 1;
        p.a_slab_bytes = (int)slab;
        p.stage_bytes = (int)bstage;
        stages = (int)((tc::SMEM_BUDGET - fixed - slab) / bstage);
    } else {
        if (fixed + 2 * (size_t)p.stage_bytes > tc::SMEM_BUDGET) return CAPHN_EINVAL;
        stages = (int)((tc::SMEM_BUDGET - fixed) / p.stage_bytes);
    }
    if (stages > tc::MAX_STAGES) stages = tc::MAX_STAGES;
    if (stages < 2) return CAPHN_EINVAL;
    p.stages = stages;
    p.tmem_cols = (2 * p.BN <= 256) ? 256u : 512u;
    const size_t smem = (size_t)p.a_slab_bytes + (size_t)stages * p.stage_bytes + fixed;
    if (bn_used) *bn_used = p.BN;
    if (amax_val) {
        if (amax_ld < 2 * ceil_div(N, p.BN)) return CAPHN_EINVAL;
        p.amax_val = amax_val; p.amax_idx = amax_idx; p.amax_ld = amax_ld;
    }
    if (p.splitk > 1) {
        if (ldc == N) {
            CAPHN_CHECK(cudaMemsetAsync(C, 0, (size_t)M * N * sizeof(float), st));
        } else {
            CAPHN_CHECK(cudaMemset2DAsync(C, (size_t)ldc * sizeof(float), 0, (size_t)N * sizeof(float), (size_t)M, st));
        }
    }
    CUtensorMap mAh, mAl, mBh, mBl;
    int rc;
    // K-major: dims {K, rows}, box {64, rows-tile}.  MN-major: dims {MN, K}, box {64, 64}.
    if (!a_mn) {
        if ((rc = tc::make_map(&mAh, Ahi, M, K, tc::BM, a_ld))) return rc;
        if ((rc = tc::make_map(&mAl, split ? Alo : Ahi, M, K, tc::BM, a_ld))) return rc;
    } else {
        if ((rc = tc::make_map(&mAh, Ahi, K, M, 64, a_ld))) return rc;
        if ((rc = tc::make_map(&mAl, split ? Alo : Ahi, K, M, 64, a_ld))) return rc;
    }
    if (!b_mn) {
        if ((rc = tc::make_map(&mBh, Bhi, N, K, p.BN, b_ld))) return rc;
        if ((rc = tc::make_map(&mBl, split ? Blo : Bhi, N, K, p.BN, b_ld))) return rc;
    } else {
        if ((rc = tc::make_map(&mBh, Bhi, K, N, 64, b_ld))) return rc;
        if ((rc = tc::make_map(&mBl, split ? Blo : Bhi, K, N, 64, b_ld))) return rc;
    }
    const long units = (long)tiles * p.splitk;
    const int grid = units < kNumSMs ? (int)units : kNumSMs;
    CUtensorMap mC{};
    if (tma_store && (rc = tc::make_map_c(&mC, C, M, N, ldc))) return rc;
    if (split && tma_store) {
        CAPHN_CHECK(cudaFuncSetAttribute(tc::gemm_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc_kernel<true, true><<<grid, tc::THREADS_V2, smem, st>>>(mAh, mAl, mBh, mBl, mC, p);
    } else if (split) {
        CAPHN_CHECK(cudaFuncSetAttribute(tc::gemm_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc_kernel<true><<<grid, tc::THREADS_V2, smem, st>>>(mAh, mAl, mBh, mBl, mC, p);
    } else if (tma_store) {
        CAPHN_CHECK(cudaFuncSetAttribute(tc::gemm_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc_kernel<false, true><<<grid, tc::THREADS_V2, smem, st>>>(mAh, mAl, mBh, mBl, mC, p);
    } else {
        CAPHN_CHECK(cudaFuncSetAttribute(tc::gemm_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc_kernel<false><<<grid, tc::THREADS_V2, smem, st>>>(mAh, mAl, mBh, mBl, mC, p);
    }
    CAPHN_RETURN_LAST();
}

// Grouped product (the per-style grouped GEMM of BASELINE.json's north star): `num_units` output tiles, each described by
// one GUnit record (12 int32 words = 48 bytes, see struct GUnit): which A rows / B rows / K range it multiplies and where it writes.
// Operands are 2-D bf16 arrays (hi, optional lo) with `*_inner` contiguous elements per row, `*_outer` rows and row pitch
// `*_ld`: K-major (x_mn = 0: inner = K, outer = operand rows) or MN-major (x_mn = 1: inner = operand rows, outer = K).
// A tile reads 128 A rows and BN B rows starting at the unit's a_row / b_row (rows beyond m_valid / n_valid are read --
// TMA zero-fills past the array -- but never written), accumulates nkb 64-wide k blocks from ka0 (in A) and kb0 (in B) (the caller pads each
// group's K range to a multiple of 64 with zero rows/columns in at least one operand) and writes C + c_off (+ bias), or,
// with `rowmap`, row r of the tile to C row rowmap[map0 + r] (negative = skip).  BN: multiple of 16 (64 for MN-major B).
int caphn_gemm_tc_grouped(const void* Ahi, const void* Alo, long a_inner, long a_outer, long a_ld, int a_mn,
                          const void* Bhi, const void* Blo, long b_inner, long b_outer, long b_ld, int b_mn, float* C,
                          long ldc, const float* bias, const int* rowmap, const void* units, int num_units, int BN,
                          void* stream) {
    if (num_units <= 0 || !units || !Ahi || !Bhi || ((Alo == nullptr) != (Blo == nullptr))) return CAPHN_EINVAL;
    if (((uintptr_t)Ahi & 15) || ((uintptr_t)Bhi & 15) || ((uintptr_t)Alo & 15) || ((uintptr_t)Blo & 15) || (a_ld & 7) ||
        (b_ld & 7) || ((uintptr_t)units & 3))
        return CAPHN_EINVAL;
    if (BN < 16 || BN > 256 || (BN % (b_mn ? 64 : 16)) != 0) return CAPHN_EINVAL;
    const bool split = Alo != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    tc::TcParams p{};
    p.C = C; p.ldc = ldc; p.bias = bias; p.units = (const tc::GUnit*)units; p.rowmap = rowmap; p.num_units = num_units;
    p.M = 0; p.N = 0; p.relu = 0; p.a_mn = a_mn ? 1 : 0; p.b_mn = b_mn ? 1 : 0; p.num_kb = 0; p.BN = BN;
    p.splitk = 1; p.kb_per = 0;
    p.b_bytes = p.BN * tc::BK * 2;
    p.stage_bytes = (split ? 2 : 1) * (tc::TILE_BYTES + p.b_bytes);
    const size_t fixed = (size_t)tc::STG_FLOATS_V2 * 4 + (2 * tc::MAX_STAGES + 6) * 8 + 16 + 1024;
    int stages = (int)((tc::SMEM_BUDGET - fixed) / p.stage_bytes);
    if (stages > tc::MAX_STAGES) stages = tc::MAX_STAGES;
    if (stages < 2) return CAPHN_EINVAL;
    p.stages = stages;
    p.tmem_cols = (2 * p.BN <= 256) ? 256u : 512u;
    const size_t smem = (size_t)stages * p.stage_bytes + fixed;
    CUtensorMap mAh, mAl, mBh, mBl, mC{};
    int rc;
    // make_map(map, base, rows = outer extent, Kp = inner extent, box rows, pitch): box = 64 inner x box rows
    if ((rc = tc::make_map(&mAh, Ahi, a_outer, a_inner, a_mn ? 64 : tc::BM, a_ld))) return rc;
    if ((rc = tc::make_map(&mAl, split ? Alo : Ahi, a_outer, a_inner, a_mn ? 64 : tc::BM, a_ld))) return rc;
    if ((rc = tc::make_map(&mBh, Bhi, b_outer, b_inner, b_mn ? 64 : p.BN, b_ld))) return rc;
    if ((rc = tc::make_map(&mBl, split ? Blo : Bhi, b_outer, b_inner, b_mn ? 64 : p.BN, b_ld))) return rc;
    const int grid = num_units < kNumSMs ? num_units : kNumSMs;
    if (split) {
        CAPHN_CHECK(cudaFuncSetAttribute(tc::gemm_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc_kernel<true><<<grid, tc::THREADS_V2, smem, st>>>(mAh, mAl, mBh, mBl, mC, p);
    } else {
        CAPHN_CHECK(cudaFuncSetAttribute(tc::gemm_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::gemm_tc_kernel<false><<<grid, tc::THREADS_V2, smem, st>>>(mAh, mAl, mBh, mBl, mC, p);
    }
    CAPHN_RETURN_LAST();
}

int caphn_gemm_tc_ex(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                     int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, int relu, int splitk,
                     void* stream) {
    return gemm_tc_impl(Ahi, Alo, a_ld, a_mn, Bhi, Blo, b_ld, b_mn, K, C, ldc, bias, M, N, relu, splitk, nullptr, nullptr, 0,
                        stream);
}

// caphn_gemm_tc_ex with a device-side scalar on the product: C = (scale_num[0] / max(scale_den[0], 1)) * A B^T (+bias).
// scale_den may be NULL (= 1).  Used by the fused cross-entropy nodes: A or B is the unscaled gradient operand written by
// caphn_ce_fwd_split, scale_num = grad_output of the loss, scale_den = number of valid rows (lossbuf + 1).
int caphn_gemm_tc_scaled(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                         int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, int splitk,
                         const float* scale_num, const float* scale_den, void* stream) {
    if (!scale_num) return CAPHN_EINVAL;
    return gemm_tc_impl(Ahi, Alo, a_ld, a_mn, Bhi, Blo, b_ld, b_mn, K, C, ldc, bias, M, N, 0, splitk, nullptr, nullptr, 0,
                        stream, nullptr, scale_num, scale_den);
}

// caphn_gemm_tc_ex + row arg-max partials in the epilogue (greedy decode: logits_t = h_t W^T + b, next word = arg-max):
// amax_val / amax_idx [M, amax_ld] receive, per row, one (max, column) pair per (n-tile, epilogue-warp half) in slots
// 0 .. 2*ceil(N/BN)-1 (slots of halves that read no column hold -inf).  amax_ld >= 2*ceil(N/128) always suffices.
// *nparts (host int, optional) = number of slots written.  Finish with caphn_argmax_finish_gather.
int caphn_gemm_tc_amax(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                       int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, float* amax_val,
                       int* amax_idx, int amax_ld, int* nparts, void* stream) {
    if (!amax_val || !amax_idx) return CAPHN_EINVAL;
    int bn = 0;
    const int rc = gemm_tc_impl(Ahi, Alo, a_ld, a_mn, Bhi, Blo, b_ld, b_mn, K, C, ldc, bias, M, N, 0, 1, amax_val, amax_idx,
                                amax_ld, stream, &bn);
    if (nparts && bn > 0) *nparts = 2 * ceil_div(N, bn);
    return rc;
}

// Both operands K-major with the same padded pitch Kp (Kp % 64 == 0): the original entry point.
int caphn_gemm_tc(const void* Ahi, const void* Alo, const void* Bhi, const void* Blo, long Kp, float* C, long ldc,
                  const float* bias, int M, int N, int relu, int splitk, void* stream) {
    if (Kp <= 0 || (Kp & 63)) return CAPHN_EINVAL;
    return caphn_gemm_tc_ex(Ahi, Alo, Kp, 0, Bhi, Blo, Kp, 0, Kp, C, ldc, bias, M, N, relu, splitk, stream);
}

}  // extern "C"
