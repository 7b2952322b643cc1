// tc_gemm.cu -- tcgen05 (5th-gen tensor core) GEMM with fp32-level accuracy for the IQN / ensemble dense
// layers, forward and backward (sm_100a only).
//
//     C[b] (M x N) = act( sum_kb  A[kb|b] (M x K) . B[kb|b]^T (N x K)  + bias[b] )        fp32 in, fp32 out
//
// The reference computes these layers in fp32 (nn.Linear, prism/agents/models/ffnn_model.py:61-76,
// iqn_model.py:30-46, 89-93, q_ensemble.py:26-48) and parity is judged at 1e-4 relative on losses and
// gradients, which a single TF32 or BF16 pass (~1e-3) cannot hold.  So every operand is split on the fly
// into a TF32 "hi" part and a TF32 "lo" residual and each product is issued as three tensor-core MMAs
// lo.hi + hi.lo + hi.hi accumulating in fp32 in TENSOR MEMORY -- error ~1e-6 at a third of the TF32 rate.
//
// Structure: persistent, warp-specialised, one CTA per SM, 448 threads:
//   warp 0      TMA producer: cp.async.bulk.tensor (128-byte swizzle) of the raw fp32 A (128 x 32) and
//               B (BN x 32) tiles into a ring of shared-memory stages, completion on mbarriers;
//   warps 2-5   splitters: one element-wise pass over the landed stage, lo = x - tf32(x) written to a twin
//               tile at the SAME swizzled offset (layout-agnostic, bank-conflict-free); the raw tile itself
//               is the "hi" operand (the tensor core reads only the upper 19 bits of each fp32 word; mode 1
//               rewrites it in place with the round-to-nearest TF32 value instead);
//   warp 1      MMA issuer: one thread issues tcgen05.mma.cta_group::1.kind::tf32 (M 128, N BN, K 8) from
//               shared-memory descriptors, 12 per stage; tcgen05.commit frees the stage / publishes the tile;
//   warps 6-13  epilogue: tcgen05.ld 32x32b of the finished accumulator (double-buffered in TMEM for BN <= 128, so
//               the next tile's MMAs overlap), + bias, ReLU, optional row-broadcast multiplier, 128-byte-swizzled
//               32 x 32 tile in shared memory, cp.async.bulk.tensor store (or a raw stream-K partial tile).
// Scheduling is stream-K: equal contiguous ranges of (tile, K block) work per CTA; tiles cut by a range
// boundary leave partial tiles in a bounded workspace and a fix-up kernel sums them in a fixed order.
// Operands may be K-major (row-major M x K) or MN-major (row-major K x M, i.e. the transposed view), which
// is what the backward GEMMs need (dX = dZ W, dW = dZ^T X) -- no transposed copies are ever made.
#include "common.cuh"
#include <cuda.h>

namespace {

using namespace pb;

constexpr int BM = 128;           // K block (BK, template): 32 floats = one 128-byte swizzled row, or 16 = 64-byte rows
constexpr int NUM_THREADS = 448;           // warp 0 TMA, warp 1 MMA, warps 2-5 splitters, warps 6-13 epilogue
constexpr int SMEM_BUDGET = 200 * 1024;          // operand stages; barriers live in static shared memory

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred P1;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
                     "selp.b32 %0, 1, 0, P1;\n\t}"
                     : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap *map, uint32_t src, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor, descriptor version 1 (sm_100).
//   K-major tile  (rows x 32 floats, row = 128 B), layout 2 = SWIZZLE_128B (16-byte chunks, 8-row atom):
//       SBO = 1024 (next 8 rows), LBO unused
//   MN-major tile (groups of [32 K-rows x 32 M/N floats], K-row = 128 B), layout 1 = SWIZZLE_128B_BASE32B
//   (32-byte chunks, 4-row atom) -- the only swizzle the tensor core accepts for MN-major 32-bit operands
//   (TMA side: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B):
//       SBO = 512 (next 4 K-rows), LBO = 4096 (next 32 M/N)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}

// instruction descriptor: D fp32, A/B tf32, M = 128, N = n; major bits: 0 = K-major, 1 = MN-major
__host__ __device__ constexpr uint32_t make_idesc(int n, int a_mn, int b_mn)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_c, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
                 ::"r"(tmem_c), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
                 : "memory");
}

struct TcParams {
    float *C;
    const float *bias;
    float *ws;                     // partial tiles [3 * grid][128][BN]: per CTA its first cut tile, its last cut tile, and
                                   // the running sum of a whole tile accumulated in chunks (kc)
    int kc;                        // longest accumulation chain in TMEM, in K blocks (0 = unlimited), see SegIter
    long long c_bs, bias_bs;
    int ldc;
    int M, N;
    int kblocks;                   // 32-wide K blocks per K batch
    int kbatches;                  // operand batches summed into one output (shared-input dgrad); else 1
    int batch;                     // output batches
    int a_batched, b_batched;
    int tiles_m, tiles_n;
    int bn;                        // tile width of this launch (fix-up kernel)
    int fix_by_boundary;           // fix-up grid: 1 = one block column per CTA-range boundary, 0 = one per tile
    long long work, per_cta;       // stream-K: work = tiles * kb_total K blocks, dealt out in equal contiguous ranges
    int act;                       // 0 none, 1 ReLU
    int split_mode;                // 0: hi = raw word (hardware truncation); 1: hi rewritten as cvt.rna.tf32
    const float *mul;              // optional epilogue multiplier: out *= mul[(row % mul_rows) * ld_mul + col]
    int mul_rows, ld_mul;
    int deep_epi;                  // 1: two operand stages + four store buffers per epilogue warp (short K loops)
    int tma_store;                 // 1: epilogue through a swizzled shared-memory tile + cp.async.bulk.tensor store (tmC);
                                   // 0: direct per-row stores (C rows not 16-byte aligned)
};

// Stream-K schedule: the (tile, K block) work items are numbered tile-major (tn fastest, then tm, then batch)
// and CTA c owns the contiguous range [c * per_cta, (c + 1) * per_cta).  A range is cut into segments at tile
// boundaries; a segment covering all of a tile's K blocks is finished by the epilogue directly, any other
// segment leaves a raw partial tile in the workspace (slot 2c for the CTA's first segment, 2c + 1 for its
// last -- the segments in between are whole tiles) and tc_streamk_fixup_kernel sums the cut tiles.
//
// Accumulation chains.  The tensor core adds into its fp32 accumulator with truncation, not round-to-nearest: every
// MMA loses ~half an ulp of the accumulator in the same direction, so a chain of n MMAs drifts by ~n * 3e-8
// relative (measured: -4.2e-5 of the result per 2048 floats of K on same-signed products) -- 1.4e-4 for the K = 32768
// weight gradients of configs[4] against the fp32 CPU oracle (tests/test_gpu_config_shapes.py).  g.kc > 0 caps a chain at kc K blocks: a segment is
// issued as CHUNKS of <= kc blocks, each into a fresh TMEM accumulator (the two accumulators alternate, so the tensor
// pipe never waits), and the epilogue warps add the chunks in round-to-nearest fp32 -- the running sum lives in the
// CTA's own workspace slot (L2-resident, read and written by the same thread, fixed order: deterministic).
constexpr int SLOTS_PER_CTA = 3;

struct Seg { int b, tm, tn, kb0, kb1, slot; bool whole, first, last; };

struct SegIter {
    long long pos, end, start;
    int kb_total;
    __device__ __forceinline__ SegIter(const TcParams &g)
    {
        start = pos = (long long)blockIdx.x * g.per_cta;
        end = min(g.work, pos + g.per_cta);
        kb_total = g.kblocks * g.kbatches;
    }
    // one CHUNK per call: [kb0, kb1) of tile (b, tm, tn); first / last chunk of its segment
    __device__ __forceinline__ bool next(const TcParams &g, Seg &w)
    {
        if (pos >= end) return false;
        const long long t = pos / kb_total;
        const long long t0 = t * kb_total;
        const long long s0 = max(start, t0), s1 = min(end, t0 + kb_total);      // the segment of this tile
        w.whole = (s0 == t0 && s1 == t0 + kb_total);
        long long c1 = s1;
        if (g.kc > 0 && s1 - s0 > g.kc) {
            const long long n_chunks = (s1 - s0 + g.kc - 1) / g.kc, len = (s1 - s0 + n_chunks - 1) / n_chunks;
            c1 = min(s1, s0 + ((pos - s0) / len + 1) * len);
        }
        w.first = (pos == s0);
        w.last = (c1 == s1);
        w.kb0 = (int)(pos - t0);
        w.kb1 = (int)(c1 - t0);
        w.slot = SLOTS_PER_CTA * (int)blockIdx.x + (w.whole ? 2 : (s0 == start ? 0 : 1));
        int u = (int)t;
        w.tn = u % g.tiles_n; u /= g.tiles_n;
        w.tm = u % g.tiles_m; w.b = u / g.tiles_m;
        pos = c1;
        return true;
    }
};

template <int BN, int BK, int A_MN, int B_MN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const TcParams g)
{
    constexpr int A_BYTES = BM * BK * 4, B_BYTES = BN * BK * 4, RAW_BYTES = A_BYTES + B_BYTES;
    constexpr int STAGE_BYTES = 2 * RAW_BYTES;                       // raw (hi) | lo
    constexpr int MAX_STAGES = SMEM_BUDGET / STAGE_BYTES;
    // short K loops (epilogue-bound, e.g. the 64-wide cosine basis) trade operand stages for a deeper ring of
    // epilogue store buffers: g.deep_epi = 4 x 4 KB per epilogue warp and only two operand stages
    constexpr bool DEEP_OK = 2 * STAGE_BYTES + 65536 <= MAX_STAGES * STAGE_BYTES + 32768;
    const bool deep = DEEP_OK && g.deep_epi;
    const int STAGES = deep ? 2 : MAX_STAGES;
    const int EPI_BUFS = deep ? 2 : 1;                               // 4 KB store buffers per epilogue warp (8 warps)
    constexpr int ACC = (2 * BN <= 512) ? 2 : 1;
    constexpr uint32_t TMEM_COLS = (uint32_t)(ACC * BN);
    static_assert(MAX_STAGES >= 2, "pipeline needs two stages");
    static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS >= 32 && TMEM_COLS <= 512, "TMEM columns");

    extern __shared__ uint8_t smem_dyn[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    uint8_t *staging = smem + STAGES * STAGE_BYTES;                  // 8 epilogue warps x EPI_BUFS x (32 rows x 128 B)
    __shared__ uint64_t bar_full[MAX_STAGES], bar_ready[MAX_STAGES], bar_empty[MAX_STAGES];
    __shared__ uint64_t bar_acc_full[ACC], bar_acc_empty[ACC];
    __shared__ uint32_t tmem_base_slot;
    __shared__ __align__(16) float bias_s[BN];

    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;

    if (t == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_ready[s], 4); mbar_init(&bar_empty[s], 1); }
        for (int a = 0; a < ACC; ++a) { mbar_init(&bar_acc_full[a], 1); mbar_init(&bar_acc_empty[a], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
        if (g.tma_store) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmC) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                     "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            uint32_t it = 0;
            SegIter segs(g);
            Seg w;
            while (segs.next(g, w)) {
                const int m0 = w.tm * BM, n0 = w.tn * BN;
                for (int kb = w.kb0; kb < w.kb1; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&bar_empty[s], ((it / STAGES) & 1) ^ 1);
                    const int kbatch = kb / g.kblocks, k0 = (kb % g.kblocks) * BK;
                    const int zb = g.kbatches > 1 ? kbatch : w.b;
                    const int za = g.a_batched ? zb : 0, zbb = g.b_batched ? zb : 0;
                    const uint32_t a_dst = smem_u32(smem + s * STAGE_BYTES), b_dst = a_dst + A_BYTES;
                    mbar_expect_tx(&bar_full[s], RAW_BYTES);
                    if (A_MN) {
#pragma unroll
                        for (int gI = 0; gI < BM / 32; ++gI) tma_load_3d(a_dst + gI * (BK * 128), &tmA, &bar_full[s], m0 + gI * 32, k0, za);
                    } else {
                        tma_load_3d(a_dst, &tmA, &bar_full[s], k0, m0, za);
                    }
                    if (B_MN) {
#pragma unroll
                        for (int gI = 0; gI < BN / 32; ++gI) tma_load_3d(b_dst + gI * (BK * 128), &tmB, &bar_full[s], n0 + gI * 32, k0, zbb);
                    } else {
                        tma_load_3d(b_dst, &tmB, &bar_full[s], k0, n0, zbb);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(BN, A_MN, B_MN);
            // K-major rows are BK * 4 bytes: SWIZZLE_128B (layout 2, 8-row group = 1024 B) for BK = 32,
            // SWIZZLE_64B (layout 4, 8-row group = 512 B) for BK = 16
            constexpr uint32_t K_LAY = BK == 32 ? 2 : 4, K_SBO = BK * 4 * 8;
            constexpr uint32_t A_LBO = A_MN ? BK * 128 : 16, B_LBO = B_MN ? BK * 128 : 16;
            constexpr uint32_t A_SBO = A_MN ? 512 : K_SBO, B_SBO = B_MN ? 512 : K_SBO;
            constexpr uint32_t A_LAY = A_MN ? 1 : K_LAY, B_LAY = B_MN ? 1 : K_LAY;
            constexpr uint32_t A_KSTEP = A_MN ? 1024 : 32, B_KSTEP = B_MN ? 1024 : 32;   // bytes per K = 8
            uint32_t it = 0, ui = 0;
            SegIter segs(g);
            Seg w;
            for (; segs.next(g, w); ++ui) {
                const int acc = ui % ACC;
                mbar_wait(&bar_acc_empty[acc], ((ui / ACC) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tmem_c = tmem_base + (uint32_t)(acc * BN);
                for (int kb = w.kb0; kb < w.kb1; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(&bar_full[s], ph);
                    mbar_wait(&bar_ready[s], ph);
                    tc_fence_after();
                    const uint32_t ah = smem_u32(smem + s * STAGE_BYTES), bh = ah + A_BYTES;
                    const uint32_t al = ah + RAW_BYTES, bl = bh + RAW_BYTES;
#pragma unroll
                    for (int ks = 0; ks < BK / 8; ++ks) {
                        const uint64_t dah = make_desc(ah + ks * A_KSTEP, A_LBO, A_SBO, A_LAY);
                        const uint64_t dal = make_desc(al + ks * A_KSTEP, A_LBO, A_SBO, A_LAY);
                        const uint64_t dbh = make_desc(bh + ks * B_KSTEP, B_LBO, B_SBO, B_LAY);
                        const uint64_t dbl = make_desc(bl + ks * B_KSTEP, B_LBO, B_SBO, B_LAY);
                        umma_tf32(tmem_c, dal, dbh, idesc, (kb > w.kb0 || ks > 0) ? 1u : 0u);   // small terms first
                        umma_tf32(tmem_c, dah, dbl, idesc, 1u);
                        umma_tf32(tmem_c, dah, dbh, idesc, 1u);
                    }
                    umma_commit(&bar_empty[s]);                       // stage reusable once these MMAs retire
                }
                umma_commit(&bar_acc_full[acc]);                      // accumulator complete
            }
        }
    } else if (warp < 6) {
        // ------------------------------------------------------------------ splitters (128 threads)
        const int st = t - 64;
        uint32_t it = 0;
        SegIter segs(g);
        Seg w;
        while (segs.next(g, w)) {
            for (int kb = w.kb0; kb < w.kb1; ++kb, ++it) {
                const int s = it % STAGES;
                mbar_wait(&bar_full[s], (it / STAGES) & 1);
                float4 *raw = reinterpret_cast<float4 *>(smem + s * STAGE_BYTES);
                float4 *lo = reinterpret_cast<float4 *>(smem + s * STAGE_BYTES + RAW_BYTES);
                constexpr int N4 = RAW_BYTES / 16, PER = N4 / 128;
                static_assert(N4 % 128 == 0 && PER % 2 == 0, "split loop shape");
                if (g.split_mode == 0) {
                    constexpr int UN = (PER % 4 == 0) ? 4 : 2;
#pragma unroll
                    for (int j0 = 0; j0 < PER; j0 += UN) {
                        float4 v[UN];
#pragma unroll
                        for (int j = 0; j < UN; ++j) v[j] = raw[st + (j0 + j) * 128];
#pragma unroll
                        for (int j = 0; j < UN; ++j) {
                            float4 l;
                            l.x = v[j].x - __uint_as_float(__float_as_uint(v[j].x) & 0xFFFFE000u);
                            l.y = v[j].y - __uint_as_float(__float_as_uint(v[j].y) & 0xFFFFE000u);
                            l.z = v[j].z - __uint_as_float(__float_as_uint(v[j].z) & 0xFFFFE000u);
                            l.w = v[j].w - __uint_as_float(__float_as_uint(v[j].w) & 0xFFFFE000u);
                            lo[st + (j0 + j) * 128] = l;
                        }
                    }
                } else {
#pragma unroll 2
                    for (int j = 0; j < PER; ++j) {
                        const float4 v = raw[st + j * 128];
                        float4 h, l;
                        uint32_t r;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v.x)); h.x = __uint_as_float(r); l.x = v.x - h.x;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v.y)); h.y = __uint_as_float(r); l.y = v.y - h.y;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v.z)); h.z = __uint_as_float(r); l.z = v.z - h.z;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v.w)); h.w = __uint_as_float(r); l.w = v.w - h.w;
                        raw[st + j * 128] = h;
                        lo[st + j * 128] = l;
                    }
                }
                fence_async_smem();                                   // generic-proxy writes -> tensor-core (async) proxy
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_ready[s]);
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 6-13)
        // two warps per TMEM lane quarter (a warp may only touch lanes 32 * (warp % 4) ..): one takes the even
        // 32-column chunks of the tile, the other the odd ones -- twice the loads / stores in flight
        const int q = warp & 3;
        const int half = (warp - 6) >> 2;
        const int et = t - 192;                                       // 0..255 within the epilogue warps
        uint32_t ui = 0, chunk = 0;
        const bool vec_ok = (g.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0) && (g.c_bs % 4 == 0);
        const bool mul_vec = g.mul && ((reinterpret_cast<uintptr_t>(g.mul) & 15) == 0) && (g.ld_mul % 4 == 0);
        const bool staged = g.tma_store != 0;
        uint8_t *stg = staging + (warp - 6) * (EPI_BUFS * 4096);
        SegIter segs(g);
        Seg w;
        for (; segs.next(g, w); ++ui) {
            const int acc = ui % ACC;
            const bool partial = !w.whole;                            // the segment's result goes to the workspace
            const bool fin = w.last;                                  // this chunk completes its segment
            const int row0 = w.tm * BM + q * 32, row = row0 + lane, n0 = w.tn * BN;
            // the tile's bias row goes to shared memory while the MMAs are still running (named barriers among the
            // four epilogue warps: everyone is done with the previous tile's row / the new row is published)
            float *bias_t = bias_s;
            const bool has_bias = g.bias && !partial && fin;
            if (g.bias) {
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (has_bias) {
                    const float *bsrc = g.bias + (size_t)w.b * g.bias_bs;
                    for (int c = et; c < BN; c += 256) bias_t[c] = (n0 + c < g.N) ? __ldg(bsrc + n0 + c) : 0.f;
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
            }
            mbar_wait(&bar_acc_full[acc], (ui / ACC) & 1);
            tc_fence_after();
            const bool relu = g.act == 1 && !partial && fin;
            const bool use_mul = g.mul && !partial && fin;
            float *crow = g.C + (size_t)w.b * g.c_bs + (size_t)row * g.ldc;
            float4 *prow = reinterpret_cast<float4 *>(g.ws + ((size_t)w.slot * BM + q * 32 + lane) * BN);
            // multiplier tile of one chunk, COALESCED (lane l: 16-byte chunk (l & 7) of rows 4i + (l >> 3)); requested one
            // chunk ahead so that its latency hides behind the previous chunk's TMEM load and stores
            float4 mreg[8], mnext[8];
            auto load_mul = [&](float4 (&m)[8], int c0) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int rr = 4 * i + (lane >> 3), col = c0 + (lane & 7) * 4;
                    const float *mrow = g.mul + (size_t)((row0 + rr) % g.mul_rows) * g.ld_mul;
                    if (mul_vec && col + 3 < g.N) m[i] = __ldg(reinterpret_cast<const float4 *>(mrow + col));
                    else {
                        m[i].x = col < g.N ? __ldg(mrow + col) : 0.f;
                        m[i].y = col + 1 < g.N ? __ldg(mrow + col + 1) : 0.f;
                        m[i].z = col + 2 < g.N ? __ldg(mrow + col + 2) : 0.f;
                        m[i].w = col + 3 < g.N ? __ldg(mrow + col + 3) : 0.f;
                    }
                }
            };
            const bool pre_mul = use_mul && staged;
            if (pre_mul && n0 + half * 32 < g.N) load_mul(mnext, n0 + half * 32);
#pragma unroll 1
            for (int cc = half; cc < BN / 32; cc += 2) {
                const int c0 = n0 + cc * 32;
                if (c0 >= g.N) break;                                 // warp-uniform (fix-up never reads these columns)
                if (pre_mul) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) mreg[i] = mnext[i];
                    if (cc + 2 < BN / 32 && c0 + 64 < g.N) load_mul(mnext, c0 + 64);
                }
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + cc * 32);
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32"
                             "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
                             " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                               "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                               "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                               "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                             : "r"(taddr) : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (!w.first) {
                    // running sum of the segment's earlier chunks (this thread's own stores), round-to-nearest adds
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 sacc = prow[(cc * 32 + j) >> 2];
                        r[j] = __float_as_uint(__uint_as_float(r[j]) + sacc.x);
                        r[j + 1] = __float_as_uint(__uint_as_float(r[j + 1]) + sacc.y);
                        r[j + 2] = __float_as_uint(__uint_as_float(r[j + 2]) + sacc.z);
                        r[j + 3] = __float_as_uint(__uint_as_float(r[j + 3]) + sacc.w);
                    }
                }
                if (partial || !fin) {
                    // raw partial tile, dense [128][BN] in the workspace: every lane writes 128 contiguous bytes
#pragma unroll
                    for (int j = 0; j < 32; j += 4)
                        prow[(cc * 32 + j) >> 2] = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                               __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                } else if (staged) {
                    // bias / ReLU in registers -> 128-byte-swizzled 32 x 32 tile in shared memory -> multiplier pass ->
                    // one bulk tensor store (full 128-byte lines; TMA clips rows >= M and columns >= N)
                    uint8_t *buf = stg + (chunk % EPI_BUFS) * 4096;
                    if (lane == 0) {
                        if (deep) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float4 v = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                               __uint_as_float(r[j + 3]));
                        if (has_bias) {
                            const float4 bb = *reinterpret_cast<const float4 *>(bias_t + cc * 32 + j);   // broadcast read
                            v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
                        }
                        if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                        *reinterpret_cast<float4 *>(buf + lane * 128 + (((j >> 2) ^ (lane & 7)) << 4)) = v;
                    }
                    if (use_mul) {
                        __syncwarp();
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int rr = 4 * i + (lane >> 3), ch = lane & 7;
                            float4 *cell = reinterpret_cast<float4 *>(buf + rr * 128 + ((ch ^ (rr & 7)) << 4));
                            float4 v = *cell;
                            v.x *= mreg[i].x; v.y *= mreg[i].y; v.z *= mreg[i].z; v.w *= mreg[i].w;
                            *cell = v;
                        }
                    }
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) tma_store_3d(&tmC, smem_u32(buf), c0, row0, w.b);
                    ++chunk;
                } else if (row < g.M) {
                    // C rows are not 16-byte aligned (e.g. 18 actions): per-row stores
                    const float *mul = use_mul ? g.mul + (size_t)(row % g.mul_rows) * g.ld_mul : nullptr;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const int col = c0 + j;
                        const float e[4] = {__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                            __uint_as_float(r[j + 3])};
                        float o[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            float x = e[i];
                            if (col + i < g.N) {
                                if (has_bias) x += bias_t[cc * 32 + j + i];
                                if (relu) x = fmaxf(x, 0.f);
                                if (mul) x *= __ldg(mul + col + i);
                            }
                            o[i] = x;
                        }
                        if (vec_ok && col + 3 < g.N) {
                            *reinterpret_cast<float4 *>(crow + col) = make_float4(o[0], o[1], o[2], o[3]);
                        } else {
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                if (col + i < g.N) crow[col + i] = o[i];
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_acc_empty[acc]);
        }
        if (staged && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// Stream-K fix-up: block (range boundary, strip of FIX_ROWS rows) sums the partial tiles of a cut tile in CTA order (a
// fixed order: results do not depend on scheduling), applies bias / ReLU / multiplier and writes C.
constexpr int FIX_ROWS = 4;

__global__ void __launch_bounds__(256) tc_streamk_fixup_kernel(TcParams g)
{
    const int kb_total = g.kblocks * g.kbatches;
    // many tiles, few cuts: one block column per CTA-range boundary -- the tile it falls into is cut (unless the boundary
    // sits on a tile edge); a tile holding several boundaries is summed at its first one.  Few tiles: one per tile.
    long long t = blockIdx.x;                                         // fix_by_boundary == 0: one block column per tile
    if (g.fix_by_boundary) {
        const long long wb = (long long)(blockIdx.x + 1) * g.per_cta;
        if (wb >= g.work || wb % kb_total == 0) return;
        t = wb / kb_total;
        if ((long long)blockIdx.x * g.per_cta > t * kb_total) return;
    }
    const long long w0 = t * kb_total, w1 = w0 + kb_total;
    const int c_first = (int)(w0 / g.per_cta), c_last = (int)((w1 - 1) / g.per_cta);
    if (c_first == c_last) return;                                    // whole tile: written by the GEMM epilogue
    int u = (int)t;
    const int tn = u % g.tiles_n; u /= g.tiles_n;
    const int tm = u % g.tiles_m, b = u / g.tiles_m;
    const int bn4 = g.bn >> 2;
    const float *bias = g.bias ? g.bias + (size_t)b * g.bias_bs : nullptr;
    const bool cvec = (g.ldc % 4 == 0) && (g.c_bs % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
    const int first_slot = SLOTS_PER_CTA * c_first + ((long long)c_first * g.per_cta < w0 ? 1 : 0);
    for (int i = threadIdx.x; i < FIX_ROWS * bn4; i += blockDim.x) {
        const int r = blockIdx.y * FIX_ROWS + i / bn4, c = (i % bn4) << 2;
        const int row = tm * BM + r, col = tn * g.bn + c;
        if (row >= g.M || col >= g.N) continue;
        const size_t off = (size_t)r * g.bn + c, slot_stride = (size_t)BM * g.bn;
        float4 a = *reinterpret_cast<const float4 *>(g.ws + first_slot * slot_stride + off);
#pragma unroll 4
        for (int cta = c_first + 1; cta <= c_last; ++cta) {          // every later CTA reaches this tile as its first segment
            const float4 v = *reinterpret_cast<const float4 *>(g.ws + (size_t)(SLOTS_PER_CTA * cta) * slot_stride + off);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        float o[4] = {a.x, a.y, a.z, a.w};
        float *dst = g.C + (size_t)b * g.c_bs + (size_t)row * g.ldc + col;
        const float *mm = g.mul ? g.mul + (size_t)(row % g.mul_rows) * g.ld_mul + col : nullptr;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (col + k < g.N) {
                float x = o[k];
                if (bias) x += bias[col + k];
                if (g.act == 1) x = fmaxf(x, 0.f);
                if (mm) x *= mm[k];
                o[k] = x;
            }
        }
        if (cvec && col + 3 < g.N) *reinterpret_cast<float4 *>(dst) = make_float4(o[0], o[1], o[2], o[3]);
        else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (col + k < g.N) dst[k] = o[k];
        }
    }
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// operand with logical shape rows x kdim (x nbatch).  major 0: stored row-major [rows][kdim] (ld floats);
// major 1: stored row-major [kdim][rows] (ld floats).  Box = 32 floats along the contiguous dimension.
int make_map(CUtensorMap *map, const float *ptr, int major, long long rows, long long kdim, long long ld, long long bs,
             long long nbatch, int tile_rows, int bk)
{
    EncodeTiledFn enc = encode_fn();
    if (!enc) return PB_E_UNSUPPORTED;
    if ((ld % 4) != 0 || (bs % 4) != 0 || (reinterpret_cast<uintptr_t>(ptr) & 15)) return PB_E_ARG;
    cuuint64_t dims[3], strides[2];
    cuuint32_t box[3], estr[3] = {1, 1, 1};
    const long long outer_rows = major ? kdim : rows;
    dims[0] = (cuuint64_t)(major ? rows : kdim);
    dims[1] = (cuuint64_t)outer_rows;
    dims[2] = (cuuint64_t)(nbatch > 0 ? nbatch : 1);
    strides[0] = (cuuint64_t)ld * 4;
    strides[1] = (cuuint64_t)((nbatch > 1 && bs > 0) ? bs : outer_rows * ld) * 4;
    box[0] = (cuuint32_t)(major ? 32 : bk);
    box[1] = (cuuint32_t)(major ? bk : tile_rows);
    box[2] = 1;
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE,
                     major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : (bk == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B),
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? PB_OK : PB_E_ARG;
}

// output tile map: row-major [rows][cols] (row stride ld floats) x nbatch, 32 x 32 boxes, 128-byte swizzle
int make_out_map(CUtensorMap *map, float *ptr, long long rows, long long cols, long long ld, long long bs, long long nbatch)
{
    EncodeTiledFn enc = encode_fn();
    if (!enc) return PB_E_UNSUPPORTED;
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(nbatch > 0 ? nbatch : 1)};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)((nbatch > 1 && bs > 0) ? bs : rows * ld) * 4};
    cuuint32_t box[3] = {32, 32, 1}, estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? PB_OK : PB_E_ARG;
}

template <int BN, int BK, int A_MN, int B_MN>
int launch_cfg(const CUtensorMap &ta, const CUtensorMap &tb, const CUtensorMap &tc, const TcParams &g, int grid, void *stream)
{
    static PbPerDeviceOnce attr_set;
    const int smem = SMEM_BUDGET / (2 * (BM + BN) * BK * 4) * (2 * (BM + BN) * BK * 4) + 32768 + 1024;
    if (!attr_set.done()) {
        cudaError_t e = cudaFuncSetAttribute(tc_gemm_kernel<BN, BK, A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr_set.mark();
    }
    PB_LAUNCH((tc_gemm_kernel<BN, BK, A_MN, B_MN>), grid, NUM_THREADS, smem, stream, ta, tb, tc, g);
    return PB_OK;
}

template <int BN, int BK>
int launch_bn(int a_mn, int b_mn, const CUtensorMap &ta, const CUtensorMap &tb, const CUtensorMap &tc, const TcParams &g,
              int grid, void *stream)
{
    if (!a_mn && !b_mn) return launch_cfg<BN, BK, 0, 0>(ta, tb, tc, g, grid, stream);
    if (!a_mn && b_mn) return launch_cfg<BN, BK, 0, 1>(ta, tb, tc, g, grid, stream);
    if (a_mn && b_mn) return launch_cfg<BN, BK, 1, 1>(ta, tb, tc, g, grid, stream);
    return launch_cfg<BN, BK, 1, 0>(ta, tb, tc, g, grid, stream);
}

// K block per tile width
int pick_bk(int bn, int K)
{
    return (bn == 256 && K >= 256) ? 16 : 32;    // 4 x 48 KB stages instead of 2 x 96 KB once the K loop is long
}

constexpr int TC_CHAIN_FLOATS = 2048;

// modelled cost (SM clocks) of one K block and one epilogue at tile width bn: the MMA time and the shared-memory
// traffic (12 operand reads + the split pass) whichever is larger -- see DESIGN.md section 4
double kb_clocks(int bn)                       // per 32 floats of K
{
    const double mma = 12.0 * bn / 2.0;
    const double smem = (12.0 * (4096 + bn * 32) + 2.0 * (BM + bn) * 128) / 128.0;
    return mma > smem ? mma : smem;
}

}  // namespace

extern "C" {

int pb_tc_gemm_supported(int M, int N, int K, long long lda, long long ldb, long long ldc)
{
    return (M > 0 && N > 0 && K > 0 && (lda % 4) == 0 && (ldb % 4) == 0 && ldc >= N) ? 1 : 0;
}

// C[b] = act(sum over K (and over kbatches operand batches) A . B^T + bias[b]); see the header.
int pb_tc_gemm(int batch, int kbatches, int M, int N, int K,
               const float *A, int a_major, long long lda, long long a_bs,
               const float *B, int b_major, long long ldb, long long b_bs,
               const float *bias, long long bias_bs, int act,
               const float *mul, int mul_rows, long long ld_mul,
               float *C, long long ldc, long long c_bs,
               float *workspace, long long workspace_floats, int split_mode, void *stream)
{
    if (batch <= 0 || kbatches <= 0 || !A || !B || !C || (act != 0 && act != 1)) return PB_E_ARG;
    if (mul && (mul_rows <= 0 || ld_mul < N)) return PB_E_ARG;
    if (kbatches > 1 && batch != 1) return PB_E_ARG;
    if (!pb_tc_gemm_supported(M, N, K, lda, ldb, ldc)) return PB_E_UNSUPPORTED;
    if (split_mode != 0 && split_mode != 1) return PB_E_ARG;
    const int sms = pb_sm_count();
    TcParams g = {};
    g.C = C; g.bias = bias; g.ws = workspace;
    g.c_bs = c_bs; g.bias_bs = bias_bs; g.ldc = (int)ldc;
    g.M = M; g.N = N;
    g.kbatches = kbatches;
    g.batch = batch;
    g.a_batched = a_bs != 0; g.b_batched = b_bs != 0;
    g.tiles_m = (M + BM - 1) / BM;
    g.act = act; g.split_mode = split_mode;
    g.mul = mul; g.mul_rows = mul ? mul_rows : 1; g.ld_mul = (int)ld_mul;
    const int kb32 = ((K + 31) / 32) * kbatches;                       // cost model works in 32-float K blocks

    // tile width and schedule: whole tiles per CTA (data-parallel waves) or equal K-block ranges per CTA
    // (stream-K: no wave quantisation, but cut tiles pay a partial-tile round trip and the fix-up launch)
    int best_bn = 64;
    bool best_sk = false;
    double best = 1e300;
    const int bns[3] = {256, 128, 64};
    for (int bi = 0; bi < 3; ++bi) {
        const int bn = bns[bi];
        if (bn > 64 && bn / 2 >= N) continue;                          // tile twice as wide as the matrix
        const long long tiles = (long long)batch * g.tiles_m * ((N + bn - 1) / bn);
        // epilogue ~18 clocks per column of the tile; it overlaps the next tile's K loop only when the two
        // accumulators fit in TMEM (bn <= 128)
        const double t_main = kb32 * kb_clocks(bn), t_drain = 18.0 * bn + 600.0;
        const double t_epi = bn > 128 ? t_drain : (t_drain > t_main ? t_drain - t_main : 0.0) + 500.0;
        const double dp = (double)((tiles + sms - 1) / sms) * (t_main + t_epi);
        if (dp < best) { best = dp; best_bn = bn; best_sk = false; }
        const double work = (double)tiles * kb32;
        const double ctas = work / 4 < sms ? (work + 3) / 4 : sms;
        const bool ws_ok = workspace && SLOTS_PER_CTA * (long long)ctas * BM * bn <= workspace_floats;
        const double sk = work / ctas * kb_clocks(bn) + (tiles / ctas + 1.0) * t_epi + 2.0 * bn * BM * 4 / 48.0 + 14000.0;
        if (ws_ok && sk < best) { best = sk; best_bn = bn; best_sk = true; }
    }
    g.bn = best_bn;
    const int bk = pick_bk(best_bn, K);
    g.kblocks = (K + bk - 1) / bk;
    const int kb_total = g.kblocks * kbatches;
    g.tiles_n = (N + best_bn - 1) / best_bn;
    const long long tiles = (long long)batch * g.tiles_m * g.tiles_n;
    g.work = tiles * kb_total;
    long long grid;
    g.deep_epi = kb_total * bk <= 256 ? 1 : 0;
    if (best_sk) {
        const int min_kb = 128 / bk;                                   // at least 128 floats of K per CTA
        grid = g.work / min_kb < sms ? (g.work + min_kb - 1) / min_kb : sms;
        g.per_cta = (g.work + grid - 1) / grid;
    } else {
        grid = tiles < sms ? tiles : sms;
        g.per_cta = ((tiles + grid - 1) / grid) * kb_total;
    }
    grid = (g.work + g.per_cta - 1) / g.per_cta;
    // accumulation chains of at most ~2048 floats of K once a tile's K loop is twice that (see SegIter): the K = 32768
    // weight gradients; the K = 3136 forward / input-gradient GEMMs keep one chain (their drift, ~3e-5 worst case,
    // is inside the 1e-4 parity bar, and chunking them costs 18 % of their time)
    if ((long long)kb_total * bk >= 2 * TC_CHAIN_FLOATS && workspace &&
        SLOTS_PER_CTA * grid * BM * best_bn <= workspace_floats)
        g.kc = TC_CHAIN_FLOATS / bk;

    CUtensorMap ta, tb;
    const long long nb = kbatches > 1 ? kbatches : batch;
    int rc = make_map(&ta, A, a_major, M, K, lda, a_bs, g.a_batched ? nb : 1, BM, bk);
    if (rc != PB_OK) return rc;
    rc = make_map(&tb, B, b_major, N, K, ldb, b_bs, g.b_batched ? nb : 1, best_bn, bk);
    if (rc != PB_OK) return rc;
    CUtensorMap tc = ta;                                               // placeholder when the direct-store epilogue runs
    if ((ldc % 4) == 0 && (c_bs % 4) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0) {
        rc = make_out_map(&tc, C, M, N, ldc, c_bs, batch);
        if (rc != PB_OK) return rc;
        g.tma_store = 1;
    }

    if (bk == 16) {                                                    // only at bn 256 (pick_bk)
        rc = launch_bn<256, 16>(a_major, b_major, ta, tb, tc, g, (int)grid, stream);
    } else {
        if (best_bn == 256) rc = launch_bn<256, 32>(a_major, b_major, ta, tb, tc, g, (int)grid, stream);
        else if (best_bn == 128) rc = launch_bn<128, 32>(a_major, b_major, ta, tb, tc, g, (int)grid, stream);
        else rc = launch_bn<64, 32>(a_major, b_major, ta, tb, tc, g, (int)grid, stream);
    }
    if (rc != PB_OK) return rc;
    if ((g.per_cta % kb_total) != 0 && grid > 1) {                     // some tile is cut
        g.fix_by_boundary = tiles > grid - 1 ? 1 : 0;
        dim3 fgrid((unsigned)(g.fix_by_boundary ? grid - 1 : tiles), BM / FIX_ROWS);
        PB_LAUNCH(tc_streamk_fixup_kernel, fgrid, 256, 0, stream, g);
    }
    return PB_OK;
}

// Forward dense layer on the tensor cores: Y[k] (M x N) = act(X[k] (M x J) W[k]^T (N x J) + b[k]).
int pb_linear_fwd_tc_supported(int M, int N, int J)
{
    return (M > 0 && N > 0 && J > 0 && (J % 4) == 0) ? 1 : 0;
}

int pb_linear_fwd_tc(int K, int M, int N, int J, const float *X, long long x_head_stride, const float *W,
                     const float *b, int act, float *Y, void *stream)
{
    return pb_tc_gemm(K, 1, M, N, J, X, 0, J, x_head_stride, W, 0, J, (long long)N * J, b, N, act, nullptr, 0, 0, Y, N,
                      (long long)M * N, nullptr, 0, 0, stream);
}

}  // extern "C"
