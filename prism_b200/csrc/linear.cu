// linear.cu -- dense layers of the Q heads / IQN MLP as one fused launch each (sm_100a).
//
// The reference evaluates its heads with nn.Linear inside nn.Sequential
// (prism/agents/models/ffnn_model.py:61-76, q_ensemble.py:26-48, iqn_model.py:30-46): per layer a
// cuBLAS sgemm + bias add + activation, and autograd mirrors.  At learner batch sizes (64-512 rows)
// cuBLAS picks a 32x32 SIMT tile on <= 64 CTAs (29 us per layer on a B200, profiles/launches_r01_step.txt)
// and the element-wise glue costs as much again.  Here one kernel does
//     forward   Y = act(X W^T + b)                       (bias + ReLU fused)
//     backward  dX = (dY . relu') W,  dW = (dY . relu')^T X,  db = colsum(dY . relu')   (mask fused on load,
//               bias gradient fused into the dW launch)
// batched over the K ensemble heads, products as 3xTF32 on the tensor cores (fp32-grade: parity 1e-4 needs it),
// and fills the chip on small problems with split-K over a THREAD-BLOCK CLUSTER: the S CTAs of a
// cluster each reduce a slice of the inner dimension and combine their 64x64 partial tiles through
// distributed shared memory in a fixed order -- deterministic, no atomics, no workspace, one launch.
#include "common.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace {

using namespace pb;

constexpr int TM = 64, TN = 64, TK = 32, PAD = 8;   // 2 x (A,B) stages of 32 x 72 floats (18 KB each; a row stride of 72 words
                                                    // makes the tensor-core fragment loads conflict-free); C tile aliases them


// phase marks of one launch for measurement runs (pb_gemm_trace; profiles/kernel_chain.py): slot 0 <- the EARLIEST
// %globaltimer at which a CTA started, slots 1.. <- the LATEST at which any CTA passed the mark.  Off by default: one
// cached load per CTA.
__device__ unsigned long long g_gemm_trace[8];
__device__ int g_gemm_trace_on;
__device__ __forceinline__ void gemm_mark(int on, int slot)
{
    if (on && threadIdx.x == 0) {
        unsigned long long v;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
        if (slot == 0) atomicMin(&g_gemm_trace[0], v); else atomicMax(&g_gemm_trace[slot], v);
    }
}

struct GemmArgs {
    const float *A, *B, *bias, *mask;
    float *C, *colsum;
    long long a_bs, b_bs, c_bs, bias_bs, colsum_bs;     // batch (head) strides, elements
    long long a_ss, b_ss;                               // segment strides (inner dimension made of n_seg pieces)
    int lda, ldb, ldc;
    int M, N, K;                                        // C is M x N, inner dimension K per segment
    int n_seg, splits, act, m_tiles;
};

// r[q] = 0 where !(m[q] > 0): the ReLU mask of four consecutive elements.  The mask has the operand's layout but its own
// base address, so a float4 load is taken only when it is 16-byte aligned itself.
__device__ __forceinline__ void mask4(float (&r)[4], const float *m)
{
    if ((reinterpret_cast<uintptr_t>(m) & 15) == 0) {
        const float4 v = *reinterpret_cast<const float4 *>(m);
        r[0] = v.x > 0.f ? r[0] : 0.f; r[1] = v.y > 0.f ? r[1] : 0.f;
        r[2] = v.z > 0.f ? r[2] : 0.f; r[3] = v.w > 0.f ? r[3] : 0.f;
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) r[q] = m[q] > 0.f ? r[q] : 0.f;
    }
}

template <bool KMAJOR>
__device__ __forceinline__ void load_tile(float (&r)[4], const float *__restrict__ P, const float *__restrict__ mask,
                                          int ld, int row0, int k0, int rows, int kmax, int t, int half)
{
    // tile is [TK][64] in smem (k-major), fetched as two halves of 16 k.  KMAJOR: memory contiguous along k ->
    // thread owns 4 consecutive k of one row.  else: contiguous along the row index -> 4 consecutive rows of one k.
    int row, k;
    if (KMAJOR) { row = row0 + (t >> 2); k = k0 + half * 16 + ((t & 3) << 2); }
    else        { k = k0 + half * 16 + (t >> 4); row = row0 + ((t & 15) << 2); }
    const bool vec_ok = (ld & 3) == 0 && ((reinterpret_cast<uintptr_t>(P) & 15) == 0);
    if (KMAJOR) {
        const long long off = (long long)row * ld + k;
        if (vec_ok && row < rows && k + 3 < kmax && (k & 3) == 0) {
            float4 v = *reinterpret_cast<const float4 *>(P + off);
            r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
            if (mask) mask4(r, mask + off);
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float v = 0.f;
                if (row < rows && k + q < kmax) {
                    v = P[off + q];
                    if (mask && !(mask[off + q] > 0.f)) v = 0.f;
                }
                r[q] = v;
            }
        }
    } else {
        const long long off = (long long)k * ld + row;
        if (vec_ok && k < kmax && row + 3 < rows && (row & 3) == 0) {
            float4 v = *reinterpret_cast<const float4 *>(P + off);
            r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
            if (mask) mask4(r, mask + off);
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float v = 0.f;
                if (k < kmax && row + q < rows) {
                    v = P[off + q];
                    if (mask && !(mask[off + q] > 0.f)) v = 0.f;
                }
                r[q] = v;
            }
        }
    }
}

template <bool KMAJOR>
__device__ __forceinline__ void store_tile(float (*S)[TM + PAD], const float (&r)[4], int t, int half)
{
    if (KMAJOR) {
        const int row = t >> 2, k = half * 16 + ((t & 3) << 2);
#pragma unroll
        for (int q = 0; q < 4; ++q) S[k + q][row] = r[q];
    } else {
        const int k = half * 16 + (t >> 4), row = (t & 15) << 2;
        *reinterpret_cast<float4 *>(&S[k][row]) = make_float4(r[0], r[1], r[2], r[3]);
    }
}

// C[i][j] = epilogue( sum_seg sum_k A(i,k) B(k,j) )   grid: (n tiles, m tiles * batch, splits); cluster (1,1,splits)
// The products run on the tensor cores as 3xTF32 (mma.sync m16n8k8; every operand is split in registers into a TF32
// hi part and its fp32 residual lo, and each k step issues lo.hi + hi.lo + hi.hi into fp32 accumulators -- error ~1e-6,
// the same recipe as csrc/tc_gemm.cu).  These tiles are far too small and too many for the persistent tcgen05 kernel
// (one 128 x N tile per SM, 200 KB of shared memory: it serialised the step's graph branches).
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2])
{
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void split_tf32(float x, uint32_t &hi, uint32_t &lo)
{
    hi = __float_as_uint(x) & 0xFFFFE000u;                       // the 19 bits the tensor core reads
    lo = __float_as_uint(x - __uint_as_float(hi));                // exact; the tensor core reads ITS top 19 bits
}

// The split-K meeting point: CTA `rank` of the cluster owns TM / S rows of the tile and sums the S partial tiles in rank
// order.  Every remote (distributed shared memory) load of a thread is requested before the first add -- as a loop over
// the ranks with one scalar load each, the 2-4 rounds x S dependent round trips were a third of a 13 us launch.
template <int S, typename Emit4>
__device__ __forceinline__ void splitk_reduce(cg::cluster_group &cluster, float *cs, float *rsm, int rank, int t, int i0,
                                              int j0, Emit4 &emit4, float *colsum, int M)
{
    constexpr int rows_per = TM / S, units = rows_per * (TN / 4);      // float4 units of this rank's rows
    const float *remote[S];
#pragma unroll
    for (int s = 0; s < S; ++s) remote[s] = cluster.map_shared_rank(cs, s);
    for (int e = t; e < units; e += 256) {
        const int r = rank * rows_per + e / (TN / 4), c = (e % (TN / 4)) * 4;
        float4 v[S];
#pragma unroll
        for (int s = 0; s < S; ++s) v[s] = *reinterpret_cast<const float4 *>(remote[s] + r * (TN + PAD) + c);
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int s = 0; s < S; ++s) { a.x += v[s].x; a.y += v[s].y; a.z += v[s].z; a.w += v[s].w; }
        emit4(i0 + r, j0 + c, a);
    }
    if (colsum && t < rows_per) {
        const int r = rank * rows_per + t;
        float v[S];
#pragma unroll
        for (int s = 0; s < S; ++s) v[s] = cluster.map_shared_rank(rsm, s)[r];
        float a = 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) a += v[s];
        if (i0 + r < M) colsum[i0 + r] = a;
    }
}

// Everything after the K loop, shared by the two kernels below: fragments -> C tile -> 4 x 4 thread tiles; bias /
// activation / store when the tile is complete; otherwise the split-K meeting in distributed shared memory.
template <bool ROWSUM>
__device__ __forceinline__ void finish_tile(const GemmArgs &g, float (*Cs)[TN + PAD], float *Rs, float (&cf)[4][4], float rsum,
                                            int batch, int i0, int j0, bool want_rowsum, int tr_on)
{
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int lane = t & 31, gq = lane >> 2, tq = lane & 3;
    const int wm = ((t >> 5) & 3) * 16, wn = (t >> 7) * 32;
    // fragments -> the C tile (it aliases the stages: every warp is past its last read, see the barriers in the
    // callers) -> the 4 x 4 thread tiles the epilogue and the split-K reduction work with
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        *reinterpret_cast<float2 *>(&Cs[wm + gq][wn + nt * 8 + 2 * tq]) = make_float2(cf[nt][0], cf[nt][1]);
        *reinterpret_cast<float2 *>(&Cs[wm + gq + 8][wn + nt * 8 + 2 * tq]) = make_float2(cf[nt][2], cf[nt][3]);
    }
    if (ROWSUM && t < TM) Rs[t] = rsum;
    __syncthreads();
    float acc[4][4];
    float rs[4] = {};
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const float4 v = *reinterpret_cast<const float4 *>(&Cs[(ty << 2) + r][tx << 2]);
        acc[r][0] = v.x; acc[r][1] = v.y; acc[r][2] = v.z; acc[r][3] = v.w;
        if (ROWSUM) rs[r] = Rs[(ty << 2) + r];
    }
    __syncthreads();                                               // the split-K path rewrites the C tile below
    float *C = g.C + batch * g.c_bs;
    const float *bias = g.bias ? g.bias + batch * g.bias_bs : nullptr;
    auto emit = [&](int i, int j, float v) {
        if (i < g.M && j < g.N) {
            if (bias) v += bias[j];
            if (g.act == 1) v = fmaxf(v, 0.f);
            C[(long long)i * g.ldc + j] = v;
        }
    };
    if (g.splits == 1) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int i = i0 + (ty << 2) + r, j = j0 + (tx << 2);
            if (i < g.M && j + 3 < g.N && (g.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0) {
                float4 v = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
                if (bias) { v.x += bias[j]; v.y += bias[j + 1]; v.z += bias[j + 2]; v.w += bias[j + 3]; }
                if (g.act == 1) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                *reinterpret_cast<float4 *>(C + (long long)i * g.ldc + j) = v;
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c) emit(i, j + c, acc[r][c]);
            }
        }
        if (want_rowsum && tx == 0) {
            float *cs = g.colsum + batch * g.colsum_bs;
#pragma unroll
            for (int r = 0; r < 4; ++r) if (i0 + (ty << 2) + r < g.M) cs[i0 + (ty << 2) + r] = rs[r];
        }
        return;
    }

    // split-K: partial tiles meet in distributed shared memory, summed in rank order (deterministic)
    cg::cluster_group cluster = cg::this_cluster();
#pragma unroll
    for (int r = 0; r < 4; ++r)
        *reinterpret_cast<float4 *>(&Cs[(ty << 2) + r][tx << 2]) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
    if (tx == 0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) Rs[(ty << 2) + r] = rs[r];
    }
    gemm_mark(tr_on, 3);
    cluster.sync();
    gemm_mark(tr_on, 4);
    const bool c_vec = (g.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0;
    auto emit4 = [&](int i, int j, float4 v) {
        if (i < g.M && j + 3 < g.N && c_vec) {
            if (bias) { v.x += bias[j]; v.y += bias[j + 1]; v.z += bias[j + 2]; v.w += bias[j + 3]; }
            if (g.act == 1) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            *reinterpret_cast<float4 *>(C + (long long)i * g.ldc + j) = v;
        } else {
            emit(i, j, v.x); emit(i, j + 1, v.y); emit(i, j + 2, v.z); emit(i, j + 3, v.w);
        }
    };
    const int rank = (int)cluster.block_rank();
    switch (g.splits) {                                    // 2, 4 or 8 (pick_splits)
        case 2: splitk_reduce<2>(cluster, &Cs[0][0], Rs, rank, t, i0, j0, emit4, want_rowsum ? g.colsum + batch * g.colsum_bs : nullptr, g.M); break;
        case 4: splitk_reduce<4>(cluster, &Cs[0][0], Rs, rank, t, i0, j0, emit4, want_rowsum ? g.colsum + batch * g.colsum_bs : nullptr, g.M); break;
        default: splitk_reduce<8>(cluster, &Cs[0][0], Rs, rank, t, i0, j0, emit4, want_rowsum ? g.colsum + batch * g.colsum_bs : nullptr, g.M); break;
    }
    gemm_mark(tr_on, 5);
    cluster.sync();                                        // nobody exits while its tile is still being read
    gemm_mark(tr_on, 6);
}

// Operand tiles staged through registers in a two-stage pipeline, 4 CTAs per SM: the kernel for operands the cp.async
// kernel below cannot copy in 16-byte pieces.
template <bool A_KMAJOR, bool B_KMAJOR, bool ROWSUM>
__global__ void __launch_bounds__(256, 4) gemm_kernel(GemmArgs g)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const int tr_on = __ldg(&g_gemm_trace_on);
    gemm_mark(tr_on, 0);
    extern __shared__ __align__(16) float tiles[];
    __shared__ float Rs[TM];
    float (*As)[TK][TM + PAD] = reinterpret_cast<float (*)[TK][TM + PAD]>(tiles);
    float (*Bs)[TK][TN + PAD] = reinterpret_cast<float (*)[TK][TN + PAD]>(tiles + 2 * TK * (TM + PAD));
    float (*Cs)[TN + PAD] = reinterpret_cast<float (*)[TN + PAD]>(tiles);      // reused once the K loop is over

    const int t = threadIdx.x;
    const int batch = blockIdx.y / g.m_tiles, mt = blockIdx.y % g.m_tiles;
    const int i0 = mt * TM, j0 = blockIdx.x * TN;
    const int split = blockIdx.z;
    const float *A = g.A + batch * g.a_bs, *B = g.B + batch * g.b_bs;
    const float *mask = g.mask ? g.mask + batch * g.a_bs : nullptr;

    // iteration space: n_seg segments x ceil(K/TK) chunks, dealt to the splits in contiguous ranges
    const int chunks_per_seg = (g.K + TK - 1) / TK;
    const int total = g.n_seg * chunks_per_seg;
    const int per = (total + g.splits - 1) / g.splits;
    const int it0 = split * per, it1 = min(total, it0 + per);
    const bool want_rowsum = ROWSUM && g.colsum != nullptr && blockIdx.x == 0;

    auto fetch = [&](int it, float (&ra)[2][4], float (&rb)[2][4]) {
        const int seg = it / chunks_per_seg, k0 = (it % chunks_per_seg) * TK;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            load_tile<A_KMAJOR>(ra[h], A + seg * g.a_ss, mask ? mask + seg * g.a_ss : nullptr, g.lda, i0, k0, g.M, g.K, t, h);
            load_tile<B_KMAJOR>(rb[h], B + seg * g.b_ss, nullptr, g.ldb, j0, k0, g.N, g.K, t, h);
        }
    };
    auto stash = [&](int b, const float (&ra)[2][4], const float (&rb)[2][4]) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            store_tile<A_KMAJOR>(As[b], ra[h], t, h);
            store_tile<B_KMAJOR>(Bs[b], rb[h], t, h);
        }
    };
    // warp w owns rows wm .. wm+15, columns wn .. wn+31 of the tile (one m16 x four n8 fragments)
    const int lane = t & 31, gq = lane >> 2, tq = lane & 3;
    const int wm = ((t >> 5) & 3) * 16, wn = (t >> 7) * 32;
    float cf[4][4] = {};
    float rsum = 0.f;                                              // ROWSUM: thread t < 64 sums row t
    auto compute = [&](int b) {
        // a warp whose 16 rows lie past M has nothing to add (zero-filled rows): the padded static batch of the
        // data-parallel step (272 rows: a fifth tile with one live warp row) stays cheap
        if (i0 + wm < g.M) {
#pragma unroll
            for (int k0 = 0; k0 < TK; k0 += 8) {
                uint32_t ah[4], al[4];
                split_tf32(As[b][k0 + tq][wm + gq], ah[0], al[0]);
                split_tf32(As[b][k0 + tq][wm + gq + 8], ah[1], al[1]);
                split_tf32(As[b][k0 + tq + 4][wm + gq], ah[2], al[2]);
                split_tf32(As[b][k0 + tq + 4][wm + gq + 8], ah[3], al[3]);
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    uint32_t bh[2], bl[2];
                    split_tf32(Bs[b][k0 + tq][wn + nt * 8 + gq], bh[0], bl[0]);
                    split_tf32(Bs[b][k0 + tq + 4][wn + nt * 8 + gq], bh[1], bl[1]);
                    mma_tf32(cf[nt], al, bh);                      // small terms first
                    mma_tf32(cf[nt], ah, bl);
                    mma_tf32(cf[nt], ah, bh);
                }
            }
        }
        if (ROWSUM && t < TM) {
#pragma unroll
            for (int k = 0; k < TK; ++k) rsum += As[b][k][t];
        }
    };
    float ra[2][4], rb[2][4];
    int buf = 0;
    if (it0 < it1) {
        fetch(it0, ra, rb);
        stash(0, ra, rb);
    }
    __syncthreads();
    gemm_mark(tr_on, 1);
    for (int it = it0; it < it1; ++it) {
        const bool more = it + 1 < it1;
        if (more) fetch(it + 1, ra, rb);
        compute(buf);
        if (more) stash(buf ^ 1, ra, rb);
        __syncthreads();
        buf ^= 1;
    }

    gemm_mark(tr_on, 2);
    finish_tile<ROWSUM>(g, Cs, Rs, cf, rsum, batch, i0, j0, want_rowsum, tr_on);
}

// ---------------------------------------------------------------------------------------------------------------
// The same GEMM with the operand tiles brought in by cp.async (16-byte copies straight into shared memory, the whole
// pipeline of a split requested at kernel entry) -- used whenever the operands are 16-byte aligned, which every layer of
// the learner step is.  pb_gemm_trace on the register-staged kernel above: per 32-wide chunk 1.2 us went to staging
// (address arithmetic, LDG -> STS through registers, 4-way conflicted transposing stores) IN SERIES with 0.9 us of
// MMAs; here staging is 4 instructions per thread per chunk and overlaps the MMAs of earlier chunks.
// Tiles keep the layout of global memory: an operand contiguous along k sits row-major ([64][TK + 4] words), one
// contiguous along the row index k-major ([TK][64 + 8]) -- both strides make the m16n8k8 fragment loads conflict-free.
// The ReLU mask of the backward GEMMs gets its own tile and is applied when the A fragments are read.
constexpr int RS = TK + 4;                                  // row-major tile: words per row
constexpr int TILE_WORDS = TK * (TM + PAD);                 // = TM * RS = 2304 words either way
static_assert(TM * RS == TILE_WORDS && TN * RS == TILE_WORDS, "tile sizes");

__device__ __forceinline__ void cp_async16(float *dst, const float *src, bool valid)
{
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
    const int n = valid ? 16 : 0;                            // 0 source bytes: the 16 destination bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// one 64 x TK operand tile: 512 16-byte copies, two per thread
template <bool KMAJOR>
__device__ __forceinline__ void tile_async(float *dst, const float *__restrict__ P, int ld, int row0, int k0, int rows,
                                           int kmax, int t)
{
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int f = t + h * 256;
        if (KMAJOR) {
            const int row = f >> 3, kq = (f & 7) << 2;
            const bool ok = row0 + row < rows && k0 + kq < kmax;
            cp_async16(dst + row * RS + kq, ok ? P + (long long)(row0 + row) * ld + k0 + kq : P, ok);
        } else {
            const int k = f >> 4, rq = (f & 15) << 2;
            const bool ok = k0 + k < kmax && row0 + rq < rows;
            cp_async16(dst + k * (TM + PAD) + rq, ok ? P + (long long)(k0 + k) * ld + row0 + rq : P, ok);
        }
    }
}
template <bool KMAJOR>
__device__ __forceinline__ float tile_at(const float *tile, int row, int k)
{
    return KMAJOR ? tile[row * RS + k] : tile[k * (TM + PAD) + row];
}

template <bool A_KMAJOR, bool B_KMAJOR, bool ROWSUM, int STAGES>
__global__ void __launch_bounds__(256, STAGES == 2 ? 4 : 3) gemm_async_kernel(GemmArgs g)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const int tr_on = __ldg(&g_gemm_trace_on);
    gemm_mark(tr_on, 0);
    extern __shared__ __align__(16) float tiles[];
    __shared__ float Rs[TM];
    const bool masked = g.mask != nullptr;
    const int stage_words = (masked ? 3 : 2) * TILE_WORDS;        // A, B, (mask) tiles of one stage
    float (*Cs)[TN + PAD] = reinterpret_cast<float (*)[TN + PAD]>(tiles);      // reused once the K loop is over

    const int t = threadIdx.x;
    const int batch = blockIdx.y / g.m_tiles, mt = blockIdx.y % g.m_tiles;
    const int i0 = mt * TM, j0 = blockIdx.x * TN;
    const int split = blockIdx.z;
    const float *A = g.A + batch * g.a_bs, *B = g.B + batch * g.b_bs;
    const float *mask = masked ? g.mask + batch * g.a_bs : nullptr;
    const int chunks_per_seg = (g.K + TK - 1) / TK;
    const int total = g.n_seg * chunks_per_seg;
    const int per = (total + g.splits - 1) / g.splits;
    const int it0 = split * per, it1 = min(total, it0 + per);

    auto issue = [&](int it, int st) {
        if (it < it1) {
            const int seg = it / chunks_per_seg, k0 = (it % chunks_per_seg) * TK;
            float *base = tiles + st * stage_words;
            tile_async<A_KMAJOR>(base, A + seg * g.a_ss, g.lda, i0, k0, g.M, g.K, t);
            tile_async<B_KMAJOR>(base + TILE_WORDS, B + seg * g.b_ss, g.ldb, j0, k0, g.N, g.K, t);
            if (masked) tile_async<A_KMAJOR>(base + 2 * TILE_WORDS, mask + seg * g.a_ss, g.lda, i0, k0, g.M, g.K, t);
        }
        cp_async_commit();                                         // one group per chunk, empty ones included
    };
#pragma unroll
    for (int s = 0; s < STAGES; ++s) issue(it0 + s, s);

    const int lane = t & 31, gq = lane >> 2, tq = lane & 3;
    const int wm = ((t >> 5) & 3) * 16, wn = (t >> 7) * 32;
    float cf[4][4] = {};
    float rsum = 0.f;
    const bool want_rowsum = ROWSUM && g.colsum != nullptr && blockIdx.x == 0;
    const bool live = i0 + wm < g.M;                               // a warp whose 16 rows lie past M has nothing to add

    for (int it = it0, st = 0; it < it1; ++it) {
        cp_async_wait<STAGES - 1>();                               // all but the STAGES - 1 newest groups: chunk `it` landed
        __syncthreads();
        if (it == it0) gemm_mark(tr_on, 1);
        const float *sa = tiles + st * stage_words, *sb = sa + TILE_WORDS, *sm = sb + TILE_WORDS;
        if (live) {
#pragma unroll
            for (int k0 = 0; k0 < TK; k0 += 8) {
                float av[4] = {tile_at<A_KMAJOR>(sa, wm + gq, k0 + tq), tile_at<A_KMAJOR>(sa, wm + gq + 8, k0 + tq),
                               tile_at<A_KMAJOR>(sa, wm + gq, k0 + tq + 4), tile_at<A_KMAJOR>(sa, wm + gq + 8, k0 + tq + 4)};
                if (masked) {
                    av[0] = tile_at<A_KMAJOR>(sm, wm + gq, k0 + tq) > 0.f ? av[0] : 0.f;
                    av[1] = tile_at<A_KMAJOR>(sm, wm + gq + 8, k0 + tq) > 0.f ? av[1] : 0.f;
                    av[2] = tile_at<A_KMAJOR>(sm, wm + gq, k0 + tq + 4) > 0.f ? av[2] : 0.f;
                    av[3] = tile_at<A_KMAJOR>(sm, wm + gq + 8, k0 + tq + 4) > 0.f ? av[3] : 0.f;
                }
                uint32_t ah[4], al[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) split_tf32(av[q], ah[q], al[q]);
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    uint32_t bh[2], bl[2];
                    split_tf32(tile_at<B_KMAJOR>(sb, wn + nt * 8 + gq, k0 + tq), bh[0], bl[0]);
                    split_tf32(tile_at<B_KMAJOR>(sb, wn + nt * 8 + gq, k0 + tq + 4), bh[1], bl[1]);
                    mma_tf32(cf[nt], al, bh);                      // small terms first
                    mma_tf32(cf[nt], ah, bl);
                    mma_tf32(cf[nt], ah, bh);
                }
            }
        }
        if (ROWSUM && t < TM) {
#pragma unroll
            for (int k = 0; k < TK; ++k) {
                const float a = tile_at<A_KMAJOR>(sa, t, k);
                rsum += (!masked || tile_at<A_KMAJOR>(sm, t, k) > 0.f) ? a : 0.f;
            }
        }
        if (it + STAGES < it1) {
            __syncthreads();                                       // every warp is done with this stage
            issue(it + STAGES, st);
        } else {
            cp_async_commit();                                     // keeps the group count in step with `it`
        }
        st = st + 1 == STAGES ? 0 : st + 1;
    }
    cp_async_wait<0>();
    __syncthreads();                                               // the C tile aliases the stages
    gemm_mark(tr_on, 2);
    finish_tile<ROWSUM>(g, Cs, Rs, cf, rsum, batch, i0, j0, want_rowsum, tr_on);
}

int pick_splits(long long tiles, int total_chunks)
{
    const int sms = pb_sm_count();
    int s = 1;
    while (s < 8 && tiles * (s * 2) <= 2LL * sms && total_chunks / (s * 2) >= 2) s *= 2;
    return s;
}

// one launch of a GEMM kernel: grid (n tiles, m tiles * batch, splits), the splits of a tile forming one cluster
int launch_cluster(void (*kernel)(GemmArgs), const GemmArgs &g, int batch, int n_tiles, size_t smem, void *stream)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)n_tiles, (unsigned)(g.m_tiles * batch), (unsigned)g.splits);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = (unsigned)g.splits;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, g);
    g_pb_launches.fetch_add(1, std::memory_order_relaxed);
    if (e != cudaSuccess) return (int)e;
    e = cudaGetLastError();
    return e == cudaSuccess ? PB_OK : (int)e;
}

template <bool AK, bool BK, bool ROWSUM>
int launch_gemm_reg(GemmArgs g, int batch, int n_tiles, void *stream)
{
    constexpr int SMEM = 2 * 2 * TK * (TM + PAD) * 4;
    static PbPerDeviceOnce smem_set;                // one flag per template instantiation
    if (!smem_set.done()) {
        cudaError_t e = cudaFuncSetAttribute(gemm_kernel<AK, BK, ROWSUM>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) return (int)e;
        smem_set.mark();
    }
    return launch_cluster(gemm_kernel<AK, BK, ROWSUM>, g, batch, n_tiles, SMEM, stream);
}

template <bool AK, bool BK, bool ROWSUM, int STAGES>
int launch_gemm_async(GemmArgs g, int batch, int n_tiles, void *stream)
{
    static PbPerDeviceOnce smem_set;                // one flag per template instantiation
    if (!smem_set.done()) {
        cudaError_t e = cudaFuncSetAttribute(gemm_async_kernel<AK, BK, ROWSUM, STAGES>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, STAGES * 3 * TILE_WORDS * 4);
        if (e != cudaSuccess) return (int)e;
        smem_set.mark();
    }
    const size_t smem = (size_t)STAGES * (g.mask ? 3 : 2) * TILE_WORDS * 4;
    return launch_cluster(gemm_async_kernel<AK, BK, ROWSUM, STAGES>, g, batch, n_tiles, smem, stream);
}

bool async_eligible(const GemmArgs &g, bool ak, bool bk)
{
    const uintptr_t p = reinterpret_cast<uintptr_t>(g.A) | reinterpret_cast<uintptr_t>(g.B) | reinterpret_cast<uintptr_t>(g.mask);
    if (p & 15) return false;
    if ((g.lda | g.ldb) & 3) return false;
    if ((g.a_bs | g.b_bs | g.a_ss | g.b_ss) & 3) return false;
    if (((ak ? g.K : g.M) & 3) || ((bk ? g.K : g.N) & 3)) return false;      // a 16-byte copy is all inside or all outside
    return true;
}

template <bool AK, bool BK, bool ROWSUM>
int launch_gemm(GemmArgs g, int batch, void *stream)
{
    g.m_tiles = (g.M + TM - 1) / TM;
    const int n_tiles = (g.N + TN - 1) / TN;
    const int total_chunks = g.n_seg * ((g.K + TK - 1) / TK);
    g.splits = pick_splits((long long)g.m_tiles * n_tiles * batch, total_chunks);
    const int per = (total_chunks + g.splits - 1) / g.splits;      // chunks per split
    // 16-byte aligned operands (every layer of the learner step): the cp.async kernel
    if (async_eligible(g, AK, BK)) {
        if (per <= 2) return launch_gemm_async<AK, BK, ROWSUM, 2>(g, batch, n_tiles, stream);
        return launch_gemm_async<AK, BK, ROWSUM, 4>(g, batch, n_tiles, stream);
    }
    return launch_gemm_reg<AK, BK, ROWSUM>(g, batch, n_tiles, stream);
}

}  // namespace

extern "C" {

// Y[k] (M x N) = act(X[k] (M x J) W[k]^T (N x J) + b[k]);  x_head_stride 0 = one X shared by every head
int pb_linear_fwd(int K, int M, int N, int J, const float *X, long long x_head_stride, const float *W,
                  const float *b, int act, float *Y, void *stream)
{
    if (K <= 0 || M <= 0 || N <= 0 || J <= 0 || !X || !W || !Y || (act != 0 && act != 1)) return PB_E_ARG;
    GemmArgs g = {};
    g.A = X; g.a_bs = x_head_stride; g.lda = J;
    g.B = W; g.b_bs = (long long)N * J; g.ldb = J;
    g.C = Y; g.c_bs = (long long)M * N; g.ldc = N;
    g.bias = b; g.bias_bs = N; g.act = act;
    g.M = M; g.N = N; g.K = J; g.n_seg = 1;
    return launch_gemm<true, true, false>(g, K, stream);
}

// dX[k] (M x J) = (dY[k] . [Ymask[k] > 0]) (M x N) W[k] (N x J).
// sum_heads != 0: ONE dX (M x J) = sum over the K heads (X was shared): heads become segments of the inner dimension.
int pb_linear_bwd_input(int K, int M, int N, int J, const float *dY, const float *Ymask, const float *W,
                        int sum_heads, float *dX, void *stream)
{
    if (K <= 0 || M <= 0 || N <= 0 || J <= 0 || !dY || !W || !dX) return PB_E_ARG;
    GemmArgs g = {};
    g.A = dY; g.mask = Ymask; g.lda = N;
    g.B = W; g.ldb = J;
    g.C = dX; g.ldc = J;
    g.M = M; g.N = J; g.K = N;
    if (sum_heads) {
        g.n_seg = K; g.a_ss = (long long)M * N; g.b_ss = (long long)N * J;
        return launch_gemm<true, false, false>(g, 1, stream);
    }
    g.n_seg = 1; g.a_bs = (long long)M * N; g.b_bs = (long long)N * J; g.c_bs = (long long)M * J;
    return launch_gemm<true, false, false>(g, K, stream);
}

// dW[k] (N x J) = (dY[k] . mask)^T X[k];  db[k] (N) = column sums of (dY[k] . mask)   (db optional)
int pb_linear_bwd_weight(int K, int M, int N, int J, const float *dY, const float *Ymask, const float *X,
                         long long x_head_stride, float *dW, float *db, void *stream)
{
    if (K <= 0 || M <= 0 || N <= 0 || J <= 0 || !dY || !X || !dW) return PB_E_ARG;
    GemmArgs g = {};
    g.A = dY; g.mask = Ymask; g.lda = N; g.a_bs = (long long)M * N;      // A(i = n, k = m): contiguous along i
    g.B = X; g.ldb = J; g.b_bs = x_head_stride;                          // B(k = m, j): contiguous along j
    g.C = dW; g.ldc = J; g.c_bs = (long long)N * J;
    g.colsum = db; g.colsum_bs = N;
    g.M = N; g.N = J; g.K = M; g.n_seg = 1;
    return db ? launch_gemm<false, false, true>(g, K, stream) : launch_gemm<false, false, false>(g, K, stream);
}

// measurement runs only (synchronous): copy out the phase marks of the launches since the last call, reset them, switch
// marking on / off.  out[0] = earliest CTA start, out[1..6] = latest CTA past: first chunk staged, K loop, partial tile
// written, cluster barrier, split-K sum + epilogue, exit barrier.
int pb_gemm_trace(int enable, unsigned long long *out, int n_out)
{
    unsigned long long host[8];
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyFromSymbol(host, g_gemm_trace, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    if (out) for (int k = 0; k < n_out && k < 8; ++k) out[k] = host[k];
    for (int k = 0; k < 8; ++k) host[k] = 0;
    host[0] = ~0ULL;
    e = cudaMemcpyToSymbol(g_gemm_trace, host, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    const int on = enable ? 1 : 0;
    e = cudaMemcpyToSymbol(g_gemm_trace_on, &on, sizeof(on));
    return e == cudaSuccess ? PB_OK : (int)e;
}

}  // extern "C"
