// narrow.cu -- the small pieces around the tensor-core GEMMs of the IQN / ensemble heads that used to leave this
// library (sm_100a, HBM-bound streaming kernels):
//
//   pb_narrow_linear_fwd / _bwd   the A-wide output layer of the IQN head on (T*B) rows
//                                 (nn.Linear(width, n_actions), prism/agents/models/iqn_model.py:42-46): N = 3..18
//                                 outputs per row is no GEMM tile -- the layer is one pass over its input
//                                 (forward: read x once; backward: read x once, write dx once, dW / db from
//                                 per-CTA register partials combined in a fixed order)
//   pb_sum_heads                  out[i] = sum_k in[k][i]: the state embedding's gradient summed over the K ensemble
//                                 heads that share it (q_ensemble.py:44-48)
//   pb_iqn_draw_cos_basis         tau ~ U[0,1) drawn on the device (Philox4x32-10, counter = (row, call number)) and
//                                 its cos(pi i tau) basis in the same launch (iqn_model.py:64-66, 89-92): no
//                                 framework RNG kernel in the captured step
#include "common.cuh"
#include <math.h>

namespace {

using namespace pb;

// ---------------------------------------------------------------------------------
// values p[0..NP) per lane -> lane l returns the warp-wide sum of p[l % NP] (NP a power of two <= 32):
// butterfly transpose-reduce, NP - 1 + log2(32 / NP) shuffles instead of 5 * NP
// ---------------------------------------------------------------------------------
template <int NP>
__device__ __forceinline__ float warp_reduce_multi(float (&p)[NP])
{
    const int lane = lane_id();
#pragma unroll
    for (int s = NP / 2; s >= 1; s >>= 1) {
#pragma unroll
        for (int k = 0; k < s; ++k) {
            const bool up = (lane & s) != 0;
            const float keep = up ? p[k + s] : p[k];
            const float send = up ? p[k] : p[k + s];
            p[k] = keep + __shfl_xor_sync(FULL, send, s);
        }
    }
    float v = p[0];
#pragma unroll
    for (int s = NP; s < 32; s <<= 1) v += __shfl_xor_sync(FULL, v, s);
    return v;
}

// forward: one warp per row; W staged in shared memory as float4 [N][J/4]
template <int NP>
__global__ void __launch_bounds__(256) narrow_fwd_kernel(long long M, int N, int J4, const float4 *__restrict__ x,
                                                         long long x_hs4, const float4 *__restrict__ w,
                                                         const float *__restrict__ bias, float *__restrict__ y)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    extern __shared__ float4 ws[];
    // grid.y = heads: head k works on x + k * x_hs (x_hs = 0: the heads share x), W + k * N * J, bias + k * N, y + k * M * N
    x += (size_t)blockIdx.y * x_hs4;
    w += (size_t)blockIdx.y * N * J4;
    if (bias) bias += (size_t)blockIdx.y * N;
    y += (size_t)blockIdx.y * M * N;
    for (int e = threadIdx.x; e < N * J4; e += blockDim.x) ws[e] = w[e];
    __syncthreads();
    const int lane = lane_id();
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const float b = (bias && lane < N) ? bias[lane] : 0.0f;
    for (long long m = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; m < M; m += n_warps) {
        float p[NP];
#pragma unroll
        for (int n = 0; n < NP; ++n) p[n] = 0.0f;
        const float4 *xr = x + m * J4;
        for (int c = lane; c < J4; c += 32) {
            const uint4 u = ldg_stream(reinterpret_cast<const uint4 *>(xr + c));
            const float4 xv = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                if (n < N) {
                    const float4 wv = ws[n * J4 + c];
                    p[n] += (xv.x * wv.x + xv.y * wv.y) + (xv.z * wv.z + xv.w * wv.w);
                }
            }
        }
        const float v = warp_reduce_multi<NP>(p);
        if (lane < N) y[m * N + lane] = v + b;
    }
}

// backward: thread t owns input columns 2t, 2t+1 (blockDim = J/2); rows are staged rpc (<= 32) at a time -- 32 for the
// (T*B)-row IQN layers (few partials), 4 at learner-batch sizes (a 256-row layer on 8 CTAs of 32 serial rows each was
// 11 us of pure load latency on the step's critical path).
//   dx[m][j]  = sum_n dy[m][n] W[n][j]          (W column pair in registers)
//   dWp[cta][n][j] = sum_{m in cta} dy[m][n] x[m][j],  dbp[cta][n] = sum_{m in cta} dy[m][n]
template <int NP>
__global__ void __launch_bounds__(512) narrow_bwd_kernel(long long M, int N, int J, const float *__restrict__ x,
                                                         long long x_hs, const float *__restrict__ w,
                                                         const float *__restrict__ dy, float *__restrict__ dx,
                                                         float *__restrict__ dWp, float *__restrict__ dbp, int rpc)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ float sdy[32 * NP];
    // grid.y = heads (dx is per head: (K, M, J); the caller sums it over the heads when they share x)
    x += (size_t)blockIdx.y * x_hs;
    w += (size_t)blockIdx.y * N * J;
    dy += (size_t)blockIdx.y * M * N;
    if (dx) dx += (size_t)blockIdx.y * M * J;
    if (dWp) dWp += (size_t)blockIdx.y * gridDim.x * N * J;
    if (dbp) dbp += (size_t)blockIdx.y * gridDim.x * N;
    const int t = threadIdx.x, j = 2 * t;
    float2 wr[NP], acc[NP];
#pragma unroll
    for (int n = 0; n < NP; ++n) {
        wr[n] = (n < N) ? *reinterpret_cast<const float2 *>(w + (size_t)n * J + j) : make_float2(0.f, 0.f);
        acc[n] = make_float2(0.f, 0.f);
    }
    float db = 0.0f;
    const long long chunks = (M + rpc - 1) / rpc;
    for (long long ch = blockIdx.x; ch < chunks; ch += gridDim.x) {
        const long long m0 = ch * rpc;
        const int rows = (int)((M - m0) < rpc ? (M - m0) : rpc);
        __syncthreads();
        for (int e = t; e < rpc * NP; e += blockDim.x) {
            const int r = e / NP, n = e - r * NP;
            sdy[e] = (r < rows && n < N) ? dy[(m0 + r) * N + n] : 0.0f;
        }
        __syncthreads();
        if (t < NP) {
            for (int r = 0; r < rows; ++r) db += sdy[r * NP + t];
        }
        for (int r0 = 0; r0 < rows; r0 += 4) {                      // four rows' loads in flight
            float2 xv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                xv[u] = r0 + u < rows ? *reinterpret_cast<const float2 *>(x + (size_t)(m0 + r0 + u) * J + j) : make_float2(0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int r = r0 + u;
                if (r >= rows) break;
                float2 d = make_float2(0.f, 0.f);
#pragma unroll
                for (int n = 0; n < NP; ++n) {
                    const float g = sdy[r * NP + n];
                    d.x += g * wr[n].x; d.y += g * wr[n].y;
                    acc[n].x += g * xv[u].x; acc[n].y += g * xv[u].y;
                }
                if (dx) *reinterpret_cast<float2 *>(dx + (size_t)(m0 + r) * J + j) = d;
            }
        }
    }
    if (dWp) {
#pragma unroll
        for (int n = 0; n < NP; ++n)
            if (n < N) *reinterpret_cast<float2 *>(dWp + ((size_t)blockIdx.x * N + n) * J + j) = acc[n];
    }
    if (dbp && t < N) dbp[(size_t)blockIdx.x * N + t] = db;
}


// dW and db of the narrow backward in ONE launch (two dependent launches sat on the step's critical path):
// e < n_w: dW[e] = sum_b wpart[b][e];  else db[e - n_w] = sum_b bpart[b][e - n_w].  Eight lanes per element stride over
// the partials (64 of them at learner-batch sizes: a thread per element was 64 dependent-latency loads deep), combined
// by three shuffles in a fixed order.
__global__ void __launch_bounds__(256) narrow_reduce_kernel(int nblocks, long long n_w, int n_b,
                                                            const float *__restrict__ wpart,
                                                            const float *__restrict__ bpart, float *__restrict__ dW,
                                                            float *__restrict__ db)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    wpart += (size_t)blockIdx.y * nblocks * n_w;                  // grid.y = heads
    bpart += (size_t)blockIdx.y * nblocks * n_b;
    const long long e = (long long)blockIdx.x * 32 + (threadIdx.x >> 3);
    const int pl = threadIdx.x & 7;
    const bool live = e < n_w + n_b, is_w = e < n_w;
    const float *src = is_w ? wpart + e : bpart + (e - n_w);
    const long long stride = is_w ? n_w : n_b;
    float a0 = 0.0f, a1 = 0.0f;
    if (live) {
        int b = pl;
        for (; b + 8 < nblocks; b += 16) { a0 += src[(size_t)b * stride]; a1 += src[(size_t)(b + 8) * stride]; }
        if (b < nblocks) a0 += src[(size_t)b * stride];
    }
    float a = a0 + a1;
    a += __shfl_xor_sync(FULL, a, 1);
    a += __shfl_xor_sync(FULL, a, 2);
    a += __shfl_xor_sync(FULL, a, 4);
    if (live && pl == 0) {
        if (is_w) { if (dW) dW[(size_t)blockIdx.y * n_w + e] = a; }
        else if (db) db[(size_t)blockIdx.y * n_b + (e - n_w)] = a;
    }
}

__global__ void sum_heads_kernel(int K, long long n4, const float4 *__restrict__ in, float4 *__restrict__ out)
{
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n4; e += (long long)gridDim.x * blockDim.x) {
        float4 a = in[e];
        for (int k = 1; k < K; ++k) {
            const float4 b = in[(size_t)k * n4 + e];
            a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
        }
        out[e] = a;
    }
}

// ---------------------------------------------------------------------------------
// tau draw + cosine basis.  rng: device long long[4] = {seed, call number, ticket, unused}; the last CTA of the launch
// advances the call number, so a replayed CUDA graph draws fresh quantiles every iteration.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ unsigned philox_word(unsigned seed, unsigned call, unsigned long long k)
{
    unsigned c0 = (unsigned)k, c1 = (unsigned)(k >> 32), c2 = call, c3 = 0x49514E21u;
    unsigned k0 = seed, k1 = 0x9E3779B9u ^ seed;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

__global__ void __launch_bounds__(256) draw_cos_basis_kernel(long long n_rows, int n_basis, long long *rng,
                                                             float *__restrict__ tau_out, float *__restrict__ out)
{
    const unsigned seed = (unsigned)rng[0], call = (unsigned)rng[1];
    const long long total = n_rows * n_basis;
    const float pi = 3.14159265358979323846f;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / n_basis;
        const int i = (int)(e - r * n_basis);
        // 24 random bits -> [0, 1), the resolution of torch.rand on fp32
        const float tau = (float)(philox_word(seed, call, (unsigned long long)r) >> 8) * (1.0f / 16777216.0f);
        if (i == 0) tau_out[r] = tau;
        out[e] = cosf(__fmul_rn(__fmul_rn(tau, (float)(i + 1)), pi));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned long long ticket = atomicAdd(reinterpret_cast<unsigned long long *>(rng + 2), 1ull);
        if (ticket == (unsigned long long)gridDim.x - 1) { rng[1] += 1; rng[2] = 0; }
    }
}

int narrow_np(int N) { return N <= 4 ? 4 : (N <= 8 ? 8 : (N <= 16 ? 16 : 32)); }

}  // namespace

extern "C" {

int pb_narrow_linear_supported(long long M, int N, int J)
{
    if (M <= 0 || N <= 0 || N > 32 || J <= 0) return 0;
    if ((J % 64) != 0 || J > 1024) return 0;                       // backward: J / 2 threads per CTA, whole warps
    if ((size_t)N * J * sizeof(float) > 160 * 1024) return 0;      // forward: W staged in shared memory
    return 1;
}

static int narrow_rpc(long long M) { return M <= 2048 ? 4 : 32; }

int pb_narrow_linear_bwd_blocks(long long M)
{
    const int rpc = narrow_rpc(M);
    long long nb = (M + rpc - 1) / rpc;
    const long long cap = (long long)pb_sm_count() * 2;
    if (nb > cap) nb = cap;
    return (int)(nb < 1 ? 1 : nb);
}

// y (K, M, N) = x . W^T + bias per head: x (K, M, J) with head stride x_head_stride floats (0: one (M, J) input shared by
// the heads), W (K, N, J), bias (K, N) or NULL
int pb_narrow_linear_fwd(int K, long long M, int N, int J, const float *x, long long x_head_stride, const float *w,
                         const float *bias, float *y, void *stream)
{
    if (K < 1 || K > 65535 || !pb_narrow_linear_supported(M, N, J) || !x || !w || !y || x_head_stride < 0 || (x_head_stride & 3))
        return PB_E_ARG;
    if ((((uintptr_t)x) | ((uintptr_t)w)) & 15) return PB_E_ARG;
    const size_t smem = (size_t)N * J * sizeof(float);
    long long nb = (M + 7) / 8;
    long long cap = ((long long)pb_sm_count() * 4 + K - 1) / K;
    if (cap < 1) cap = 1;
    if (nb > cap) nb = cap;
    const dim3 grid((unsigned)nb, (unsigned)K);
    const float4 *x4 = reinterpret_cast<const float4 *>(x), *w4 = reinterpret_cast<const float4 *>(w);
#define PB_NARROW_FWD(NP)                                                                                          \
    do {                                                                                                           \
        static PbPerDeviceOnce once;                                                                               \
        if (!once.done()) {                                                                                        \
            cudaError_t e = cudaFuncSetAttribute(narrow_fwd_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                 160 * 1024);                                                      \
            if (e != cudaSuccess) return (int)e;                                                                   \
            once.mark();                                                                                           \
        }                                                                                                          \
        PB_LAUNCH(narrow_fwd_kernel<NP>, grid, 256, smem, stream, M, N, J / 4, x4, x_head_stride / 4, w4, bias, y); \
    } while (0)
    switch (narrow_np(N)) {
        case 4: PB_NARROW_FWD(4); break;
        case 8: PB_NARROW_FWD(8); break;
        case 16: PB_NARROW_FWD(16); break;
        default: PB_NARROW_FWD(32); break;
    }
#undef PB_NARROW_FWD
    return PB_OK;
}

// per head: dx (K, M, J; optional) = dy . W ; dW (K, N, J; optional) = dy^T . x ; db (K, N; optional) = column sums of dy.
// partials: K * pb_narrow_linear_bwd_blocks(M) * (N * J + N) floats of scratch.  With partials given but dW = db = NULL
// only the per-CTA partial sums are written: pb_narrow_linear_bwd_reduce (below) finishes them, on any stream ordered
// after this call -- LearnerStep puts it on the weight-gradient branch of its graph.
int pb_narrow_linear_bwd(int K, long long M, int N, int J, const float *x, long long x_head_stride, const float *w,
                         const float *dy, float *dx, float *dW, float *db, float *partials, void *stream)
{
    if (K < 1 || K > 65535 || !pb_narrow_linear_supported(M, N, J) || !x || !w || !dy || x_head_stride < 0) return PB_E_ARG;
    if ((dW || db) && !partials) return PB_E_ARG;
    if ((((uintptr_t)x) | ((uintptr_t)w) | ((uintptr_t)dx) | ((uintptr_t)partials)) & 7) return PB_E_ARG;
    const int nb = pb_narrow_linear_bwd_blocks(M);
    const int rpc = narrow_rpc(M);
    float *dWp = partials;
    float *dbp = partials ? partials + (size_t)K * nb * N * J : nullptr;
    const dim3 grid((unsigned)nb, (unsigned)K);
    switch (narrow_np(N)) {
        case 4: PB_LAUNCH(narrow_bwd_kernel<4>, grid, J / 2, 0, stream, M, N, J, x, x_head_stride, w, dy, dx, dWp, dbp, rpc); break;
        case 8: PB_LAUNCH(narrow_bwd_kernel<8>, grid, J / 2, 0, stream, M, N, J, x, x_head_stride, w, dy, dx, dWp, dbp, rpc); break;
        case 16: PB_LAUNCH(narrow_bwd_kernel<16>, grid, J / 2, 0, stream, M, N, J, x, x_head_stride, w, dy, dx, dWp, dbp, rpc); break;
        default: PB_LAUNCH(narrow_bwd_kernel<32>, grid, J / 2, 0, stream, M, N, J, x, x_head_stride, w, dy, dx, dWp, dbp, rpc); break;
    }
    if (dW || db) {
        const long long n = (long long)N * J;
        PB_LAUNCH(narrow_reduce_kernel, dim3((unsigned)((n + N + 31) / 32), (unsigned)K), 256, 0, stream, nb, n, N, dWp, dbp,
                  dW, db);
    }
    return PB_OK;
}

// the second half of pb_narrow_linear_bwd: dW (K, N, J; optional) and db (K, N; optional) from the partial sums
int pb_narrow_linear_bwd_reduce(int K, long long M, int N, int J, const float *partials, float *dW, float *db, void *stream)
{
    if (K < 1 || K > 65535 || !pb_narrow_linear_supported(M, N, J) || !partials) return PB_E_ARG;
    if (!dW && !db) return PB_OK;
    const int nb = pb_narrow_linear_bwd_blocks(M);
    const long long n = (long long)N * J;
    PB_LAUNCH(narrow_reduce_kernel, dim3((unsigned)((n + N + 31) / 32), (unsigned)K), 256, 0, stream, nb, n, N, partials,
              partials + (size_t)K * nb * N * J, dW, db);
    return PB_OK;
}

int pb_sum_heads(int K, long long n, const float *in, float *out, void *stream)
{
    if (K <= 0 || n <= 0 || (n % 4) != 0 || !in || !out) return PB_E_ARG;
    if ((((uintptr_t)in) | ((uintptr_t)out)) & 15) return PB_E_ARG;
    long long nb = (n / 4 + 255) / 256;
    const long long cap = (long long)pb_sm_count() * 8;
    if (nb > cap) nb = cap;
    PB_LAUNCH(sum_heads_kernel, (unsigned)nb, 256, 0, stream, K, n / 4, reinterpret_cast<const float4 *>(in),
              reinterpret_cast<float4 *>(out));
    return PB_OK;
}

int pb_iqn_draw_cos_basis(long long n_rows, int n_basis, long long *rng, float *tau_out, float *out, void *stream)
{
    if (n_rows < 0 || n_basis <= 0) return PB_E_ARG;
    if (n_rows == 0) return PB_OK;
    if (!rng || !tau_out || !out) return PB_E_ARG;
    const long long total = n_rows * n_basis;
    long long nb = (total + 255) / 256;
    const long long cap = (long long)pb_sm_count() * 16;
    if (nb > cap) nb = cap;
    PB_LAUNCH(draw_cos_basis_kernel, (unsigned)nb, 256, 0, stream, n_rows, n_basis, rng, tau_out, out);
    return PB_OK;
}

}  // extern "C"
