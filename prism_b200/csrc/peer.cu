// peer.cu -- data-parallel exchange steps over NVLink / NVSwitch PEER MEMORY (sm_100a), no NCCL on the path.
//
// SURVEY 8(e): the replay buffer shards by collector, so the learner needs exactly two exchanges per step:
//   1. the 64-byte shard state blocks {len, p_sum, p_min, ...} of every rank (global stratified sampling), and
//   2. the sum of the flat gradient arenas, followed by the SAME clip + Adam step on every rank
//      (prism/agents/agent.py:73-74 runs clip_grad_norm_ + Adam.step on one process).
// Both are latency-bound at these sizes (64 B; 9.5 MB for configs[1]), where a library collective costs tens of
// microseconds per call inside a CUDA graph.  Here every rank maps every other rank's buffers (CUDA IPC) and
//   * pb_peer_state_allgather: one 1-block kernel stores the local block into every peer and runs the flag
//     handshake (release/acquire at system scope);
//   * pb_peer_reduce_scatter: rank r PULLS slice r of every rank's gradient arena with 128-bit loads, adds in rank
//     order (one owner per slice: no two ranks ever disagree), keeps the reduced slice locally and publishes the
//     slice's sum of squares to every peer;
//   * pb_peer_adam: the fused clip + Adam sweep reads each slice of the reduced gradient straight from its owner
//     (the all-gather half of the all-reduce is fused into the optimizer kernel), derives the global norm from the
//     published partial sums in rank order (bit-identical on every rank) and updates the local parameter replica.
// pb_peer_barrier is a 1-block epoch barrier (flags in peer memory, monotonically increasing: graph-replay safe).
#include "common.cuh"

namespace {

using namespace pb;

__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// peer data is re-written every step by another GPU: never serve it from this SM's L1
__device__ __forceinline__ float4 ld_peer_f4(const float *p)
{
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_peer_f64(const double *p)
{
    double v;
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Poll a flag in (local) peer-mapped memory until it reaches e (acquire loads at system scope; relaxed polls + one
// fence.acq_rel.sys measured slower: 26 vs 17 us for the fused exchange at 2 GPUs).  Bounded by timeout_ns
// (0 = forever); false on a timeout.
__device__ __forceinline__ bool wait_flag_sys(const unsigned long long *p, unsigned long long e, unsigned long long timeout_ns)
{
    if (ld_acquire_sys(p) < e) {
        const unsigned long long t0 = global_timer_ns();
        unsigned spins = 0;
        while (ld_acquire_sys(p) < e) {
            if ((++spins & 1023u) == 0 && timeout_ns && global_timer_ns() - t0 > timeout_ns) return false;
        }
    }
    return true;
}

// phase marks for measurement runs (pb_peer_trace): slot <- the latest %globaltimer at which any CTA passed the mark
__device__ unsigned long long g_ptrace[16];
__device__ int g_ptrace_on;
__device__ __forceinline__ void ptrace(int on, int slot)
{
    if (on) atomicMax(&g_ptrace[slot], global_timer_ns());
}

// one warp: lane i signals rank i and waits for rank i.  Two independent CHANNELS (own flags, own epoch): calls on
// one channel must be issued in the same order by every rank, but they may interleave with the other channel.
// The wait is BOUNDED: a rank that does not show up within g.timeout_ns (dead process, missed launch) makes the
// waiting lanes give up, set bit (1 << channel) of the local status word and let the kernel finish -- results are
// garbage from then on, but no GPU hangs in a kernel that cannot be cancelled; the host checks the status word
// (PeerGroup.check) and raises.
__device__ __forceinline__ void epoch_handshake(const pb_peer_group &g, int ch)
{
    const int lane = threadIdx.x & 31;
    unsigned long long *epoch = g.epoch + ch;
    const unsigned long long e = *epoch + 1;
    __threadfence_system();
    if (lane < g.world) {
        st_release_sys(g.flags[lane] + ch * PB_PEER_MAX + g.rank, e);
        const unsigned long long *mine = g.flags[g.rank] + ch * PB_PEER_MAX + lane;
        if (!wait_flag_sys(mine, e, g.timeout_ns) && g.status) atomicOr(g.status, 1u << ch);
    }
    __syncwarp();
    if (lane == 0) *epoch = e;
}

// which half of the double-buffered gradient arena the exchange in flight uses: the parity of the number of
// COMPLETED state exchanges (channel 1).  Writers (pack) run before the exchange of their step, readers (pulls)
// after it, so a fast rank packing step t+1 never touches the half a slow rank still pulls for step t, and it
// cannot reach step t+2 before that rank has signalled exchange t+1, i.e. finished pulling t.
__device__ __forceinline__ long long grad_parity_offset(const pb_peer_group &g, bool after_exchange)
{
    const unsigned long long e = g.epoch[1];
    return (long long)((after_exchange ? e - 1 : e) & 1ull) * g.grad_stride;
}

__global__ void __launch_bounds__(32) peer_barrier_kernel(pb_peer_group g) { epoch_handshake(g, 0); }

// The gathered blocks land in one of two peer-visible slots (parity of the channel-1 epoch) and are copied to a
// local buffer after the handshake: a fast rank's NEXT all-gather then never writes where a slower rank still reads.
__global__ void __launch_bounds__(64) peer_state_allgather_kernel(pb_peer_group g, const unsigned int *__restrict__ state,
                                                                  unsigned int *__restrict__ out_local)
{
    const int t = threadIdx.x;
    const unsigned long long slot = (g.epoch[1] + 1) & 1;
    const size_t slot_words = (size_t)slot * PB_PEER_MAX * 16;
    if (t < 16) {
        const unsigned int v = state[t];
        for (int p = 0; p < g.world; ++p) reinterpret_cast<unsigned int *>(g.state[p])[slot_words + g.rank * 16 + t] = v;
        __threadfence_system();
    }
    __syncthreads();
    if (t < 32) epoch_handshake(g, 1);
    __syncthreads();
    const volatile unsigned int *mine = reinterpret_cast<const volatile unsigned int *>(g.state[g.rank]) + slot_words;
    for (int i = t; i < g.world * 16; i += blockDim.x) out_local[i] = mine[i];
}

constexpr int RS_THREADS = 256;

__global__ void __launch_bounds__(RS_THREADS) peer_reduce_scatter_kernel(pb_peer_group g, long long n, long long slice,
                                                                         float *__restrict__ partials,
                                                                         unsigned int *__restrict__ ticket,
                                                                         long long *__restrict__ step_count)
{
    __shared__ double part[RS_THREADS / 32];
    __shared__ bool last;
    const long long lo = (long long)g.rank * slice, hi = min(n, lo + slice);
    const long long n4 = hi > lo ? (hi - lo) >> 2 : 0;                  // slices are multiples of 4 floats; n % 4 == 0
    float *out = g.reduced[g.rank];
    const long long po = grad_parity_offset(g, true);
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const long long e = lo + (i << 2);
        float4 s = ld_peer_f4(g.grad[0] + po + e);
        for (int p = 1; p < g.world; ++p) {
            const float4 v = ld_peer_f4(g.grad[p] + po + e);
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        *reinterpret_cast<float4 *>(out + e) = s;
        acc += (double)(s.x * s.x + s.y * s.y) + (double)(s.z * s.z + s.w * s.w);
    }
    acc = warp_sum(acc);
    if (lane_id() == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < RS_THREADS / 32; ++k) t += part[k];
        reinterpret_cast<double *>(partials)[blockIdx.x] = t;
        __threadfence();
        last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        __threadfence();
        double t = 0.0;
        for (unsigned k = 0; k < gridDim.x; ++k) t += reinterpret_cast<volatile double *>(partials)[k];   // fixed order
        for (int p = 0; p < g.world; ++p) g.norm_parts[p][g.rank] = t;
        __threadfence_system();
        *ticket = 0;
        if (step_count) *step_count += 1;
    }
}

// One-shot variant for small arenas (latency-bound: n * world * 4 B of NVLink pulls cost less than a second
// cross-GPU barrier): every rank pulls ALL ranks' gradients, adds them in rank order into its local reduced buffer
// and leaves per-block sums of squares -- same grid and order on every rank, so the replicas agree bit for bit --
// for the ordinary single-GPU clip + Adam kernel that follows.
__global__ void __launch_bounds__(RS_THREADS) peer_pull_sum_kernel(pb_peer_group g, long long n, float *__restrict__ partials,
                                                                   long long *__restrict__ step_count)
{
    __shared__ double part[RS_THREADS / 32];
    const long long n4 = n >> 2;
    float *out = g.reduced[g.rank];
    const long long po = grad_parity_offset(g, true);
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const long long e = i << 2;
        float4 s = ld_peer_f4(g.grad[0] + po + e);
        for (int p = 1; p < g.world; ++p) {
            const float4 v = ld_peer_f4(g.grad[p] + po + e);
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        *reinterpret_cast<float4 *>(out + e) = s;
        acc += (double)(s.x * s.x + s.y * s.y) + (double)(s.z * s.z + s.w * s.w);
    }
    acc = warp_sum(acc);
    if (lane_id() == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < RS_THREADS / 32; ++k) t += part[k];
        partials[blockIdx.x] = (float)t;
        if (blockIdx.x == 0 && step_count) *step_count += 1;
    }
}

__global__ void __launch_bounds__(256) peer_adam_kernel(pb_peer_group g, long long n, long long slice,
                                                        float *__restrict__ param, float *__restrict__ exp_avg,
                                                        float *__restrict__ exp_avg_sq,
                                                        const long long *__restrict__ step_count, float lr, float beta1,
                                                        float beta2, float adam_eps, float max_grad_norm,
                                                        float *__restrict__ norm_out, float *__restrict__ grad_out)
{
    double sq = 0.0;
    for (int r = 0; r < g.world; ++r) sq += ld_peer_f64(g.norm_parts[g.rank] + r);          // rank order: identical everywhere
    const float total_norm = (float)sqrt(sq);
    float coef = max_grad_norm / (total_norm + 1e-6f);                                       // clip_grad_norm_
    coef = coef > 1.0f ? 1.0f : coef;
    if (!(max_grad_norm > 0.0f)) coef = 1.0f;
    if (blockIdx.x == 0 && threadIdx.x == 0 && norm_out) { norm_out[0] = total_norm; norm_out[1] = coef; }
    const double step = (double)(*step_count);
    const float bc1 = (float)(1.0 - pow((double)beta1, step));
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, step));
    const float step_size = lr / bc1;
    auto upd = [&](float &p, float gg, float &m, float &v) {                                 // same arithmetic as adam_clip_kernel
        gg *= coef;
        m = m + (gg - m) * (1.0f - beta1);
        v = v * beta2 + (1.0f - beta2) * gg * gg;
        const float denom = sqrtf(v) / bc2_sqrt + adam_eps;
        p = p - step_size * (m / denom);
    };
    const long long n4 = n >> 2;
    float4 *p4 = reinterpret_cast<float4 *>(param), *m4 = reinterpret_cast<float4 *>(exp_avg),
           *v4 = reinterpret_cast<float4 *>(exp_avg_sq);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const long long e = i << 2;
        const int owner = (int)(e / slice);
        const float4 gr = ld_peer_f4(g.reduced[owner] + e);                                   // all-gather fused into the sweep
        float4 p = p4[i], m = m4[i], v = v4[i];
        upd(p.x, gr.x, m.x, v.x); upd(p.y, gr.y, m.y, v.y); upd(p.z, gr.z, m.z, v.z); upd(p.w, gr.w, m.w, v.w);
        p4[i] = p; m4[i] = m; v4[i] = v;
        if (grad_out) *reinterpret_cast<float4 *>(grad_out + e) = gr;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Small arenas, ONE kernel for the whole data-parallel optimizer step (after pack): handshake -> pull + sum ->
// global norm -> clip + Adam.  Every CTA waits on the local signal pad itself (no separate barrier launch), pulls its
// elements of every rank's gradient with 128-bit loads and adds them in rank order INTO REGISTERS, publishes its
// sum of squares, meets the other CTAs of this grid at a counter (all CTAs are co-resident: grid <= 4 per SM), and
// applies clip + Adam to the elements it still holds -- the summed gradient is never re-read.  Same grid and the
// same order of additions on every rank: the replicas stay bit-identical.
// Channel 1 carries the handshake (its completed count is the parity of the double-buffered gradient arena).
// ---------------------------------------------------------------------------------------------------------------
constexpr int FA_THREADS = 256;
constexpr int FA_U = 8;                                               // 128-bit elements per thread held in registers
constexpr int FA_MAX_PEERS = PB_PEER_MAX - 1;                         // other ranks a thread pulls from

__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(FA_THREADS) peer_allreduce_adam_kernel(pb_peer_group g, long long n,
                                                                         float *__restrict__ param,
                                                                         float *__restrict__ exp_avg,
                                                                         float *__restrict__ exp_avg_sq,
                                                                         long long *__restrict__ step_count, float lr,
                                                                         float beta1, float beta2, float adam_eps,
                                                                         float max_grad_norm, float *__restrict__ partials,
                                                                         unsigned int *__restrict__ counters,
                                                                         float *__restrict__ norm_out)
{
    __shared__ double red[FA_THREADS / 32];
    __shared__ float s_coef;
    __shared__ unsigned s_last;
    const int lane = threadIdx.x & 31;
    const unsigned long long e = g.epoch[1] + 1;                      // this exchange (epoch[1] advances at the very end)
    const long long step_now = *step_count + 1;                       // likewise
    const int tr = __ldg(&g_ptrace_on);
    if (tr && blockIdx.x == 0 && threadIdx.x == 0) g_ptrace[0] = global_timer_ns();
    // ---- everything that does not depend on the other ranks is requested BEFORE the wait: the optimizer state of this
    // thread's first element (the only one for arenas up to one element per thread) and the bias corrections
    const long long n4 = n >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x, i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float4 *p4 = reinterpret_cast<float4 *>(param), *m4 = reinterpret_cast<float4 *>(exp_avg),
           *v4 = reinterpret_cast<float4 *>(exp_avg_sq), *r4 = reinterpret_cast<float4 *>(g.reduced[g.rank]);
    float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f), m0 = p0, v0 = p0;
    if (i0 < n4) { p0 = p4[i0]; m0 = m4[i0]; v0 = v4[i0]; }
    const double step = (double)step_now;
    const float bc1 = (float)(1.0 - pow((double)beta1, step));
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, step));
    const float step_size = lr / bc1;
    // (launched as a programmatic dependent of the pack kernel: everything above overlaps its tail)
    pdl_wait();
    // ---- handshake: CTA 0 tells every rank "my gradient is packed"; every CTA waits for all ranks on the local pad
    if (threadIdx.x < 32) {
        if (blockIdx.x == 0) {
            __threadfence_system();
            if (lane < g.world) st_release_sys(g.flags[lane] + 1 * PB_PEER_MAX + g.rank, e);
        }
        if (lane < g.world) {
            const unsigned long long *mine = g.flags[g.rank] + 1 * PB_PEER_MAX + lane;
            if (!wait_flag_sys(mine, e, g.timeout_ns) && g.status) atomicOr(g.status, 1u << 1);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) ptrace(tr, 1);                              // handshake done
    const long long po = (long long)((e - 1) & 1ull) * g.grad_stride;  // the half packed for this exchange
    float4 sum[FA_U];
    // ---- pull + sum every rank's whole arena in rank order, kept in registers
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < FA_U; ++k) {
        const long long i = i0 + k * stride;
        sum[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n4) {
            float4 s4 = ld_peer_f4(g.grad[0] + po + (i << 2));
            // fully unrolled, the kernel fits 80 registers: 3 resident CTAs per SM, which sizes the grid (fa_max_blocks)
#pragma unroll FA_MAX_PEERS
            for (int p = 1; p < g.world; ++p) {
                const float4 v = ld_peer_f4(g.grad[p] + po + (i << 2));
                s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
            }
            sum[k] = s4;
            acc += (double)(s4.x * s4.x + s4.y * s4.y) + (double)(s4.z * s4.z + s4.w * s4.w);
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        ptrace(tr, 2);                                                // pulled + summed
        double t = 0.0;
        for (int k = 0; k < FA_THREADS / 32; ++k) t += red[k];
        partials[blockIdx.x] = (float)t;
        __threadfence();
        atomicAdd(&counters[0], 1u);
        // ---- meet the other CTAs of this grid (all resident)
        while (ld_acquire_gpu_u32(&counters[0]) < gridDim.x) { }
    }
    __syncthreads();
    if (threadIdx.x == 0) ptrace(tr, 3);                              // met the other CTAs
    // ---- global norm: every CTA adds the partials in the same order
    double a2 = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) a2 += (double)__ldcg(partials + k);
    a2 = warp_sum(a2);
    __syncthreads();                                                  // red[] is reused
    if (lane == 0) red[threadIdx.x >> 5] = a2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < FA_THREADS / 32; ++k) t += red[k];
        const float total_norm = (float)sqrt(t);
        float coef = max_grad_norm / (total_norm + 1e-6f);            // clip_grad_norm_
        coef = coef > 1.0f ? 1.0f : coef;
        if (!(max_grad_norm > 0.0f)) coef = 1.0f;
        s_coef = coef;
        if (blockIdx.x == 0 && norm_out) { norm_out[0] = total_norm; norm_out[1] = coef; }
    }
    __syncthreads();
    const float coef = s_coef;
    auto upd = [&](float &p, float gg, float &m, float &v) {          // same arithmetic as adam_clip_kernel
        gg *= coef;
        m = m + (gg - m) * (1.0f - beta1);
        v = v * beta2 + (1.0f - beta2) * gg * gg;
        const float denom = sqrtf(v) / bc2_sqrt + adam_eps;
        p = p - step_size * (m / denom);
    };
#pragma unroll
    for (int k = 0; k < FA_U; ++k) {
        const long long i = i0 + k * stride;
        if (i < n4) {
            float4 p = p0, m = m0, v = v0;
            if (k > 0) { p = p4[i]; m = m4[i]; v = v4[i]; }
            const float4 gr = sum[k];
            upd(p.x, gr.x, m.x, v.x); upd(p.y, gr.y, m.y, v.y); upd(p.z, gr.z, m.z, v.z); upd(p.w, gr.w, m.w, v.w);
            p4[i] = p; m4[i] = m; v4[i] = v;
            r4[i] = gr;                                               // the summed gradient (diagnostics, tests)
        }
    }
    // ---- the last CTA out closes the exchange: counters back to zero, epoch and step count advanced
    __syncthreads();
    if (threadIdx.x == 0) ptrace(tr, 4);                              // Adam applied
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&counters[1], 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        counters[0] = 0u; counters[1] = 0u;
        g.epoch[1] = e;
        *step_count = step_now;
    }
}

// Non-blocking half of the shard-state exchange (channel 2): store this rank's 64-byte state block into every rank's
// slot (parity of the put count) and raise this rank's flag there.  Nobody waits here: the consumer -- the global
// sampling kernel (pb_tree_sample_global_peer) -- waits on its local pad, so the exchange hides behind whatever runs
// between the priority write-back and the next batch's sampling (the backward pass).
__global__ void __launch_bounds__(32) peer_state_put_kernel(pb_peer_group g, const unsigned int *__restrict__ state)
{
    const int lane = threadIdx.x;
    const unsigned long long e = g.epoch[2] + 1;
    const size_t slot_words = (size_t)(2 + (e & 1)) * PB_PEER_MAX * 16;
    if (lane < 16) {
        const unsigned int v = state[lane];
        for (int p = 0; p < g.world; ++p) reinterpret_cast<unsigned int *>(g.state[p])[slot_words + g.rank * 16 + lane] = v;
    }
    __threadfence_system();
    __syncwarp();
    if (lane < g.world) st_release_sys(g.flags[lane] + 2 * PB_PEER_MAX + g.rank, e);
    __syncwarp();
    if (lane == 0) g.epoch[2] = e;
}

int check_group(const pb_peer_group *g)
{
    if (!g || g->world < 1 || g->world > PB_PEER_MAX || g->rank < 0 || g->rank >= g->world || !g->epoch) return PB_E_ARG;
    for (int p = 0; p < g->world; ++p)
        if (!g->flags[p]) return PB_E_ARG;
    return PB_OK;
}

}  // namespace

extern "C" {

int pb_peer_alloc(long long bytes, void **ptr)
{
    if (bytes <= 0 || !ptr) return PB_E_ARG;
    cudaError_t e = cudaMalloc(ptr, (size_t)bytes);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemset(*ptr, 0, (size_t)bytes);
    if (e != cudaSuccess) return (int)e;
    e = cudaDeviceSynchronize();
    return e == cudaSuccess ? PB_OK : (int)e;
}

int pb_peer_free(void *ptr) { return ptr ? (int)cudaFree(ptr) : PB_OK; }

// Force the (lazily loaded) exchange kernels into the context.  Loading a kernel can synchronise the device; done
// up front it can never wait behind a barrier kernel that spins on a rank whose work is not launched yet.
int pb_peer_preload(void)
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, peer_barrier_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, peer_state_allgather_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, peer_reduce_scatter_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, peer_adam_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, peer_pull_sum_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, peer_allreduce_adam_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, peer_state_put_kernel);
    return e == cudaSuccess ? PB_OK : (int)e;
}

int pb_peer_export(const void *ptr, void *handle64)
{
    if (!ptr || !handle64) return PB_E_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    return (int)cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(handle64), const_cast<void *>(ptr));
}

int pb_peer_open(const void *handle64, void **ptr)
{
    if (!handle64 || !ptr) return PB_E_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    return (int)cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
}

int pb_peer_close(void *ptr) { return ptr ? (int)cudaIpcCloseMemHandle(ptr) : PB_OK; }

int pb_peer_barrier(const pb_peer_group *g, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    PB_LAUNCH(peer_barrier_kernel, 1, 32, 0, stream, *g);
    return PB_OK;
}

int pb_peer_state_allgather(const pb_peer_group *g, const void *state64, void *all_state_out, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    if (!state64 || !all_state_out) return PB_E_ARG;
    for (int p = 0; p < g->world; ++p)
        if (!g->state[p]) return PB_E_ARG;
    PB_LAUNCH(peer_state_allgather_kernel, 1, 64, 0, stream, *g, reinterpret_cast<const unsigned int *>(state64),
              reinterpret_cast<unsigned int *>(all_state_out));
    return PB_OK;
}

long long pb_peer_slice(long long n, int world)
{
    if (n <= 0 || world <= 0) return 0;
    const long long q = ((n + 3) / 4 + world - 1) / world;
    return q * 4;
}

int pb_peer_reduce_scatter(const pb_peer_group *g, long long n, float *partial_scratch, long long *step_count, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    if (n <= 0 || (n % 4) != 0 || !partial_scratch) return PB_E_ARG;
    for (int p = 0; p < g->world; ++p)
        if (!g->grad[p] || !g->reduced[p] || !g->norm_parts[p]) return PB_E_ARG;
    const long long slice = pb_peer_slice(n, g->world);
    long long nb = ((slice >> 2) + RS_THREADS - 1) / RS_THREADS;
    const long long cap = (long long)pb_sm_count() * 4;
    if (nb > cap) nb = cap;
    if (nb > 1024) nb = 1024;                                          // partial_scratch: 4096 floats = 2040 doubles + ticket
    if (nb < 1) nb = 1;
    unsigned int *ticket = reinterpret_cast<unsigned int *>(partial_scratch + 4092);
    PB_LAUNCH(peer_reduce_scatter_kernel, (unsigned)nb, RS_THREADS, 0, stream, *g, n, slice, partial_scratch, ticket, step_count);
    return PB_OK;
}

int pb_peer_pull_sum(const pb_peer_group *g, long long n, float *partial_scratch, long long *step_count,
                     int *n_partials_out_h, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    if (n <= 0 || (n % 4) != 0 || !partial_scratch) return PB_E_ARG;
    for (int p = 0; p < g->world; ++p)
        if (!g->grad[p]) return PB_E_ARG;
    if (!g->reduced[g->rank]) return PB_E_ARG;
    long long nb = ((n >> 2) + RS_THREADS - 1) / RS_THREADS;
    const long long cap = (long long)pb_sm_count() * 4;
    if (nb > cap) nb = cap;
    if (nb < 1) nb = 1;
    PB_LAUNCH(peer_pull_sum_kernel, (unsigned)nb, RS_THREADS, 0, stream, *g, n, partial_scratch, step_count);
    if (n_partials_out_h) *n_partials_out_h = (int)nb;
    return PB_OK;
}

// CTAs of the fused kernel that are resident at once (its grid never exceeds this: the CTAs meet at a counter)
static int fa_max_blocks()
{
    static std::atomic<int> cached[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    int c = cached[dev].load(std::memory_order_relaxed);
    if (c > 0) return c;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, peer_allreduce_adam_kernel, FA_THREADS, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    c = pb_sm_count() * per_sm;
    cached[dev].store(c, std::memory_order_relaxed);
    return c;
}

long long pb_peer_allreduce_adam_max_n(void) { return (long long)fa_max_blocks() * FA_THREADS * FA_U * 4; }

int pb_peer_allreduce_adam(const pb_peer_group *g, long long n, float *param, float *exp_avg, float *exp_avg_sq,
                           long long *step_count, float lr, float beta1, float beta2, float adam_eps, float max_grad_norm,
                           float *partial_scratch, float *norm_out, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    if (n <= 0 || (n % 4) != 0 || n > pb_peer_allreduce_adam_max_n()) return PB_E_ARG;
    if (!param || !exp_avg || !exp_avg_sq || !step_count || !partial_scratch) return PB_E_ARG;
    if ((((uintptr_t)param) | ((uintptr_t)exp_avg) | ((uintptr_t)exp_avg_sq)) & 15) return PB_E_ARG;
    for (int p = 0; p < g->world; ++p)
        if (!g->grad[p]) return PB_E_ARG;
    if (!g->reduced[g->rank]) return PB_E_ARG;
    // one 128-bit element per thread while that fits the resident grid, then up to FA_U
    long long nb = ((n >> 2) + FA_THREADS - 1) / FA_THREADS;
    const long long cap = fa_max_blocks();
    if (nb > cap) nb = cap;
    if (nb < 1) nb = 1;
    unsigned int *counters = reinterpret_cast<unsigned int *>(partial_scratch + 4092);    // zero between calls
    PB_LAUNCH_PDL(peer_allreduce_adam_kernel, (unsigned)nb, FA_THREADS, 0, stream, *g, n, param, exp_avg, exp_avg_sq, step_count,
              lr, beta1, beta2, adam_eps, max_grad_norm, partial_scratch, counters, norm_out);
    return PB_OK;
}

int pb_peer_trace(int enable, unsigned long long *out, int n_out)
{
    // synchronous (measurement runs only): copy out the marks of the fused exchange kernel, clear them, switch marking
    unsigned long long host[16];
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyFromSymbol(host, g_ptrace, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    if (out) for (int k = 0; k < n_out && k < 16; ++k) out[k] = host[k];
    for (int k = 0; k < 16; ++k) host[k] = 0;
    e = cudaMemcpyToSymbol(g_ptrace, host, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    const int on = enable ? 1 : 0;
    e = cudaMemcpyToSymbol(g_ptrace_on, &on, sizeof(on));
    return e == cudaSuccess ? PB_OK : (int)e;
}

int pb_peer_state_put(const pb_peer_group *g, const void *state64, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    if (!state64) return PB_E_ARG;
    for (int p = 0; p < g->world; ++p)
        if (!g->state[p]) return PB_E_ARG;
    PB_LAUNCH(peer_state_put_kernel, 1, 32, 0, stream, *g, reinterpret_cast<const unsigned int *>(state64));
    return PB_OK;
}

int pb_peer_adam(const pb_peer_group *g, long long n, float *param, float *exp_avg, float *exp_avg_sq,
                 const long long *step_count, float lr, float beta1, float beta2, float adam_eps, float max_grad_norm,
                 float *norm_out, float *grad_out, void *stream)
{
    int rc = check_group(g);
    if (rc) return rc;
    if (n <= 0 || (n % 4) != 0 || !param || !exp_avg || !exp_avg_sq || !step_count) return PB_E_ARG;
    if ((((uintptr_t)param) | ((uintptr_t)exp_avg) | ((uintptr_t)exp_avg_sq) | ((uintptr_t)grad_out)) & 15) return PB_E_ARG;
    const long long slice = pb_peer_slice(n, g->world);
    long long nb = ((n >> 2) + 255) / 256;
    const long long cap = (long long)pb_sm_count() * 4;
    if (nb > cap) nb = cap;
    PB_LAUNCH(peer_adam_kernel, (unsigned)nb, 256, 0, stream, *g, n, slice, param, exp_avg, exp_avg_sq, step_count, lr, beta1,
              beta2, adam_eps, max_grad_norm, norm_out, grad_out);
    return PB_OK;
}

}  // extern "C"
