// common.cuh -- shared helpers for libprism_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "prism_b200.h"

extern std::atomic<long long> g_pb_launches;

#define PB_CHECK_ARG(cond) do { if (!(cond)) return PB_E_ARG; } while (0)

// Launch + count + surface launch errors as positive cudaError_t codes.
#define PB_LAUNCH(kernel, grid, block, smem, stream, ...)                                   \
    do {                                                                                    \
        kernel<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__);           \
        g_pb_launches.fetch_add(1, std::memory_order_relaxed);                              \
        cudaError_t pb_e_ = cudaGetLastError();                                             \
        if (pb_e_ != cudaSuccess) return (int)pb_e_;                                        \
    } while (0)

// Same, as a PROGRAMMATIC DEPENDENT LAUNCH: the kernel may be scheduled while its predecessor on the stream (or the
// graph branch it is captured on) is still running; it must call pb::pdl_wait() before touching anything the
// predecessor wrote.  Chains of short dependent kernels (the priority store's sample -> mark -> lines -> rebuild) save
// the launch latency at every boundary.  The kernels of the agent's update chain are launched the ordinary way
// (PB_LAUNCH): a dependent kernel that is resident early holds SM slots while it waits, and in the step graph those
// slots belong to the GEMMs of the parallel branches (measured: 86.8 vs 83.8 us per step with PDL on that chain).
#define PB_LAUNCH_PDL(kernel, grid, block, smem, stream, ...)                               \
    do {                                                                                    \
        cudaLaunchConfig_t pb_cfg_ = {};                                                    \
        pb_cfg_.gridDim = dim3(grid); pb_cfg_.blockDim = dim3(block);                       \
        pb_cfg_.dynamicSmemBytes = (smem); pb_cfg_.stream = (cudaStream_t)(stream);         \
        cudaLaunchAttribute pb_at_[1];                                                      \
        pb_at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                  \
        pb_at_[0].val.programmaticStreamSerializationAllowed = 1;                           \
        pb_cfg_.attrs = pb_at_; pb_cfg_.numAttrs = 1;                                       \
        cudaError_t pb_e_ = cudaLaunchKernelEx(&pb_cfg_, kernel, __VA_ARGS__);              \
        g_pb_launches.fetch_add(1, std::memory_order_relaxed);                              \
        if (pb_e_ != cudaSuccess) return (int)pb_e_;                                        \
    } while (0)

// argument check of the rule-parameterised optimizer entries: PB_E_ARG for an unknown rule or a NULL state array that
// the rule reads (m: Adam, centered RMSprop; v: every rule but SGD)
static inline bool pb_opt_known(int rule) { return rule >= PB_OPT_ADAM && rule <= PB_OPT_SGD; }
static inline int pb_opt_check(int rule, const void *m, const void *v)
{
    if (!pb_opt_known(rule)) return PB_E_ARG;
    const bool has_m = rule == PB_OPT_ADAM || rule == PB_OPT_RMSPROP_CENTERED, has_v = rule != PB_OPT_SGD;
    return ((has_m && !m) || (has_v && !v)) ? PB_E_ARG : PB_OK;
}

static inline int pb_ilog2(long long v) { int l = 0; while ((1LL << l) < v) ++l; return l; }
static inline bool pb_is_pow2(long long v) { return v > 0 && (v & (v - 1)) == 0; }

// SM count of the current device (148 on B200); cached per device.
int pb_sm_count();

// One-time per-device setup (cudaFuncSetAttribute is a per-device property): a bitmask over device ordinals.
struct PbPerDeviceOnce {
    std::atomic<unsigned long long> mask{0};
    static int device() { int d = 0; return cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < 64 ? d : 0; }
    bool done() const { return (mask.load(std::memory_order_acquire) >> device()) & 1ull; }
    void mark() { mask.fetch_or(1ull << device(), std::memory_order_release); }
};

namespace pb {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// programmatic dependent launch (PB_LAUNCH_PDL): wait until the preceding grid has completed and its writes are
// visible / allow the next grid to be scheduled.  Both are no-ops in a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// streaming 128-bit accesses that do not pollute L1
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream(uint4 *p, const uint4 &v)
{
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
    return v;
}

// ---------------------------------------------------------------------------------
// device-side uniforms of the replay samplers (per_tree.cu, uniform.cu): Philox4x32-10 keyed by the shard seed,
// counter = (sample number, call number).  Every rank of a sharded buffer draws the same u_k without communication;
// the call number lives in the state block (pad[2], seed pad[3]) and is advanced by the last CTA of the launch (ticket
// pad[1]), so a replayed CUDA graph gets fresh numbers every iteration with no extra launch.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ double philox_uniform(unsigned seed, unsigned call, unsigned long long k)
{
    unsigned c0 = (unsigned)k, c1 = (unsigned)(k >> 32), c2 = call, c3 = 0x50455221u;
    unsigned k0 = seed, k1 = 0x9E3779B9u ^ seed;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    // 53 random bits -> [0, 1)
    return ((double)(c0 >> 5) * 67108864.0 + (double)(c1 >> 6)) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ void rng_advance(pb_per_state *st)
{
    // call after a __syncthreads(): every thread of this CTA has read the call number
    if (threadIdx.x == 0) {
        __threadfence();
        const int ticket = atomicAdd(&st->pad[1], 1);
        if (ticket == (int)(gridDim.x * gridDim.y) - 1) {
            st->pad[2] += 1;
            st->pad[1] = 0;
        }
    }
}

// peer wait of the global samplers (pb_tree_sample_global_peer, pb_uniform_sample_global_peer): the shard states were
// PUT into this rank's slots by every rank (peer_state_put_kernel, csrc/peer.cu); every CTA waits on the local signal
// pad until all ranks' puts of the current exchange have landed (bounded: gives up after timeout_ns and raises bit 2 of
// *status), then reads the slot.
struct PeerWait {
    const unsigned long long *flags;      // local pad, channel 2: [src] = number of that rank's completed puts
    const unsigned long long *epoch;      // local count of this rank's own puts (the exchange to wait for)
    const unsigned char *slots;           // local state area: slot (2 + (epoch & 1)) holds the blocks of that exchange
    unsigned int *status;
    unsigned long long timeout_ns;
    int slot_bytes;                       // bytes per slot
};

// gathered shard states may sit in peer-mapped memory that other GPUs write: read them past this SM's L1
__device__ __forceinline__ float ld_state_f32(const float *p)
{
    float v;
    asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ long long ld_state_s64(const long long *p)
{
    long long v;
    asm volatile("ld.volatile.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// every thread of the CTA: wait for the puts of G ranks (pw.flags set), returns the slot holding their state blocks
__device__ __forceinline__ const pb_per_state *peer_wait_states(const PeerWait &pw, int G)
{
    const unsigned long long e = *pw.epoch;
    if (threadIdx.x < G) {
        const unsigned long long *f = pw.flags + threadIdx.x;
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        if (v < e) {
            const unsigned long long t0 = global_ns();
            unsigned spins = 0;
            for (;;) {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
                if (v >= e) break;
                if ((++spins & 1023u) == 0 && pw.timeout_ns && global_ns() - t0 > pw.timeout_ns) {
                    if (pw.status) atomicOr(pw.status, 1u << 2);
                    break;
                }
            }
        }
    }
    __syncthreads();
    return reinterpret_cast<const pb_per_state *>(pw.slots + (size_t)(2 + (e & 1)) * pw.slot_bytes);
}

// ---------------------------------------------------------------------------------
// Update rules of the flat optimizers (PB_OPT_*), one instantiation of every clip + update kernel family per rule
// (agent_kernels.cu, peer.cu).  State slots: m = Adam's exp_avg / centered RMSprop's grad_avg, v = Adam's exp_avg_sq /
// RMSprop's square_avg; plain RMSprop keeps v only, SGD neither (its state pointers may be null).  Adam's arithmetic is
// written out in each kernel; opt_update is every other rule, per element after clip_grad_norm_'s g *= coef, in the
// order of torch's foreach implementation (torch/optim/rmsprop.py _multi_tensor_rmsprop, torch/optim/sgd.py
// _multi_tensor_sgd).  Each foreach op is one rounding; inside one, ATen's functors compute a + s * op(b, c), which
// the compiler contracts to fma(s, op(b, c), a):
//   square_avg.mul_(alpha)                      v = v * alpha
//   square_avg.addcmul_(g, g, 1 - alpha)        v = fma(1 - alpha, g * g, v)
//   grad_avg.lerp_(g, w = 1 - alpha)            m = |w| < 0.5 ? fma(w, g - m, m) : fma(-(g - m), 1 - w, g)
//                                                   (ATen's two-branch lerp, ATen/native/Lerp.h)
//   avg = addcmul(square_avg, grad_avg, grad_avg, -1).sqrt_().add_(eps)     centered: sqrt(v - m * m) + eps
//   avg = square_avg.sqrt().add_(eps)                                       not centered: sqrt(v) + eps
//   param.addcdiv_(g, avg, -lr)                 p = fma(-lr, g / avg, p)
//   SGD: param.add_(g, alpha=-lr)               p = fma(-lr, g, p)
// ---------------------------------------------------------------------------------
template <int R> struct OptRule {
    static_assert(R == PB_OPT_ADAM || R == PB_OPT_RMSPROP || R == PB_OPT_RMSPROP_CENTERED || R == PB_OPT_SGD, "rule");
    static constexpr bool has_m = R == PB_OPT_ADAM || R == PB_OPT_RMSPROP_CENTERED;   // reads / writes the m slot
    static constexpr bool has_v = R != PB_OPT_SGD;                                     // reads / writes the v slot
};

template <int R>
__device__ __forceinline__ void opt_update(float &p, float g, float &m, float &v, float lr, float alpha, float eps)
{
    if constexpr (R == PB_OPT_SGD) {
        p = __fmaf_rn(-lr, g, p);
    } else {
        v = __fmaf_rn(1.0f - alpha, __fmul_rn(g, g), __fmul_rn(v, alpha));
        float avg;
        if constexpr (R == PB_OPT_RMSPROP_CENTERED) {
            const float w = 1.0f - alpha, d = __fsub_rn(g, m);
            m = fabsf(w) < 0.5f ? __fmaf_rn(w, d, m) : __fmaf_rn(-d, __fsub_rn(1.0f, w), g);
            avg = __fadd_rn(__fsqrt_rn(__fsub_rn(v, __fmul_rn(m, m))), eps);
        } else {
            avg = __fadd_rn(__fsqrt_rn(v), eps);
        }
        p = __fmaf_rn(-lr, __fdiv_rn(g, avg), p);
    }
}

// ---------------------------------------------------------------------------------
// Value squashing (PB_SQUASH_*, Config.loss_squish_fn_id): h maps returns into the space the networks predict in, h^-1
// maps predictions back.  S = PB_SQUASH_NONE is the identity and adds no instruction to a kernel templated on S.
//   PB_SQUASH_OBS_LOOK_FURTHER  h(x)    = sign(x) (sqrt(|x| + 1) - 1) + eps x                   (Pohlen et al. 2018)
//                               h^-1(x) = sign(x) ((t - 1)^2 + 2 (t - 1)),  t = (sqrt(1 + 4 eps (|x| + 1 + eps)) - 1) / (2 eps)
//   PB_SQUASH_SYMLOG            h(x)    = sign(x) log1p(|x|),  h^-1(x) = sign(x) expm1(|x|)
// The textbook forms cancel in fp32 (sqrt(a + 1) - 1 near a = 0, and the 1/(2 eps)-scaled difference of h^-1, up to
// 1.2e-5 max(1, |x|)); the forms below have no cancellation: sqrt(a + 1) - 1 = a / (sqrt(a + 1) + 1) and, with
// s = sqrt(1 + 4 eps (a + 1 + eps)), t - 1 = 2 a / (s + 1 + 2 eps).  Explicit _rn operations: no FMA contraction, so
// tests/squash_oracle.py restates the same roundings.  copysignf keeps the sign of +-0 and propagates NaN.
// ---------------------------------------------------------------------------------
template <int S>
__device__ __forceinline__ float squash(float x)
{
    static_assert(S == PB_SQUASH_NONE || S == PB_SQUASH_OBS_LOOK_FURTHER || S == PB_SQUASH_SYMLOG, "squash kind");
    if constexpr (S == PB_SQUASH_OBS_LOOK_FURTHER) {
        const float a = fabsf(x);
        const float r = __fdiv_rn(a, __fadd_rn(__fsqrt_rn(__fadd_rn(a, 1.0f)), 1.0f));
        return __fadd_rn(copysignf(r, x), __fmul_rn(PB_SQUASH_OLF_EPS, x));
    } else if constexpr (S == PB_SQUASH_SYMLOG) {
        return copysignf(log1pf(fabsf(x)), x);
    } else {
        return x;
    }
}

template <int S>
__device__ __forceinline__ float unsquash(float x)
{
    static_assert(S == PB_SQUASH_NONE || S == PB_SQUASH_OBS_LOOK_FURTHER || S == PB_SQUASH_SYMLOG, "squash kind");
    if constexpr (S == PB_SQUASH_OBS_LOOK_FURTHER) {
        constexpr float e = PB_SQUASH_OLF_EPS;
        const float a = fabsf(x);
        const float s = __fsqrt_rn(__fadd_rn(1.0f, __fmul_rn(4.0f * e, __fadd_rn(a, 1.0f + e))));
        const float tm1 = __fdiv_rn(__fmul_rn(2.0f, a), __fadd_rn(s, 1.0f + 2.0f * e));
        return copysignf(__fmul_rn(tm1, __fadd_rn(tm1, 2.0f)), x);
    } else if constexpr (S == PB_SQUASH_SYMLOG) {
        return copysignf(expm1f(fabsf(x)), x);
    } else {
        return x;
    }
}

}  // namespace pb
