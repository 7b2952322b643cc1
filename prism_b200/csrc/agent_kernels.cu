// agent_kernels.cu -- fused warp-level kernels of the learner update and of acting (sm_100a).
//
//   pb_iqn_cos_basis   IQNModel._embed_quantiles basis      prism/agents/models/iqn_model.py:89-92
//   pb_iqn_qh_loss     IQNModel.get_loss target+loss+grad   prism/agents/models/iqn_model.py:110-201
//   pb_ens_q_loss      QEnsemble.get_loss (MSE, double-Q)   prism/agents/models/q_ensemble.py:50-92
//   pb_ids_select      IDSActionSelector                    prism/agents/action_selectors.py:125-176
//   pb_greedy_select   GreedyActionSelector                 prism/agents/action_selectors.py:70-82
//   pb_value_squash    squish / unsquish functions          prism/agents/squish_functions.py (the *_sq entries: the
//                      loss and IDS kernels with value squashing as a template parameter, common.cuh)
//   pb_loss_combine    PER-weighted total + new priorities  prism/agents/agent.py:58-66, composite_model.py:135-142
//   pb_adam_clip_step  clip_grad_norm_ + Adam               prism/agents/agent.py:73-74, factory/agent_factory.py:44-47
//   pb_opt_*           clip_grad_norm_ + Adam / RMSprop / SGD  factory/agent_factory.py:40-58
//
// The reference runs each of these as 10-30 tiny ATen kernels (plus their autograd
// mirrors) with B*T'*T temporaries; here each is one launch, one warp per batch row,
// everything in registers/shared memory, forward and backward in the same pass.
#include "common.cuh"
#include <math.h>

namespace {

using namespace pb;

// ---------------------------------------------------------------------------------
__global__ void cos_basis_kernel(long long n_rows, int n_basis, const float *__restrict__ tau,
                                 float *__restrict__ out)
{
    const long long total = n_rows * n_basis;
    const float pi = 3.14159265358979323846f;  // np.pi rounded to fp32, as torch does for a python scalar
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / n_basis;
        const int i = (int)(e - r * n_basis);
        // (tile(tau) * arange(1..n)) * pi, each product rounded to fp32 (iqn_model.py:90-91)
        const float x = __fmul_rn(__fmul_rn(tau[r], (float)(i + 1)), pi);
        out[e] = cosf(x);
    }
}

// ---------------------------------------------------------------------------------
// quantile-Huber loss: one warp per batch row.  smem per warp: y[Tp], theta[T], tq[T].  S: value squashing of the
// target (PB_SQUASH_*, common.cuh).
// ---------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(128) qh_loss_kernel(int B, int T, int Tp, int A, const float *__restrict__ z_cur,
                                                      const float *__restrict__ tau,
                                                      const float *__restrict__ z_next_online,
                                                      const float *__restrict__ z_next_target,
                                                      const long long *__restrict__ action,
                                                      const float *__restrict__ ret, const float *__restrict__ gdn,
                                                      const uint8_t *__restrict__ nonterm, float kappa,
                                                      float loss_weight, const float *__restrict__ row_weight,
                                                      float grad_scale, float *__restrict__ loss_out,
                                                      float *__restrict__ grad_z)
{
    extern __shared__ float smem[];
    const int warp = threadIdx.x >> 5, lane = lane_id();
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b >= B) return;
    float *y = smem + (size_t)warp * (Tp + 2 * T);
    float *theta = y + Tp;
    float *tq = theta + T;

    // a* = argmax_a mean_j Z_online(s', tau'_j)[a]   (iqn_model.py:129-133), first index on ties
    int best_a = 0;
    float best_v = -INFINITY;
    for (int a = 0; a < A; ++a) {
        float acc = 0.0f;
        for (int j = lane; j < Tp; j += 32) acc += z_next_online[((size_t)j * B + b) * A + a];
        acc = warp_sum(acc) / (float)Tp;
        if (acc > best_v) { best_v = acc; best_a = a; }
    }
    // y_j = h(R + gamma^k * nonterminal * h^-1(Z_target(s', tau'_j)[a*]))   (:136-145)
    const float R = ret[b], g = nonterm ? __fmul_rn(gdn[b], nonterm[b] ? 1.0f : 0.0f) : gdn[b];
    for (int j = lane; j < Tp; j += 32)
        y[j] = squash<S>(__fadd_rn(R, __fmul_rn(unsquash<S>(z_next_target[((size_t)j * B + b) * A + best_a]), g)));
    const int act = (int)action[b];
    for (int i = lane; i < T; i += 32) {
        theta[i] = z_cur[((size_t)i * B + b) * A + act];
        tq[i] = tau[(size_t)i * B + b];
    }
    __syncwarp();

    const float w_row = (row_weight ? row_weight[b] : 1.0f) * grad_scale * loss_weight / (float)Tp;
    float loss_acc = 0.0f;
    for (int i = lane; i < T; i += 32) {
        const float th = theta[i], tqi = tq[i];
        float li = 0.0f, gi = 0.0f;
        for (int j = 0; j < Tp; ++j) {
            const float d = y[j] - th;                           // (:171)
            const float ad = fabsf(d);
            const bool quad = ad <= kappa;                       // (:174-178)
            const float hub = quad ? 0.5f * d * d : kappa * (ad - 0.5f * kappa);
            const float dh = quad ? d : (d > 0.0f ? kappa : -kappa);
            const float wq = fabsf(tqi - (d < 0.0f ? 1.0f : 0.0f));  // (:191-193)
            li += wq * hub;
            gi -= wq * dh;                                       // d/d theta = - d/d delta
        }
        loss_acc += li / kappa;
        gi = gi / kappa * w_row;
        float *grow = grad_z + ((size_t)i * B + b) * A;
        for (int a = 0; a < A; ++a) grow[a] = (a == act) ? gi : 0.0f;
    }
    loss_acc = warp_sum(loss_acc);
    if (lane == 0) loss_out[b] = loss_acc / (float)Tp * loss_weight;  // (:196-201)
}

// ---------------------------------------------------------------------------------
// ensemble MSE loss: one warp per batch row, lanes over heads.  tables are [K][B][A].
// ---------------------------------------------------------------------------------
// ticket != NULL: the LAST CTA to finish also does what loss_combine_kernel does (total = mean(dist * w) + mean(q' * w)
// with q' = q_scale * (loss - *q_offset), td_b = the TD mix) -- one launch less on the step's critical path.
// S: value squashing of the target (PB_SQUASH_*, common.cuh).
template <int S>
__global__ void __launch_bounds__(128) ens_loss_kernel(int B, int A, int K, const float *__restrict__ q_cur,
                                                       const float *__restrict__ q_next_online,
                                                       const float *__restrict__ q_next_target,
                                                       const long long *__restrict__ action,
                                                       const float *__restrict__ ret, const float *__restrict__ gdn,
                                                       const uint8_t *__restrict__ nonterm, float loss_weight,
                                                       const float *__restrict__ row_weight, float grad_scale,
                                                       float *__restrict__ loss_out, float *__restrict__ grad_q,
                                                       const float *__restrict__ dist, float q_scale,
                                                       const float *__restrict__ q_offset, float *__restrict__ total_out,
                                                       float *__restrict__ td_out, unsigned int *__restrict__ ticket)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const int warp = threadIdx.x >> 5, lane = lane_id();
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b < B) {
        const int act = (int)action[b];
        const float R = ret[b], g = nonterm ? __fmul_rn(gdn[b], nonterm[b] ? 1.0f : 0.0f) : gdn[b];
        const float gs = (row_weight ? row_weight[b] : 1.0f) * grad_scale * loss_weight * 2.0f / (float)K;
        float acc = 0.0f;
        for (int k = lane; k < K; k += 32) {
            const size_t row = ((size_t)k * B + b) * A;
            int best = 0;
            float bv = q_next_online[row];
            for (int a = 1; a < A; ++a) {
                float v = q_next_online[row + a];
                if (v > bv) { bv = v; best = a; }                    // argmax(dim=-2), first index (q_ensemble.py:70)
            }
            const float yk = squash<S>(__fadd_rn(R, __fmul_rn(unsquash<S>(q_next_target[row + best]), g)));  // (:80)
            const float diff = q_cur[row + act] - yk;
            acc += diff * diff;                                      // MSELoss(reduction='none') (:84)
            for (int a = 0; a < A; ++a) grad_q[row + a] = (a == act) ? gs * diff : 0.0f;
        }
        acc = warp_sum(acc);
        if (lane == 0) loss_out[b] = acc / (float)K * loss_weight;
    }
    if (!ticket) return;
    __shared__ unsigned s_last;
    __shared__ float part[4];
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
        if (s_last) { __threadfence(); *ticket = 0u; }
    }
    __syncthreads();
    if (!s_last) return;
    float acc = 0.0f;
    const float off = q_offset ? *q_offset : 0.0f;
    for (int r = threadIdx.x; r < B; r += blockDim.x) {
        const float wb = row_weight ? row_weight[r] : 1.0f;
        const float d = dist ? dist[r] : 0.0f, qq = q_scale * (__ldcg(loss_out + r) - off);
        acc += d * wb + qq * wb;
        if (td_out) td_out[r] = dist ? (d * 0.5f + qq * 0.5f) : fabsf(qq);
    }
    acc = warp_sum(acc);
    if (lane == 0) part[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0 && total_out) *total_out = (part[0] + part[1] + part[2] + part[3]) / (float)B;
}

// ---------------------------------------------------------------------------------
// IDS: one warp per state, lane = action (A <= 32).  S: every q and z value is read through h^-1 (PB_SQUASH_*).
// ---------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(128) ids_select_kernel(int N, int A, int K, int Nq, const float *__restrict__ q,
                                                         const float *__restrict__ z, float lambda, float eps,
                                                         float rho_lb, long long *__restrict__ action_out,
                                                         float *__restrict__ scores_out)
{
    const int warp = threadIdx.x >> 5, lane = lane_id();
    const int n = blockIdx.x * (blockDim.x >> 5) + warp;
    if (n >= N) return;
    const bool on = lane < A;
    // mean / unbiased std over heads (action_selectors.py:132-135; "variance" is std, "std" is sqrt(std))
    double mu = 0.0;
    if (on) for (int k = 0; k < K; ++k) mu += (double)unsquash<S>(q[((size_t)k * N + n) * A + lane]);
    mu /= (double)K;
    double ss = 0.0;
    if (on) for (int k = 0; k < K; ++k) { double d = (double)unsquash<S>(q[((size_t)k * N + n) * A + lane]) - mu; ss += d * d; }
    const float mean = (float)mu;
    const float s1 = (float)sqrt(ss / (double)(K - 1));          // torch.std (unbiased); K==1 -> nan like torch
    const float s2 = sqrtf(s1);
    // regret (:137-139)
    float ub = on ? mean + lambda * s2 : -INFINITY;
    const float best = warp_max(ub);
    float regret = best - (mean - lambda * s2);
    const float regret_sq = regret * regret;
    // unbiased variance of the return distribution over quantile samples (:141)
    double zm = 0.0;
    if (on) for (int j = 0; j < Nq; ++j) zm += (double)unsquash<S>(z[((size_t)j * N + n) * A + lane]);
    zm /= (double)Nq;
    double zs = 0.0;
    if (on) for (int j = 0; j < Nq; ++j) { double d = (double)unsquash<S>(z[((size_t)j * N + n) * A + lane]) - zm; zs += d * d; }
    const float var_z = (float)(zs / (double)(Nq - 1));
    const float mean_var = warp_sum(on ? var_z : 0.0f) / (float)A;
    const float normalized = var_z / (eps + mean_var);           // (:142)
    const float rho = fmaxf(normalized, rho_lb);                 // (:143)
    const float info_gain = logf(1.0f + s1 / rho) + eps;         // (:146)
    float score = regret_sq / info_gain;                         // (:148)
    if (scores_out && on) scores_out[(size_t)n * A + lane] = score;
    // argmin, first index on ties; NaN never wins (torch.argmin would pick a NaN: flagged in DESIGN.md)
    float bs = on ? score : INFINITY;
    int bi = on ? lane : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float os = __shfl_xor_sync(FULL, bs, o);
        int oi = __shfl_xor_sync(FULL, bi, o);
        if (os < bs || (os == bs && oi < bi)) { bs = os; bi = oi; }
    }
    if (lane == 0) action_out[n] = (bi == 0x7fffffff) ? 0 : bi;
}

// elementwise h / h^-1 (pb_value_squash)
template <int S>
__global__ void __launch_bounds__(256) value_squash_kernel(long long n, const float *x, float *y, int inverse)
{
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        y[e] = inverse ? unsquash<S>(x[e]) : squash<S>(x[e]);
}

__global__ void __launch_bounds__(128) greedy_select_kernel(int N, int A, int K, const float *__restrict__ q,
                                                            long long *__restrict__ action_out)
{
    const int warp = threadIdx.x >> 5, lane = lane_id();
    const int n = blockIdx.x * (blockDim.x >> 5) + warp;
    if (n >= N) return;
    const bool on = lane < A;
    float acc = 0.0f;
    if (on) for (int k = 0; k < K; ++k) acc += q[((size_t)k * N + n) * A + lane];
    float bs = on ? acc / (float)K : -INFINITY;
    int bi = on ? lane : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float os = __shfl_xor_sync(FULL, bs, o);
        int oi = __shfl_xor_sync(FULL, bi, o);
        if (os > bs || (os == bs && oi < bi)) { bs = os; bi = oi; }
    }
    if (lane == 0) action_out[n] = (bi == 0x7fffffff) ? 0 : bi;
}

// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) loss_combine_kernel(int B, const float *__restrict__ dist,
                                                            const float *__restrict__ q, const float *__restrict__ w,
                                                            float q_scale, const float *__restrict__ q_offset,
                                                            float *__restrict__ total_out, float *__restrict__ td_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ float part[32];
    float acc = 0.0f;
    const float off = q_offset ? *q_offset : 0.0f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const float wb = w ? w[b] : 1.0f;
        const float d = dist ? dist[b] : 0.0f, qq = q ? q_scale * (q[b] - off) : 0.0f;
        acc += d * wb + qq * wb;
        if (td_out) td_out[b] = (dist && q) ? (d * 0.5f + qq * 0.5f) : (dist ? d : fabsf(qq));
    }
    acc = warp_sum(acc);
    if (lane_id() == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.0f;
        v = warp_sum(v);
        if (threadIdx.x == 0 && total_out) *total_out = v / (float)B;
    }
}

// ---------------------------------------------------------------------------------
// clip_grad_norm_ + Adam over one flat arena.  Kernel 1: per-CTA partial sum of squares
// (fp64 accumulate of fp32 squares is overkill; fp32 per thread, fp64 across), step++.
// Kernel 2: every CTA re-reduces the <=1024 partials, derives the clip coefficient and
// applies the update with 128-bit accesses.
// adam_clip_kernel and adam_fused_kernel are templates on the update rule R (PB_OPT_*, common.cuh: OptRule,
// opt_update); their names are the Adam family's.  For the RMSprop rules beta1 carries alpha and beta2 is unused; a
// state slot the rule does not keep is never dereferenced.  R = PB_OPT_ADAM compiles to the code of the Adam-only kernels.
// ---------------------------------------------------------------------------------
constexpr int ADAM_THREADS = 256;
constexpr int ADAM_MAX_PARTIALS = 4096;
constexpr int PACK_BLOCKS_PER_TENSOR = 16;

// multi-tensor gather of autograd's per-parameter gradients into the flat arena (scaled), with the
// sum of squares of the scaled values folded in.  table[t] = {grad pointer, arena offset, numel}.
__global__ void __launch_bounds__(ADAM_THREADS) pack_grads_kernel(const long long *__restrict__ table, float scale,
                                                                  float *__restrict__ flat,
                                                                  const unsigned long long *__restrict__ epoch,
                                                                  long long stride, float *__restrict__ partial,
                                                                  long long *__restrict__ step_count)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ double part[ADAM_THREADS / 32];
    if (epoch) flat += (long long)(*epoch & 1ull) * stride;      // double-buffered arena of the peer exchange
    const int t = blockIdx.y;
    const float *__restrict__ src = reinterpret_cast<const float *>(table[3 * t + 0]);
    float *__restrict__ dst = flat + table[3 * t + 1];
    const long long n = table[3 * t + 2];
    double acc = 0.0;
    if (src != nullptr) {
        const bool vec = ((((uintptr_t)src) | ((uintptr_t)dst)) & 15) == 0;
        const long long n4 = vec ? (n >> 2) : 0;
        const long long stride = (long long)gridDim.x * blockDim.x;
        long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + 3 * stride < n4; i += 4 * stride) {               // 4 independent 128-bit loads in flight
            float4 v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = reinterpret_cast<const float4 *>(src)[i + k * stride];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                v[k].x *= scale; v[k].y *= scale; v[k].z *= scale; v[k].w *= scale;
                reinterpret_cast<float4 *>(dst)[i + k * stride] = v[k];
                acc += (double)(v[k].x * v[k].x + v[k].y * v[k].y) + (double)(v[k].z * v[k].z + v[k].w * v[k].w);
            }
        }
        for (; i < n4; i += stride) {
            float4 v = reinterpret_cast<const float4 *>(src)[i];
            v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
            reinterpret_cast<float4 *>(dst)[i] = v;
            acc += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
        }
        for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
             i += (long long)gridDim.x * blockDim.x) {
            float v = src[i] * scale;
            dst[i] = v;
            acc += (double)v * (double)v;
        }
    } else {
        // parameter that received no gradient this step: zero its slice
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
            dst[i] = 0.0f;
    }
    acc = warp_sum(acc);
    if (lane_id() == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int k = 0; k < ADAM_THREADS / 32; ++k) tot += part[k];
        if (partial) partial[blockIdx.y * gridDim.x + blockIdx.x] = (float)tot;
        if (blockIdx.x == 0 && blockIdx.y == 0 && step_count) *step_count += 1;
    }
}

__global__ void __launch_bounds__(ADAM_THREADS) grad_sumsq_kernel(long long n, const float *__restrict__ grad,
                                                                  float *__restrict__ partial,
                                                                  long long *__restrict__ step_count)
{
    __shared__ double part[ADAM_THREADS / 32];
    double acc = 0.0;
    const long long n4 = n >> 2;
    const float4 *g4 = reinterpret_cast<const float4 *>(grad);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        float4 v = g4[i];
        acc += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
    }
    if (blockIdx.x == 0)
        for (long long i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) acc += (double)grad[i] * (double)grad[i];
    acc = warp_sum(acc);
    if (lane_id() == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < ADAM_THREADS / 32; ++k) t += part[k];
        partial[blockIdx.x] = (float)t;
        if (blockIdx.x == 0 && step_count) *step_count += 1;
    }
}

template <int R>
__global__ void __launch_bounds__(ADAM_THREADS) adam_clip_kernel(long long n, float *__restrict__ param,
                                                                 const float *__restrict__ grad,
                                                                 float *__restrict__ exp_avg,
                                                                 float *__restrict__ exp_avg_sq,
                                                                 const long long *__restrict__ step_count, float lr,
                                                                 float beta1, float beta2, float adam_eps,
                                                                 float max_grad_norm, const float *__restrict__ partial,
                                                                 int n_partials, float *__restrict__ norm_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ double red[ADAM_THREADS / 32];
    __shared__ float s_coef, s_bc2_sqrt, s_step_size;
    double acc = 0.0;
    for (int k = threadIdx.x; k < n_partials; k += blockDim.x) acc += (double)partial[k];
    acc = warp_sum(acc);
    if (lane_id() == 0) red[threadIdx.x >> 5] = acc;
    if constexpr (R == PB_OPT_ADAM) {
        if (threadIdx.x == 32) {
            // bias corrections: two fp64 pow() -- once per CTA (another warp than the one that finishes the norm), not
            // once per thread
            const double step = (double)(*step_count);
            const float bc1 = (float)(1.0 - pow((double)beta1, step));
            s_bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, step));
            s_step_size = lr / bc1;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < ADAM_THREADS / 32; ++k) t += red[k];
        const float total_norm = (float)sqrt(t);
        // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
        float coef = max_grad_norm / (total_norm + 1e-6f);
        coef = coef > 1.0f ? 1.0f : coef;
        if (!(max_grad_norm > 0.0f)) coef = 1.0f;
        s_coef = coef;
        if (blockIdx.x == 0 && norm_out) { norm_out[0] = total_norm; norm_out[1] = coef; }
    }
    __syncthreads();
    const float coef = s_coef;
    const float bc2_sqrt = R == PB_OPT_ADAM ? s_bc2_sqrt : 0.0f;
    const float step_size = R == PB_OPT_ADAM ? s_step_size : 0.0f;
    auto upd = [&](float &p, float g, float &m, float &v) {
        g *= coef;
        if constexpr (R == PB_OPT_ADAM) {
            m = m + (g - m) * (1.0f - beta1);                    // exp_avg.lerp_(grad, 1-beta1)
            v = v * beta2 + (1.0f - beta2) * g * g;              // mul_(beta2).addcmul_(g, g, 1-beta2)
            const float denom = sqrtf(v) / bc2_sqrt + adam_eps;
            p = p - step_size * (m / denom);                     // addcdiv_(exp_avg, denom, -step_size)
        } else {
            opt_update<R>(p, g, m, v, lr, beta1, adam_eps);      // beta1 = RMSprop's alpha (common.cuh)
        }
    };
    constexpr bool HM = OptRule<R>::has_m, HV = OptRule<R>::has_v;
    const long long n4 = n >> 2;
    float4 *p4 = reinterpret_cast<float4 *>(param);
    const float4 *g4 = reinterpret_cast<const float4 *>(grad);
    float4 *m4 = reinterpret_cast<float4 *>(exp_avg);
    float4 *v4 = reinterpret_cast<float4 *>(exp_avg_sq);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        float4 p = p4[i], g = g4[i], m, v;
        if constexpr (HM) m = m4[i];
        if constexpr (HV) v = v4[i];
        upd(p.x, g.x, m.x, v.x); upd(p.y, g.y, m.y, v.y); upd(p.z, g.z, m.z, v.z); upd(p.w, g.w, m.w, v.w);
        p4[i] = p;
        if constexpr (HM) m4[i] = m;
        if constexpr (HV) v4[i] = v;
    }
    if (blockIdx.x == 0)
        for (long long i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) {
            float unused = 0.0f;
            upd(param[i], grad[i], HM ? exp_avg[i] : unused, HV ? exp_avg_sq[i] : unused);
        }
}


// ---------------------------------------------------------------------------------
// Small arenas, ONE launch for gather + clip_grad_norm_ + Adam (agent.py:73-74): a thread gathers its 128-bit elements
// of autograd's per-parameter gradients (scaled) INTO REGISTERS (and into the flat gradient arena, for whoever reads
// it), publishes its CTA's sum of squares, meets the other CTAs of the grid at a counter (all resident: the grid is
// sized by the occupancy API), derives the norm from the partials in a fixed order and applies Adam to the elements
// it still holds.  The optimizer state of the first element and the bias corrections are requested before the
// barrier.  Replaces pack_grads_kernel + adam_clip_kernel (two launches, the gradient written and re-read) on the
// configs[0] / [1] steps; arenas beyond FUSED_U elements per thread keep the two-launch path.
// ---------------------------------------------------------------------------------
constexpr int FUSED_U = 8;
constexpr int FUSED_MAX_TENSORS = 64;

template <int R>
__global__ void __launch_bounds__(ADAM_THREADS) adam_fused_kernel(const long long *__restrict__ table, int n_tensors,
                                                                  float scale, long long n, float *__restrict__ param,
                                                                  float *__restrict__ grad, float *__restrict__ exp_avg,
                                                                  float *__restrict__ exp_avg_sq,
                                                                  long long *__restrict__ step_count, float lr,
                                                                  float beta1, float beta2, float adam_eps,
                                                                  float max_grad_norm, float *__restrict__ partials,
                                                                  unsigned int *__restrict__ counters,
                                                                  float *__restrict__ norm_out)
{
    __shared__ long long s_tab[3 * FUSED_MAX_TENSORS];
    __shared__ double red[ADAM_THREADS / 32];
    __shared__ float s_coef;
    __shared__ unsigned s_last;
    for (int e = threadIdx.x; e < 3 * n_tensors; e += blockDim.x) s_tab[e] = table[e];
    const long long step_now = *step_count + 1;
    const long long n4 = n >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x, i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float4 *p4 = reinterpret_cast<float4 *>(param), *m4 = reinterpret_cast<float4 *>(exp_avg),
           *v4 = reinterpret_cast<float4 *>(exp_avg_sq), *g4 = reinterpret_cast<float4 *>(grad);
    constexpr bool HM = OptRule<R>::has_m, HV = OptRule<R>::has_v;
    float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f), m0 = p0, v0 = p0;
    if (i0 < n4) {
        p0 = p4[i0];
        if constexpr (HM) m0 = m4[i0];
        if constexpr (HV) v0 = v4[i0];
    }
    float bc2_sqrt = 0.0f, step_size = 0.0f;
    if constexpr (R == PB_OPT_ADAM) {
        const double step = (double)step_now;
        const float bc1 = (float)(1.0 - pow((double)beta1, step));
        bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, step));
        step_size = lr / bc1;
    }
    __syncthreads();
    // ---- gather: arena offset -> (tensor, offset within it); tensors are laid out in table order, 16-byte aligned
    float4 gsum[FUSED_U];
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < FUSED_U; ++k) {
        const long long i = i0 + k * stride;
        gsum[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n4) {
            const long long o = i << 2;
            int t = 0;
            for (int q = 1; q < n_tensors; ++q) t = s_tab[3 * q + 1] <= o ? q : t;
            const float *src = reinterpret_cast<const float *>(s_tab[3 * t]);
            const long long within = o - s_tab[3 * t + 1], numel = s_tab[3 * t + 2];
            float4 gv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (src != nullptr && within < numel) {
                if (within + 3 < numel && ((reinterpret_cast<uintptr_t>(src + within) & 15) == 0)) {
                    gv = *reinterpret_cast<const float4 *>(src + within);
                } else {
                    gv.x = src[within];
                    gv.y = within + 1 < numel ? src[within + 1] : 0.f;
                    gv.z = within + 2 < numel ? src[within + 2] : 0.f;
                    gv.w = within + 3 < numel ? src[within + 3] : 0.f;
                }
                gv.x *= scale; gv.y *= scale; gv.z *= scale; gv.w *= scale;
            }
            gsum[k] = gv;
            g4[i] = gv;
            acc += (double)(gv.x * gv.x + gv.y * gv.y) + (double)(gv.z * gv.z + gv.w * gv.w);
        }
    }
    acc = warp_sum(acc);
    if (lane_id() == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < ADAM_THREADS / 32; ++k) t += red[k];
        partials[blockIdx.x] = (float)t;
        __threadfence();
        atomicAdd(&counters[0], 1u);
        unsigned seen;
        do {                                                          // meet the other CTAs of this grid (all resident)
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(&counters[0]) : "memory");
        } while (seen < gridDim.x);
    }
    __syncthreads();
    double a2 = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) a2 += (double)__ldcg(partials + k);
    a2 = warp_sum(a2);
    __syncthreads();                                                  // red[] is reused
    if (lane_id() == 0) red[threadIdx.x >> 5] = a2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < ADAM_THREADS / 32; ++k) t += red[k];
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
        if constexpr (R == PB_OPT_ADAM) {
            m = m + (gg - m) * (1.0f - beta1);
            v = v * beta2 + (1.0f - beta2) * gg * gg;
            const float denom = sqrtf(v) / bc2_sqrt + adam_eps;
            p = p - step_size * (m / denom);
        } else {
            opt_update<R>(p, gg, m, v, lr, beta1, adam_eps);
        }
    };
#pragma unroll
    for (int k = 0; k < FUSED_U; ++k) {
        const long long i = i0 + k * stride;
        if (i < n4) {
            float4 p = p0, m = m0, v = v0;
            if (k > 0) {
                p = p4[i];
                if constexpr (HM) m = m4[i];
                if constexpr (HV) v = v4[i];
            }
            const float4 gr = gsum[k];
            upd(p.x, gr.x, m.x, v.x); upd(p.y, gr.y, m.y, v.y); upd(p.z, gr.z, m.z, v.z); upd(p.w, gr.w, m.w, v.w);
            p4[i] = p;
            if constexpr (HM) m4[i] = m;
            if constexpr (HV) v4[i] = v;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&counters[1], 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        counters[0] = 0u; counters[1] = 0u;
        *step_count = step_now;
    }
}

// rule -> kernel instantiation (nullptr: unknown rule)
static decltype(&adam_fused_kernel<PB_OPT_ADAM>) fused_kernel(int rule)
{
    switch (rule) {
    case PB_OPT_ADAM: return adam_fused_kernel<PB_OPT_ADAM>;
    case PB_OPT_RMSPROP: return adam_fused_kernel<PB_OPT_RMSPROP>;
    case PB_OPT_RMSPROP_CENTERED: return adam_fused_kernel<PB_OPT_RMSPROP_CENTERED>;
    case PB_OPT_SGD: return adam_fused_kernel<PB_OPT_SGD>;
    }
    return nullptr;
}

static decltype(&adam_clip_kernel<PB_OPT_ADAM>) clip_kernel(int rule)
{
    switch (rule) {
    case PB_OPT_ADAM: return adam_clip_kernel<PB_OPT_ADAM>;
    case PB_OPT_RMSPROP: return adam_clip_kernel<PB_OPT_RMSPROP>;
    case PB_OPT_RMSPROP_CENTERED: return adam_clip_kernel<PB_OPT_RMSPROP_CENTERED>;
    case PB_OPT_SGD: return adam_clip_kernel<PB_OPT_SGD>;
    }
    return nullptr;
}

// squash kind -> kernel instantiation (nullptr: unknown kind)
#define PB_SQUASH_PICK(kernel, s)                                                                          \
    ((s) == PB_SQUASH_NONE ? kernel<PB_SQUASH_NONE>                                                      \
     : (s) == PB_SQUASH_OBS_LOOK_FURTHER ? kernel<PB_SQUASH_OBS_LOOK_FURTHER>                            \
     : (s) == PB_SQUASH_SYMLOG ? kernel<PB_SQUASH_SYMLOG> : nullptr)

// CTAs of the rule's fused kernel that are resident at once (its grid never exceeds this: the CTAs meet at a counter)
static int fused_max_blocks(int rule)
{
    static std::atomic<int> cached[4][64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    int c = cached[rule][dev].load(std::memory_order_relaxed);
    if (c > 0) return c;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fused_kernel(rule), ADAM_THREADS, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    c = pb_sm_count() * per_sm;
    cached[rule][dev].store(c, std::memory_order_relaxed);
    return c;
}

}  // namespace

extern "C" {

int pb_iqn_cos_basis(long long n_rows, int n_basis, const float *tau, float *out, void *stream)
{
    if (n_rows < 0 || n_basis <= 0) return PB_E_ARG;
    if (n_rows == 0) return PB_OK;
    if (!tau || !out) return PB_E_ARG;
    const long long total = n_rows * n_basis;
    long long nb = (total + 255) / 256;
    const long long cap = (long long)pb_sm_count() * 16;
    if (nb > cap) nb = cap;
    PB_LAUNCH(cos_basis_kernel, (unsigned)nb, 256, 0, stream, n_rows, n_basis, tau, out);
    return PB_OK;
}

int pb_iqn_qh_loss(int B, int T, int Tp, int A, const float *z_cur, const float *tau, const float *z_next_online,
                   const float *z_next_target, const long long *action, const float *ret, const float *gdn,
                   const uint8_t *nonterminal, float kappa, float loss_weight, const float *row_weight,
                   float grad_scale, float *loss_out, float *grad_z_cur, void *stream)
{
    return pb_iqn_qh_loss_sq(B, T, Tp, A, z_cur, tau, z_next_online, z_next_target, action, ret, gdn, nonterminal, kappa,
                             loss_weight, row_weight, grad_scale, loss_out, grad_z_cur, stream, PB_SQUASH_NONE);
}

int pb_iqn_qh_loss_sq(int B, int T, int Tp, int A, const float *z_cur, const float *tau, const float *z_next_online,
                      const float *z_next_target, const long long *action, const float *ret, const float *gdn,
                      const uint8_t *nonterminal, float kappa, float loss_weight, const float *row_weight,
                      float grad_scale, float *loss_out, float *grad_z_cur, void *stream, int squash)
{
    const auto kernel = PB_SQUASH_PICK(qh_loss_kernel, squash);
    if (!kernel) return PB_E_UNSUPPORTED;
    if (B < 0 || T <= 0 || Tp <= 0 || A <= 0 || !(kappa > 0.0f)) return PB_E_ARG;
    if (B == 0) return PB_OK;
    if (!z_cur || !tau || !z_next_online || !z_next_target || !action || !ret || !gdn || !loss_out || !grad_z_cur)
        return PB_E_ARG;
    const int warps = 4;
    const size_t smem = sizeof(float) * warps * (size_t)(Tp + 2 * T);
    if (smem > 48 * 1024) return PB_E_UNSUPPORTED;
    PB_LAUNCH(kernel, (unsigned)((B + warps - 1) / warps), warps * 32, smem, stream, B, T, Tp, A, z_cur, tau,
              z_next_online, z_next_target, action, ret, gdn, nonterminal, kappa, loss_weight, row_weight, grad_scale,
              loss_out, grad_z_cur);
    return PB_OK;
}

int pb_ens_q_loss(int B, int A, int K, const float *q_cur, const float *q_next_online, const float *q_next_target,
                  const long long *action, const float *ret, const float *gdn, const uint8_t *nonterminal,
                  float loss_weight, const float *row_weight, float grad_scale, float *loss_out, float *grad_q_cur,
                  void *stream)
{
    return pb_ens_q_loss_sq(B, A, K, q_cur, q_next_online, q_next_target, action, ret, gdn, nonterminal, loss_weight,
                            row_weight, grad_scale, loss_out, grad_q_cur, stream, PB_SQUASH_NONE);
}

int pb_ens_q_loss_sq(int B, int A, int K, const float *q_cur, const float *q_next_online, const float *q_next_target,
                     const long long *action, const float *ret, const float *gdn, const uint8_t *nonterminal,
                     float loss_weight, const float *row_weight, float grad_scale, float *loss_out, float *grad_q_cur,
                     void *stream, int squash)
{
    const auto kernel = PB_SQUASH_PICK(ens_loss_kernel, squash);
    if (!kernel) return PB_E_UNSUPPORTED;
    if (B < 0 || A <= 0 || K <= 0) return PB_E_ARG;
    if (B == 0) return PB_OK;
    if (!q_cur || !q_next_online || !q_next_target || !action || !ret || !gdn || !loss_out || !grad_q_cur)
        return PB_E_ARG;
    PB_LAUNCH(kernel, (unsigned)((B + 3) / 4), 128, 0, stream, B, A, K, q_cur, q_next_online, q_next_target,
              action, ret, gdn, nonterminal, loss_weight, row_weight, grad_scale, loss_out, grad_q_cur,
              (const float *)nullptr, 1.0f, (const float *)nullptr, (float *)nullptr, (float *)nullptr, (unsigned int *)nullptr);
    return PB_OK;
}

int pb_ens_q_loss_total(int B, int A, int K, const float *q_cur, const float *q_next_online, const float *q_next_target,
                        const long long *action, const float *ret, const float *gdn, const uint8_t *nonterminal,
                        float loss_weight, const float *row_weight, float grad_scale, float *loss_out, float *grad_q_cur,
                        const float *dist, float q_scale, const float *q_offset, float *total_out, float *td_out,
                        unsigned int *ticket, void *stream)
{
    return pb_ens_q_loss_total_sq(B, A, K, q_cur, q_next_online, q_next_target, action, ret, gdn, nonterminal,
                                  loss_weight, row_weight, grad_scale, loss_out, grad_q_cur, dist, q_scale, q_offset,
                                  total_out, td_out, ticket, stream, PB_SQUASH_NONE);
}

int pb_ens_q_loss_total_sq(int B, int A, int K, const float *q_cur, const float *q_next_online,
                           const float *q_next_target, const long long *action, const float *ret, const float *gdn,
                           const uint8_t *nonterminal, float loss_weight, const float *row_weight, float grad_scale,
                           float *loss_out, float *grad_q_cur, const float *dist, float q_scale,
                           const float *q_offset, float *total_out, float *td_out, unsigned int *ticket,
                           void *stream, int squash)
{
    const auto kernel = PB_SQUASH_PICK(ens_loss_kernel, squash);
    if (!kernel) return PB_E_UNSUPPORTED;
    if (B < 0 || A <= 0 || K <= 0) return PB_E_ARG;
    if (B == 0) return PB_OK;
    if (!q_cur || !q_next_online || !q_next_target || !action || !ret || !gdn || !loss_out || !grad_q_cur || !total_out ||
        !ticket)
        return PB_E_ARG;
    PB_LAUNCH(kernel, (unsigned)((B + 3) / 4), 128, 0, stream, B, A, K, q_cur, q_next_online, q_next_target,
              action, ret, gdn, nonterminal, loss_weight, row_weight, grad_scale, loss_out, grad_q_cur, dist, q_scale,
              q_offset, total_out, td_out, ticket);
    return PB_OK;
}

int pb_ids_select(int N, int A, int K, int Nq, const float *q, const float *z, float lambda, float eps,
                  float rho_lower_bound, long long *action_out, float *scores_out, void *stream)
{
    return pb_ids_select_sq(N, A, K, Nq, q, z, lambda, eps, rho_lower_bound, action_out, scores_out, stream,
                            PB_SQUASH_NONE);
}

int pb_ids_select_sq(int N, int A, int K, int Nq, const float *q, const float *z, float lambda, float eps,
                     float rho_lower_bound, long long *action_out, float *scores_out, void *stream, int squash)
{
    const auto kernel = PB_SQUASH_PICK(ids_select_kernel, squash);
    if (!kernel) return PB_E_UNSUPPORTED;
    if (N < 0 || A <= 0 || K <= 0 || Nq <= 0) return PB_E_ARG;
    if (A > 32) return PB_E_UNSUPPORTED;
    if (N == 0) return PB_OK;
    if (!q || !z || !action_out) return PB_E_ARG;
    PB_LAUNCH(kernel, (unsigned)((N + 3) / 4), 128, 0, stream, N, A, K, Nq, q, z, lambda, eps,
              rho_lower_bound, action_out, scores_out);
    return PB_OK;
}

int pb_value_squash(long long n, const float *x, float *y, int squash, int inverse, void *stream)
{
    const auto kernel = PB_SQUASH_PICK(value_squash_kernel, squash);
    if (!kernel) return PB_E_UNSUPPORTED;
    if (n < 0 || (inverse != 0 && inverse != 1)) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (!x || !y) return PB_E_ARG;
    long long nb = (n + 255) / 256;
    const long long cap = (long long)pb_sm_count() * 16;
    if (nb > cap) nb = cap;
    PB_LAUNCH(kernel, (unsigned)nb, 256, 0, stream, n, x, y, inverse);
    return PB_OK;
}

int pb_greedy_select(int N, int A, int K, const float *q, long long *action_out, void *stream)
{
    if (N < 0 || A <= 0 || K <= 0) return PB_E_ARG;
    if (A > 32) return PB_E_UNSUPPORTED;
    if (N == 0) return PB_OK;
    if (!q || !action_out) return PB_E_ARG;
    PB_LAUNCH(greedy_select_kernel, (unsigned)((N + 3) / 4), 128, 0, stream, N, A, K, q, action_out);
    return PB_OK;
}

int pb_loss_combine(int B, const float *dist, const float *q, const float *w, float q_scale, const float *q_offset,
                    float *total_out, float *td_out, void *stream)
{
    if (B <= 0 || (!dist && !q)) return PB_E_ARG;
    PB_LAUNCH(loss_combine_kernel, 1, 1024, 0, stream, B, dist, q, w, q_scale, q_offset, total_out, td_out);
    return PB_OK;
}

int pb_pack_grads(int n_tensors, const long long *table, float scale, float *flat, float *partial_scratch,
                  long long *step_count, int *n_partials_out_h, void *stream)
{
    return pb_pack_grads_parity(n_tensors, table, scale, flat, nullptr, 0, partial_scratch, step_count, n_partials_out_h,
                                stream);
}

int pb_pack_grads_parity(int n_tensors, const long long *table, float scale, float *flat,
                         const unsigned long long *epoch, long long stride, float *partial_scratch,
                         long long *step_count, int *n_partials_out_h, void *stream)
{
    if (n_tensors <= 0 || !table || !flat || stride < 0 || (stride & 3)) return PB_E_ARG;
    if ((long long)n_tensors * PACK_BLOCKS_PER_TENSOR > ADAM_MAX_PARTIALS) return PB_E_UNSUPPORTED;
    // as many blocks per tensor as the partial-sum table allows (blocks of small tensors exit at once; the
    // multi-million-element tensors need the whole machine)
    int per = ADAM_MAX_PARTIALS / n_tensors;
    if (per > 128) per = 128;
    if (per < PACK_BLOCKS_PER_TENSOR) per = PACK_BLOCKS_PER_TENSOR;
    dim3 grid((unsigned)per, (unsigned)n_tensors);
    PB_LAUNCH(pack_grads_kernel, grid, ADAM_THREADS, 0, stream, table, scale, flat, epoch, stride, partial_scratch,
              step_count);
    if (n_partials_out_h) *n_partials_out_h = n_tensors * per;
    return PB_OK;
}

int pb_grad_sumsq(long long n, const float *grad, float *partial_scratch, long long *step_count,
                  int *n_partials_out_h, void *stream)
{
    if (n <= 0 || !grad || !partial_scratch) return PB_E_ARG;
    if (((uintptr_t)grad) & 15) return PB_E_ARG;
    long long nb = ((n >> 2) + ADAM_THREADS - 1) / ADAM_THREADS;
    if (nb < 1) nb = 1;
    const long long cap = (long long)pb_sm_count() * 4;
    if (nb > cap) nb = cap;
    if (nb > ADAM_MAX_PARTIALS) nb = ADAM_MAX_PARTIALS;
    PB_LAUNCH(grad_sumsq_kernel, (unsigned)nb, ADAM_THREADS, 0, stream, n, grad, partial_scratch, step_count);
    if (n_partials_out_h) *n_partials_out_h = (int)nb;
    return PB_OK;
}

int pb_opt_clip_apply(int rule, long long n, float *param, const float *grad, float *m, float *v,
                      const long long *step_count, float lr, float h1, float h2, float eps, float max_grad_norm,
                      const float *partial_scratch, int n_partials, float *norm_out, void *stream)
{
    if (pb_opt_check(rule, m, v)) return PB_E_ARG;
    if (n <= 0 || !param || !grad || !step_count || !partial_scratch) return PB_E_ARG;
    if (n_partials <= 0 || n_partials > ADAM_MAX_PARTIALS) return PB_E_ARG;
    if ((((uintptr_t)param) | ((uintptr_t)grad) | ((uintptr_t)m) | ((uintptr_t)v)) & 15) return PB_E_ARG;
    long long nb = ((n >> 2) + ADAM_THREADS - 1) / ADAM_THREADS;
    if (nb < 1) nb = 1;
    const long long cap = (long long)pb_sm_count() * 4;
    if (nb > cap) nb = cap;
    PB_LAUNCH(clip_kernel(rule), (unsigned)nb, ADAM_THREADS, 0, stream, n, param, grad, m, v, step_count,
              lr, h1, h2, eps, max_grad_norm, partial_scratch, n_partials, norm_out);
    return PB_OK;
}

int pb_adam_clip_apply(long long n, float *param, const float *grad, float *exp_avg, float *exp_avg_sq,
                       const long long *step_count, float lr, float beta1, float beta2, float adam_eps,
                       float max_grad_norm, const float *partial_scratch, int n_partials, float *norm_out,
                       void *stream)
{
    return pb_opt_clip_apply(PB_OPT_ADAM, n, param, grad, exp_avg, exp_avg_sq, step_count, lr, beta1, beta2, adam_eps,
                             max_grad_norm, partial_scratch, n_partials, norm_out, stream);
}

// load the optimizer kernels now (see pb_peer_preload)
int pb_optimizer_preload(void)
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, pack_grads_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, grad_sumsq_kernel);
    for (int rule = PB_OPT_ADAM; rule <= PB_OPT_SGD && e == cudaSuccess; ++rule) {
        e = cudaFuncGetAttributes(&a, clip_kernel(rule));
        if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, fused_kernel(rule));
    }
    return e == cudaSuccess ? PB_OK : (int)e;
}

long long pb_opt_fused_max_n(int rule)
{
    if (!pb_opt_known(rule)) return 0;
    return (long long)fused_max_blocks(rule) * ADAM_THREADS * FUSED_U * 4;
}

long long pb_adam_fused_max_n(void) { return pb_opt_fused_max_n(PB_OPT_ADAM); }

int pb_opt_fused_step(int rule, int n_tensors, const long long *table, float scale, long long n, float *param, float *grad,
                      float *m, float *v, long long *step_count, float lr, float h1, float h2, float eps,
                      float max_grad_norm, float *partial_scratch, float *norm_out, void *stream)
{
    if (pb_opt_check(rule, m, v)) return PB_E_ARG;
    if (n_tensors <= 0 || !table || n <= 0 || (n % 4) != 0 || !param || !grad || !step_count || !partial_scratch)
        return PB_E_ARG;
    if (n_tensors > FUSED_MAX_TENSORS || n > pb_opt_fused_max_n(rule)) return PB_E_UNSUPPORTED;
    if ((((uintptr_t)param) | ((uintptr_t)grad) | ((uintptr_t)m) | ((uintptr_t)v)) & 15) return PB_E_ARG;
    long long nb = ((n >> 2) + ADAM_THREADS - 1) / ADAM_THREADS;
    const long long cap = fused_max_blocks(rule);
    if (nb > cap) nb = cap;
    if (nb < 1) nb = 1;
    unsigned int *counters = reinterpret_cast<unsigned int *>(partial_scratch + 4092);    // zero between calls
    PB_LAUNCH(fused_kernel(rule), (unsigned)nb, ADAM_THREADS, 0, stream, table, n_tensors, scale, n, param, grad, m, v,
              step_count, lr, h1, h2, eps, max_grad_norm, partial_scratch, counters, norm_out);
    return PB_OK;
}

int pb_adam_fused_step(int n_tensors, const long long *table, float scale, long long n, float *param, float *grad,
                       float *exp_avg, float *exp_avg_sq, long long *step_count, float lr, float beta1, float beta2,
                       float adam_eps, float max_grad_norm, float *partial_scratch, float *norm_out, void *stream)
{
    return pb_opt_fused_step(PB_OPT_ADAM, n_tensors, table, scale, n, param, grad, exp_avg, exp_avg_sq, step_count, lr,
                             beta1, beta2, adam_eps, max_grad_norm, partial_scratch, norm_out, stream);
}

int pb_adam_clip_step(long long n, float *param, const float *grad, float *exp_avg, float *exp_avg_sq,
                      long long *step_count, float lr, float beta1, float beta2, float adam_eps,
                      float max_grad_norm, float *norm_out, float *partial_scratch, void *stream)
{
    int n_partials = 0;
    int rc = pb_grad_sumsq(n, grad, partial_scratch, step_count, &n_partials, stream);
    if (rc) return rc;
    return pb_adam_clip_apply(n, param, grad, exp_avg, exp_avg_sq, step_count, lr, beta1, beta2, adam_eps,
                              max_grad_norm, partial_scratch, n_partials, norm_out, stream);
}

}  // extern "C"
