// uniform.cu -- device-resident uniform replay sampler (sm_100a).
//
// Replaces the sampler of torchrl's uniform ``ReplayBuffer`` that the reference builds when ``use_per`` is off
// (prism/factory/exp_buffer_factory.py:29-33) -- its DEFAULT_CONFIG.  The sampler's whole state is the 64-byte
// pb_per_state block of the prioritized store, of which it reads len, seq, status, owned_lo / owned_n and the rng words
// pad[1..3] (ticket, call number, seed; same meaning as in per_tree.cu).  Because it is the same block, the peer
// exchange (pb_peer_state_put) carries it unchanged and the learner's data-parallel step works as for PER.
//  * init / extend are single-thread launches: the length lives on the device, so a step graph that ingests new
//    transitions and samples the next batch replays without a host round trip.
//  * sample: idx = floor(u * len) (iid, the eager path of TimestepBuffer.sample) or floor((k + u) / n * len)
//    (stratified), fp64 with explicit round-to-nearest operations; weight 1.
//  * global sampling over the concatenated shards: g_k = floor((k + u) / n_global * total), owner from the prefix sums
//    of the shard lengths.  g_k is monotone in k, so each rank's strata are one contiguous run, found by a search.
#include "common.cuh"

namespace {

using namespace pb;

constexpr int US_THREADS = 256;
constexpr int MAX_RANKS = 64;

__global__ void uniform_init_kernel(pb_per_state *st, long long size, long long seq, int seed)
{
    pb_per_state s;
    s.len = seq < size ? seq : size; s.seq = seq; s.max_priority = 0.0f; s.p_sum = 0.0f; s.p_min = 0.0f; s.status = 0;
    s.batch_max = 0.0f; s.owned_lo = 0; s.owned_n = 0;
    for (int k = 0; k < 5; ++k) s.pad[k] = 0;
    s.pad[3] = seed;
    *st = s;
}

__global__ void uniform_extend_kernel(pb_per_state *st, long long size, long long n)
{
    const long long seq = st->seq + n;
    st->seq = seq;
    st->len = seq < size ? seq : size;
}

// idx of sample k: fp64 u * len (iid) or (k + u) / n * len (stratified), truncated, clamped to len - 1
__device__ __forceinline__ long long uniform_index(int mode, long long k, double uk, long long n, long long len)
{
    const double x = mode == 0 ? __dmul_rn(uk, (double)len)
                               : __dmul_rn(__ddiv_rn(__dadd_rn((double)k, uk), (double)n), (double)len);
    const long long i = (long long)x;
    return i > len - 1 ? len - 1 : i;
}

__global__ void __launch_bounds__(US_THREADS) uniform_sample_kernel(pb_per_state *st, long long n, const double *u,
                                                                    int mode, long long *idx_out, float *w_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const unsigned call = (unsigned)st->pad[2], seed = (unsigned)st->pad[3];
    const long long len = st->len;
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) {
        if (len <= 0) {
            idx_out[k] = 0; w_out[k] = 0.0f;
            if (k == 0) atomicOr(&st->status, PB_ST_EMPTY);
        } else {
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            idx_out[k] = uniform_index(mode, k, uk, n, len);
            w_out[k] = 1.0f;
        }
    }
    if (!u) { __syncthreads(); rng_advance(st); }
}

// first stratum k in [0, n] whose global index g_k (stratified over the concatenated shards) is >= bound (n when there is none); one warp, 32-ary search over the monotone
// predicate (the search of first_owned in per_tree.cu)
__device__ long long first_at_or_past(long long bound, long long n, long long total, const double *u, unsigned seed,
                                      unsigned call)
{
    const int lane = lane_id();
    long long lo = 0, hi = n;                                     // the answer lies in [lo, hi]
    while (lo < hi) {
        const long long step = (hi - lo + 31) / 32;
        const long long k = lo + (long long)lane * step;          // 32 probes, lo first
        bool ge = true;                                           // probes at or past hi count as "past"
        if (k < hi) {
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            ge = uniform_index(1, k, uk, n, total) >= bound;
        }
        const unsigned m = __ballot_sync(FULL, ge);
        if (m == 0u) { lo = lo + 31 * step + 1; continue; }       // all 32 probes below hi and none past yet
        const int first = __ffs(m) - 1;
        if (first == 0) { hi = lo; break; }
        const long long k_first = lo + (long long)first * step;
        lo = k_first - step + 1;                                  // probe first-1 was not past
        hi = k_first < hi ? k_first : hi;
    }
    return hi;
}

__global__ void __launch_bounds__(US_THREADS) uniform_global_sample_kernel(pb_per_state *st, const pb_per_state *all_state,
                                                                           int G, int rank, long long n_global,
                                                                           const double *u, long long *idx_out,
                                                                           float *w_out, long long *stratum_out,
                                                                           PeerWait pw)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ long long prefix[MAX_RANKS + 1];                   // prefix[r] = sum of the lengths of ranks < r
    __shared__ long long run[2];
    if (pw.flags) all_state = peer_wait_states(pw, G);
    if (threadIdx.x == 0) {
        long long acc = 0;
        for (int r = 0; r < G; ++r) {
            prefix[r] = acc;
            const long long len = ld_state_s64(&all_state[r].len);
            acc += len > 0 ? len : 0;
        }
        prefix[G] = acc;
    }
    __syncthreads();
    const long long total = prefix[G], base = prefix[rank];
    const unsigned call = (unsigned)st->pad[2], seed = (unsigned)st->pad[3];
    if (threadIdx.x < 32) {
        long long lo = n_global, hi = n_global;                   // an empty global buffer: nothing is owned
        if (total > 0) {
            lo = first_at_or_past(base, n_global, total, u, seed, call);
            hi = first_at_or_past(prefix[rank + 1], n_global, total, u, seed, call);
        }
        if (threadIdx.x == 0) { run[0] = lo; run[1] = hi; }
    }
    __syncthreads();
    const long long lo = run[0], cnt = run[1] - run[0];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        st->owned_lo = (int)lo; st->owned_n = (int)cnt;
        if (total <= 0) atomicOr(&st->status, PB_ST_EMPTY);
    }
    const long long pos = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // output row
    if (pos < n_global) {
        if (pos < cnt) {
            const long long k = lo + pos;
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            idx_out[pos] = uniform_index(1, k, uk, n_global, total) - base;
            w_out[pos] = 1.0f;
            if (stratum_out) stratum_out[pos] = k;
        } else {                                                  // padding rows of the static batch: skipped downstream
            idx_out[pos] = -1; w_out[pos] = 0.0f;
            if (stratum_out) stratum_out[pos] = -1;
        }
    }
    if (!u) { __syncthreads(); rng_advance(st); }
}

unsigned grid_for(long long n) { return (unsigned)((n + US_THREADS - 1) / US_THREADS); }

}  // namespace

extern "C" {

int pb_uniform_init(pb_per_state *state, long long size, long long seq, int seed, void *stream)
{
    if (!state || size <= 0 || seq < 0) return PB_E_ARG;
    PB_LAUNCH(uniform_init_kernel, 1, 1, 0, stream, state, size, seq, seed);
    return PB_OK;
}

int pb_uniform_extend(pb_per_state *state, long long size, long long n, void *stream)
{
    if (!state || size <= 0 || n < 0) return PB_E_ARG;
    PB_LAUNCH(uniform_extend_kernel, 1, 1, 0, stream, state, size, n);
    return PB_OK;
}

int pb_uniform_sample(pb_per_state *state, long long n, const double *u, int mode, long long *idx_out,
                      float *weight_out, void *stream)
{
    if (!state || n < 0 || n >= (1LL << 31) || (mode != 0 && mode != 1)) return PB_E_ARG;
    if (n > 0 && (!idx_out || !weight_out)) return PB_E_ARG;
    if (n == 0) return PB_OK;
    PB_LAUNCH_PDL(uniform_sample_kernel, grid_for(n), US_THREADS, 0, stream, state, n, u, mode, idx_out, weight_out);
    return PB_OK;
}

int pb_uniform_sample_global(pb_per_state *state, int n_ranks, int rank, const pb_per_state *all_state,
                             long long n_global, const double *u, long long *idx_out, float *weight_out,
                             long long *stratum_out, void *stream)
{
    if (!state || !all_state || n_ranks < 1 || n_ranks > MAX_RANKS || rank < 0 || rank >= n_ranks) return PB_E_ARG;
    if (n_global < 0 || n_global >= (1LL << 31)) return PB_E_ARG;
    if (n_global > 0 && (!idx_out || !weight_out)) return PB_E_ARG;
    if (n_global == 0) return PB_OK;
    PeerWait pw = {};
    PB_LAUNCH_PDL(uniform_global_sample_kernel, grid_for(n_global), US_THREADS, 0, stream, state, all_state, n_ranks,
                  rank, n_global, u, idx_out, weight_out, stratum_out, pw);
    return PB_OK;
}

int pb_uniform_sample_global_peer(pb_per_state *state, const pb_peer_group *g, long long n_global, const double *u,
                                  long long *idx_out, float *weight_out, long long *stratum_out, void *stream)
{
    if (!state || !g || g->world < 1 || g->world > PB_PEER_MAX || g->rank < 0 || g->rank >= g->world) return PB_E_ARG;
    if (!g->flags[g->rank] || !g->state[g->rank] || !g->epoch || n_global < 0 || n_global >= (1LL << 31))
        return PB_E_ARG;
    if (n_global > 0 && (!idx_out || !weight_out)) return PB_E_ARG;
    if (n_global == 0) return PB_OK;
    PeerWait pw;
    pw.flags = g->flags[g->rank] + 2 * PB_PEER_MAX;
    pw.epoch = g->epoch + 2;
    pw.slots = g->state[g->rank];
    pw.status = g->status;
    pw.timeout_ns = g->timeout_ns;
    pw.slot_bytes = PB_PEER_MAX * 64;
    PB_LAUNCH_PDL(uniform_global_sample_kernel, grid_for(n_global), US_THREADS, 0, stream, state,
                  (const pb_per_state *)nullptr, g->world, g->rank, n_global, u, idx_out, weight_out, stratum_out, pw);
    return PB_OK;
}

}  // extern "C"
