/*
 * prism_b200.h -- C ABI of libprism_b200.so (hand-written sm_100a CUDA).
 *
 * Drop-in boundary for the learner-side hot path of AechPro/Prism.  The
 * reference is 100 % Python and has no FFI of its own; the only native code it
 * touches is torchrl's segment tree (a pybind C++ extension inside a
 * third-party wheel).  Each entry point below therefore cites the reference
 * *call site* it replaces (paths relative to the reference repository).
 *
 * Conventions
 *   - every function returns int: 0 ok, <0 argument error (PB_E_*), >0 a
 *     cudaError_t.  Nothing throws, nothing synchronises the stream, nothing
 *     allocates device memory: the caller (PyTorch) owns every buffer and the
 *     library borrows raw pointers for the duration of the stream-ordered call.
 *   - `stream` is a cudaStream_t passed as void*.
 *   - all entry points are CUDA-graph capturable (no host reads of device data).
 *   - pointers are DEVICE pointers unless the name ends in _h (host).
 *   - a few entry points are HOST functions (no stream argument, no device work): the ingest planner
 *     (pb_store_extend_plan, pb_store_stage_block), the wire codec (pb_wire_*), the peer-memory set-up
 *     (pb_peer_alloc / export / open / close / free, which do allocate or map) and the event / copy wrappers.
 *   - thread-compatible: no globals except a launch counter (atomic) and per-device one-time kernel attributes.
 */
#ifndef PRISM_B200_H
#define PRISM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_ABI_VERSION 2

enum {
    PB_OK = 0,
    PB_E_ARG = -1,          /* null pointer / negative size / unsupported shape */
    PB_E_CAPACITY = -2,     /* capacity not a power of two or size > capacity   */
    PB_E_UNSUPPORTED = -3,  /* dtype / option not implemented                   */
    PB_E_POOL = -4          /* aux observation pool exhausted (host planner)    */
};

/* device-side status bits accumulated in pb_per_state.status */
enum {
    PB_ST_EMPTY = 1,        /* sample on an empty shard        (torchrl: RuntimeError) */
    PB_ST_PSUM_NONPOS = 2,  /* p_sum <= 0                      (torchrl: RuntimeError) */
    PB_ST_PMIN_NONPOS = 4   /* p_min <= 0                      (torchrl: RuntimeError) */
};

int         pb_abi_version(void);
/* Thin stream / event / copy wrappers (cudaEvent_t / cudaStream_t as void*): the per-iteration host path of the
 * fused ingest orders its pinned->device staging copy against the step graph through these. */
int pb_event_create(void **event);
int pb_event_destroy(void *event);
int pb_event_record(void *event, void *stream);
int pb_event_synchronize(void *event);
int pb_stream_wait_event(void *stream, void *event);
int pb_copy_h2d_async(void *dst, const void *src, long long bytes, void *stream);
int pb_copy_d2h_async(void *dst, const void *src, long long bytes, void *stream);
int pb_copy_d2d_async(void *dst, const void *src, long long bytes, void *stream);
/* one host call per iteration of the fused ingest: copy_stream waits for after_event (NULL: none), copies the pinned
 * block src -> dst, records copied_event; main_stream waits for copied_event */
int pb_staged_copy_submit(void *copy_stream, void *after_event, void *dst, const void *src, long long bytes,
                          void *copied_event, void *main_stream);
const char *pb_error_string(int code);
/* number of kernels this library has launched in this process (bench: gpu_launches) */
long long   pb_launch_count(void);

/* ------------------------------------------------------------------------- *
 * Prioritized replay: sum-tree + min-tree priority store.
 * Replaces torchrl.data.PrioritizedReplayBuffer's sampler as constructed at
 * prism/factory/exp_buffer_factory.py:22-28.
 * Every node is fl32(left + right) / min(left, right) of a binary tree over the
 * leaves: the reference's add order.  Layout ("compact"): a warp rebuilds the 5
 * levels above a 128-byte line of 32 sibling nodes with shuffles, bit-identical to
 * the nodes a pointer-walking tree would store, so only every 5th level is kept:
 *     levels 0 .. TL               one level-ordered heap array of 2^(TL+1) floats
 *                                  (node i: children 2i, 2i+1; TL <= 14)
 *     levels TL+5, TL+10, .., L    one array of 2^level floats each, L = leaves
 * and the min tree has no leaf array of its own (a leaf holds the same value in both
 * trees; slots >= len read as +inf on the min side).  pb_tree_layout() gives the
 * sizes; pb_tree_export() materialises the full 2*capacity arrays.
 * ------------------------------------------------------------------------- */

/* 64-byte device-resident state block of one shard */
typedef struct pb_per_state {
    long long len;           /* filled slots                                   */
    long long seq;           /* number of transitions ever written (cursor = seq % size) */
    float     max_priority;  /* torchrl _max_priority, starts at 1             */
    float     p_sum;         /* query_sum(0, len), refreshed by every mutation */
    float     p_min;         /* query_min(0, len)                              */
    int       status;        /* PB_ST_* bits (sticky)                          */
    float     batch_max;     /* scratch: max priority of the batch in flight   */
    int       owned_lo;      /* global sampling: first stratum owned by this rank */
    int       owned_n;       /* global sampling: number of strata owned        */
    int       pad[5];        /* [0] top-kernel ticket, [1] rng ticket, [2] rng call number, [3] rng seed, [4] spare */
} pb_per_state;

typedef struct pb_tree {
    float        *sum;       /* compact sum store, pb_tree_layout() floats (leaves last) */
    float        *min;       /* compact min store, pb_tree_layout() floats (no leaf level) */
    int          *owner;     /* reserved, may be NULL (unsorted updates dedup on the leaf slots themselves) */
    int          *counters;  /* pb_tree_layout() ints of reserved scratch, all 0 (no kernel uses a side array any more) */
    pb_per_state *state;
    long long     capacity;  /* power of two */
    long long     size;      /* addressable slots N <= capacity */
    float         alpha;     /* priority exponent (0.5 in every reference config) */
    float         eps_f32;   /* eps as torch adds it to an fp32 tensor */
    double        eps_f64;   /* eps as python adds it to a float */
    int           weight_eps_in_denominator; /* w = (p/(p_min+eps))^-beta variant */
    int           default_priority_fp64;     /* (max_p+eps)^alpha in double, then cast */
} pb_tree;

/* HOST: sizes of the compact stores for a power-of-two capacity (any output may be NULL): floats of the sum store,
 * floats of the min store, ints of the reserved scratch, float offset of leaf 0 inside the sum store, and TL. */
int pb_tree_layout(long long capacity, long long *sum_floats, long long *min_floats, long long *counter_ints,
                   long long *leaf_offset, int *top_level);

/* zero the trees (sum 0, min +inf), counters = 0, state = {len 0, max_priority 1} */
int pb_tree_init(const pb_tree *t, void *stream);

/* HOST, synchronous, measurement runs only (profiles/per_phases.py): copies the phase marks of the priority-store kernels
 * (%globaltimer ns per slot, 0 = not reached; slot numbering in csrc/per_tree.cu) into out[0 .. n_out), clears them and
 * switches marking on (enable != 0) or off.  Marking is off by default and costs one cached load per mark when off. */
int pb_tree_trace(int enable, unsigned long long *out, int n_out);

/* the full level-ordered arrays a pointer-walking tree would hold (2*capacity floats each, node i has children 2i and
 * 2i+1, leaves at [capacity, 2*capacity); either may be NULL): parity tests and checkpoints, not the hot path */
int pb_tree_export(const pb_tree *t, float *sum_heap, float *min_heap, void *stream);

/* bulk load n post-pow fp32 leaves (rest padded with the identity) and rebuild
 * every internal node pairwise; sets len=min(n,size), seq=n.  Streaming kernel. */
int pb_tree_build(const pb_tree *t, const float *leaves, long long n, void *stream);

/* recompute state->p_sum / p_min = query(0, len) exactly as torchrl's interval
 * walk associates them (timestep_buffer.py:37 -> PrioritizedSampler.sample) */
int pb_tree_stats(const pb_tree *t, void *stream);

/* raw leaf write + ancestor recompute (both trees).  Duplicates: last wins,
 * like the sequential reference loop.  sorted!=0 promises idx is non-decreasing
 * (true for stratified samples; out-of-range entries such as the -1 padding rows of
 * a sharded sample may only form a suffix) and takes the one-launch path. */
int pb_tree_set_leaves(const pb_tree *t, long long n, const long long *idx,
                       const float *leaves, int sorted, void *stream);

/* TimestepBuffer.update_priority (prism/experience/timestep_buffer.py:53-54,
 * called from prism/learner.py:119-120): max_priority = max(max_priority, max p);
 * leaf = (p + eps)^alpha in fp32; ancestors; refreshes p_sum/p_min.
 * No device->host copy (the reference syncs here). */
int pb_tree_update_priority(const pb_tree *t, long long n, const long long *idx,
                            const float *priority, int sorted, void *stream);

/* TimestepBuffer.extend (timestep_buffer.py:32-33): the n slots starting at the
 * ring cursor get the default priority (max_priority+eps)^alpha; advances
 * seq/len.  idx_out (optional) receives the slots written. */
int pb_tree_extend(const pb_tree *t, long long n, long long *idx_out, void *stream);

/* scan_lower_bound on injected fp32 masses (parity entry point) */
int pb_tree_scan(const pb_tree *t, long long n, const float *mass, long long *idx_out,
                 void *stream);

/* PrioritizedSampler.sample (timestep_buffer.py:37): u are fp64 uniforms in [0,1); u == NULL draws them
 * on the device (Philox4x32-10 keyed by state->pad[3], counter = (k, state->pad[2]); the call number
 * advances by one per launch, so graph replays see fresh numbers and all ranks of a sharded buffer
 * that share a seed draw identical strata).
 * mode 0 iid: mass = p_sum*u (numpy uniform(0,p_sum)); mode 1 stratified:
 * mass = (k+u_k)/n * p_sum.  idx clamped to len-1; weight=(leaf/p_min)^-beta.
 * mass_out optional. */
int pb_tree_sample(const pb_tree *t, long long n, const double *u, int mode, float beta,
                   long long *idx_out, float *weight_out, float *mass_out, void *stream);

/* n_batches independent batches of `batch` samples in ONE launch, all against the current tree state ("batches in
 * flight": a learner that samples several batches before their priorities come back).  Sample k = b*batch + j is
 * stratum j of batch b (mode 1: mass = (j + u_k)/batch * p_sum); outputs are [n_batches][batch].  The matching
 * write-back is pb_tree_update_priority on the concatenation with sorted = 0 (later batches win, like n_batches
 * successive reference calls). */
int pb_tree_sample_batches(const pb_tree *t, long long n_batches, long long batch, const double *u, int mode,
                           float beta, long long *idx_out, float *weight_out, float *mass_out, void *stream);

/* Sharded global stratified sampling (new design, SURVEY 8e).  Every rank holds
 * one shard; all_state is the all-gathered array of the G shards' 64-byte state
 * blocks (one NCCL all-gather; only p_sum, p_min and len are read; G a power of two).  The G shard roots form the virtual top of one tree of
 * G*capacity leaves, summed pairwise in fp32.  Each rank evaluates all n_global
 * strata, keeps the contiguous run that lands in its shard and descends its own
 * tree with the residual mass.  Outputs are compacted to [0, owned_n);
 * state->owned_lo / owned_n report the run.  Rows >= owned_n get idx -1 (skipped by
 * pb_store_gather and pb_tree_update_priority) and weight 0. */
int pb_tree_sample_global(const pb_tree *t, int n_ranks, int rank,
                          const pb_per_state *all_state, long long n_global, const double *u,
                          float beta, long long *idx_out, float *weight_out,
                          long long *stratum_out, void *stream);

/* ------------------------------------------------------------------------- *
 * Transition ring (replaces the linked list of Timestep objects,
 * prism/experience/timestep.py:12-28, and ListStorage).
 * SoA; slot = seq % size; links hold sequence numbers and die on overwrite
 * exactly like the reference's weakrefs.
 * ------------------------------------------------------------------------- */
typedef struct pb_store {
    void      *obs;        /* [size][obs_elems] of obs_dtype            */
    void      *aux_obs;    /* [aux_size][obs_elems]: in-flight / truncated-final observations */
    int       *action;     /* [size] */
    float     *reward;     /* [size] */
    uint8_t   *done;       /* [size] */
    uint8_t   *trunc;      /* [size] */
    long long *slot_seq;   /* [size], -1 = empty */
    long long *next_link;  /* [size]: >=0 seq of successor; -1 none; <=-2 aux row -(v+2) */
    long long *prev_link;  /* [size]: >=0 seq of predecessor; -1 none */
    long long  size;
    long long  aux_size;
    int        obs_elems;  /* elements of ONE frame */
    int        obs_dtype;  /* 0 fp32, 1 uint8 */
    int        obs_scale;  /* uint8 only: 0 -> (float)v, 1 -> (float)v / 255.0f */
    int        frame_stack;
    int        n_step;
    int        pad;
    double     gamma;
} pb_store;

/* per-step flags handed to the host planner */
enum { PB_STEP_DONE = 1, PB_STEP_TRUNC = 2, PB_STEP_NO_NEXT = 4 };

/* one staged step: 64 bytes, filled on pinned host memory and copied to the device in one piece */
typedef struct pb_step_meta {
    long long seq;         /* planner: global sequence number (slot = seq % size)            */
    long long prev_link;   /* planner */
    long long next_link;   /* planner */
    long long aux_row;     /* planner: aux_obs row that receives next_obs[j], -1 = discard    */
    long long patch_slot;  /* planner: already-stored predecessor whose next_link is fixed up */
    long long patch_val;   /* planner */
    float     reward;      /* caller */
    int       action;      /* caller */
    uint8_t   done;        /* caller */
    uint8_t   trunc;       /* caller */
    uint8_t   pad[6];
} pb_step_meta;

/* HOST planner for TimestepBuffer.extend: turns n new steps (in arrival order, each tagged
 * with its collector stream) into slot/link values, following the link rules of
 * multiprocessing_experience_collection/collector_process_interface.py:146-173
 * (done -> no next; truncated -> next is the final observation, never stored; else prev/next
 * neighbours).  All arrays are HOST memory.
 *   stream_last_h[n_streams]  in/out: seq of the newest stored step of each stream, -1 none
 *   seq0                      seq of the first new step
 *   trunc_cursor_h            in/out: next free row of the truncated-obs pool
 *                             (rows [n_streams, aux_size) of aux_obs, used as a ring)
 *   trunc_owner_h[aux_size-n_streams] in/out: seq of the step owning each pool row (-1 free);
 *                             recycling a row whose owner is still stored returns PB_E_POOL
 *                             with no side effect (the caller grows the pool and retries)
 *   meta_h[n]                 out: the six planner fields of every step */
int pb_store_extend_plan(long long size, long long aux_size, int n_streams, long long n,
                         long long seq0, const int *stream_id_h, const uint8_t *flags_h,
                         long long *stream_last_h, long long *trunc_cursor_h,
                         long long *trunc_owner_h, pb_step_meta *meta_h);

/* HOST: fill a staging block and plan it in one call -- rows_h [2][n][row_bytes] <- obs_h, next_obs_h (n contiguous rows
 * of the store dtype each), the caller fields of meta_h <- action (int32 or int64: action_bytes 4 | 8) / reward / done / trunc, then pb_store_extend_plan
 * with flags = done * PB_STEP_DONE + trunc * PB_STEP_TRUNC.  On PB_E_POOL (or any error) the rows are left untouched. */
int pb_store_stage_block(long long size, long long aux_size, int n_streams, long long n, long long seq0,
                         long long row_bytes, const void *obs_h, const void *next_obs_h, const int *stream_id_h,
                         const void *action_h, int action_bytes, const float *reward_h, const uint8_t *done_h,
                         const uint8_t *trunc_h, void *rows_h, long long *stream_last_h, long long *trunc_cursor_h,
                         long long *trunc_owner_h, pb_step_meta *meta_h);

/* device scatter of n planned steps: obs rows -> ring, next_obs rows -> aux pool, metadata,
 * link patches.  obs/next_obs are device staging buffers [n][obs_elems] of the store dtype,
 * meta the device copy of the planned pb_step_meta array. */
int pb_store_scatter(const pb_store *s, long long n, const void *obs, const void *next_obs,
                     const pb_step_meta *meta, void *stream);
/* Same scatter for an ingest fused into a replayed CUDA graph: two staging blocks (A, B) with frozen addresses; the
 * block of this replay is chosen on the device by the parity of *replay_counter (even: A), which the call then
 * increments -- the host fills and copies the other block for the next replay meanwhile. */
int pb_store_scatter_dbuf(const pb_store *st, long long n, const void *obs_a, const void *next_obs_a,
                          const pb_step_meta *meta_a, const void *obs_b, const void *next_obs_b,
                          const pb_step_meta *meta_b, long long *replay_counter, void *stream);
/* dst[0..n) = (parity of *replay_counter + bias) ? src_b : src_a -- the per-iteration fp64 uniforms ride in the same
 * double-buffered staging block as the new steps and are picked by the same replay counter. */
int pb_select_copy_f64(double *dst, const double *src_a, const double *src_b, const long long *replay_counter,
                       long long bias, long long n, void *stream);

/* TimestepBuffer._timesteps_to_batch + _compute_n_step + _stack_obs_into
 * (prism/experience/timestep_buffer.py:79-257) fused: for each sampled slot walk
 * <= n_step links (fp64 return accumulation), resolve the successor observation,
 * and write the static batch with 128-bit coalesced row copies (uint8 widened
 * on the fly).  Rows with idx < 0 are skipped.
 *   obs_out/next_obs_out  [n][frame_stack][obs_elems] fp32
 *   ret_out [n] fp32, gamma_out [n] fp32, nonterm_out [n] u8 (torch.bool),
 *   action_out [n] int64 */
int pb_store_gather(const pb_store *s, long long n, const long long *idx, float *obs_out,
                    float *next_obs_out, float *ret_out, float *gamma_out,
                    uint8_t *nonterm_out, long long *action_out, void *stream);

/* n-step metadata only (parity entry point): same walk, no observation traffic */
int pb_store_nstep(const pb_store *s, long long n, const long long *idx, float *ret_out,
                   float *gamma_out, uint8_t *done_out, long long *last_out,
                   long long *succ_out, void *stream);

/* ------------------------------------------------------------------------- *
 * Agent-side fused kernels
 * ------------------------------------------------------------------------- */

/* IQNModel._embed_quantiles basis (prism/agents/models/iqn_model.py:89-92):
 * out[r][i] = cos(fl32(fl32(tau[r] * (i+1)) * pi)), i in [0, n_basis) */
int pb_iqn_cos_basis(long long n_rows, int n_basis, const float *tau, float *out, void *stream);

/* IQNModel.get_loss (prism/agents/models/iqn_model.py:110-201) from the three
 * quantile tables, fused with its own backward:
 *   z_cur   [T*B][A]  online Z(s, tau_i)   (quantile-major rows: r = i*B + b)
 *   tau     [T*B]
 *   z_next_online / z_next_target [Tp*B][A]  (same pointer when not double-Q)
 *   a* = argmax_a mean_j z_next_online; y_bj = R_b + gdn_b * z_next_target[j,b,a*]
 *   delta = y_bj - theta_bi; Huber(kappa); rho = |tau_bi - 1{delta<0}| * L / kappa
 *   loss_b = loss_weight * mean_j sum_i rho
 *   nonterminal (optional, torch.bool bytes): the bootstrap factor is gdn_b * nonterminal_b, i.e.
 *   gdn = gamma^k alone (composite_model.py:110 fused in); NULL = gdn already holds the product.
 * grad_z_cur [T*B][A] = grad_scale * row_weight[b] * d loss_b / d z_cur (zero outside the
 * taken action; row_weight NULL = 1).  With row_weight = PER weights and grad_scale = 1/B
 * this is d mean(loss*w) / d z_cur (prism/agents/agent.py:58-60). */
int pb_iqn_qh_loss(int B, int T, int Tp, int A, const float *z_cur, const float *tau,
                   const float *z_next_online, const float *z_next_target,
                   const long long *action, const float *ret, const float *gdn,
                   const uint8_t *nonterminal, float kappa, float loss_weight,
                   const float *row_weight, float grad_scale, float *loss_out, float *grad_z_cur,
                   void *stream);

/* QEnsemble.get_loss (prism/agents/models/q_ensemble.py:50-92) without the
 * Theil term: tables are head-major [K][B][A].
 *   a*_k = argmax_a q_next_online[k,b,:]; y_k = R + gdn * q_next_target[k,b,a*_k]
 *   loss_b = loss_weight * mean_k (q_cur[k,b,a_b] - y_k)^2;  grad_q_cur [K][B][A] */
int pb_ens_q_loss(int B, int A, int K, const float *q_cur, const float *q_next_online,
                  const float *q_next_target, const long long *action, const float *ret,
                  const float *gdn, const uint8_t *nonterminal, float loss_weight,
                  const float *row_weight, float grad_scale, float *loss_out, float *grad_q_cur,
                  void *stream);
/* pb_ens_q_loss whose LAST CTA also does pb_loss_combine (one launch less on the step's critical path):
 * *total_out = mean_b(dist_b * w_b) + mean_b(q'_b * w_b), q'_b = q_scale * (loss_b - *q_offset); td_out as pb_loss_combine.
 * dist (B per-row distributional losses, may be NULL) must be complete in stream order.  ticket: one device word,
 * zero between calls. */
int pb_ens_q_loss_total(int B, int A, int K, const float *q_cur, const float *q_next_online, const float *q_next_target,
                        const long long *action, const float *ret, const float *gdn, const uint8_t *nonterminal,
                        float loss_weight, const float *row_weight, float grad_scale, float *loss_out, float *grad_q_cur,
                        const float *dist, float q_scale, const float *q_offset, float *total_out, float *td_out,
                        unsigned int *ticket, void *stream);

/* IDSActionSelector.generate_action_probs + select_action
 * (prism/agents/action_selectors.py:125-176), deterministic branch.
 *   q [K][N][A] head-major ensemble values, z [Nq][N][A] quantile values.
 *   action_out [N] int64; scores_out optional [N][A]. Reproduces the reference's
 *   std-for-variance / sqrt(std)-for-std naming quirk. */
int pb_ids_select(int N, int A, int K, int Nq, const float *q, const float *z, float lambda,
                  float eps, float rho_lower_bound, long long *action_out, float *scores_out,
                  void *stream);

/* GreedyActionSelector (action_selectors.py:70-82): argmax_a mean_k q */
int pb_greedy_select(int N, int A, int K, const float *q, long long *action_out, void *stream);

/* Agent._update_without_cuda_graph tail (prism/agents/agent.py:71-74):
 * clip_grad_norm_(max_norm) + Adam (torch.optim.Adam semantics, factory/agent_factory.py:44-47)
 * over ONE flat fp32 parameter arena -- two launches instead of ~10 per parameter tensor.
 *
 * pb_pack_grads: gather autograd's per-parameter gradients into the flat arena, multiplied by
 *   `scale` (1/world_size under data parallelism), folding in the per-CTA sum of squares.
 *   table (device) = n_tensors x {grad pointer (0 = no grad), arena offset, numel} as int64.
 *   step_count (device int64, optional) is incremented.  n_partials_out_h (host) receives the
 *   number of partial sums written to partial_scratch (>= 4096 floats).
 * pb_grad_sumsq: same partial sums for a gradient that is already flat (after an all-reduce).
 * pb_adam_clip_apply: total_norm = sqrt(sum partials); coef = min(1, max_norm/(norm+1e-6));
 *   g *= coef; Adam with bias correction from *step_count.  norm_out (optional, device
 *   float[2]) = {total_norm, coef}.
 * pb_adam_clip_step = pb_grad_sumsq + pb_adam_clip_apply. */
#define PB_ADAM_MAX_PARTIALS 4096
/* pb_pack_grads_parity: the same gather into one half of a double-buffered arena: destination = flat +
 * (*epoch & 1) * stride, epoch a device counter (the peer exchange's count of completed state gathers, csrc/peer.cu). */
int pb_pack_grads_parity(int n_tensors, const long long *table, float scale, float *flat,
                         const unsigned long long *epoch, long long stride, float *partial_scratch,
                         long long *step_count, int *n_partials_out_h, void *stream);
int pb_pack_grads(int n_tensors, const long long *table, float scale, float *flat,
                  float *partial_scratch, long long *step_count, int *n_partials_out_h,
                  void *stream);
int pb_grad_sumsq(long long n, const float *grad, float *partial_scratch, long long *step_count,
                  int *n_partials_out_h, void *stream);
int pb_adam_clip_apply(long long n, float *param, const float *grad, float *exp_avg,
                       float *exp_avg_sq, const long long *step_count, float lr, float beta1,
                       float beta2, float adam_eps, float max_grad_norm,
                       const float *partial_scratch, int n_partials, float *norm_out,
                       void *stream);
/* Small arenas (n <= pb_adam_fused_max_n(), at most 64 tensors): pb_pack_grads + pb_adam_clip_apply as ONE launch -- the
 * gathered gradient stays in registers between the norm (the CTAs of the grid meet at a counter) and the Adam update;
 * it is also written to `grad` (the flat arena).  table as for pb_pack_grads, tensors in arena order.
 * partial_scratch: 4096 floats, the last 4 zero between calls.  PB_E_UNSUPPORTED: use the two-launch path. */
long long pb_adam_fused_max_n(void);
int pb_adam_fused_step(int n_tensors, const long long *table, float scale, long long n, float *param, float *grad,
                       float *exp_avg, float *exp_avg_sq, long long *step_count, float lr, float beta1, float beta2,
                       float adam_eps, float max_grad_norm, float *partial_scratch, float *norm_out, void *stream);
int pb_adam_clip_step(long long n, float *param, const float *grad, float *exp_avg, float *exp_avg_sq,
                      long long *step_count, float lr, float beta1, float beta2, float adam_eps,
                      float max_grad_norm, float *norm_out, float *partial_scratch, void *stream);

/* MinAtarModel embedding (prism/agents/models/minatar_cnn_model.py:13-18, 41-44) in one launch:
 * x (B, H, W, C) channels-last fp32 -> conv3x3 stride 1 no padding (weight (OC, C, 3, 3), torch layout)
 * + bias + ReLU -> out (B, OC*(H-2)*(W-2)) in NCHW-flatten order.
 * Backward (observations need no gradient): dw (OC, C, 3, 3), db (OC) from dout masked by out > 0;
 * partial_scratch holds pb_conv3x3_relu_bwd_groups(B) * (OC*C*9 + OC) floats.
 * pb_conv3x3_relu_supported: 1 when both entries accept an H x W x C frame with OC filters (at most 2048 weights +
 * biases, 4096 frame floats, 6272 output floats per image, 48 KB of shared memory per CTA), else 0: run the
 * convolution elsewhere.  The backward takes the tensor cores for OC == 16, an output plane that is a multiple of 8
 * and at most 64, and 4 <= C <= 10; every other accepted shape takes the FMA kernel. */
int pb_conv3x3_relu_supported(int H, int W, int C, int OC);
int pb_conv3x3_relu_fwd(int B, int H, int W, int C, int OC, const float *x, const float *w,
                        const float *bias, float *out, void *stream);
int pb_conv3x3_relu_bwd_groups(int B);
int pb_conv3x3_relu_bwd(int B, int H, int W, int C, int OC, const float *x, const float *out,
                        const float *dout, float *partial_scratch, float *dw, float *db,
                        void *stream);

/* Dense layers of the Q heads / IQN MLP (nn.Linear inside nn.Sequential in the reference:
 * prism/agents/models/ffnn_model.py:61-76, q_ensemble.py:26-48, iqn_model.py:30-46), one launch
 * each, batched over K heads, fp32 FFMA, split-K across a thread-block cluster (DSMEM reduce).
 *   fwd:        Y[k] (M x N) = act(X[k] (M x J) . W[k]^T (N x J) + b[k]);  act 0 none / 1 ReLU;
 *               x_head_stride = 0 shares one X between all heads
 *   bwd_input:  dX[k] (M x J) = (dY[k] . [Ymask[k] > 0]) . W[k];  Ymask NULL = no activation;
 *               sum_heads != 0: one dX = sum over heads (X was shared)
 *   bwd_weight: dW[k] (N x J) = (dY[k] . mask)^T . X[k];  db[k] (N) = column sums (optional) */
int pb_linear_fwd(int K, int M, int N, int J, const float *X, long long x_head_stride, const float *W,
                  const float *b, int act, float *Y, void *stream);
int pb_linear_bwd_input(int K, int M, int N, int J, const float *dY, const float *Ymask, const float *W,
                        int sum_heads, float *dX, void *stream);
int pb_linear_bwd_weight(int K, int M, int N, int J, const float *dY, const float *Ymask, const float *X,
                         long long x_head_stride, float *dW, float *db, void *stream);
/* Measurement runs only (synchronous): phase marks (%globaltimer, ns) of the cluster split-K kernel's launches since the
 * last call -- out[0] earliest CTA start, out[1..6] latest CTA past: first chunk staged, K loop, partial tile written,
 * cluster barrier, split-K sum + epilogue, exit barrier -- then reset, and marking switched on / off. */
int pb_gemm_trace(int enable, unsigned long long *out, int n_out);

/* Dense layers on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM, operands
 * staged by TMA; csrc/tc_gemm.cu).  Every fp32 operand is split on the fly into TF32 hi + lo parts and each
 * product issued as lo.hi + hi.lo + hi.hi (3xTF32), which keeps fp32-level accuracy (parity bar 1e-4) at
 * tensor-core speed.  Replaces the nn.Linear GEMMs of the (T*B)-row IQN layers and of the K-head ensemble
 * (iqn_model.py:30-46,89-93; ffnn_model.py:61-76; q_ensemble.py:26-48) and their autograd transposes.
 *
 *   C[b] (M x N, row stride ldc) = act( sum_k A[b](m,k) B[b](n,k) + bias[b](n) ),   b < batch
 *
 * a_major / b_major: 0 = the operand is stored row-major [M or N][K] (row stride lda/ldb); 1 = it is stored
 * row-major [K][M or N] -- the transposed view the backward GEMMs need (dX = dZ W: b_major 1; dW = dZ^T X:
 * both 1).  a_bs / b_bs: batch strides in floats (0 = shared by every batch).  kbatches > 1 (batch must be 1):
 * the K loop also runs over kbatches operand batches, i.e. C = sum_h A[h] B[h]^T (input gradient of a layer
 * whose input is shared by all heads).  workspace: optional scratch for split-K partials (the kernel picks the
 * split so that batch*splits*M*N <= workspace_floats).  split_mode 0: hi = the raw fp32 word (the tensor core
 * reads its upper 19 bits); 1: hi = cvt.rna.tf32.  Requirements: 16-byte aligned A/B, lda/ldb/a_bs/b_bs % 4 == 0
 * (PB_E_UNSUPPORTED / PB_E_ARG otherwise).  act: 0 none, 1 ReLU.  mul (optional): after bias and activation
 * every output is multiplied by mul[(m % mul_rows) * ld_mul + n] -- the IQN product phi(tau) (.) x with the
 * state embedding x broadcast over the quantile-major rows (iqn_model.py:70-71), fused into the phi GEMM. */
int pb_tc_gemm_supported(int M, int N, int K, long long lda, long long ldb, long long ldc);
int pb_tc_gemm(int batch, int kbatches, int M, int N, int K,
               const float *A, int a_major, long long lda, long long a_bs,
               const float *B, int b_major, long long ldb, long long b_bs,
               const float *bias, long long bias_bs, int act,
               const float *mul, int mul_rows, long long ld_mul,
               float *C, long long ldc, long long c_bs,
               float *workspace, long long workspace_floats, int split_mode, void *stream);
/* nn.Linear forward through pb_tc_gemm: Y[k] (M x N) = act(X[k] (M x J) W[k]^T + b[k]), J % 4 == 0. */
int pb_linear_fwd_tc_supported(int M, int N, int J);
int pb_linear_fwd_tc(int K, int M, int N, int J, const float *X, long long x_head_stride, const float *W,
                     const float *b, int act, float *Y, void *stream);

/* Backward of the IQN product h[q,b,:] = relu(pre[q,b,:]) (.) x[b,:]  (iqn_model.py:70-71, 89-93; rows are
 * quantile-major r = q*B + b) in one pass: dpre = dh * x * [phi > 0], dx[b] = sum_q dh * phi,
 * dbias_partial[b] = sum_q dpre (the bias gradient is its column sum over b).  F % 4 == 0, 16-byte aligned
 * pointers; dx may be NULL. */
int pb_iqn_phi_bwd(int n, int B, int F, const float *dh, const float *phi, const float *x, float *dpre, float *dx,
                   float *dbias_partial, void *stream);

/* ---- data-parallel exchange over NVLink / NVSwitch peer memory (csrc/peer.cu; SURVEY 8e) -----------------------
 * Replaces, for ranks on one box, the two collectives of the sharded learner step: the all-gather of the 64-byte
 * shard state blocks and the all-reduce of the flat gradient arena followed by clip + Adam (agent.py:73-74).
 * Every rank allocates one block with pb_peer_alloc, exports it (pb_peer_export, a 64-byte CUDA IPC handle that
 * the host side exchanges any way it likes), opens the other ranks' blocks (pb_peer_open) and fills a
 * pb_peer_group with the per-rank addresses.  All calls are stream-ordered, graph-capturable and must be issued
 * by every rank in the same order (the barriers are epoch counters in peer memory). */
#define PB_PEER_MAX 8
typedef struct pb_peer_group {
    int world, rank;
    float *grad[PB_PEER_MAX];                 /* every rank's flat gradient arena (n floats)                         */
    float *reduced[PB_PEER_MAX];              /* every rank's reduced-gradient buffer (n floats; rank r fills slice r) */
    unsigned long long *flags[PB_PEER_MAX];   /* every rank's signal pad, 3 channels x PB_PEER_MAX: [dst][ch][src] = epoch */
    double *norm_parts[PB_PEER_MAX];          /* every rank's [PB_PEER_MAX] slice sums of squares                    */
    unsigned char *state[PB_PEER_MAX];        /* every rank's gathered shard states, 4 slots x [PB_PEER_MAX][64]: 0-1 the
                                                 parity slots of pb_peer_state_allgather, 2-3 those of pb_peer_state_put */
    unsigned long long *epoch;                /* local counters, one per channel (0 barrier, 1 gradient exchange /
                                                 state gather, 2 state puts)                                          */
    unsigned int *status;                     /* local status word: bit ch set = a wait on channel ch timed out (may be NULL) */
    unsigned long long timeout_ns;            /* bound of every flag wait; 0 = wait forever                          */
    long long grad_stride;                    /* floats between the two halves of the double-buffered gradient arena
                                                 (0: single buffer); the half in use = parity of completed state gathers */
} pb_peer_group;
int pb_peer_alloc(long long bytes, void **ptr);            /* cudaMalloc + zero fill; blocking                      */
int pb_peer_free(void *ptr);
int pb_optimizer_preload(void);                            /* same for pack_grads / grad_sumsq / adam_clip          */
int pb_peer_preload(void);                                  /* load the exchange kernels now (blocking)              */
int pb_peer_export(const void *ptr, void *handle64);
int pb_peer_open(const void *handle64, void **ptr);        /* maps a peer block, enabling peer access               */
int pb_peer_close(void *ptr);
int pb_peer_barrier(const pb_peer_group *g, void *stream);
/* state64: this rank's 64-byte tree state block (pb_tree state).  On return (stream order) all_state_out (local,
 * world x 64 bytes) holds every rank's block. */
int pb_peer_state_allgather(const pb_peer_group *g, const void *state64, void *all_state_out, void *stream);
long long pb_peer_slice(long long n, int world);           /* floats per rank slice (multiple of 4)                 */
/* reduced[rank][slice rank] = sum over ranks (rank order) of grad[p][slice]; publishes the slice's sum of squares
 * to every rank; increments *step_count (may be NULL).  Needs a pb_peer_barrier between the writers of grad and
 * this call, and another one before pb_peer_adam.  partial_scratch: 4096 floats.  n % 4 == 0. */
int pb_peer_reduce_scatter(const pb_peer_group *g, long long n, float *partial_scratch, long long *step_count, void *stream);
/* One-shot all-reduce for small arenas: reduced[rank] = sum over ranks (rank order) of grad[p], all n floats pulled
 * by every rank, + per-block sums of squares in partial_scratch (*n_partials_out_h of them) for pb_adam_clip_apply on
 * (param, reduced[rank]).  One pb_peer_barrier before it, none after. */
int pb_peer_pull_sum(const pb_peer_group *g, long long n, float *partial_scratch, long long *step_count,
                     int *n_partials_out_h, void *stream);
/* clip_grad_norm_(max_grad_norm) + Adam over the local replica, reading the reduced gradient slice by slice from its
 * owner rank.  grad_out (optional): receives the full reduced gradient. */
int pb_peer_adam(const pb_peer_group *g, long long n, float *param, float *exp_avg, float *exp_avg_sq,
                 const long long *step_count, float lr, float beta1, float beta2, float adam_eps, float max_grad_norm,
                 float *norm_out, float *grad_out, void *stream);
/* Small arenas (n <= pb_peer_allreduce_adam_max_n()), ONE launch for everything after the pack: handshake on channel 1
 * (every CTA waits on the local pad), pull + sum of every rank's gradient in rank order into registers, global norm
 * (the CTAs of the grid meet at a counter), clip + Adam -- agent.py:73-74 on W replicas.  Advances *step_count and
 * the channel-1 epoch (the parity of the double-buffered gradient arena); reduced[rank] receives the summed gradient.
 * partial_scratch: 4096 floats, the last 4 zero between calls. */
long long pb_peer_allreduce_adam_max_n(void);
int pb_peer_allreduce_adam(const pb_peer_group *g, long long n, float *param, float *exp_avg, float *exp_avg_sq,
                           long long *step_count, float lr, float beta1, float beta2, float adam_eps, float max_grad_norm,
                           float *partial_scratch, float *norm_out, void *stream);
/* HOST, synchronous, measurement runs only: phase marks of pb_peer_allreduce_adam's kernel (%globaltimer ns: 0 CTA 0
 * starts, 1 handshake done, 2 pulled + summed, 3 the CTAs met, 4 Adam applied; latest CTA each), cleared on read. */
int pb_peer_trace(int enable, unsigned long long *out, int n_out);
/* Non-blocking half of the shard-state exchange (channel 2): this rank's 64-byte state block goes into slot
 * 2 + (count & 1) of every rank's state area and this rank's flag is raised there.  The matching wait is inside
 * pb_tree_sample_global_peer.  The state area holds 4 slots of PB_PEER_MAX x 64 bytes (0-1: pb_peer_state_allgather). */
int pb_peer_state_put(const pb_peer_group *g, const void *state64, void *stream);
/* pb_tree_sample_global on the states of the latest pb_peer_state_put exchange: every CTA first waits (bounded by
 * g->timeout_ns; bit 2 of *g->status on a timeout) until every rank's put has landed in the local slot. */
int pb_tree_sample_global_peer(const pb_tree *t, const pb_peer_group *g, long long n_global, const double *u, float beta,
                               long long *idx_out, float *weight_out, long long *stratum_out, void *stream);

/* ------------------------------------------------------------------------- *
 * Uniform replay (the reference's default, use_per = False: torchrl's uniform ReplayBuffer).
 * The whole sampler is one 64-byte pb_per_state block; only len, seq, status, owned_lo / owned_n and pad[1..3]
 * (rng ticket, call number, seed -- as for pb_tree_sample) are used, so pb_peer_state_put carries it unchanged.
 * Every entry returns PB_E_ARG for a NULL state before it launches anything.
 * ------------------------------------------------------------------------- */
/* seq = the given value, len = min(seq, size), seed = pad[3], call number 0, status 0 (one single-thread launch) */
int pb_uniform_init(pb_per_state *state, long long size, long long seq, int seed, void *stream);
/* seq += n, len = min(seq, size): one single-thread launch, capturable (the ring's fused ingest) */
int pb_uniform_extend(pb_per_state *state, long long size, long long n, void *stream);
/* mode 0 iid: idx = (long long)(u_k * len); mode 1 stratified: idx = (long long)((k + u_k) / n * len) -- fp64,
 * round-to-nearest, in that order; clamped to len - 1; weight 1.  u == NULL draws u_k on the device (Philox4x32-10,
 * key pad[3], counter (k, pad[2]); the last CTA advances the call number).  len == 0 sets PB_ST_EMPTY. */
int pb_uniform_sample(pb_per_state *state, long long n, const double *u, int mode, long long *idx_out,
                      float *weight_out, void *stream);
/* Global stratified uniform sampling over the concatenation of n_ranks shards (all_state: their gathered state
 * blocks, only len is read): total = sum of len_r, g_k = (long long)((k + u_k) / n_global * total) clamped to
 * total - 1, owner from the prefix sums of len_r, local index g_k - prefix[rank].  This rank's strata form one
 * contiguous run; outputs are compacted to [0, owned_n) and the run is written to owned_lo / owned_n.  Rows past it
 * get idx -1, weight 0, stratum -1.  stratum_out optional. */
int pb_uniform_sample_global(pb_per_state *state, int n_ranks, int rank, const pb_per_state *all_state,
                             long long n_global, const double *u, long long *idx_out, float *weight_out,
                             long long *stratum_out, void *stream);
/* pb_uniform_sample_global on the states of the latest pb_peer_state_put exchange (bounded wait as for
 * pb_tree_sample_global_peer: bit 2 of *g->status on a timeout). */
int pb_uniform_sample_global_peer(pb_per_state *state, const pb_peer_group *g, long long n_global, const double *u,
                                  long long *idx_out, float *weight_out, long long *stratum_out, void *stream);

/* LayerNorm over the last dimension of a (rows x F) fp32 matrix, forward and backward (csrc/ln.cu), for the
 * (T*B)-row IQN activations (nn.LayerNorm in ffnn_model.py:17-18, iqn_model.py:42-46).  F % 4 == 0, F <= 4096,
 * 16-byte aligned pointers.  gamma / beta may be NULL (no affine); mean_out / rstd_out may be NULL (no backward).
 * Backward makes ONE pass over (x, dy): dx plus per-CTA partial column sums, then a column reduction;
 * partials = scratch of 2 * pb_layer_norm_bwd_blocks(rows, F) * F floats; dgamma / dbeta may be NULL. */
int pb_layer_norm_supported(long long rows, int F);
int pb_layer_norm_bwd_blocks(long long rows, int F);
int pb_layer_norm_fwd(long long rows, int F, float eps, const float *x, const float *gamma, const float *beta, float *y,
                      float *mean_out, float *rstd_out, void *stream);
int pb_layer_norm_bwd(long long rows, int F, const float *x, const float *dy, const float *gamma, const float *mean,
                      const float *rstd, float *dx, float *dgamma, float *dbeta, float *partials, void *stream);

/* ReLU backward + bias gradient of a dense layer (heads stacked (heads, rows, N) matrices) in one pass:
 * dz = dy * [y > 0] (y NULL: no activation, dz untouched) and dbias[h] = column sums of dz -- the autograd glue
 * around the tensor-core GEMMs (nn.Linear + ReLU backward, ffnn_model.py:61-76).  N % 4 == 0; partials =
 * heads * pb_relu_bwd_bias_strips(rows) * N floats of scratch. */
int pb_relu_bwd_bias_strips(long long rows);
int pb_relu_bwd_bias(int heads, long long rows, int N, const float *dy, const float *y, float *dz, float *dbias,
                     float *partials, void *stream);

/* Theil index of the K heads' parameter L2 norms (q_ensemble.py:86-92) over stacked parameter tensors (K, ...), and
 * its gradient.  table (device): per tensor {address, elements per head, offset of its gradient in `out`} as int64
 * triples.  forward: *theil_out = mean_k r_k log r_k, coef[k] = d T / d theta_k divided by theta_k; chunks = blocks per
 * (tensor, head) from pb_theil_chunks(largest per-head size); partial = scratch of n_tensors * K * chunks floats;
 * K <= 64.  backward: out = *upstream * coef[k] * theta. */
int pb_theil_chunks(long long max_per_head);
int pb_theil_fwd(int n_tensors, int K, int chunks, const long long *table, float *partial, float *theil_out, float *coef,
                 void *stream);
int pb_theil_bwd(int n_tensors, int K, int chunks, const long long *table, const float *coef, const float *upstream,
                 float *out, void *stream);

/* total_loss = mean_b(dist*w) + mean_b(q'*w);  td_b = 0.5*dist + 0.5*q' | dist | |q'|
 * (composite_model.py:135-142, agent.py:58-64) with q' = q_scale * (q - *q_offset)
 * (q_ensemble.py:92: q_loss_weight * (q_loss - theil * coef); q_offset NULL = 0).
 * dist or q may be NULL; w NULL = 1. */
int pb_loss_combine(int B, const float *dist, const float *q, const float *w, float q_scale,
                    const float *q_offset, float *total_out, float *td_out, void *stream);

/* Timeline mark for measurement runs: *dst (device) = %globaltimer (ns) when the stream -- or the graph branch the call
 * was captured on -- reaches this point.  One single-thread launch; the product path never calls it unless a trace was
 * asked for (LearnerStep.enable_trace), since nsys is not available on the measurement boxes. */
int pb_stamp_time(unsigned long long *dst, void *stream);

/* ---- wire codec of the remote-actor transport (SURVEY 8f-4).  HOST functions: plain host pointers, no stream, no
 * device work.  They replace the per-element Python walks of the reference's Redis path:
 *   msgpack array of numbers -> float64   prism/async_components/compression_methods.py:72-80 (msgpack.unpackb)
 *   Timestep records -> offsets           prism/experience/timestep.py:103-187 (Timestep.deserialize)
 *   tensor memory -> msgpack numbers      prism/async_components/async_experience_buffer.py:90-96 (tensor.tolist())
 * pb_wire_unpack_numbers: buf holds exactly ONE msgpack array of ints / floats / bools; *n_out = its length; out NULL
 *   = validate and count only; PB_E_UNSUPPORTED for any other element type (nil, str, bin, containers).
 * pb_wire_array_header: msgpack array header of n elements (out >= 5 bytes).
 * pb_wire_pack_numbers: n elements (dtype 0 float32, 1 float64, 2 int64, 3 bool bytes) as msgpack encodes the
 *   corresponding Python list (floats as float64, ints in their shortest form); cap >= 9 * n.
 * pb_wire_index_timesteps: flat = the decoded numbers of a block of serialized Timesteps (timestep.py:30-101); per
 *   record 12 int64 columns: id | obs offset (-1 none), values, shape offset, shape values | truncated successor id
 *   (-1313 none) and the same four columns of its observation | offset of the 12 scalar fields (reward .. next id) |
 *   offset one past the record.  rec NULL = count only.  PB_E_ARG on a malformed block. */
int pb_wire_unpack_numbers(const unsigned char *buf, long long len, double *out, long long cap, long long *n_out);
int pb_wire_array_header(long long n, unsigned char *out, long long *written);
int pb_wire_pack_numbers(const void *src, int dtype, long long n, unsigned char *out, long long cap, long long *written);
int pb_wire_index_timesteps(const double *flat, long long n, long long max_records, long long *rec, long long *n_rec);

/* ------------------------------------------------------------------------- *
 * Grouped LayerNorm (csrc/ln.cu): `groups` affine pairs, gamma / beta (groups, F).  Output row r of
 * groups * rows_per_group rows normalises input row r % x_rows with the pair r / rows_per_group.  K ensemble heads on
 * one shared embedding (prism/agents/models/q_ensemble.py:26-48: every head starts with its own LayerNorm):
 * groups = K, x_rows = rows_per_group = B.  Backward: dx per OUTPUT row (sum it over the heads with pb_sum_heads
 * when the input is shared); partials = 2 * groups * pb_layer_norm_grouped_bwd_blocks() * F floats of scratch.
 * ------------------------------------------------------------------------- */
int pb_layer_norm_grouped_fwd(int groups, long long rows_per_group, long long x_rows, int F, float eps, const float *x,
                              const float *gamma, const float *beta, float *y, float *mean_out, float *rstd_out,
                              void *stream);
int pb_layer_norm_grouped_bwd_blocks(int groups, long long rows_per_group, int F);
int pb_layer_norm_grouped_bwd(int groups, long long rows_per_group, long long x_rows, int F, const float *x,
                              const float *dy, const float *gamma, const float *mean, const float *rstd, float *dx,
                              float *dgamma, float *dbeta, float *partials, void *stream);

/* ------------------------------------------------------------------------- *
 * Narrow dense layer (csrc/narrow.cu): y (M x N) = x (M x J) . W^T (N x J) + bias with N <= 32 outputs -- the
 * n_actions-wide output layer of the IQN head on (T*B) rows (prism/agents/models/iqn_model.py:42-46, autograd of
 * nn.Linear) and of the K ensemble heads (q_ensemble.py:26-48), batched over K heads: x (K, M, J) with head stride
 * x_head_stride floats (0 = the heads share one (M, J) input), W (K, N, J), bias (K, N), y / dy (K, M, N), dx (K, M, J).
 * One streaming pass over x forward; backward reads x once, writes dx once, and combines per-CTA partials of dW / db in a
 * fixed order.  partials: K * pb_narrow_linear_bwd_blocks(M) * (N * J + N) floats.
 * ------------------------------------------------------------------------- */
int pb_narrow_linear_supported(long long M, int N, int J);
int pb_narrow_linear_bwd_blocks(long long M);
int pb_narrow_linear_fwd(int K, long long M, int N, int J, const float *x, long long x_head_stride, const float *w,
                         const float *bias, float *y, void *stream);
int pb_narrow_linear_bwd(int K, long long M, int N, int J, const float *x, long long x_head_stride, const float *w,
                         const float *dy, float *dx, float *dW, float *db, float *partials, void *stream);
/* pb_narrow_linear_bwd with partials given and dW = db = NULL writes the per-CTA partial sums only; this finishes them
 * (dW / db optional) on any stream ordered after that call -- the weight-gradient branch of the learner step graph. */
int pb_narrow_linear_bwd_reduce(int K, long long M, int N, int J, const float *partials, float *dW, float *db, void *stream);

/* out[i] = sum_k in[k][i], i < n (n % 4 == 0): gradients of an input shared by K heads (q_ensemble.py:44-48) */
int pb_sum_heads(int K, long long n, const float *in, float *out, void *stream);

/* IQN quantile draw + cosine basis in one launch (prism/agents/models/iqn_model.py:64-66, 89-92): tau_out (n_rows)
 * ~ U[0,1) from Philox4x32-10 keyed by rng[0] with counter (row, rng[1]); out (n_rows, n_basis) = cos(pi i tau).
 * rng: device long long[4] = {seed, call number, ticket, unused}; the call number advances once per launch, so a
 * replayed CUDA graph draws fresh quantiles. */
int pb_iqn_draw_cos_basis(long long n_rows, int n_basis, long long *rng, float *tau_out, float *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PRISM_B200_H */
