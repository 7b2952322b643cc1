// store.cu -- device-resident transition ring: ingest scatter, n-step assembly and the
// fused batch gather (sm_100a).
//
// Replaces the reference's linked list of Python Timestep objects
// (prism/experience/timestep.py:12-28, linked by
// multiprocessing_experience_collection/collector_process_interface.py:146-173) and the
// per-row Python loop of TimestepBuffer._timesteps_to_batch / _compute_n_step /
// _stack_obs_into (prism/experience/timestep_buffer.py:79-257).
//
// Layout in HBM: struct-of-arrays ring, slot = seq % size.  Links are sequence numbers,
// alive iff slot_seq[link % size] == link -- the weakref-dies-on-overwrite rule without
// any invalidation pass.  Each observation frame is stored once (fp32 or uint8); frame
// stacks and n-step successors are resolved at gather time.  In-flight successors and
// truncated final observations live in a small aux pool (never sampled).
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include <math.h>

namespace {

using namespace pb;

constexpr int MAX_NSTEP = 16;

struct StoreView {
    const uint8_t *obs, *aux;
    uint8_t *obs_w, *aux_w;
    int *action;
    float *reward;
    uint8_t *done, *trunc;
    long long *slot_seq, *next_link, *prev_link;
    long long size, aux_size;
    long long row_bytes;
    int obs_elems, dtype, scale, fs, n_step;
    double gammas[MAX_NSTEP + 1];
};

int make_store(const pb_store *s, StoreView *v)
{
    if (!s || !s->obs || !s->action || !s->reward || !s->done || !s->trunc || !s->slot_seq || !s->next_link ||
        !s->prev_link)
        return PB_E_ARG;
    if (s->size <= 0 || s->obs_elems <= 0 || s->frame_stack < 1 || s->n_step < 1 || s->aux_size < 0)
        return PB_E_ARG;
    if (s->n_step > MAX_NSTEP || (s->obs_dtype != 0 && s->obs_dtype != 1)) return PB_E_UNSUPPORTED;
    if (s->aux_size > 0 && !s->aux_obs) return PB_E_ARG;
    v->obs = (const uint8_t *)s->obs; v->aux = (const uint8_t *)s->aux_obs;
    v->obs_w = (uint8_t *)s->obs; v->aux_w = (uint8_t *)s->aux_obs;
    v->action = s->action; v->reward = s->reward; v->done = s->done; v->trunc = s->trunc;
    v->slot_seq = s->slot_seq; v->next_link = s->next_link; v->prev_link = s->prev_link;
    v->size = s->size; v->aux_size = s->aux_size;
    v->obs_elems = s->obs_elems; v->dtype = s->obs_dtype; v->scale = s->obs_scale;
    v->fs = s->frame_stack; v->n_step = s->n_step;
    v->row_bytes = (long long)s->obs_elems * (s->obs_dtype == 0 ? 4 : 1);
    // python: self.gammas = [gamma ** i for i in range(n_step + 1)]  (timestep_buffer.py:17)
    for (int i = 0; i <= s->n_step; ++i) v->gammas[i] = pow(s->gamma, (double)i);
    return PB_OK;
}

// ---- ingest ------------------------------------------------------------------------
__device__ __forceinline__ void copy_row_bytes(uint8_t *dst, const uint8_t *src, long long bytes)
{
    if ((bytes & 15) == 0 && ((((uintptr_t)dst) | ((uintptr_t)src)) & 15) == 0) {
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        for (long long i = threadIdx.x; i < (bytes >> 4); i += blockDim.x) stg_stream(d4 + i, ldg_stream(s4 + i));
    } else {
        for (long long i = threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
    }
}

__global__ void __launch_bounds__(128) store_scatter_kernel(StoreView s, long long n, const uint8_t *obs,
                                                            const uint8_t *next_obs, const pb_step_meta *meta)
{
    const long long j = blockIdx.x;
    const pb_step_meta m = meta[j];
    const long long slot = m.seq % s.size;
    if (blockIdx.y == 0) {
        copy_row_bytes(s.obs_w + slot * s.row_bytes, obs + j * s.row_bytes, s.row_bytes);
        if (threadIdx.x == 0) {
            s.action[slot] = m.action;
            s.reward[slot] = m.reward;
            s.done[slot] = m.done;
            s.trunc[slot] = m.trunc;
            s.slot_seq[slot] = m.seq;
            s.prev_link[slot] = m.prev_link;
            s.next_link[slot] = m.next_link;
            if (m.patch_slot >= 0) s.next_link[m.patch_slot] = m.patch_val;
        }
    } else {
        const long long row = m.aux_row;
        if (row >= 0 && row < s.aux_size && next_obs)
            copy_row_bytes(s.aux_w + row * s.row_bytes, next_obs + j * s.row_bytes, s.row_bytes);
    }
}

// Double-buffered variant for an ingest that is fused into a replayed CUDA graph: the graph's kernel arguments are
// frozen, so the staging block in use is picked on the device from the parity of a replay counter (block A on even
// replays, B on odd ones) while the host fills / copies the other block for the next replay.
__global__ void __launch_bounds__(128) store_scatter_dbuf_kernel(StoreView s, long long n, const uint8_t *obs_a,
                                                                 const uint8_t *next_a, const pb_step_meta *meta_a,
                                                                 const uint8_t *obs_b, const uint8_t *next_b,
                                                                 const pb_step_meta *meta_b, const long long *counter)
{
    const bool odd = (*counter) & 1;
    const uint8_t *obs = odd ? obs_b : obs_a, *next_obs = odd ? next_b : next_a;
    const pb_step_meta *meta = odd ? meta_b : meta_a;
    const long long j = blockIdx.x;
    const pb_step_meta m = meta[j];
    const long long slot = m.seq % s.size;
    if (blockIdx.y == 0) {
        copy_row_bytes(s.obs_w + slot * s.row_bytes, obs + j * s.row_bytes, s.row_bytes);
        if (threadIdx.x == 0) {
            s.action[slot] = m.action;
            s.reward[slot] = m.reward;
            s.done[slot] = m.done;
            s.trunc[slot] = m.trunc;
            s.slot_seq[slot] = m.seq;
            s.prev_link[slot] = m.prev_link;
            s.next_link[slot] = m.next_link;
            if (m.patch_slot >= 0) s.next_link[m.patch_slot] = m.patch_val;
        }
    } else {
        const long long row = m.aux_row;
        if (row >= 0 && row < s.aux_size && next_obs)
            copy_row_bytes(s.aux_w + row * s.row_bytes, next_obs + j * s.row_bytes, s.row_bytes);
    }
}

__global__ void counter_inc_kernel(long long *counter) { *counter += 1; }

// dst = (parity of (*counter + bias)) ? src_b : src_a  -- picks this replay's half of a double-buffered staging block
// (the per-iteration uniforms ride in the same block as the new steps)
__global__ void __launch_bounds__(256) select_copy_kernel(double *__restrict__ dst, const double *__restrict__ src_a,
                                                          const double *__restrict__ src_b,
                                                          const long long *__restrict__ counter, long long bias, long long n)
{
    const double *src = ((*counter + bias) & 1) ? src_b : src_a;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// ---- n-step walk (uniform across the CTA: every thread reads the same addresses) ----
struct Walk {
    float ret, gamma;
    uint8_t done;
    long long last, succ;
};

__device__ __forceinline__ bool link_alive(const StoreView &s, long long link)
{
    return link >= 0 && s.slot_seq[link % s.size] == link;
}

__device__ __forceinline__ Walk nstep_walk(const StoreView &s, long long start)
{
    // _compute_n_step (timestep_buffer.py:198-238): python float (fp64) accumulation,
    // separate multiply and add (no fma), stored to fp32 tensors afterwards (:175-177).
    long long cur = start;
    double ret = 0.0, g = 1.0;
    for (int i = 0; i < s.n_step; ++i) {
        ret = __dadd_rn(ret, __dmul_rn((double)s.reward[cur], s.gammas[i]));
        g = s.gammas[i + 1];
        const bool incomplete = (i != s.n_step - 1);
        const long long nl = s.next_link[cur];
        if (nl >= 0 && !s.trunc[cur] && incomplete) {
            if (link_alive(s, nl)) cur = nl % s.size; else break;
        } else break;
    }
    Walk w;
    w.ret = (float)ret;
    w.gamma = (float)g;
    w.done = s.done[cur];
    w.last = cur;
    long long nl = s.next_link[cur];
    if (nl >= 0 && !link_alive(s, nl)) nl = -1;                   // dead weakref
    if (nl <= -2 && (-(nl) - 2) >= s.aux_size) nl = -1;           // defensive
    w.succ = nl;
    return w;
}

// walk `hops` prev links from slot; false if the chain is shorter
__device__ __forceinline__ bool prev_walk(const StoreView &s, long long &slot, int hops)
{
    for (int h = 0; h < hops; ++h) {
        const long long pl = s.prev_link[slot];
        if (!link_alive(s, pl)) return false;
        slot = pl % s.size;
    }
    return true;
}

__device__ __forceinline__ void emit_row(const StoreView &s, float *dst, const uint8_t *src)
{
    const int n = s.obs_elems;
    if (src == nullptr) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = 0.0f;
        return;
    }
    if (s.dtype == 0) {
        const float *f = reinterpret_cast<const float *>(src);
        if ((n & 3) == 0) {
            const uint4 *s4 = reinterpret_cast<const uint4 *>(f);
            uint4 *d4 = reinterpret_cast<uint4 *>(dst);
            for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x) stg_stream(d4 + i, ldg_stream(s4 + i));
        } else {
            for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = f[i];
        }
        return;
    }
    // uint8 storage, widened on the fly
    if ((n & 15) == 0) {
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        for (int i = threadIdx.x; i < (n >> 4); i += blockDim.x) {
            uint4 p = ldg_stream(s4 + i);
            unsigned w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float4 o;
                o.x = (float)(w[k] & 0xff); o.y = (float)((w[k] >> 8) & 0xff);
                o.z = (float)((w[k] >> 16) & 0xff); o.w = (float)(w[k] >> 24);
                if (s.scale) {
                    o.x = __fdiv_rn(o.x, 255.0f); o.y = __fdiv_rn(o.y, 255.0f);
                    o.z = __fdiv_rn(o.z, 255.0f); o.w = __fdiv_rn(o.w, 255.0f);
                }
                d4[i * 4 + k] = o;
            }
        }
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            float v = (float)src[i];
            dst[i] = s.scale ? __fdiv_rn(v, 255.0f) : v;
        }
    }
}

// grid (n, 2*frame_stack): blockIdx.y = which*fs + c; which 0 obs / 1 next_obs; c = chain
// position counted back from the newest frame (output frame fs-1-c).
__global__ void __launch_bounds__(256) store_gather_kernel(StoreView s, long long n, const long long *idx,
                                                           float *obs_out, float *next_out, float *ret_out,
                                                           float *gamma_out, uint8_t *nonterm_out,
                                                           long long *action_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const long long b = blockIdx.x;
    const long long start = idx[b];
    if (start < 0 || start >= s.size) return;
    const int which = blockIdx.y / s.fs;
    const int c = blockIdx.y % s.fs;
    const Walk w = nstep_walk(s, start);
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        ret_out[b] = w.ret;
        gamma_out[b] = w.gamma;
        nonterm_out[b] = w.done ? 0 : 1;
        action_out[b] = (long long)s.action[start];
    }
    // _stack_obs_into: frames are filled in lock-step while the START chain continues
    long long cur = start;
    const bool reach = prev_walk(s, cur, c);
    const uint8_t *src = nullptr;
    if (reach) {
        if (which == 0 || w.succ == -1) {
            src = s.obs + cur * s.row_bytes;          // obs frame; terminal: next_obs := obs
        } else if (c == 0) {
            src = w.succ >= 0 ? s.obs + (w.succ % s.size) * s.row_bytes
                              : s.aux + (-(w.succ) - 2) * s.row_bytes;
        } else {
            long long cur2 = w.last;                  // successor.prev is always the last walked step
            if (prev_walk(s, cur2, c - 1)) src = s.obs + cur2 * s.row_bytes;
        }
    }
    float *dst = (which ? next_out : obs_out) + ((b * s.fs) + (s.fs - 1 - c)) * (long long)s.obs_elems;
    emit_row(s, dst, src);
}

__global__ void store_nstep_kernel(StoreView s, long long n, const long long *idx, float *ret_out,
                                   float *gamma_out, uint8_t *done_out, long long *last_out, long long *succ_out)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const long long start = idx[b];
    if (start < 0 || start >= s.size) return;
    const Walk w = nstep_walk(s, start);
    ret_out[b] = w.ret; gamma_out[b] = w.gamma; done_out[b] = w.done;
    last_out[b] = w.last; succ_out[b] = w.succ;
}

}  // namespace

extern "C" {

int pb_store_extend_plan(long long size, long long aux_size, int n_streams, long long n, long long seq0,
                         const int *stream_id_h, const uint8_t *flags_h, long long *stream_last_h,
                         long long *trunc_cursor_h, long long *trunc_owner_h, pb_step_meta *meta_h)
{
    if (size <= 0 || n < 0 || n > size || n_streams <= 0 || aux_size < n_streams) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (!stream_id_h || !flags_h || !stream_last_h || !trunc_cursor_h || !meta_h) return PB_E_ARG;
    const long long pool = aux_size - n_streams;
    // dry run (no side effects on failure): stream ids valid; every truncated-pool row this
    // batch would recycle must belong to a step that has already left the ring
    {
        long long n_trunc = 0;
        for (long long j = 0; j < n; ++j) {
            if (stream_id_h[j] < 0 || stream_id_h[j] >= n_streams) return PB_E_ARG;
            n_trunc += ((flags_h[j] & PB_STEP_TRUNC) && !(flags_h[j] & PB_STEP_DONE));
        }
        if (n_trunc > 0) {
            if (n_trunc > pool || !trunc_owner_h) return PB_E_POOL;
            long long cur = *trunc_cursor_h;
            for (long long q = 0; q < n_trunc; ++q) {
                const long long owner = trunc_owner_h[cur];
                if (owner >= 0 && seq0 - owner < size) return PB_E_POOL;  // owner still in the ring
                cur = (cur + 1) % pool;
            }
        }
    }
    const long long end_seq = seq0 + n - 1;
    for (long long j = 0; j < n; ++j) {
        const int sid = stream_id_h[j];
        const long long s = seq0 + j;
        meta_h[j].seq = s;
        meta_h[j].patch_slot = -1; meta_h[j].patch_val = -1;
        const long long prev = stream_last_h[sid];
        meta_h[j].prev_link = prev;
        if (prev >= 0) {
            if (prev >= seq0) {                       // predecessor is in this batch: link directly
                meta_h[prev - seq0].next_link = s;
                meta_h[prev - seq0].aux_row = -1;     // its in-flight row is superseded by this step
            } else if (end_seq - prev < size) {       // still stored after this batch lands
                meta_h[j].patch_slot = prev % size;
                meta_h[j].patch_val = s;
            }
        }
        if (flags_h[j] & PB_STEP_DONE) {
            // collector_process_interface.py:167: done -> no next link
            meta_h[j].next_link = -1; meta_h[j].aux_row = -1; stream_last_h[sid] = -1;
        } else if (flags_h[j] & PB_STEP_NO_NEXT) {
            // a step handed over before its successor observation exists (hand-linked chains):
            // no next yet; the stream stays open so a later step can still link to it
            meta_h[j].next_link = -1; meta_h[j].aux_row = -1; stream_last_h[sid] = (flags_h[j] & PB_STEP_TRUNC) ? -1 : s;
        } else if (flags_h[j] & PB_STEP_TRUNC) {
            // :155-165: truncated -> next is the final observation, held only by this step
            const long long row = n_streams + *trunc_cursor_h;
            trunc_owner_h[*trunc_cursor_h] = s;
            *trunc_cursor_h = (*trunc_cursor_h + 1) % pool;
            meta_h[j].next_link = -(row + 2); meta_h[j].aux_row = row; stream_last_h[sid] = -1;
        } else {
            // :168-169: successor is the in-flight step (observation only) of the same stream
            meta_h[j].next_link = -((long long)sid + 2); meta_h[j].aux_row = sid; stream_last_h[sid] = s;
        }
    }
    return PB_OK;
}

// Fill a staging block from the collector's arrays and plan it, in one host call (what IngestSlot.fill does with a
// dozen small numpy assignments per learner iteration).
int pb_store_stage_block(long long size, long long aux_size, int n_streams, long long n, long long seq0,
                         long long row_bytes, const void *obs_h, const void *next_obs_h, const int *stream_id_h,
                         const void *action_h, int action_bytes, const float *reward_h, const uint8_t *done_h,
                         const uint8_t *trunc_h, void *rows_h, long long *stream_last_h, long long *trunc_cursor_h,
                         long long *trunc_owner_h, pb_step_meta *meta_h)
{
    if (n < 0 || row_bytes <= 0 || (action_bytes != 4 && action_bytes != 8)) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (!obs_h || !next_obs_h || !stream_id_h || !action_h || !reward_h || !done_h || !trunc_h || !rows_h || !meta_h)
        return PB_E_ARG;
    uint8_t small[256];
    uint8_t *flags = n <= 256 ? small : (uint8_t *)malloc((size_t)n);
    if (!flags) return PB_E_ARG;
    for (long long j = 0; j < n; ++j) {
        const uint8_t d = done_h[j] ? 1 : 0, t = trunc_h[j] ? 1 : 0;
        flags[j] = (uint8_t)(d * PB_STEP_DONE + t * PB_STEP_TRUNC);
        meta_h[j].action = action_bytes == 8 ? (int)((const long long *)action_h)[j] : ((const int *)action_h)[j];
        meta_h[j].reward = reward_h[j];
        meta_h[j].done = d;
        meta_h[j].trunc = t;
    }
    const int rc = pb_store_extend_plan(size, aux_size, n_streams, n, seq0, stream_id_h, flags, stream_last_h,
                                        trunc_cursor_h, trunc_owner_h, meta_h);
    if (flags != small) free(flags);
    if (rc != PB_OK) return rc;                                     // nothing planned: leave the rows alone too
    memcpy(rows_h, obs_h, (size_t)(n * row_bytes));
    memcpy((char *)rows_h + n * row_bytes, next_obs_h, (size_t)(n * row_bytes));
    return PB_OK;
}

int pb_store_scatter(const pb_store *st, long long n, const void *obs, const void *next_obs,
                     const pb_step_meta *meta, void *stream)
{
    StoreView v;
    int rc = make_store(st, &v);
    if (rc) return rc;
    if (n < 0 || n > v.size) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (!obs || !meta) return PB_E_ARG;
    dim3 grid((unsigned)n, 2);
    PB_LAUNCH(store_scatter_kernel, grid, 128, 0, stream, v, n, (const uint8_t *)obs, (const uint8_t *)next_obs, meta);
    return PB_OK;
}

int pb_store_scatter_dbuf(const pb_store *st, long long n, const void *obs_a, const void *next_obs_a,
                          const pb_step_meta *meta_a, const void *obs_b, const void *next_obs_b,
                          const pb_step_meta *meta_b, long long *replay_counter, void *stream)
{
    StoreView v;
    int rc = make_store(st, &v);
    if (rc) return rc;
    if (n <= 0 || n > v.size || !obs_a || !meta_a || !obs_b || !meta_b || !replay_counter) return PB_E_ARG;
    dim3 grid((unsigned)n, 2);
    PB_LAUNCH(store_scatter_dbuf_kernel, grid, 128, 0, stream, v, n, (const uint8_t *)obs_a, (const uint8_t *)next_obs_a,
              meta_a, (const uint8_t *)obs_b, (const uint8_t *)next_obs_b, meta_b, (const long long *)replay_counter);
    PB_LAUNCH(counter_inc_kernel, 1, 1, 0, stream, replay_counter);
    return PB_OK;
}

int pb_select_copy_f64(double *dst, const double *src_a, const double *src_b, const long long *replay_counter,
                       long long bias, long long n, void *stream)
{
    if (!dst || !src_a || !src_b || !replay_counter || n <= 0) return PB_E_ARG;
    long long nb = (n + 255) / 256;
    if (nb > 64) nb = 64;
    PB_LAUNCH(select_copy_kernel, (unsigned)nb, 256, 0, stream, dst, src_a, src_b, replay_counter, bias, n);
    return PB_OK;
}

int pb_store_gather(const pb_store *st, long long n, const long long *idx, float *obs_out, float *next_obs_out,
                    float *ret_out, float *gamma_out, uint8_t *nonterm_out, long long *action_out, void *stream)
{
    StoreView v;
    int rc = make_store(st, &v);
    if (rc) return rc;
    if (n < 0) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (!idx || !obs_out || !next_obs_out || !ret_out || !gamma_out || !nonterm_out || !action_out) return PB_E_ARG;
    dim3 grid((unsigned)n, (unsigned)(2 * v.fs));
    const int threads = v.row_bytes >= 4096 ? 256 : 128;
    PB_LAUNCH(store_gather_kernel, grid, threads, 0, stream, v, n, idx, obs_out, next_obs_out, ret_out, gamma_out,
              nonterm_out, action_out);
    return PB_OK;
}

int pb_store_nstep(const pb_store *st, long long n, const long long *idx, float *ret_out, float *gamma_out,
                   uint8_t *done_out, long long *last_out, long long *succ_out, void *stream)
{
    StoreView v;
    int rc = make_store(st, &v);
    if (rc) return rc;
    if (n < 0) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (!idx || !ret_out || !gamma_out || !done_out || !last_out || !succ_out) return PB_E_ARG;
    PB_LAUNCH(store_nstep_kernel, (unsigned)((n + 127) / 128), 128, 0, stream, v, n, idx, ret_out, gamma_out,
              done_out, last_out, succ_out);
    return PB_OK;
}

}  // extern "C"
