// per_tree.cu -- sum-tree / min-tree priority store for prioritized replay (sm_100a).
//
// Replaces the segment tree + PrioritizedSampler that the reference reaches through
// torchrl (prism/factory/exp_buffer_factory.py:22-28; call sites
// prism/experience/timestep_buffer.py:33,37,54; prism/learner.py:100,120).
//
// Design (B200-first, not a port of a pointer-walking CPU tree):
//  * every node is fl32(left + right) / min(left, right) of a binary tree over the leaves -- the reference add
//    order, so sampled indices are bit-exact whatever order updates arrive in.
//  * one primitive everywhere: 32 sibling nodes (one aligned 128-byte line) are reduced over 5 levels in registers
//    and shuffles.  The rebuilt intermediate values are bit-identical to the nodes a pointer-walking tree would
//    store, so they are NOT stored: the tree keeps only every 5th level below its top ("compact" layout)
//        levels 0 .. TL          one level-ordered heap array (TL <= 9: <= 4 KB)
//        levels TL+5, TL+10, .., L   one array per level; L = leaves
//    and the min tree shares the leaf array of the sum tree (a leaf is written with the same value in both;
//    slots that were never written -- index >= len -- read as +inf on the min side).
//    16M leaves: 64 MiB + 2 x 2.1 MiB instead of 2 x 128 MiB, i.e. the whole store fits the 126 MB L2.
//      - sampling descends 5 levels per dependent 128-byte load: 8 lanes per sample for one learner batch (latency),
//        a thread per sample over a shared-memory copy of the top 14 levels for many batches in flight (throughput:
//        the warp fetches its 32 lines together and transposes them through shared memory);
//      - an update is a LINE phase -- every touched 32-leaf line is patched and reduced to its node of level L-5 by one
//        thread holding the line in registers -- followed by a streaming rebuild of the (32 x smaller) tree above
//        level L-5, whose last CTA (ticket) rebuilds the top heap and the state block.  Sorted batches (one
//        stratified learner batch, the ring's extends): the first entry of every line's run is its leader, 2 launches.
//        Any other batch (unsorted, duplicates, K batches in flight): a mark pass leaves a dedup tag on every touched
//        leaf slot, then the entry whose tag sits in a line's lowest tagged slot leads that line, 3 launches;
//      - batches beyond cap/16 entries scatter their leaves and rebuild every line with one streaming pass over the
//        leaf array (4.3 B per leaf of traffic, independent of the batch size);
//      - the bulk build is that same streaming pass;
//      - the launches of one call (and the sampling launch that follows) are programmatic dependent launches.
//  * duplicates in an update batch: last occurrence wins (sequential reference loop), resolved deterministically
//    (adjacency when sorted; otherwise atomicMax of a NaN-tagged entry number on the leaf slot itself -- no side array).
//  * no host sync anywhere: len / cursor / max_priority / p_sum / p_min live in a 64-byte device state block, so
//    the whole sample->update loop is CUDA-graph capturable.
#include "common.cuh"
#include <math.h>

namespace {

using namespace pb;

constexpr int TOP_MAX = 9;         // the top heap holds levels [0, TL], TL <= 9: rebuilt whole by ONE CTA after every update
constexpr int MAX_DEEP = 8;        // stored levels below the heap (capacity <= 2^30 -> at most 4)

struct TreeView {
    float *sum, *min;
    int *owner, *cnt;
    pb_per_state *st;
    long long cap, size;
    int L, TL, P;                  // P = (L - TL) / 5 deep levels: L, L-5, .., TL+5
    long long off[MAX_DEEP];       // off[m]: float offset of level TL + 5m in the sum / min store (m >= 1)
    float alpha, eps32;
    double eps64;
    int weps, dp64;
};

enum { MODE_RAW = 0, MODE_PRIORITY = 1, MODE_EXTEND = 2 };
constexpr float INF = __builtin_huge_valf();

__device__ __forceinline__ float op_sum(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float op_min(float a, float b) { return fminf(a, b); }

// level s of the sum tree (node i of that level at [i])
__device__ __forceinline__ float *sum_level(const TreeView &t, int s)
{
    return s <= t.TL ? t.sum + (1LL << s) : t.sum + t.off[(s - t.TL) / 5];
}
// level s < L of the min tree (the leaf level is shared with the sum tree, see min_of_leaf)
__device__ __forceinline__ float *min_level(const TreeView &t, int s)
{
    return s <= t.TL ? t.min + (1LL << s) : t.min + t.off[(s - t.TL) / 5];
}
__device__ __forceinline__ float *leaf_ptr(const TreeView &t) { return sum_level(t, t.L); }
__device__ __forceinline__ float min_of_leaf(float v, long long i, long long len) { return i < len ? v : INF; }

__device__ __forceinline__ float ldcg(const float *p) { return __ldcg(p); }

// arrival-counter update with release (my node store is visible to whoever reads the counter after me) and acquire
// (I see the node stores of everyone who updated it before me) semantics in ONE instruction -- no MEMBAR.SC
__device__ __forceinline__ int atom_add_acq_rel(int *p, int v)
{
    int old;
    asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}

// ---------------------------------------------------------------------------------
// phase marks for measurement runs (pb_tree_trace; profiles/per_phases.py): slot <- the LATEST %globaltimer at which
// any CTA passed the mark (start marks: slot <- CTA 0's own time).  Off by default: one cached load per mark.
// ---------------------------------------------------------------------------------
constexpr int TRACE_SLOTS = 48;
__device__ unsigned long long g_trace[TRACE_SLOTS];
__device__ int g_trace_on;

// `on` = g_trace_on read ONCE at kernel entry (TRACE_ON).  Call from one thread per CTA (or per warp).
#define TRACE_ON() (__ldg(&g_trace_on))
__device__ __forceinline__ void trace_max(int on, int slot)
{
    if (on) atomicMax(&g_trace[slot], global_ns());
}
__device__ __forceinline__ void trace_cta0(int on, int slot)
{
    if (on && blockIdx.x == 0 && threadIdx.x == 0) g_trace[slot] = global_ns();
}
enum {
    TR_SAMPLE_START = 0, TR_SAMPLE_STAGED, TR_SAMPLE_END,
    TR_CHAIN_START = 4, TR_CHAIN_REGISTERED, TR_CHAIN_LEAVES, TR_CHAIN_GROUP, TR_CHAIN_CLIMBED, TR_CHAIN_TICKET, TR_CHAIN_TOP,
    TR_CHAIN_END,
    TR_MARK_START = 16, TR_MARK_END, TR_LEAF_START, TR_LEAF_END, TR_SPARSE_START, TR_SPARSE_SPANS, TR_SPARSE_TICKET,
    TR_SPARSE_TOP, TR_SPARSE_END,
    TR_REBUILD_START = 28, TR_REBUILD_END, TR_REBUILD_TICKET, TR_REBUILD_TOP, TR_REBUILD_STATE,
    TR_LINES_START = 36, TR_LINES_END
};

// cold paths (every reference configuration has alpha = 0.5): kept out of line so that the latency-bound update
// kernels stay small in the instruction cache
__device__ __noinline__ float powf_cold(float x, float a) { return powf(x, a); }
__device__ __noinline__ double pow_cold(double x, double a) { return pow(x, a); }

__device__ __forceinline__ float pow_leaf(float p, const TreeView &t)
{
    // torch.pow(priority + eps, alpha) on an fp32 tensor; alpha == 0.5 is torch's sqrt path
    float x = __fadd_rn(p, t.eps32);
    if (t.alpha == 0.5f) return __fsqrt_rn(x);
    if (t.alpha == 1.0f) return x;
    return powf_cold(x, t.alpha);
}

__device__ __forceinline__ float default_priority(const TreeView &t)
{
    float mp = t.st->max_priority;
    if (t.dp64) {
        double x = (double)mp + t.eps64;
        double r = (t.alpha == 0.5f) ? __dsqrt_rn(x) : ((t.alpha == 1.0f) ? x : pow_cold(x, (double)t.alpha));
        return (float)r;
    }
    return pow_leaf(mp, t);
}

__device__ __forceinline__ long long entry_index(const TreeView &t, const long long *idx, long long j, int mode,
                                                 long long seq0)
{
    if (mode == MODE_EXTEND) return (seq0 + j) % t.size;
    return idx[j];
}

__device__ __forceinline__ float entry_leaf(const TreeView &t, const float *val, long long j, int mode, float defp)
{
    if (mode == MODE_RAW) return val[j];
    if (mode == MODE_PRIORITY) return pow_leaf(fabsf(val[j]), t);   // learner.py:120 passes |td|; idempotent
    return defp;
}

__device__ __forceinline__ long long len_after(const TreeView &t, int mode, long long n_new, long long set_len)
{
    long long len = t.st->len;
    if (mode == MODE_EXTEND) len = len + n_new < t.size ? len + n_new : t.size;
    else if (set_len >= 0) len = set_len < t.size ? set_len : t.size;
    return len;
}

// reduce one line: every lane holds one of 32 sibling nodes; returns the 5-level pairwise total in every lane
__device__ __forceinline__ void line_reduce(float &vs, float &vm)
{
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        vs = op_sum(vs, __shfl_xor_sync(FULL, vs, 1 << s));
        vm = op_min(vm, __shfl_xor_sync(FULL, vm, 1 << s));
    }
}

// ---------------------------------------------------------------------------------
// value of ANY node (level d, index i), stored or not: an unstored level is rebuilt pairwise from the next
// stored level below it (<= 16 nodes).
// ---------------------------------------------------------------------------------
template <bool IS_MIN>
__device__ float node_value(const TreeView &t, int d, long long i, long long len)
{
    const float ident = IS_MIN ? INF : 0.0f;
    const int r = d <= t.TL ? 0 : (t.L - d) % 5;     // levels to the next stored level below
    const int s = d + r;
    const long long base = i << r;
    float v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (k < (1 << r)) {
            // L2 loads: the state block is finalised by the last CTA of a launch whose other CTAs wrote these nodes
            if (s == t.L) {
                float x = ldcg(leaf_ptr(t) + base + k);
                v[k] = IS_MIN ? min_of_leaf(x, base + k, len) : x;
            } else {
                v[k] = IS_MIN ? ldcg(min_level(t, s) + base + k) : ldcg(sum_level(t, s) + base + k);
            }
        } else {
            v[k] = ident;
        }
    }
#pragma unroll
    for (int w = 8; w >= 1; w >>= 1) {
        if (w < (1 << r)) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (k < w) v[k] = IS_MIN ? op_min(v[2 * k], v[2 * k + 1]) : op_sum(v[2 * k], v[2 * k + 1]);
        }
    }
    return v[0];
}

// ---------------------------------------------------------------------------------
// query(0, len) with torchrl's interval-walk association (one warp)
// ---------------------------------------------------------------------------------
template <bool IS_MIN>
__device__ float tree_query_prefix(const TreeView &t, long long len)
{
    const float ident = IS_MIN ? INF : 0.0f;
    if (len >= t.size) return IS_MIN ? ldcg(t.min + 1) : ldcg(t.sum + 1);
    if (len <= 0) return ident;
    const int k = lane_id();
    float v = ident;
    // bit k of len set: the walk takes node (len >> k) - 1 of level L - k (a node fully inside [0, len))
    if (k < t.L && ((len >> k) & 1)) v = node_value<IS_MIN>(t, t.L - k, (len >> k) - 1, len);
    float ret = ident;
    for (int b = 0; b < t.L; ++b) {
        float vb = __shfl_sync(FULL, v, b);
        if ((len >> b) & 1) ret = IS_MIN ? op_min(ret, vb) : op_sum(ret, vb);
    }
    return ret;
}

// one warp: advance len / seq, merge max_priority, refresh p_sum / p_min.  have_roots: the caller rebuilt the top heap and
// hands over the roots (a full tree's query(0, len) IS the root: no load, no fence)
__device__ void finalize_state(const TreeView &t, int mode, long long n_new, long long set_len, bool have_roots = false,
                               float root_s = 0.0f, float root_m = 0.0f)
{
    const long long len = len_after(t, mode, n_new, set_len);
    float ps, pm;
    if (have_roots && len >= t.size) { ps = root_s; pm = root_m; }
    else {
        if (have_roots) __threadfence();          // partial fill: the walk reads heap nodes other warps of this CTA just stored
        ps = tree_query_prefix<false>(t, len);
        pm = tree_query_prefix<true>(t, len);
    }
    if (lane_id() == 0) {
        pb_per_state *s = t.st;
        if (mode == MODE_EXTEND) s->seq += n_new;
        else if (set_len >= 0) s->seq = set_len;
        s->len = len;
        if (mode == MODE_PRIORITY) {
            const float bm = s->batch_max;
            if (bm > s->max_priority) s->max_priority = bm;
        }
        s->batch_max = 0.0f;
        s->p_sum = ps; s->p_min = pm;
        s->pad[0] = 0;
    }
}

// ---------------------------------------------------------------------------------
// top phase: rebuild heap levels TL-1 .. 0 of BOTH trees from level TL (32 .. 512 nodes).  Called by every thread of ONE
// CTA (blockDim.x threads, a multiple of 64; the first half works on the sum tree, the second on the min tree).
// Every warp reduces lines of 32 level-TL nodes with shuffles, storing the intermediate levels as it goes; the
// <= 16 line totals (level TL-5) meet in shared memory and one warp per tree finishes the last levels.
// ---------------------------------------------------------------------------------
constexpr int TOP_SM_FLOATS = 32;                   // per tree: the line totals

__device__ void top_rebuild(const TreeView &t, float *sm, long long len)
{
    const int half = blockDim.x >> 1;
    const bool is_min = threadIdx.x >= half;
    const int tid = is_min ? threadIdx.x - half : threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5, n_warps = half >> 5;
    float *heap = is_min ? t.min : t.sum;
    float *s = sm + (is_min ? TOP_SM_FLOATS : 0);
    const int TL = t.TL;                                        // 5 .. 9
    const bool shared_leaves = is_min && TL == t.L;             // tiny trees: level TL is the shared leaf level
    const float *src = shared_leaves ? t.sum + (1 << TL) : heap + (1 << TL);
    const int n_lines = 1 << (TL - 5);
    for (int base = warp; base < n_lines; base += 4 * n_warps) {
        float v4[4];                                            // up to 4 lines per warp with their loads in flight
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int line = base + u * n_warps, e = (line << 5) + lane;
            v4[u] = line < n_lines ? ldcg(src + e) : 0.0f;
            if (shared_leaves && line < n_lines) v4[u] = min_of_leaf(v4[u], e, len);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int line = base + u * n_warps, e = (line << 5) + lane;
            if (line >= n_lines) break;                         // warp-uniform
            float v = v4[u];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float o = __shfl_xor_sync(FULL, v, 1 << k);
                v = is_min ? op_min(v, o) : op_sum(v, o);
                if ((lane & ((2 << k) - 1)) == 0) heap[(1 << (TL - 1 - k)) + (e >> (k + 1))] = v;
            }
            if (lane == 0) s[line] = v;                          // node `line` of level TL - 5 (already stored above)
        }
    }
    __syncthreads();
    if (warp == 0 && TL > 5) {
        float v = lane < n_lines ? s[lane] : (is_min ? INF : 0.0f);
        for (int k = 0; k < TL - 5; ++k) {
            const float o = __shfl_xor_sync(FULL, v, 1 << k);
            v = is_min ? op_min(v, o) : op_sum(v, o);
            if (lane < n_lines && (lane & ((2 << k) - 1)) == 0) heap[(1 << (TL - 6 - k)) + (lane >> (k + 1))] = v;
        }
        if (lane == 0) s[0] = v;                                  // the root (TL == 5: s[0] already is)
    }
}

// last-CTA ticket: returns true in every thread of the CTA that arrives last.  pad[0] is reset by finalize_state.
__device__ bool last_cta(const TreeView &t)
{
    __shared__ int is_last;
    __syncthreads();                                  // the CTA's stores happen-before thread 0's release below
    if (threadIdx.x == 0) {
        const int ticket = atom_add_acq_rel(&t.st->pad[0], 1);
        is_last = (ticket == (int)gridDim.x - 1);
    }
    __syncthreads();
    return is_last != 0;
}

__device__ void top_and_finalize(const TreeView &t, float *sm, int mode, long long n_new, long long set_len,
                                 int tr_top = -1, int tr_end = -1)
{
    const long long len = len_after(t, mode, n_new, set_len);
    top_rebuild(t, sm, len);
    __syncthreads();
    if (tr_top >= 0 && threadIdx.x == 0) trace_max(1, tr_top);
    if (threadIdx.x < 32) finalize_state(t, mode, n_new, set_len, true, sm[0], sm[TOP_SM_FLOATS]);
    if (tr_end >= 0 && threadIdx.x == 0) trace_max(1, tr_end);
}

// ---------------------------------------------------------------------------------
// init
// ---------------------------------------------------------------------------------
__global__ void tree_init_kernel(TreeView t, long long n_sum, long long n_min, long long n_cnt)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = i; k < n_sum; k += stride) t.sum[k] = 0.0f;
    for (long long k = i; k < n_min; k += stride) t.min[k] = INF;
    for (long long k = i; k < n_cnt; k += stride) t.cnt[k] = 0;
    if (i == 0) {
        pb_per_state s;
        s.len = 0; s.seq = 0; s.max_priority = 1.0f; s.p_sum = 0.0f; s.p_min = INF; s.status = 0;
        s.batch_max = 0.0f; s.owned_lo = 0; s.owned_n = 0;
        for (int k = 0; k < 5; ++k) s.pad[k] = 0;
        *t.st = s;
    }
}

__global__ void tree_stats_kernel(TreeView t)
{
    const long long len = t.st->len;
    const float ps = tree_query_prefix<false>(t, len);
    const float pm = tree_query_prefix<true>(t, len);
    if (threadIdx.x == 0) { t.st->p_sum = ps; t.st->p_min = pm; }
}

// ---------------------------------------------------------------------------------
// streaming rebuild: every line of level s is reduced to its node of level s-5 and, when that level is stored
// too, on to level s-10.  Warp-autonomous, no shared memory: per iteration a warp streams 1024 consecutive source
// nodes with 8 coalesced float4 loads per lane in flight (8 lanes per 128-byte line), reduces every line in
// registers + 3 shuffle levels, transposes the 32 line totals into one lane each with shuffles (= one coalesced
// 128-byte store of level s-5) and reduces those 5 more levels for the node of level s-10.  Persistent grid.
// s == L reads the shared leaf array (optionally first loading it from `ext`, the bulk build).
// FUSE_TOP: the last CTA (ticket) rebuilds the top heap and the state block.
// ---------------------------------------------------------------------------------
constexpr int RB_THREADS = 256;
constexpr int RB_TILE = 1024;                                    // source nodes per warp iteration

// n_lv = 1, 2 or 3 levels per pass (s-5, s-10, s-15).  The third level needs 32 warp tiles in one CTA: a CTA then takes
// 32768 consecutive source nodes per iteration (4 warp tiles per warp) and combines their level s-10 nodes through
// shared memory.
__global__ void __launch_bounds__(RB_THREADS) tree_rebuild_kernel(TreeView t, int s, int n_lv, const float *ext,
                                                                  long long n_ext, int fuse_top, int mode,
                                                                  long long n_new, long long set_len)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ float sm_top[2 * TOP_SM_FLOATS];
    __shared__ float l2s[32], l2m[32];
    const int two_levels = n_lv >= 2;
    const long long len = len_after(t, mode, n_new, set_len);
    const bool leaves = (s == t.L);
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_REBUILD_START);
    float *src_s = sum_level(t, s);
    const float *src_m = leaves ? src_s : min_level(t, s);
    float *dst1_s = sum_level(t, s - 5), *dst1_m = min_level(t, s - 5);
    const long long n_tiles = (1LL << s) / RB_TILE;
    const int lane = lane_id();
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    // n_lv < 3: warps stride over the warp tiles on their own.  n_lv == 3: CTAs stride over groups of 32 warp tiles.
    const int wic = threadIdx.x >> 5;                            // warp in CTA (RB_THREADS / 32 = 8 of them)
    const long long n_outer = n_lv == 3 ? n_tiles / 32 : 1;
    for (long long outer = n_lv == 3 ? blockIdx.x : 0; outer < n_outer; outer += n_lv == 3 ? gridDim.x : 1) {
    const long long t_first = n_lv == 3 ? outer * 32 + wic : (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const long long t_step = n_lv == 3 ? RB_THREADS / 32 : n_warps;
    const long long t_end = n_lv == 3 ? outer * 32 + 32 : n_tiles;
    for (long long tile = t_first; tile < t_end; tile += t_step) {
        const long long base = tile * RB_TILE + lane * 4;        // load q covers nodes base + 128 q .. + 3
        float4 a[8], m[8];
        if (ext) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const long long e = base + 128 * q;
                if (e + 4 <= n_ext) a[q] = __ldcs(reinterpret_cast<const float4 *>(ext + e));
                else {
                    a[q].x = e + 0 < n_ext ? ext[e + 0] : 0.0f; a[q].y = e + 1 < n_ext ? ext[e + 1] : 0.0f;
                    a[q].z = e + 2 < n_ext ? ext[e + 2] : 0.0f; a[q].w = e + 3 < n_ext ? ext[e + 3] : 0.0f;
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) *reinterpret_cast<float4 *>(src_s + base + 128 * q) = a[q];
        } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) a[q] = __ldcg(reinterpret_cast<const float4 *>(src_s + base + 128 * q));
        }
        if (leaves) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const long long e = base + 128 * q;
                m[q] = a[q];
                if (e + 4 > len) {
                    m[q].x = min_of_leaf(a[q].x, e + 0, len); m[q].y = min_of_leaf(a[q].y, e + 1, len);
                    m[q].z = min_of_leaf(a[q].z, e + 2, len); m[q].w = min_of_leaf(a[q].w, e + 3, len);
                }
            }
        } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) m[q] = __ldcg(reinterpret_cast<const float4 *>(src_m + base + 128 * q));
        }
        // line totals: load q holds 4 lines (8 lanes each); afterwards lane l owns line l of the tile
        float ps = 0.0f, pm = 0.0f;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float vs = op_sum(op_sum(a[q].x, a[q].y), op_sum(a[q].z, a[q].w));
            float vm = op_min(op_min(m[q].x, m[q].y), op_min(m[q].z, m[q].w));
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                vs = op_sum(vs, __shfl_xor_sync(FULL, vs, 1 << k));
                vm = op_min(vm, __shfl_xor_sync(FULL, vm, 1 << k));
            }
            // line 4q + g sits in the lanes of group g: hand it to lane 4q + g
            const float gs = __shfl_sync(FULL, vs, (lane & 3) << 3);
            const float gm = __shfl_sync(FULL, vm, (lane & 3) << 3);
            if ((lane >> 2) == q) { ps = gs; pm = gm; }
        }
        dst1_s[tile * 32 + lane] = ps;                           // 32 nodes of level s-5: one coalesced line
        dst1_m[tile * 32 + lane] = pm;
        if (two_levels) {
            line_reduce(ps, pm);
            if (lane == 0) {
                sum_level(t, s - 10)[tile] = ps; min_level(t, s - 10)[tile] = pm;
                if (n_lv == 3) { l2s[tile & 31] = ps; l2m[tile & 31] = pm; }
            }
        }
    }
    if (n_lv == 3) {
        __syncthreads();
        if (wic == 0) {
            float ps = l2s[lane], pm = l2m[lane];
            line_reduce(ps, pm);
            if (lane == 0) { sum_level(t, s - 15)[outer] = ps; min_level(t, s - 15)[outer] = pm; }
        }
        __syncthreads();
    }
    }
    if (threadIdx.x == 0) trace_max(tr_on, TR_REBUILD_END);
    if (!fuse_top) return;
    if (!last_cta(t)) return;
    if (threadIdx.x == 0) trace_max(tr_on, TR_REBUILD_TICKET);
    top_and_finalize(t, sm_top, mode, n_new, set_len, tr_on ? TR_REBUILD_TOP : -1, tr_on ? TR_REBUILD_STATE : -1);
}

// trees without deep levels (L <= 14): copy the leaves (identity padded) into the heap's leaf level
__global__ void tree_fill_leaves_kernel(TreeView t, const float *leaves, long long n_leaves)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= t.cap) return;
    leaf_ptr(t)[i] = i < n_leaves ? leaves[i] : 0.0f;
}

// standalone top phase (one CTA)
__global__ void __launch_bounds__(512) tree_top_kernel(TreeView t, int mode, long long n_new, long long set_len)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ float sm_top[2 * TOP_SM_FLOATS];
    top_and_finalize(t, sm_top, mode, n_new, set_len);
}

// ---------------------------------------------------------------------------------
// leaf scatter, general (unsorted) path.  Duplicates: the LAST occurrence wins (sequential reference loop).  No side
// array: the leaf slot itself is the scratch.  A) every entry j does atomicMax(int view of leaf[i], TAG + j): TAG + j
// is a NaN bit pattern, as a signed int larger than every non-NaN float's, so the slot ends up holding the tag of the
// highest j that targets it.  B) the entry whose tag it finds there writes the value.  Dense path, sorted input: the
// last entry of every run of equal indices writes the leaf.
// ---------------------------------------------------------------------------------
constexpr int LEAF_TAG = 0x7F800001;                 // first NaN pattern; TAG + j stays a positive int for j < 2^23 - 1
constexpr long long LEAF_TAG_MAX_N = (1LL << 23) - 2;

// the batch's largest |priority| (max_priority is merged by the finalising CTA): one conditional atomic per CTA -- an
// atomic per warp on this ONE address serialises in L2 (measured: 73 us of a 1M-entry mark pass).  Every thread calls.
__device__ __forceinline__ void cta_batch_max(const TreeView &t, float bm)
{
    __shared__ float s_bm[32];
    bm = warp_max(bm);
    if (lane_id() == 0) s_bm[threadIdx.x >> 5] = bm;
    __syncthreads();
    if (threadIdx.x < 32) {
        const int nw = (blockDim.x + 31) >> 5;
        bm = warp_max(threadIdx.x < nw ? s_bm[threadIdx.x] : 0.0f);
        if (threadIdx.x == 0 && bm > 0.0f && bm > __ldcg(&t.st->batch_max))
            atomicMax(reinterpret_cast<int *>(&t.st->batch_max), __float_as_int(bm));
    }
}

__global__ void upd_mark_kernel(TreeView t, long long n, const long long *idx, const float *val, int mode,
                                long long *idx_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long seq0 = t.st->seq;
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_MARK_START);
    float bm = 0.0f;
    if (j < n) {
        const long long i = entry_index(t, idx, j, mode, seq0);
        if (idx_out) idx_out[j] = i;
        if (i >= 0 && i < t.size) {
            atomicMax(reinterpret_cast<int *>(leaf_ptr(t) + i), LEAF_TAG + (int)j);
            if (mode == MODE_PRIORITY) bm = fabsf(val[j]);
        }
    }
    if (mode == MODE_PRIORITY) cta_batch_max(t, bm);
    if (threadIdx.x == 0) trace_max(tr_on, TR_MARK_END);
}

__global__ void upd_leaf_kernel(TreeView t, long long n, const long long *idx, const float *val, int mode,
                                long long *idx_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_LEAF_START);
    if (j < n) {
        const long long i = entry_index(t, idx, j, mode, t.st->seq);
        if (idx_out) idx_out[j] = i;
        if (i >= 0 && i < t.size && __ldcg(reinterpret_cast<const int *>(leaf_ptr(t) + i)) == LEAF_TAG + (int)j) {
            const float defp = (mode == MODE_EXTEND) ? default_priority(t) : 0.0f;
            leaf_ptr(t)[i] = entry_leaf(t, val, j, mode, defp);
        }
    }
    if (threadIdx.x == 0) trace_max(tr_on, TR_LEAF_END);
}

__global__ void upd_leaf_sorted_kernel(TreeView t, long long n, const long long *idx, const float *val, int mode,
                                       long long *idx_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long seq0 = t.st->seq;
    float bm = 0.0f;
    if (j < n) {
        const long long i = entry_index(t, idx, j, mode, seq0);
        if (idx_out) idx_out[j] = i;
        if (i >= 0 && i < t.size) {
            if (mode == MODE_PRIORITY) bm = fabsf(val[j]);
            const long long nx = (j + 1 < n) ? entry_index(t, idx, j + 1, mode, seq0) : -1;
            if (nx != i) {
                const float defp = (mode == MODE_EXTEND) ? default_priority(t) : 0.0f;
                leaf_ptr(t)[i] = entry_leaf(t, val, j, mode, defp);
            }
        }
    }
    if (mode == MODE_PRIORITY) cta_batch_max(t, bm);
}

// ---------------------------------------------------------------------------------
// LINE PHASE of an update: every touched leaf line (32 leaves, 128 bytes) is reduced to its node of level L-5 by ONE
// thread that holds the whole line in registers (8 x 128-bit loads in flight, tree-order sums in registers).  Nothing
// above level L-5 is touched here: from there the tree is small (2^-5 of the leaves) and a streaming pass rebuilds it
// whole (tree_rebuild_kernel from level L-5, top heap and state block by its last CTA) -- two short launches with no
// dependency between CTAs instead of a climb through arrival counters (measured at 2^24 leaves, batch 4096: 15 us for
// the one-launch climb, of which 5 us waiting on store -> load round trips, profiles/per_phases_r02.txt).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void line_total(const float4 (&v)[8], long long base, long long len, float &vs, float &vm)
{
    float ps[8], pm[8];
    const bool whole = base + 32 <= len;                          // every leaf of the line is a filled slot
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float4 m = v[k];
        if (!whole) {
            const long long e = base + 4 * k;
            m.x = min_of_leaf(m.x, e + 0, len); m.y = min_of_leaf(m.y, e + 1, len);
            m.z = min_of_leaf(m.z, e + 2, len); m.w = min_of_leaf(m.w, e + 3, len);
        }
        ps[k] = op_sum(op_sum(v[k].x, v[k].y), op_sum(v[k].z, v[k].w));
        pm[k] = op_min(op_min(m.x, m.y), op_min(m.z, m.w));
    }
    vs = op_sum(op_sum(op_sum(ps[0], ps[1]), op_sum(ps[2], ps[3])), op_sum(op_sum(ps[4], ps[5]), op_sum(ps[6], ps[7])));
    vm = op_min(op_min(op_min(pm[0], pm[1]), op_min(pm[2], pm[3])), op_min(op_min(pm[4], pm[5]), op_min(pm[6], pm[7])));
}

struct RunScan { long long seq0; const long long *idx; long long n; int mode; };

__device__ __forceinline__ bool valid_at(const TreeView &t, const RunScan &r, long long j, long long &i)
{
    if (j < 0 || j >= r.n) return false;
    i = entry_index(t, r.idx, j, r.mode, r.seq0);
    return i >= 0 && i < t.size;
}

// Every lane of a warp wants one 128-byte line (line index `node` of the array `lvl`).  Fetched TOGETHER: 4 lines per
// load instruction (8 lanes x 16 bytes per line -- one L1 wavefront per line instead of eight when every lane
// streams its own line, which is what bounded the first thread-per-sample / thread-per-entry kernels), transposed
// through 4 KB of shared memory per warp (XOR-swizzled 16-byte chunks, conflict-free both ways).  All 32 lanes call.
__device__ __forceinline__ void warp_fetch_lines_raw(const float *__restrict__ lvl, long long node, float4 *wbuf, float4 (&q)[8])
{
    const int lane = lane_id();
    const int g = lane >> 3, c = lane & 7;
    float4 r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const long long ln = __shfl_sync(FULL, node, 4 * k + g);
        r[k] = __ldcg(reinterpret_cast<const float4 *>(lvl + (ln << 5)) + c);
    }
    __syncwarp();                                                 // everyone is done reading the previous fetch
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int slot = 4 * k + g;
        wbuf[slot * 8 + (c ^ (slot & 7))] = r[k];
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 8; ++k) q[k] = wbuf[lane * 8 + (k ^ (lane & 7))];
}

// Sorted input (one stratified learner batch, the ring's extends), thread per entry.  The first entry of every run of
// entries that fall into the same leaf line is the line's leader: it loads the line, applies the run in entry order
// (last of equal indices wins, like the sequential reference loop) to its registers AND to the leaf array, and stores
// the line's node of level L-5.  No thread reads what another one wrote in this launch.  Needs P >= 1.
constexpr int LS_THREADS = 128;
constexpr long long SORTED_LINES_MAX_N = 1 << 20;   // thread per entry; beyond this the streaming pass over all leaves wins

__global__ void __launch_bounds__(LS_THREADS) upd_lines_sorted_kernel(TreeView t, long long n, const long long *idx,
                                                                      const float *val, int mode, long long *idx_out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_LINES_START);
    RunScan r;
    r.seq0 = mode == MODE_EXTEND ? t.st->seq : 0; r.idx = idx; r.n = n; r.mode = mode;     // the cursor only names slots of an extend
    const long long len = len_after(t, mode, n, -1);
    const float defp = (mode == MODE_EXTEND) ? default_priority(t) : 0.0f;
    float *leaf = leaf_ptr(t);
    float *n1s = sum_level(t, t.L - 5), *n1m = min_level(t, t.L - 5);
    float bm = 0.0f;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
        // everything the common case needs is requested up front: own index, both neighbours, own value
        long long i = -1, ip = -1, inx = -1;
        const bool ok = valid_at(t, r, j, i);
        const bool ok_prev = valid_at(t, r, j - 1, ip), ok_next = valid_at(t, r, j + 1, inx);
        const float vj = (ok && mode != MODE_EXTEND) ? val[j] : 0.0f;
        if (!ok) continue;
        if (idx_out) idx_out[j] = i;
        if (mode == MODE_PRIORITY) bm = fmaxf(bm, fabsf(vj));
        const long long line = i >> 5;
        if (ok_prev && (ip >> 5) == line) continue;               // the line's leader does this entry
        float4 v[8];
        const float4 *src = reinterpret_cast<const float4 *>(leaf + (line << 5));
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = __ldcg(src + k);
        long long ii = i;
        float x = mode == MODE_RAW ? vj : (mode == MODE_PRIORITY ? pow_leaf(fabsf(vj), t) : defp);
        bool more = ok_next && (inx >> 5) == line;
        for (long long jj = j;;) {
            leaf[ii] = x;                                         // equal indices: the later entry overwrites (last wins)
            const int pos = (int)(ii & 31);
#pragma unroll
            for (int k = 0; k < 8; ++k) {                         // 32 selects: the line stays in registers
                v[k].x = pos == 4 * k ? x : v[k].x;
                v[k].y = pos == 4 * k + 1 ? x : v[k].y;
                v[k].z = pos == 4 * k + 2 ? x : v[k].z;
                v[k].w = pos == 4 * k + 3 ? x : v[k].w;
            }
            if (!more) break;
            ++jj;
            ii = jj == j + 1 ? inx : entry_index(t, idx, jj, mode, r.seq0);
            x = entry_leaf(t, val, jj, mode, defp);
            long long nx;
            more = valid_at(t, r, jj + 1, nx) && (nx >> 5) == line;
        }
        float vs, vm;
        line_total(v, line << 5, len, vs, vm);
        n1s[line] = vs; n1m[line] = vm;
    }
    if (mode == MODE_PRIORITY) cta_batch_max(t, bm);
    if (threadIdx.x == 0) trace_max(tr_on, TR_LINES_END);
}

// Any other batch (unsorted, duplicates, K batches in flight), after upd_mark_kernel: thread per ENTRY.  Every entry
// loads its leaf line (8 x 128-bit) and looks at the dedup tags in it: the entry whose tag sits in the LOWEST tagged
// slot of the line is the line's leader -- it resolves every tagged slot (a NaN-tagged slot names its winning entry:
// that entry's value is computed and stored), reduces the line and stores its node of level L-5; everybody else is
// done.  No side structure, no barrier, every lane of every warp works on a touched line (a pass over a touched-line
// bitmap spends its instructions on empty lines: 9 us at 64K entries against 4 us here, profiles/per_phases_r02.txt).
// Entries of one line may run at different times: a late one finds slots already resolved by the leader.  It is then
// either no leader (nothing to do) or the leader of what is left, and rebuilds the same node from the same final
// values -- stores of equal values, a benign race.
constexpr int LT_THREADS = 128;

__global__ void __launch_bounds__(LT_THREADS) upd_lines_tagged_kernel(TreeView t, long long n, const long long *idx,
                                                                      const float *val, int mode)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_LINES_START);
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long len = len_after(t, mode, n, -1);
    const float defp = (mode == MODE_EXTEND) ? default_priority(t) : 0.0f;
    float *leaf = leaf_ptr(t);
    __shared__ float4 wbuf_all[(LT_THREADS / 32) * 256];
    long long i = -1;
    if (j < n) i = entry_index(t, idx, j, mode, mode == MODE_EXTEND ? t.st->seq : 0);
    const bool live = i >= 0 && i < t.size;
    const long long line = live ? i >> 5 : 0;
    float4 v[8];                                                  // the line; NaN-tagged slots carry entry numbers
    warp_fetch_lines_raw(leaf, line, wbuf_all + (threadIdx.x >> 5) * 256, v);      // the warp's 32 lines, fetched together
    if (live) {
        unsigned tagged = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            tagged |= (__float_as_int(v[k].x) >= LEAF_TAG ? 1u : 0u) << (4 * k);
            tagged |= (__float_as_int(v[k].y) >= LEAF_TAG ? 1u : 0u) << (4 * k + 1);
            tagged |= (__float_as_int(v[k].z) >= LEAF_TAG ? 1u : 0u) << (4 * k + 2);
            tagged |= (__float_as_int(v[k].w) >= LEAF_TAG ? 1u : 0u) << (4 * k + 3);
        }
        // the slot at dynamic position p of the register copy (32 selects)
        auto slot = [&](int p) {
            float r = 0.0f;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                r = p == 4 * k ? v[k].x : r;
                r = p == 4 * k + 1 ? v[k].y : r;
                r = p == 4 * k + 2 ? v[k].z : r;
                r = p == 4 * k + 3 ? v[k].w : r;
            }
            return r;
        };
        const int p0 = __ffs(tagged) - 1;                         // -1: everything resolved already
        if (p0 >= 0 && __float_as_int(slot(p0)) == LEAF_TAG + (int)j) {       // my tag sits in the lowest tagged slot: leader
            while (tagged) {                                      // one or two per line; ONE copy of the entry code
                const int pos = __ffs(tagged) - 1;
                tagged &= tagged - 1;
                const int tag = __float_as_int(slot(pos));        // the tag this thread SAW in slot pos (its snapshot)
                const float nv = entry_leaf(t, val, (long long)(tag - LEAF_TAG), mode, defp);
                leaf[(line << 5) + pos] = nv;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    v[k].x = pos == 4 * k ? nv : v[k].x;
                    v[k].y = pos == 4 * k + 1 ? nv : v[k].y;
                    v[k].z = pos == 4 * k + 2 ? nv : v[k].z;
                    v[k].w = pos == 4 * k + 3 ? nv : v[k].w;
                }
            }
            float vs, vm;
            line_total(v, line << 5, len, vs, vm);
            sum_level(t, t.L - 5)[line] = vs;
            min_level(t, t.L - 5)[line] = vm;
        }
    }
    if (threadIdx.x == 0) trace_max(tr_on, TR_LINES_END);
}

// ---------------------------------------------------------------------------------
// prefix-sum descent: 8 lanes per sample (4 samples per warp), 5 levels per dependent 128-byte load: every lane
// loads 4 of the line's 32 nodes (one float4), two levels are reduced in registers and three with shuffles.  Same
// comparisons in the same order as the reference loop (go right and subtract iff mass > left).  All 32 lanes of the
// warp must call this together.  Returns the leaf index (or size when mass > root) and the leaf's value.
// ---------------------------------------------------------------------------------
template <int U>
__device__ __forceinline__ void group_descend_multi(const TreeView &t, float (&m)[U], long long (&node)[U],
                                                    float (&leafv)[U])
{
    // U independent descents per 8-lane group, interleaved level by level: U 128-byte loads in flight per group
    const int gl = threadIdx.x & 7;
    const float root = t.sum[1];
    bool over[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        over[u] = m[u] > root;
        if (over[u]) m[u] = 0.0f;                                 // stay on real nodes; the result is discarded
        node[u] = 0;                                              // index within the current level
        leafv[u] = 0.0f;
    }
    int d = 0;
    int c = t.L % 5;                                              // short chunk first: deeper chunks are full aligned lines
    if (c == 0) c = 5;
    while (d < t.L) {
        const int s = d + c;
        const float *lvl = sum_level(t, s);
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float *p = lvl + (node[u] << c);
            if (c == 5) {
                v[u] = *reinterpret_cast<const float4 *>(p + 4 * gl);
            } else {
                const int cnt = 1 << c, b = 4 * gl;
                v[u].x = b + 0 < cnt ? p[b + 0] : 0.0f; v[u].y = b + 1 < cnt ? p[b + 1] : 0.0f;
                v[u].z = b + 2 < cnt ? p[b + 2] : 0.0f; v[u].w = b + 3 < cnt ? p[b + 3] : 0.0f;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float a = op_sum(v[u].x, v[u].y), b2 = op_sum(v[u].z, v[u].w);
            const float c4 = op_sum(a, b2);
            const float s1 = op_sum(c4, __shfl_xor_sync(FULL, c4, 1, 8));
            const float s2 = op_sum(s1, __shfl_xor_sync(FULL, s1, 2, 8));
            float mm = m[u];
            int pos = 0;
            float l = __shfl_sync(FULL, s2, 0, 8);
            if (mm > l) { mm = __fsub_rn(mm, l); pos = 4; }
            l = __shfl_sync(FULL, s1, pos, 8);
            if (mm > l) { mm = __fsub_rn(mm, l); pos += 2; }
            l = __shfl_sync(FULL, c4, pos, 8);
            if (mm > l) { mm = __fsub_rn(mm, l); pos += 1; }
            const float la = __shfl_sync(FULL, a, pos, 8);
            const float lx = __shfl_sync(FULL, v[u].x, pos, 8), ly = __shfl_sync(FULL, v[u].y, pos, 8);
            const float lz = __shfl_sync(FULL, v[u].z, pos, 8), lw = __shfl_sync(FULL, v[u].w, pos, 8);
            int sub = 0;
            float l0 = lx, l1 = ly;
            if (mm > la) { mm = __fsub_rn(mm, la); sub = 2; l0 = lz; l1 = lw; }
            float lf = l0;
            if (mm > l0) { mm = __fsub_rn(mm, l0); sub += 1; lf = l1; }
            m[u] = mm;
            leafv[u] = lf;
            node[u] = (c == 5 ? (node[u] << 5) : 0) + 4 * pos + sub;
        }
        d = s;
        c = 5;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) if (over[u]) node[u] = t.size;
}

__device__ __forceinline__ long long group_descend(const TreeView &t, float m, float *leaf_out)
{
    float mm[1] = {m}, lf[1];
    long long nd[1];
    group_descend_multi<1>(t, mm, nd, lf);
    *leaf_out = lf[0];
    return nd[0];
}

// R sub-rounds of 4 descents each (one per 8-lane group): lane l = 4 sub + g hands its mass to group g in sub-round
// `sub` and collects the result.  R = 8 runs the sub-rounds four at a time (interleaved descents).
__device__ __forceinline__ void warp_descend_rounds(const TreeView &t, float m, int R, long long &mine, float &my_leaf)
{
    const int lane = lane_id();
    mine = 0; my_leaf = 0.0f;
    if (R == 8) {
#pragma unroll 1
        for (int sub = 0; sub < 8; sub += 4) {
            float mg[4], lf[4];
            long long nd[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) mg[u] = __shfl_sync(FULL, m, 4 * (sub + u) + (lane >> 3));
            group_descend_multi<4>(t, mg, nd, lf);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const long long gi = __shfl_sync(FULL, nd[u], (lane & 3) << 3);
                const float gf = __shfl_sync(FULL, lf[u], (lane & 3) << 3);
                if ((lane >> 2) == sub + u) { mine = gi; my_leaf = gf; }
            }
        }
    } else {
#pragma unroll 1
        for (int sub = 0; sub < R; ++sub) {
            const float mg = __shfl_sync(FULL, m, 4 * sub + (lane >> 3));
            float leafv;
            const long long i = group_descend(t, mg, &leafv);
            const long long gi = __shfl_sync(FULL, i, (lane & 3) << 3);
            const float gf = __shfl_sync(FULL, leafv, (lane & 3) << 3);
            if ((lane >> 2) == sub) { mine = gi; my_leaf = gf; }
        }
    }
}

__global__ void __launch_bounds__(256) tree_scan_kernel(TreeView t, long long n, const float *mass, long long *idx_out)
{
    const int lane = lane_id();
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long w0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long rounds = (n + 32 * n_warps - 1) / (32 * n_warps);
    for (long long rd = 0; rd < rounds; ++rd) {
        const long long k = (w0 + rd * n_warps) * 32 + lane;
        const float m = k < n ? mass[k] : 0.0f;
        long long mine;
        float my_leaf;
        warp_descend_rounds(t, m, 8, mine, my_leaf);
        if (k < n) idx_out[k] = mine;
    }
}

__device__ __forceinline__ float is_weight(float leaf, float p_min, float beta, const TreeView &t)
{
    float denom = t.weps ? __fadd_rn(p_min, t.eps32) : p_min;
    float ratio = __fdiv_rn(leaf, denom);
    // np.power(fp32, -beta) -> libm powf (< 1 ulp).  beta = 0.5 (the value the learner forces, learner.py:105-107):
    // hardware rsqrt + one Newton step in fp32 -- within 2 ulp of powf (the parity bar on IS weights is 1e-6 relative;
    // tests/test_gpu_per.py), a tenth of the instructions of the fp64 evaluation that every other beta takes.
    if (beta == 0.5f) {
        const float y = rsqrtf(ratio);
        return y * fmaf(-0.5f * ratio * y, y, 1.5f);
    }
    return (float)pow_cold((double)ratio, -(double)beta);
}

// device-side uniforms: philox_uniform / rng_advance (common.cuh), keyed by the state block's seed and call number

__device__ __forceinline__ float stratified_mass(long long k, double uk, long long n, float total)
{
    return (float)__dmul_rn(__ddiv_rn(__dadd_rn((double)k, uk), (double)n), (double)total);
}

// n = n_batches * batch samples; sample k belongs to batch k / batch, stratum k % batch of its batch (every batch
// is stratified on its own, all against the same tree state).  Persistent grid.  A warp takes 32 consecutive samples
// per round: every lane prepares ONE sample (uniform, fp64 mass), the descents run 4 at a time (8 lanes each, 8
// sub-rounds, masses and results handed over by shuffles), then every lane finishes its own sample (clamp, fp64
// importance weight) and the 32 results leave as coalesced stores.
// R sub-rounds per warp round (4 R samples per warp): 8 for large n (throughput), 1 for small batches (a warp then
// runs ONE descent chain, the latency of a single learner batch).
__global__ void __launch_bounds__(256) tree_sample_kernel(TreeView t, long long n, long long batch, const double *u,
                                                          int mode, float beta, long long *idx_out, float *w_out,
                                                          float *mass_out, int R)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const unsigned call = (unsigned)t.st->pad[2], seed = (unsigned)t.st->pad[3];
    const long long len = t.st->len;
    const float p_sum = t.st->p_sum, p_min = t.st->p_min;
    int bad = 0;
    if (len <= 0) bad = PB_ST_EMPTY;
    else if (!(p_sum > 0.0f)) bad = PB_ST_PSUM_NONPOS;
    else if (!(p_min > 0.0f)) bad = PB_ST_PMIN_NONPOS;
    const int lane = lane_id();
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long w0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int per_warp = 4 * R;
    const long long rounds = (n + per_warp * n_warps - 1) / (per_warp * n_warps);
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_SAMPLE_START);
    for (long long rd = 0; rd < rounds; ++rd) {
        const long long k = (w0 + rd * n_warps) * per_warp + lane;
        const bool live = lane < per_warp && k < n;
        if (bad) {
            if (live) {
                idx_out[k] = 0; w_out[k] = 0.0f;
                if (mass_out) mass_out[k] = 0.0f;
                if (k == 0) atomicOr(&t.st->status, bad);
            }
            continue;
        }
        float m = 0.0f;
        if (live) {
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            m = (mode == 0) ? (float)(0.0 + ((double)p_sum - 0.0) * uk) : stratified_mass(k % batch, uk, batch, p_sum);
        }
        long long mine;
        float my_leaf;
        warp_descend_rounds(t, m, R, mine, my_leaf);
        if (live) {
            if (mine > len - 1) { mine = len - 1; my_leaf = leaf_ptr(t)[mine]; }
            idx_out[k] = mine;
            w_out[k] = is_weight(my_leaf, p_min, beta, t);
            if (mass_out) mass_out[k] = m;
        }
    }
    if (threadIdx.x == 0) trace_max(tr_on, TR_SAMPLE_END);
    if (!u) { __syncthreads(); rng_advance(t.st); }
}

// ---------------------------------------------------------------------------------
// throughput mode (many batches in flight): one THREAD per sample.
//  * The CTA stages the top of the tree as a full level-ordered heap in shared memory: heap levels 0..TL copied, and
//    every thread streams one line of the stored level S = TL + 5 (<= 14) and rebuilds the four levels in between in
//    registers (bit-identical to a stored tree) -- one round trip, one barrier.  The first S levels of a descent then
//    cost one shared-memory load each.
//  * Every deeper stored level costs the thread one 128-byte line whose 5 levels it resolves in registers.  The warp
//    fetches its 32 lines TOGETHER: 4 lines per load instruction (8 lanes x 16 bytes each, one L1 wavefront per line
//    instead of eight when every lane streams its own line -- the unit that bounded the first version of this
//    kernel), transposed through 4 KB of shared memory per warp (XOR-swizzled 16-byte chunks, conflict-free both ways).
// Same comparisons in the same order as the reference loop and as group_descend: both modes return identical indices.
// ---------------------------------------------------------------------------------
constexpr int ST_THREADS = 512;

__device__ __forceinline__ void warp_fetch_lines(const float *__restrict__ lvl, long long node, float4 *wbuf, float (&v)[32])
{
    const int lane = lane_id();
    const int g = lane >> 3, c = lane & 7;
    float4 q[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const long long ln = __shfl_sync(FULL, node, 4 * r + g);
        q[r] = __ldg(reinterpret_cast<const float4 *>(lvl + (ln << 5)) + c);
    }
    __syncwarp();                                                 // everyone is done reading the previous level's lines
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int slot = 4 * r + g;
        wbuf[slot * 8 + (c ^ (slot & 7))] = q[r];
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float4 x = wbuf[lane * 8 + (k ^ (lane & 7))];
        v[4 * k] = x.x; v[4 * k + 1] = x.y; v[4 * k + 2] = x.z; v[4 * k + 3] = x.w;
    }
}

// one line (32 nodes of a stored level, children of `node`): go right and subtract iff mass > left, 5 times.  The three
// upper levels come from tree-order sums in registers (v: the line); the two lower ones from ONE 128-bit read of the
// line's copy that warp_fetch_lines left in shared memory (row: this lane's 8 swizzled chunks) -- a dynamic index is a
// shared-memory address, not a cascade of 37 selects.
__device__ __forceinline__ void thread_line_descend(const float (&v)[32], const float4 *row, long long &node, float &m,
                                                    float &leaf)
{
    float t16[16], t8[8], t4[4], t2[2];
#pragma unroll
    for (int i = 0; i < 16; ++i) t16[i] = op_sum(v[2 * i], v[2 * i + 1]);
#pragma unroll
    for (int i = 0; i < 8; ++i) t8[i] = op_sum(t16[2 * i], t16[2 * i + 1]);
#pragma unroll
    for (int i = 0; i < 4; ++i) t4[i] = op_sum(t8[2 * i], t8[2 * i + 1]);
#pragma unroll
    for (int i = 0; i < 2; ++i) t2[i] = op_sum(t4[2 * i], t4[2 * i + 1]);
    int pos = 0;
    float l = t2[0];
    if (m > l) { m = __fsub_rn(m, l); pos = 1; }
    l = pos ? t4[2] : t4[0];
    pos <<= 1;
    if (m > l) { m = __fsub_rn(m, l); pos |= 1; }
    {   // left child of node `pos` at the 4-node level: t8[2 pos]
        const float a = (pos & 1) ? t8[2] : t8[0], b = (pos & 1) ? t8[6] : t8[4];
        l = (pos & 2) ? b : a;
    }
    pos <<= 1;
    if (m > l) { m = __fsub_rn(m, l); pos |= 1; }
    // pos in 0..7 names the 128-bit chunk {v[4 pos] .. v[4 pos + 3]}: its two pairs are the last two levels
    const float4 c = row[pos ^ (lane_id() & 7)];
    l = op_sum(c.x, c.y);                                         // == t16[2 pos]
    float lo = c.x, hi = c.y;
    pos <<= 1;
    if (m > l) { m = __fsub_rn(m, l); pos |= 1; lo = c.z; hi = c.w; }
    pos <<= 1;
    leaf = lo;
    if (m > lo) { m = __fsub_rn(m, lo); pos |= 1; leaf = hi; }
    node = (node << 5) + pos;
}

__global__ void __launch_bounds__(ST_THREADS) tree_sample_thread_kernel(TreeView t, long long n, long long batch,
                                                                        const double *u, int mode, float beta,
                                                                        long long *idx_out, float *w_out,
                                                                        float *mass_out, int S)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    extern __shared__ float4 sh4[];
    float *sh = reinterpret_cast<float *>(sh4);                   // heap of levels 0..S: node i of level d at [2^d + i]
    float4 *wbuf = sh4 + ((2u << S) >> 2) + (threadIdx.x >> 5) * 256;     // this warp's 32 lines x 8 chunks
    const unsigned call = (unsigned)t.st->pad[2], seed = (unsigned)t.st->pad[3];
    const int TL = t.TL;                                          // S == TL + 5
    const int tr_on = TRACE_ON();
    trace_cta0(tr_on, TR_SAMPLE_START);
    for (int i = threadIdx.x; i < (2 << TL); i += blockDim.x) sh[i] = i ? __ldg(t.sum + i) : 0.0f;
    {
        // level S, coalesced: 128-bit word i holds nodes 4i .. 4i+3 of level S = 2 nodes of level S-1 = 1 node of level
        // S-2; neighbouring lanes hold neighbouring words, so levels S-3 and S-4 come from two shuffles.  Conflict-free
        // shared-memory stores; no barrier until everything is in place.
        const float4 *lv = reinterpret_cast<const float4 *>(sum_level(t, S));
        const int n4 = 1 << (S - 2);                              // 128-bit words of level S (a multiple of 32)
        float4 *d0 = reinterpret_cast<float4 *>(sh + (1 << S));
        float2 *d1 = reinterpret_cast<float2 *>(sh + (1 << (S - 1)));
        float *d2 = sh + (1 << (S - 2)), *d3 = sh + (1 << (S - 3)), *d4 = sh + (1 << (S - 4));
        const int lane = threadIdx.x & 31;
        for (int i0 = threadIdx.x; i0 < n4; i0 += 8 * blockDim.x) {
            float4 q[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = i0 + k * blockDim.x;
                q[k] = i < n4 ? __ldg(lv + i) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = i0 + k * blockDim.x;
                if (i - lane >= n4) break;                        // warp-uniform: whole warps are in or out (n4 % 32 == 0)
                const float a = op_sum(q[k].x, q[k].y), b = op_sum(q[k].z, q[k].w);
                const float c = op_sum(a, b);
                const float c2 = op_sum(c, __shfl_xor_sync(FULL, c, 1));
                const float c3 = op_sum(c2, __shfl_xor_sync(FULL, c2, 2));
                d0[i] = q[k];
                d1[i] = make_float2(a, b);
                d2[i] = c;
                if ((lane & 1) == 0) d3[i >> 1] = c2;
                if ((lane & 3) == 0) d4[i >> 2] = c3;
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) trace_max(tr_on, TR_SAMPLE_STAGED);
    const long long len = t.st->len;
    const float p_sum = t.st->p_sum, p_min = t.st->p_min;
    int bad = 0;
    if (len <= 0) bad = PB_ST_EMPTY;
    else if (!(p_sum > 0.0f)) bad = PB_ST_PSUM_NONPOS;
    else if (!(p_min > 0.0f)) bad = PB_ST_PMIN_NONPOS;
    const float root = sh[1];
    const bool batch_p2 = (batch & (batch - 1)) == 0;             // (k + u) / batch == (k + u) * (1 / batch) exactly
    const double inv_batch = 1.0 / (double)batch;
    // whole warps iterate together (the line fetch is a warp-wide operation); lanes past n ride along on node 0
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); k0 < n; k0 += stride) {
        const long long k = k0 + (threadIdx.x & 31);
        const bool live = k < n;
        if (bad) {
            if (live) {
                idx_out[k] = 0; w_out[k] = 0.0f;
                if (mass_out) mass_out[k] = 0.0f;
                if (k == 0) atomicOr(&t.st->status, bad);
            }
            continue;
        }
        float m0 = 0.0f;
        if (live) {
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            if (mode == 0) m0 = (float)(0.0 + ((double)p_sum - 0.0) * uk);
            else if (batch_p2) m0 = (float)__dmul_rn(__dmul_rn(__dadd_rn((double)(k & (batch - 1)), uk), inv_batch), (double)p_sum);
            else m0 = stratified_mass(k % batch, uk, batch, p_sum);
        }
        float m = m0;
        const bool over = m > root;
        if (over) m = 0.0f;
        int hn = 1;                                               // heap index in shared memory
        for (int d = 0; d < S; ++d) {
            hn <<= 1;
            const float left = sh[hn];
            if (m > left) { m = __fsub_rn(m, left); hn |= 1; }
        }
        long long node = hn - (1 << S);                           // index within level S
        float leafv = sh[hn];
        for (int s = S + 5; s <= t.L; s += 5) {
            float v[32];
            warp_fetch_lines(sum_level(t, s), node, wbuf, v);
            thread_line_descend(v, wbuf + (threadIdx.x & 31) * 8, node, m, leafv);
        }
        if (live) {
            long long i = over ? t.size : node;
            if (i > len - 1) { i = len - 1; leafv = leaf_ptr(t)[i]; }
            idx_out[k] = i;
            w_out[k] = is_weight(leafv, p_min, beta, t);
            if (mass_out) mass_out[k] = m0;
        }
    }
    if (threadIdx.x == 0) trace_max(tr_on, TR_SAMPLE_END);
    if (!u) { __syncthreads(); rng_advance(t.st); }
}

// ---------------------------------------------------------------------------------
// sharded global stratified sampling: the G shard roots are the leaves of a virtual
// top tree, summed pairwise in fp32 (so shards concatenated == one big tree).  ONE launch: masses are
// non-decreasing in the stratum number and the descent is monotone, so the strata a rank owns are a contiguous
// range [lo, lo + cnt) that every CTA finds by a warp-parallel 32-ary search (no counting pass, no atomics).
// ---------------------------------------------------------------------------------
constexpr int MAX_RANKS = 64;

struct GlobalTop {
    float psum[2 * MAX_RANKS];  // heap layout of the virtual top: leaves (shard p_sums) at [G, 2G)
    float pmin;
    long long lo, hi;           // this rank owns strata [lo, hi)
};

__device__ __forceinline__ void build_top(GlobalTop *g, const pb_per_state *all_state, int G)
{
    if (threadIdx.x < G) g->psum[G + threadIdx.x] = ld_state_f32(&all_state[threadIdx.x].p_sum);
    __syncthreads();
    for (int n = G >> 1; n >= 1; n >>= 1) {
        if (threadIdx.x < n) g->psum[n + threadIdx.x] = op_sum(g->psum[2 * (n + threadIdx.x)], g->psum[2 * (n + threadIdx.x) + 1]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        float m = ld_state_f32(&all_state[0].p_min);
        for (int r = 1; r < G; ++r) m = op_min(m, ld_state_f32(&all_state[r].p_min));
        g->pmin = m;
    }
    __syncthreads();
}

__device__ __forceinline__ int route_stratum(const GlobalTop &g, int G, long long k, long long n_global,
                                             double uk, float *residual)
{
    const float total = g.psum[1];
    float m = stratified_mass(k, uk, n_global, total);
    *residual = m;
    if (m > total) return G - 1;  // unreachable for u < 1; clamp like idx.clamp_max(len-1)
    int node = 1;
    while (node < G) {
        node <<= 1;
        float left = g.psum[node];
        if (m > left) { m = __fsub_rn(m, left); node |= 1; }
    }
    *residual = m;
    return node - G;
}

// first stratum k in [0, n] whose owner is >= rank_bound (n when there is none); one warp, 32-ary search over the
// monotone predicate owner(k) >= rank_bound
__device__ long long first_owned(const GlobalTop &g, int G, long long n, int rank_bound, const double *u,
                                 unsigned seed, unsigned call)
{
    const int lane = lane_id();
    long long lo = 0, hi = n;                                     // the answer lies in [lo, hi]
    while (lo < hi) {
        const long long step = (hi - lo + 31) / 32;
        const long long k = lo + (long long)lane * step;          // 32 probes, lo first
        bool ge = true;                                           // probes at or past hi count as "owned"
        if (k < hi) {
            float res;
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            ge = route_stratum(g, G, k, n, uk, &res) >= rank_bound;
        }
        const unsigned m = __ballot_sync(FULL, ge);
        if (m == 0u) { lo = lo + 31 * step + 1; continue; }       // all 32 probes below hi and none owned yet
        const int first = __ffs(m) - 1;
        if (first == 0) { hi = lo; break; }
        const long long k_first = lo + (long long)first * step;
        lo = k_first - step + 1;                                  // probe first-1 was not owned
        hi = k_first < hi ? k_first : hi;
    }
    return hi;
}

// peer wait (pb_tree_sample_global_peer): PeerWait / peer_wait_states, common.cuh
__global__ void __launch_bounds__(256) global_sample_kernel(TreeView t, const pb_per_state *all_state, int G, int rank,
                                                            long long n_global, const double *u, float beta,
                                                            long long *idx_out, float *w_out, long long *stratum_out,
                                                            int R, PeerWait pw)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    __shared__ GlobalTop g;
    if (pw.flags) all_state = peer_wait_states(pw, G);
    build_top(&g, all_state, G);
    const unsigned call = (unsigned)t.st->pad[2], seed = (unsigned)t.st->pad[3];
    if (threadIdx.x < 32) {
        const long long lo = first_owned(g, G, n_global, rank, u, seed, call);
        const long long hi = first_owned(g, G, n_global, rank + 1, u, seed, call);
        if (threadIdx.x == 0) { g.lo = lo; g.hi = hi; }
    }
    __syncthreads();
    const long long lo = g.lo, cnt = g.hi - g.lo;
    const long long len = ld_state_s64(&all_state[rank].len);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        t.st->owned_lo = (int)lo; t.st->owned_n = (int)cnt;
        if (cnt > 0 && (len <= 0 || !(g.psum[1] > 0.0f) || !(g.pmin > 0.0f)))
            atomicOr(&t.st->status, len <= 0 ? PB_ST_EMPTY : (!(g.psum[1] > 0.0f) ? PB_ST_PSUM_NONPOS : PB_ST_PMIN_NONPOS));
    }
    const int lane = lane_id();
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long w0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int per_warp = 4 * R;
    const long long rounds = (n_global + per_warp * n_warps - 1) / (per_warp * n_warps);
    for (long long rd = 0; rd < rounds; ++rd) {
        const long long pos = (w0 + rd * n_warps) * per_warp + lane;    // output row
        const bool mine_row = lane < per_warp;
        const bool live = mine_row && pos < cnt;
        float res = 0.0f;
        if (live) {
            const long long k = lo + pos;
            const double uk = u ? u[k] : philox_uniform(seed, call, (unsigned long long)k);
            route_stratum(g, G, k, n_global, uk, &res);
        }
        long long mine;
        float my_leaf;
        warp_descend_rounds(t, res, R, mine, my_leaf);
        if (mine_row && pos < n_global) {
            if (live) {
                if (mine > len - 1) { mine = len - 1; if (mine < 0) mine = 0; my_leaf = leaf_ptr(t)[mine]; }
                idx_out[pos] = mine;
                w_out[pos] = is_weight(my_leaf, g.pmin, beta, t);
                if (stratum_out) stratum_out[pos] = lo + pos;
            } else {                                              // padding rows of the static batch: skipped downstream
                idx_out[pos] = -1; w_out[pos] = 0.0f;
                if (stratum_out) stratum_out[pos] = -1;
            }
        }
    }
    if (!u) { __syncthreads(); rng_advance(t.st); }
}

// ---------------------------------------------------------------------------------
// export: the full level-ordered arrays (2 * capacity floats per tree) a pointer-walking tree would hold --
// parity tests and checkpoints.  One launch per level.
// ---------------------------------------------------------------------------------
__global__ void tree_export_kernel(TreeView t, int d, float *sum_heap, float *min_heap)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (1LL << d)) return;
    const long long len = t.st->len;
    if (sum_heap) sum_heap[(1LL << d) + i] = node_value<false>(t, d, i, len);
    if (min_heap) min_heap[(1LL << d) + i] = node_value<true>(t, d, i, len);
    if (d == 0 && i == 0) {
        if (sum_heap) sum_heap[0] = 0.0f;
        if (min_heap) min_heap[0] = INF;
    }
}

// ---------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------
struct Layout { int L, TL, P; long long off[MAX_DEEP]; long long n_sum, n_min, n_cnt; };

void make_layout(long long cap, Layout *y)
{
    y->L = pb_ilog2(cap);
    y->P = y->L <= TOP_MAX ? 0 : (y->L - TOP_MAX + 4) / 5;
    y->TL = y->L - 5 * y->P;
    long long off = 2LL << y->TL;
    for (int m = 0; m < MAX_DEEP; ++m) y->off[m] = 0;
    y->n_min = off;
    for (int m = 1; m <= y->P; ++m) {
        y->off[m] = off;
        off += 1LL << (y->TL + 5 * m);
        if (m < y->P) y->n_min = off;                             // the min store ends before the leaf level
    }
    y->n_sum = off;
    y->n_cnt = 32;                                                // reserved scratch (no kernel needs a side array any more)
}

int make_view(const pb_tree *t, TreeView *v)
{
    if (!t || !t->sum || !t->min || !t->state) return PB_E_ARG;
    if (!pb_is_pow2(t->capacity) || t->size <= 0 || t->size > t->capacity) return PB_E_CAPACITY;
    if (t->capacity < 32 || t->capacity > (1LL << 30)) return PB_E_CAPACITY;     // at least one 32-leaf line
    Layout y;
    make_layout(t->capacity, &y);
    if (!t->counters) return PB_E_ARG;
    v->sum = t->sum; v->min = t->min; v->owner = t->owner; v->cnt = t->counters; v->st = t->state;
    v->cap = t->capacity; v->size = t->size; v->L = y.L; v->TL = y.TL; v->P = y.P;
    for (int m = 0; m < MAX_DEEP; ++m) v->off[m] = y.off[m];
    v->alpha = t->alpha; v->eps32 = t->eps_f32; v->eps64 = t->eps_f64;
    v->weps = t->weight_eps_in_denominator; v->dp64 = t->default_priority_fp64;
    return PB_OK;
}

int persistent_grid(long long work_items, int per_cta, int ctas_per_sm)
{
    long long need = (work_items + per_cta - 1) / per_cta;
    long long cap = (long long)pb_sm_count() * ctas_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// every line of every deep level from level s_start (default: the leaves) up, then the top heap + state
// (streaming; ext: bulk build source)
int launch_rebuild(const TreeView &v, const float *ext, long long n_ext, int mode, long long n_new, long long set_len,
                   void *stream, int s_start = -1)
{
    if (s_start < 0) s_start = v.L;
    if (v.P == 0 || s_start <= v.TL) {
        if (ext) PB_LAUNCH_PDL(tree_fill_leaves_kernel, (unsigned)((v.cap + 255) / 256), 256, 0, stream, v, ext, n_ext);
        PB_LAUNCH_PDL(tree_top_kernel, 1, 512, 0, stream, v, mode, n_new, set_len);
        return PB_OK;
    }
    for (int s = s_start; s > v.TL;) {
        int n_lv = (s - v.TL) / 5;
        if (n_lv > 3) n_lv = 3;
        const int fuse = (s - 5 * n_lv <= v.TL) ? 1 : 0;
        const int grid = n_lv == 3 ? persistent_grid(1LL << s, 32 * RB_TILE, 4)
                                   : persistent_grid(1LL << s, RB_TILE * (RB_THREADS / 32), 8);
        PB_LAUNCH_PDL(tree_rebuild_kernel, grid, RB_THREADS, 0, stream, v, s, n_lv, s == v.L ? ext : (const float *)nullptr,
                  n_ext, fuse, mode, n_new, set_len);
        s -= 5 * n_lv;
    }
    return PB_OK;
}

int launch_update(const pb_tree *t, long long n, const long long *idx, const float *val, int mode, int sorted,
                  long long *idx_out, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (n < 0 || n >= (1LL << 31)) return PB_E_ARG;
    if (mode != MODE_EXTEND && (!idx || !val)) return n == 0 ? PB_OK : PB_E_ARG;
    if (n == 0) return PB_OK;
    if (mode == MODE_EXTEND) {
        if (n > v.size) return PB_E_ARG;
        sorted = (2 * n <= v.size);     // a contiguous run of slots; a long one may wrap onto lines it already touched
    }
    const int nb = (int)((n + 255) / 256);
    // Trees without a deep level (capacity <= 512): the leaves ARE the heap's bottom level.
    if (v.P == 0) {
        if (sorted) {
            PB_LAUNCH_PDL(upd_leaf_sorted_kernel, nb, 256, 0, stream, v, n, idx, val, mode, idx_out);
        } else {
            if (n > LEAF_TAG_MAX_N) return PB_E_UNSUPPORTED;
            PB_LAUNCH_PDL(upd_mark_kernel, nb, 256, 0, stream, v, n, idx, val, mode, idx_out);
            PB_LAUNCH_PDL(upd_leaf_kernel, nb, 256, 0, stream, v, n, idx, val, mode, (long long *)nullptr);
        }
        PB_LAUNCH_PDL(tree_top_kernel, 1, 512, 0, stream, v, mode, n, -1LL);
        return PB_OK;
    }
    // Three regimes, each a LINE phase (touched leaf lines -> nodes of level L-5) followed by the streaming rebuild of
    // the small tree above level L-5 (its last CTA rebuilds the top heap and the state block):
    //   (1) sorted batches (one learner batch, the ring's extends): the line leaders apply their runs -- 2 launches;
    //   (2) anything else below cap/16 entries: mark (dedup tags on the leaf slots), entry-driven lines -- 3 launches;
    //   (3) beyond that: scatter the leaves and stream the whole leaf array.
    if (sorted && n <= SORTED_LINES_MAX_N) {
        const int grid = (int)((n + LS_THREADS - 1) / LS_THREADS);
        PB_LAUNCH_PDL(upd_lines_sorted_kernel, grid, LS_THREADS, 0, stream, v, n, idx, val, mode, idx_out);
        return launch_rebuild(v, nullptr, 0, mode, n, -1, stream, v.L - 5);
    }
    if (n < v.cap / 16 && n <= LEAF_TAG_MAX_N) {
        PB_LAUNCH_PDL(upd_mark_kernel, nb, 256, 0, stream, v, n, idx, val, mode, idx_out);
        PB_LAUNCH_PDL(upd_lines_tagged_kernel, (int)((n + LT_THREADS - 1) / LT_THREADS), LT_THREADS, 0, stream, v, n, idx, val,
                      mode);
        return launch_rebuild(v, nullptr, 0, mode, n, -1, stream, v.L - 5);
    }
    if (sorted) {
        PB_LAUNCH_PDL(upd_leaf_sorted_kernel, nb, 256, 0, stream, v, n, idx, val, mode, idx_out);
    } else {
        if (n > LEAF_TAG_MAX_N) return PB_E_UNSUPPORTED;        // the dedup tags are NaN payloads: 2^23 - 2 of them
        PB_LAUNCH_PDL(upd_mark_kernel, nb, 256, 0, stream, v, n, idx, val, mode, idx_out);
        PB_LAUNCH_PDL(upd_leaf_kernel, nb, 256, 0, stream, v, n, idx, val, mode, (long long *)nullptr);
    }
    return launch_rebuild(v, nullptr, 0, mode, n, -1, stream);
}

}  // namespace

extern "C" {

int pb_tree_layout(long long capacity, long long *sum_floats, long long *min_floats, long long *counter_ints,
                   long long *leaf_offset, int *top_level)
{
    if (!pb_is_pow2(capacity) || capacity < 32 || capacity > (1LL << 30)) return PB_E_CAPACITY;
    Layout y;
    make_layout(capacity, &y);
    if (sum_floats) *sum_floats = y.n_sum;
    if (min_floats) *min_floats = y.n_min;
    if (counter_ints) *counter_ints = y.n_cnt;
    if (leaf_offset) *leaf_offset = y.P == 0 ? (1LL << y.L) : y.off[y.P];
    if (top_level) *top_level = y.TL;
    return PB_OK;
}

int pb_tree_init(const pb_tree *t, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (!t->counters) return PB_E_ARG;
    Layout y;
    make_layout(t->capacity, &y);
    int nb = pb_sm_count() * 8;
    PB_LAUNCH(tree_init_kernel, nb, 256, 0, stream, v, y.n_sum, y.n_min, y.n_cnt);
    return PB_OK;
}

int pb_tree_stats(const pb_tree *t, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    PB_LAUNCH(tree_stats_kernel, 1, 32, 0, stream, v);
    return PB_OK;
}

int pb_tree_build(const pb_tree *t, const float *leaves, long long n, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (!leaves || n < 0 || n > v.size) return PB_E_ARG;
    return launch_rebuild(v, leaves, n, MODE_RAW, 0, n, stream);
}

int pb_tree_set_leaves(const pb_tree *t, long long n, const long long *idx, const float *leaves, int sorted,
                       void *stream)
{
    return launch_update(t, n, idx, leaves, MODE_RAW, sorted, nullptr, stream);
}

int pb_tree_update_priority(const pb_tree *t, long long n, const long long *idx, const float *priority,
                            int sorted, void *stream)
{
    return launch_update(t, n, idx, priority, MODE_PRIORITY, sorted, nullptr, stream);
}

int pb_tree_extend(const pb_tree *t, long long n, long long *idx_out, void *stream)
{
    return launch_update(t, n, nullptr, nullptr, MODE_EXTEND, 1, idx_out, stream);
}

int pb_tree_scan(const pb_tree *t, long long n, const float *mass, long long *idx_out, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (n < 0 || (n > 0 && (!mass || !idx_out))) return PB_E_ARG;
    if (n == 0) return PB_OK;
    PB_LAUNCH(tree_scan_kernel, persistent_grid(n, 256, 6), 256, 0, stream, v, n, mass, idx_out);
    return PB_OK;
}

int pb_tree_sample_batches(const pb_tree *t, long long n_batches, long long batch, const double *u, int mode,
                           float beta, long long *idx_out, float *weight_out, float *mass_out, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (n_batches < 0 || batch < 0 || (mode != 0 && mode != 1)) return PB_E_ARG;
    const long long n = n_batches * batch;
    if (n >= (1LL << 31) || (n > 0 && (!idx_out || !weight_out))) return PB_E_ARG;
    if (n == 0) return PB_OK;
    if (n > 16384 && v.L >= 10) {
        // throughput mode: a thread per sample over a shared-memory heap of the top S = TL + 5 (<= 14) levels
        const int S = v.TL + 5;
        const size_t smem = sizeof(float) * (2ull << S) + (ST_THREADS / 32) * 4096;      // top heap + a line buffer per warp
        static PbPerDeviceOnce attr_set;
        if (!attr_set.done()) {
            cudaError_t e = cudaFuncSetAttribute(tree_sample_thread_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(sizeof(float) * (2ull << 14) + (ST_THREADS / 32) * 4096));
            if (e != cudaSuccess) return (int)e;
            attr_set.mark();
        }
        const int per_sm = smem > 100 * 1024 ? 1 : 2;
        PB_LAUNCH_PDL(tree_sample_thread_kernel, persistent_grid(n, ST_THREADS, per_sm), ST_THREADS, smem, stream, v, n, batch, u,
                  mode, beta, idx_out, weight_out, mass_out, S);
        return PB_OK;
    }
    // one learner batch: one 8-lane descent chain per group, 4 samples per warp (latency)
    const int R = 1;
    const int sgrid = persistent_grid(n, 8 * 4 * R, 6);
    PB_LAUNCH_PDL(tree_sample_kernel, sgrid, 256, 0, stream, v, n, batch, u, mode, beta, idx_out, weight_out, mass_out, R);
    return PB_OK;
}

int pb_tree_sample(const pb_tree *t, long long n, const double *u, int mode, float beta, long long *idx_out,
                   float *weight_out, float *mass_out, void *stream)
{
    return pb_tree_sample_batches(t, n > 0 ? 1 : 0, n, u, mode, beta, idx_out, weight_out, mass_out, stream);
}

int pb_tree_sample_global(const pb_tree *t, int n_ranks, int rank, const pb_per_state *all_state,
                          long long n_global, const double *u, float beta, long long *idx_out,
                          float *weight_out, long long *stratum_out, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (n_ranks < 1 || n_ranks > MAX_RANKS || !pb_is_pow2(n_ranks) || rank < 0 || rank >= n_ranks) return PB_E_ARG;
    if (!all_state || n_global < 0) return PB_E_ARG;
    if (n_global > 0 && (!idx_out || !weight_out)) return PB_E_ARG;
    if (n_global == 0) return PB_OK;
    const int R = n_global <= 16384 ? 1 : 8;
    PeerWait pw = {};
    PB_LAUNCH_PDL(global_sample_kernel, persistent_grid(n_global, 8 * 4 * R, 6), 256, 0, stream, v, all_state, n_ranks, rank,
              n_global, u, beta, idx_out, weight_out, stratum_out, R, pw);
    return PB_OK;
}

int pb_tree_sample_global_peer(const pb_tree *t, const pb_peer_group *g, long long n_global, const double *u, float beta,
                               long long *idx_out, float *weight_out, long long *stratum_out, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (!g || g->world < 1 || g->world > PB_PEER_MAX || !pb_is_pow2(g->world) || g->rank < 0 || g->rank >= g->world)
        return PB_E_ARG;
    if (!g->flags[g->rank] || !g->state[g->rank] || !g->epoch || n_global < 0) return PB_E_ARG;
    if (n_global > 0 && (!idx_out || !weight_out)) return PB_E_ARG;
    if (n_global == 0) return PB_OK;
    const int R = n_global <= 16384 ? 1 : 8;
    PeerWait pw;
    pw.flags = g->flags[g->rank] + 2 * PB_PEER_MAX;
    pw.epoch = g->epoch + 2;
    pw.slots = g->state[g->rank];
    pw.status = g->status;
    pw.timeout_ns = g->timeout_ns;
    pw.slot_bytes = PB_PEER_MAX * 64;
    PB_LAUNCH_PDL(global_sample_kernel, persistent_grid(n_global, 8 * 4 * R, 6), 256, 0, stream, v,
                  (const pb_per_state *)nullptr, g->world, g->rank, n_global, u, beta, idx_out, weight_out, stratum_out, R, pw);
    return PB_OK;
}

int pb_tree_trace(int enable, unsigned long long *out, int n_out)
{
    // synchronous (measurement runs only): copy out the marks, clear them, switch marking on / off
    unsigned long long host[TRACE_SLOTS];
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyFromSymbol(host, g_trace, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    if (out) for (int k = 0; k < n_out && k < TRACE_SLOTS; ++k) out[k] = host[k];
    for (int k = 0; k < TRACE_SLOTS; ++k) host[k] = 0;
    e = cudaMemcpyToSymbol(g_trace, host, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    const int on = enable ? 1 : 0;
    e = cudaMemcpyToSymbol(g_trace_on, &on, sizeof(on));
    return e == cudaSuccess ? PB_OK : (int)e;
}

int pb_tree_export(const pb_tree *t, float *sum_heap, float *min_heap, void *stream)
{
    TreeView v;
    int rc = make_view(t, &v);
    if (rc) return rc;
    if (!sum_heap && !min_heap) return PB_E_ARG;
    for (int d = v.L; d >= 0; --d)
        PB_LAUNCH(tree_export_kernel, (unsigned)(((1LL << d) + 255) / 256), 256, 0, stream, v, d, sum_heap, min_heap);
    return PB_OK;
}

}  // extern "C"
