// conv.cu -- MinAtar embedding network as one launch: conv3x3 (stride 1, no padding) on a
// channels-last observation + bias + ReLU + NCHW flatten (sm_100a).
//
// Reference: MinAtarModel (prism/agents/models/minatar_cnn_model.py:13-18, 41-44):
//     x.permute(0,3,1,2) -> Conv2d(C,16,3,1) -> ReLU -> Flatten.
// Through PyTorch/cuDNN that is 5 launches forward (layout copy, NHWC conv engine, bias add, clamp,
// flatten copy) and ~8 backward for a 14 MFLOP problem.  Here: one CTA per observation holds the
// 10x10xC frame and the whole filter bank in shared memory.  The observation needs no gradient
// (it comes from the replay ring), so backward is only dW / db: one CTA per group of samples
// accumulates its share in registers, partial sums are combined by a second tiny launch in a fixed
// order (deterministic).
#include "common.cuh"

namespace {

using namespace pb;

constexpr int MAX_X = 16 * 16 * 16;      // floats of one frame in smem
constexpr int MAX_W = 32 * 16 * 9;       // floats of the filter bank in smem
constexpr int MAX_OUT = 32 * 14 * 14;

struct ConvDims { int B, H, W, C, OC, OH, OW; };

// One CTA per observation.  Shared memory: the frame and the filter bank transposed to
// [c][ky][kx][oc] so that a thread reads the OCG = 8 consecutive output channels of one tap as two
// float4.  Thread = (output position, group of 8 output channels): 1 frame load feeds 8 FMAs.
// The frame is staged channel-major with its rows pitched to frame_pitch(W) words ([c][y][pitch]): the lanes of a warp
// are 32 consecutive output positions (4 rows of 8 for MinAtar) reading one tap, and with a pitch of 8 mod 16 those
// rows land on disjoint banks.  Channels-last as in global memory ((y*W + x)*C + c) the same read was 2-4-way
// conflicted, and the conflicts -- not the FMAs -- set this kernel's time (three of them run concurrently per step).
constexpr int OCG = 8;

__host__ __device__ inline int frame_pitch(int W) { return ((W + 7) / 16) * 16 + 8; }   // smallest >= W with pitch % 16 == 8

// channels-last word i of a frame -> its word in the staged layout.  mC, mW = div_magic(C), div_magic(W): the staging
// loop maps 8 words per thread, and two runtime divisions each were a third of the forward kernel's instructions.
// n / d == umulhi(n, magic) for 2 <= d, n < 2^32 / d.  d = 1 would need 2^32: the magic wraps to 0.
__device__ __forceinline__ unsigned div_magic(int d) { return 0xFFFFFFFFu / (unsigned)d + 1u; }
__device__ __forceinline__ int frame_slot(int i, int H, int W, int C, int P, unsigned mC, unsigned mW)
{
    // W >= 3 always; a one-channel frame (C = 1) is its own pixel index
    const int pix = C == 1 ? i : (int)__umulhi((unsigned)i, mC), c = i - pix * C;
    const int y = (int)__umulhi((unsigned)pix, mW), x = pix - y * W;
    return (c * H + y) * P + x;
}

__global__ void __launch_bounds__(256) conv3x3_relu_fwd_kernel(ConvDims d, const float *__restrict__ x,
                                                               const float *__restrict__ w,
                                                               const float *__restrict__ bias, float *__restrict__ out)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    extern __shared__ __align__(16) float sm[];
    const int nx = d.H * d.W * d.C, ocp = (d.OC + OCG - 1) / OCG * OCG, taps = d.C * 9;
    const int P = frame_pitch(d.W), cstride = d.H * P;
    const unsigned mC = div_magic(d.C), mW = div_magic(d.W), mO = div_magic(ocp);
    float *sw = sm, *sx = sm + taps * ocp;               // sw first: keeps it 16-byte aligned
    const int b = blockIdx.x;
    const float *xb = x + (size_t)b * nx;
    // staging with every global load requested before the first shared-memory store (a load -> store loop of up to 7
    // dependent round trips per thread was a third of this kernel)
    {
        const int nwp = taps * ocp;
        for (int i0 = threadIdx.x; i0 < nx || i0 < nwp; i0 += 8 * blockDim.x) {
            float fx[8], fw[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                fx[u] = i < nx ? xb[i] : 0.0f;
                const int tap = (int)__umulhi((unsigned)i, mO), oc = i - tap * ocp;     // tap = c*9 + ky*3 + kx
                fw[u] = (i < nwp && oc < d.OC) ? w[oc * taps + tap] : 0.0f;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i < nx) sx[frame_slot(i, d.H, d.W, d.C, P, mC, mW)] = fx[u];
                if (i < nwp) sw[i] = fw[u];
            }
        }
    }
    __syncthreads();
    const int plane = d.OH * d.OW, groups = ocp / OCG;
    float *ob = out + (size_t)b * d.OC * plane;
    for (int item = threadIdx.x; item < plane * groups; item += blockDim.x) {
        const int g = item / plane, p = item - g * plane, y = p / d.OW, xx = p - y * d.OW;
        float acc[OCG];
#pragma unroll
        for (int q = 0; q < OCG; ++q) acc[q] = 0.0f;
        for (int ky = 0; ky < 3; ++ky)
            for (int kx = 0; kx < 3; ++kx) {
                const float *px = sx + (y + ky) * P + (xx + kx);
                for (int c = 0; c < d.C; ++c) {
                    const float v = px[c * cstride];
                    const float4 *wv = reinterpret_cast<const float4 *>(sw + (c * 9 + ky * 3 + kx) * ocp + g * OCG);
                    const float4 w0 = wv[0], w1 = wv[1];
                    acc[0] = fmaf(v, w0.x, acc[0]); acc[1] = fmaf(v, w0.y, acc[1]);
                    acc[2] = fmaf(v, w0.z, acc[2]); acc[3] = fmaf(v, w0.w, acc[3]);
                    acc[4] = fmaf(v, w1.x, acc[4]); acc[5] = fmaf(v, w1.y, acc[5]);
                    acc[6] = fmaf(v, w1.z, acc[6]); acc[7] = fmaf(v, w1.w, acc[7]);
                }
            }
#pragma unroll
        for (int q = 0; q < OCG; ++q) {
            const int oc = g * OCG + q;
            if (oc < d.OC) ob[oc * plane + p] = fmaxf(acc[q] + (bias ? bias[oc] : 0.0f), 0.0f);
        }
    }
}

// partial[g][e], e in [0, OC*C*9) = dW, e in [OC*C*9, OC*C*9+OC) = db, for the samples of CTA g.
// Thread -> (tap, output channel) with the CHANNEL fastest, and the masked output gradient staged position-major
// ([p][oc]): the threads of a warp read consecutive words of the gradient and one or two broadcast words of the frame per
// tap -- both shared-memory reads of the inner FMA are conflict-free (element-major threads over a channel-major
// gradient strided the frame reads by 6 and 60 words: 17 us on the step's critical path).
__global__ void __launch_bounds__(512) conv3x3_relu_bwd_kernel(ConvDims d, const float *__restrict__ x,
                                                               const float *__restrict__ out,
                                                               const float *__restrict__ dout,
                                                               float *__restrict__ partial)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    extern __shared__ float sm[];
    const int nx = d.H * d.W * d.C, plane = d.OH * d.OW, n_out = d.OC * plane;
    float *sx = sm, *sg = sm + nx;                           // sg[p * OC + oc]
    const int taps = d.C * 9, nw = d.OC * taps, ne = nw + d.OC;
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.0f;
    for (int b = blockIdx.x; b < d.B; b += gridDim.x) {
        __syncthreads();
        const float *xb = x + (size_t)b * nx;
        for (int i = threadIdx.x; i < nx; i += blockDim.x) sx[i] = xb[i];
        const float *ob = out + (size_t)b * n_out, *gb = dout + (size_t)b * n_out;
        for (int i = threadIdx.x; i < n_out; i += blockDim.x) {
            const int oc = i / plane, p = i - oc * plane;
            sg[p * d.OC + oc] = ob[i] > 0.0f ? gb[i] : 0.0f;  // ReLU mask
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int u = threadIdx.x + q * blockDim.x;      // u = tap * OC + oc for the weights, nw + oc for the bias
            if (u >= ne) break;
            float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
            if (u < nw) {
                const int tap = u / d.OC, oc = u - tap * d.OC, c = tap / 9, k = tap - c * 9, ky = k / 3, kx = k - ky * 3;
                const float *g = sg + oc;
                for (int y = 0; y < d.OH; ++y) {
                    const float *gy = g + y * d.OW * d.OC, *xy = sx + ((y + ky) * d.W + kx) * d.C + c;
                    int xx = 0;
                    for (; xx + 3 < d.OW; xx += 4) {
                        a0 = fmaf(gy[xx * d.OC], xy[xx * d.C], a0);
                        a1 = fmaf(gy[(xx + 1) * d.OC], xy[(xx + 1) * d.C], a1);
                        a2 = fmaf(gy[(xx + 2) * d.OC], xy[(xx + 2) * d.C], a2);
                        a3 = fmaf(gy[(xx + 3) * d.OC], xy[(xx + 3) * d.C], a3);
                    }
                    for (; xx < d.OW; ++xx) a0 = fmaf(gy[xx * d.OC], xy[xx * d.C], a0);
                }
            } else {
                const float *g = sg + (u - nw);
                int p = 0;
                for (; p + 3 < plane; p += 4) {
                    a0 += g[p * d.OC]; a1 += g[(p + 1) * d.OC]; a2 += g[(p + 2) * d.OC]; a3 += g[(p + 3) * d.OC];
                }
                for (; p < plane; ++p) a0 += g[p * d.OC];
            }
            acc[q] += (a0 + a1) + (a2 + a3);
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int u = threadIdx.x + q * blockDim.x;
        if (u >= ne) break;
        // back to the weight layout (OC, C, 3, 3): e = oc * taps + tap
        int e = u;
        if (u < nw) { const int tap = u / d.OC, oc = u - tap * d.OC; e = oc * taps + tap; }
        partial[(size_t)blockIdx.x * ne + e] = acc[q];
    }
}

// ---------------------------------------------------------------------------------
// Backward on the tensor cores, 16 output channels (every MinAtar embedding): for one sample
//     dW[oc][tap] = sum_p dY[oc][p] * Xcol[p][tap],   db[oc] = sum_p dY[oc][p]
// is a 16 x (taps + 1) x (OH*OW) product (the bias is one more column, of ones): m16n8k8 3xTF32 MMAs -- the masked
// gradient is the A operand (rows padded to 68 words: conflict-free fragment loads), the frame is gathered into B
// fragments through two small offset tables (position -> frame word, tap -> frame word).  One CTA of 4 warps per
// sample: staged together (8 rounds of loads in flight), the warps split the n-tiles.  ~0.2 MFLOP per sample: the FMA
// kernel above spends its time on 2 shared-memory reads per FMA.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void conv_mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2])
{
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void conv_split_tf32(float x, uint32_t &hi, uint32_t &lo)
{
    hi = __float_as_uint(x) & 0xFFFFE000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}

constexpr int CM_WARPS = 4;                 // warps per CTA: they share one sample and split its n-tiles
constexpr int CM_MAX_NT = 12;               // n-tiles of 8 columns: taps + 1 <= 96 (C <= 10)
constexpr int CM_GSTRIDE = 68;              // words per gradient row in shared memory

template <int NT>
__global__ void __launch_bounds__(CM_WARPS * 32) conv3x3_relu_bwd_mma_kernel(ConvDims d, const float *__restrict__ x,
                                                                            const float *__restrict__ out,
                                                                            const float *__restrict__ dout,
                                                                            float *__restrict__ partial, int n_groups)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    extern __shared__ float sm[];
    constexpr int NTW = (NT + CM_WARPS - 1) / CM_WARPS;            // n-tiles per warp
    const int nx = d.H * d.W * d.C, plane = d.OH * d.OW, taps = d.C * 9, ne = 16 * taps + 16;
    const int P = frame_pitch(d.W), cstride = d.H * P;            // frame staged [c][y][pitch]: see frame_pitch
    const unsigned mC = div_magic(d.C), mW = div_magic(d.W);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gq = lane >> 2, tq = lane & 3;
    float *sx = sm, *sg = sx + cstride * d.C;
    // offset tables: pos_off[p] = frame word of output position p's window origin; tap_off[tap] = frame word of the
    // tap inside the window, -1 for the bias column, -2 past it
    int *pos_off = reinterpret_cast<int *>(sg + 16 * CM_GSTRIDE), *tap_off = pos_off + plane;
    for (int p = threadIdx.x; p < plane; p += blockDim.x) pos_off[p] = (p / d.OW) * P + (p % d.OW);
    for (int tp = threadIdx.x; tp < NT * 8; tp += blockDim.x) {
        int v = -2;
        if (tp < taps) { const int c = tp / 9, k = tp - c * 9; v = c * cstride + (k / 3) * P + (k % 3); }
        else if (tp == taps) v = -1;
        tap_off[tp] = v;
    }
    float cf[NTW][4];
#pragma unroll
    for (int j = 0; j < NTW; ++j) cf[j][0] = cf[j][1] = cf[j][2] = cf[j][3] = 0.0f;
    const int g = blockIdx.x;                                      // this CTA's partial
    for (int b = g; b < d.B; b += n_groups) {
        __syncthreads();
        const float *xb = x + (size_t)b * nx, *ob = out + (size_t)b * 16 * plane, *gb = dout + (size_t)b * 16 * plane;
        // staging with the loads of 8 rounds in flight
        for (int i0 = threadIdx.x; i0 < nx; i0 += 8 * blockDim.x) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; v[u] = i < nx ? xb[i] : 0.0f; }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i < nx) sx[frame_slot(i, d.H, d.W, d.C, P, mC, mW)] = v[u];
            }
        }
        for (int i0 = threadIdx.x; i0 < 16 * plane; i0 += 8 * blockDim.x) {
            float vo[8], vg[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                vo[u] = i < 16 * plane ? ob[i] : 0.0f;
                vg[u] = i < 16 * plane ? gb[i] : 0.0f;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i < 16 * plane) {
                    const int oc = i / plane, p = i - oc * plane;
                    sg[oc * CM_GSTRIDE + p] = vo[u] > 0.0f ? vg[u] : 0.0f;   // ReLU mask
                }
            }
        }
        __syncthreads();
        int toff[NTW];
#pragma unroll
        for (int j = 0; j < NTW; ++j) { const int nt = warp + j * CM_WARPS; toff[j] = nt < NT ? tap_off[nt * 8 + gq] : -2; }
        for (int k0 = 0; k0 < plane; k0 += 8) {
            uint32_t ah[4], al[4];
            conv_split_tf32(sg[gq * CM_GSTRIDE + k0 + tq], ah[0], al[0]);
            conv_split_tf32(sg[(gq + 8) * CM_GSTRIDE + k0 + tq], ah[1], al[1]);
            conv_split_tf32(sg[gq * CM_GSTRIDE + k0 + tq + 4], ah[2], al[2]);
            conv_split_tf32(sg[(gq + 8) * CM_GSTRIDE + k0 + tq + 4], ah[3], al[3]);
            const int p0 = pos_off[k0 + tq], p1 = pos_off[k0 + tq + 4];
#pragma unroll
            for (int j = 0; j < NTW; ++j) {
                if (warp + j * CM_WARPS >= NT) break;              // warp-uniform
                const int to = toff[j];
                const float b0 = to >= 0 ? sx[p0 + to] : (to == -1 ? 1.0f : 0.0f);
                const float b1 = to >= 0 ? sx[p1 + to] : (to == -1 ? 1.0f : 0.0f);
                uint32_t bh[2], bl[2];
                conv_split_tf32(b0, bh[0], bl[0]);
                conv_split_tf32(b1, bh[1], bl[1]);
                conv_mma_tf32(cf[j], al, bh);
                conv_mma_tf32(cf[j], ah, bl);
                conv_mma_tf32(cf[j], ah, bh);
            }
        }
    }
    if (g < n_groups) {
        // fragment (row gq / gq + 8 = output channel, columns 2 tq, 2 tq + 1 of n-tile nt = tap) -> partial[g][e]:
        // e = oc * taps + tap for the weights, 16 * taps + oc for the bias column
        float *pg = partial + (size_t)g * ne;
#pragma unroll
        for (int j = 0; j < NTW; ++j) {
            const int nt = warp + j * CM_WARPS;
            if (nt >= NT) break;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int oc = gq + (q >> 1) * 8, tp = nt * 8 + 2 * tq + (q & 1);
                if (tp < taps) pg[oc * taps + tp] = cf[j][q];
                else if (tp == taps) pg[16 * taps + oc] = cf[j][q];
            }
        }
    }
}

// one warp per gradient element: lanes stride over the per-CTA partials, fixed-order shuffle reduction
__global__ void __launch_bounds__(256) conv_bwd_reduce_kernel(int n_groups, int nw, int n_bias,
                                                              const float *__restrict__ partial,
                                                              float *__restrict__ dw, float *__restrict__ db)
{
    pdl_wait();                                                   // programmatic dependent launch (PB_LAUNCH_PDL)
    pdl_trigger();
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, ne = nw + n_bias;
    if (e >= ne) return;
    float a = 0.0f;
    for (int g = lane_id(); g < n_groups; g += 32) a += partial[(size_t)g * ne + e];
    a = warp_sum(a);
    if (lane_id() == 0) {
        if (e < nw) dw[e] = a; else if (db) db[e - nw] = a;
    }
}

// dynamic shared memory of the forward and of the FMA backward (the tensor-core backward is a fast path: a shape it
// cannot stage takes the FMA kernel, so its own limit never refuses a shape)
size_t fwd_smem(const ConvDims &d)
{
    const int ocp = (d.OC + OCG - 1) / OCG * OCG;
    return sizeof(float) * (size_t)(d.H * frame_pitch(d.W) * d.C + ocp * d.C * 9);
}
size_t fma_bwd_smem(const ConvDims &d) { return sizeof(float) * (size_t)(d.H * d.W * d.C + d.OC * d.OH * d.OW); }

// every limit of both entries: pb_conv3x3_relu_supported answers with the same function, so they cannot drift apart
int check_dims(const ConvDims &d)
{
    if (d.B <= 0 || d.H < 3 || d.W < 3 || d.C <= 0 || d.OC <= 0) return PB_E_ARG;
    const long long H = d.H, W = d.W, C = d.C, OC = d.OC;          // no int overflow for absurd arguments
    if (H * W * C > MAX_X || OC * C * 9 > MAX_W || OC * (H - 2) * (W - 2) > MAX_OUT) return PB_E_UNSUPPORTED;
    if (OC * C * 9 + OC > 8 * 256) return PB_E_UNSUPPORTED;         // FMA backward: 8 gradient elements per thread
    if (fwd_smem(d) > 48 * 1024 || fma_bwd_smem(d) > 48 * 1024) return PB_E_UNSUPPORTED;
    return PB_OK;
}

}  // namespace

extern "C" {

int pb_conv3x3_relu_supported(int H, int W, int C, int OC)
{
    const ConvDims d = {1, H, W, C, OC, H - 2, W - 2};
    return check_dims(d) == PB_OK ? 1 : 0;
}

int pb_conv3x3_relu_fwd(int B, int H, int W, int C, int OC, const float *x, const float *w, const float *bias,
                        float *out, void *stream)
{
    ConvDims d = {B, H, W, C, OC, H - 2, W - 2};
    int rc = check_dims(d);
    if (rc) return rc;
    if (!x || !w || !out) return PB_E_ARG;
    const int ocp = (OC + 7) / 8 * 8;
    const size_t smem = fwd_smem(d);
    const int items = d.OH * d.OW * (ocp / 8);
    const int threads = items >= 256 ? 256 : (items + 31) / 32 * 32;
    PB_LAUNCH(conv3x3_relu_fwd_kernel, (unsigned)B, threads, smem, stream, d, x, w, bias, out);
    return PB_OK;
}

int pb_conv3x3_relu_bwd_groups(int B) { return B < 296 ? B : 296; }

int pb_conv3x3_relu_bwd(int B, int H, int W, int C, int OC, const float *x, const float *out, const float *dout,
                        float *partial_scratch, float *dw, float *db, void *stream)
{
    ConvDims d = {B, H, W, C, OC, H - 2, W - 2};
    int rc = check_dims(d);
    if (rc) return rc;
    if (!x || !out || !dout || !partial_scratch || !dw) return PB_E_ARG;
    const int groups = pb_conv3x3_relu_bwd_groups(B);
    const int ne = OC * C * 9 + OC;
    // 16 output channels, output plane a multiple of 8: the tensor-core kernel.  NT = (9C + 8) / 8 n-tiles: C = 4..10
    // gives 5, 6, 7, 8, 10, 11, 12 (no C gives 9)
    const int plane = d.OH * d.OW, nt = (C * 9 + 1 + 7) / 8;
    const size_t msmem = sizeof(float) * (size_t)(H * frame_pitch(W) * C + 16 * CM_GSTRIDE + plane + nt * 8);
    if (OC == 16 && (plane % 8) == 0 && plane <= 64 && nt >= 5 && nt <= CM_MAX_NT && msmem <= 48 * 1024) {
        const unsigned grid = (unsigned)groups;
#define PB_CONV_TC_CASE(NTV)                                                                                       \
        case NTV: PB_LAUNCH(conv3x3_relu_bwd_mma_kernel<NTV>, grid, CM_WARPS * 32, msmem, stream, d, x, out, dout, \
                            partial_scratch, groups); break;
        switch (nt) {
            PB_CONV_TC_CASE(5) PB_CONV_TC_CASE(6) PB_CONV_TC_CASE(7) PB_CONV_TC_CASE(8)
            PB_CONV_TC_CASE(10) PB_CONV_TC_CASE(11) PB_CONV_TC_CASE(12)
        }
#undef PB_CONV_TC_CASE
        PB_LAUNCH(conv_bwd_reduce_kernel, (unsigned)((ne + 7) / 8), 256, 0, stream, groups, OC * C * 9, OC,
                  partial_scratch, dw, db);
        return PB_OK;
    }
    const size_t smem = fma_bwd_smem(d);
    // two gradient elements per thread for the MinAtar embedding (880 elements, 512 threads): several CTAs per SM, so
    // one CTA's staging loads overlap another's FMA loop and the 256 per-sample CTAs are resident in one wave
    const int ne_all = OC * C * 9 + OC;
    const int bthreads = ne_all > 256 ? 512 : 256;
    PB_LAUNCH(conv3x3_relu_bwd_kernel, (unsigned)groups, bthreads, smem, stream, d, x, out, dout, partial_scratch);
    PB_LAUNCH(conv_bwd_reduce_kernel, (unsigned)((ne + 7) / 8), 256, 0, stream, groups, OC * C * 9, OC,
              partial_scratch, dw, db);
    return PB_OK;
}

}  // extern "C"
