// BALF detector forward (multi-axis gated-MLP encoder + detector head) for sm_100a.
//
// Reference semantics (restated in oracle/detector.py):
//   balf/model/mlp_ma_decoder.py:201-244  Down           :119-149 split-head multi-axis gMLP
//   balf/model/mlp_ma_decoder.py:25-70    grid gMLP      :72-117  block gMLP
//   balf/model/mlp_ma_decoder.py:151-199  channel attention (LN, Linear, LeakyReLU, Linear, SE)
//   balf/model/decoder.py:16-30           DetectorHead   balf/utils/tensor_op.py:1-27 pixel_shuffle
//
// Precision 0 ("fp32") path.  Each Down stage runs as five fused kernels; all activations that
// cross kernels are channels-last fp32 in HBM, everything inside a kernel lives in shared memory
// as [channel][pixel] tiles so that the per-pixel Linear layers are register-blocked FFMA GEMMs:
//   branch<grid>  x -> conv.0 -> ReLU -> LN -> dense1[u half] -> GELU -> grid gMLP  -> u'
//   branch<block> x -> conv.0 -> ReLU -> LN -> dense1[v half] -> GELU -> block gMLP -> v'
//                 (the 64x64 token-mixing matmul runs over the pixel axis of the tile, which is
//                  why a tile is 64 grid cells x NF offsets, or NB whole 8x8 blocks)
//   merge         x, u', v' -> x0, dense2 + x0 -> LN -> conv1 -> LeakyReLU -> conv2 = r,
//                 q = x1 + x0, per-tile channel sums of r (deterministic two-level reduction)
//   se            mean -> excite.0 -> ReLU -> excite.2 -> sigmoid = s
//   pool          max-pool2x2(r * s + q)            (stages 1-3)
//   head          conv2(r * s + q) -> ReLU -> dense -> BN -> softmax -> depth-to-space (stage 4)
#include <cuda_fp16.h>
#include "detector.cuh"

namespace balf {

constexpr int NT = 256;          // threads per CTA in every tile kernel
constexpr int kWbufFloats = 4096;   // weight staging: 16 k-rows x <=256 outputs, or one 64x64 mixing matrix

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2, ACT_LRELU = 3 };

template <int ACT> __device__ __forceinline__ float act_fn(float v) {
    if (ACT == ACT_RELU) return fmaxf(v, 0.0f);
    if (ACT == ACT_GELU) return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f));
    if (ACT == ACT_LRELU) return v > 0.0f ? v : 0.2f * v;
    return v;
}

// ------------------------------------------------------------------------------------------ tile primitives
// Activation tiles are [channels][MP] fp32 in shared memory, MP = M + 4 (row stride == 4 mod 32
// banks: transposing loads/stores and vector reads are conflict-free).

// out[n][m] = act(sum_k in[k][m] * wT[k][n] + bias[n]) (+ res[n][m]).  out may alias in when
// N <= one pass (ALIAS).  Thread tile: 8 pixels (two float4 groups) x TN outputs.
template <int M, int K, int N, int ACT, bool ALIAS>
__device__ __forceinline__ void linear_tile(const float* in_s, const float* __restrict__ wT, int ldw,
                                            const float* __restrict__ bias, float* out_s, const float* res_s,
                                            float* wbuf) {
    constexpr int MP = M + 4;
    constexpr int TMB = M / 8, NTH = NT / TMB;
    constexpr int NC = N < NTH * 8 ? N : NTH * 8;
    constexpr int TN = NC / NTH;
    constexpr int KC = K < 16 ? K : 16;
    static_assert(N % NC == 0 && NC % NTH == 0 && TN >= 1 && K % KC == 0 && NC % 4 == 0, "tile shape");
    static_assert(!ALIAS || N == NC, "in-place needs a single output pass");
    static_assert(KC * NC <= kWbufFloats, "weight staging buffer too small");
    const int tid = threadIdx.x, tm = tid % TMB, tn = tid / TMB;
    for (int n0 = 0; n0 < N; n0 += NC) {
        float acc[TN][8];
#pragma unroll
        for (int j = 0; j < TN; ++j)
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[j][i] = 0.0f;
        for (int k0 = 0; k0 < K; k0 += KC) {
            __syncthreads();
            for (int i = tid; i < KC * NC / 4; i += NT) {
                int kk = i / (NC / 4), c4 = i - kk * (NC / 4);
                reinterpret_cast<float4*>(wbuf)[i] =
                    __ldg(reinterpret_cast<const float4*>(wT + (size_t)(k0 + kk) * ldw + n0 + c4 * 4));
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < KC; ++kk) {
                const float* arow = in_s + (size_t)(k0 + kk) * MP + tm * 4;
                float4 a0 = *reinterpret_cast<const float4*>(arow);
                float4 a1 = *reinterpret_cast<const float4*>(arow + M / 2);
                float w[TN];
                const float* wrow = wbuf + kk * NC + tn * TN;
                if (TN % 4 == 0) {
#pragma unroll
                    for (int j = 0; j < TN / 4; ++j) *reinterpret_cast<float4*>(&w[4 * j]) = reinterpret_cast<const float4*>(wrow)[j];
                } else if (TN % 2 == 0) {
#pragma unroll
                    for (int j = 0; j < TN / 2; ++j) *reinterpret_cast<float2*>(&w[2 * j]) = reinterpret_cast<const float2*>(wrow)[j];
                } else {
#pragma unroll
                    for (int j = 0; j < TN; ++j) w[j] = wrow[j];
                }
#pragma unroll
                for (int j = 0; j < TN; ++j) {
                    acc[j][0] = fmaf(w[j], a0.x, acc[j][0]); acc[j][1] = fmaf(w[j], a0.y, acc[j][1]);
                    acc[j][2] = fmaf(w[j], a0.z, acc[j][2]); acc[j][3] = fmaf(w[j], a0.w, acc[j][3]);
                    acc[j][4] = fmaf(w[j], a1.x, acc[j][4]); acc[j][5] = fmaf(w[j], a1.y, acc[j][5]);
                    acc[j][6] = fmaf(w[j], a1.z, acc[j][6]); acc[j][7] = fmaf(w[j], a1.w, acc[j][7]);
                }
            }
        }
        if (ALIAS) __syncthreads();
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int n = n0 + tn * TN + j;
            const float bv = bias ? __ldg(bias + n) : 0.0f;
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = act_fn<ACT>(acc[j][i] + bv);
            if (res_s) {
                const float* rr = res_s + (size_t)n * MP + tm * 4;
                float4 r0 = *reinterpret_cast<const float4*>(rr), r1 = *reinterpret_cast<const float4*>(rr + M / 2);
                o[0] += r0.x; o[1] += r0.y; o[2] += r0.z; o[3] += r0.w;
                o[4] += r1.x; o[5] += r1.y; o[6] += r1.z; o[7] += r1.w;
            }
            float* orow = out_s + (size_t)n * MP + tm * 4;
            *reinterpret_cast<float4*>(orow) = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<float4*>(orow + M / 2) = make_float4(o[4], o[5], o[6], o[7]);
        }
    }
    __syncthreads();
}

// LayerNorm over channels for every pixel of the tile (eps 1e-5, affine); src may equal dst.
template <int M, int C>
__device__ __forceinline__ void layernorm_tile(const float* src, float* dst, const float* __restrict__ g,
                                               const float* __restrict__ b, float* red) {
    constexpr int MP = M + 4, PARTS = NT / M;
    const int p = threadIdx.x % M, part = threadIdx.x / M;
    float s = 0.0f;
    for (int c = part; c < C; c += PARTS) s += src[(size_t)c * MP + p];
    red[part * M + p] = s;
    __syncthreads();
    float mean = 0.0f;
#pragma unroll
    for (int i = 0; i < PARTS; ++i) mean += red[i * M + p];
    mean *= (1.0f / C);
    float q = 0.0f;
    for (int c = part; c < C; c += PARTS) { float d = src[(size_t)c * MP + p] - mean; q = fmaf(d, d, q); }
    red[NT + part * M + p] = q;
    __syncthreads();
    float var = 0.0f;
#pragma unroll
    for (int i = 0; i < PARTS; ++i) var += red[NT + i * M + p];
    const float rstd = 1.0f / sqrtf(var * (1.0f / C) + 1e-5f);
    for (int c = part; c < C; c += PARTS)
        dst[(size_t)c * MP + p] = (src[(size_t)c * MP + p] - mean) * rstd * __ldg(g + c) + __ldg(b + c);
    __syncthreads();
}

// Token mixing of the gating units, in place: buf[c][g*64 + t'] = sum_t buf[c][g*64 + t] * wT[t][t'] + bias[t']
// for every 64-pixel group g of the tile (grid: the 64 cells of one offset; block: one 8x8 block).
template <int M, int C>
__device__ __forceinline__ void mix_tile(float* buf, const float* __restrict__ wT, const float* __restrict__ bias,
                                         float* wbuf) {
    constexpr int MP = M + 4, TQ = M / 4, TCB = NT / TQ, TC = C / TCB;
    static_assert(C % TCB == 0 && TC >= 1, "mix tile shape");
    const int tid = threadIdx.x, tq = tid % TQ, tc = tid / TQ, grp = tq / 16, mq = tq % 16;
    __syncthreads();
    for (int i = tid; i < 1024; i += NT) reinterpret_cast<float4*>(wbuf)[i] = __ldg(reinterpret_cast<const float4*>(wT) + i);
    __syncthreads();
    float acc[TC][4];
#pragma unroll
    for (int i = 0; i < TC; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
#pragma unroll 4
    for (int t4 = 0; t4 < 16; ++t4) {
        const float4 w0 = *reinterpret_cast<const float4*>(wbuf + (t4 * 4 + 0) * 64 + mq * 4);
        const float4 w1 = *reinterpret_cast<const float4*>(wbuf + (t4 * 4 + 1) * 64 + mq * 4);
        const float4 w2 = *reinterpret_cast<const float4*>(wbuf + (t4 * 4 + 2) * 64 + mq * 4);
        const float4 w3 = *reinterpret_cast<const float4*>(wbuf + (t4 * 4 + 3) * 64 + mq * 4);
#pragma unroll
        for (int i = 0; i < TC; ++i) {
            const float4 a = *reinterpret_cast<const float4*>(buf + (size_t)(tc * TC + i) * MP + grp * 64 + t4 * 4);
            acc[i][0] = fmaf(a.x, w0.x, acc[i][0]); acc[i][1] = fmaf(a.x, w0.y, acc[i][1]);
            acc[i][2] = fmaf(a.x, w0.z, acc[i][2]); acc[i][3] = fmaf(a.x, w0.w, acc[i][3]);
            acc[i][0] = fmaf(a.y, w1.x, acc[i][0]); acc[i][1] = fmaf(a.y, w1.y, acc[i][1]);
            acc[i][2] = fmaf(a.y, w1.z, acc[i][2]); acc[i][3] = fmaf(a.y, w1.w, acc[i][3]);
            acc[i][0] = fmaf(a.z, w2.x, acc[i][0]); acc[i][1] = fmaf(a.z, w2.y, acc[i][1]);
            acc[i][2] = fmaf(a.z, w2.z, acc[i][2]); acc[i][3] = fmaf(a.z, w2.w, acc[i][3]);
            acc[i][0] = fmaf(a.w, w3.x, acc[i][0]); acc[i][1] = fmaf(a.w, w3.y, acc[i][1]);
            acc[i][2] = fmaf(a.w, w3.z, acc[i][2]); acc[i][3] = fmaf(a.w, w3.w, acc[i][3]);
        }
    }
    __syncthreads();
    const float4 bv = __ldg(reinterpret_cast<const float4*>(bias) + mq);
#pragma unroll
    for (int i = 0; i < TC; ++i)
        *reinterpret_cast<float4*>(buf + (size_t)(tc * TC + i) * MP + grp * 64 + mq * 4) =
            make_float4(acc[i][0] + bv.x, acc[i][1] + bv.y, acc[i][2] + bv.z, acc[i][3] + bv.w);
    __syncthreads();
}

// channels-last global ([pixel][C]) <-> [C][MP] tile.  pix(m) = pixel index inside the image.
// A warp moves 16 pixels x 2 channel quads: 32-byte global segments, conflict-free shared accesses.
template <int M, int C, typename Pix>
__device__ __forceinline__ void load_cl(const float* __restrict__ g, float* s, Pix pix) {
    constexpr int MP = M + 4, QP = C / 8;
    for (int it = threadIdx.x; it < M * (C / 4); it += NT) {
        int blk = it >> 5, l = it & 31, m = (blk / QP) * 16 + (l & 15), q = (blk % QP) * 2 + (l >> 4);
        float4 v = __ldg(reinterpret_cast<const float4*>(g + (size_t)pix(m) * C) + q);
        float* d = s + (size_t)(q * 4) * MP + m;
        d[0] = v.x; d[MP] = v.y; d[2 * MP] = v.z; d[3 * MP] = v.w;
    }
}
template <int M, int C, typename Pix>
__device__ __forceinline__ void store_cl(float* __restrict__ g, const float* s, Pix pix) {
    constexpr int MP = M + 4, QP = C / 8;
    for (int it = threadIdx.x; it < M * (C / 4); it += NT) {
        int blk = it >> 5, l = it & 31, m = (blk / QP) * 16 + (l & 15), q = (blk % QP) * 2 + (l >> 4);
        const float* d = s + (size_t)(q * 4) * MP + m;
        *(reinterpret_cast<float4*>(g + (size_t)pix(m) * C) + q) = make_float4(d[0], d[MP], d[2 * MP], d[3 * MP]);
    }
}

// stage input of a level: either the NCHW network input (CIN = 3) or the previous stage's
// channels-last pooled output
template <int M, int CIN, typename Pix>
__device__ __forceinline__ void load_level_input(const float* __restrict__ xin, bool nchw, size_t npix, float* s, Pix pix) {
    constexpr int MP = M + 4;
    if (nchw) {
        for (int it = threadIdx.x; it < M * CIN; it += NT) {
            int c = it / M, m = it - c * M;
            s[(size_t)c * MP + m] = __ldg(xin + (size_t)c * npix + pix(m));
        }
    } else if constexpr (CIN % 8 == 0) {
        load_cl<M, CIN>(xin, s, pix);
    }
}

struct LevelGeom {
    int h, w;          // spatial size at this level
    int fh, fw;        // grid-cell extent (h/8, w/8)
};

// ------------------------------------------------------------------------------------------ branch kernel
template <int CIN, int C, int M>
struct BranchSmem {
    static constexpr int MP = M + 4;
    static constexpr size_t floats = 3 * (size_t)C * MP + kWbufFloats + 2 * NT;
    static constexpr size_t bytes = floats * sizeof(float);
};

template <int CIN, int C, int M, int BR>   // BR 0 = grid, 1 = block
__global__ void __launch_bounds__(NT, 1) branch_kernel(const float* __restrict__ xin, int in_nchw, DownW w, LevelGeom g,
                                                      float* __restrict__ out) {
    extern __shared__ __align__(16) float smem[];
    constexpr int MP = M + 4, G = M / 64;
    float* A = smem;
    float* Bf = A + (size_t)C * MP;
    float* Cf = Bf + (size_t)C * MP;
    float* wbuf = Cf + (size_t)C * MP;
    float* red = wbuf + kWbufFloats;
    const int b = blockIdx.y, t = blockIdx.x;
    const size_t npix = (size_t)g.h * g.w;
    int o0, o1;                                    // tile origin
    if (BR == 0) { int per_row = g.fw / G; o0 = t / per_row; o1 = (t % per_row) * G; }      // (fy, fx0)
    else { o0 = t * G; o1 = g.w / 8; }                                                      // (first block, blocks per row)
    auto pix = [&](int m) -> int {
        if (BR == 0) { int f = m >> 6, c = m & 63; return ((c >> 3) * g.fh + o0) * g.w + (c & 7) * g.fw + o1 + f; }
        int blk = o0 + (m >> 6), i = m & 63;
        return ((blk / o1) * 8 + (i >> 3)) * g.w + (blk % o1) * 8 + (i & 7);
    };
    const float* xb = xin + (size_t)b * npix * CIN;
    load_level_input<M, CIN>(xb, in_nchw != 0, npix, Cf, pix);
    const DownW::Branch& r = w.br[BR];
    linear_tile<M, CIN, C, ACT_RELU, false>(Cf, w.conv0_w, C, w.conv0_b, A, nullptr, wbuf);              // x0
    layernorm_tile<M, C>(A, A, w.pn_w, w.pn_b, red);
    linear_tile<M, C, C, ACT_GELU, false>(A, w.pd1_w + BR * C, 2 * C, w.pd1_b + BR * C, Bf, nullptr, wbuf);   // u | v
    layernorm_tile<M, C>(Bf, A, r.n_w, r.n_b, red);
    linear_tile<M, C, C, ACT_GELU, false>(A, r.d1_w, 2 * C, r.d1_b, Cf, nullptr, wbuf);                  // y1
    linear_tile<M, C, C, ACT_GELU, true>(A, r.d1_w + C, 2 * C, r.d1_b + C, A, nullptr, wbuf);            // y2 (in place)
    layernorm_tile<M, C>(A, A, r.gn_w, r.gn_b, red);
    mix_tile<M, C>(A, r.gd_w, r.gd_b, wbuf);
    for (int i = threadIdx.x; i < C * (M / 4); i += NT) {                                               // y1 * (y2' + 1)
        int c = i / (M / 4), m4 = i - c * (M / 4);
        float4 y2 = *reinterpret_cast<const float4*>(A + (size_t)c * MP + m4 * 4);
        float4* y1 = reinterpret_cast<float4*>(Cf + (size_t)c * MP + m4 * 4);
        float4 v = *y1;
        v.x *= y2.x + 1.0f; v.y *= y2.y + 1.0f; v.z *= y2.z + 1.0f; v.w *= y2.w + 1.0f;
        *y1 = v;
    }
    linear_tile<M, C, C, ACT_NONE, false>(Cf, r.d2_w, C, r.d2_b, A, Bf, wbuf);                           // + residual
    store_cl<M, C>(out + (size_t)b * npix * C, A, pix);
}

// ------------------------------------------------------------------------------------------ merge kernel
template <int CIN, int C, int M>
struct MergeSmem {
    static constexpr int MP = M + 4;
    static constexpr size_t floats = 4 * (size_t)C * MP + kWbufFloats + 2 * NT;
    static constexpr size_t bytes = floats * sizeof(float);
};

template <int CIN, int C, int M>
__global__ void __launch_bounds__(NT, 1) merge_kernel(const float* __restrict__ xin, int in_nchw, DownW w, LevelGeom g,
                                                     const float* __restrict__ u, const float* __restrict__ v,
                                                     float* __restrict__ rout, float* __restrict__ qout,
                                                     float* __restrict__ partial) {
    extern __shared__ __align__(16) float smem[];
    constexpr int MP = M + 4;
    float* UV = smem;                         // [2C][MP]
    float* A = UV + (size_t)2 * C * MP;       // x0
    float* X1 = A + (size_t)C * MP;
    float* wbuf = X1 + (size_t)C * MP;
    float* red = wbuf + kWbufFloats;
    const int b = blockIdx.y, t = blockIdx.x;
    const size_t npix = (size_t)g.h * g.w;
    const int p0 = t * M;
    auto pix = [&](int m) -> int { return p0 + m; };
    load_level_input<M, CIN>(xin + (size_t)b * npix * CIN, in_nchw != 0, npix, X1, pix);
    load_cl<M, C>(u + (size_t)b * npix * C, UV, pix);
    load_cl<M, C>(v + (size_t)b * npix * C, UV + (size_t)C * MP, pix);
    linear_tile<M, CIN, C, ACT_RELU, false>(X1, w.conv0_w, C, w.conv0_b, A, nullptr, wbuf);              // x0
    linear_tile<M, 2 * C, C, ACT_NONE, false>(UV, w.pd2_w, C, w.pd2_b, X1, A, wbuf);                     // x1
    layernorm_tile<M, C>(X1, UV, w.rn_w, w.rn_b, red);
    linear_tile<M, C, C, ACT_LRELU, false>(UV, w.rc1_w, C, w.rc1_b, UV + (size_t)C * MP, nullptr, wbuf);
    linear_tile<M, C, C, ACT_NONE, false>(UV + (size_t)C * MP, w.rc2_w, C, w.rc2_b, UV, nullptr, wbuf);  // r
    // squeeze: channel sums of r over this tile (fixed order -> deterministic)
    for (int c = threadIdx.x; c < C; c += NT) {
        float s = 0.0f;
        for (int m = 0; m < M; ++m) s += UV[(size_t)c * MP + m];
        partial[((size_t)b * gridDim.x + t) * C + c] = s;
    }
    for (int i = threadIdx.x; i < C * (M / 4); i += NT) {                                               // q = x1 + x0
        int c = i / (M / 4), m4 = i - c * (M / 4);
        float4 a = *reinterpret_cast<const float4*>(A + (size_t)c * MP + m4 * 4);
        float4* x = reinterpret_cast<float4*>(X1 + (size_t)c * MP + m4 * 4);
        float4 v4 = *x;
        v4.x += a.x; v4.y += a.y; v4.z += a.z; v4.w += a.w;
        *x = v4;
    }
    __syncthreads();
    store_cl<M, C>(rout + (size_t)b * npix * C, UV, pix);
    store_cl<M, C>(qout + (size_t)b * npix * C, X1, pix);
}

// ------------------------------------------------------------------------------------------ squeeze-excite
// One CTA per image.  The per-unit channel sums are reduced in a fixed order (thread (seg, c) walks units seg,
// seg + NSEG, ...; then a fixed shared-memory tree over seg), so the mean -- and with it the score map -- is
// bit-reproducible run to run and independent of the batch the image sits in.
constexpr int kSeThreads = 1024;
template <int C>
__global__ void __launch_bounds__(kSeThreads) se_kernel(const float* __restrict__ partial, int tiles, float inv_npix, DownW w,
                                                        float* __restrict__ scale) {
    constexpr int NSEG = kSeThreads / C;
    __shared__ float red[kSeThreads];
    __shared__ float mean[C];
    __shared__ float hid[C / 4];
    const int b = blockIdx.x, c = threadIdx.x % C, seg = threadIdx.x / C;
    const float* src = partial + (size_t)b * tiles * C + c;
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
    int t = seg;
    for (; t + 3 * NSEG < tiles; t += 4 * NSEG) {
        s0 += src[(size_t)t * C]; s1 += src[(size_t)(t + NSEG) * C];
        s2 += src[(size_t)(t + 2 * NSEG) * C]; s3 += src[(size_t)(t + 3 * NSEG) * C];
    }
    for (; t < tiles; t += NSEG) s0 += src[(size_t)t * C];
    red[threadIdx.x] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    for (int n = NSEG / 2; n >= 1; n >>= 1) {
        if (seg < n) red[threadIdx.x] += red[threadIdx.x + n * C];
        __syncthreads();
    }
    if (threadIdx.x < C) mean[c] = red[c] * inv_npix;
    __syncthreads();
    if (threadIdx.x < C / 4) {
        float h = __ldg(w.ex0_b + c);
        for (int k = 0; k < C; ++k) h = fmaf(mean[k], __ldg(w.ex0_w + (size_t)k * (C / 4) + c), h);
        hid[c] = fmaxf(h, 0.0f);
    }
    __syncthreads();
    if (threadIdx.x < C) {
        float o = __ldg(w.ex2_b + c);
        for (int k = 0; k < C / 4; ++k) o = fmaf(hid[k], __ldg(w.ex2_w + (size_t)k * C + c), o);
        scale[(size_t)b * C + c] = 1.0f / (1.0f + expf(-o));
    }
}

// ------------------------------------------------------------------------------------------ pool (stages 1-3)
// out[b, py, px, :] = max over the 2x2 window of (r * s + q)
// swz: 0 = r, q channels-last; 1 = q in swizzled-panel tiles, r in fp16 tiles; 2 = r and q in swizzled-panel tiles (split precision);
//      3 = q channels-last, r channels-last fp16 (stage 3 of the single-rounded tensor path)
// OH: the output is fp16 (channels-last halves) -- the next stage runs on the single-rounded tensor-core path, whose only use of
// its level input is the fp16 A operand of conv.0: same values as rounding at load time, half the bytes written once and read 3x
template <int C, int swz, bool OH>
__global__ void pool_kernel(const float* __restrict__ r, const float* __restrict__ q, const float* __restrict__ scale,
                            int h, int w, float* __restrict__ out, size_t total) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    constexpr int Q = C / 4;
    const int c4 = (int)(i % Q);
    size_t t = i / Q;
    const int wo = w / 2, ho = h / 2;
    const int px = (int)(t % wo);
    t /= wo;
    const int py = (int)(t % ho);
    const size_t b = t / ho;
    const float4 s = __ldg(reinterpret_cast<const float4*>(scale + b * C) + c4);
    float4 best = make_float4(kNegInf, kNegInf, kNegInf, kNegInf);
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            size_t p = (b * h + 2 * py + dy) * w + 2 * px + dx;
            // swz: r / q of the tensor-core merge kernels of the first two stages are tiles of 128 pixels in the swizzled
            // panel layout (detector_tc.cu sw_off): panels of 32 channels, 128-byte rows, chunks permuted by (pixel % 8)
            const size_t rowi = p & 127;
            const size_t cs = (swz == 1 || swz == 2) ? (((p - rowi) * C) >> 2) + (size_t)(c4 >> 3) * (128 * 8) + rowi * 8 + ((c4 & 7) ^ (rowi & 7))
                                  : ((p * C) >> 2) + c4;
            float4 rv;
            if constexpr (swz == 1) {
                // r of those stages is an fp16 tile [C / 8 chunks][128 pixels][8 halves] (tc_merge_bulk_kernel)
                const uint2 h = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(r) + (p - rowi) * C +
                                                                     (size_t)(c4 >> 1) * (128 * 8) + rowi * 8 + (c4 & 1) * 4));
                const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&h.x)), hi = __half22float2(*reinterpret_cast<const __half2*>(&h.y));
                rv = make_float4(lo.x, lo.y, hi.x, hi.y);
            } else if constexpr (swz == 3) {
                const uint2 h = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(r) + p * C) + c4);
                const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&h.x)), hi = __half22float2(*reinterpret_cast<const __half2*>(&h.y));
                rv = make_float4(lo.x, lo.y, hi.x, hi.y);
            } else {
                rv = __ldg(reinterpret_cast<const float4*>(r) + cs);
            }
            float4 qv;
            if constexpr (swz == 1) {
                // q of those stages: 24 bits per value in two planes per tile of 128 pixels (tc_merge_bulk_kernel): [C / 8][128][8 x u16]
                // = the top halves of the fp32 patterns, then [C / 16][128][16 x u8] = the next byte
                const unsigned char* qt = reinterpret_cast<const unsigned char*>(q) + (p - rowi) * C * 3;
                const uint2 t16 = __ldg(reinterpret_cast<const uint2*>(qt + ((size_t)(c4 >> 1) * 128 + rowi) * 16 + (c4 & 1) * 8));
                const uint32_t m8 = __ldg(reinterpret_cast<const uint32_t*>(qt + (size_t)128 * C * 2 + ((size_t)(c4 >> 2) * 128 + rowi) * 16 + (c4 & 3) * 4));
                qv.x = __uint_as_float(((t16.x & 0xFFFFu) << 16) | ((m8 & 0xFFu) << 8));
                qv.y = __uint_as_float((t16.x & 0xFFFF0000u) | (m8 & 0xFF00u));
                qv.z = __uint_as_float(((t16.y & 0xFFFFu) << 16) | ((m8 >> 8) & 0xFF00u));
                qv.w = __uint_as_float((t16.y & 0xFFFF0000u) | ((m8 >> 16) & 0xFF00u));
            } else {
                qv = __ldg(reinterpret_cast<const float4*>(q) + cs);
            }
            best.x = fmaxf(best.x, rv.x * s.x + qv.x); best.y = fmaxf(best.y, rv.y * s.y + qv.y);
            best.z = fmaxf(best.z, rv.z * s.z + qv.z); best.w = fmaxf(best.w, rv.w * s.w + qv.w);
        }
    if constexpr (OH) {
        uint2 o;
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(o.x) : "f"(best.y), "f"(best.x));
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(o.y) : "f"(best.w), "f"(best.z));
        *(reinterpret_cast<uint2*>(reinterpret_cast<__half*>(out) + ((b * ho + py) * wo + px) * C) + c4) = o;
    } else {
        *(reinterpret_cast<float4*>(out + ((b * ho + py) * wo + px) * C) + c4) = best;
    }
}

// ------------------------------------------------------------------------------------------ head (stage 4)
template <int C, int M>
struct HeadSmem {
    static constexpr int MP = M + 4;
    static constexpr size_t floats = (2 * (size_t)C + kHeadPad) * MP + kWbufFloats;
    static constexpr size_t bytes = floats * sizeof(float);
};

template <int C, int M>
__global__ void __launch_bounds__(NT, 1) head_kernel(const float* __restrict__ r, const float* __restrict__ q,
                                                    const float* __restrict__ scale, DownW w, HeadW hw, int hc, int wc,
                                                    int cell, float* __restrict__ logits, float* __restrict__ prob) {
    extern __shared__ __align__(16) float smem[];
    constexpr int MP = M + 4;
    float* A = smem;
    float* T = A + (size_t)C * MP;
    float* Z = T + (size_t)C * MP;            // [kHeadPad][MP]
    float* wbuf = Z + (size_t)kHeadPad * MP;
    const int b = blockIdx.y, p0 = blockIdx.x * M;
    const size_t npix = (size_t)hc * wc;
    auto pix = [&](int m) -> int { return p0 + m; };
    load_cl<M, C>(r + (size_t)b * npix * C, A, pix);
    load_cl<M, C>(q + (size_t)b * npix * C, T, pix);
    __syncthreads();
    for (int i = threadIdx.x; i < C * M; i += NT) {
        int c = i / M, m = i - c * M;
        A[(size_t)c * MP + m] = A[(size_t)c * MP + m] * __ldg(scale + (size_t)b * C + c) + T[(size_t)c * MP + m];
    }
    linear_tile<M, C, C, ACT_RELU, false>(A, w.c2_w, C, w.c2_b, T, nullptr, wbuf);     // conv2, then the head's ReLU
    linear_tile<M, C, kHeadPad, ACT_NONE, false>(T, hw.w, kHeadPad, hw.b, Z, nullptr, wbuf);
    const int nlog = cell * cell + 1;
    // eval BatchNorm (folded affine); logits are NCHW
    for (int i = threadIdx.x; i < nlog * M; i += NT) {
        int n = i / M, m = i - n * M;
        float z = Z[(size_t)n * MP + m] * __ldg(hw.alpha + n) + __ldg(hw.beta + n);
        Z[(size_t)n * MP + m] = z;
        if (logits) logits[((size_t)b * nlog + n) * npix + p0 + m] = z;
    }
    __syncthreads();
    // softmax over the nlog channels, drop the dustbin, depth-to-space
    for (int m = threadIdx.x; m < M; m += NT) {
        float mx = kNegInf;
        for (int n = 0; n < nlog; ++n) mx = fmaxf(mx, Z[(size_t)n * MP + m]);
        float den = 0.0f;
        for (int n = 0; n < nlog; ++n) den += expf(Z[(size_t)n * MP + m] - mx);
        T[m] = mx;
        T[MP + m] = den;
    }
    __syncthreads();
    const int Wp = wc * cell;
    for (int i = threadIdx.x; i < (nlog - 1) * M; i += NT) {
        int m = i / (nlog - 1), n = i - m * (nlog - 1);
        int p = p0 + m, cy = p / wc, cx = p - cy * wc;
        float v = expf(Z[(size_t)n * MP + m] - T[m]) / T[MP + m];
        prob[((size_t)b * hc * cell + cy * cell + n / cell) * Wp + cx * cell + n % cell] = v;
    }
}

// ------------------------------------------------------------------------------------------ weight packing
__global__ void transpose_pack_kernel(const float* __restrict__ src, int rows, int cols, float* __restrict__ dst, int ld) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols) return;
    int r = i / cols, c = i - r * cols;             // src[r][c] -> dst[c][r]
    dst[(size_t)c * ld + r] = src[i];
}
__global__ void copy_pack_kernel(const float* __restrict__ src, int n, float* __restrict__ dst) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}
// F.batch_norm(eval): y = (x - mean) / sqrt(var + eps) * gamma + beta = x * alpha + beta'
__global__ void bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                               const float* __restrict__ var, int n, float* __restrict__ a, float* __restrict__ bb) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float al = gamma[i] / sqrtf(var[i] + 1e-5f);
    a[i] = al;
    bb[i] = beta[i] - mean[i] * al;
}

// ------------------------------------------------------------------------------------------ host
static int check_arch(const balf_detector_arch* a) {
    BALF_REQUIRE(a != nullptr, "null architecture");
    BALF_REQUIRE(a->dims[0] == 3 && a->dims[1] == 32 && a->dims[2] == 64 && a->dims[3] == 128 && a->dims[4] == 256,
                 "only en_embed_dims = [3,32,64,128,256] is built (got [%d,%d,%d,%d,%d])", a->dims[0], a->dims[1],
                 a->dims[2], a->dims[3], a->dims[4]);
    BALF_REQUIRE(a->grid_h == 8 && a->grid_w == 8 && a->block_h == 8 && a->block_w == 8,
                 "only grid_size = block_size = [8,8] is built");
    BALF_REQUIRE(a->grid_factor == 2 && a->block_factor == 2 && a->proj_factor == 2, "only gMLP / projection factor 2 is built");
    BALF_REQUIRE(a->reduction == 4, "only channels_reduction = 4 is built");
    BALF_REQUIRE(a->cell == 8, "only cell_size = 8 is built");
    return 0;
}

static int64_t raw_count(const balf_detector_arch& a) {
    int64_t n = 0;
    for (int l = 0; l < 4; ++l) {
        int64_t ci = a.dims[l], c = a.dims[l + 1], red = c / a.reduction;
        n += ci * c + c + 2 * c + (2 * c * c + 2 * c);
        n += 2 * (2 * c + (2 * c * c + 2 * c) + 2 * c + (64 * 64 + 64) + (c * c + c));
        n += (2 * c * c + c) + 2 * c + 2 * (c * c + c) + (c * red + red) + (red * c + c) + (c * c + c);
    }
    int64_t nl = a.cell * a.cell + 1;
    return n + nl * a.dims[4] + nl + 4 * nl;
}

struct Workspace {
    float *u, *v, *r, *q;       // [Bc, h1*w1*32] each (largest level)
    float* pooled[3];           // stage outputs
    float* partial;             // [Bc, tiles, C]
    float* scale;               // [Bc, 256]
};

static size_t ws_layout(const balf_detector_arch& a, int Bc, int Hp, int Wp, void* base, Workspace* ws) {
    size_t off = 0;
    char* p = static_cast<char*>(base);
    auto take = [&](size_t floats) { size_t o = off; off = align_up(off + floats * sizeof(float), 256); return o; };
    const size_t px = (size_t)Hp * Wp;
    const size_t big = (size_t)Bc * px * a.dims[1];
    size_t o[9];
    for (int i = 0; i < 4; ++i) o[i] = take(big);
    for (int l = 0; l < 3; ++l) o[4 + l] = take((size_t)Bc * (px >> (2 * (l + 1))) * a.dims[l + 1]);
    o[7] = take((size_t)Bc * (px / 64) * a.dims[1]);       // partial sums: (64-pixel units) * C is largest at level 1
    o[8] = take((size_t)Bc * a.dims[4]);
    if (ws) {
        ws->u = reinterpret_cast<float*>(p + o[0]); ws->v = reinterpret_cast<float*>(p + o[1]);
        ws->r = reinterpret_cast<float*>(p + o[2]); ws->q = reinterpret_cast<float*>(p + o[3]);
        for (int l = 0; l < 3; ++l) ws->pooled[l] = reinterpret_cast<float*>(p + o[4 + l]);
        ws->partial = reinterpret_cast<float*>(p + o[7]);
        ws->scale = reinterpret_cast<float*>(p + o[8]);
    }
    return off;
}

extern int g_tc_trace_sel;        // detector_tc.cu
extern int g_match_impl;          // match.cu
extern int g_greedy_impl;         // nms.cu
extern int g_greedy_rounds;       // nms.cu
extern int g_nms_tma;             // nms.cu
int g_tc_mask = 0x1F;              // debug hook (balf_debug_set key 0): bit l = stage l on the tensor-core path, bit 4 = head

int g_chunk_images = 0;            // images per internal pass; 0 = automatic (debug hook key 1 pins it)
// Automatic chunk: as many images as fit a 16 GB workspace, at most 64.  Larger passes mean fewer launches, shorter
// persistent-grid tails and full waves at the two coarsest stages (measured at 512x640: 8 -> 2433, 16 -> 2669, 32 -> 2827,
// 64 -> 2879 images/s); 16 GB of a 180 GB HBM3e stack is the price.  fast_div limits a pass to 2^23 units.
static int chunk_images(const balf_detector_arch& a, int B, int Hp, int Wp) {
    int c = g_chunk_images;
    if (c <= 0) {
        const size_t per_image = ws_layout(a, 1, Hp, Wp, nullptr, nullptr);
        size_t n = ((size_t)16 << 30) / (per_image ? per_image : 1);
        const size_t unit_cap = ((size_t)1 << 22) / ((size_t)Hp * Wp / 64);
        if (unit_cap < n) n = unit_cap;
        c = n < 1 ? 1 : n > 64 ? 64 : (int)n;
    }
    return B < c ? B : c;
}

template <typename K> static int set_smem(K kernel, size_t bytes) {
    BALF_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

template <int CIN, int C, int MB, int MM>
static int run_level(const float* xin, bool nchw, const DownW& w, int Bc, int h, int wd, const Workspace& ws,
                     cudaStream_t st, int* merge_tiles) {
    LevelGeom g{h, wd, h / 8, wd / 8};
    const int npix = h * wd;
    if (int e = set_smem(branch_kernel<CIN, C, MB, 0>, BranchSmem<CIN, C, MB>::bytes)) return e;
    if (int e = set_smem(branch_kernel<CIN, C, MB, 1>, BranchSmem<CIN, C, MB>::bytes)) return e;
    if (int e = set_smem(merge_kernel<CIN, C, MM>, MergeSmem<CIN, C, MM>::bytes)) return e;
    dim3 gb(npix / MB, Bc);
    {
        ProfScope p(C == 32 ? "det_branch_grid_c32" : C == 64 ? "det_branch_grid_c64" : C == 128 ? "det_branch_grid_c128" : "det_branch_grid_c256", st);
        branch_kernel<CIN, C, MB, 0><<<gb, NT, BranchSmem<CIN, C, MB>::bytes, st>>>(xin, nchw, w, g, ws.u);
    }
    {
        ProfScope p(C == 32 ? "det_branch_block_c32" : C == 64 ? "det_branch_block_c64" : C == 128 ? "det_branch_block_c128" : "det_branch_block_c256", st);
        branch_kernel<CIN, C, MB, 1><<<gb, NT, BranchSmem<CIN, C, MB>::bytes, st>>>(xin, nchw, w, g, ws.v);
    }
    dim3 gm(npix / MM, Bc);
    {
        ProfScope p(C == 32 ? "det_merge_c32" : C == 64 ? "det_merge_c64" : C == 128 ? "det_merge_c128" : "det_merge_c256", st);
        merge_kernel<CIN, C, MM><<<gm, NT, MergeSmem<CIN, C, MM>::bytes, st>>>(xin, nchw, w, g, ws.u, ws.v, ws.r, ws.q, ws.partial);
    }
    {
        ProfScope p("det_se", st);
        se_kernel<C><<<Bc, kSeThreads, 0, st>>>(ws.partial, npix / MM, 1.0f / (float)npix, w, ws.scale);
    }
    BALF_COUNT_LAUNCH(4);
    BALF_LAUNCH_OK();
    *merge_tiles = npix / MM;
    return 0;
}

template <int C>
static int run_se(const Workspace& ws, const DownW& w, int Bc, int npix, int parts, cudaStream_t st) {
    {
        ProfScope p("det_se", st);
        se_kernel<C><<<Bc, kSeThreads, 0, st>>>(ws.partial, parts, 1.0f / (float)npix, w, ws.scale);
    }
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}

template <int C>
static int run_pool(const Workspace& ws, int Bc, int h, int wd, float* out, cudaStream_t st, int swz = 0, bool oh = false) {
    size_t total = (size_t)Bc * (h / 2) * (wd / 2) * (C / 4);
    {
        ProfScope p("det_pool", st);
        const unsigned grid = (unsigned)((total + 255) / 256);
        if (swz == 1 && oh) pool_kernel<C, 1, true><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
        else if (swz == 1) pool_kernel<C, 1, false><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
        else if (swz == 2) pool_kernel<C, 2, false><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
        else if (swz == 3 && oh) pool_kernel<C, 3, true><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
        else if (swz == 3) pool_kernel<C, 3, false><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
        else if (oh) pool_kernel<C, 0, true><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
        else pool_kernel<C, 0, false><<<grid, 256, 0, st>>>(ws.r, ws.q, ws.scale, h, wd, out, total);
    }
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}

}  // namespace balf

using namespace balf;

extern "C" int balf_debug_set(int key, int value) {
    BALF_REQUIRE(key >= 0 && key <= 7 && key != 4, "unknown debug key %d", key);
    if (key == 7) { g_nms_tma = value ? 1 : 0; return 0; }
    if (key == 6) { g_greedy_rounds = value < 0 ? 0 : value > 64 ? 64 : value; return 0; }
    if (key == 5) { g_greedy_impl = value ? 1 : 0; return 0; }
    if (key == 3) { g_match_impl = value ? 1 : 0; return 0; }
    if (key == 0) g_tc_mask = value & 0x1F;
    else if (key == 2) g_tc_trace_sel = value;
    else { BALF_REQUIRE(value >= 0 && value <= 64, "chunk must be in [0, 64] (0 = automatic)"); g_chunk_images = value; }
    return 0;
}

extern "C" int balf_detector_check_arch(const balf_detector_arch* arch) { return check_arch(arch); }

extern "C" int64_t balf_detector_raw_weight_count(const balf_detector_arch* arch) {
    if (check_arch(arch)) return -1;
    return raw_count(*arch);
}

extern "C" int64_t balf_detector_packed_weight_count(const balf_detector_arch* arch) {
    if (check_arch(arch)) return -1;
    return (int64_t)(walk_packed(*arch, nullptr, nullptr) + tc_blob_floats(*arch));
}

extern "C" int balf_detector_pack_weights(const balf_detector_arch* arch, const float* raw, float* packed, void* stream) {
    if (int e = check_arch(arch)) return e;
    BALF_REQUIRE(raw && packed, "null pointer argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const balf_detector_arch& a = *arch;
    DetW w;
    size_t total = walk_packed(a, packed, &w);
    BALF_CUDA_OK(cudaMemsetAsync(packed, 0, total * sizeof(float), st));
    const float* src = raw;
    auto mat = [&](const float* dst, int out_f, int in_f, int ld) {     // Linear.weight [out][in] -> wT[in][ld]
        int n = out_f * in_f;
        transpose_pack_kernel<<<cdiv(n, 256), 256, 0, st>>>(src, out_f, in_f, const_cast<float*>(dst), ld);
        src += n;
    };
    auto vec = [&](const float* dst, int n) {
        copy_pack_kernel<<<cdiv(n, 256), 256, 0, st>>>(src, n, const_cast<float*>(dst));
        src += n;
    };
    for (int l = 0; l < 4; ++l) {
        const int ci = a.dims[l], c = a.dims[l + 1], red = c / a.reduction;
        const DownW& d = w.down[l];
        mat(d.conv0_w, c, ci, c); vec(d.conv0_b, c);
        vec(d.pn_w, c); vec(d.pn_b, c);
        mat(d.pd1_w, 2 * c, c, 2 * c); vec(d.pd1_b, 2 * c);
        for (int b = 0; b < 2; ++b) {
            const DownW::Branch& r = d.br[b];
            vec(r.n_w, c); vec(r.n_b, c);
            mat(r.d1_w, 2 * c, c, 2 * c); vec(r.d1_b, 2 * c);
            vec(r.gn_w, c); vec(r.gn_b, c);
            mat(r.gd_w, 64, 64, 64); vec(r.gd_b, 64);
            mat(r.d2_w, c, c, c); vec(r.d2_b, c);
        }
        mat(d.pd2_w, c, 2 * c, c); vec(d.pd2_b, c);
        vec(d.rn_w, c); vec(d.rn_b, c);
        mat(d.rc1_w, c, c, c); vec(d.rc1_b, c);
        mat(d.rc2_w, c, c, c); vec(d.rc2_b, c);
        mat(d.ex0_w, red, c, red); vec(d.ex0_b, red);
        mat(d.ex2_w, c, red, c); vec(d.ex2_b, c);
        mat(d.c2_w, c, c, c); vec(d.c2_b, c);
    }
    const int nl = a.cell * a.cell + 1;
    mat(w.head.w, nl, a.dims[4], kHeadPad); vec(w.head.b, nl);
    bn_fold_kernel<<<1, 128, 0, st>>>(src, src + nl, src + 2 * nl, src + 3 * nl, nl, const_cast<float*>(w.head.alpha),
                                      const_cast<float*>(w.head.beta));
    src += 4 * nl;
    BALF_LAUNCH_OK();
    BALF_REQUIRE(src - raw == raw_count(a), "internal: raw weight walk mismatch");
    return tc_pack_weights(a, w, packed + total, st);       // second half of the blob: tensor-core operand images
}

extern "C" size_t balf_detector_workspace_bytes(const balf_detector_arch* arch, int B, int Hp, int Wp) {
    if (check_arch(arch) || B <= 0 || Hp <= 0 || Wp <= 0) return 0;
    return ws_layout(*arch, chunk_images(*arch, B, Hp, Wp), Hp, Wp, nullptr, nullptr);
}

extern "C" int balf_detector_forward(const balf_detector_arch* arch, const float* packed, const float* x, int B, int Hp,
                                     int Wp, float* logits, float* prob, void* workspace, size_t workspace_bytes,
                                     int precision, void* stream) {
    if (int e = check_arch(arch)) return e;
    BALF_REQUIRE(packed && x && prob && workspace, "null pointer argument");
    BALF_REQUIRE(B > 0 && Hp > 0 && Wp > 0, "B, Hp, Wp must be positive");
    BALF_REQUIRE(Hp % 64 == 0 && Wp % 64 == 0, "input %dx%d: height and width must be multiples of 64 "
                 "(3 max-pools x 8x8 grid/block tokens; pad with mod_padding_symmetric)", Hp, Wp);
    BALF_REQUIRE(precision >= 0 && precision <= 2, "precision %d is not built in this library (0 = fp32, 1 = tf32-class, 2 = f16x3)", precision);
    const balf_detector_arch& a = *arch;
    const int chunk = chunk_images(a, B, Hp, Wp);
    BALF_REQUIRE(workspace_bytes >= ws_layout(a, chunk, Hp, Wp, nullptr, nullptr), "workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DetW w;
    const float* tc_blob = packed + walk_packed(a, packed, &w);
    Workspace ws;
    ws_layout(a, chunk, Hp, Wp, workspace, &ws);
    const int nl = a.cell * a.cell + 1, hc = Hp / 8, wc = Wp / 8;
    if (int e = set_smem(head_kernel<256, 32>, HeadSmem<256, 32>::bytes)) return e;
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int Bc = B - b0 < chunk ? B - b0 : chunk;
        const float* xb = x + (size_t)b0 * 3 * Hp * Wp;
        // precision 1: tensor-core kernels (detector_tc.cu); g_tc_mask (debug hook) can send single
        // stages back to the fp32 kernels -- both paths share the workspace formats.
        const int tcm = precision >= 1 ? g_tc_mask : 0;
        const int px = precision == 2 ? 1 : 0;                 // split precision: fp16 hi + lo operands, three MMAs per product
        const DownW* d = w.down;
        int tiles = 0;
        if (tcm & 1) {
            if (int e = tc_run_level_dispatch(0, xb, d[0], a, tc_blob, Bc, Hp, Wp, ws.u, ws.v, ws.r, ws.q, ws.partial, st, px, 0)) return e;
            if (int e = run_se<32>(ws, d[0], Bc, Hp * Wp, Hp * Wp / 64, st)) return e;
        } else if (int e = run_level<3, 32, 128, 128>(xb, true, w.down[0], Bc, Hp, Wp, ws, st, &tiles)) return e;
        if (int e = run_pool<32>(ws, Bc, Hp, Wp, ws.pooled[0], st, (tcm & 1) ? 1 + px : 0, (tcm & 2) && !px)) return e;
        if (tcm & 2) {
            if (int e = tc_run_level_dispatch(1, ws.pooled[0], d[1], a, tc_blob, Bc, Hp / 2, Wp / 2, ws.u, ws.v, ws.r, ws.q, ws.partial, st, px, 0)) return e;
            if (int e = run_se<64>(ws, d[1], Bc, Hp * Wp / 4, Hp * Wp / 256, st)) return e;
        } else if (int e = run_level<32, 64, 128, 128>(ws.pooled[0], false, w.down[1], Bc, Hp / 2, Wp / 2, ws, st, &tiles)) return e;
        if (int e = run_pool<64>(ws, Bc, Hp / 2, Wp / 2, ws.pooled[1], st, (tcm & 2) ? 1 + px : 0, (tcm & 4) && !px)) return e;
        if (tcm & 4) {
            if (int e = tc_run_level_dispatch(2, ws.pooled[1], d[2], a, tc_blob, Bc, Hp / 4, Wp / 4, ws.u, ws.v, ws.r, ws.q, ws.partial, st, px, px == 0)) return e;
            if (int e = run_se<128>(ws, d[2], Bc, Hp * Wp / 16, Hp * Wp / 1024, st)) return e;
        } else if (int e = run_level<64, 128, 64, 64>(ws.pooled[1], false, w.down[2], Bc, Hp / 4, Wp / 4, ws, st, &tiles)) return e;
        if (int e = run_pool<128>(ws, Bc, Hp / 4, Wp / 4, ws.pooled[2], st, ((tcm & 4) && !px) ? 3 : 0, (tcm & 8) && !px)) return e;
        if (tcm & 8) {
            if (int e = tc_run_level_dispatch(3, ws.pooled[2], d[3], a, tc_blob, Bc, hc, wc, ws.u, ws.v, ws.r, ws.q, ws.partial, st, px, px == 0 && (tcm & 16) != 0)) return e;
            if (int e = run_se<256>(ws, d[3], Bc, hc * wc, hc * wc / 64, st)) return e;
        } else if (int e = run_level<128, 256, 64, 32>(ws.pooled[2], false, w.down[3], Bc, hc, wc, ws, st, &tiles)) return e;
        if (tcm & 16) {
            if (int e = tc_run_head(ws.r, ws.q, ws.scale, a, tc_blob, Bc, hc, wc,
                                    logits ? logits + (size_t)b0 * nl * hc * wc : nullptr, prob + (size_t)b0 * Hp * Wp, st, px, px == 0 && (tcm & 8) != 0)) return e;
            continue;
        }
        dim3 gh(hc * wc / 32, Bc);
        {
            ProfScope p("det_head", st);
            head_kernel<256, 32><<<gh, NT, HeadSmem<256, 32>::bytes, st>>>(
                ws.r, ws.q, ws.scale, w.down[3], w.head, hc, wc, a.cell,
                logits ? logits + (size_t)b0 * nl * hc * wc : nullptr, prob + (size_t)b0 * Hp * Wp);
        }
        BALF_COUNT_LAUNCH(1);
        BALF_LAUNCH_OK();
    }
    return 0;
}
