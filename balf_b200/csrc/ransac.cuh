// Pieces shared by the RANSAC estimators (homography.cu, fundamental.cu, essential.cu): the counter-based sampler, the
// partial-pivot elimination, point normalisation, the chunked scoring kernel with its packed winner key, the refit kernels'
// fixed-order block sums, the unit-norm scaling, det3 and the cyclic Jacobi.  Every translation unit is compiled with
// -fmad=false, and oracle/homography.py and oracle/fundamental.py restate every piece (oracle/essential.py reuses them).
#pragma once
#include "common.cuh"

namespace balf {
namespace {

typedef unsigned long long u64;

constexpr int kMaxMatches = 16384;       // test_utils.K_MAX: the largest keypoint list the library produces
constexpr int kMaxIters = 1 << 17;
constexpr double kSqrt2 = 1.4142135623730951;
constexpr int kScoreThreads = 256;
constexpr int kHypThreads = 128;
constexpr int kChunk = 1024;             // points per shared-memory chunk of the scoring kernel (32 KB)
constexpr int kRefitThreads = 256;
constexpr int kJacobiSweeps = 32;
constexpr double kJacobiTol2 = 4.930380657631324e-32;   // 2^-104: off-diagonal sum of squares / diagonal sum of squares
constexpr double kInf = __builtin_huge_val();

__device__ __forceinline__ u64 splitmix64(u64 z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// K distinct indices of n for hypothesis h of pair b, in draw order: counter c = 0, 1, ... gives
// splitmix64(stream + c) mod n, stream = splitmix64(splitmix64(seed) ^ (b << 32 | h)), and a repeated index is skipped.
// False when Draws counters did not give K distinct indices.
template <int K, int Draws>
__device__ __forceinline__ bool draw_sample(u64 seed, int b, int h, int n, int (&idx)[K]) {
    const u64 stream = splitmix64(splitmix64(seed) ^ (((u64)b << 32) | (u64)h));
    int k = 0;
    for (int c = 0; c < Draws && k < K; ++c) {
        const int i = (int)(splitmix64(stream + (u64)c) % (u64)n);
        bool dup = false;
#pragma unroll
        for (int j = 0; j < K; ++j) dup |= (j < k) && idx[j] == i;
        if (!dup) {
#pragma unroll
            for (int j = 0; j < K; ++j) if (j == k) idx[j] = i;
            ++k;
        }
    }
    return k == K;
}

// Gaussian elimination with partial pivoting on the augmented system a [8][9] -> h [8].  The pivot is the first row with
// the largest |a[r][k]| (a NaN counts as the largest, like np.argmax); false when a pivot is 0 or not finite.  Loops are
// unrolled so that the row swap is a set of selects on registers.
__device__ __forceinline__ bool solve8(double (&a)[8][9], double (&h)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        double best = fabs(a[k][k]);
        int p = k;
#pragma unroll
        for (int r = k + 1; r < 8; ++r) {
            const double v = fabs(a[r][k]);
            if (!isnan(best) && (isnan(v) || v > best)) { best = v; p = r; }
        }
        if (!(best > 0.0 && best < __longlong_as_double(0x7ff0000000000000ll))) return false;
#pragma unroll
        for (int r = k + 1; r < 8; ++r)
            if (p == r) {
#pragma unroll
                for (int c = k; c < 9; ++c) { const double t = a[k][c]; a[k][c] = a[r][c]; a[r][c] = t; }
            }
        const double d = a[k][k];
#pragma unroll
        for (int r = k + 1; r < 8; ++r) {
            const double f = a[r][k] / d;
#pragma unroll
            for (int c = k + 1; c < 9; ++c) a[r][c] = a[r][c] - f * a[k][c];
        }
    }
#pragma unroll
    for (int k = 7; k >= 0; --k) {
        double s = a[k][8];
#pragma unroll
        for (int c = k + 1; c < 8; ++c) s = s - a[k][c] * h[c];
        h[k] = s / a[k][k];
    }
    return true;
}

// Normalisation (u, v) = ((x - cx) * s, (y - cy) * s) of each image.
struct Norm { double cx1, cy1, s1, cx2, cy2, s2; };

// normalises K points in place to centroid 0 and mean distance sqrt(2), sums in index order -> centroid and scale
template <int K>
__device__ __forceinline__ void normalise(double (&x)[K], double (&y)[K], double& cx, double& cy, double& s) {
    cx = x[0]; cy = y[0];
#pragma unroll
    for (int i = 1; i < K; ++i) { cx = cx + x[i]; cy = cy + y[i]; }
    cx = cx / (double)K;
    cy = cy / (double)K;
    double sd = 0.0;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        const double dx = x[i] - cx, dy = y[i] - cy, d = sqrt((dx * dx) + (dy * dy));
        sd = i ? sd + d : d;
    }
    s = kSqrt2 / (sd / (double)K);
#pragma unroll
    for (int i = 0; i < K; ++i) { x[i] = (x[i] - cx) * s; y[i] = (y[i] - cy) * s; }
}

__device__ __forceinline__ int clamp_count(const int32_t* count, int b, int M) {
    const int n = count[b];
    return n < 0 ? 0 : (n > M ? M : n);
}

// One thread per model slot g (0 <= g < slots) of a pair, 9 doubles each in hyp [B][slots][9]; the pair's points are
// streamed through shared memory in chunks.  Model supplies kMinMatches (fewer matches: the pair has no model),
// kPairThr (true: pair b's squared threshold is thr2_pair[b], not thr2), valid(P) (false for an empty slot) and
// inlier(P, x1, y1, x2, y2, thr2).
// key = (inliers + 1) << 32 | (0xFFFFFFFF - g): an empty slot scores -1 (key < 2^32), the maximum key is the highest
// count, and among equal counts the lowest slot.  Each warp combines its keys and issues one atomicMax into best[b].
template <class Model>
__global__ void __launch_bounds__(kScoreThreads) ransac_score_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                     const int32_t* __restrict__ count, int M, int slots,
                                                                     double thr2, const double* __restrict__ hyp,
                                                                     u64* __restrict__ best,
                                                                     const double* __restrict__ thr2_pair = nullptr) {
    __shared__ double4 pts[kChunk];
    const int g = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    const int n = clamp_count(count, b, M);
    if (n < Model::kMinMatches) return;                              // every slot of the pair is empty
    if constexpr (Model::kPairThr) thr2 = thr2_pair[b];
    double P[9];
    bool ok = g < slots;
    if (ok) {
        const double* src = hyp + ((size_t)b * slots + g) * 9;
#pragma unroll
        for (int i = 0; i < 9; ++i) P[i] = src[i];
        ok = Model::valid(P);
    }
    const double* q1 = p1 + (size_t)b * M * 2;
    const double* q2 = p2 + (size_t)b * M * 2;
    int inl = 0;
    for (int base = 0; base < n; base += kChunk) {
        const int m = min(kChunk, n - base);
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += blockDim.x) {
            const size_t q = 2 * (size_t)(base + i);
            pts[i] = make_double4(q1[q], q1[q + 1], q2[q], q2[q + 1]);
        }
        __syncthreads();
        if (ok) {
#pragma unroll 4
            for (int i = 0; i < m; ++i) {
                const double4 p = pts[i];
                inl += Model::inlier(P, p.x, p.y, p.z, p.w, thr2) ? 1 : 0;
            }
        }
    }
    u64 key = g < slots ? ((u64)(ok ? inl + 1 : 0) << 32) | (u64)(0xFFFFFFFFu - (unsigned)g) : 0ull;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const u64 v = __shfl_xor_sync(0xffffffffu, key, o);
        key = v > key ? v : key;
    }
    if ((threadIdx.x & 31) == 0 && key) atomicMax(best + b, key);
}

// Block sum of K per-thread partials in a fixed order (restated by oracle/homography.py: block_sum): a tree inside each
// warp (lane t += lane t + o, o = 16 .. 1), then a tree over the 8 warp sums (w += w + o, o = 4, 2, 1).
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double (*warp_part)[kRefitThreads / 32], double* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        double s = v[q];
#pragma unroll
        for (int o = 16; o; o >>= 1) s = s + __shfl_down_sync(0xffffffffu, s, o);
        if (lane == 0) warp_part[q][warp] = s;
    }
    __syncthreads();
    for (int q = threadIdx.x; q < K; q += blockDim.x) {
        double w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = warp_part[q][j];
#pragma unroll
        for (int o = 4; o; o >>= 1)
#pragma unroll
            for (int j = 0; j < o; ++j) w[j] = w[j] + w[j + o];
        out[q] = w[0];
    }
    __syncthreads();
}

// The refit kernels' normalisation of the cnt points where mask is set.  Thread t accumulates points t, t + 256, ...
// (a point outside the mask adds 0.0) and block_sum combines them:
//   pass A: sums of x1, y1, x2, y2 -> centroids = sum / cnt;
//   pass B: sums of the distances to the centroids -> s = sqrt(2) / (sum / cnt).
__device__ __forceinline__ Norm refit_norm(const double* q1, const double* q2, int n, int cnt, const uint8_t* m,
                                           double (*warp_part)[kRefitThreads / 32], double* tot) {
    const int t = threadIdx.x, rows = (n + kRefitThreads - 1) / kRefitThreads;
    const double dn = (double)cnt;
    double sA[4] = {0.0, 0.0, 0.0, 0.0};
    for (int r = 0; r < rows; ++r) {
        const int i = r * kRefitThreads + t;
        const bool in = i < n && m[i];
        sA[0] = sA[0] + (in ? q1[2 * i] : 0.0);
        sA[1] = sA[1] + (in ? q1[2 * i + 1] : 0.0);
        sA[2] = sA[2] + (in ? q2[2 * i] : 0.0);
        sA[3] = sA[3] + (in ? q2[2 * i + 1] : 0.0);
    }
    block_sum<4>(sA, warp_part, tot);
    Norm nm;
    nm.cx1 = tot[0] / dn; nm.cy1 = tot[1] / dn; nm.cx2 = tot[2] / dn; nm.cy2 = tot[3] / dn;
    __syncthreads();
    double sB[2] = {0.0, 0.0};
    for (int r = 0; r < rows; ++r) {
        const int i = r * kRefitThreads + t;
        const bool in = i < n && m[i];
        double d1 = 0.0, d2 = 0.0;
        if (in) {
            const double ax = q1[2 * i] - nm.cx1, ay = q1[2 * i + 1] - nm.cy1;
            const double bx = q2[2 * i] - nm.cx2, by = q2[2 * i + 1] - nm.cy2;
            d1 = sqrt((ax * ax) + (ay * ay));
            d2 = sqrt((bx * bx) + (by * by));
        }
        sB[0] = sB[0] + d1;
        sB[1] = sB[1] + d2;
    }
    block_sum<2>(sB, warp_part, tot);
    nm.s1 = kSqrt2 / (tot[0] / dn);
    nm.s2 = kSqrt2 / (tot[1] / dn);
    __syncthreads();
    return nm;
}

// The inliers of model G among the n points, written to mask -> their count (every thread of the CTA gets it).
template <class Model>
__device__ __forceinline__ int mark_inliers(const double (&G)[9], const double* q1, const double* q2, int n, double thr2,
                                            uint8_t* mask, int* cnt_sh) {
    const int t = threadIdx.x;
    if (t == 0) *cnt_sh = 0;
    __syncthreads();
    int c = 0;
    for (int i = t; i < n; i += blockDim.x) {
        const bool in = Model::inlier(G, q1[2 * i], q1[2 * i + 1], q2[2 * i], q2[2 * i + 1], thr2);
        mask[i] = in ? 1 : 0;
        c += in ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((t & 31) == 0) atomicAdd(cnt_sh, c);
    __syncthreads();
    const int r = *cnt_sh;
    __syncthreads();
    return r;
}

__device__ __forceinline__ double det3(const double (&m)[9]) {
    return ((m[0] * ((m[4] * m[8]) - (m[5] * m[7]))) - (m[1] * ((m[3] * m[8]) - (m[5] * m[6])))) +
           (m[2] * ((m[3] * m[7]) - (m[4] * m[6])));
}

// F / |F|_F (sum of squares in index order) with its first largest-magnitude entry made positive (oracle/fundamental.py:
// scale_unit).  False when the norm is 0 or not finite.
__device__ __forceinline__ bool scale_unit(double (&F)[9]) {
    double s = F[0] * F[0];
#pragma unroll
    for (int i = 1; i < 9; ++i) s = s + (F[i] * F[i]);
    const double nrm = sqrt(s);
    if (!(nrm > 0.0 && nrm < kInf)) return false;
#pragma unroll
    for (int i = 0; i < 9; ++i) F[i] = F[i] / nrm;
    double big = F[0];
#pragma unroll
    for (int i = 1; i < 9; ++i) big = fabs(F[i]) > fabs(big) ? F[i] : big;
    if (big < 0.0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) F[i] = -F[i];
    }
    return true;
}

// Cyclic Jacobi on the symmetric A (oracle/fundamental.py: jacobi_eigh); V receives the eigenvectors as columns, the
// diagonal of A the eigenvalues, and the return value is the column of the first smallest eigenvalue.
template <int N>
__device__ int jacobi_smallest(double (&A)[N][N], double (&V)[N][N]) {
    for (int i = 0; i < N; ++i)
        for (int j = 0; j < N; ++j) V[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
        double off = 0.0, dsq = 0.0;
        for (int p = 0; p < N; ++p) {
            dsq = dsq + (A[p][p] * A[p][p]);
            for (int q = p + 1; q < N; ++q) off = off + (A[p][q] * A[p][q]);
        }
        if (!(off > kJacobiTol2 * dsq)) break;
        for (int p = 0; p < N - 1; ++p)
            for (int q = p + 1; q < N; ++q) {
                const double apq = A[p][q];
                if (apq == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                double t = 1.0 / (fabs(theta) + sqrt((theta * theta) + 1.0));
                if (theta < 0.0) t = -t;
                const double c = 1.0 / sqrt((t * t) + 1.0), s = t * c;
                for (int k = 0; k < N; ++k) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = (c * akp) - (s * akq);
                    A[k][q] = (s * akp) + (c * akq);
                }
                for (int k = 0; k < N; ++k) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = (c * apk) - (s * aqk);
                    A[q][k] = (s * apk) + (c * aqk);
                }
                A[p][q] = 0.0;
                A[q][p] = 0.0;
                for (int k = 0; k < N; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = (c * vkp) - (s * vkq);
                    V[k][q] = (s * vkp) + (c * vkq);
                }
            }
    }
    int j = 0;
    for (int i = 1; i < N; ++i) if (A[i][i] < A[j][j]) j = i;
    return j;
}

inline size_t best_bytes(int B) { return align_up((size_t)B * sizeof(u64), 256); }

}  // namespace
}  // namespace balf
