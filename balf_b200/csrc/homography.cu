// RANSAC homography estimation from matched keypoints, batched over image pairs.
//
// No reference counterpart: the reference stops at the SMNN match list (demo/demo_match.py:97-112) and its evaluation
// parsers (balf/configs/config_hpatches.py, config_gopro_eval.py) name homography estimation without implementing it.  The
// semantics are defined here, documented in include/balf_b200.h and restated in oracle/homography.py; the tests check the
// kernels against that restatement bit for bit and against cv2.findHomography(RANSAC) on accuracy.
//
// All arithmetic is float64 compiled with -fmad=false (build.py), so every product and sum rounds once, like NumPy's.
//
// Three kernels per call:
//   ransac_hyp_kernel    one thread per (pair, hypothesis): 4 distinct indices from the counter-based hash, normalised
//                        4-point DLT, H written to the workspace (H[8] = 0 marks a degenerate sample).
//   ransac_score_kernel  one thread per (pair, hypothesis), the pair's points streamed through shared memory in chunks;
//                        the inlier count and the hypothesis index are packed into one 64-bit key and atomicMax'ed into the
//                        pair's slot, which is order-independent and yields (highest count, lowest index).
//   ransac_refit_kernel  one CTA per pair: the winner's inliers, then least-squares refits while the inlier set grows.
// Splitting the hypothesis from the scoring keeps the 8x9 elimination out of the scoring kernel.  With the solver inside,
// the scoring kernel needs 106 registers and a 576-byte stack frame (2 CTAs of 256 threads per SM); split, it needs 60
// registers and no stack (4 CTAs per SM).  DESIGN.md section 4.4 has the timing of both layouts.
#include "ransac.cuh"
#include "../../include/balf_b200.h"

namespace balf {
namespace {

constexpr int kMaxDraws = 32;            // hash counters per hypothesis before the sample is declared degenerate
constexpr int kRefitPasses = 8;          // least-squares refits of the winner, stopping early once the set stops growing
constexpr double kCollinearTol = 1e-6;   // |cross| of two edges of a sample triangle, in normalised coordinates
constexpr int kNormalTerms = 44;         // 36 upper-triangle entries of the 8x8 normal matrix + 8 right-hand sides

// The solved hn maps normalised points of image 1 to those of image 2 (Norm: ransac.cuh); H = T2^-1 Hn T1, scaled so that
// H[2][2] = 1.  False when H[2][2] is 0 or not finite.
__device__ __forceinline__ bool denormalise(const double (&hn)[8], const Norm& n, double (&H)[9]) {
    const double Hn[9] = {hn[0], hn[1], hn[2], hn[3], hn[4], hn[5], hn[6], hn[7], 1.0};
    double G[9];                                                     // Hn T1, T1 = [[s1, 0, -s1 cx1], [0, s1, -s1 cy1], [0, 0, 1]]
    const double tx = -(n.s1 * n.cx1), ty = -(n.s1 * n.cy1);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        G[3 * r] = Hn[3 * r] * n.s1;
        G[3 * r + 1] = Hn[3 * r + 1] * n.s1;
        G[3 * r + 2] = ((Hn[3 * r] * tx) + (Hn[3 * r + 1] * ty)) + Hn[3 * r + 2];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {                                    // T2^-1 = [[1/s2, 0, cx2], [0, 1/s2, cy2], [0, 0, 1]]
        H[c] = (G[c] / n.s2) + (n.cx2 * G[6 + c]);
        H[3 + c] = (G[3 + c] / n.s2) + (n.cy2 * G[6 + c]);
        H[6 + c] = G[6 + c];
    }
    const double w = H[8];
    if (!(fabs(w) > 0.0 && fabs(w) < __longlong_as_double(0x7ff0000000000000ll))) return false;
#pragma unroll
    for (int i = 0; i < 8; ++i) H[i] = H[i] / w;
    H[8] = 1.0;
    return true;
}

// The inlier rule: w = (H p1)_z > 0 and |proj(H p1) - p2|^2 <= thr^2, with proj = (X, Y) * (1 / w).
__device__ __forceinline__ bool is_inlier(const double (&H)[9], double x1, double y1, double x2, double y2, double thr2) {
    const double X = ((H[0] * x1) + (H[1] * y1)) + H[2];
    const double Y = ((H[3] * x1) + (H[4] * y1)) + H[5];
    const double w = ((H[6] * x1) + (H[7] * y1)) + H[8];
    const double iw = 1.0 / w;
    const double dx = (X * iw) - x2, dy = (Y * iw) - y2;
    return w > 0.0 && ((dx * dx) + (dy * dy)) <= thr2;
}

// The model of ransac_score_kernel / mark_inliers (ransac.cuh); H[8] = 0 marks a degenerate hypothesis.
struct Homography {
    static constexpr int kMinMatches = 4;
    static __device__ __forceinline__ bool valid(const double (&H)[9]) { return H[8] != 0.0; }
    static __device__ __forceinline__ bool inlier(const double (&H)[9], double x1, double y1, double x2, double y2,
                                                  double thr2) {
        return is_inlier(H, x1, y1, x2, y2, thr2);
    }
};

__device__ __forceinline__ bool collinear3(double ax, double ay, double bx, double by, double cx, double cy) {
    const double dx1 = bx - ax, dy1 = by - ay, dx2 = cx - ax, dy2 = cy - ay;
    return !(fabs((dx1 * dy2) - (dy1 * dx2)) > kCollinearTol);       // NaN (coincident points) counts as collinear
}

// DLT rows of one correspondence (u, v) -> (u', v') with h33 = 1:
//   a = [u, v, 1, 0, 0, 0, -u u', -v u'] . h = u'      b = [0, 0, 0, u, v, 1, -u v', -v v'] . h = v'
__device__ __forceinline__ void dlt_rows(double u, double v, double up, double vp, double (&a)[8], double (&b)[8]) {
    a[0] = u; a[1] = v; a[2] = 1.0; a[3] = 0.0; a[4] = 0.0; a[5] = 0.0; a[6] = -(u * up); a[7] = -(v * up);
    b[0] = 0.0; b[1] = 0.0; b[2] = 0.0; b[3] = u; b[4] = v; b[5] = 1.0; b[6] = -(u * vp); b[7] = -(v * vp);
}

// hypothesis h of pair b (n valid matches) -> H; false for a degenerate sample
__device__ __forceinline__ bool make_hypothesis(const double* __restrict__ p1, const double* __restrict__ p2, int n, int M, int b,
                                                int h, u64 seed, double (&H)[9]) {
    int idx[4] = {0, 0, 0, 0};
    bool ok = n >= 4 && draw_sample<4, kMaxDraws>(seed, b, h, n, idx);
    if (ok) {
        const double* q1 = p1 + (size_t)b * M * 2;
        const double* q2 = p2 + (size_t)b * M * 2;
        double x1[4], y1[4], x2[4], y2[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            x1[j] = q1[2 * idx[j]]; y1[j] = q1[2 * idx[j] + 1];
            x2[j] = q2[2 * idx[j]]; y2[j] = q2[2 * idx[j] + 1];
        }
        Norm nm;
        normalise<4>(x1, y1, nm.cx1, nm.cy1, nm.s1);
        normalise<4>(x2, y2, nm.cx2, nm.cy2, nm.s2);
        const int tri[4][3] = {{0, 1, 2}, {0, 1, 3}, {0, 2, 3}, {1, 2, 3}};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int i0 = tri[t][0], i1 = tri[t][1], i2 = tri[t][2];
            ok = ok && !collinear3(x1[i0], y1[i0], x1[i1], y1[i1], x1[i2], y1[i2]) &&
                 !collinear3(x2[i0], y2[i0], x2[i1], y2[i1], x2[i2], y2[i2]);
        }
        if (ok) {
            double a[8][9], hn[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                double ra[8], rb[8];
                dlt_rows(x1[j], y1[j], x2[j], y2[j], ra, rb);
#pragma unroll
                for (int c = 0; c < 8; ++c) { a[2 * j][c] = ra[c]; a[2 * j + 1][c] = rb[c]; }
                a[2 * j][8] = x2[j];
                a[2 * j + 1][8] = y2[j];
            }
            ok = solve8(a, hn) && denormalise(hn, nm, H);
        }
    }
    return ok;
}

__global__ void __launch_bounds__(kHypThreads) ransac_hyp_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                 const int32_t* __restrict__ count, int M, int iters, u64 seed,
                                                                 double* __restrict__ hyp) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (h >= iters) return;
    double H[9];
    const bool ok = make_hypothesis(p1, p2, clamp_count(count, b, M), M, b, h, seed, H);
    double* out = hyp + ((size_t)b * iters + h) * 9;
#pragma unroll
    for (int i = 0; i < 9; ++i) out[i] = ok ? H[i] : 0.0;
}

// One CTA per pair.  refit_norm (ransac.cuh) normalises the inliers (passes A and B), then, with the same strided
// per-thread sums and block_sum:
//   pass C: the 36 upper-triangle entries a_i a_j + b_i b_j (row-major, i <= j) and the 8 right-hand sides a_i u' + b_i v'
//           of the normal equations -> the same solve8 / denormalise as the minimal solver.
// Each refit replaces the current H and its inliers (the least-squares fit is kept even when one more point fell inside
// the threshold of the 4-point sample); the refits repeat while the inlier count grows, at most kRefitPasses of them.
__global__ void __launch_bounds__(kRefitThreads) ransac_refit_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                     const int32_t* __restrict__ count, int M, int iters,
                                                                     double thr2, const double* __restrict__ hyp,
                                                                     const u64* __restrict__ best, double* __restrict__ H_out,
                                                                     uint8_t* __restrict__ mask_out, int32_t* __restrict__ n_out) {
    __shared__ uint8_t mask[kMaxMatches];
    __shared__ double warp_part[kNormalTerms][kRefitThreads / 32];
    __shared__ double tot[kNormalTerms];
    __shared__ double Hs[9];
    __shared__ int cnt_sh, ok_sh;
    const int b = blockIdx.x, t = threadIdx.x;
    const int n = clamp_count(count, b, M);
    const u64 key = best[b];
    const double* q1 = p1 + (size_t)b * M * 2;
    const double* q2 = p2 + (size_t)b * M * 2;
    if (n < 4 || (key >> 32) == 0) {
        if (t < 9) H_out[9 * b + t] = 0.0;
        if (t == 0) n_out[b] = 0;
        for (int i = t; i < M; i += blockDim.x) mask_out[(size_t)b * M + i] = 0;
        return;
    }
    const unsigned h = 0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull);
    double H[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) H[i] = hyp[((size_t)b * iters + h) * 9 + i];

    int cnt = mark_inliers<Homography>(H, q1, q2, n, thr2, mask, &cnt_sh);
    const int rows = (n + kRefitThreads - 1) / kRefitThreads;
    for (int pass = 0; pass < kRefitPasses && cnt >= 4; ++pass) {
        const uint8_t* m = mask;
        const Norm nm = refit_norm(q1, q2, n, cnt, m, warp_part, tot);
        double sC[kNormalTerms];
#pragma unroll
        for (int q = 0; q < kNormalTerms; ++q) sC[q] = 0.0;
        for (int r = 0; r < rows; ++r) {
            const int i = r * kRefitThreads + t;
            const bool in = i < n && m[i];
            double a[8], bb[8], up = 0.0, vp = 0.0;
            if (in) {
                up = (q2[2 * i] - nm.cx2) * nm.s2;
                vp = (q2[2 * i + 1] - nm.cy2) * nm.s2;
                dlt_rows((q1[2 * i] - nm.cx1) * nm.s1, (q1[2 * i + 1] - nm.cy1) * nm.s1, up, vp, a, bb);
            }
            int q = 0;
#pragma unroll
            for (int ii = 0; ii < 8; ++ii)
#pragma unroll
                for (int jj = ii; jj < 8; ++jj, ++q) sC[q] = sC[q] + (in ? (a[ii] * a[jj]) + (bb[ii] * bb[jj]) : 0.0);
#pragma unroll
            for (int ii = 0; ii < 8; ++ii) sC[36 + ii] = sC[36 + ii] + (in ? (a[ii] * up) + (bb[ii] * vp) : 0.0);
        }
        block_sum<kNormalTerms>(sC, warp_part, tot);
        if (t == 0) {
            double A[8][9], hn[8], G[9];
            int q = 0;
            for (int ii = 0; ii < 8; ++ii)
                for (int jj = ii; jj < 8; ++jj, ++q) { A[ii][jj] = tot[q]; A[jj][ii] = tot[q]; }
            for (int ii = 0; ii < 8; ++ii) A[ii][8] = tot[36 + ii];
            ok_sh = solve8(A, hn) && denormalise(hn, nm, G);
            for (int i = 0; i < 9; ++i) Hs[i] = G[i];
        }
        __syncthreads();
        if (!ok_sh) break;
#pragma unroll
        for (int i = 0; i < 9; ++i) H[i] = Hs[i];
        const int c2 = mark_inliers<Homography>(H, q1, q2, n, thr2, mask, &cnt_sh);                                      // the sums above are complete: the mask is free
        const bool grew = c2 > cnt;
        cnt = c2;
        if (!grew) break;
    }
    if (t < 9) H_out[9 * b + t] = H[t];
    if (t == 0) n_out[b] = cnt;
    for (int i = t; i < M; i += blockDim.x) mask_out[(size_t)b * M + i] = i < n ? mask[i] : 0;
}

}  // namespace
}  // namespace balf

using namespace balf;

extern "C" size_t balf_homography_workspace_bytes(int B, int M, int iters) {
    if (B < 0 || M < 0 || iters < 1 || iters > kMaxIters) return 0;
    return best_bytes(B) + (size_t)B * iters * 9 * sizeof(double) + 256;
}

extern "C" int balf_find_homography_ransac(const double* p1, const double* p2, const int32_t* count, int B, int M, double thr,
                                           int iters, uint64_t seed, double* H, uint8_t* inlier_mask, int32_t* n_inliers,
                                           void* workspace, size_t workspace_bytes, void* stream) {
    BALF_REQUIRE(B >= 0 && B <= 65535, "find_homography_ransac: B = %d outside [0, 65535]", B);
    BALF_REQUIRE(M >= 0 && M <= kMaxMatches, "find_homography_ransac: M = %d outside [0, %d]", M, kMaxMatches);
    BALF_REQUIRE(thr > 0.0, "find_homography_ransac: thr must be > 0");
    BALF_REQUIRE(iters >= 1 && iters <= kMaxIters, "find_homography_ransac: iters = %d outside [1, %d]", iters, kMaxIters);
    if (B == 0) return 0;
    BALF_REQUIRE(count && H && n_inliers && workspace && (M == 0 || (p1 && p2 && inlier_mask)),
                 "find_homography_ransac: null pointer argument");
    BALF_REQUIRE(workspace_bytes >= balf_homography_workspace_bytes(B, M, iters),
                 "find_homography_ransac: workspace of %zu bytes is too small (%zu needed)", workspace_bytes,
                 balf_homography_workspace_bytes(B, M, iters));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* base = reinterpret_cast<unsigned char*>(align_up((size_t)workspace, 256));
    u64* best = reinterpret_cast<u64*>(base);
    double* hyp = reinterpret_cast<double*>(base + best_bytes(B));
    const double thr2 = thr * thr;
    BALF_CUDA_OK(cudaMemsetAsync(best, 0, (size_t)B * sizeof(u64), st));
    {
        ProfScope p("ransac_hyp", st);
        ransac_hyp_kernel<<<dim3(cdiv(iters, kHypThreads), B), kHypThreads, 0, st>>>(p1, p2, count, M, iters, seed, hyp);
    }
    {
        ProfScope p("ransac_score", st);
        ransac_score_kernel<Homography><<<dim3(cdiv(iters, kScoreThreads), B), kScoreThreads, 0, st>>>(p1, p2, count, M, iters, thr2, hyp,
                                                                                           best);
    }
    {
        ProfScope p("ransac_refit", st);
        ransac_refit_kernel<<<B, kRefitThreads, 0, st>>>(p1, p2, count, M, iters, thr2, hyp, best, H, inlier_mask, n_inliers);
    }
    BALF_COUNT_LAUNCH(3);
    BALF_LAUNCH_OK();
    return 0;
}
