// RANSAC fundamental-matrix estimation from matched keypoints, batched over image pairs.
//
// No reference counterpart: the reference's GoPro evaluation parser (balf/configs/config_gopro_eval.py) names epipolar
// verification of consecutive frames without implementing it.  The semantics are defined here, documented in
// include/balf_b200.h and restated in oracle/fundamental.py; the tests check the kernels against that restatement bit for
// bit and against cv2.findFundamentalMat on accuracy.
//
// float64 compiled with -fmad=false (build.py), and only + - * / sqrt and comparisons: every one of them is correctly
// rounded on both the GPU and the host, so the restatement can match bit for bit.  That rules out cbrt / acos / cos of the
// usual closed-form cubic: its roots are bracketed and bisected instead.
//
// Three kernels per call, in the homography's pattern (ransac.cuh holds the shared pieces):
//   fundamental_hyp_kernel  one thread per (pair, hypothesis): 7 distinct indices, the 7-point solver, up to 3 models
//                           written to slots 3 h + m of the workspace (an all-zero slot holds no model).
//   ransac_score_kernel     one thread per (pair, model slot), the points streamed through shared memory; the packed key
//                           gives (highest count, lowest 3 h + m).  Holding the 3 models of a hypothesis in one thread
//                           needs 27 doubles more per thread (DESIGN.md section 4.4 has the register counts), so each
//                           slot is a thread of its own.
//   fundamental_refit_kernel  one CTA per pair: the winner's inliers, then normalised 8-point refits (smallest
//                           eigenvector of the 9x9 normal matrix by cyclic Jacobi, rank 2 by a 3x3 Jacobi of F^T F) while
//                           the inlier set grows.
#include "ransac.cuh"
#include "../../include/balf_b200.h"

namespace balf {
namespace {

constexpr int kSample = 7;
constexpr int kMaxDraws = 64;            // 32 counters leave about 5 % of the samples of n = 7 without 7 distinct indices
constexpr int kModels = 3;               // real roots of the 7-point cubic
constexpr int kRefitPasses = 8;
constexpr int kRefitMin = 8;             // the 8-point refit needs 8 inliers
constexpr int kMaxBisect = 200;
constexpr int kNormalTerms = 45;         // upper triangle of the 9x9 normal matrix

// F = T2^T Fn T1 with T = [[s, 0, -s cx], [0, s, -s cy], [0, 0, 1]], then unit Frobenius norm with the first
// largest-magnitude entry positive.  False when the norm is 0 or not finite.
__device__ __forceinline__ bool denormalise(const double (&Fn)[9], const Norm& n, double (&F)[9]) {
    double G[9];
    const double tx = -(n.s1 * n.cx1), ty = -(n.s1 * n.cy1);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        G[3 * r] = Fn[3 * r] * n.s1;
        G[3 * r + 1] = Fn[3 * r + 1] * n.s1;
        G[3 * r + 2] = ((Fn[3 * r] * tx) + (Fn[3 * r + 1] * ty)) + Fn[3 * r + 2];
    }
    const double ux = -(n.s2 * n.cx2), uy = -(n.s2 * n.cy2);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        F[c] = n.s2 * G[c];
        F[3 + c] = n.s2 * G[3 + c];
        F[6 + c] = ((ux * G[c]) + (uy * G[3 + c])) + G[6 + c];
    }
    return scale_unit(F);
}

// Epipolar inlier rule: l2 = F x1 = (a, b, c), s = x2^T l2, l1 = F^T x2 = (a', b', .); both point-to-line distances at
// most thr, in squared form: s^2 <= thr^2 (a^2 + b^2) and s^2 <= thr^2 (a'^2 + b'^2), each a^2 + b^2 finite and > 0.
struct Fundamental {
    static constexpr int kMinMatches = kSample;
    static constexpr bool kPairThr = false;
    static __device__ __forceinline__ bool valid(const double (&F)[9]) {
        bool nz = false;
#pragma unroll
        for (int i = 0; i < 9; ++i) nz |= F[i] != 0.0;
        return nz;
    }
    static __device__ __forceinline__ bool inlier(const double (&F)[9], double x1, double y1, double x2, double y2,
                                                  double thr2) {
        const double a = ((F[0] * x1) + (F[1] * y1)) + F[2];
        const double b = ((F[3] * x1) + (F[4] * y1)) + F[5];
        const double c = ((F[6] * x1) + (F[7] * y1)) + F[8];
        const double s = ((x2 * a) + (y2 * b)) + c;
        const double ap = ((F[0] * x2) + (F[3] * y2)) + F[6];
        const double bp = ((F[1] * x2) + (F[4] * y2)) + F[7];
        const double s2 = s * s, n2 = (a * a) + (b * b), n1 = (ap * ap) + (bp * bp);
        return n2 > 0.0 && n2 < kInf && n1 > 0.0 && n1 < kInf && s2 <= thr2 * n2 && s2 <= thr2 * n1;
    }
};

__device__ __forceinline__ double poly3(const double (&c)[4], double x) {
    return ((((c[3] * x) + c[2]) * x + c[1]) * x) + c[0];
}

// Real roots of c0 + c1 x + c2 x^2 + c3 x^3 in ascending order -> their count (oracle/fundamental.py: cubic_roots).  The
// degree is the highest whose Cauchy bound R is finite; the derivative's roots, clamped to [-R, R], split [-R, R] into
// monotone pieces, and each piece whose ends differ in sign is bisected at a / 2 + b / 2.
__device__ int cubic_roots(const double (&c)[4], double (&root)[kModels]) {
    const double a0 = fabs(c[0]), a1 = fabs(c[1]), a2 = fabs(c[2]), a3 = fabs(c[3]);
    const double R3 = 1.0 + (fmax(fmax(a0, a1), a2) / a3);
    const double R2 = 1.0 + (fmax(a0, a1) / a2);
    const double R1 = 1.0 + (a0 / a1);
    double R, k1, k2;
    if (R3 > 0.0 && R3 < kInf) {
        R = R3;
        k1 = k2 = -R;
        const double disc = (c[2] * c[2]) - ((3.0 * c[3]) * c[1]);
        if (disc > 0.0) {
            const double sq = sqrt(disc);
            const double q = c[2] >= 0.0 ? -(c[2] + sq) : sq - c[2];
            const double x1 = q / (3.0 * c[3]), x2 = c[1] / q;
            k1 = fmin(x1, x2);
            k2 = fmax(x1, x2);
        }
    } else if (R2 > 0.0 && R2 < kInf) {
        R = R2;
        k1 = k2 = (-c[1]) / (2.0 * c[2]);
    } else if (R1 > 0.0 && R1 < kInf) {
        R = R1;
        k1 = k2 = -R;
    } else {
        return 0;
    }
    k1 = k1 < -R ? -R : (k1 > R ? R : k1);
    k2 = k2 < -R ? -R : (k2 > R ? R : k2);
    const double knot[4] = {-R, k1, k2, R};
    int cnt = 0;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        const double a = knot[p], b = knot[p + 1];
        double flo = poly3(c, a);
        const double fb = poly3(c, b);
        if (!(a < b && (fb == 0.0 || (flo != 0.0 && (flo < 0.0) != (fb < 0.0))))) continue;
        double lo = a, hi = b, mid = b;
        if (fb != 0.0) {
            for (int it = 0; it < kMaxBisect; ++it) {
                mid = (0.5 * lo) + (0.5 * hi);
                if (!(lo < mid && mid < hi)) break;
                const double fm = poly3(c, mid);
                if (fm == 0.0) break;
                if ((fm < 0.0) == (flo < 0.0)) { lo = mid; flo = fm; } else { hi = mid; }
            }
        }
#pragma unroll
        for (int j = 0; j < kModels; ++j) if (j == cnt) root[j] = mid;
        ++cnt;
    }
    return cnt;
}

// One vector of the 2-D null space of the 7x9 system x2^T F x1 = 0 (normalised points), by solve8 with an eighth row
// that fixes f7: v = 0 gives F1 with f8 = 1, f7 = 0 and v = 1 gives F2 with f8 = 0, f7 = 1.  The unit row is never a
// pivot before column 7, so both run the same elimination of the 7 rows.  Not inlined: the two eliminations then share
// one register allocation, and the hypothesis kernel does not spill.
__device__ __noinline__ bool null_vector(const double (&u1)[kSample], const double (&v1)[kSample], const double (&u2)[kSample],
                                         const double (&v2)[kSample], int v, double (&out)[9]) {
    double a[8][9], f[8];
#pragma unroll
    for (int j = 0; j < kSample; ++j) {
        a[j][0] = u2[j] * u1[j]; a[j][1] = u2[j] * v1[j]; a[j][2] = u2[j];
        a[j][3] = v2[j] * u1[j]; a[j][4] = v2[j] * v1[j]; a[j][5] = v2[j];
        a[j][6] = u1[j]; a[j][7] = v1[j]; a[j][8] = v == 0 ? -1.0 : 0.0;
    }
#pragma unroll
    for (int c = 0; c < 9; ++c) a[7][c] = 0.0;
    a[7][7] = 1.0;
    a[7][8] = v == 0 ? 0.0 : 1.0;
    if (!solve8(a, f)) return false;
#pragma unroll
    for (int i = 0; i < 8; ++i) out[i] = f[i];
    out[8] = v == 0 ? 1.0 : 0.0;
    return true;
}

// hypothesis h of pair b (n valid matches) -> up to 3 models in F (slots without one are zeros)
__device__ __forceinline__ void make_hypothesis(const double* __restrict__ p1, const double* __restrict__ p2, int n, int M,
                                                int b, int h, u64 seed, double (&F)[kModels][9]) {
#pragma unroll
    for (int m = 0; m < kModels; ++m)
#pragma unroll
        for (int i = 0; i < 9; ++i) F[m][i] = 0.0;
    int idx[kSample];
#pragma unroll
    for (int j = 0; j < kSample; ++j) idx[j] = 0;
    if (!(n >= kSample && draw_sample<kSample, kMaxDraws>(seed, b, h, n, idx))) return;
    const double* q1 = p1 + (size_t)b * M * 2;
    const double* q2 = p2 + (size_t)b * M * 2;
    double x1[kSample], y1[kSample], x2[kSample], y2[kSample];
#pragma unroll
    for (int j = 0; j < kSample; ++j) {
        x1[j] = q1[2 * idx[j]]; y1[j] = q1[2 * idx[j] + 1];
        x2[j] = q2[2 * idx[j]]; y2[j] = q2[2 * idx[j] + 1];
    }
    Norm nm;
    normalise<kSample>(x1, y1, nm.cx1, nm.cy1, nm.s1);
    normalise<kSample>(x2, y2, nm.cx2, nm.cy2, nm.s2);
    double F1[9], F2[9];
    if (!null_vector(x1, y1, x2, y2, 0, F1) || !null_vector(x1, y1, x2, y2, 1, F2)) return;
    // det(lam F1 + (1 - lam) F2) = det(F2 + lam D), D = F1 - F2: c1 sums the determinants of F2 with column j taken from D,
    // c2 those of D with column j taken from F2.
    double D[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) D[i] = F1[i] - F2[i];
    double c[4];
    c[0] = det3(F2);
    c[3] = det3(D);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        double A[9], E[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            A[i] = i % 3 == j ? D[i] : F2[i];
            E[i] = i % 3 == j ? F2[i] : D[i];
        }
        c[1] = j ? c[1] + det3(A) : det3(A);
        c[2] = j ? c[2] + det3(E) : det3(E);
    }
    double root[kModels];
    const int nr = cubic_roots(c, root);
#pragma unroll
    for (int m = 0; m < kModels; ++m) {
        if (m >= nr) break;
        const double lam = root[m], mu = 1.0 - lam;
        double Fn[9], G[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) Fn[i] = (lam * F1[i]) + (mu * F2[i]);
        if (denormalise(Fn, nm, G)) {
#pragma unroll
            for (int i = 0; i < 9; ++i) F[m][i] = G[i];
        }
    }
}

__global__ void __launch_bounds__(kHypThreads) fundamental_hyp_kernel(const double* __restrict__ p1,
                                                                      const double* __restrict__ p2,
                                                                      const int32_t* __restrict__ count, int M, int iters,
                                                                      u64 seed, double* __restrict__ hyp) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (h >= iters) return;
    double F[kModels][9];
    make_hypothesis(p1, p2, clamp_count(count, b, M), M, b, h, seed, F);
    double* out = hyp + ((size_t)b * iters + h) * (kModels * 9);
#pragma unroll
    for (int m = 0; m < kModels; ++m)
#pragma unroll
        for (int i = 0; i < 9; ++i) out[9 * m + i] = F[m][i];
}

// The normalised 8-point fit from the 45 normal-matrix sums: the smallest eigenvector f, then F - (F v3) v3^T with v3 the
// smallest eigenvector of F^T F (the nearest rank-2 matrix), denormalised and scaled.
__device__ bool solve_normal(const double* tot, const Norm& nm, double (&F)[9]) {
    double A[9][9], V[9][9];
    int q = 0;
    for (int i = 0; i < 9; ++i)
        for (int j = i; j < 9; ++j, ++q) { A[i][j] = tot[q]; A[j][i] = tot[q]; }
    const int e = jacobi_smallest<9>(A, V);
    double f[3][3];
    for (int i = 0; i < 9; ++i) f[i / 3][i % 3] = V[i][e];
    double T[3][3], U[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) T[i][j] = ((f[0][i] * f[0][j]) + (f[1][i] * f[1][j])) + (f[2][i] * f[2][j]);
    const int e3 = jacobi_smallest<3>(T, U);
    const double v0 = U[0][e3], v1 = U[1][e3], v2 = U[2][e3];
    double Fn[9];
    for (int r = 0; r < 3; ++r) {
        const double w = ((f[r][0] * v0) + (f[r][1] * v1)) + (f[r][2] * v2);
        Fn[3 * r] = f[r][0] - (w * v0);
        Fn[3 * r + 1] = f[r][1] - (w * v1);
        Fn[3 * r + 2] = f[r][2] - (w * v2);
    }
    return denormalise(Fn, nm, F);
}

// One CTA per pair.  refit_norm (ransac.cuh) normalises the inliers; thread t then sums the 45 products r_i r_j (i <= j,
// row-major) of the epipolar rows r = [u2 u1, u2 v1, u2, v2 u1, v2 v1, v2, u1, v1, 1] of its points t, t + 256, ... and
// block_sum combines them; thread 0 solves.  Each refit replaces F and its inliers; the refits repeat while the inlier
// count grows, at most kRefitPasses of them, and only while it is at least kRefitMin.
__global__ void __launch_bounds__(kRefitThreads) fundamental_refit_kernel(
    const double* __restrict__ p1, const double* __restrict__ p2, const int32_t* __restrict__ count, int M, int iters,
    double thr2, const double* __restrict__ hyp, const u64* __restrict__ best, double* __restrict__ F_out,
    uint8_t* __restrict__ mask_out, int32_t* __restrict__ n_out) {
    __shared__ uint8_t mask[kMaxMatches];
    __shared__ double warp_part[kNormalTerms][kRefitThreads / 32];
    __shared__ double tot[kNormalTerms];
    __shared__ double Fs[9];
    __shared__ int cnt_sh, ok_sh;
    const int b = blockIdx.x, t = threadIdx.x;
    const int n = clamp_count(count, b, M);
    const u64 key = best[b];
    const double* q1 = p1 + (size_t)b * M * 2;
    const double* q2 = p2 + (size_t)b * M * 2;
    if (n < kSample || (key >> 32) == 0) {
        if (t < 9) F_out[9 * b + t] = 0.0;
        if (t == 0) n_out[b] = 0;
        for (int i = t; i < M; i += blockDim.x) mask_out[(size_t)b * M + i] = 0;
        return;
    }
    const unsigned g = 0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull);
    double F[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) F[i] = hyp[((size_t)b * iters * kModels + g) * 9 + i];
    int cnt = mark_inliers<Fundamental>(F, q1, q2, n, thr2, mask, &cnt_sh);
    const int rows = (n + kRefitThreads - 1) / kRefitThreads;
    for (int pass = 0; pass < kRefitPasses && cnt >= kRefitMin; ++pass) {
        const uint8_t* m = mask;
        const Norm nm = refit_norm(q1, q2, n, cnt, m, warp_part, tot);
        double sC[kNormalTerms];
#pragma unroll
        for (int q = 0; q < kNormalTerms; ++q) sC[q] = 0.0;
        for (int r = 0; r < rows; ++r) {
            const int i = r * kRefitThreads + t;
            const bool in = i < n && m[i];
            double e[9];
            if (in) {
                const double u1 = (q1[2 * i] - nm.cx1) * nm.s1, v1 = (q1[2 * i + 1] - nm.cy1) * nm.s1;
                const double u2 = (q2[2 * i] - nm.cx2) * nm.s2, v2 = (q2[2 * i + 1] - nm.cy2) * nm.s2;
                e[0] = u2 * u1; e[1] = u2 * v1; e[2] = u2; e[3] = v2 * u1; e[4] = v2 * v1; e[5] = v2;
                e[6] = u1; e[7] = v1; e[8] = 1.0;
            }
            int q = 0;
#pragma unroll
            for (int ii = 0; ii < 9; ++ii)
#pragma unroll
                for (int jj = ii; jj < 9; ++jj, ++q) sC[q] = sC[q] + (in ? e[ii] * e[jj] : 0.0);
        }
        block_sum<kNormalTerms>(sC, warp_part, tot);
        if (t == 0) {
            double G[9];
            ok_sh = solve_normal(tot, nm, G);
            for (int i = 0; i < 9; ++i) Fs[i] = G[i];
        }
        __syncthreads();
        if (!ok_sh) break;
#pragma unroll
        for (int i = 0; i < 9; ++i) F[i] = Fs[i];
        const int c2 = mark_inliers<Fundamental>(F, q1, q2, n, thr2, mask, &cnt_sh);   // the sums above are complete
        const bool grew = c2 > cnt;
        cnt = c2;
        if (!grew) break;
    }
    if (t < 9) F_out[9 * b + t] = F[t];
    if (t == 0) n_out[b] = cnt;
    for (int i = t; i < M; i += blockDim.x) mask_out[(size_t)b * M + i] = i < n ? mask[i] : 0;
}

}  // namespace
}  // namespace balf

using namespace balf;

extern "C" size_t balf_fundamental_workspace_bytes(int B, int M, int iters) {
    if (B < 0 || M < 0 || iters < 1 || iters > kMaxIters) return 0;
    return best_bytes(B) + (size_t)B * iters * kModels * 9 * sizeof(double) + 256;
}

extern "C" int balf_find_fundamental_ransac(const double* p1, const double* p2, const int32_t* count, int B, int M, double thr,
                                            int iters, uint64_t seed, double* F, uint8_t* inlier_mask, int32_t* n_inliers,
                                            void* workspace, size_t workspace_bytes, void* stream) {
    BALF_REQUIRE(B >= 0 && B <= 65535, "find_fundamental_ransac: B = %d outside [0, 65535]", B);
    BALF_REQUIRE(M >= 0 && M <= kMaxMatches, "find_fundamental_ransac: M = %d outside [0, %d]", M, kMaxMatches);
    BALF_REQUIRE(thr > 0.0, "find_fundamental_ransac: thr must be > 0");
    BALF_REQUIRE(iters >= 1 && iters <= kMaxIters, "find_fundamental_ransac: iters = %d outside [1, %d]", iters, kMaxIters);
    if (B == 0) return 0;
    BALF_REQUIRE(count && F && n_inliers && workspace && (M == 0 || (p1 && p2 && inlier_mask)),
                 "find_fundamental_ransac: null pointer argument");
    BALF_REQUIRE(workspace_bytes >= balf_fundamental_workspace_bytes(B, M, iters),
                 "find_fundamental_ransac: workspace of %zu bytes is too small (%zu needed)", workspace_bytes,
                 balf_fundamental_workspace_bytes(B, M, iters));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* base = reinterpret_cast<unsigned char*>(align_up((size_t)workspace, 256));
    u64* best = reinterpret_cast<u64*>(base);
    double* hyp = reinterpret_cast<double*>(base + best_bytes(B));
    const double thr2 = thr * thr;
    const int slots = iters * kModels;
    BALF_CUDA_OK(cudaMemsetAsync(best, 0, (size_t)B * sizeof(u64), st));
    {
        ProfScope p("fundamental_hyp", st);
        fundamental_hyp_kernel<<<dim3(cdiv(iters, kHypThreads), B), kHypThreads, 0, st>>>(p1, p2, count, M, iters, seed, hyp);
    }
    {
        ProfScope p("fundamental_score", st);
        ransac_score_kernel<Fundamental><<<dim3(cdiv(slots, kScoreThreads), B), kScoreThreads, 0, st>>>(p1, p2, count, M, slots,
                                                                                                       thr2, hyp, best);
    }
    {
        ProfScope p("fundamental_refit", st);
        fundamental_refit_kernel<<<B, kRefitThreads, 0, st>>>(p1, p2, count, M, iters, thr2, hyp, best, F, inlier_mask,
                                                              n_inliers);
    }
    BALF_COUNT_LAUNCH(3);
    BALF_LAUNCH_OK();
    return 0;
}
