// RANSAC essential-matrix estimation and relative pose recovery for calibrated image pairs, batched over pairs.
//
// No reference counterpart.  The semantics are defined here, documented in include/balf_b200.h and restated in
// oracle/essential.py; the tests check the kernels against that restatement bit for bit and against cv2.findEssentialMat /
// cv2.recoverPose on accuracy.
//
// float64 compiled with -fmad=false (build.py), and only + - * / sqrt and comparisons: every one of them is correctly
// rounded on both the GPU and the host, so the restatement can match bit for bit.  That rules out cbrt, eigen-solvers and
// complex root finders for the degree-10 polynomial of the 5-point solver: its real roots come from a Sturm sequence and
// bisection instead.
//
// Five kernels, in the pattern of the homography and the fundamental matrix (ransac.cuh holds the shared pieces):
//   essential_calib_kernel  the calibrated points of every pair and its squared threshold, into the workspace; a pair
//                           whose K is invalid gets a count of 0 there, so every later kernel sees it as empty.
//   essential_hyp_kernel    one thread per (pair, hypothesis): 5 distinct indices, the 5-point solver, up to 10 models
//                           written to slots 10 h + m of the workspace (an all-zero slot holds no model).  The 10x20
//                           matrix and the Sturm sequence live in the thread's stack frame.
//   ransac_score_kernel     one thread per (pair, model slot), with the pair's threshold; the packed key gives (highest
//                           count, lowest 10 h + m).
//   essential_finish_kernel one CTA per pair: the winner and its inliers (no refit, as cv2.findEssentialMat).
//   recover_pose_kernel     one CTA per pair (balf_recover_pose): thread 0 decomposes E into 4 candidate poses, every
//                           thread counts the matches in front of both cameras for each of them.
#include "ransac.cuh"
#include "../../include/balf_b200.h"

namespace balf {
namespace {

constexpr int kSample = 5;
constexpr int kMaxDraws = 64;            // as the fundamental matrix: 5 of n = 5 need more than 32 counters now and then
constexpr int kModels = 10;              // real roots of the degree-10 polynomial
constexpr int kMaxBisect = 200;
constexpr int kSeq = 11;                 // Sturm sequence p0 .. p10 of a degree-10 polynomial
constexpr int kPoseThreads = 256;

// product tables (oracle/essential.py: LL, QL): term (i, j) of linear x linear forms [x, y, z, 1] goes to quadratic
// monomial LL[i][j] (x^2, xy, xz, x, y^2, yz, y, z^2, z, 1); term (m, k) of quadratic x linear to cubic monomial QL[m][k]
// in the column order of the 10x20 matrix (x^3, y^3, x^2y, xy^2, x^2z, x^2, y^2z, y^2, xyz, xy | xz^2, xz, x, yz^2, yz, y,
// z^3, z^2, z, 1).
__device__ constexpr int kLL[4][4] = {{0, 1, 2, 3}, {1, 4, 5, 6}, {2, 5, 7, 8}, {3, 6, 8, 9}};
__device__ constexpr int kQL[10][4] = {{0, 2, 4, 5},   {2, 3, 8, 9},   {4, 8, 10, 11},  {5, 9, 11, 12},  {3, 1, 6, 7},
                                       {8, 6, 13, 14}, {9, 7, 14, 15}, {10, 13, 16, 17}, {11, 14, 17, 18}, {12, 15, 18, 19}};

// fx, fy finite and > 0, last row (0, 0, 1)
__device__ __forceinline__ bool k_valid(const double* K) {
    return K[0] > 0.0 && K[0] < kInf && K[4] > 0.0 && K[4] < kInf && K[6] == 0.0 && K[7] == 0.0 && K[8] == 1.0;
}

// y' = (y - cy) / fy, x' = ((x - cx) - s y') / fx
__device__ __forceinline__ void calibrate(const double* K, double x, double y, double& xc, double& yc) {
    yc = (y - K[5]) / K[4];
    xc = ((x - K[2]) - (K[1] * yc)) / K[0];
}

// Inlier rule of cv2's EMEstimatorCallback::computeError in squared form: (a, b, c) = E x1, s = x2^T E x1,
// (a', b', .) = E^T x2, d = ((a^2 + b^2) + a'^2) + b'^2; an inlier has d finite and > 0 and s^2 <= thr2 d.
struct Essential {
    static constexpr int kMinMatches = kSample;
    static constexpr bool kPairThr = true;
    static __device__ __forceinline__ bool valid(const double (&E)[9]) {
        bool nz = false;
#pragma unroll
        for (int i = 0; i < 9; ++i) nz |= E[i] != 0.0;
        return nz;
    }
    static __device__ __forceinline__ bool inlier(const double (&E)[9], double x1, double y1, double x2, double y2,
                                                  double thr2) {
        const double a = ((E[0] * x1) + (E[1] * y1)) + E[2];
        const double b = ((E[3] * x1) + (E[4] * y1)) + E[5];
        const double c = ((E[6] * x1) + (E[7] * y1)) + E[8];
        const double s = ((x2 * a) + (y2 * b)) + c;
        const double ap = ((E[0] * x2) + (E[3] * y2)) + E[6];
        const double bp = ((E[1] * x2) + (E[4] * y2)) + E[7];
        const double d = (((a * a) + (b * b)) + (ap * ap)) + (bp * bp);
        return d > 0.0 && d < kInf && (s * s) <= thr2 * d;
    }
};

// ------------------------------------------------------------------------------------------ null space
// The 4-D null space of the 5x9 epipolar system (oracle/essential.py: null_basis, orthonormalise): the 5x5 system in
// e0..e4 with right-hand sides -a[.][5 + j] by one partial-pivot elimination (solve8's pivot rule) and four back
// substitutions (basis j has e_{5+j} = 1), then modified Gram-Schmidt in the order W, Z, Y, X.  False when a pivot or a
// norm is 0 or not finite.
__device__ __noinline__ bool null_basis(const double (&u1)[kSample], const double (&v1)[kSample],
                                        const double (&u2)[kSample], const double (&v2)[kSample], double (&N)[4][9]) {
    double a[kSample][9];
#pragma unroll
    for (int j = 0; j < kSample; ++j) {
        a[j][0] = u2[j] * u1[j]; a[j][1] = u2[j] * v1[j]; a[j][2] = u2[j];
        a[j][3] = v2[j] * u1[j]; a[j][4] = v2[j] * v1[j];
        a[j][5] = -v2[j]; a[j][6] = -u1[j]; a[j][7] = -v1[j]; a[j][8] = -1.0;   // minus the entries of e5 .. e8
    }
#pragma unroll
    for (int k = 0; k < kSample; ++k) {
        double best = fabs(a[k][k]);
        int p = k;
#pragma unroll
        for (int r = k + 1; r < kSample; ++r) {
            const double v = fabs(a[r][k]);
            if (!isnan(best) && (isnan(v) || v > best)) { best = v; p = r; }
        }
        if (!(best > 0.0 && best < kInf)) return false;
#pragma unroll
        for (int r = k + 1; r < kSample; ++r)
            if (p == r) {
#pragma unroll
                for (int c = k; c < 9; ++c) { const double t = a[k][c]; a[k][c] = a[r][c]; a[r][c] = t; }
            }
        const double d = a[k][k];
#pragma unroll
        for (int r = k + 1; r < kSample; ++r) {
            const double f = a[r][k] / d;
#pragma unroll
            for (int c = k + 1; c < 9; ++c) a[r][c] = a[r][c] - f * a[k][c];
        }
    }
    double B[4][9];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int i = 5; i < 9; ++i) B[j][i] = i == 5 + j ? 1.0 : 0.0;
#pragma unroll
        for (int k = kSample - 1; k >= 0; --k) {
            double s = a[k][5 + j];
#pragma unroll
            for (int c = k + 1; c < kSample; ++c) s = s - a[k][c] * B[j][c];
            B[j][k] = s / a[k][k];
        }
    }
    // Gram-Schmidt: N[3] = W', N[2] = Z', N[1] = Y', N[0] = X'
#pragma unroll
    for (int q = 3; q >= 0; --q) {
        double v[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) v[i] = B[q][i];
#pragma unroll
        for (int u = 3; u > q; --u) {
            double s = v[0] * N[u][0];
#pragma unroll
            for (int i = 1; i < 9; ++i) s = s + (v[i] * N[u][i]);
#pragma unroll
            for (int i = 0; i < 9; ++i) v[i] = v[i] - s * N[u][i];
        }
        double s = v[0] * v[0];
#pragma unroll
        for (int i = 1; i < 9; ++i) s = s + (v[i] * v[i]);
        const double nrm = sqrt(s);
        if (!(nrm > 0.0 && nrm < kInf)) return false;
#pragma unroll
        for (int i = 0; i < 9; ++i) N[q][i] = v[i] / nrm;
    }
    return true;
}

// ------------------------------------------------------------------------------------------ 10x20 matrix
// q = a x b, terms added in (i, j) row-major order onto 0.0
__device__ __forceinline__ void mul_ll(const double (&a)[4], const double (&b)[4], double (&q)[10]) {
#pragma unroll
    for (int m = 0; m < 10; ++m) q[m] = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) q[kLL[i][j]] = q[kLL[i][j]] + (a[i] * b[j]);
}

// c = q x b, terms added in (m, k) row-major order onto 0.0
__device__ __forceinline__ void mul_ql(const double (&q)[10], const double (&b)[4], double (&c)[20]) {
#pragma unroll
    for (int m = 0; m < 20; ++m) c[m] = 0.0;
#pragma unroll
    for (int m = 0; m < 10; ++m)
#pragma unroll
        for (int k = 0; k < 4; ++k) c[kQL[m][k]] = c[kQL[m][k]] + (q[m] * b[k]);
}

// The 10x20 matrix of E = x X + y Y + z Z + W (oracle/essential.py: constraint_matrix): row 0 det E, rows 1 + 3 i + j
// (L E)_ij with L = E E^T - (tr(E E^T) * 0.5) I.
__device__ __noinline__ void constraint_matrix(const double (&N)[4][9], double (*C)[20]) {
    double e[9][4];
#pragma unroll
    for (int i = 0; i < 9; ++i)
#pragma unroll
        for (int v = 0; v < 4; ++v) e[i][v] = N[v][i];
    {
        double p[10], q[10], m[10], c0[20], c1[20];
        mul_ll(e[4], e[8], p); mul_ll(e[5], e[7], q);
#pragma unroll
        for (int i = 0; i < 10; ++i) m[i] = p[i] - q[i];
        mul_ql(m, e[0], c0);
        mul_ll(e[3], e[8], p); mul_ll(e[5], e[6], q);
#pragma unroll
        for (int i = 0; i < 10; ++i) m[i] = p[i] - q[i];
        mul_ql(m, e[1], c1);
#pragma unroll
        for (int i = 0; i < 20; ++i) c0[i] = c0[i] - c1[i];
        mul_ll(e[3], e[7], p); mul_ll(e[4], e[6], q);
#pragma unroll
        for (int i = 0; i < 10; ++i) m[i] = p[i] - q[i];
        mul_ql(m, e[2], c1);
#pragma unroll
        for (int i = 0; i < 20; ++i) C[0][i] = c0[i] + c1[i];
    }
    double L[3][3][10];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double p[10], q[10];
            mul_ll(e[3 * i], e[3 * j], p);
            mul_ll(e[3 * i + 1], e[3 * j + 1], q);
#pragma unroll
            for (int k = 0; k < 10; ++k) p[k] = p[k] + q[k];
            mul_ll(e[3 * i + 2], e[3 * j + 2], q);
#pragma unroll
            for (int k = 0; k < 10; ++k) L[i][j][k] = p[k] + q[k];
        }
    double half[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) half[k] = ((L[0][0][k] + L[1][1][k]) + L[2][2][k]) * 0.5;
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 10; ++k) L[i][i][k] = L[i][i][k] - half[k];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double c0[20], c1[20];
            mul_ql(L[i][0], e[j], c0);
            mul_ql(L[i][1], e[3 + j], c1);
#pragma unroll
            for (int k = 0; k < 20; ++k) c0[k] = c0[k] + c1[k];
            mul_ql(L[i][2], e[6 + j], c1);
#pragma unroll
            for (int k = 0; k < 20; ++k) C[1 + 3 * i + j][k] = c0[k] + c1[k];
        }
}

// Gauss-Jordan on the first 10 columns with partial pivoting (oracle/essential.py: gauss_jordan); false when a pivot is
// 0 or not finite.
__device__ __noinline__ bool gauss_jordan(double (*C)[20]) {
    for (int k = 0; k < 10; ++k) {
        double best = fabs(C[k][k]);
        int p = k;
        for (int r = k + 1; r < 10; ++r) {
            const double v = fabs(C[r][k]);
            if (!isnan(best) && (isnan(v) || v > best)) { best = v; p = r; }
        }
        if (!(best > 0.0 && best < kInf)) return false;
        if (p != k)
            for (int c = k; c < 20; ++c) { const double t = C[k][c]; C[k][c] = C[p][c]; C[p][c] = t; }
        const double d = C[k][k];
        for (int c = k + 1; c < 20; ++c) C[k][c] = C[k][c] / d;
        for (int r = 0; r < 10; ++r) {
            if (r == k) continue;
            const double f = C[r][k];
            for (int c = k + 1; c < 20; ++c) C[r][c] = C[r][c] - f * C[k][c];
        }
    }
    return true;
}

// B(z) (oracle/essential.py: action_rows): row k = row(2k + 4) - z row(2k + 5), the x and y entries cubics, the 1 entry a
// quartic in z (ascending powers).
__device__ __forceinline__ void action_rows(double (*C)[20], double (&Bz)[3][3][5]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double* a = C[2 * k + 4];
        const double* b = C[2 * k + 5];
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int c2 = v ? 13 : 10, c1 = c2 + 1, c0 = c2 + 2;
            Bz[k][v][0] = a[c0];
            Bz[k][v][1] = a[c1] - b[c0];
            Bz[k][v][2] = a[c2] - b[c1];
            Bz[k][v][3] = -b[c2];
            Bz[k][v][4] = 0.0;
        }
        Bz[k][2][0] = a[19];
        Bz[k][2][1] = a[18] - b[19];
        Bz[k][2][2] = a[17] - b[18];
        Bz[k][2][3] = a[16] - b[17];
        Bz[k][2][4] = -b[16];
    }
}

// out (na + nb - 1 terms) = a x b, terms added in (i, j) row-major order onto 0.0
template <int NA, int NB>
__device__ __forceinline__ void pmul(const double* a, const double* b, double* out) {
#pragma unroll
    for (int i = 0; i < NA + NB - 1; ++i) out[i] = 0.0;
#pragma unroll
    for (int i = 0; i < NA; ++i)
#pragma unroll
        for (int j = 0; j < NB; ++j) out[i + j] = out[i + j] + (a[i] * b[j]);
}

// det B(z) (oracle/essential.py: det_poly)
__device__ __noinline__ void det_poly(const double (&Bz)[3][3][5], double (&P)[11]) {
    double p[8], q[8], m0[8], m1[8], m2[7], t0[11], t1[11], t2[11];
    pmul<4, 5>(Bz[1][1], Bz[2][2], p); pmul<5, 4>(Bz[1][2], Bz[2][1], q);
    for (int i = 0; i < 8; ++i) m0[i] = p[i] - q[i];
    pmul<4, 5>(Bz[1][0], Bz[2][2], p); pmul<5, 4>(Bz[1][2], Bz[2][0], q);
    for (int i = 0; i < 8; ++i) m1[i] = p[i] - q[i];
    pmul<4, 4>(Bz[1][0], Bz[2][1], p); pmul<4, 4>(Bz[1][1], Bz[2][0], q);
    for (int i = 0; i < 7; ++i) m2[i] = p[i] - q[i];
    pmul<4, 8>(Bz[0][0], m0, t0);
    pmul<4, 8>(Bz[0][1], m1, t1);
    pmul<5, 7>(Bz[0][2], m2, t2);
    for (int i = 0; i < 11; ++i) P[i] = (t0[i] - t1[i]) + t2[i];
}

// ------------------------------------------------------------------------------------------ Sturm roots
struct Sturm {
    double s[kSeq][11];
    int deg[kSeq];
    int n;
};

// max |a[j]|, j <= d, by strict comparisons in index order
__device__ __forceinline__ double max_abs(const double* a, int d) {
    double m = fabs(a[0]);
    for (int j = 1; j <= d; ++j) {
        const double v = fabs(a[j]);
        m = v > m ? v : m;
    }
    return m;
}

// sign changes of the sequence at x (zeros skipped, a NaN counts as positive)
__device__ int sign_changes(const Sturm& S, double x) {
    int cnt = 0;
    bool have = false, prev = false;
    for (int k = 0; k < S.n; ++k) {
        const int d = S.deg[k];
        double v = S.s[k][d];
        for (int i = d - 1; i >= 0; --i) v = (v * x) + S.s[k][i];
        if (v != 0.0) {
            const bool neg = v < 0.0;
            if (have && neg != prev) ++cnt;
            prev = neg;
            have = true;
        }
    }
    return cnt;
}

// Real roots of c0 + c1 z + ... + c10 z^10 in ascending order -> their count (oracle/essential.py: sturm_sequence,
// poly_roots).
__device__ __noinline__ int poly_roots(const double (&c)[11], Sturm& S, double (&root)[kModels]) {
    for (int i = 0; i < 11; ++i)
        if (!(fabs(c[i]) < kInf)) return 0;
    int d = -1;
    double R = 0.0;
    for (int k = 10; k >= 1; --k) {
        double m = fabs(c[0]);
        for (int j = 1; j < k; ++j) { const double v = fabs(c[j]); m = v > m ? v : m; }
        const double Rk = 1.0 + (m / fabs(c[k]));
        if (Rk > 0.0 && Rk < kInf) { d = k; R = Rk; break; }
    }
    if (d < 1) return 0;
    const double m0 = max_abs(c, d);
    for (int j = 0; j <= d; ++j) S.s[0][j] = c[j] / m0;
    S.deg[0] = d;
    double a[11];
    for (int j = 0; j < d; ++j) a[j] = (double)(j + 1) * S.s[0][j + 1];
    const double m1 = max_abs(a, d - 1);
    for (int j = 0; j < d; ++j) S.s[1][j] = a[j] / m1;
    S.deg[1] = d - 1;
    S.n = 2;
    for (int k = 2; k < kSeq; ++k) {
        const int da = S.deg[k - 2], db = S.deg[k - 1];
        if (db < 1) break;
        for (int j = 0; j <= da; ++j) a[j] = S.s[k - 2][j];
        const double lead = S.s[k - 1][db];
        for (int i = da; i >= db; --i) {
            const double q = a[i] / lead;
            for (int j = 0; j < db; ++j) a[i - db + j] = a[i - db + j] - q * S.s[k - 1][j];
        }
        int nd = -1;
        for (int j = 0; j < db; ++j) if (a[j] != 0.0) nd = j;
        if (nd < 0) break;
        const double m = max_abs(a, nd);
        for (int j = 0; j <= nd; ++j) S.s[k][j] = -(a[j] / m);
        S.deg[k] = nd;
        S.n = k + 1;
    }
    const int vA = sign_changes(S, -R);
    int n = vA - sign_changes(S, R);
    n = n < 0 ? 0 : (n > kModels ? kModels : n);
    for (int r = 0; r < n; ++r) {
        double lo = -R, hi = R;
        int vlo = vA, k = r;
        for (int it = 0; it < kMaxBisect; ++it) {
            const double mid = (0.5 * lo) + (0.5 * hi);
            if (!(lo < mid && mid < hi)) break;
            const int vm = sign_changes(S, mid);
            if (vlo - vm > k) {
                hi = mid;
            } else {
                k -= vlo - vm;
                lo = mid;
                vlo = vm;
            }
        }
        root[r] = hi;
    }
    return n;
}

template <int N>
__device__ __forceinline__ double horner(const double* p, double z) {
    double v = p[N - 1];
#pragma unroll
    for (int i = N - 2; i >= 0; --i) v = (v * z) + p[i];
    return v;
}

// ------------------------------------------------------------------------------------------ hypotheses
// hypothesis h of pair b (n valid calibrated matches c1, c2 [n][2]) -> its 10 slots in out (zeros where no model)
__device__ __noinline__ void make_hypothesis(const double* __restrict__ c1, const double* __restrict__ c2, int n, int b,
                                             int h, u64 seed, double* __restrict__ out) {
    for (int i = 0; i < kModels * 9; ++i) out[i] = 0.0;
    int idx[kSample];
#pragma unroll
    for (int j = 0; j < kSample; ++j) idx[j] = 0;
    if (!(n >= kSample && draw_sample<kSample, kMaxDraws>(seed, b, h, n, idx))) return;
    double u1[kSample], v1[kSample], u2[kSample], v2[kSample];
#pragma unroll
    for (int j = 0; j < kSample; ++j) {
        u1[j] = c1[2 * idx[j]]; v1[j] = c1[2 * idx[j] + 1];
        u2[j] = c2[2 * idx[j]]; v2[j] = c2[2 * idx[j] + 1];
    }
    double N[4][9];
    if (!null_basis(u1, v1, u2, v2, N)) return;
    double C[10][20];
    constraint_matrix(N, C);
    if (!gauss_jordan(C)) return;
    double Bz[3][3][5];
    action_rows(C, Bz);
    double P[11];
    det_poly(Bz, P);
    Sturm S;
    double root[kModels];
    const int nr = poly_roots(P, S, root);
    for (int m = 0; m < nr; ++m) {
        const double z = root[m];
        double r[2][3];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            r[k][0] = horner<4>(Bz[k][0], z);
            r[k][1] = horner<4>(Bz[k][1], z);
            r[k][2] = horner<5>(Bz[k][2], z);
        }
        const double xp = (r[0][1] * r[1][2]) - (r[0][2] * r[1][1]);
        const double yp = (r[0][2] * r[1][0]) - (r[0][0] * r[1][2]);
        const double wp = (r[0][0] * r[1][1]) - (r[0][1] * r[1][0]);
        if (wp == 0.0) continue;
        const double x = xp / wp, y = yp / wp;
        double E[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) E[i] = (((x * N[0][i]) + (y * N[1][i])) + (z * N[2][i])) + N[3][i];
        if (!scale_unit(E)) continue;
#pragma unroll
        for (int i = 0; i < 9; ++i) out[9 * m + i] = E[i];
    }
}

// ------------------------------------------------------------------------------------------ kernels
// Workspace views: best [B] u64, n_eff [B] int32 (0 for a pair with an invalid K), thr2 [B], c1, c2 [B][M][2].
struct Views {
    u64* best;
    int32_t* n_eff;
    double* thr2;
    double* c1;
    double* c2;
    double* hyp;
};

__global__ void __launch_bounds__(kRefitThreads) essential_calib_kernel(const double* __restrict__ p1,
                                                                        const double* __restrict__ p2,
                                                                        const int32_t* __restrict__ count,
                                                                        const double* __restrict__ K, int M, double thr,
                                                                        Views w) {
    const int b = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    const double* K1 = K + 18 * (size_t)b;
    const double* K2 = K1 + 9;
    const bool ok = k_valid(K1) && k_valid(K2);
    const int n = clamp_count(count, b, M);
    if (i == 0) {
        const double f = (((K1[0] + K1[4]) + K2[0]) + K2[4]) / 4.0;
        const double t = thr / f;
        w.n_eff[b] = ok ? n : 0;
        w.thr2[b] = t * t;
    }
    if (!ok || i >= n) return;
    const size_t q = ((size_t)b * M + i) * 2;
    calibrate(K1, p1[q], p1[q + 1], w.c1[q], w.c1[q + 1]);
    calibrate(K2, p2[q], p2[q + 1], w.c2[q], w.c2[q + 1]);
}

__global__ void __launch_bounds__(kHypThreads) essential_hyp_kernel(int M, int iters, u64 seed, Views w) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (h >= iters) return;
    make_hypothesis(w.c1 + (size_t)b * M * 2, w.c2 + (size_t)b * M * 2, w.n_eff[b], b, h, seed,
                    w.hyp + ((size_t)b * iters + h) * (kModels * 9));
}

// One CTA per pair: the winner's E, its inliers and their count; zeros for a pair without a model.
__global__ void __launch_bounds__(kRefitThreads) essential_finish_kernel(int M, int iters, Views w, double* __restrict__ E_out,
                                                                         uint8_t* __restrict__ mask_out,
                                                                         int32_t* __restrict__ n_out) {
    __shared__ int cnt_sh;
    const int b = blockIdx.x, t = threadIdx.x;
    const int n = w.n_eff[b];
    const u64 key = w.best[b];
    uint8_t* mask = mask_out + (size_t)b * M;
    if (n < kSample || (key >> 32) == 0) {
        if (t < 9) E_out[9 * b + t] = 0.0;
        if (t == 0) n_out[b] = 0;
        for (int i = t; i < M; i += blockDim.x) mask[i] = 0;
        return;
    }
    const unsigned g = 0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull);
    double E[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) E[i] = w.hyp[((size_t)b * iters * kModels + g) * 9 + i];
    const int cnt = mark_inliers<Essential>(E, w.c1 + (size_t)b * M * 2, w.c2 + (size_t)b * M * 2, n, w.thr2[b], mask,
                                            &cnt_sh);
    for (int i = n + t; i < M; i += blockDim.x) mask[i] = 0;
    if (t < 9) E_out[9 * b + t] = E[t];
    if (t == 0) n_out[b] = cnt;
}

// ------------------------------------------------------------------------------------------ pose
// E -> R1, R2 [9] and t [3] (oracle/essential.py: decompose); false when |E v1| or |E v2| is 0 or not finite.
__device__ __noinline__ bool decompose(const double (&E)[9], double (&R1)[9], double (&R2)[9], double (&t)[3]) {
    double A[3][3], V[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) A[i][j] = ((E[i] * E[j]) + (E[3 + i] * E[3 + j])) + (E[6 + i] * E[6 + j]);
    jacobi_smallest<3>(A, V);
    int o[3] = {0, 1, 2};
    const int pa[3] = {0, 1, 0}, pb[3] = {1, 2, 1};
    for (int s = 0; s < 3; ++s)
        if (A[o[pb[s]]][o[pb[s]]] > A[o[pa[s]]][o[pa[s]]]) { const int x = o[pa[s]]; o[pa[s]] = o[pb[s]]; o[pb[s]] = x; }
    double v[3][3], u[2][3];
    for (int k = 0; k < 3; ++k)
        for (int r = 0; r < 3; ++r) v[k][r] = V[r][o[k]];
    for (int k = 0; k < 2; ++k) {
        double Ev[3];
        for (int r = 0; r < 3; ++r) Ev[r] = ((E[3 * r] * v[k][0]) + (E[3 * r + 1] * v[k][1])) + (E[3 * r + 2] * v[k][2]);
        const double nrm = sqrt(((Ev[0] * Ev[0]) + (Ev[1] * Ev[1])) + (Ev[2] * Ev[2]));
        if (!(nrm > 0.0 && nrm < kInf)) return false;
        for (int r = 0; r < 3; ++r) u[k][r] = Ev[r] / nrm;
    }
    const double u3[3] = {(u[0][1] * u[1][2]) - (u[0][2] * u[1][1]), (u[0][2] * u[1][0]) - (u[0][0] * u[1][2]),
                          (u[0][0] * u[1][1]) - (u[0][1] * u[1][0])};
    double Vm[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) Vm[3 * r + c] = v[c][r];
    if (det3(Vm) < 0.0)
        for (int r = 0; r < 3; ++r) v[2][r] = -v[2][r];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            R1[3 * r + c] = ((u[1][r] * v[0][c]) - (u[0][r] * v[1][c])) + (u3[r] * v[2][c]);
            R2[3 * r + c] = ((u[0][r] * v[1][c]) - (u[1][r] * v[0][c])) + (u3[r] * v[2][c]);
        }
    for (int r = 0; r < 3; ++r) t[r] = u3[r];
    return true;
}

// the least-squares depths of z2 x2 = z1 R x1 + t: 0 < z1 < dist and 0 < (R z1 x1 + t)_z < dist
__device__ __forceinline__ bool cheirality(const double* R, const double* t, double u1, double v1, double u2, double v2,
                                           double dist) {
    const double a0 = ((R[0] * u1) + (R[1] * v1)) + R[2];
    const double a1 = ((R[3] * u1) + (R[4] * v1)) + R[5];
    const double a2 = ((R[6] * u1) + (R[7] * v1)) + R[8];
    const double aa = ((a0 * a0) + (a1 * a1)) + (a2 * a2);
    const double bb = ((u2 * u2) + (v2 * v2)) + 1.0;
    const double ab = ((a0 * u2) + (a1 * v2)) + a2;
    const double at = ((a0 * t[0]) + (a1 * t[1])) + (a2 * t[2]);
    const double bt = ((u2 * t[0]) + (v2 * t[1])) + t[2];
    const double det = (aa * bb) - (ab * ab);
    const double z1 = ((ab * bt) - (at * bb)) / det;
    const double z = (((R[6] * (z1 * u1)) + (R[7] * (z1 * v1))) + (R[8] * z1)) + t[2];
    return z1 > 0.0 && z1 < dist && z > 0.0 && z < dist;
}

__global__ void __launch_bounds__(kPoseThreads) recover_pose_kernel(
    const double* __restrict__ E_in, const double* __restrict__ p1, const double* __restrict__ p2,
    const int32_t* __restrict__ count, const double* __restrict__ K, const uint8_t* __restrict__ mask_in, int M,
    double dist, double* __restrict__ R_out, double* __restrict__ t_out, uint8_t* __restrict__ mask_out,
    int32_t* __restrict__ n_out) {
    __shared__ double Rs[2][9], ts[3];
    __shared__ int ok_sh, cnt_sh[4];
    __shared__ uint8_t flags[kMaxMatches];
    const int b = blockIdx.x, t = threadIdx.x;
    const int n = clamp_count(count, b, M);
    const double* K1 = K + 18 * (size_t)b;
    const double* K2 = K1 + 9;
    uint8_t* mask = mask_out + (size_t)b * M;
    if (t == 0) {
        double E[9];
        bool nz = false;
        for (int i = 0; i < 9; ++i) { E[i] = E_in[9 * (size_t)b + i]; nz |= E[i] != 0.0; }
        ok_sh = nz && k_valid(K1) && k_valid(K2) && decompose(E, Rs[0], Rs[1], ts);
        for (int q = 0; q < 4; ++q) cnt_sh[q] = 0;
    }
    __syncthreads();
    if (!ok_sh) {
        if (t < 9) R_out[9 * b + t] = 0.0;
        if (t < 3) t_out[3 * b + t] = 0.0;
        if (t == 0) n_out[b] = 0;
        for (int i = t; i < M; i += blockDim.x) mask[i] = 0;
        return;
    }
    double R[2][9], tv[2][3];
#pragma unroll
    for (int i = 0; i < 9; ++i) { R[0][i] = Rs[0][i]; R[1][i] = Rs[1][i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { tv[0][i] = ts[i]; tv[1][i] = -ts[i]; }
    int c[4] = {0, 0, 0, 0};
    for (int i = t; i < n; i += blockDim.x) {
        uint8_t f = 0;
        if (!mask_in || mask_in[(size_t)b * M + i]) {
            const size_t q = ((size_t)b * M + i) * 2;
            double u1, v1, u2, v2;
            calibrate(K1, p1[q], p1[q + 1], u1, v1);
            calibrate(K2, p2[q], p2[q + 1], u2, v2);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (cheirality(R[k & 1], tv[k >> 1], u1, v1, u2, v2, dist)) { f |= (uint8_t)(1 << k); ++c[k]; }
        }
        flags[i] = f;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int s = c[k];
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((t & 31) == 0) atomicAdd(&cnt_sh[k], s);
    }
    __syncthreads();
    int best = 0;
    for (int k = 1; k < 4; ++k) best = cnt_sh[k] > cnt_sh[best] ? k : best;
    for (int i = t; i < M; i += blockDim.x) mask[i] = i < n ? (uint8_t)((flags[i] >> best) & 1) : (uint8_t)0;
    if (t < 9) R_out[9 * b + t] = Rs[best & 1][t];
    if (t < 3) t_out[3 * b + t] = tv[best >> 1][t];
    if (t == 0) n_out[b] = cnt_sh[best];
}

// workspace layout (offsets from the 256-aligned base)
struct Layout {
    size_t n_eff, thr2, c1, c2, hyp, total;
};

inline Layout layout(int B, int M, int iters) {
    Layout l;
    l.n_eff = best_bytes(B);
    l.thr2 = l.n_eff + align_up((size_t)B * sizeof(int32_t), 256);
    l.c1 = l.thr2 + align_up((size_t)B * sizeof(double), 256);
    const size_t pts = align_up((size_t)B * M * 2 * sizeof(double), 256);
    l.c2 = l.c1 + pts;
    l.hyp = l.c2 + pts;
    l.total = l.hyp + (size_t)B * iters * kModels * 9 * sizeof(double);
    return l;
}

}  // namespace
}  // namespace balf

using namespace balf;

extern "C" size_t balf_essential_workspace_bytes(int B, int M, int iters) {
    if (B < 0 || M < 0 || iters < 1 || iters > kMaxIters) return 0;
    return layout(B, M, iters).total + 256;
}

extern "C" int balf_find_essential_ransac(const double* p1, const double* p2, const int32_t* count, const double* K, int B,
                                          int M, double thr, int iters, uint64_t seed, double* E, uint8_t* inlier_mask,
                                          int32_t* n_inliers, void* workspace, size_t workspace_bytes, void* stream) {
    BALF_REQUIRE(B >= 0 && B <= 65535, "find_essential_ransac: B = %d outside [0, 65535]", B);
    BALF_REQUIRE(M >= 0 && M <= kMaxMatches, "find_essential_ransac: M = %d outside [0, %d]", M, kMaxMatches);
    BALF_REQUIRE(thr > 0.0, "find_essential_ransac: thr must be > 0");
    BALF_REQUIRE(iters >= 1 && iters <= kMaxIters, "find_essential_ransac: iters = %d outside [1, %d]", iters, kMaxIters);
    if (B == 0) return 0;
    BALF_REQUIRE(count && K && E && n_inliers && workspace && (M == 0 || (p1 && p2 && inlier_mask)),
                 "find_essential_ransac: null pointer argument");
    BALF_REQUIRE(workspace_bytes >= balf_essential_workspace_bytes(B, M, iters),
                 "find_essential_ransac: workspace of %zu bytes is too small (%zu needed)", workspace_bytes,
                 balf_essential_workspace_bytes(B, M, iters));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* base = reinterpret_cast<unsigned char*>(align_up((size_t)workspace, 256));
    const Layout l = layout(B, M, iters);
    Views w;
    w.best = reinterpret_cast<u64*>(base);
    w.n_eff = reinterpret_cast<int32_t*>(base + l.n_eff);
    w.thr2 = reinterpret_cast<double*>(base + l.thr2);
    w.c1 = reinterpret_cast<double*>(base + l.c1);
    w.c2 = reinterpret_cast<double*>(base + l.c2);
    w.hyp = reinterpret_cast<double*>(base + l.hyp);
    const int slots = iters * kModels;
    BALF_CUDA_OK(cudaMemsetAsync(w.best, 0, (size_t)B * sizeof(u64), st));
    {
        ProfScope p("essential_calib", st);
        essential_calib_kernel<<<dim3(cdiv(M > 0 ? M : 1, kRefitThreads), B), kRefitThreads, 0, st>>>(p1, p2, count, K, M,
                                                                                                      thr, w);
    }
    {
        ProfScope p("essential_hyp", st);
        essential_hyp_kernel<<<dim3(cdiv(iters, kHypThreads), B), kHypThreads, 0, st>>>(M, iters, seed, w);
    }
    {
        ProfScope p("essential_score", st);
        ransac_score_kernel<Essential><<<dim3(cdiv(slots, kScoreThreads), B), kScoreThreads, 0, st>>>(
            w.c1, w.c2, w.n_eff, M, slots, 0.0, w.hyp, w.best, w.thr2);
    }
    {
        ProfScope p("essential_finish", st);
        essential_finish_kernel<<<B, kRefitThreads, 0, st>>>(M, iters, w, E, inlier_mask, n_inliers);
    }
    BALF_COUNT_LAUNCH(4);
    BALF_LAUNCH_OK();
    return 0;
}

extern "C" int balf_recover_pose(const double* E, const double* p1, const double* p2, const int32_t* count, const double* K,
                                 const uint8_t* mask_in, int B, int M, double dist_thresh, double* R, double* t,
                                 uint8_t* pose_mask, int32_t* n_good, void* stream) {
    BALF_REQUIRE(B >= 0 && B <= 65535, "recover_pose: B = %d outside [0, 65535]", B);
    BALF_REQUIRE(M >= 0 && M <= kMaxMatches, "recover_pose: M = %d outside [0, %d]", M, kMaxMatches);
    BALF_REQUIRE(dist_thresh > 0.0, "recover_pose: dist_thresh must be > 0");
    if (B == 0) return 0;
    BALF_REQUIRE(E && count && K && R && t && n_good && (M == 0 || (p1 && p2 && pose_mask)),
                 "recover_pose: null pointer argument");
    cudaStream_t st = (cudaStream_t)stream;
    {
        ProfScope p("recover_pose", st);
        recover_pose_kernel<<<B, kPoseThreads, 0, st>>>(E, p1, p2, count, K, mask_in, M, dist_thresh, R, t, pose_mask,
                                                        n_good);
    }
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}
