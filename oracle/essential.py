"""RANSAC essential matrix and relative pose of ``balf_find_essential_ransac`` / ``balf_recover_pose``
(balf_b200/csrc/essential.cu), restated in NumPy.

No reference counterpart: the semantics are defined in include/balf_b200.h and restated here operation for operation.
PARITY UNPINNABLE against the reference; anchored instead on OpenCV (tests/test_oracle_essential.py: the 5-point solver
against ``cv2.findEssentialMat`` on 5 points, the decomposition against ``cv2.decomposeEssentialMat``, the pose against
``cv2.recoverPose``, the inlier rule against a transcription of cv2's error, recovery of seeded two-view geometry).

The hash, the block structure of the workspace and the scaling are those of oracle/fundamental.py and
oracle/homography.py; the Jacobi is ``oracle.fundamental.jacobi_eigh``.  Every float64 operation is elementwise IEEE
arithmetic (+ - * / sqrt and comparisons only) in the order the kernels perform it, so the results are bit-identical:
vectorising over hypotheses changes no rounding.
"""
import numpy as np

from oracle import fundamental as of

SAMPLE = 5
MAX_DRAWS = 64
MAX_MODELS = 10
MAX_BISECT = 200
NSEQ = 11                            # Sturm sequence of a degree-10 polynomial: p0 .. p10

# The 20 monomials of the cubic constraints, in the column order of the 10x20 matrix: the first 10 are eliminated,
# the last 10 stay (Nister's order).  Exponents (of x, y, z).
MONOS = [(3, 0, 0), (0, 3, 0), (2, 1, 0), (1, 2, 0), (2, 0, 1), (2, 0, 0), (0, 2, 1), (0, 2, 0), (1, 1, 1), (1, 1, 0),
         (1, 0, 2), (1, 0, 1), (1, 0, 0), (0, 1, 2), (0, 1, 1), (0, 1, 0), (0, 0, 3), (0, 0, 2), (0, 0, 1), (0, 0, 0)]
# A linear form is [x, y, z, 1]; a quadratic form has these 10 monomials.
LIN = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, 0)]
QUAD = [(2, 0, 0), (1, 1, 0), (1, 0, 1), (1, 0, 0), (0, 2, 0), (0, 1, 1), (0, 1, 0), (0, 0, 2), (0, 0, 1), (0, 0, 0)]


def _add(a, b):
    return tuple(i + j for i, j in zip(a, b))


# product tables: term (i, j) of lin x lin goes to QUAD index LL[i][j]; term (m, k) of quad x lin to MONOS index QL[m][k]
LL = [[QUAD.index(_add(LIN[i], LIN[j])) for j in range(4)] for i in range(4)]
QL = [[MONOS.index(_add(QUAD[m], LIN[k])) for k in range(4)] for m in range(10)]


# ------------------------------------------------------------------------------------------ calibration
def k_valid(K):
    """K [...,9] row-major -> bool: fx, fy finite and > 0, last row (0, 0, 1)."""
    K = np.asarray(K, np.float64)
    fin = lambda v: (v > 0) & (v < np.inf)
    return fin(K[..., 0]) & fin(K[..., 4]) & (K[..., 6] == 0) & (K[..., 7] == 0) & (K[..., 8] == 1)


def calibrate(p, K):
    """p [...,2] pixels, K [9] -> calibrated [...,2]: y' = (y - cy) / fy, x' = ((x - cx) - s y') / fx."""
    with np.errstate(all="ignore"):
        yc = (p[..., 1] - K[5]) / K[4]
        xc = ((p[..., 0] - K[2]) - (K[1] * yc)) / K[0]
    return np.stack([xc, yc], -1)


def pair_thr2(thr, K1, K2):
    """thr_b^2, thr_b = thr / (((fx1 + fy1) + fx2) + fy2) / 4."""
    f = (((K1[0] + K1[4]) + K2[0]) + K2[4]) / 4.0
    t = thr / f
    return t * t


# ------------------------------------------------------------------------------------------ null space
def null_basis(a):
    """a [N,5,9] epipolar rows -> (X, Y, Z, W [N,9], ok): the 5x5 system in e0..e4 with right-hand sides -a[:,5+j], j = 0..3
    (e5 .. e8 free), one partial-pivot elimination (the pivot is the first largest |a[r][k]|, NaN counting as the
    largest; ok = False when a pivot is 0 or not finite) and four back substitutions.  Basis j has e_{5+j} = 1 and the
    other free entries 0."""
    N = a.shape[0]
    r = np.arange(N)
    A = np.concatenate([a[:, :, :5], -a[:, :, 5:]], 2).copy()
    ok = np.ones(N, bool)
    with np.errstate(all="ignore"):
        for k in range(5):
            col = np.abs(A[:, k:, k])
            p = k + np.argmax(col, axis=1)
            best = col[r, p - k]
            ok &= (best > 0) & (best < np.inf)
            rk, rp = A[r, k].copy(), A[r, p].copy()
            A[r, k], A[r, p] = rp, rk
            d = A[:, k, k]
            f = A[:, k + 1:, k] / d[:, None]
            A[:, k + 1:, k + 1:] = A[:, k + 1:, k + 1:] - f[:, :, None] * A[:, k, None, k + 1:]
        out = []
        for j in range(4):
            h = np.zeros((N, 9))
            h[:, 5 + j] = 1.0
            for k in range(4, -1, -1):
                s = A[:, k, 5 + j].copy()
                for c in range(k + 1, 5):
                    s = s - A[:, k, c] * h[:, c]
                h[:, k] = s / A[:, k, k]
            out.append(h)
    return out[0], out[1], out[2], out[3], ok


def _dot9(a, b):
    s = a[:, 0] * b[:, 0]
    for i in range(1, 9):
        s = s + (a[:, i] * b[:, i])
    return s


def orthonormalise(X, Y, Z, W):
    """Modified Gram-Schmidt in the order W, Z, Y, X -> (X', Y', Z', W', ok): each vector in turn loses its projections
    on the ones already done, v = v - (v . u) u (dot products summed in index order), and is divided by its norm
    (ok = False when a norm is 0 or not finite).  The elimination's basis is far from orthogonal; in this basis the
    degree-10 polynomial below is much better conditioned (on noise-free samples, the median error of E drops from about
    1e-10 to about 1e-14)."""
    done = []
    ok = np.ones(len(X), bool)
    with np.errstate(all="ignore"):
        for v in (W, Z, Y, X):
            v = v.copy()
            for u in done:
                v = v - _dot9(v, u)[:, None] * u
            nrm = np.sqrt(_dot9(v, v))
            ok &= (nrm > 0) & (nrm < np.inf)
            done.append(v / nrm[:, None])
    return done[3], done[2], done[1], done[0], ok


# ------------------------------------------------------------------------------------------ constraint matrix
def _mul_ll(a, b):
    """linear x linear [N,4] -> quadratic [N,10]; terms added in (i, j) row-major order onto 0.0."""
    q = np.zeros((a.shape[0], 10))
    for i in range(4):
        for j in range(4):
            q[:, LL[i][j]] = q[:, LL[i][j]] + (a[:, i] * b[:, j])
    return q


def _mul_ql(q, b):
    """quadratic [N,10] x linear [N,4] -> cubic [N,20] (MONOS order); terms added in (m, k) row-major order onto 0.0."""
    c = np.zeros((q.shape[0], 20))
    for m in range(10):
        for k in range(4):
            c[:, QL[m][k]] = c[:, QL[m][k]] + (q[:, m] * b[:, k])
    return c


def constraint_matrix(X, Y, Z, W):
    """The 10x20 coefficient matrix [N,10,20] of E = x X + y Y + z Z + W: row 0 is det E by the first row's cofactors,
    E00 (E11 E22 - E12 E21) - E01 (E10 E22 - E12 E20) + E02 (E10 E21 - E11 E20); rows 1 + 3 i + j are (L E)_ij with
    L = E E^T - (tr(E E^T) / 2) I, i.e. half of 2 E E^T E - tr(E E^T) E, where (E E^T)_ij = (E_i0 E_j0 + E_i1 E_j1) + E_i2 E_j2,
    tr = ((E E^T)_00 + (E E^T)_11) + (E E^T)_22 and (L E)_ij = (L_i0 E_0j + L_i1 E_1j) + L_i2 E_2j."""
    E = np.stack([X, Y, Z, W], -1)                               # [N,9,4]: entry e of E as a linear form
    N = E.shape[0]
    with np.errstate(all="ignore"):
        e = lambda i, j: E[:, 3 * i + j]
        m1 = _mul_ll(e(1, 1), e(2, 2)) - _mul_ll(e(1, 2), e(2, 1))
        m2 = _mul_ll(e(1, 0), e(2, 2)) - _mul_ll(e(1, 2), e(2, 0))
        m3 = _mul_ll(e(1, 0), e(2, 1)) - _mul_ll(e(1, 1), e(2, 0))
        det = (_mul_ql(m1, e(0, 0)) - _mul_ql(m2, e(0, 1))) + _mul_ql(m3, e(0, 2))
        EE = [[(_mul_ll(e(i, 0), e(j, 0)) + _mul_ll(e(i, 1), e(j, 1))) + _mul_ll(e(i, 2), e(j, 2)) for j in range(3)]
              for i in range(3)]
        half = ((EE[0][0] + EE[1][1]) + EE[2][2]) * 0.5
        L = [[EE[i][j] - half if i == j else EE[i][j] for j in range(3)] for i in range(3)]
        C = np.zeros((N, 10, 20))
        C[:, 0] = det
        for i in range(3):
            for j in range(3):
                C[:, 1 + 3 * i + j] = (_mul_ql(L[i][0], e(0, j)) + _mul_ql(L[i][1], e(1, j))) + _mul_ql(L[i][2], e(2, j))
    return C


def gauss_jordan(C):
    """Gauss-Jordan elimination of the first 10 columns of C [N,10,20] (modified) with partial pivoting (first largest
    |C[r][k]|, r >= k, NaN counting as the largest) -> ok [N] (False when a pivot is 0 or not finite).  Step k swaps the
    pivot row into row k, divides C[k][c] by the pivot for c > k, then for every other row r subtracts
    C[r][k] * C[k][c] from C[r][c], c > k.  Afterwards row i reads MONOS[i] + sum_c C[i][c] MONOS[c] = 0, c >= 10."""
    N = C.shape[0]
    r = np.arange(N)
    ok = np.ones(N, bool)
    with np.errstate(all="ignore"):
        for k in range(10):
            col = np.abs(C[:, k:, k])
            p = k + np.argmax(col, axis=1)
            best = col[r, p - k]
            ok &= (best > 0) & (best < np.inf)
            rk, rp = C[r, k].copy(), C[r, p].copy()
            C[r, k], C[r, p] = rp, rk
            d = C[:, k, k].copy()
            C[:, k, k + 1:] = C[:, k, k + 1:] / d[:, None]
            others = [i for i in range(10) if i != k]
            f = C[:, others, k].copy()
            C[:, others, k + 1:] = C[:, others, k + 1:] - f[:, :, None] * C[:, k, None, k + 1:]
    return ok


def action_rows(C):
    """The reduced rows of x^2 z, x^2, y^2 z, y^2, x y z, x y (rows 4 .. 9) -> B(z) [N,3,3,5]: row k of B is
    row(2 k + 4) - z row(2 k + 5) as the coefficients (ascending powers of z) of x, y and 1 in B(z) (x, y, 1)^T = 0:
      x: [a12, a11 - b12, a10 - b11, -b10, 0], y: [a15, a14 - b15, a13 - b14, -b13, 0],
      1: [a19, a18 - b19, a17 - b18, a16 - b17, -b16]   (a = row 2 k + 4, b = row 2 k + 5, indices = MONOS columns)."""
    N = C.shape[0]
    Bz = np.zeros((N, 3, 3, 5))
    for k in range(3):
        a, b = C[:, 2 * k + 4], C[:, 2 * k + 5]
        for v, (c2, c1, c0) in enumerate(((10, 11, 12), (13, 14, 15))):
            Bz[:, k, v, 0] = a[:, c0]
            Bz[:, k, v, 1] = a[:, c1] - b[:, c0]
            Bz[:, k, v, 2] = a[:, c2] - b[:, c1]
            Bz[:, k, v, 3] = -b[:, c2]
        Bz[:, k, 2, 0] = a[:, 19]
        Bz[:, k, 2, 1] = a[:, 18] - b[:, 19]
        Bz[:, k, 2, 2] = a[:, 17] - b[:, 18]
        Bz[:, k, 2, 3] = a[:, 16] - b[:, 17]
        Bz[:, k, 2, 4] = -b[:, 16]
    return Bz


def _pmul(a, b):
    """polynomial product [N,na] x [N,nb] -> [N,na+nb-1] (ascending); terms added in (i, j) row-major order onto 0.0."""
    out = np.zeros((a.shape[0], a.shape[1] + b.shape[1] - 1))
    for i in range(a.shape[1]):
        for j in range(b.shape[1]):
            out[:, i + j] = out[:, i + j] + (a[:, i] * b[:, j])
    return out


def det_poly(Bz):
    """det B(z) [N,11] (ascending) by the first row's cofactors, each minor a difference of products of 4 x 5 or 4 x 4
    coefficients: B00 (B11 B22 - B12 B21) - B01 (B10 B22 - B12 B20) + B02 (B10 B21 - B11 B20)."""
    b = lambda i, j, n: Bz[:, i, j, :n]                       # x, y entries are cubics (4), the 1 entries quartics (5)
    with np.errstate(all="ignore"):
        m0 = _pmul(b(1, 1, 4), b(2, 2, 5)) - _pmul(b(1, 2, 5), b(2, 1, 4))      # degree 7
        m1 = _pmul(b(1, 0, 4), b(2, 2, 5)) - _pmul(b(1, 2, 5), b(2, 0, 4))      # degree 7
        m2 = _pmul(b(1, 0, 4), b(2, 1, 4)) - _pmul(b(1, 1, 4), b(2, 0, 4))      # degree 6
        t0, t1, t2 = _pmul(b(0, 0, 4), m0), _pmul(b(0, 1, 4), m1), _pmul(b(0, 2, 5), m2)
        return (t0 - t1) + t2


# ------------------------------------------------------------------------------------------ real roots (Sturm)
def _maxabs(c, upto):
    """max |c[:, i]|, i < upto, by strict comparisons in index order (c finite)."""
    m = np.abs(c[:, 0])
    for i in range(1, upto):
        a = np.abs(c[:, i])
        m = np.where(a > m, a, m)
    return m


def sturm_sequence(c):
    """c [N,11] (ascending; finite) -> (seq [N,11,11], deg [N,11] (-1: no polynomial), R [N], ok [N]).

    The degree d is the highest i with a finite Cauchy bound R = 1 + max_{j<i} |c_j| / |c_i| (ok = False below degree 1
    or when a coefficient is not finite).  p0 = c[0..d] / max|c|, p1 = p0' / max|p0'|, and p_{k+1} = -(p_{k-1} mod p_k)
    divided by its largest magnitude, until the remainder is 0.  The remainder: for i = deg a .. deg b,
    q = a_i / b_db, a_{i-db+j} = a_{i-db+j} - q b_j (j < db); its degree is the highest index with a nonzero entry."""
    N = c.shape[0]
    rows = np.arange(N)
    with np.errstate(all="ignore"):
        fin = np.isfinite(c).all(1)
        c = np.where(fin[:, None], c, 0.0)
        deg = np.full(N, -1)
        R = np.zeros(N)
        for d in range(1, 11):
            Rd = 1.0 + (_maxabs(c, d) / np.abs(c[:, d]))
            good = (Rd > 0) & (Rd < np.inf)
            deg = np.where(good, d, deg)
            R = np.where(good, Rd, R)
        ok = fin & (deg >= 1)
        deg = np.where(ok, deg, -1)
        seq = np.zeros((N, NSEQ, 11))
        sdeg = np.full((N, NSEQ), -1)
        keep = np.arange(11)[None, :] <= deg[:, None]
        p0 = np.where(keep, c, 0.0)
        p0 = p0 / _maxabs(p0, 11)[:, None]
        p0 = np.where(keep, p0, 0.0)
        seq[:, 0], sdeg[:, 0] = p0, deg
        d1 = np.zeros((N, 11))
        for j in range(10):
            d1[:, j] = float(j + 1) * p0[:, j + 1]
        d1 = d1 / _maxabs(d1, 11)[:, None]
        seq[:, 1], sdeg[:, 1] = np.where(ok[:, None], d1, 0.0), np.where(ok, deg - 1, -1)
        for k in range(2, NSEQ):
            a, b = seq[:, k - 2].copy(), seq[:, k - 1]
            da, db = sdeg[:, k - 2], sdeg[:, k - 1]
            act = (db >= 1) & (da >= db)                     # p_{k-1} of degree 0 (or none) ends the chain
            lead = b[rows, np.maximum(db, 0)]
            for i in range(10, -1, -1):
                on = act & (i <= da) & (i >= db)
                q = a[:, i] / lead
                for j in range(10):
                    on_j = on & (j < db)
                    t = i - db + j
                    sel = rows[on_j]
                    a[sel, t[on_j]] = a[sel, t[on_j]] - q[on_j] * b[sel, j]
            a = np.where(np.arange(11)[None, :] < db[:, None], a, 0.0)
            nd = np.full(N, -1)
            for j in range(11):
                nd = np.where((a[:, j] != 0) & (j < db), j, nd)
            act = act & (nd >= 0)
            a = -(a / _maxabs(a, 11)[:, None])
            seq[:, k] = np.where(act[:, None], a, 0.0)
            sdeg[:, k] = np.where(act, nd, -1)
    return seq, sdeg, R, ok


def sign_changes(seq, sdeg, x):
    """Sign changes of the Sturm sequence at x [N] (zeros skipped; a NaN value counts as positive).  Each p_k is evaluated
    by Horner from its leading coefficient: v = p_d; v = v x + p_i, i = d - 1 .. 0."""
    N = seq.shape[0]
    cnt = np.zeros(N, np.int64)
    have = np.zeros(N, bool)
    prev = np.zeros(N, bool)
    with np.errstate(all="ignore"):
        for k in range(NSEQ):
            d = sdeg[:, k]
            v = np.zeros(N)
            for i in range(10, -1, -1):
                v = np.where(d == i, seq[:, k, i], np.where(d > i, (v * x) + seq[:, k, i], v))
            live = d >= 0
            nz = live & (v != 0)
            neg = v < 0
            cnt += nz & have & (neg != prev)
            prev = np.where(nz, neg, prev)
            have |= nz
    return cnt


def poly_roots(c):
    """Real roots of c0 + c1 z + ... + c10 z^10, c [N,11] -> (roots [N,10] ascending, NaN-padded; count [N]).

    With the Sturm sequence and the Cauchy bound R of ``sturm_sequence``, the count is V(-R) - V(R) clamped to [0, 10]
    (V: sign changes).  Root i is found by bisection of (lo, hi] = (-R, R] at mid = lo / 2 + hi / 2: when the interval
    (lo, mid] holds more than k roots (k = roots of rank < i above lo), hi = mid, else lo = mid and k drops by the roots
    passed.  It stops when mid is no longer strictly inside or after 200 steps; the root is hi."""
    N = c.shape[0]
    seq, sdeg, R, ok = sturm_sequence(c)
    vlo0 = sign_changes(seq, sdeg, -R)
    n = np.where(ok, np.clip(vlo0 - sign_changes(seq, sdeg, R), 0, MAX_MODELS), 0)
    roots = np.full((N, MAX_MODELS), np.nan)
    hs, ranks = np.nonzero(np.arange(MAX_MODELS)[None, :] < n[:, None])
    if len(hs) == 0:
        return roots, n
    S, D = seq[hs], sdeg[hs]
    lo, hi = -R[hs], R[hs].copy()
    vlo = vlo0[hs].copy()
    k = ranks.copy()
    act = np.ones(len(hs), bool)
    with np.errstate(all="ignore"):
        for _ in range(MAX_BISECT):
            mid = (0.5 * lo) + (0.5 * hi)
            act &= (lo < mid) & (mid < hi)
            if not act.any():
                break
            idx = np.nonzero(act)[0]
            vm = sign_changes(S[idx], D[idx], mid[idx])
            left = (vlo[idx] - vm) > k[idx]
            hi[idx] = np.where(left, mid[idx], hi[idx])
            k[idx] = np.where(left, k[idx], k[idx] - (vlo[idx] - vm))
            lo[idx] = np.where(left, lo[idx], mid[idx])
            vlo[idx] = np.where(left, vlo[idx], vm)
    roots[hs, ranks] = hi
    return roots, n


# ------------------------------------------------------------------------------------------ minimal solver
def _horner(p, z):
    v = p[..., -1]
    for i in range(p.shape[-1] - 2, -1, -1):
        v = (v * z) + p[..., i]
    return v


def minimal_solve(c1, c2):
    """5-point solver on calibrated points c1, c2 [N,5,2] -> (E [N,10,9] in root order, ok [N,10]); a slot without a
    model is zeros.  For root z: rows 0 and 1 of B(z) (Horner, the x and y entries as cubics, the 1 entry as a quartic),
    (x', y', w') = row0 x row1 = (b01 b12 - b02 b11, b02 b10 - b00 b12, b00 b11 - b01 b10), no model when w' = 0, x = x' / w',
    y = y' / w', E = ((x X + y Y) + z Z) + W scaled by ``oracle.fundamental.scale_unit``."""
    N = c1.shape[0]
    with np.errstate(all="ignore"):
        X, Y, Z, W, ok = null_basis(of.epipolar_rows(c1[..., 0], c1[..., 1], c2[..., 0], c2[..., 1]))
        X, Y, Z, W, ok_o = orthonormalise(X, Y, Z, W)
        ok &= ok_o
        C = constraint_matrix(X, Y, Z, W)
        ok &= gauss_jordan(C)
        Bz = action_rows(C)
        roots, cnt = poly_roots(det_poly(Bz))
    cnt = np.where(ok, cnt, 0)
    out, oks = np.zeros((N, MAX_MODELS, 9)), np.zeros((N, MAX_MODELS), bool)
    for m in range(MAX_MODELS):
        z = roots[:, m]
        with np.errstate(all="ignore"):
            b = [[_horner(Bz[:, r, v, :4 if v < 2 else 5], z) for v in range(3)] for r in range(2)]
            xp = (b[0][1] * b[1][2]) - (b[0][2] * b[1][1])
            yp = (b[0][2] * b[1][0]) - (b[0][0] * b[1][2])
            wp = (b[0][0] * b[1][1]) - (b[0][1] * b[1][0])
            x, y = xp / wp, yp / wp
            E = (((x[:, None] * X) + (y[:, None] * Y)) + (z[:, None] * Z)) + W
        G, okd = of.scale_unit(E)
        oks[:, m] = ok & (cnt > m) & (wp != 0) & okd
        out[:, m] = np.where(oks[:, m, None], G, 0.0)
    return out, oks


# ------------------------------------------------------------------------------------------ inliers
def inliers(E, c1, c2, thr2):
    """E [N,9], calibrated c1, c2 [n,2] -> bool [N,n]: with (a, b, c) = E x1, s = x2^T E x1, (a', b', .) = E^T x2 and
    d = ((a^2 + b^2) + a'^2) + b'^2, an inlier has d finite and > 0 and s^2 <= thr2 d (cv2's EMEstimatorCallback error,
    s^2 / d <= thr^2, without its rounding to float32)."""
    x1, y1, x2, y2 = c1[:, 0], c1[:, 1], c2[:, 0], c2[:, 1]
    f = [E[:, i, None] for i in range(9)]
    with np.errstate(all="ignore"):
        a = ((f[0] * x1) + (f[1] * y1)) + f[2]
        b = ((f[3] * x1) + (f[4] * y1)) + f[5]
        c = ((f[6] * x1) + (f[7] * y1)) + f[8]
        s = ((x2 * a) + (y2 * b)) + c
        ap = ((f[0] * x2) + (f[3] * y2)) + f[6]
        bp = ((f[1] * x2) + (f[4] * y2)) + f[7]
        d = (((a * a) + (b * b)) + (ap * ap)) + (bp * bp)
        return (d > 0) & (d < np.inf) & ((s * s) <= thr2 * d)


# ------------------------------------------------------------------------------------------ RANSAC
def hypotheses(c1, c2, n, b, iters, seed):
    """All hypotheses of pair b -> (E [iters*10,9], ok [iters*10]), slot 10 h + m = model m of hypothesis h."""
    idx, ok = of.sample_indices(seed, b, np.arange(iters), max(n, 1), k=SAMPLE, draws=MAX_DRAWS)
    idx = np.where(ok[:, None], idx, 0)
    E, ok_m = minimal_solve(c1[idx], c2[idx])
    ok_m &= ok[:, None]
    return np.where(ok_m[..., None], E, 0.0).reshape(-1, 9), ok_m.reshape(-1)


def find_essential_ransac_pair(p1, p2, n, K1, K2, b, thr, iters, seed, chunk=256):
    """One pair (index b of its batch, n valid rows) -> (E [9], mask uint8 [n], n_inliers)."""
    p1, p2 = np.asarray(p1, np.float64)[:n], np.asarray(p2, np.float64)[:n]
    K1, K2 = np.asarray(K1, np.float64).reshape(9), np.asarray(K2, np.float64).reshape(9)
    if n < SAMPLE or not (k_valid(K1) and k_valid(K2)):
        return np.zeros(9), np.zeros(n, np.uint8), 0
    c1, c2, t2 = calibrate(p1, K1), calibrate(p2, K2), pair_thr2(thr, K1, K2)
    E, ok = hypotheses(c1, c2, n, b, iters, seed)
    S = len(E)
    score = np.full(S, -1, np.int64)
    for s in range(0, S, chunk):
        e = min(S, s + chunk)
        score[s:e] = np.where(ok[s:e], inliers(E[s:e], c1, c2, t2).sum(1), -1)
    win = int(np.argmax(score))                                 # first maximum = lowest 10 h + m
    if score[win] < 0:
        return np.zeros(9), np.zeros(n, np.uint8), 0
    mask = inliers(E[win][None], c1, c2, t2)[0]
    return E[win], mask.astype(np.uint8), int(mask.sum())


def find_essential_ransac(p1, p2, count, K, thr, iters, seed):
    """Batched form of ``balf_find_essential_ransac``: p1, p2 [B,M,2], count [B], K [B,2,3,3] -> (E [B,3,3],
    mask uint8 [B,M], n_inliers int32 [B])."""
    p1, p2 = np.asarray(p1, np.float64), np.asarray(p2, np.float64)
    K = np.asarray(K, np.float64).reshape(-1, 2, 9)
    B, M = p1.shape[:2]
    Es, masks, ns = np.zeros((B, 9)), np.zeros((B, M), np.uint8), np.zeros(B, np.int32)
    for b in range(B):
        n = int(min(max(int(count[b]), 0), M))
        Es[b], masks[b, :n], ns[b] = find_essential_ransac_pair(p1[b], p2[b], n, K[b, 0], K[b, 1], b, thr, iters, seed)
    return Es.reshape(B, 3, 3), masks, ns


# ------------------------------------------------------------------------------------------ pose
def _dot3(a, b):
    return ((a[0] * b[0]) + (a[1] * b[1])) + (a[2] * b[2])


def decompose(E):
    """E [9] -> [(R [9], t [3])] x 4 in candidate order (R1, t), (R2, t), (R1, -t), (R2, -t), or None.  V: the
    eigenvectors of E^T E ((E^T E)_ij = (E_0i E_0j + E_1i E_1j) + E_2i E_2j) by ``oracle.fundamental.jacobi_eigh``, in
    descending eigenvalue order (a stable sort: equal eigenvalues keep their column order); u_k = E v_k / |E v_k|
    (k = 1, 2; None when a norm is 0 or not finite), u3 = u1 x u2, v3 negated when det [v1 v2 v3] < 0;
    R1 = U W V^T = u2 v1^T - u1 v2^T + u3 v3^T, R2 = U W^T V^T = u1 v2^T - u2 v1^T + u3 v3^T (W = [[0,-1,0],[1,0,0],[0,0,1]]),
    entries ((a_r b_c) - (d_r e_c)) + (u3_r v3_c); t = u3."""
    E = [float(v) for v in np.asarray(E, np.float64).reshape(9)]
    e = lambda i, j: E[3 * i + j]
    A = [[((e(0, i) * e(0, j)) + (e(1, i) * e(1, j))) + (e(2, i) * e(2, j)) for j in range(3)] for i in range(3)]
    w, V = of.jacobi_eigh(A)
    o = [0, 1, 2]
    for a, b in ((0, 1), (1, 2), (0, 1)):
        if w[o[b]] > w[o[a]]:
            o[a], o[b] = o[b], o[a]
    v = [[V[r][o[k]] for r in range(3)] for k in range(3)]
    u = []
    for k in range(2):
        Ev = [((e(r, 0) * v[k][0]) + (e(r, 1) * v[k][1])) + (e(r, 2) * v[k][2]) for r in range(3)]
        nrm = float(np.sqrt(((Ev[0] * Ev[0]) + (Ev[1] * Ev[1])) + (Ev[2] * Ev[2])))
        if not (nrm > 0 and nrm < np.inf):
            return None
        u.append([Ev[r] / nrm for r in range(3)])
    u1, u2 = u
    u3 = [(u1[1] * u2[2]) - (u1[2] * u2[1]), (u1[2] * u2[0]) - (u1[0] * u2[2]), (u1[0] * u2[1]) - (u1[1] * u2[0])]
    Vm = np.array([[v[c][r] for c in range(3)] for r in range(3)]).reshape(1, 9)
    v3 = v[2]
    if of.det3(Vm)[0] < 0:
        v3 = [-x for x in v3]
    v1, v2 = v[0], v[1]
    R1 = [((u2[r] * v1[c]) - (u1[r] * v2[c])) + (u3[r] * v3[c]) for r in range(3) for c in range(3)]
    R2 = [((u1[r] * v2[c]) - (u2[r] * v1[c])) + (u3[r] * v3[c]) for r in range(3) for c in range(3)]
    nt = [-x for x in u3]
    return [(np.array(R1), np.array(u3)), (np.array(R2), np.array(u3)), (np.array(R1), np.array(nt)),
            (np.array(R2), np.array(nt))]


def cheirality(R, t, c1, c2, dist):
    """bool [n]: a = R x1 (x = (u, v, 1)), b = x2, the least-squares (z1, z2) of z2 x2 = z1 R x1 + t through the normal
    equations, det = (a.a)(b.b) - (a.b)^2, z1 = ((a.b)(b.t) - (a.t)(b.b)) / det; X = z1 x1, z = ((R20 X0 + R21 X1) + R22 X2)
    + t2; good when 0 < z1 < dist and 0 < z < dist."""
    u1, v1, u2, v2 = c1[:, 0], c1[:, 1], c2[:, 0], c2[:, 1]
    with np.errstate(all="ignore"):
        a = [((R[3 * r] * u1) + (R[3 * r + 1] * v1)) + R[3 * r + 2] for r in range(3)]
        b = [u2, v2, np.ones_like(u2)]
        aa, bb, ab = _dot3(a, a), _dot3(b, b), _dot3(a, b)
        at, bt = _dot3(a, t), _dot3(b, t)
        det = (aa * bb) - (ab * ab)
        z1 = ((ab * bt) - (at * bb)) / det
        X = [z1 * u1, z1 * v1, z1]
        z = (((R[6] * X[0]) + (R[7] * X[1])) + (R[8] * X[2])) + t[2]
        return (z1 > 0) & (z1 < dist) & (z > 0) & (z < dist)


def recover_pose_pair(E, p1, p2, n, K1, K2, mask, dist):
    """One pair -> (R [9], t [3], pose mask uint8 [n], n_good): the candidate with the most good matches among the masked
    valid ones, the first on ties; all zeros for an all-zero E, an invalid K or a failed decomposition."""
    p1, p2 = np.asarray(p1, np.float64)[:n], np.asarray(p2, np.float64)[:n]
    K1, K2 = np.asarray(K1, np.float64).reshape(9), np.asarray(K2, np.float64).reshape(9)
    zero = (np.zeros(9), np.zeros(3), np.zeros(n, np.uint8), 0)
    E = np.asarray(E, np.float64).reshape(9)
    if not E.any() or not (k_valid(K1) and k_valid(K2)):
        return zero
    cands = decompose(E)
    if cands is None:
        return zero
    c1, c2 = calibrate(p1, K1), calibrate(p2, K2)
    m = np.ones(n, bool) if mask is None else np.asarray(mask)[:n].astype(bool)
    goods = [cheirality(R, t, c1, c2, dist) & m for R, t in cands]
    cnt = [int(g.sum()) for g in goods]
    best = 0
    for i in range(1, 4):
        if cnt[i] > cnt[best]:
            best = i
    R, t = cands[best]
    return R, t, goods[best].astype(np.uint8), cnt[best]


def recover_pose(E, p1, p2, count, K, mask=None, dist=50.0):
    """Batched form of ``balf_recover_pose`` -> (R [B,3,3], t [B,3], pose mask uint8 [B,M], n_good int32 [B])."""
    p1, p2 = np.asarray(p1, np.float64), np.asarray(p2, np.float64)
    E = np.asarray(E, np.float64).reshape(-1, 9)
    K = np.asarray(K, np.float64).reshape(-1, 2, 9)
    B, M = p1.shape[:2]
    Rs, ts, masks, ns = np.zeros((B, 9)), np.zeros((B, 3)), np.zeros((B, M), np.uint8), np.zeros(B, np.int32)
    for b in range(B):
        n = int(min(max(int(count[b]), 0), M))
        Rs[b], ts[b], masks[b, :n], ns[b] = recover_pose_pair(E[b], p1[b], p2[b], n, K[b, 0], K[b, 1],
                                                              None if mask is None else mask[b], dist)
    return Rs.reshape(B, 3, 3), ts, masks, ns
