"""RANSAC fundamental matrix of ``balf_find_fundamental_ransac`` (balf_b200/csrc/fundamental.cu), restated in NumPy.

No reference counterpart: the reference's GoPro evaluation parser (config_gopro_eval.py) names epipolar verification
without implementing it, so the semantics are defined in include/balf_b200.h and restated here operation for operation.
PARITY UNPINNABLE against the reference; anchored instead on OpenCV (tests/test_oracle_fundamental.py: the 7-point solver
against ``cv2.findFundamentalMat(FM_7POINT)``, the refit against ``FM_8POINT``, the inlier rule against a transcription of
``FM_RANSAC``'s error, recovery of seeded two-view geometry).

The hash, the elimination and the fixed-order block sum are those of oracle/homography.py.  Every float64 operation is
elementwise IEEE arithmetic (+ - * / sqrt and comparisons only) in the order the kernels perform it, so the results are
bit-identical: vectorising over hypotheses changes no rounding.
"""
import math

import numpy as np

from oracle import homography as oh

SAMPLE = 7
MAX_DRAWS = 64
MAX_MODELS = 3
REFIT_PASSES = 8
REFIT_MIN = 8
MAX_BISECT = 200
JACOBI_SWEEPS = 32
JACOBI_TOL2 = 2.0 ** -104           # stop once the off-diagonal sum of squares is below this share of the diagonal's
SQRT2 = oh.SQRT2


def sample_indices(seed, b, hyps, n, k=SAMPLE, draws=MAX_DRAWS):
    """-> (idx int64 [len(hyps),k], ok bool [len(hyps)]): the k distinct match indices of hypotheses ``hyps`` of pair b drawn
    from n matches, in draw order; ok = False when ``draws`` counters did not give k distinct indices.  The kernels share
    one sampler; with k = 4, draws = 32 this is ``oracle.homography.sample_indices``."""
    hyps = np.asarray(hyps, dtype=np.uint64)
    base = np.uint64(oh.splitmix64(seed & oh.MASK64))
    stream = oh._splitmix64_np(base ^ ((np.uint64(b) << np.uint64(32)) | hyps))
    idx = np.full((len(hyps), k), -1, np.int64)
    got = np.zeros(len(hyps), np.int64)
    rows = np.arange(len(hyps))
    with np.errstate(over="ignore"):
        for c in range(draws):
            cand = (oh._splitmix64_np(stream + np.uint64(c)) % np.uint64(n)).astype(np.int64)
            take = (got < k) & ~(idx == cand[:, None]).any(1)
            idx[rows[take], got[take]] = cand[take]
            got += take
    return idx, got == k


def _normalise(x, y):
    """x, y [N,K] -> (u, v, cx, cy, s): centroid 0 and mean distance sqrt(2), sums in index order."""
    K = x.shape[1]
    with np.errstate(all="ignore"):
        cx, cy = x[:, 0].copy(), y[:, 0].copy()
        for i in range(1, K):
            cx, cy = cx + x[:, i], cy + y[:, i]
        cx, cy = cx / float(K), cy / float(K)
        dx, dy = x - cx[:, None], y - cy[:, None]
        d = np.sqrt((dx * dx) + (dy * dy))
        sd = d[:, 0].copy()
        for i in range(1, K):
            sd = sd + d[:, i]
        s = SQRT2 / (sd / float(K))
        return (x - cx[:, None]) * s[:, None], (y - cy[:, None]) * s[:, None], cx, cy, s


def epipolar_rows(u1, v1, u2, v2):
    """The row of x2^T F x1 = 0 in the entries of F (row-major): [u2 u1, u2 v1, u2, v2 u1, v2 v1, v2, u1, v1, 1]."""
    return np.stack([u2 * u1, u2 * v1, u2, v2 * u1, v2 * v1, v2, u1, v1, np.ones_like(u1)], -1)


def det3(m):
    """m [...,9] row-major -> determinant by the first row's cofactors."""
    return (((m[..., 0] * ((m[..., 4] * m[..., 8]) - (m[..., 5] * m[..., 7])))
             - (m[..., 1] * ((m[..., 3] * m[..., 8]) - (m[..., 5] * m[..., 6]))))
            + (m[..., 2] * ((m[..., 3] * m[..., 7]) - (m[..., 4] * m[..., 6]))))


def cubic_coeffs(F1, F2):
    """det(lam F1 + (1 - lam) F2) = det(F2 + lam D), D = F1 - F2, -> c [N,4] (c0 + c1 lam + c2 lam^2 + c3 lam^3): c1 sums the
    determinants of F2 with column j taken from D (j = 0, 1, 2), c2 those of D with column j taken from F2."""
    D = F1 - F2
    c1 = c2 = None
    for j in range(3):
        a, d = F2.copy(), D.copy()
        a[:, j::3], d[:, j::3] = D[:, j::3], F2[:, j::3]
        c1 = det3(a) if c1 is None else c1 + det3(a)
        c2 = det3(d) if c2 is None else c2 + det3(d)
    return np.stack([det3(F2), c1, c2, det3(D)], 1)


def _poly(c, x):
    return (((c[:, 3] * x) + c[:, 2]) * x + c[:, 1]) * x + c[:, 0]


def cubic_roots(c):
    """Real roots of c0 + c1 x + c2 x^2 + c3 x^3, c [N,4] -> (roots [N,3] ascending, NaN-padded; count [N]).

    The degree is the highest one whose Cauchy bound R = 1 + max |c_i / c_d| is finite.  The roots of the derivative
    (the stable quadratic formula; -c1 / (2 c2) for a quadratic), clamped to [-R, R], split [-R, R] into up to three
    monotone pieces [a, b].  A piece with a < b holds a root when f(b) = 0 (the root is b) or f(a) != 0 and the signs of
    f(a) and f(b) differ; bisection at mid = a / 2 + b / 2 keeps the half whose ends differ in sign, and stops when f(mid)
    = 0, when mid is no longer strictly inside, or after 200 steps.  The root is the last mid."""
    N = c.shape[0]
    inf = np.inf
    with np.errstate(all="ignore"):
        a0, a1, a2, a3 = (np.abs(c[:, i]) for i in range(4))
        R3 = 1.0 + (np.maximum(np.maximum(a0, a1), a2) / a3)
        R2 = 1.0 + (np.maximum(a0, a1) / a2)
        R1 = 1.0 + (a0 / a1)
        fin = lambda r: (r > 0) & (r < inf)
        d3, d2, d1 = fin(R3), ~fin(R3) & fin(R2), ~fin(R3) & ~fin(R2) & fin(R1)
        R = np.where(d3, R3, np.where(d2, R2, np.where(d1, R1, 0.0)))
        k1, k2 = -R, -R
        # cubic: 3 c3 x^2 + 2 c2 x + c1 = 0
        disc = (c[:, 2] * c[:, 2]) - ((3.0 * c[:, 3]) * c[:, 1])
        sq = np.sqrt(disc)
        q = np.where(c[:, 2] >= 0, -(c[:, 2] + sq), sq - c[:, 2])
        x1, x2 = q / (3.0 * c[:, 3]), c[:, 1] / q
        lo, hi = np.minimum(x1, x2), np.maximum(x1, x2)
        two = d3 & (disc > 0)
        k1, k2 = np.where(two, lo, k1), np.where(two, hi, k2)
        xq = (-c[:, 1]) / (2.0 * c[:, 2])
        k1 = np.where(d2, xq, k1)
        k2 = np.where(d2, xq, k2)
        clamp = lambda x: np.where(x < -R, -R, np.where(x > R, R, x))
        k1, k2 = clamp(k1), clamp(k2)
        knots = [-R, k1, k2, R]
        roots = np.full((N, 3), np.nan)
        cnt = np.zeros(N, np.int64)
        for p in range(3):
            a, b = knots[p], knots[p + 1]
            fa, fb = _poly(c, a), _poly(c, b)
            has = (d3 | d2 | d1) & (a < b) & ((fb == 0) | ((fa != 0) & ((fa < 0) != (fb < 0))))
            lo_, hi_, flo = a.copy(), b.copy(), fa.copy()
            mid = b.copy()
            act = has & (fb != 0)
            for _ in range(MAX_BISECT):
                if not act.any():
                    break
                m = (0.5 * lo_) + (0.5 * hi_)
                inside = act & (lo_ < m) & (m < hi_)
                mid = np.where(act, m, mid)
                fm = _poly(c, m)
                step = inside & (fm != 0)
                left = (fm < 0) == (flo < 0)
                lo_ = np.where(step & left, m, lo_)
                flo = np.where(step & left, fm, flo)
                hi_ = np.where(step & ~left, m, hi_)
                act = step
            roots[has, cnt[has]] = mid[has]
            cnt += has
    return roots, cnt


def scale_unit(F):
    """F [N,9] -> (F / |F|_F with its first largest-magnitude entry made positive, ok = the norm is > 0 and finite)."""
    with np.errstate(all="ignore"):
        s = F[:, 0] * F[:, 0]
        for i in range(1, 9):
            s = s + (F[:, i] * F[:, i])
        nrm = np.sqrt(s)
        ok = (nrm > 0) & (nrm < np.inf)
        G = F / nrm[:, None]
        j = np.zeros(len(F), np.int64)
        r = np.arange(len(F))
        for i in range(1, 9):
            j = np.where(np.abs(G[:, i]) > np.abs(G[r, j]), i, j)
        G = np.where((G[r, j] < 0)[:, None], -G, G)
    return G, ok


def denormalise(Fn, cx1, cy1, s1, cx2, cy2, s2):
    """F = T2^T Fn T1 (T = [[s, 0, -s cx], [0, s, -s cy], [0, 0, 1]]), scaled by ``scale_unit`` -> (F [N,9], ok [N])."""
    with np.errstate(all="ignore"):
        tx, ty = -(s1 * cx1), -(s1 * cy1)
        G = np.empty_like(Fn)
        for r in range(3):
            G[:, 3 * r] = Fn[:, 3 * r] * s1
            G[:, 3 * r + 1] = Fn[:, 3 * r + 1] * s1
            G[:, 3 * r + 2] = ((Fn[:, 3 * r] * tx) + (Fn[:, 3 * r + 1] * ty)) + Fn[:, 3 * r + 2]
        ux, uy = -(s2 * cx2), -(s2 * cy2)
        F = np.empty_like(Fn)
        for c in range(3):
            F[:, c] = s2 * G[:, c]
            F[:, 3 + c] = s2 * G[:, 3 + c]
            F[:, 6 + c] = ((ux * G[:, c]) + (uy * G[:, 3 + c])) + G[:, 6 + c]
    return scale_unit(F)


def null_space(a):
    """a [N,7,9] -> (F1, F2 [N,9], ok): the null space of the 7x9 system by two solves of oracle.homography.solve8, the
    eighth row fixing f7: F1 has f8 = 1, f7 = 0 and F2 has f8 = 0, f7 = 1.  The unit row is never a pivot before column 7,
    so both solves run the same elimination of the 7 rows."""
    N = a.shape[0]
    s1, s2 = np.zeros((N, 8, 9)), np.zeros((N, 8, 9))
    s1[:, :7, :8] = a[:, :, :8]
    s1[:, :7, 8] = -a[:, :, 8]
    s1[:, 7, 7] = 1.0
    s2[:, :7, :8] = a[:, :, :8]
    s2[:, 7, 7] = 1.0
    s2[:, 7, 8] = 1.0
    h1, ok1 = oh.solve8(s1)
    h2, ok2 = oh.solve8(s2)
    F1 = np.concatenate([h1, np.ones((N, 1))], 1)
    F2 = np.concatenate([h2, np.zeros((N, 1))], 1)
    return F1, F2, ok1 & ok2


def minimal_solve(q1, q2):
    """7-point solver: q1, q2 [N,7,2] -> (F [N,3,9] in root order, ok [N,3]); a slot without a model is zeros."""
    x1, y1 = q1[..., 0].astype(np.float64), q1[..., 1].astype(np.float64)
    x2, y2 = q2[..., 0].astype(np.float64), q2[..., 1].astype(np.float64)
    u1, v1, cx1, cy1, s1 = _normalise(x1, y1)
    u2, v2, cx2, cy2, s2 = _normalise(x2, y2)
    N = len(x1)
    with np.errstate(all="ignore"):
        F1, F2, ok = null_space(epipolar_rows(u1, v1, u2, v2))
        roots, cnt = cubic_roots(cubic_coeffs(F1, F2))
    out, oks = np.zeros((N, MAX_MODELS, 9)), np.zeros((N, MAX_MODELS), bool)
    for m in range(MAX_MODELS):
        lam = roots[:, m, None]
        with np.errstate(all="ignore"):
            Fn = (lam * F1) + ((1.0 - lam) * F2)
        F, okd = denormalise(Fn, cx1, cy1, s1, cx2, cy2, s2)
        oks[:, m] = ok & (cnt > m) & okd
        out[:, m] = np.where(oks[:, m, None], F, 0.0)
    return out, oks


def inliers(F, p1, p2, thr):
    """F [N,9], p1, p2 [n,2] -> bool [N,n]: with l2 = F x1 = (a, b, c), s = x2^T l2 and l1 = F^T x2 = (a', b', .), a match is
    an inlier when s^2 <= thr^2 (a^2 + b^2) and s^2 <= thr^2 (a'^2 + b'^2), each a^2 + b^2 finite and > 0 (the larger of
    the two point-to-line distances is at most thr)."""
    x1, y1, x2, y2 = p1[:, 0], p1[:, 1], p2[:, 0], p2[:, 1]
    f = [F[:, i, None] for i in range(9)]
    thr2 = thr * thr
    with np.errstate(all="ignore"):
        a = ((f[0] * x1) + (f[1] * y1)) + f[2]
        b = ((f[3] * x1) + (f[4] * y1)) + f[5]
        c = ((f[6] * x1) + (f[7] * y1)) + f[8]
        s = ((x2 * a) + (y2 * b)) + c
        ap = ((f[0] * x2) + (f[3] * y2)) + f[6]
        bp = ((f[1] * x2) + (f[4] * y2)) + f[7]
        s2, n2, n1 = s * s, (a * a) + (b * b), (ap * ap) + (bp * bp)
        return ((n2 > 0) & (n2 < np.inf) & (n1 > 0) & (n1 < np.inf) & (s2 <= thr2 * n2) & (s2 <= thr2 * n1))


def jacobi_eigh(A):
    """Cyclic Jacobi on a symmetric n x n matrix (a list of lists of floats, modified) -> (eigenvalues, V with the
    eigenvectors in its columns).  Each sweep first sums the squared off-diagonal entries and the squared diagonal in
    row-major order and stops when the former is not above 2^-104 times the latter (or after 32 sweeps); then it rotates
    every (p, q), p < q in row-major order, with a_pq != 0: theta = (a_qq - a_pp) / (2 a_pq),
    t = sign(theta) / (|theta| + sqrt(theta^2 + 1)), c = 1 / sqrt(t^2 + 1), s = t c; A <- A J column-wise, then J^T A
    row-wise, a_pq = a_qq = 0, V <- V J."""
    n = len(A)
    V = [[1.0 if i == j else 0.0 for j in range(n)] for i in range(n)]
    for _ in range(JACOBI_SWEEPS):
        off = 0.0
        dsq = 0.0
        for p in range(n):
            dsq = dsq + (A[p][p] * A[p][p])
            for q in range(p + 1, n):
                off = off + (A[p][q] * A[p][q])
        if not (off > JACOBI_TOL2 * dsq):
            break
        for p in range(n - 1):
            for q in range(p + 1, n):
                apq = A[p][q]
                if apq == 0.0:
                    continue
                theta = (A[q][q] - A[p][p]) / (2.0 * apq)
                t = 1.0 / (abs(theta) + math.sqrt((theta * theta) + 1.0))
                if theta < 0:
                    t = -t
                c = 1.0 / math.sqrt((t * t) + 1.0)
                s = t * c
                for k in range(n):
                    akp, akq = A[k][p], A[k][q]
                    A[k][p], A[k][q] = (c * akp) - (s * akq), (s * akp) + (c * akq)
                for k in range(n):
                    apk, aqk = A[p][k], A[q][k]
                    A[p][k], A[q][k] = (c * apk) - (s * aqk), (s * apk) + (c * aqk)
                A[p][q] = 0.0
                A[q][p] = 0.0
                for k in range(n):
                    vkp, vkq = V[k][p], V[k][q]
                    V[k][p], V[k][q] = (c * vkp) - (s * vkq), (s * vkp) + (c * vkq)
    return [A[i][i] for i in range(n)], V


def smallest_eigvec(A):
    """The column of V of the first smallest eigenvalue of ``jacobi_eigh``."""
    w, V = jacobi_eigh([list(map(float, r)) for r in A])
    j = 0
    for i in range(1, len(w)):
        if w[i] < w[j]:
            j = i
    return [V[k][j] for k in range(len(w))]


def rank2(f):
    """f [9] (row-major F) -> F - (F v3) v3^T, v3 the smallest eigenvector of F^T F: the nearest rank-2 matrix."""
    F = [[float(f[3 * r + c]) for c in range(3)] for r in range(3)]
    M = [[((F[0][i] * F[0][j]) + (F[1][i] * F[1][j])) + (F[2][i] * F[2][j]) for j in range(3)] for i in range(3)]
    v = smallest_eigvec(M)
    out = []
    for r in range(3):
        w = ((F[r][0] * v[0]) + (F[r][1] * v[1])) + (F[r][2] * v[2])
        out += [F[r][c] - (w * v[c]) for c in range(3)]
    return np.array(out)


def refit(p1, p2, mask):
    """Normalised 8-point least squares on the points where mask is set -> (F [9], ok): the smallest eigenvector of the
    9x9 normal matrix (its 45 upper-triangle sums in the block_sum order), made rank 2, denormalised and scaled."""
    n = len(p1)
    m = mask.astype(bool)
    dn = float(m.sum())
    x1, y1, x2, y2 = p1[:, 0], p1[:, 1], p2[:, 0], p2[:, 1]
    with np.errstate(all="ignore"):
        sA = oh.block_sum(np.where(m[:, None], np.stack([x1, y1, x2, y2], 1), 0.0), n)
        cx1, cy1, cx2, cy2 = sA / dn
        ax, ay, bx, by = x1 - cx1, y1 - cy1, x2 - cx2, y2 - cy2
        d = np.stack([np.sqrt((ax * ax) + (ay * ay)), np.sqrt((bx * bx) + (by * by))], 1)
        sB = oh.block_sum(np.where(m[:, None], d, 0.0), n)
        s1, s2 = SQRT2 / (sB[0] / dn), SQRT2 / (sB[1] / dn)
        r = epipolar_rows((x1 - cx1) * s1, (y1 - cy1) * s1, (x2 - cx2) * s2, (y2 - cy2) * s2)
        cols = [r[:, i] * r[:, j] for i in range(9) for j in range(i, 9)]
        sC = oh.block_sum(np.where(m[:, None], np.stack(cols, 1), 0.0), n)
        A = np.zeros((9, 9))
        q = 0
        for i in range(9):
            for j in range(i, 9):
                A[i, j] = A[j, i] = sC[q]
                q += 1
        Fn = rank2(smallest_eigvec(A))
        F, ok = denormalise(Fn[None], cx1, cy1, s1, cx2, cy2, s2)
    return F[0], bool(ok[0])


def hypotheses(p1, p2, n, b, iters, seed):
    """All hypotheses of pair b -> (F [iters*3,9], ok [iters*3]), slot 3 h + m = model m of hypothesis h."""
    idx, ok = sample_indices(seed, b, np.arange(iters), max(n, 1))
    idx = np.where(ok[:, None], idx, 0)
    F, ok_m = minimal_solve(p1[idx], p2[idx])
    ok_m &= ok[:, None]
    return np.where(ok_m[..., None], F, 0.0).reshape(-1, 9), ok_m.reshape(-1)


def find_fundamental_ransac_pair(p1, p2, n, b, thr, iters, seed, chunk=256):
    """One pair (index b of its batch, n valid rows) -> (F [9], mask uint8 [n], n_inliers)."""
    p1, p2 = np.asarray(p1, np.float64)[:n], np.asarray(p2, np.float64)[:n]
    if n < SAMPLE:
        return np.zeros(9), np.zeros(n, np.uint8), 0
    F, ok = hypotheses(p1, p2, n, b, iters, seed)
    S = len(F)
    score = np.full(S, -1, np.int64)
    for s in range(0, S, chunk):
        e = min(S, s + chunk)
        score[s:e] = np.where(ok[s:e], inliers(F[s:e], p1, p2, thr).sum(1), -1)
    win = int(np.argmax(score))                                 # first maximum = lowest 3 h + m
    if score[win] < 0:
        return np.zeros(9), np.zeros(n, np.uint8), 0
    Fc = F[win]
    mask = inliers(Fc[None], p1, p2, thr)[0]
    cnt = int(mask.sum())
    for _ in range(REFIT_PASSES):
        if cnt < REFIT_MIN:
            break
        G, ok_r = refit(p1, p2, mask)
        if not ok_r:
            break
        m2 = inliers(G[None], p1, p2, thr)[0]
        c2 = int(m2.sum())
        grew = c2 > cnt
        Fc, mask, cnt = G, m2, c2
        if not grew:
            break
    return Fc, mask.astype(np.uint8), cnt


def find_fundamental_ransac(p1, p2, count, thr, iters, seed):
    """Batched form of ``balf_find_fundamental_ransac``: p1, p2 [B,M,2], count [B] -> (F [B,3,3], mask uint8 [B,M],
    n_inliers int32 [B])."""
    p1, p2 = np.asarray(p1, np.float64), np.asarray(p2, np.float64)
    B, M = p1.shape[:2]
    Fs, masks, ns = np.zeros((B, 9)), np.zeros((B, M), np.uint8), np.zeros(B, np.int32)
    for b in range(B):
        n = int(min(max(int(count[b]), 0), M))
        Fs[b], masks[b, :n], ns[b] = find_fundamental_ransac_pair(p1[b], p2[b], n, b, thr, iters, seed)
    return Fs.reshape(B, 3, 3), masks, ns
