"""RANSAC homography of ``balf_find_homography_ransac`` (balf_b200/csrc/homography.cu), restated in NumPy.

No reference counterpart: the reference has no homography estimation (its evaluation parsers name the measure only), so the
semantics are defined in include/balf_b200.h and restated here operation for operation.  PARITY UNPINNABLE against the
reference; anchored instead on OpenCV (tests/test_oracle_homography.py: the minimal solver against
``cv2.getPerspectiveTransform``, the refit against ``cv2.findHomography(..., 0)``, recovery of seeded ground truths next to
``cv2.findHomography(..., cv2.RANSAC)``).

Every float64 operation below is elementwise IEEE arithmetic in the order the kernel performs it (the kernel is compiled
without FMA contraction), so results are bit-identical: vectorising over hypotheses changes no rounding.
"""
import numpy as np

MASK64 = (1 << 64) - 1
MAX_DRAWS = 32
REFIT_PASSES = 8
COLLINEAR_TOL = 1e-6
SQRT2 = 1.4142135623730951
REFIT_THREADS = 256


def splitmix64(z):
    """The hash on Python integers (the definition)."""
    z = (z + 0x9E3779B97F4A7C15) & MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    return z ^ (z >> 31)


def _splitmix64_np(z):
    """splitmix64 on uint64 arrays (wrapping arithmetic); equal to ``splitmix64`` elementwise."""
    z = np.asarray(z, dtype=np.uint64) + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def sample_indices(seed, b, hyps, n):
    """-> (idx int64 [len(hyps),4], ok bool [len(hyps)]): the 4 distinct match indices of hypotheses ``hyps`` of pair b
    drawn from n matches, in draw order; ok = False when 32 counters did not give 4 distinct indices."""
    hyps = np.asarray(hyps, dtype=np.uint64)
    base = np.uint64(splitmix64(seed & MASK64))
    stream = _splitmix64_np(base ^ ((np.uint64(b) << np.uint64(32)) | hyps))
    idx = np.full((len(hyps), 4), -1, np.int64)
    k = np.zeros(len(hyps), np.int64)
    rows = np.arange(len(hyps))
    with np.errstate(over="ignore"):
        draws = [(_splitmix64_np(stream + np.uint64(c)) % np.uint64(n)).astype(np.int64) for c in range(MAX_DRAWS)]
    for c in range(MAX_DRAWS):
        cand = draws[c]
        take = (k < 4) & ~(idx == cand[:, None]).any(1)
        idx[rows[take], k[take]] = cand[take]
        k += take
    return idx, k == 4


def solve8(a):
    """Gaussian elimination with partial pivoting on augmented systems a [N,8,9] (modified) -> (h [N,8], ok [N]).
    The pivot is np.argmax of |column| (first maximum; NaN counts as the maximum); ok = False when a pivot is 0 or not
    finite."""
    N = a.shape[0]
    r = np.arange(N)
    ok = np.ones(N, bool)
    with np.errstate(all="ignore"):
        for k in range(8):
            col = np.abs(a[:, k:, k])
            p = k + np.argmax(col, axis=1)
            best = col[r, p - k]
            ok &= (best > 0) & (best < np.inf)
            rk, rp = a[r, k].copy(), a[r, p].copy()
            a[r, k], a[r, p] = rp, rk
            d = a[:, k, k]
            f = a[:, k + 1:, k] / d[:, None]
            a[:, k + 1:, k + 1:] = a[:, k + 1:, k + 1:] - f[:, :, None] * a[:, k, None, k + 1:]
        h = np.zeros((N, 8))
        for k in range(7, -1, -1):
            s = a[:, k, 8].copy()
            for c in range(k + 1, 8):
                s = s - a[:, k, c] * h[:, c]
            h[:, k] = s / a[:, k, k]
    return h, ok


def denormalise(hn, cx1, cy1, s1, cx2, cy2, s2):
    """H = T2^-1 Hn T1 scaled to H[8] = 1 -> (H [N,9], ok [N]); arguments are [N] arrays (or scalars)."""
    N = hn.shape[0]
    Hn = np.concatenate([hn, np.ones((N, 1))], 1)
    with np.errstate(all="ignore"):
        tx, ty = -(s1 * cx1), -(s1 * cy1)
        G = np.empty((N, 9))
        for r in range(3):
            G[:, 3 * r] = Hn[:, 3 * r] * s1
            G[:, 3 * r + 1] = Hn[:, 3 * r + 1] * s1
            G[:, 3 * r + 2] = ((Hn[:, 3 * r] * tx) + (Hn[:, 3 * r + 1] * ty)) + Hn[:, 3 * r + 2]
        H = np.empty((N, 9))
        for c in range(3):
            H[:, c] = (G[:, c] / s2) + (cx2 * G[:, 6 + c])
            H[:, 3 + c] = (G[:, 3 + c] / s2) + (cy2 * G[:, 6 + c])
            H[:, 6 + c] = G[:, 6 + c]
        w = H[:, 8].copy()
        ok = (np.abs(w) > 0) & (np.abs(w) < np.inf)
        H[:, :8] = H[:, :8] / w[:, None]
        H[:, 8] = 1.0
    return H, ok


def _dlt_rows(u, v, up, vp):
    z, o = np.zeros_like(u), np.ones_like(u)
    a = np.stack([u, v, o, z, z, z, -(u * up), -(v * up)], -1)
    b = np.stack([z, z, z, u, v, o, -(u * vp), -(v * vp)], -1)
    return a, b


def _normalise4(x, y):
    """x, y [N,4] -> (u, v, cx, cy, s)."""
    with np.errstate(all="ignore"):
        cx = (((x[:, 0] + x[:, 1]) + x[:, 2]) + x[:, 3]) / 4.0
        cy = (((y[:, 0] + y[:, 1]) + y[:, 2]) + y[:, 3]) / 4.0
        dx, dy = x - cx[:, None], y - cy[:, None]
        d = np.sqrt((dx * dx) + (dy * dy))
        s = SQRT2 / ((((d[:, 0] + d[:, 1]) + d[:, 2]) + d[:, 3]) / 4.0)
        return (x - cx[:, None]) * s[:, None], (y - cy[:, None]) * s[:, None], cx, cy, s


def _collinear(x, y, i0, i1, i2):
    with np.errstate(all="ignore"):
        dx1, dy1 = x[:, i1] - x[:, i0], y[:, i1] - y[:, i0]
        dx2, dy2 = x[:, i2] - x[:, i0], y[:, i2] - y[:, i0]
        return ~(np.abs((dx1 * dy2) - (dy1 * dx2)) > COLLINEAR_TOL)


def minimal_solve(q1, q2):
    """4-point normalised DLT: q1, q2 [N,4,2] -> (H [N,9], ok [N]) (ok = False for a degenerate sample)."""
    x1, y1 = q1[..., 0].astype(np.float64), q1[..., 1].astype(np.float64)
    x2, y2 = q2[..., 0].astype(np.float64), q2[..., 1].astype(np.float64)
    u1, v1, cx1, cy1, s1 = _normalise4(x1, y1)
    u2, v2, cx2, cy2, s2 = _normalise4(x2, y2)
    ok = np.ones(len(x1), bool)
    for t in ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3)):
        ok &= ~_collinear(u1, v1, *t) & ~_collinear(u2, v2, *t)
    a = np.zeros((len(x1), 8, 9))
    with np.errstate(all="ignore"):
        ra, rb = _dlt_rows(u1, v1, u2, v2)                      # [N,4,8]
    a[:, 0::2, :8], a[:, 1::2, :8] = ra, rb
    a[:, 0::2, 8], a[:, 1::2, 8] = u2, v2
    hn, ok_s = solve8(a)
    H, ok_d = denormalise(hn, cx1, cy1, s1, cx2, cy2, s2)
    return H, ok & ok_s & ok_d


def inliers(H, p1, p2, thr):
    """H [N,9], p1, p2 [n,2] -> bool [N,n]: w > 0 and |(X, Y) * (1 / w) - p2|^2 <= thr^2."""
    x1, y1, x2, y2 = p1[:, 0], p1[:, 1], p2[:, 0], p2[:, 1]
    h = [H[:, i, None] for i in range(9)]
    with np.errstate(all="ignore"):
        X = ((h[0] * x1) + (h[1] * y1)) + h[2]
        Y = ((h[3] * x1) + (h[4] * y1)) + h[5]
        w = ((h[6] * x1) + (h[7] * y1)) + h[8]
        iw = 1.0 / w
        dx, dy = (X * iw) - x2, (Y * iw) - y2
        return (w > 0) & (((dx * dx) + (dy * dy)) <= thr * thr)


def block_sum(terms, n):
    """The refit kernel's sum of terms [n,K] (zeros where a point does not contribute) -> [K]: thread t of 256 adds rows
    t, t + 256, ... in order starting from 0.0, then a tree inside each 32-lane warp (lane t += lane t + o, o = 16 .. 1) and
    a tree over the 8 warp sums (o = 4, 2, 1)."""
    R = -(-n // REFIT_THREADS)
    T = np.zeros((R * REFIT_THREADS, terms.shape[1]))
    T[:n] = terms
    T = T.reshape(R, REFIT_THREADS, -1)
    acc = np.zeros((REFIT_THREADS, terms.shape[1]))
    for r in range(R):
        acc = acc + T[r]
    w = acc.reshape(8, 32, -1)
    for o in (16, 8, 4, 2, 1):
        w = w[:, :o] + w[:, o:2 * o]
    w = w[:, 0]
    for o in (4, 2, 1):
        w = w[:o] + w[o:2 * o]
    return w[0]


def refit(p1, p2, mask):
    """Least-squares normalised DLT on the points where mask is set -> (H [9], ok)."""
    n = len(p1)
    m = mask.astype(bool)
    dn = float(m.sum())
    x1, y1, x2, y2 = p1[:, 0], p1[:, 1], p2[:, 0], p2[:, 1]
    with np.errstate(all="ignore"):
        sA = block_sum(np.where(m[:, None], np.stack([x1, y1, x2, y2], 1), 0.0), n)
        cx1, cy1, cx2, cy2 = sA / dn
        ax, ay, bx, by = x1 - cx1, y1 - cy1, x2 - cx2, y2 - cy2
        d = np.stack([np.sqrt((ax * ax) + (ay * ay)), np.sqrt((bx * bx) + (by * by))], 1)
        sB = block_sum(np.where(m[:, None], d, 0.0), n)
        s1, s2 = SQRT2 / (sB[0] / dn), SQRT2 / (sB[1] / dn)
        up, vp = (x2 - cx2) * s2, (y2 - cy2) * s2
        a, b = _dlt_rows((x1 - cx1) * s1, (y1 - cy1) * s1, up, vp)
        cols = [(a[:, i] * a[:, j]) + (b[:, i] * b[:, j]) for i in range(8) for j in range(i, 8)]
        cols += [(a[:, i] * up) + (b[:, i] * vp) for i in range(8)]
        sC = block_sum(np.where(m[:, None], np.stack(cols, 1), 0.0), n)
    A = np.zeros((1, 8, 9))
    q = 0
    for i in range(8):
        for j in range(i, 8):
            A[0, i, j] = A[0, j, i] = sC[q]
            q += 1
    A[0, :, 8] = sC[36:]
    hn, ok_s = solve8(A)
    H, ok_d = denormalise(hn, cx1, cy1, s1, cx2, cy2, s2)
    return H[0], bool(ok_s[0] and ok_d[0])


def hypotheses(p1, p2, n, b, iters, seed):
    """All hypotheses of pair b -> (H [iters,9], ok [iters])."""
    idx, ok = sample_indices(seed, b, np.arange(iters), max(n, 1))
    idx = np.where(ok[:, None], idx, 0)
    H, ok_h = minimal_solve(p1[idx], p2[idx])
    return H, ok & ok_h


def find_homography_ransac_pair(p1, p2, n, b, thr, iters, seed, chunk=256):
    """One pair (index b of its batch, n valid rows) -> (H [9], mask uint8 [n], n_inliers)."""
    p1, p2 = np.asarray(p1, np.float64)[:n], np.asarray(p2, np.float64)[:n]
    if n < 4:
        return np.zeros(9), np.zeros(n, np.uint8), 0
    H, ok = hypotheses(p1, p2, n, b, iters, seed)
    score = np.full(iters, -1, np.int64)
    for s in range(0, iters, chunk):
        e = min(iters, s + chunk)
        score[s:e] = np.where(ok[s:e], inliers(H[s:e], p1, p2, thr).sum(1), -1)
    win = int(np.argmax(score))                                 # first maximum = lowest hypothesis index
    if score[win] < 0:
        return np.zeros(9), np.zeros(n, np.uint8), 0
    Hc = H[win]
    mask = inliers(Hc[None], p1, p2, thr)[0]
    cnt = int(mask.sum())
    for _ in range(REFIT_PASSES):
        if cnt < 4:
            break
        G, ok_r = refit(p1, p2, mask)
        if not ok_r:
            break
        m2 = inliers(G[None], p1, p2, thr)[0]
        c2 = int(m2.sum())
        grew = c2 > cnt
        Hc, mask, cnt = G, m2, c2
        if not grew:
            break
    return Hc, mask.astype(np.uint8), cnt


def find_homography_ransac(p1, p2, count, thr, iters, seed):
    """Batched form of ``balf_find_homography_ransac``: p1, p2 [B,M,2], count [B] -> (H [B,3,3], mask uint8 [B,M],
    n_inliers int32 [B])."""
    p1, p2 = np.asarray(p1, np.float64), np.asarray(p2, np.float64)
    B, M = p1.shape[:2]
    Hs, masks, ns = np.zeros((B, 9)), np.zeros((B, M), np.uint8), np.zeros(B, np.int32)
    for b in range(B):
        n = int(min(max(int(count[b]), 0), M))
        Hs[b], masks[b, :n], ns[b] = find_homography_ransac_pair(p1[b], p2[b], n, b, thr, iters, seed)
    return Hs.reshape(B, 3, 3), masks, ns
