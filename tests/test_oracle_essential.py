"""RANSAC essential-matrix and relative-pose restatement (oracle/essential.py) on the CPU, anchored on NumPy and on OpenCV.

The essential-matrix stage has no reference counterpart, so its semantics (include/balf_b200.h,
balf_find_essential_ransac and balf_recover_pose) are defined by this project; these tests pin the restatement that
tests/test_gpu_essential.py holds the kernels to."""
import numpy as np
import pytest

from oracle import essential as oe
from oracle import fundamental as of
from oracle import homography as oh

cv2 = pytest.importorskip("cv2")

W, H = 1200, 900
K = np.array([[800.0, 0, W / 2], [0, 800.0, H / 2], [0, 0, 1]])
K9 = K.reshape(9)


def rot(v):
    a = np.linalg.norm(v)
    k = v / a
    S = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(a) * S + (1 - np.cos(a)) * S @ S


def skew(t):
    return np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])


def two_view(rng, n, ratio, sigma=0.5, K1=K, K2=K):
    """test_gpu_fundamental's seeded two-view scene with known cameras: 3-D points 4 - 10 units in front of camera 1,
    camera 2 rotated by up to 0.1 rad and translated by about one unit; a fraction `ratio` of the matches with N(0, sigma)
    pixel noise, the rest uniform outliers, shuffled -> (p1, p2, E_gt (unit, library sign), R, t (unit), is_inlier)."""
    X = np.c_[rng.uniform(-3, 3, (n, 2)), rng.uniform(4, 10, n)]
    R = rot(rng.uniform(-0.1, 0.1, 3))
    t = np.array([1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)])
    a, b = X @ K1.T, (X @ R.T + t) @ K2.T
    p1, p2 = a[:, :2] / a[:, 2:], b[:, :2] / b[:, 2:]
    k = int(round(ratio * n))
    p2[:k] += rng.normal(0, sigma, (k, 2))
    p2[k:] = rng.uniform([0, 0], [W, H], (n - k, 2))
    perm = rng.permutation(n)
    return p1[perm], p2[perm], unit(skew(t) @ R), R, t / np.linalg.norm(t), perm < k


def unit(E):
    f = np.asarray(E, np.float64).reshape(-1)
    f = f / np.linalg.norm(f)
    return f * np.sign(f[np.argmax(np.abs(f))])


def calibrated_sample(rng):
    """5 noise-free calibrated correspondences of a random pose -> (c1, c2 [5,2], E_gt)."""
    X = np.c_[rng.uniform(-3, 3, (5, 2)), rng.uniform(4, 10, 5)]
    R = rot(rng.uniform(-0.2, 0.2, 3))
    t = np.array([1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)])
    b = X @ R.T + t
    return X[:, :2] / X[:, 2:], b[:, :2] / b[:, 2:], unit(skew(t) @ R)


def em_error(E, c1, c2):
    """cv2's EMEstimatorCallback::computeError, transcribed (without its float32 rounding)."""
    E = np.asarray(E, np.float64).reshape(3, 3)
    x1, x2 = np.c_[c1, np.ones(len(c1))], np.c_[c2, np.ones(len(c2))]
    Ex1, Etx2 = x1 @ E.T, x2 @ E
    s = (x2 * Ex1).sum(1)
    d = Ex1[:, 0] ** 2 + Ex1[:, 1] ** 2 + Etx2[:, 0] ** 2 + Etx2[:, 1] ** 2
    return s * s / d


# ------------------------------------------------------------------------------------------ sampler
def test_sampler_five_distinct_on_the_shared_streams():
    for n in (5, 6, 50, 16384):
        idx, ok = of.sample_indices(11, 2, np.arange(2000), n, k=5, draws=oe.MAX_DRAWS)
        good = idx[ok]
        assert ((good >= 0) & (good < n)).all()
        assert all(len(set(r)) == 5 for r in good.tolist())
        assert ok.mean() > 0.999
    # the streams are the homography's and the fundamental matrix's: the same first draws
    a, _ = of.sample_indices(3, 5, np.arange(3000), 1000, k=5, draws=oe.MAX_DRAWS)
    b, _ = oh.sample_indices(3, 5, np.arange(3000), 1000)
    c, _ = of.sample_indices(3, 5, np.arange(3000), 1000)
    np.testing.assert_array_equal(a[:, :4], b)
    np.testing.assert_array_equal(a, c[:, :5])


# ------------------------------------------------------------------------------------------ null space
def test_null_space():
    rng = np.random.default_rng(1)
    c1 = rng.uniform(-1, 1, (200, 5, 2))
    c2 = rng.uniform(-1, 1, (200, 5, 2))
    rows = of.epipolar_rows(c1[..., 0], c1[..., 1], c2[..., 0], c2[..., 1])
    X, Y, Z, Wv, ok = oe.null_basis(rows)
    assert ok.all()
    Xo, Yo, Zo, Wo, ok2 = oe.orthonormalise(X, Y, Z, Wv)
    assert ok2.all()
    for basis in ((X, Y, Z, Wv), (Xo, Yo, Zo, Wo)):
        for v in basis:
            r = np.einsum("nij,nj->ni", rows, v)
            assert np.abs(r).max() < 1e-12 * np.abs(v).max(1).max()
    G = np.stack([Xo, Yo, Zo, Wo], 1)
    np.testing.assert_allclose(G @ G.transpose(0, 2, 1), np.broadcast_to(np.eye(4), (200, 4, 4)), atol=1e-12)


# ------------------------------------------------------------------------------------------ Sturm roots
def real_roots(c):
    c = np.trim_zeros(c, "b")
    r = np.roots(c[::-1])
    return np.sort(r[np.abs(r.imag) <= 1e-7 * np.maximum(1, np.abs(r))].real)


def poly_of(roots, extra=()):
    """ascending coefficients of prod (z - r) times the quadratic factors in extra (each (p, q): z^2 + p z + q)."""
    c = np.poly(roots) if len(roots) else np.array([1.0])
    for p, q in extra:
        c = np.polymul(c, [1.0, p, q])
    return c[::-1].copy()


@pytest.mark.parametrize("roots,extra,tol", [
    ((-3.0, -1.5, -0.2, 0.1, 0.7, 1.0, 2.5, 4.0, 9.0, 30.0), (), 1e-9),      # ten real roots
    ((-0.5, 0.25, 2.0), ((0.0, 1.0), (2.0, 5.0), (-1.0, 3.0)), 1e-12),
    ((1.0, 1.0 + 1e-4, 1.0 + 2e-4, 5.0), ((0.0, 4.0), (1.0, 1.0), (0.0, 9.0)), 1e-6),   # a cluster
    ((), ((0.0, 1.0), (1.0, 2.0), (-2.0, 5.0), (0.3, 0.2), (0.0, 7.0)), 0.0),           # no real roots, degree 10
])
def test_sturm_roots_vs_np_roots(roots, extra, tol):
    c = poly_of(roots, extra) * 0.37
    got, cnt = oe.poly_roots(np.pad(c, (0, 11 - len(c)))[None])
    want = np.sort(np.array(roots))
    assert cnt[0] == len(want)
    np.testing.assert_allclose(got[0, :cnt[0]], want, rtol=tol, atol=tol)
    np.testing.assert_allclose(got[0, :cnt[0]], real_roots(c), rtol=max(tol, 1e-7), atol=max(tol, 1e-7))


def test_sturm_roots_random_and_degree_drop():
    rng = np.random.default_rng(2)
    c = rng.normal(size=(500, 11))
    got, cnt = oe.poly_roots(c)
    for i in range(len(c)):
        want = real_roots(c[i])
        assert cnt[i] == len(want)
        np.testing.assert_allclose(got[i, :cnt[i]], want, rtol=1e-7, atol=1e-7)
    # vanishing leading coefficients: the degree drops to the highest finite Cauchy bound
    q = np.zeros((3, 11))
    q[0, :4] = poly_of((-2.0, 0.5, 3.0))
    q[1, :4] = poly_of((-2.0, 0.5, 3.0))
    q[1, 10] = 1e-320                                               # denormal: 1 + max / |c10| overflows
    q[2, :3] = poly_of((1.0, 2.0))
    got, cnt = oe.poly_roots(q)
    np.testing.assert_allclose(got[0, :3], [-2.0, 0.5, 3.0], rtol=1e-13)
    np.testing.assert_allclose(got[1, :3], [-2.0, 0.5, 3.0], rtol=1e-13)
    np.testing.assert_allclose(got[2, :2], [1.0, 2.0], rtol=1e-13)
    assert list(cnt) == [3, 3, 2]
    bad = np.zeros((3, 11))
    bad[0, 0] = 1.0                                                 # a constant
    bad[2, :3] = [np.nan, 1.0, 1.0]
    assert (oe.poly_roots(bad)[1] == 0).all()


# ------------------------------------------------------------------------------------------ minimal solver
def test_minimal_solver_vs_cv2_five_points():
    rng = np.random.default_rng(3)
    samples = [calibrated_sample(rng) for _ in range(300)]
    c1, c2 = np.array([s[0] for s in samples]), np.array([s[1] for s in samples])
    E, ok = oe.minimal_solve(c1, c2)
    gt_err, cv_err, resid = [], [], []
    for i, (a, b, Eg) in enumerate(samples):
        sols = E[i][ok[i]]
        assert len(sols) >= 1
        gt_err.append(min(np.abs(s - Eg).max() for s in sols))
        Ec, _ = cv2.findEssentialMat(a, b, np.eye(3), cv2.RANSAC, 0.999, 1e-3)
        for j in range(0 if Ec is None else len(Ec) // 3):
            cv_err.append(min(np.abs(s - unit(Ec[3 * j:3 * j + 3])).max() for s in sols))
        for s in sols:                                               # every model is an essential matrix of its sample
            M = s.reshape(3, 3)
            resid.append(max(abs(np.linalg.det(M)), np.abs(2 * M @ M.T @ M - np.trace(M @ M.T) * M).max(),
                             np.abs((np.c_[b, np.ones(5)] * (np.c_[a, np.ones(5)] @ M.T)).sum(1)).max()))
    # measured over these 300 samples: ground truth max 3.0e-3, median 1.8e-14; cv2's 1400 solutions max 5.2e-2, median
    # 8.6e-14 (both lose accuracy on the same few ill-conditioned samples)
    print("ground truth: max %.2e median %.2e; cv2 (%d): max %.2e median %.2e" %
          (max(gt_err), np.median(gt_err), len(cv_err), max(cv_err), np.median(cv_err)))
    # every model is an essential matrix of its sample (|E| = 1, so the bounds are relative): det E, the trace constraint
    # and the epipolar residuals.  Measured: max 2.7e-2, 99th percentile 1.0e-7 (the largest from nearly coincident roots)
    print("residuals: max %.2e, 99th percentile %.2e over %d models" % (max(resid), np.quantile(resid, 0.99), len(resid)))
    assert np.quantile(resid, 0.99) < 1e-6 and max(resid) < 0.1
    assert np.quantile(gt_err, 0.99) < 1e-5 and max(gt_err) < 1e-2 and np.median(gt_err) < 1e-12
    assert np.quantile(cv_err, 0.99) < 1e-5 and max(cv_err) < 0.1 and np.median(cv_err) < 1e-12


def test_minimal_solver_degenerate_samples():
    rng = np.random.default_rng(4)
    a, b, _ = calibrated_sample(rng)
    same = np.tile(a[:1], (5, 1))
    pair1, pair2 = np.r_[a[:2], a[:2], a[:1]], np.r_[b[:2], b[:2], b[:1]]      # two matches repeated: rank 3
    # one image's points identical (a zero pivot or a NaN scale), two matches repeated (rank 3), everything identical
    E, ok = oe.minimal_solve(np.stack([same, pair1, same]), np.stack([b, pair2, same]))
    assert not ok.any() and not E.any()


# ------------------------------------------------------------------------------------------ inlier rule and threshold
def test_inlier_rule_vs_cv2_error():
    rng = np.random.default_rng(6)
    p1, p2, Eg, _, _, truth = two_view(rng, 3000, 0.6, sigma=2.0)
    c1, c2 = oe.calibrate(p1, K9), oe.calibrate(p2, K9)
    for thr in (0.5, 1.0, 3.0):
        t2 = oe.pair_thr2(thr, K9, K9)
        got = oe.inliers(Eg[None], c1, c2, t2)[0]
        err = em_error(Eg, c1, c2)
        close = np.abs(err - t2) < 1e-9 * t2
        assert (got == (err <= t2))[~close].all() and got.sum() > 100
    assert not oe.inliers(np.zeros((1, 9)), c1, c2, 1.0).any()


def test_threshold_rule_matches_cv2_two_camera_overload():
    """cv2's two-camera findEssentialMat scores with thr / ((fx1 + fy1 + fx2 + fy2) / 4): its own E and that rule give its
    mask (up to its float32 rounding of the error)."""
    rng = np.random.default_rng(7)
    K1 = np.array([[700.0, 0, 590], [0, 760.0, 440], [0, 0, 1]])
    K2 = np.array([[1100.0, 0, 610], [0, 1000.0, 455], [0, 0, 1]])
    p1, p2, _, _, _, _ = two_view(rng, 2000, 0.6, sigma=1.0, K1=K1, K2=K2)
    Ec, mc = cv2.findEssentialMat(p1, p2, K1, np.zeros(5), K2, np.zeros(5), cv2.RANSAC, 0.999, 1.0)
    c1, c2 = oe.calibrate(p1, K1.reshape(9)), oe.calibrate(p2, K2.reshape(9))
    t2 = oe.pair_thr2(1.0, K1.reshape(9), K2.reshape(9))
    err = em_error(Ec[:3], c1, c2)
    decided = np.abs(err - t2) > 1e-6 * t2
    np.testing.assert_array_equal((err <= t2)[decided], mc[decided, 0].astype(bool))
    for f in ((700 + 760) / 2, (1100 + 1000) / 2):                  # either camera's own focal length alone differs
        assert ((err <= (1.0 / f) ** 2) != mc[:, 0].astype(bool)).sum() > 10


# ------------------------------------------------------------------------------------------ decomposition and pose
def test_decomposition_vs_cv2():
    rng = np.random.default_rng(8)
    for _ in range(50):
        _, _, Eg = calibrated_sample(rng)
        E = unit(Eg + rng.normal(0, 1e-3, 9))                      # not exactly rank 2
        cands = oe.decompose(E)
        R1, R2, t = cv2.decomposeEssentialMat(E.reshape(3, 3))
        Rs = [c[0].reshape(3, 3) for c in cands[:2]]
        for R in Rs:
            np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-13)
            assert abs(np.linalg.det(R) - 1) < 1e-13
        assert min(np.abs(Rs[0] - R1).max(), np.abs(Rs[1] - R1).max()) < 1e-9
        assert min(np.abs(Rs[0] - R2).max(), np.abs(Rs[1] - R2).max()) < 1e-9
        assert min(np.abs(cands[0][1] - t[:, 0]).max(), np.abs(cands[0][1] + t[:, 0]).max()) < 1e-9
        np.testing.assert_array_equal(cands[2][0], cands[0][0])
        np.testing.assert_array_equal(cands[2][1], -cands[0][1])


def test_recover_pose_vs_cv2():
    rng = np.random.default_rng(9)
    for trial in range(10):
        p1, p2, Eg, R, t, truth = two_view(rng, 500, 0.7, sigma=0.3)
        dist = 50.0 if trial % 2 else 8.0                         # 8: the far points fail the distance test
        mask = truth.astype(np.uint8) if trial % 3 else None
        Ro, to, mo, no = oe.recover_pose_pair(Eg, p1, p2, 500, K9, K9, mask, dist)
        kw = {} if mask is None else {"mask": mask.reshape(-1, 1).copy()}
        nc, Rc, tc, mc, _ = cv2.recoverPose(Eg.reshape(3, 3), p1, p2, K, distanceThresh=dist, **kw)
        np.testing.assert_allclose(Ro.reshape(3, 3), Rc, atol=1e-9)
        np.testing.assert_allclose(to, tc[:, 0], atol=1e-9)
        np.testing.assert_allclose(Ro.reshape(3, 3), R, atol=0.02)
        np.testing.assert_allclose(to, t, atol=0.05)
        # the good counts agree except for matches within a margin of a bound: recompute the depths exactly
        c1, c2 = oe.calibrate(p1, K9), oe.calibrate(p2, K9)
        X = np.array([cv2.triangulatePoints(np.eye(3, 4), np.c_[Rc, tc], c1[i:i + 1].T, c2[i:i + 1].T)[:, 0]
                      for i in range(500)])
        z1 = X[:, 2] / X[:, 3]
        z2 = (X[:, :3] / X[:, 3:]) @ Rc[2] + tc[2, 0]
        margin = 1e-6 * dist
        near = (np.minimum(np.abs(z1), np.abs(z1 - dist)) < margin) | (np.minimum(np.abs(z2), np.abs(z2 - dist)) < margin)
        # on an outlier the two triangulations are different least-squares problems, so they can disagree anywhere
        np.testing.assert_array_equal(mo[truth & ~near], (mc[:, 0] != 0)[truth & ~near])
        assert abs(int(mo[truth].sum()) - int((mc[truth] != 0).sum())) <= near.sum()
        assert (mo == (mc[:, 0] != 0)).mean() > 0.9
        if dist == 8.0:
            assert no < (truth.sum() if mask is not None else 500)


def test_recover_pose_zero_outputs():
    rng = np.random.default_rng(10)
    p1, p2, Eg, _, _, _ = two_view(rng, 50, 1.0)
    for E, K1 in ((np.zeros(9), K9), (Eg, np.r_[K9[:8], 2.0])):
        R, t, m, n = oe.recover_pose_pair(E, p1, p2, 50, K1, K9, None, 50.0)
        assert not R.any() and not t.any() and not m.any() and n == 0


# ------------------------------------------------------------------------------------------ ground truth
@pytest.mark.parametrize("ratio", [0.3, 0.5, 0.9])
def test_ransac_recovers_ground_truth(ratio):
    rng = np.random.default_rng(int(ratio * 10))
    n = 400
    p1, p2, Eg, R, t, truth = two_view(rng, n, ratio)
    iters = 1000 if ratio < 0.4 else 300
    E, mask, cnt = oe.find_essential_ransac_pair(p1, p2, n, K9, K9, 0, 1.0, iters, 0)
    c1, c2 = oe.calibrate(p1, K9), oe.calibrate(p2, K9)
    n_gt = oe.inliers(Eg[None], c1, c2, oe.pair_thr2(1.0, K9, K9))[0].sum()   # 0.5 px noise: not every match is within 1 px
    # no refit: the winner is a minimal model of 5 noisy matches (measured 0.87 - 0.90 of n_gt at ratios 0.3 / 0.5)
    assert cnt == mask.sum() and cnt >= 0.8 * n_gt and mask[~truth].mean() < 0.05
    Ro, to, mo, no = oe.recover_pose_pair(E, p1, p2, n, K9, K9, mask, 50.0)
    rot_err = np.degrees(np.arccos(np.clip((np.trace(Ro.reshape(3, 3).T @ R) - 1) / 2, -1, 1)))
    t_err = np.degrees(np.arccos(np.clip(to @ t, -1, 1)))
    assert rot_err < 2.0 and t_err < 5.0 and no >= 0.95 * cnt      # degrees; measured up to 0.79 and 2.1


def test_invalid_k_and_small_counts_give_no_model():
    rng = np.random.default_rng(11)
    p1, p2, _, _, _, _ = two_view(rng, 50, 1.0)
    for K1 in (np.r_[K9[:8], 2.0], np.r_[0.0, K9[1:]], np.r_[K9[:4], np.inf, K9[5:]], np.r_[K9[:6], 1e-3, K9[7:]]):
        assert not oe.k_valid(K1)
        E, m, c = oe.find_essential_ransac_pair(p1, p2, 50, K1, K9, 0, 1.0, 10, 0)
        assert c == 0 and not E.any() and not m.any()
    E, m, c = oe.find_essential_ransac_pair(p1, p2, 4, K9, K9, 0, 1.0, 10, 0)
    assert c == 0 and not E.any() and len(m) == 4
