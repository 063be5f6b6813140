"""RANSAC fundamental-matrix restatement (oracle/fundamental.py) on the CPU, anchored on NumPy and on OpenCV.

The fundamental-matrix stage has no reference counterpart, so its semantics (include/balf_b200.h,
balf_find_fundamental_ransac) are defined by this project; these tests pin the restatement that
tests/test_gpu_fundamental.py holds the kernels to."""
import numpy as np
import pytest

from oracle import fundamental as of
from oracle import homography as oh

cv2 = pytest.importorskip("cv2")

W, H = 1200, 900
K = np.array([[800.0, 0, W / 2], [0, 800.0, H / 2], [0, 0, 1]])


def rot(v):
    a = np.linalg.norm(v)
    k = v / a
    S = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(a) * S + (1 - np.cos(a)) * S @ S


def two_view(rng, n, ratio, sigma=0.5):
    """n matches of a seeded two-view scene (random 3-D points 4 - 10 units in front of camera 1, camera 2 rotated by up to
    0.1 rad and translated by about one unit), a fraction `ratio` with N(0, sigma) pixel noise, the rest uniform outliers,
    shuffled -> (p1, p2, F_gt with unit norm, noise-free p2, is_inlier)."""
    X = np.c_[rng.uniform(-3, 3, (n, 2)), rng.uniform(4, 10, n)]
    R = rot(rng.uniform(-0.1, 0.1, 3))
    t = np.array([1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)])
    a, b = X @ K.T, (X @ R.T + t) @ K.T
    p1, c2 = a[:, :2] / a[:, 2:], b[:, :2] / b[:, 2:]
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    Ki = np.linalg.inv(K)
    Fg = Ki.T @ tx @ R @ Ki
    k = int(round(ratio * n))
    p2 = c2.copy()
    p2[:k] += rng.normal(0, sigma, (k, 2))
    p2[k:] = rng.uniform([0, 0], [W, H], (n - k, 2))
    perm = rng.permutation(n)
    return p1[perm], p2[perm], Fg / np.linalg.norm(Fg), c2[perm], perm < k


def epipolar_error(F, p1, p2):
    """cv2's FM_RANSAC error, transcribed: the larger of the two squared point-to-epipolar-line distances."""
    F = np.asarray(F, np.float64).reshape(3, 3)
    out = np.empty(len(p1))
    for i, ((x1, y1), (x2, y2)) in enumerate(zip(p1, p2)):
        a, b, c = F[0, 0] * x1 + F[0, 1] * y1 + F[0, 2], F[1, 0] * x1 + F[1, 1] * y1 + F[1, 2], F[2, 0] * x1 + F[2, 1] * y1 + F[2, 2]
        a2, b2 = F[0, 0] * x2 + F[1, 0] * y2 + F[2, 0], F[0, 1] * x2 + F[1, 1] * y2 + F[2, 1]
        s2 = 1.0 / (a * a + b * b)
        s1 = 1.0 / (a2 * a2 + b2 * b2)
        d = x2 * a + y2 * b + c
        out[i] = max(d * d * s1, d * d * s2)
    return out


def unit(F):
    """cv2's scaling (F[2,2] = 1 where it can) -> the library's: unit Frobenius norm, first largest-magnitude entry > 0."""
    f = np.asarray(F, np.float64).reshape(-1)
    f = f / np.linalg.norm(f)
    return f * np.sign(f[np.argmax(np.abs(f))])


# ------------------------------------------------------------------------------------------ sampler
def test_sampler_seven_distinct_and_shared_with_homography():
    for n in (7, 8, 50, 16384):
        idx, ok = of.sample_indices(11, 2, np.arange(2000), n)
        good = idx[ok]
        assert ((good >= 0) & (good < n)).all()
        assert all(len(set(r)) == 7 for r in good.tolist())
        assert ok.mean() > 0.999
    # one sampler: 4 of n with 32 draws is the homography's
    for n in (4, 37):
        a, oka = of.sample_indices(3, 5, np.arange(3000), n, k=4, draws=32)
        b, okb = oh.sample_indices(3, 5, np.arange(3000), n)
        np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(oka, okb)


def test_sampler_n7_exhausts_its_draws():
    """7 of 7: about 5 % of the hypotheses do not find all 7 within 32 counters, about 2.5e-4 within 64."""
    _, ok32 = of.sample_indices(0, 0, np.arange(20000), 7, draws=32)
    _, ok64 = of.sample_indices(0, 0, np.arange(20000), 7)
    assert 0.03 < (~ok32).mean() < 0.07
    assert 0 < (~ok64).sum() < 20
    for seed in (3662, 9896, 12452):
        assert not of.sample_indices(seed, 0, np.array([0]), 7)[1][0]
    assert of.sample_indices(3663, 0, np.array([0]), 7)[1][0]


# ------------------------------------------------------------------------------------------ Jacobi
def test_jacobi_vs_eigh():
    rng = np.random.default_rng(1)
    for trial in range(20):
        a, b, _, _, _ = two_view(rng, 50, 1.0, sigma=0.5 if trial % 2 else 0.0)
        u1, v1, _, _, _ = of._normalise(a[None, :, 0], a[None, :, 1])
        u2, v2, _, _, _ = of._normalise(b[None, :, 0], b[None, :, 1])
        r = of.epipolar_rows(u1[0], v1[0], u2[0], v2[0])
        A = r.T @ r                                                 # the refit's 9x9 normal matrix
        f = np.array(of.smallest_eigvec(A))
        w, V = np.linalg.eigh(A)
        assert abs(abs(f @ V[:, 0]) - 1) < 1e-9
        assert np.linalg.norm(A @ f) <= w[0] + 1e-12 * w[-1]
        vals, _ = of.jacobi_eigh([list(map(float, row)) for row in A])
        np.testing.assert_allclose(np.sort(vals), w, rtol=0, atol=1e-12 * w[-1])
        F = f.reshape(3, 3)                                         # and the 3x3 F^T F of the rank-2 step
        M = F.T @ F
        v3 = np.array(of.smallest_eigvec(M))
        w3, V3 = np.linalg.eigh(M)
        assert abs(abs(v3 @ V3[:, 0]) - 1) < 1e-9
        G = of.rank2(f).reshape(3, 3)
        s = np.linalg.svd(G, compute_uv=False)
        assert s[2] / s[0] < 1e-14
        np.testing.assert_allclose(s[:2], np.linalg.svd(F, compute_uv=False)[:2], rtol=1e-12)


# ------------------------------------------------------------------------------------------ cubic roots
def real_roots(c):
    r = np.roots(c[::-1])
    return np.sort(r[np.abs(r.imag) <= 1e-7 * np.maximum(1, np.abs(r))].real)


@pytest.mark.parametrize("roots,tol", [
    ((-2.0, 0.5, 3.0), 1e-13), ((1e-3, 2.0, -7.5), 1e-13), ((0.25, 0.25, 4.0), 2e-8), ((1.0, 1.0, 1.0), 1e-5),
    ((-1.0, 1.0 + 1e-9, 1.0), 2e-8), ((0.0, 5.0, -5.0), 1e-13)])
def test_cubic_roots_vs_np_roots(roots, tol):
    c = np.poly(roots)[::-1].copy()                                # c0 .. c3
    got, cnt = of.cubic_roots(c[None] * 0.37)
    got = got[0, :cnt[0]]
    assert 1 <= cnt[0] <= 3
    for x in got:                                                   # every root found is a root
        assert np.min(np.abs(np.array(roots) - x)) <= tol * max(1, abs(x))
    for x in real_roots(c):                                         # every simple real root of np.roots is found
        if np.sum(np.abs(np.array(roots) - x) < 1e-4) == 1:
            assert np.min(np.abs(got - x)) <= tol * max(1, abs(x))


def test_cubic_roots_random_and_degree_drop():
    rng = np.random.default_rng(2)
    c = rng.normal(size=(2000, 4))
    got, cnt = of.cubic_roots(c)
    for i in range(len(c)):
        want = real_roots(c[i])
        assert cnt[i] == len(want)
        np.testing.assert_allclose(got[i, :cnt[i]], want, rtol=1e-9, atol=1e-9)
    # leading coefficient zero: the quadratic's roots; tiny: those plus one near -c2 / c3
    q = np.array([[-6.0, 1.0, 1.0, 0.0], [2.0, -3.0, 1.0, 0.0], [-6.0, 1.0, 1.0, 1e-12], [2.0, -3.0, 1.0, -1e-9]])
    got, cnt = of.cubic_roots(q)
    np.testing.assert_allclose(got[0, :2], [-3.0, 2.0], rtol=1e-14)
    np.testing.assert_allclose(got[1, :2], [1.0, 2.0], rtol=1e-14)
    assert cnt[0] == cnt[1] == 2 and cnt[2] == cnt[3] == 3
    for i in (2, 3):
        np.testing.assert_allclose(got[i, :cnt[i]], real_roots(q[i]), rtol=1e-9)
    got, cnt = of.cubic_roots(np.array([[1.0, 0.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0], [np.nan, 1.0, 1.0, 1.0]]))
    assert (cnt == 0).all()


# ------------------------------------------------------------------------------------------ minimal solver
def test_minimal_solver_vs_cv2_7point():
    rng = np.random.default_rng(3)
    count_eq = 0
    diffs = []
    for trial in range(300):
        geometric = trial % 3 != 0
        if geometric:
            a, b, _, _, _ = two_view(rng, 7, 1.0, sigma=0.0)
        else:
            a, b = rng.uniform([0, 0], [W, H], (7, 2)), rng.uniform([0, 0], [W, H], (7, 2))
        F, ok = of.minimal_solve(a[None], b[None])
        Fc, _ = cv2.findFundamentalMat(a, b, cv2.FM_7POINT)
        nc = 0 if Fc is None else len(Fc) // 3
        if ok[0].sum() == nc:
            count_eq += 1
        else:                                                       # then np.roots agrees with the count of this cubic
            u1, v1, _, _, _ = of._normalise(a[None, :, 0], a[None, :, 1])
            u2, v2, _, _, _ = of._normalise(b[None, :, 0], b[None, :, 1])
            F1, F2, _ = of.null_space(of.epipolar_rows(u1, v1, u2, v2))
            assert ok[0].sum() == len(real_roots(of.cubic_coeffs(F1, F2)[0]))
        for m in np.where(ok[0])[0]:
            G = F[0, m].reshape(3, 3)
            s = np.linalg.svd(G, compute_uv=False)
            assert s[2] / s[0] < 1e-9                               # rank 2
            assert np.sqrt(epipolar_error(G, a, b)).max() < 1e-6    # fits its own 7 points (pixels)
            if geometric and ok[0].sum() == nc:
                diffs.append(min(np.abs(F[0, m] - unit(Fc[3 * j:3 * j + 3])).max() for j in range(nc)))
    # measured: 299 of 300 equal; in the other (geometric) sample the cubic has three real roots, two of them 0.0213 and
    # 0.0215, np.roots finds all three and cv2 returns one
    assert count_eq >= 298
    # measured over the 531 solutions of the geometric samples with equal counts: median 4.0e-8, max 5.3e-4 (the largest on
    # ill-conditioned samples)
    assert np.median(diffs) < 1e-7 and max(diffs) < 1e-3


def test_minimal_solver_degenerate_samples():
    rng = np.random.default_rng(4)
    a, b, _, _, _ = two_view(rng, 7, 1.0)
    same = np.tile(a[:1], (7, 1))
    hline = np.c_[np.linspace(0, 900, 7), np.full(7, 100.0)]
    _, ok = of.minimal_solve(np.stack([same, hline, a]), np.stack([b, b, hline]))
    assert not ok.any()


# ------------------------------------------------------------------------------------------ refit
@pytest.mark.parametrize("sigma", [0.0, 0.5])
def test_refit_vs_cv2_8point(sigma):
    rng = np.random.default_rng(5)
    a, b, Fg, _, _ = two_view(rng, 400, 1.0, sigma=sigma)
    F, ok = of.refit(a, b, np.ones(400, np.uint8))
    assert ok
    s = np.linalg.svd(F.reshape(3, 3), compute_uv=False)
    assert s[2] / s[0] < 1e-14 and abs(np.linalg.norm(F) - 1) < 1e-15
    Fc, _ = cv2.findFundamentalMat(a, b, cv2.FM_8POINT)
    d = np.abs(F - unit(Fc)).max()
    if sigma == 0:
        assert np.abs(F - unit(Fg)).max() < 1e-10 and d < 1e-7
    else:
        assert d < 1e-6                                             # both the normalised 8-point fit


# ------------------------------------------------------------------------------------------ inlier rule
def test_inlier_rule_vs_cv2_error():
    rng = np.random.default_rng(6)
    a, b, Fg, _, truth = two_view(rng, 3000, 0.6, sigma=2.0)
    F = np.stack([unit(Fg), of.refit(a[truth][:50], b[truth][:50], np.ones(50, np.uint8))[0]])
    for thr in (1.0, 3.0):
        got = of.inliers(F, a, b, thr)
        for i in range(2):
            err = epipolar_error(F[i], a, b)
            want = err <= thr * thr
            close = np.abs(err - thr * thr) < 1e-9 * thr * thr     # rounding can only differ at the threshold itself
            assert (got[i] == want)[~close].all() and got[i].sum() > 100
    zero = np.zeros((1, 9))
    assert not of.inliers(zero, a, b, 3.0).any()                    # lines with a^2 + b^2 = 0 are never inliers


# ------------------------------------------------------------------------------------------ ground truth
@pytest.mark.parametrize("ratio", [0.3, 0.5, 0.9])
def test_ransac_recovers_ground_truth(ratio):
    rng = np.random.default_rng(int(ratio * 10))
    n = 600
    a, b, Fg, clean, truth = two_view(rng, n, ratio)
    iters = 20000 if ratio < 0.4 else 1000
    F, mask, cnt = of.find_fundamental_ransac_pair(a, b, n, 0, 3.0, iters, 0)
    d = np.sqrt(epipolar_error(F, a[truth], clean[truth]))
    assert cnt == mask.sum() and mask[truth].mean() > 0.97 and mask[~truth].mean() < 0.1
    assert d.mean() < 0.5                                           # pixels, against the noise-free correspondences
