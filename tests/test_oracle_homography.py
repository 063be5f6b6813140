"""RANSAC homography restatement (oracle/homography.py) on the CPU, anchored on exact arithmetic and on OpenCV.

The homography stage has no reference counterpart, so its semantics (include/balf_b200.h, balf_find_homography_ransac) are
defined by this project; these tests pin the restatement that tests/test_gpu_homography.py holds the kernels to."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import homography as oh

cv2 = pytest.importorskip("cv2")

W, H = 1200, 900
CORNERS = np.array([[0, 0], [W, 0], [W, H], [0, H]], np.float64)


def synth_matches(rng, n, ratio, sigma=0.5):
    """n matches in a W x H frame, a fraction `ratio` of them through a seeded ground-truth homography plus N(0, sigma)
    pixel noise, the rest uniform outliers, shuffled -> (p1, p2, H_gt, is_inlier)."""
    Hg = np.array([[1 + rng.uniform(-.1, .1), rng.uniform(-.1, .1), rng.uniform(-50, 50)],
                   [rng.uniform(-.1, .1), 1 + rng.uniform(-.1, .1), rng.uniform(-50, 50)],
                   [rng.uniform(-1e-4, 1e-4), rng.uniform(-1e-4, 1e-4), 1.0]])
    p1 = rng.uniform([0, 0], [W, H], (n, 2))
    q = np.c_[p1, np.ones(n)] @ Hg.T
    p2 = q[:, :2] / q[:, 2:]
    k = int(round(ratio * n))
    p2[:k] += rng.normal(0, sigma, (k, 2))
    p2[k:] = rng.uniform([0, 0], [W, H], (n - k, 2))
    perm = rng.permutation(n)
    return p1[perm], p2[perm], Hg, perm < k


def corner_error(Hm, Hg):
    """max distance between the frame corners mapped by Hm and by Hg (pixels)."""
    a, b = np.c_[CORNERS, np.ones(4)] @ np.asarray(Hm).reshape(3, 3).T, np.c_[CORNERS, np.ones(4)] @ Hg.T
    return np.abs(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:]).max()


def exact_homography(a, b):
    """The 4-point DLT (h33 = 1) solved in rational arithmetic: the exact homography of float inputs."""
    A = []
    for (x, y), (u, v) in zip(a, b):
        x, y, u, v = map(Fraction, (x, y, u, v))
        A.append([x, y, 1, 0, 0, 0, -x * u, -y * u, u])
        A.append([0, 0, 0, x, y, 1, -x * v, -y * v, v])
    for k in range(8):
        p = max(range(k, 8), key=lambda r: abs(A[r][k]))
        A[k], A[p] = A[p], A[k]
        for r in range(k + 1, 8):
            f = A[r][k] / A[k][k]
            A[r] = [A[r][c] - f * A[k][c] for c in range(9)]
    h = [Fraction(0)] * 8
    for k in range(7, -1, -1):
        h[k] = (A[k][8] - sum(A[k][c] * h[c] for c in range(k + 1, 8))) / A[k][k]
    return np.array([float(v) for v in h] + [1.0])


def quads(rng, n):
    """n non-degenerate 4-point sets: jittered, scaled frame corners, float32-representable (cv2 takes float32)."""
    q = CORNERS[None] * rng.uniform(0.1, 0.9, (n, 1, 1)) + rng.uniform(-100, 100, (n, 4, 2)) + 100
    return q.astype(np.float32).astype(np.float64)


def test_minimal_solver_vs_exact_and_cv2():
    rng = np.random.default_rng(1)
    q1, q2 = quads(rng, 120), quads(rng, 120)
    Hm, ok = oh.minimal_solve(q1, q2)
    assert ok.all()
    for i in range(len(q1)):
        ex = exact_homography(q1[i], q2[i])
        scale = np.abs(ex).max()
        assert np.abs(Hm[i] - ex).max() / scale <= 1e-12            # measured 1.0e-14
        hc = cv2.getPerspectiveTransform(q1[i].astype(np.float32), q2[i].astype(np.float32)).reshape(9)
        # cv2's own solve (unnormalised) is the less accurate side: against the exact solution the oracle is within 1e-14,
        # while the two differ by up to 2.4e-6 (median 2e-8) on these sets
        assert np.abs(Hm[i] - hc).max() / scale <= 5e-6


def test_minimal_solver_degenerate_samples():
    rng = np.random.default_rng(2)
    q = quads(rng, 3)
    line = np.stack([np.linspace(0, 100, 4), np.linspace(5, 305, 4)], 1)
    q1 = q.copy()
    q1[0] = line                                                    # collinear in the first image
    q1[1, 3] = q1[1, 0]                                             # a repeated point: three of the four collinear
    q2 = q.copy()
    q2[2, :3] = line[:3]                                            # three collinear in the second image only
    _, ok = oh.minimal_solve(q1, q2)
    assert not ok.any()
    same = np.repeat(q[:1, :1], 4, 1)                               # four identical points: no scale at all
    assert not oh.minimal_solve(same, same)[1].any()


def test_refit_noise_free_vs_cv2():
    rng = np.random.default_rng(3)
    p1, p2, Hg, _ = synth_matches(rng, 300, 1.0, sigma=0.0)
    G, ok = oh.refit(p1, p2, np.ones(300, np.uint8))
    assert ok
    G = G.reshape(3, 3)
    assert np.abs(G - Hg).max() / np.abs(Hg).max() <= 1e-11        # measured 1.0e-13
    Hc, _ = cv2.findHomography(p1, p2, 0)
    assert np.abs(G - Hc).max() / np.abs(Hg).max() <= 1e-5         # cv2's own error: measured 1.0e-6


@pytest.mark.parametrize("ratio", [0.2, 0.5, 0.9])
def test_ransac_recovers_ground_truth(ratio):
    rng = np.random.default_rng(int(ratio * 10))
    n = 500
    p1, p2, Hg, truth = synth_matches(rng, n, ratio)
    Hm, mask, cnt = oh.find_homography_ransac_pair(p1, p2, n, 0, 3.0, 2000, 0)
    # sigma = 0.5 px on 100 .. 450 inliers: measured corner errors 0.35 / 0.37 / 0.15 px (cv2.RANSAC: 0.35 / 0.38 / 0.14)
    assert corner_error(Hm, Hg) < 1.0
    assert cnt == mask.sum() and mask[truth].mean() > 0.99 and mask[~truth].mean() < 0.02


def test_sampler_deterministic_distinct_in_range():
    for n in (4, 5, 37, 16384):
        idx, ok = oh.sample_indices(7, 3, np.arange(500), n)
        idx2, ok2 = oh.sample_indices(7, 3, np.arange(500), n)
        np.testing.assert_array_equal(idx, idx2)
        np.testing.assert_array_equal(ok, ok2)
        assert ok.mean() > 0.99
        good = idx[ok]
        assert ((good >= 0) & (good < n)).all()
        assert all(len(set(r)) == 4 for r in good.tolist())
    assert not (oh.sample_indices(8, 3, np.arange(500), 37)[0] == oh.sample_indices(7, 3, np.arange(500), 37)[0]).all()


def test_sampler_hash_matches_python_integers():
    for seed, b, h in ((0, 0, 0), (1, 63, 1999), (2 ** 64 - 1, 5, 12345)):
        stream = oh.splitmix64(oh.splitmix64(seed) ^ ((b << 32) | h))
        first = []
        for c in range(oh.MAX_DRAWS):
            i = oh.splitmix64((stream + c) & oh.MASK64) % 1000
            if i not in first:
                first.append(i)
            if len(first) == 4:
                break
        idx, ok = oh.sample_indices(seed, b, np.array([h]), 1000)
        assert ok[0] and idx[0].tolist() == first
    assert oh.splitmix64(0) == 0xE220A8397B1DCDAF                   # the published first output of splitmix64 seeded 0
