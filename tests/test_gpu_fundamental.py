"""RANSAC fundamental matrix on the GPU (balf_b200/csrc/fundamental.cu through balf_find_fundamental_ransac, _capi and
demo_match) against the NumPy restatement (oracle/fundamental.py: bit for bit) and against cv2.findFundamentalMat(FM_RANSAC)
(accuracy)."""
import copy

import numpy as np
import pytest
import torch

from conftest import synth_u8
from oracle import fundamental as of

pytestmark = pytest.mark.gpu

W, H = 1200, 900
K = np.array([[800.0, 0, W / 2], [0, 800.0, H / 2], [0, 0, 1]])


def dev():
    return torch.device("cuda:0")


def capi():
    import balf_b200._capi as c
    return c


def rot(v):
    a = np.linalg.norm(v)
    k = v / a
    S = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(a) * S + (1 - np.cos(a)) * S @ S


def two_view(rng, n, ratio, sigma=0.5):
    """n matches of a seeded two-view scene: random 3-D points 4 - 10 units in front of camera 1, camera 2 rotated by up to
    0.1 rad and translated by about one unit; a fraction `ratio` of the matches with N(0, sigma) pixel noise, the rest
    uniform outliers, shuffled -> (p1, p2, F_gt, noise-free p2, is_inlier)."""
    X = np.c_[rng.uniform(-3, 3, (n, 2)), rng.uniform(4, 10, n)]
    R = rot(rng.uniform(-0.1, 0.1, 3))
    t = np.array([1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)])
    a = X @ K.T
    b = (X @ R.T + t) @ K.T
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
    """the larger of the two point-to-epipolar-line distances of each match (pixels)."""
    F = np.asarray(F).reshape(3, 3)
    x1, x2 = np.c_[p1, np.ones(len(p1))], np.c_[p2, np.ones(len(p2))]
    l2, l1 = x1 @ F.T, x2 @ F
    s = np.abs((x2 * l2).sum(1))
    return np.maximum(s / np.hypot(l2[:, 0], l2[:, 1]), s / np.hypot(l1[:, 0], l1[:, 1]))


def batch(seed, counts, M):
    """padded batch [B,M,2] x 2 of two-view pairs with the given counts; the padding is NaN (never read)."""
    rng = np.random.default_rng(seed)
    B = len(counts)
    p1, p2 = np.full((B, M, 2), np.nan), np.full((B, M, 2), np.nan)
    for b, n in enumerate(counts):
        a, c, _, _, _ = two_view(rng, n, rng.uniform(0.3, 0.9))
        p1[b, :n], p2[b, :n] = a, c
    return p1, p2, np.asarray(counts, np.int32)


def run_gpu(p1, p2, counts, thr, iters, seed):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    F, mask, n = capi().find_fundamental_ransac(t(p1), t(p2), t(counts), thr, iters, seed)
    return F.cpu().numpy(), mask.cpu().numpy(), n.cpu().numpy()


def assert_oracle(p1, p2, cnt, thr, iters, seed):
    Fg, mg, ng = run_gpu(p1, p2, cnt, thr, iters, seed)
    Fo, mo, no = of.find_fundamental_ransac(p1, p2, cnt, thr, iters, seed)
    np.testing.assert_array_equal(ng, no)
    np.testing.assert_array_equal(mg, mo)
    np.testing.assert_array_equal(Fg, Fo)                # bit-identical: float64 without FMA on both sides, same order
    return Fg, mg, ng


# ------------------------------------------------------------------------------------------ GPU == oracle
@pytest.mark.parametrize("seed,iters,B,M", [(0, 100, 64, 16384), (1, 1, 16, 16384), (2, 1000, 4, 2048)])
def test_gpu_matches_oracle_bit_for_bit(seed, iters, B, M):
    if B >= 8:
        counts = [0, 6, 7, 8, M, 5, 1] + np.random.default_rng(100 + seed).integers(9, 2500, B - 7).tolist()
    else:
        counts = [2048, 1500, 7, 700][:B]
    p1, p2, cnt = batch(seed, counts, M)
    for thr in (3.0, 1.0):
        Fg, mg, ng = assert_oracle(p1, p2, cnt, thr, iters, seed)
        assert (ng[cnt < 7] == 0).all() and (Fg[cnt < 7] == 0).all()
        assert (mg.sum(1) == ng).all()
        found = Fg.reshape(B, 9).any(1)
        assert found[cnt >= 8].mean() > 0.9
        np.testing.assert_allclose(np.linalg.norm(Fg[found].reshape(-1, 9), axis=1), 1.0, rtol=1e-14)


def test_counts_are_clamped_and_seed_changes_the_draws():
    p1, p2, cnt = batch(4, [300, 300], 300)
    a = run_gpu(p1, p2, np.array([-5, 10 ** 6], np.int32), 3.0, 300, 9)
    b = run_gpu(p1, p2, np.array([0, 300], np.int32), 3.0, 300, 9)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    s1 = run_gpu(p1, p2, cnt, 3.0, 50, 1)
    s2 = run_gpu(p1, p2, cnt, 3.0, 50, 2)
    np.testing.assert_array_equal(s1[0], of.find_fundamental_ransac(p1, p2, cnt, 3.0, 50, 1)[0])
    assert not np.array_equal(s1[0], s2[0])


# ------------------------------------------------------------------------------------------ degenerate inputs
def test_degenerate_inputs():
    """Points on a horizontal (or vertical) line keep one normalised coordinate exactly 0, so three columns of the 7x9
    system are zero and the elimination meets a zero pivot; identical points have no scale (a NaN pivot)."""
    from balf_b200.demo import demo_match
    rng = np.random.default_rng(5)
    n = 400
    t = rng.uniform(0, 1000, n)
    hline, vline = np.stack([t, np.full(n, 300.0)], 1), np.stack([np.full(n, 250.0), t], 1)
    other = rng.uniform([0, 0], [W, H], (n, 2))
    same1, same2 = np.tile([[10.0, 20.0]], (n, 1)), np.tile([[30.0, 40.0]], (n, 1))
    for a, b in ((hline, other), (other, vline), (same1, same2)):
        F, mask = demo_match.find_fundamental(a, b)
        assert F is None and mask.shape == (n, 1) and mask.dtype == np.uint8 and not mask.any()
    for k in (0, 1, 6):
        F, mask = demo_match.find_fundamental(other[:k], other[:k])
        assert F is None and mask.shape == (k, 1)


def test_exhausted_draws():
    """7 matches: with seeds 3662, 9896 and 12452 hypothesis 0 of pair 0 has not found 7 distinct indices after its 64
    counters, so with iters = 1 the pair has no model; with many hypotheses some exhaust their draws (about 2.5e-4 of
    them) and the result is still the oracle's bit for bit."""
    p1, p2, _ = batch(6, [7], 7)
    cnt = np.array([7], np.int32)
    for seed in (3662, 9896, 12452):
        assert not of.sample_indices(seed, 0, np.array([0]), 7)[1][0]
        F, m, n = run_gpu(p1, p2, cnt, 3.0, 1, seed)
        assert n[0] == 0 and not F.any() and not m.any()
    assert (~of.sample_indices(0, 0, np.arange(20000), 7)[1]).sum() >= 1
    assert_oracle(p1, p2, cnt, 3.0, 20000, 0)


@pytest.mark.parametrize("n", [7, 8])
def test_small_counts(n):
    """Noise-free matches.  7: every sample is the whole set, so the winner fits all 7 and no refit runs; 8: the 8-point
    refit runs on all of them."""
    rng = np.random.default_rng(n)
    a, b, _, _, _ = two_view(rng, n, 1.0, sigma=0.0)
    F, m, cnt = assert_oracle(a[None], b[None], np.array([n], np.int32), 3.0, 200, 0)
    assert cnt[0] == n and m.all()
    s = np.linalg.svd(F[0], compute_uv=False)
    assert s[2] / s[0] < 1e-9
    assert epipolar_error(F[0], a, b).max() <= 3.0


# ------------------------------------------------------------------------------------------ against cv2
# Measured on these 32 pairs (B200): the mean epipolar distance of the noise-free true correspondences is below cv2's on
# every pair (by 0.14 - 0.51 px at the worst pair of each ratio, 0.62 - 0.82 px on average; cv2 keeps its 7- or 8-point
# model, this library refits on all inliers), and the inlier count is at most 3 of 1000 below cv2's (ratio 0.7).
# Margins: 0.05 px, and twice the inlier gap.
CV2_DIST_MARGIN = 0.05       # px
CV2_INLIER_MARGIN = 0.006    # fraction of the matches


@pytest.mark.parametrize("ratio,iters", [(0.3, 32768), (0.5, 1000), (0.7, 1000), (0.9, 1000)])
def test_at_least_as_good_as_cv2(ratio, iters):
    cv2 = pytest.importorskip("cv2")
    from balf_b200.demo import demo_match
    n = 1000
    rng = np.random.default_rng(int(ratio * 100))
    scenes = [two_view(rng, n, ratio) for _ in range(8)]
    got = demo_match.find_fundamental_batch([(s[0], s[1]) for s in scenes], 3.0, iters, 0)
    gaps, dinl = [], []
    for (a, b, _, clean, truth), (F, mask) in zip(scenes, got):
        Fc, mc = cv2.findFundamentalMat(a, b, cv2.FM_RANSAC, 3.0, 0.99, iters)
        assert F is not None and mask.shape == (n, 1) and Fc is not None
        dg = epipolar_error(F, a[truth], clean[truth]).mean()
        dc = epipolar_error(Fc, a[truth], clean[truth]).mean()
        gaps.append(dg - dc)
        dinl.append(int(mask.sum()) - int(mc.sum()))
    print("ratio %.1f: epipolar distance gap to cv2 max %.4f mean %.4f px, inlier gap min %d" %
          (ratio, max(gaps), np.mean(gaps), min(dinl)))
    assert max(gaps) <= CV2_DIST_MARGIN
    assert min(dinl) >= -CV2_INLIER_MARGIN * n
    np.testing.assert_array_equal(demo_match.find_fundamental(scenes[0][0], scenes[0][1], 3.0, iters)[0], got[0][0])


# ------------------------------------------------------------------------------------------ end to end
E2E_DX, E2E_DY = 128, 64
# B200, seed-0 random-init weights: 802 SMNN matches, 712 of them within 1 px of the offset, inlier fraction 0.893, every
# match that follows the offset an inlier, sigma3 / sigma1 = 9e-18; floor with margin
E2E_INLIER_FLOOR = 0.75


def test_extract_matches_then_find_fundamental(detector):
    """The homography test's two offset crops of one noise image.  The scene is planar, so the epipolar geometry is not
    determined: this checks the pipeline (F found, rank 2, the matches that follow the offset are inliers), not F."""
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    from balf_b200.third_party.hardnet.hardnet_pytorch import HardNet
    big = synth_u8(H + E2E_DY, W + E2E_DX, 31)
    rgb1 = np.ascontiguousarray(big[:H, :W])
    rgb2 = np.ascontiguousarray(big[E2E_DY:, E2E_DX:])
    torch.manual_seed(0)
    hn = HardNet().eval().to(dev())
    det = copy.deepcopy(detector).to(dev())
    args = config.default_test_args()
    p1, p2 = demo_match.extract_matches(args, rgb1, rgb1[..., 0].copy(), rgb2, rgb2[..., 0].copy(), det, hn, dev())
    F, mask = demo_match.find_fundamental(p1, p2)
    assert F is not None and mask.shape == (len(p1), 1)
    s = np.linalg.svd(F, compute_uv=False)
    good = np.abs(p1 - p2 - [E2E_DX, E2E_DY]).max(1) < 1.0
    frac, good_in = mask.mean(), mask[good, 0].mean()
    print("e2e: %d matches, %d follow the offset, inlier fraction %.4f, of those following %.4f, sigma3/sigma1 %.2e" %
          (len(p1), good.sum(), frac, good_in, s[2] / s[0]))
    assert s[2] / s[0] < 1e-9
    assert frac > E2E_INLIER_FLOOR
    assert good.sum() > 0.5 * len(p1) and good_in > 0.99


# ------------------------------------------------------------------------------------------ argument errors
def test_argument_errors():
    c = capi()
    t = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev())
    p, cnt = t(2, 10, 2), torch.full((2,), 10, dtype=torch.int32, device=dev())
    out_f, out_m, out_n = t(2, 9), torch.zeros(2, 10, dtype=torch.uint8, device=dev()), torch.zeros(2, dtype=torch.int32,
                                                                                                      device=dev())
    ws_bytes = c._fund_ws(2, 10, 100)
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev())
    raw = lambda M, thr, iters, nbytes: c._fund_ransac(c._ptr(p), c._ptr(p), c._ptr(cnt), 2, M, thr, iters, 0, c._ptr(out_f),
                                                       c._ptr(out_m), c._ptr(out_n), c._ptr(ws), nbytes, c._stream(dev()))
    assert raw(10, 3.0, 100, ws_bytes) == 0
    torch.cuda.synchronize()
    for args, what in (((10, 0.0, 100, ws_bytes), "thr"), ((10, -1.0, 100, ws_bytes), "thr"),
                       ((10, float("nan"), 100, ws_bytes), "thr"), ((10, 3.0, 0, ws_bytes), "iters"),
                       ((10, 3.0, (1 << 17) + 1, ws_bytes), "iters"), ((16385, 3.0, 100, ws_bytes), "M = 16385"),
                       ((10, 3.0, 100, ws_bytes - 1), "workspace")):
        assert raw(*args) < 0
        assert what in c._last_error().decode()
    for thr, iters, what in ((0.0, 100, "thr"), (3.0, 0, "iters")):
        with pytest.raises(ValueError, match=what):
            c.find_fundamental_ransac(p, p, cnt, thr, iters, 0)
    with pytest.raises(ValueError, match="M = 16385"):
        c.find_fundamental_ransac(t(1, 16385, 2), t(1, 16385, 2), cnt[:1], 3.0, 10, 0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        c.find_fundamental_ransac(p.cpu(), p.cpu(), cnt.cpu(), 3.0, 10, 0)
