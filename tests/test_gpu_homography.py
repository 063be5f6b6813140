"""RANSAC homography on the GPU (balf_b200/csrc/homography.cu through balf_find_homography_ransac, _capi and demo_match)
against the NumPy restatement (oracle/homography.py: bit for bit) and against cv2.findHomography(RANSAC) (accuracy)."""
import copy

import numpy as np
import pytest
import torch

from conftest import synth_u8
from oracle import homography as oh

pytestmark = pytest.mark.gpu

W, H = 1200, 900
CORNERS = np.array([[0, 0], [W, 0], [W, H], [0, H]], np.float64)


def dev():
    return torch.device("cuda:0")


def capi():
    import balf_b200._capi as c
    return c


def synth_matches(rng, n, ratio, sigma=0.5):
    """n matches in a W x H frame: a fraction `ratio` through a seeded ground-truth homography plus N(0, sigma) pixel
    noise, the rest uniform outliers, shuffled -> (p1, p2, H_gt)."""
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
    return p1[perm], p2[perm], Hg


def corner_error(Hm, Hg):
    a, b = np.c_[CORNERS, np.ones(4)] @ np.asarray(Hm).reshape(3, 3).T, np.c_[CORNERS, np.ones(4)] @ Hg.T
    return np.abs(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:]).max()


def batch(seed, counts, M):
    """padded batch [B,M,2] x 2 of synthetic pairs with the given counts; the padding is NaN (never read)."""
    rng = np.random.default_rng(seed)
    B = len(counts)
    p1, p2 = np.full((B, M, 2), np.nan), np.full((B, M, 2), np.nan)
    for b, n in enumerate(counts):
        a, c, _ = synth_matches(rng, n, rng.uniform(0.3, 0.9))
        p1[b, :n], p2[b, :n] = a, c
    return p1, p2, np.asarray(counts, np.int32)


def run_gpu(p1, p2, counts, thr, iters, seed):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    Hm, mask, n = capi().find_homography_ransac(t(p1), t(p2), t(counts), thr, iters, seed)
    return Hm.cpu().numpy(), mask.cpu().numpy(), n.cpu().numpy()


def mixed_counts(rng, B, M):
    special = [0, 3, 4, M, 5, 1]
    return special + rng.integers(5, 2500, B - len(special)).tolist()


# ------------------------------------------------------------------------------------------ GPU == oracle
@pytest.mark.parametrize("seed,iters,B,M", [(0, 200, 64, 16384), (1, 1, 16, 16384), (2, 2000, 4, 2048), (3, 500, 32, 3000)])
def test_gpu_matches_oracle_bit_for_bit(seed, iters, B, M):
    counts = mixed_counts(np.random.default_rng(100 + seed), B, M) if B >= 8 else [2048, 1500, 4, 700][:B]
    p1, p2, cnt = batch(seed, counts, M)
    for thr in (3.0, 1.5):
        Hg, mg, ng = run_gpu(p1, p2, cnt, thr, iters, seed)
        Ho, mo, no = oh.find_homography_ransac(p1, p2, cnt, thr, iters, seed)
        np.testing.assert_array_equal(ng, no)
        np.testing.assert_array_equal(mg, mo)
        np.testing.assert_array_equal(Hg, Ho)            # bit-identical: float64 without FMA on both sides, same order
        assert (ng[cnt < 4] == 0).all() and (Hg[cnt < 4] == 0).all()
        assert (mg.sum(1) == ng).all()


def test_counts_are_clamped_and_seed_changes_the_draws():
    p1, p2, cnt = batch(4, [300, 300], 300)
    a = run_gpu(p1, p2, np.array([-5, 10 ** 6], np.int32), 3.0, 300, 9)
    b = run_gpu(p1, p2, np.array([0, 300], np.int32), 3.0, 300, 9)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    s1 = run_gpu(p1, p2, cnt, 3.0, 50, 1)
    s2 = run_gpu(p1, p2, cnt, 3.0, 50, 2)
    np.testing.assert_array_equal(s1[0], oh.find_homography_ransac(p1, p2, cnt, 3.0, 50, 1)[0])
    assert not np.array_equal(s1[0], s2[0])


# ------------------------------------------------------------------------------------------ degenerate inputs
def test_degenerate_inputs():
    from balf_b200.demo import demo_match
    rng = np.random.default_rng(5)
    n = 400
    t = rng.uniform(0, 1000, n)
    line1 = np.stack([t, 0.5 * t + 20], 1)                         # every point on one line in the first image
    other = rng.uniform([0, 0], [W, H], (n, 2))
    same1, same2 = np.tile([[10.0, 20.0]], (n, 1)), np.tile([[30.0, 40.0]], (n, 1))   # every match the same point pair
    for a, b in ((line1, other), (other, line1), (same1, same2)):
        Hm, mask = demo_match.find_homography(a, b)
        assert Hm is None and mask.shape == (n, 1) and mask.dtype == np.uint8 and not mask.any()
    for k in (0, 1, 3):
        Hm, mask = demo_match.find_homography(other[:k], other[:k])
        assert Hm is None and mask.shape == (k, 1)
    # all outliers: a winner exists (a sample always fits its own points) but holds almost nothing; the result is the oracle's
    a, b = rng.uniform([0, 0], [W, H], (2048, 2)), rng.uniform([0, 0], [W, H], (2048, 2))
    Hg, mg, ng = run_gpu(a[None], b[None], np.array([2048], np.int32), 3.0, 2000, 0)
    Ho, mo, no = oh.find_homography_ransac(a[None], b[None], [2048], 3.0, 2000, 0)
    np.testing.assert_array_equal(Hg, Ho)
    np.testing.assert_array_equal(mg, mo)
    assert 4 <= ng[0] < 0.02 * 2048


def test_exhausted_draws_are_degenerate():
    """4 matches leave the sampler few distinct draws: with seeds 57, 2178 and 4543 hypothesis 0 of pair 0 has not found 4
    distinct indices after its 32 counters.  With iters = 1 that hypothesis is the only one, so the pair has no model; seed 58
    on the same points gives one."""
    p1, p2, _ = batch(6, [4], 4)
    cnt = np.array([4], np.int32)
    for seed in (57, 2178, 4543):
        assert not oh.sample_indices(seed, 0, np.array([0]), 4)[1][0]
        Hg, mg, ng = run_gpu(p1, p2, cnt, 3.0, 1, seed)
        assert ng[0] == 0 and not Hg.any() and not mg.any()
    assert oh.sample_indices(58, 0, np.array([0]), 4)[1][0]
    Hg, _, _ = run_gpu(p1, p2, cnt, 3.0, 1, 58)
    assert Hg[0, 2, 2] == 1.0
    # many hypotheses: some exhaust their draws (about 4e-4 of them), and the result is still the oracle's bit for bit
    _, ok = oh.sample_indices(57, 0, np.arange(20000), 4)
    assert (~ok).sum() >= 1
    Hg, mg, ng = run_gpu(p1, p2, cnt, 3.0, 20000, 57)
    Ho, mo, no = oh.find_homography_ransac(p1, p2, cnt, 3.0, 20000, 57)
    np.testing.assert_array_equal(Hg, Ho)
    np.testing.assert_array_equal(mg, mo)
    np.testing.assert_array_equal(ng, no)


# ------------------------------------------------------------------------------------------ against cv2
# Measured on these 48 pairs (B200): the corner error exceeds cv2's by at most 0.0126 px (mean 0.154 px against cv2's
# 0.169 px; cv2 refines with Levenberg-Marquardt, this library with least squares), and the inlier count is never below
# cv2's.  Margins: twice the corner gap, and 0.5 % of the matches.
CV2_CORNER_MARGIN = 0.025    # px
CV2_INLIER_MARGIN = 0.005    # fraction of the matches


@pytest.mark.parametrize("ratio", [0.3, 0.5, 0.9])
@pytest.mark.parametrize("n", [500, 2048])
def test_at_least_as_good_as_cv2(ratio, n):
    cv2 = pytest.importorskip("cv2")
    from balf_b200.demo import demo_match
    rng = np.random.default_rng(int(ratio * 100) + n)
    pairs, gts = [], []
    for _ in range(8):
        a, b, Hg = synth_matches(rng, n, ratio)
        pairs.append((a, b))
        gts.append(Hg)
    got = demo_match.find_homography_batch(pairs, 3.0, 2000, 0)
    for (a, b), Hg, (Hm, mask) in zip(pairs, gts, got):
        Hc, mc = cv2.findHomography(a, b, cv2.RANSAC, 3.0, maxIters=2000)
        assert Hm is not None and mask.shape == (n, 1)
        assert corner_error(Hm, Hg) <= corner_error(Hc, Hg) + CV2_CORNER_MARGIN
        assert mask.sum() >= mc.sum() - CV2_INLIER_MARGIN * n
    # a single pair is pair 0 of a batch of one: the same draws as pair 0 of the batch
    np.testing.assert_array_equal(demo_match.find_homography(*pairs[0])[0], got[0][0])


# ------------------------------------------------------------------------------------------ end to end
E2E_DX, E2E_DY = 128, 64
# B200, seed-0 random-init weights: ~800 SMNN matches, inlier fraction 0.89 and corner error 0.013 px (0.005 - 0.031 px
# and 0.88 - 0.90 over three seeds / offsets); bounds with margin
E2E_CORNER_BOUND = 0.1       # px
E2E_INLIER_FLOOR = 0.75


def test_extract_matches_then_find_homography(detector):
    """Two 900x1200 crops of one seeded noise image, the second offset by (128, 64) px: multiples of 64 keep the
    detector's 8x8 blocks aligned.  The weights are the random-init ones, so how many keypoints repeat is not known in
    advance: the bounds come from the B200 run with a margin."""
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
    Hm, mask = demo_match.find_homography(p1, p2)
    Ht = np.array([[1, 0, -E2E_DX], [0, 1, -E2E_DY], [0, 0, 1]], np.float64)
    assert Hm is not None and mask.shape == (len(p1), 1)
    err, frac = corner_error(Hm, Ht), mask.mean()
    print("e2e: %d matches, inlier fraction %.4f, corner error %.4f px" % (len(p1), frac, err))
    assert err < E2E_CORNER_BOUND
    assert frac > E2E_INLIER_FLOOR


# ------------------------------------------------------------------------------------------ argument errors
def test_argument_errors():
    c = capi()
    t = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev())
    p, cnt = t(2, 10, 2), torch.full((2,), 10, dtype=torch.int32, device=dev())
    out_h, out_m, out_n = t(2, 9), torch.zeros(2, 10, dtype=torch.uint8, device=dev()), torch.zeros(2, dtype=torch.int32,
                                                                                                      device=dev())
    ws_bytes = c._homog_ws(2, 10, 100)
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev())
    raw = lambda M, thr, iters, nbytes: c._homog_ransac(c._ptr(p), c._ptr(p), c._ptr(cnt), 2, M, thr, iters, 0, c._ptr(out_h),
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
            c.find_homography_ransac(p, p, cnt, thr, iters, 0)
    with pytest.raises(ValueError, match="M = 16385"):
        c.find_homography_ransac(t(1, 16385, 2), t(1, 16385, 2), cnt[:1], 3.0, 10, 0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        c.find_homography_ransac(p.cpu(), p.cpu(), cnt.cpu(), 3.0, 10, 0)
