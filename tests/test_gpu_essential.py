"""RANSAC essential matrix and relative pose on the GPU (balf_b200/csrc/essential.cu through balf_find_essential_ransac /
balf_recover_pose, _capi and demo_match) against the NumPy restatement (oracle/essential.py: bit for bit) and against
cv2.findEssentialMat + cv2.recoverPose (accuracy)."""
import copy

import numpy as np
import pytest
import torch

from conftest import synth_u8
from oracle import essential as oe
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


def two_view(rng, n, ratio, sigma=0.5, K1=K, K2=K):
    """test_gpu_fundamental's seeded two-view scene with known cameras (3-D points 4 - 10 units in front of camera 1,
    camera 2 rotated by up to 0.1 rad and translated by about one unit; a fraction `ratio` with N(0, sigma) pixel noise,
    the rest uniform outliers, shuffled) -> (p1, p2, R, t (unit), is_inlier)."""
    X = np.c_[rng.uniform(-3, 3, (n, 2)), rng.uniform(4, 10, n)]
    R = rot(rng.uniform(-0.1, 0.1, 3))
    t = np.array([1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)])
    a, b = X @ K1.T, (X @ R.T + t) @ K2.T
    p1, p2 = a[:, :2] / a[:, 2:], b[:, :2] / b[:, 2:]
    k = int(round(ratio * n))
    p2[:k] += rng.normal(0, sigma, (k, 2))
    p2[k:] = rng.uniform([0, 0], [W, H], (n - k, 2))
    perm = rng.permutation(n)
    return p1[perm], p2[perm], R, t / np.linalg.norm(t), perm < k


def random_k(rng, skew=False):
    f = rng.uniform(600, 1100)
    return np.array([[f * rng.uniform(0.95, 1.05), rng.uniform(-2, 2) if skew else 0.0, rng.uniform(560, 640)],
                     [0, f, rng.uniform(420, 480)], [0, 0, 1]])


def batch(seed, counts, M):
    """padded batch [B,M,2] x 2 of two-view pairs with the given counts (the padding is NaN, never read) and K [B,2,3,3]:
    pair b has K1 != K2, every third pair a K with skew."""
    rng = np.random.default_rng(seed)
    B = len(counts)
    p1, p2 = np.full((B, M, 2), np.nan), np.full((B, M, 2), np.nan)
    Ks = np.zeros((B, 2, 3, 3))
    for b, n in enumerate(counts):
        Ks[b] = random_k(rng, b % 3 == 0), random_k(rng)
        a, c, _, _, _ = two_view(rng, n, rng.uniform(0.3, 0.9), K1=Ks[b, 0], K2=Ks[b, 1])
        p1[b, :n], p2[b, :n] = a, c
    return p1, p2, np.asarray(counts, np.int32), Ks


def t_(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def run_gpu(p1, p2, counts, Ks, thr, iters, seed):
    E, mask, n = capi().find_essential_ransac(t_(p1), t_(p2), t_(counts), t_(Ks), thr, iters, seed)
    return E.cpu().numpy(), mask.cpu().numpy(), n.cpu().numpy()


def assert_oracle(p1, p2, cnt, Ks, thr, iters, seed):
    Eg, mg, ng = run_gpu(p1, p2, cnt, Ks, thr, iters, seed)
    Eo, mo, no = oe.find_essential_ransac(p1, p2, cnt, Ks, thr, iters, seed)
    np.testing.assert_array_equal(ng, no)
    np.testing.assert_array_equal(mg, mo)
    np.testing.assert_array_equal(Eg, Eo)                # bit-identical: float64 without FMA on both sides, same order
    return Eg, mg, ng


def assert_pose_oracle(E, p1, p2, cnt, Ks, mask, dist=50.0):
    R, t, m, n = capi().recover_pose(t_(E), t_(p1), t_(p2), t_(cnt), t_(Ks), None if mask is None else t_(mask), dist)
    Ro, to, mo, no = oe.recover_pose(E, p1, p2, cnt, Ks, mask, dist)
    np.testing.assert_array_equal(n.cpu().numpy(), no)
    np.testing.assert_array_equal(m.cpu().numpy(), mo)
    np.testing.assert_array_equal(R.cpu().numpy(), Ro)
    np.testing.assert_array_equal(t.cpu().numpy(), to)
    return Ro, to, mo, no


# ------------------------------------------------------------------------------------------ GPU == oracle
@pytest.mark.parametrize("seed,iters,B,M", [(0, 100, 64, 16384), (1, 1, 16, 16384), (2, 1000, 4, 2048)])
def test_gpu_matches_oracle_bit_for_bit(seed, iters, B, M):
    if B >= 8:
        counts = [0, 4, 5, 6, M, 16, 1] + np.random.default_rng(100 + seed).integers(7, 2500, B - 7).tolist()
    else:
        counts = [2048, 1500, 5, 700][:B]
    p1, p2, cnt, Ks = batch(seed, counts, M)
    for thr in (1.0, 3.0):
        Eg, mg, ng = assert_oracle(p1, p2, cnt, Ks, thr, iters, seed)
        assert (ng[cnt < 5] == 0).all() and (Eg[cnt < 5] == 0).all()
        assert (mg.sum(1) == ng).all()
        found = Eg.reshape(B, 9).any(1)
        assert found[cnt >= 6].mean() > 0.9
        np.testing.assert_allclose(np.linalg.norm(Eg[found].reshape(-1, 9), axis=1), 1.0, rtol=1e-14)
        # recover_pose on the RANSAC output, with its inlier mask and without a mask
        _, to, _, no = assert_pose_oracle(Eg, p1, p2, cnt, Ks, mg)
        assert (no <= ng).all() and (no[~found] == 0).all()
        np.testing.assert_allclose(np.linalg.norm(to[found], axis=1), 1.0, rtol=1e-14)
        if thr == 1.0:
            assert_pose_oracle(Eg, p1, p2, cnt, Ks, None, 8.0)


def test_counts_are_clamped_and_seed_changes_the_draws():
    p1, p2, cnt, Ks = batch(4, [300, 300], 300)
    a = run_gpu(p1, p2, np.array([-5, 10 ** 6], np.int32), Ks, 1.0, 300, 9)
    b = run_gpu(p1, p2, np.array([0, 300], np.int32), Ks, 1.0, 300, 9)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    s1 = run_gpu(p1, p2, cnt, Ks, 1.0, 50, 1)
    s2 = run_gpu(p1, p2, cnt, Ks, 1.0, 50, 2)
    np.testing.assert_array_equal(s1[0], oe.find_essential_ransac(p1, p2, cnt, Ks, 1.0, 50, 1)[0])
    assert not np.array_equal(s1[0], s2[0])


def test_invalid_k_gives_zeros_and_leaves_other_pairs_unchanged():
    p1, p2, cnt, Ks = batch(5, [400, 400, 400, 400], 400)
    ref = run_gpu(p1, p2, cnt, Ks, 1.0, 200, 0)
    assert ref[2].all()
    bad = [np.r_[K.reshape(9)[:8], 2.0], np.r_[0.0, K.reshape(9)[1:]], np.r_[K.reshape(9)[:4], np.nan, K.reshape(9)[5:]]]
    for i, kb in enumerate(bad):
        K2 = Ks.copy()
        K2[1, i % 2] = kb.reshape(3, 3)
        got = run_gpu(p1, p2, cnt, K2, 1.0, 200, 0)
        assert got[2][1] == 0 and not got[0][1].any() and not got[1][1].any()
        for x, y in zip(got, ref):
            np.testing.assert_array_equal(np.delete(x, 1, 0), np.delete(y, 1, 0))
        R, t, m, n = capi().recover_pose(t_(ref[0]), t_(p1), t_(p2), t_(cnt), t_(K2))
        assert n[1].item() == 0 and not R[1].any() and not t[1].any() and not m[1].any() and n[0].item() > 0


# ------------------------------------------------------------------------------------------ degenerate inputs
def test_degenerate_inputs():
    """Identical points in both images give a zero or NaN pivot; an all-zero E gives all-zero pose outputs.  (Identical
    points in one image only are not degenerate: every E with E x1 = 0 fits them.)"""
    from balf_b200.demo import demo_match
    rng = np.random.default_rng(5)
    n = 400
    other = rng.uniform([0, 0], [W, H], (n, 2))
    same1, same2 = np.tile([[10.0, 20.0]], (n, 1)), np.tile([[30.0, 40.0]], (n, 1))
    E, mask = demo_match.find_essential(same1, same2, K)
    assert E is None and mask.shape == (n, 1) and mask.dtype == np.uint8 and not mask.any()
    for k in (0, 1, 4):
        E, mask = demo_match.find_essential(other[:k], other[:k], K)
        assert E is None and mask.shape == (k, 1)
    ng, R, t, m = demo_match.recover_pose(np.zeros((3, 3)), other, other, K)
    assert ng == 0 and not R.any() and not t.any() and m.shape == (n, 1) and not m.any()


def test_exhausted_draws():
    """5 matches: with seeds 530694, 549408 and 550590 hypothesis 0 of pair 0 has not found 5 distinct indices after its
    64 counters, so with iters = 1 the pair has no model; with more hypotheses the result is the oracle's bit for bit."""
    p1, p2, _, Ks = batch(6, [5], 5)
    cnt = np.array([5], np.int32)
    for seed in (530694, 549408, 550590):
        assert not of.sample_indices(seed, 0, np.array([0]), 5, k=5, draws=oe.MAX_DRAWS)[1][0]
        E, m, n = run_gpu(p1, p2, cnt, Ks, 1.0, 1, seed)
        assert n[0] == 0 and not E.any() and not m.any()
        assert_oracle(p1, p2, cnt, Ks, 1.0, 3, seed)


# ------------------------------------------------------------------------------------------ against cv2
def rot_err(Ra, Rb):
    return np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1) / 2, -1, 1)))


def t_err(ta, tb):
    return np.degrees(np.arccos(np.clip(np.dot(ta.ravel(), tb.ravel()), -1, 1)))


# Margins set from the values measured on the B200 (printed by the test): the median rotation and translation-direction
# errors over the 8 scenes of each ratio may exceed cv2's by at most these, and the median inlier count may fall below
# cv2's by at most CV2_INLIER_MARGIN of the matches.  Neither refits its minimal model, so single scenes differ by the
# luck of the draw, hence medians: at ratio 0.3 with K1 != K2 (cv2's fixed 1000 hypotheses, about 2.4 all-inlier
# samples expected) one scene of ours was measured at 6.5 deg (mean 1.15 deg against cv2's 0.25, median 0.34 against
# 0.24).  At ratios 0.5 - 0.9 this library's means were below cv2's on every measure.
CV2_ROT_MARGIN = 0.5        # degrees
CV2_T_MARGIN = 2.0          # degrees
CV2_INLIER_MARGIN = 0.05    # fraction of the matches


def compare_cv2(cv2, scenes, got, two_camera, iters):
    rs, ts, cr, ct, dinl = [], [], [], [], []
    for (a, b, R, t, _, K1, K2), (Rg, tg, E, mask, pmask) in zip(scenes, got):
        assert Rg is not None and E is not None
        if two_camera:
            _, Ec, Rc, tc, mc = cv2.recoverPose(a, b, K1, np.zeros(5), K2, np.zeros(5), method=cv2.RANSAC, prob=0.999,
                                                threshold=1.0)
            mcount = int((mc != 0).sum())
            inl_c = int(cv2.findEssentialMat(a, b, K1, np.zeros(5), K2, np.zeros(5), cv2.RANSAC, 0.999, 1.0)[1].sum())
        else:
            Ec, mc = cv2.findEssentialMat(a, b, K1, cv2.RANSAC, 0.999, 1.0, maxIters=iters)
            inl_c = int(mc.sum())
            _, Rc, tc, _ = cv2.recoverPose(Ec[:3], a, b, K1, mask=mc)
        rs.append(rot_err(Rg, R)); ts.append(t_err(tg, t))
        cr.append(rot_err(Rc, R)); ct.append(t_err(tc, t))
        dinl.append(int(mask.sum()) - inl_c)
    return np.array(rs), np.array(ts), np.array(cr), np.array(ct), np.array(dinl)


@pytest.mark.parametrize("ratio", [0.3, 0.5, 0.7, 0.9])
def test_at_least_as_good_as_cv2(ratio):
    """One K: both at the same hypothesis cap (20000 at ratio 0.3, where 1000 leave about 9 % of the scenes without an
    all-inlier sample; cv2 stops earlier at its confidence 0.999).  K1 != K2: cv2's two-camera overload runs 1000."""
    cv2 = pytest.importorskip("cv2")
    from balf_b200.demo import demo_match
    n = 1000
    iters = 20000 if ratio < 0.4 else 1000
    rng = np.random.default_rng(int(ratio * 100))
    for two_camera in (False, True):
        scenes = []
        for _ in range(8):
            K1, K2 = (random_k(rng), random_k(rng)) if two_camera else (K, K)
            scenes.append(two_view(rng, n, ratio, K1=K1, K2=K2) + (K1, K2))
        it = 1000 if two_camera else iters
        got = demo_match.relative_pose_batch([(s[0], s[1]) for s in scenes], [(s[5], s[6]) for s in scenes], 1.0, it, 0)
        rs, ts, cr, ct, dinl = compare_cv2(cv2, scenes, got, two_camera, it)
        med = np.median
        print("ratio %.1f %s: rotation error median %.4f (cv2 %.4f) mean %.4f (cv2 %.4f) deg, translation median %.4f "
              "(cv2 %.4f) mean %.4f (cv2 %.4f) deg, inlier gap median %.1f min %d" %
              (ratio, "K1 != K2" if two_camera else "one K", med(rs), med(cr), rs.mean(), cr.mean(), med(ts), med(ct),
               ts.mean(), ct.mean(), med(dinl), dinl.min()))
        assert med(rs) <= med(cr) + CV2_ROT_MARGIN
        assert med(ts) <= med(ct) + CV2_T_MARGIN
        assert med(dinl) >= -CV2_INLIER_MARGIN * n
    # the single-pair calls return what the batch returns
    a, b = scenes[0][0], scenes[0][1]
    E1, m1 = demo_match.find_essential(a, b, scenes[0][5], scenes[0][6], 1.0, it)
    np.testing.assert_array_equal(E1, got[0][2])
    np.testing.assert_array_equal(m1, got[0][3])
    ng, R1, t1, pm = demo_match.recover_pose(E1, a, b, scenes[0][5], scenes[0][6], mask=m1)
    np.testing.assert_array_equal(R1, got[0][0])
    np.testing.assert_array_equal(t1, got[0][1])
    np.testing.assert_array_equal(pm, got[0][4])
    assert ng == int(pm.sum())


# ------------------------------------------------------------------------------------------ end to end
E2E_DX, E2E_DY = 128, 64
# B200, seed-0 random-init weights: 802 SMNN matches, 712 of them within 1 px of the offset, inlier fraction 0.8915,
# every match that follows the offset an inlier; singular values 0.70719, 0.70702, 1.2e-4 (a minimal model of noisy
# matches on a plane, where the 5-point system is near-degenerate); R 0.08 deg from I, t 0.30 deg from -(dx, dy, 0).
# Floors and bounds with margin.
E2E_INLIER_FLOOR = 0.75
E2E_SV_TOL = 2e-3            # |s1 - s2| and s3, relative to s1
E2E_ROT_DEG, E2E_T_DEG = 1.0, 3.0


def test_extract_matches_then_relative_pose(detector):
    """The fundamental-matrix test's two offset crops of one noise image: a fronto-parallel plane seen by a camera that
    translates parallel to it, so x2 = x1 - (dx, dy), R = I and t is along -(dx, dy, 0).  The scene is planar and every
    E = [t']x (for any t') fits such matches, so the pose is not determined by them: this checks the pipeline (E found with
    two equal singular values and a zero one, the matches that follow the offset are inliers).  On this input the pipeline
    picks the true pose (measured, see above), which is checked too."""
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
    R, t, E, mask, pmask = demo_match.relative_pose_batch([(p1, p2)], [K])[0]
    assert E is not None and R is not None and mask.shape == (len(p1), 1) and pmask.shape == (len(p1), 1)
    s = np.linalg.svd(E, compute_uv=False)
    good = np.abs(p1 - p2 - [E2E_DX, E2E_DY]).max(1) < 1.0
    frac, good_in = mask.mean(), mask[good, 0].mean()
    want_t = -np.array([E2E_DX, E2E_DY, 0.0]) / np.hypot(E2E_DX, E2E_DY)
    print("e2e: %d matches, %d follow the offset, inlier fraction %.4f, of those following %.4f, singular values %s, "
          "rotation from I %.4f deg, t %s (angle to -(dx, dy, 0) %.2f deg), pose mask %d" %
          (len(p1), good.sum(), frac, good_in, s, rot_err(R, np.eye(3)), t.ravel(), t_err(t, want_t), pmask.sum()))
    assert abs(s[0] - s[1]) < E2E_SV_TOL * s[0] and s[2] < E2E_SV_TOL * s[0]
    assert rot_err(R, np.eye(3)) < E2E_ROT_DEG and t_err(t, want_t) < E2E_T_DEG
    assert frac > E2E_INLIER_FLOOR
    assert good.sum() > 0.5 * len(p1) and good_in > 0.99
    np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-12)
    assert abs(np.linalg.norm(t) - 1) < 1e-12


# ------------------------------------------------------------------------------------------ argument errors
def test_argument_errors():
    c = capi()
    t = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev())
    p, cnt = t(2, 10, 2), torch.full((2,), 10, dtype=torch.int32, device=dev())
    k = torch.from_numpy(np.tile(K.reshape(9), (2, 2, 1))).to(dev())
    out_e, out_m, out_n = t(2, 9), torch.zeros(2, 10, dtype=torch.uint8, device=dev()), torch.zeros(2, dtype=torch.int32,
                                                                                                      device=dev())
    ws_bytes = c._ess_ws(2, 10, 100)
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev())
    raw = lambda M, thr, iters, nbytes, kp=k: c._ess_ransac(c._ptr(p), c._ptr(p), c._ptr(cnt), c._ptr(kp), 2, M, thr, iters,
                                                            0, c._ptr(out_e), c._ptr(out_m), c._ptr(out_n), c._ptr(ws),
                                                            nbytes, c._stream(dev()))
    assert raw(10, 1.0, 100, ws_bytes) == 0
    torch.cuda.synchronize()
    before = c.launch_count()
    for args, what in (((10, 0.0, 100, ws_bytes), "thr"), ((10, -1.0, 100, ws_bytes), "thr"),
                       ((10, float("nan"), 100, ws_bytes), "thr"), ((10, 1.0, 0, ws_bytes), "iters"),
                       ((10, 1.0, (1 << 17) + 1, ws_bytes), "iters"), ((16385, 1.0, 100, ws_bytes), "M = 16385"),
                       ((10, 1.0, 100, ws_bytes - 1), "workspace")):
        assert raw(*args) < 0
        assert what in c._last_error().decode()
    assert raw(10, 1.0, 100, ws_bytes, None) < 0 and "null pointer" in c._last_error().decode()
    R, tv, pm, ng = t(2, 9), t(2, 3), torch.zeros(2, 10, dtype=torch.uint8, device=dev()), out_n.clone()
    rawp = lambda M, dist, e=out_e: c._recover_pose(c._ptr(e), c._ptr(p), c._ptr(p), c._ptr(cnt), c._ptr(k), c._ptr(None), 2,
                                                    M, dist, c._ptr(R), c._ptr(tv), c._ptr(pm), c._ptr(ng), c._stream(dev()))
    for args, what in (((10, 0.0), "dist_thresh"), ((10, -1.0), "dist_thresh"), ((10, float("nan")), "dist_thresh"),
                       ((16385, 50.0), "M = 16385")):
        assert rawp(*args) < 0
        assert what in c._last_error().decode()
    assert rawp(10, 50.0, None) < 0 and "null pointer" in c._last_error().decode()
    for thr, iters, what in ((0.0, 100, "thr"), (1.0, 0, "iters")):
        with pytest.raises(ValueError, match=what):
            c.find_essential_ransac(p, p, cnt, k, thr, iters, 0)
    with pytest.raises(ValueError, match="M = 16385"):
        c.find_essential_ransac(t(1, 16385, 2), t(1, 16385, 2), cnt[:1], k[:1], 1.0, 10, 0)
    with pytest.raises(ValueError, match="K must be"):
        c.find_essential_ransac(p, p, cnt, k[:, :, :8], 1.0, 10, 0)
    with pytest.raises(ValueError, match="K must be"):
        c.find_essential_ransac(p, p, cnt, k[:1], 1.0, 10, 0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        c.find_essential_ransac(p.cpu(), p.cpu(), cnt.cpu(), k.cpu(), 1.0, 10, 0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        c.find_essential_ransac(p, p, cnt, k.cpu(), 1.0, 10, 0)
    with pytest.raises(ValueError, match="dist_thresh"):
        c.recover_pose(out_e, p, p, cnt, k, None, 0.0)
    with pytest.raises(ValueError, match="E must be"):
        c.recover_pose(out_e[:, :8], p, p, cnt, k)
    with pytest.raises(ValueError, match="mask must be"):
        c.recover_pose(out_e, p, p, cnt, k, torch.zeros(2, 9, dtype=torch.uint8, device=dev()))
    with pytest.raises(ValueError, match="mask must be"):
        c.recover_pose(out_e, p, p, cnt, k, torch.zeros(2, 10, dtype=torch.float32, device=dev()))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        c.recover_pose(out_e.cpu(), p, p, cnt, k)
    from balf_b200.demo import demo_match
    pts = np.zeros((10, 2))
    for bad in (np.eye(2), np.r_[K[:2], [[0, 0, 2.0]]], np.r_[[[0.0, 0, 600]], K[1:]], np.r_[[[np.inf, 0, 600]], K[1:]]):
        with pytest.raises(ValueError, match="K of pair 0"):
            demo_match.find_essential(pts, pts, bad)
        with pytest.raises(ValueError, match="K of pair 0"):
            demo_match.recover_pose(np.eye(3), pts, pts, K, bad)
    torch.cuda.synchronize()
    assert c.launch_count() == before
