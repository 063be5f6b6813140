"""Parity of the CUDA post-processing (balf_b200/csrc/nms.cu, through the C-ABI) with the oracle.
Bit-exact on indices and scores; sub-pixel offsets within a stated fp32 tolerance."""
import numpy as np
import pytest
import torch

from conftest import load_golden, load_score_480x640
from oracle import postproc, postproc_c

pytestmark = pytest.mark.gpu
SUBPIX_ATOL = 2e-5      # fp32 exp/log/sum-order differences of the 16..25-tap soft-argmax


def capi():
    import balf_b200._capi as c
    return c


def dev():
    return torch.device("cuda:0")


def gpu_windowed(score, k, border, size, crop=None):
    xy, sc, cnt = capi().windowed_nms_topk(torch.as_tensor(score).to(dev()), k, border=border, nms_size=size, crop=crop)
    xy, sc, cnt = xy.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    return [np.concatenate([xy[b, :cnt[b]].astype(np.float64), np.ones((cnt[b], 1)), sc[b, :cnt[b], None].astype(np.float64)], 1)
            for b in range(len(cnt))]


def gpu_greedy(score, k, border, thr, r, ps=0, crop=None):
    xy, sc, dxdy, cnt = capi().greedy_nms_topk(torch.as_tensor(score).to(dev()), k, border=border, thr=thr, radius=r,
                                               subpixel_ps=ps, crop=crop)
    xy, sc, cnt = xy.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    out = []
    for b in range(len(cnt)):
        p = xy[b, :cnt[b]].astype(np.float64)
        if ps:
            p = p + dxdy[b, :cnt[b]].cpu().numpy().astype(np.float64)
        out.append(np.concatenate([p, np.ones((cnt[b], 1)), sc[b, :cnt[b], None].astype(np.float64)], 1))
    return out


def oracle_greedy(score, border, thr, r, k, ps=0, fast=True):
    rb = postproc.remove_borders(score, border)
    pts = postproc.get_points_direct_from_score_map(rb, thr, r, ps > 0, ps if ps else 4,
                                                    nms=postproc_c.greedy_nms if fast else postproc.greedy_nms)
    return pts[np.argsort(-pts[:, 3], kind="stable")][:k] if len(pts) else pts.reshape(0, 4)


def test_windowed_golden_map():
    g = load_golden("postproc_480x640.npz")
    score = load_score_480x640()
    for k in (2048, 500, 5000):
        want = postproc.windowed_detect(score, 15, 15, k)
        got = gpu_windowed(score, k, 15, 15)[0]
        np.testing.assert_array_equal(got, want)
        ref = g["kth_topk%d" % k]                                # the reference's own raster-ordered rows
        np.testing.assert_array_equal(got[np.lexsort((got[:, 0], got[:, 1]))], ref)


def test_greedy_golden_map():
    g = load_golden("postproc_480x640.npz")
    score = load_score_480x640()
    for name, thr, r in (("greedy_thr001", 0.001, 15), ("greedy_thr015", 0.015, 15), ("greedy_thr001_r4", 0.001, 4)):
        got = gpu_greedy(score, 8192, 15, thr, r)[0]
        want = oracle_greedy(score, 15, thr, r, 8192)
        np.testing.assert_array_equal(got, want)
        ref = g[name]
        canon = lambda p: p[np.lexsort((p[:, 0], p[:, 1], -p[:, 3]))]
        np.testing.assert_array_equal(canon(got), canon(ref))
    got = gpu_greedy(score, 2048, 15, 0.001, 15)[0]
    assert len(got) == 800
    np.testing.assert_allclose(got[0], [28, 42, 1.0, 0.0226866342], rtol=1e-7)


def test_greedy_topk_binds():
    score = load_score_480x640()
    for k in (1, 100, 777):
        np.testing.assert_array_equal(gpu_greedy(score, k, 15, 0.001, 15)[0], oracle_greedy(score, 15, 0.001, 15, k))
    k = 300                                                       # r = 4 keeps thousands: radix-select path
    np.testing.assert_array_equal(gpu_greedy(score, k, 15, 0.001, 4)[0], oracle_greedy(score, 15, 0.001, 4, k))


def test_subpixel():
    score = load_score_480x640()
    for thr, ps in ((0.001, 4), (0.015, 5), (0.001, 3)):
        got = gpu_greedy(score, 2048, 15, thr, 15, ps)[0]
        want = oracle_greedy(score, 15, thr, 15, 2048, ps)
        np.testing.assert_array_equal(got[:, 2:], want[:, 2:])
        np.testing.assert_allclose(got[:, :2], want[:, :2], rtol=0, atol=SUBPIX_ATOL)
        assert np.abs(got[:, :2] - np.round(want[:, :2])).max() > 0.01     # offsets are really applied


@pytest.mark.parametrize("name", ["rand", "quant", "sparse", "zeros", "odd", "one"])
def test_small_maps(name):
    g = load_golden("postproc_small.npz")
    m = g["map_" + name]
    b = int(g["rb_" + name])
    for size in (15, 4, 3, 31, 1):
        for k in (1, 50, 2048):
            want = postproc.windowed_detect(m, b, size, k)
            got = gpu_windowed(m, k, b, size)[0]
            np.testing.assert_array_equal(got, want, err_msg="windowed %s size %d k %d" % (name, size, k))
    for r in (15, 4, 1, 0, 7):
        for thr in (0.015, 0.0, 0.5):
            want = oracle_greedy(m, b, thr, r, 4096)
            got = gpu_greedy(m, 4096, b, thr, r)[0]
            np.testing.assert_array_equal(got, want, err_msg="greedy %s r %d thr %g" % (name, r, thr))


def test_dense_apply_nms_and_helpers():
    from balf_b200.utils import test_utils as tu
    g = load_golden("postproc_small.npz")
    for name in ("rand", "quant", "odd"):
        m = g["map_" + name]
        for size in (15, 4, 3, 31):
            np.testing.assert_array_equal(tu.apply_nms(m, size), postproc.apply_nms(m, size))
        rb = tu.remove_borders(m, 5)
        np.testing.assert_array_equal(rb, postproc.remove_borders(m, 5))
        nm = postproc.apply_nms(rb, 15)
        for k in (1, 50, 2048):
            np.testing.assert_array_equal(tu.find_index_higher_scores(nm, k), postproc.find_index_higher_scores(nm, k))
            np.testing.assert_array_equal(tu.get_point_coordinates(nm, num_points=k), postproc.get_point_coordinates(nm, num_points=k))
        got = tu.get_points_direct_from_score_map(rb, 0.015, 4, False, 4)
        want = postproc.get_points_direct_from_score_map(rb, 0.015, 4, False, 4)
        np.testing.assert_array_equal(got, want)
        got = tu.get_points_direct_from_score_map(rb, 0.015, 4, True, 5)
        want = postproc.get_points_direct_from_score_map(rb, 0.015, 4, True, 5)
        np.testing.assert_allclose(got, want, rtol=0, atol=SUBPIX_ATOL)
        ys, xs = np.nonzero(rb >= np.float32(0.3))
        pts = np.stack([xs, ys, rb[ys, xs]]).astype(np.float64)
        out, inds = tu.nms_fast(pts, m.shape[0], m.shape[1], 4)
        keep = postproc.greedy_nms(xs, ys, pts[2], m.shape[0], m.shape[1], 4)
        np.testing.assert_array_equal(inds, keep)
        np.testing.assert_array_equal(out, pts[:, keep])
    with pytest.raises(IndexError):
        tu.find_index_higher_scores(np.ones((4, 4), np.float32), 17)
    assert tu.get_points_direct_from_score_map(np.zeros((64, 64), np.float32), 0.015, 15, True, 5).shape == (0, 4)
    assert tu.make_shape_even(np.zeros((5, 7, 3))).shape == (6, 8, 3)
    assert tu.mod_padding_symmetric(np.zeros((480, 640, 3))).shape == (512, 640, 3)
    assert tu.mod_padding_symmetric(np.zeros((900, 1200, 3))).shape == (960, 1216, 3)
    assert tu.mod_padding_symmetric(np.zeros((128, 192, 3))).shape == (128, 192, 3)
    # the stand-alone helper follows the reference arithmetic for odd sizes too (121 -> 127 rows with 3 + 3), golden pad arrays
    odd = np.arange(121 * 187 * 3, dtype=np.float64).reshape(121, 187, 3)
    p = tu.mod_padding_symmetric(odd)
    assert p.shape == (127, 191, 3) and np.array_equal(p[3:124, 2:189], odd) and p[:3].sum() == 0
    # nms_fast returns the caller's own (unrounded) columns, like the reference (test_utils.py:161)
    sub = np.stack([np.array([10.2, 30.7, 11.4, 80.0]), np.array([5.1, 5.4, 6.2, 40.0]), np.array([0.5, 0.9, 0.7, 0.1])])
    out, inds = tu.nms_fast(sub, 64, 96, 4)
    np.testing.assert_array_equal(inds, [1, 2, 3])
    np.testing.assert_array_equal(out, sub[:, [1, 2, 3]])
    # float64 maps keep their own values (the device only decides the mask)
    m64 = g["map_rand"].astype(np.float64) + 1e-12
    np.testing.assert_array_equal(tu.apply_nms(m64, 15), m64 * (postproc.apply_nms(g["map_rand"], 15) != 0))
    # no silent truncation: a radius-2 NMS on a large map can keep more than the 16384 points of one call
    with pytest.raises(ValueError):
        tu.get_points_direct_from_score_map(np.random.default_rng(0).random((600, 800), dtype=np.float32), 0.015, 2, False, 4)


def test_errors():
    c = capi()
    s = torch.rand(1, 16, 16, device=dev())
    with pytest.raises(ValueError):
        c.windowed_nms_topk(s, 257)                              # fewer than k elements (IndexError in the reference)
    with pytest.raises(ValueError):
        c.windowed_nms_topk(s, 4, crop=(8, 8, 16, 16))           # crop outside the map
    with pytest.raises(ValueError):
        c.greedy_nms_topk(s, 20000)                              # k above the supported maximum
    with pytest.raises(RuntimeError):
        c.windowed_nms_topk(s.cpu(), 4)                          # no CPU path


def test_batched_crop_full_size():
    """config-2 shape: batch of padded 512x640 maps, crop 480x640 at row 16; every image against the
    C oracle, plus size-independent properties."""
    B = 6
    rng = np.random.default_rng(11)
    maps = (rng.random((B, 512, 640), dtype=np.float32) * 0.02 + 0.005).astype(np.float32)
    maps[1] = np.round(maps[1] * 2000) / 2000                    # heavy ties / plateaus
    maps[2, 16:496] *= (rng.random((480, 640)) > 0.999)         # almost empty: fewer than k survivors
    maps[3] = 0                                                  # all-zero map quirk
    crop = (16, 0, 480, 640)
    got_w = gpu_windowed(maps, 2048, 15, 15, crop)
    got_g = gpu_greedy(maps, 2048, 15, 0.001, 15, 0, crop)
    for b in range(B):
        s = maps[b, 16:496]
        want = postproc.windowed_detect(s, 15, 15, 2048)
        np.testing.assert_array_equal(got_w[b], want, err_msg="windowed image %d" % b)
        want = oracle_greedy(s, 15, 0.001, 15, 2048)
        np.testing.assert_array_equal(got_g[b], want, err_msg="greedy image %d" % b)
        p = got_g[b]
        if len(p) > 1:
            assert np.all(np.diff(p[:, 3]) <= 0)                 # sorted by score
            d = np.maximum(np.abs(p[:, None, 0] - p[None, :, 0]), np.abs(p[:, None, 1] - p[None, :, 1]))
            np.fill_diagonal(d, 1e9)
            assert d.min() > 15                                  # exclusion box respected
            assert p[:, 0].min() >= 15 and p[:, 0].max() < 640 - 15 and p[:, 1].min() >= 15 and p[:, 1].max() < 480 - 15
    assert len(got_w[3]) == 2048 and np.all(got_w[3][:, 3] == 0)  # zero-map quirk: first k raster pixels
    assert len(got_g[3]) == 0


def test_large_map_1200x900_topk_binds():
    rng = np.random.default_rng(5)
    s = (rng.random((900, 1200), dtype=np.float32) * 0.02).astype(np.float32)
    got = gpu_greedy(s, 2048, 15, 0.001, 15)[0]
    want = oracle_greedy(s, 15, 0.001, 15, 2048)
    assert len(want) == 2048
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(gpu_windowed(s, 8192, 15, 15)[0], postproc.windowed_detect(s, 15, 15, 8192))


def test_windowed15_two_level_edge_cases():
    """nms_size 15 runs as block-maximum + coarse-select passes (csrc/nms.cu): unaligned crops (scalar load path), sizes
    that are not multiples of the 4x4 blocks, every border width, negative and zero scores, plateaus larger than the
    per-CTA survivor staging list, and isolated peaks next to the map edge."""
    rng = np.random.default_rng(23)
    base = (rng.random((3, 200, 333), dtype=np.float32) - 0.2).astype(np.float32)          # ~20 % negative
    base[1] = np.round(base[1] * 8) / 8                                                     # plateaus / ties
    base[2] *= (rng.random((200, 333)) > 0.97)                                              # sparse, many zeros
    for (top, left, H, W) in ((0, 0, 200, 333), (3, 5, 190, 321), (8, 4, 64, 128), (1, 2, 17, 29), (0, 1, 15, 15)):
        for border in (0, 1, 7, 15):
            if 2 * border >= min(H, W):
                continue
            k = min(2048, H * W)
            got = gpu_windowed(base, k, border, 15, (top, left, H, W))
            for b in range(3):
                want = postproc.windowed_detect(base[b, top:top + H, left:left + W], border, 15, k)
                np.testing.assert_array_equal(got[b], want, err_msg="crop %s border %d image %d" % ((top, left, H, W), border, b))
    # one big plateau: every pixel of the interior survives (far more than the 512-entry staging list per tile)
    flat = np.full((1, 96, 256), 0.25, np.float32)
    for k in (100, 16384):
        np.testing.assert_array_equal(gpu_windowed(flat, k, 2, 15)[0], postproc.windowed_detect(flat[0], 2, 15, k))
    # peaks at the corners and edges, equal-valued neighbours exactly 7 and 8 pixels apart
    m = np.zeros((1, 64, 64), np.float32)
    for (y, x, v) in ((0, 0, 1.0), (0, 63, 1.0), (63, 0, 2.0), (63, 63, 0.5), (20, 20, 3.0), (20, 27, 3.0), (20, 35, 2.9),
                      (27, 27, 3.0), (28, 28, 3.1), (40, 8, 1.0), (40, 16, 1.0), (47, 12, 1.0)):
        m[0, y, x] = v
    np.testing.assert_array_equal(gpu_windowed(m, 64, 0, 15)[0], postproc.windowed_detect(m[0], 0, 15, 64))


def test_windowed15_tma_and_fallback_paths():
    """nms_size 15 on maps the TMA can describe (row pitch a multiple of 16 bytes, at least one 80 x 80 window): the persistent
    double-buffered kernel (windows that leave the interior are masked in place) against the oracle and against the per-thread-load
    kernel (balf_debug_set key 7), for crops whose left edge is / is not a multiple of four pixels (the TMA faults on a box that
    does not start on a 16-byte boundary: those crops must take the fallback), partial tiles, every border class, negative scores."""
    rng = np.random.default_rng(29)
    base = (rng.random((5, 176, 336), dtype=np.float32) - 0.1).astype(np.float32)           # ~10 % negative
    base[1] = np.round(base[1] * 16) / 16                                                    # plateaus / ties
    base[2] *= (rng.random((176, 336)) > 0.97)                                               # sparse, many zeros
    c = capi()
    try:
        for (top, left, H, W) in ((0, 0, 176, 336), (3, 4, 160, 320), (2, 5, 150, 300), (25, 25, 129, 257), (8, 8, 100, 200)):
            for border in (0, 7, 15):
                k = 2048
                outs = []
                for tma in (1, 0):
                    c.debug_set(7, tma)
                    outs.append(gpu_windowed(base, k, border, 15, (top, left, H, W)))
                for b in range(base.shape[0]):
                    want = postproc.windowed_detect(base[b, top:top + H, left:left + W], border, 15, k)
                    np.testing.assert_array_equal(outs[0][b], want, err_msg="crop %s border %d image %d" % ((top, left, H, W), border, b))
                    np.testing.assert_array_equal(outs[1][b], want, err_msg="fallback: crop %s border %d image %d" % ((top, left, H, W), border, b))
    finally:
        c.debug_set(7, 1)


# ----------------------------------------------------------------------------- cell-based greedy NMS (round 2) and box_nms
def test_greedy_cells_vs_whole_image_kernel_and_oracle():
    """the multi-CTA cell rounds, the one-CTA-per-image finisher (long monotone ramps need one round per kept pixel, far
    more than the fixed multi-CTA rounds) and the round-1 whole-image kernel agree with the oracle on every radius"""
    rng = np.random.default_rng(21)
    ramp = np.tile(np.linspace(1.0, 0.2, 700, dtype=np.float32), (90, 1))            # strictly decreasing along x
    ramp += (np.arange(90, dtype=np.float32) * 1e-4)[:, None]
    maps = {"rand": rng.random((200, 333), dtype=np.float32),
            "quant": (rng.integers(0, 9, (150, 260)) / 8.0).astype(np.float32),        # heavy ties
            "ramp": ramp,
            "sparse": (rng.random((170, 190), dtype=np.float32) * (rng.random((170, 190)) > 0.98)).astype(np.float32)}
    for name, m in maps.items():
        for r in (15, 9, 4, 2, 1):
            border = 15 if name != "ramp" else 3
            want = oracle_greedy(m, border, 0.015, r, 16384)
            got = gpu_greedy(m, 16384, border, 0.015, r)[0]
            np.testing.assert_array_equal(got, want, err_msg="%s r=%d" % (name, r))
            capi().debug_set(5, 1)
            try:
                old = gpu_greedy(m, 16384, border, 0.015, r)[0]
            finally:
                capi().debug_set(5, 0)
            np.testing.assert_array_equal(old, want, err_msg="whole-image kernel %s r=%d" % (name, r))


def test_greedy_cells_batch_crop_and_subpixel():
    score = load_score_480x640()
    rng = np.random.default_rng(2)
    batch = np.stack([score, score[::-1].copy(), np.roll(score, 37, 1), rng.random((480, 640), dtype=np.float32) * 0.03])
    padded = np.zeros((4, 512, 704), np.float32)
    padded[:, 16:496, 33:673] = batch
    got = gpu_greedy(padded, 2048, 15, 0.001, 15, ps=4, crop=(16, 33, 480, 640))
    for b in range(4):
        want = oracle_greedy(batch[b], 15, 0.001, 15, 2048, ps=4)
        np.testing.assert_array_equal(got[b][:, 3], want[:, 3])
        np.testing.assert_allclose(got[b][:, :2], want[:, :2], atol=SUBPIX_ATOL)


def test_box_nms_vs_torchvision_golden():
    from balf_b200.benchmark_test import repeatability_tools as rt
    g = load_golden("r2_boxnms.npz")
    for key in [k for k in g.files if k.startswith("keep_")]:
        _, name, s, i, kk = key.split("_")
        size, iou, top = int(s[1:]), int(i[1:]) / 10, int(kk[1:]) or -1
        prob = torch.from_numpy(g["prob_" + name])[None]
        out = rt.box_nms(prob.to(dev()), size=size, iou=iou, min_prob=0.015, keep_top_k=top)
        assert out.shape == prob.shape and out.is_cuda
        out = out[0].cpu().numpy()
        np.testing.assert_array_equal(np.flatnonzero(out).astype(np.int32), g[key], err_msg=key)
        np.testing.assert_array_equal(out[out != 0], g["prob_" + name][out != 0])
        np.testing.assert_array_equal(out, postproc.box_nms(g["prob_" + name], size, iou, 0.015, top))
    small = torch.rand(1, 40, 56, generator=torch.Generator().manual_seed(8)) * 0.05       # footprints the cells do not tile
    for size, iou in ((2, 0.6), (3, 0.05), (9, 0.5)):
        got = rt.box_nms(small.to(dev()), size=size, iou=iou)[0].cpu().numpy()
        np.testing.assert_array_equal(got, postproc.box_nms(small[0].numpy(), size, iou, 0.015, -1), err_msg="%s %s" % (size, iou))
