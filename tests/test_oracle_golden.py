"""The oracle is pinned here: every restated function is checked against vectors produced by the
reference's own modules (oracle/make_golden.py, run in the build container).  CPU only."""
import numpy as np
import pytest
import torch

from conftest import load_golden, load_score_480x640, synth_u8, weight_digest
from oracle import detector as odet
from oracle import hardnet as ohn
from oracle import pipeline, postproc, postproc_c


def test_weight_init_matches_reference_digest(detector_sd, hardnet):
    g = load_golden("detector.npz")
    np.testing.assert_allclose(weight_digest(detector_sd), g["weight_digest"], rtol=1e-12)
    np.testing.assert_array_equal(detector_sd["down1.conv.0.weight"].numpy(), g["first_weight"])
    np.testing.assert_array_equal(detector_sd["detector_head.dense.bias"].numpy(), g["head_bias"])
    h = load_golden("hardnet.npz")
    np.testing.assert_allclose(weight_digest(hardnet.state_dict()), h["weight_digest"], rtol=1e-12)
    np.testing.assert_array_equal(hardnet.state_dict()["features.0.weight"].numpy(), h["first_weight"])


def test_detector_oracle_vs_reference(detector_sd):
    g = load_golden("detector.npz")
    x = torch.rand(1, 3, 128, 192, generator=torch.Generator().manual_seed(1234))
    with torch.inference_mode():
        o = odet.detector_forward(detector_sd, x)
    np.testing.assert_allclose(o["prob"][0].numpy(), g["prob_128x192"], rtol=2e-5, atol=0)
    np.testing.assert_allclose(o["logits"][0].numpy(), g["logits_128x192"], rtol=0, atol=2e-6)
    x2 = torch.rand(2, 3, 64, 128, generator=torch.Generator().manual_seed(77))
    with torch.inference_mode():
        o2 = odet.detector_forward(detector_sd, x2)
    np.testing.assert_allclose(o2["prob"].numpy(), g["prob_b2_64x128"], rtol=2e-5)
    np.testing.assert_allclose(o2["logits"].numpy(), g["logits_b2_64x128"], atol=2e-6)


def test_detector_oracle_512x640_anchors(detector_sd):
    """SURVEY.md 8c known-answer anchors of the reference (seed-0 weights, seed-1234 input)."""
    g = load_golden("detector.npz")
    x = torch.rand(1, 3, 512, 640, generator=torch.Generator().manual_seed(1234))
    with torch.inference_mode():
        p = odet.detector_forward(detector_sd, x)["prob"][0].numpy()
    np.testing.assert_allclose(p[::8, ::8], g["prob_512x640_sub8"], rtol=2e-5)
    np.testing.assert_allclose(p[255], g["prob_512x640_row255"], rtol=2e-5)
    st = g["prob_512x640_stats"]
    assert abs(p.astype(np.float64).sum() - st[0]) < 1e-3 and abs(st[0] - 5044.952016152) < 1e-3
    np.testing.assert_allclose(p[0, 0:4], [0.01324156, 0.0150795, 0.01428799, 0.01641722], rtol=1e-5)
    assert abs(p[255, 320] - 0.013534844) < 1e-7


def test_hardnet_oracle_vs_reference(hardnet):
    g = load_golden("hardnet.npz")
    x = torch.rand(8, 1, 32, 32, generator=torch.Generator().manual_seed(4321))
    with torch.inference_mode():
        o = ohn.hardnet_forward(hardnet.state_dict(), x).numpy()
    np.testing.assert_allclose(o, g["out"], atol=2e-6)
    np.testing.assert_allclose(o[0, :4], [-0.07800730, 0.07700513, 0.12284143, 0.01012279], atol=1e-6)


# ----------------------------------------------------------------------------- post-processing
def _pts_equal(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    np.testing.assert_array_equal(a, b)


def _assert_same_points(mine, ref):
    """identical rows, allowing the reference's implementation-defined order inside groups of
    exactly equal scores (its sorts are unstable / reversed -- see oracle/postproc.py)."""
    assert mine.shape == ref.shape, (mine.shape, ref.shape)
    np.testing.assert_array_equal(mine[:, 3], ref[:, 3])
    canon = lambda p: p[np.lexsort((p[:, 0], p[:, 1], -p[:, 3]))]
    np.testing.assert_array_equal(canon(mine), canon(ref))


@pytest.mark.parametrize("impl", ["numpy", "c"])
def test_postproc_480x640_vs_reference(impl):
    g = load_golden("postproc_480x640.npz")
    score = load_score_480x640()
    rb = postproc.remove_borders(score, 15)
    nms = postproc.apply_nms if impl == "numpy" else postproc_c.apply_nms
    np.testing.assert_array_equal(np.flatnonzero(nms(rb, 15)), g["apply_nms15_idx"])
    np.testing.assert_array_equal(np.flatnonzero(nms(rb, 4)), g["apply_nms4_idx"])
    assert len(g["apply_nms15_idx"]) == 2967                                   # SURVEY.md 8c anchor
    nm = postproc.apply_nms(rb, 15)
    for k in (2048, 500, 5000):
        if impl == "numpy":
            _pts_equal(postproc.get_point_coordinates(nm, num_points=k), g["kth_topk%d" % k])
        else:
            idx, _ = postproc_c.kth_value_topk(nm, k)
            ref = g["kth_topk%d" % k]
            np.testing.assert_array_equal(idx, (ref[:, 1] * 640 + ref[:, 0]).astype(np.int32))
    gnms = postproc.greedy_nms if impl == "numpy" else postproc_c.greedy_nms
    for name, thr, r in (("greedy_thr001", 0.001, 15), ("greedy_thr015", 0.015, 15), ("greedy_thr001_r4", 0.001, 4)):
        mine = postproc.get_points_direct_from_score_map(rb, thr, r, False, 4, nms=gnms)
        _assert_same_points(mine, g[name])
    assert len(g["greedy_thr001"]) == 800 and len(g["greedy_thr015"]) == 799   # SURVEY.md 8c anchors
    np.testing.assert_allclose(g["greedy_thr001"][0], [28, 42, 1.0, 0.0226866342], rtol=1e-7)


def test_nms_fast_indices_vs_reference():
    g = load_golden("postproc_480x640.npz")
    rb = postproc.remove_borders(load_score_480x640(), 15)
    ys, xs = np.nonzero(rb >= np.float32(0.001))
    keep = postproc.greedy_nms(xs, ys, rb[ys, xs].astype(np.float64), 480, 640, 15)
    np.testing.assert_array_equal(keep, g["nms_fast_inds"])
    np.testing.assert_array_equal(np.stack([xs[keep], ys[keep], rb[ys, xs][keep]]), g["nms_fast_out"])
    np.testing.assert_array_equal(postproc_c.greedy_nms(xs, ys, rb[ys, xs], 480, 640, 15), g["nms_fast_inds"])


def test_subpixel_restatement_vs_shimmed_reference():
    """unpinned third-party step (torchgeometry): checks only the reference-side arithmetic
    (patch extraction, normalisation, log) around the restated soft-argmax."""
    g = load_golden("postproc_480x640.npz")
    rb = postproc.remove_borders(load_score_480x640(), 15)
    for name, thr, ps in (("greedy_thr001_subpix4", 0.001, 4), ("greedy_thr015_subpix5", 0.015, 5)):
        mine = postproc.get_points_direct_from_score_map(rb, thr, 15, True, ps)
        canon = lambda p: p[np.lexsort((np.round(p[:, 0]), np.round(p[:, 1]), -p[:, 3]))]   # tie groups: see above
        np.testing.assert_allclose(canon(mine), canon(g[name]), rtol=0, atol=1e-5)


@pytest.mark.parametrize("name", ["rand", "quant", "sparse", "zeros", "odd", "one"])
def test_postproc_small_maps_vs_reference(name):
    g = load_golden("postproc_small.npz")
    m = g["map_" + name]
    rb = postproc.remove_borders(m, int(g["rb_" + name]))
    for size in (15, 4, 3):
        want = g["nms%d_%s" % (size, name)]
        np.testing.assert_array_equal(np.flatnonzero(postproc.apply_nms(rb, size)), want)
        np.testing.assert_array_equal(np.flatnonzero(postproc_c.apply_nms(rb, size)), want)
    nm = postproc.apply_nms(rb, 15)
    for k in (1, 50, 2048):
        for key, src in (("kth", nm), ("kthraw", rb)):
            want = g["%s%d_%s" % (key, k, name)]
            np.testing.assert_array_equal(postproc.find_index_higher_scores(src, k), want)
            idx, _ = postproc_c.kth_value_topk(src, k)
            np.testing.assert_array_equal(idx, want[:, 0] * m.shape[1] + want[:, 1])
    for r in (15, 4, 1):
        want = g["greedy%d_%s" % (r, name)]
        for fn in (postproc.greedy_nms, postproc_c.greedy_nms):
            mine = postproc.get_points_direct_from_score_map(rb, 0.015, r, False, 4, nms=fn)
            _assert_same_points(mine.reshape(-1, 4), want.reshape(-1, 4))


def test_kth_value_raises_on_short_map():
    with pytest.raises(IndexError):
        postproc.find_index_higher_scores(np.ones((4, 4), np.float32), 17)
    with pytest.raises(IndexError):
        postproc_c.kth_value_topk(np.ones((4, 4), np.float32), 17)


def test_pad_and_detect_vs_reference(detector_sd):
    g = load_golden("detect.npz")
    for h, w, seed in ((480, 640, 1234), (121, 187, 5), (128, 192, 6)):
        im = synth_u8(h, w, seed)
        x = postproc.preprocess(im)
        assert tuple(g["pad_shape_%dx%d" % (h, w)][:2]) == x.shape[2:]
        assert abs(x.astype(np.float64).sum() - g["pad_sum_%dx%d" % (h, w)][0]) < 1e-6
        if h < 480:
            np.testing.assert_array_equal(x[0].transpose(1, 2, 0), g["pad_%dx%d" % (h, w)])
            args = pipeline.default_args(sub_pixel=False)
            mine = pipeline.detect(args, detector_sd, im)
            ref = g["detect_%dx%d" % (h, w)]
            assert mine.shape == ref.shape
            inter = set(map(tuple, mine[:, :2])) & set(map(tuple, ref[:, :2]))
            assert len(inter) >= 0.99 * len(ref)      # last-ulp BLAS differences may flip a fragile maximum
