"""Generate ``tests/golden/*.npz`` by running the REFERENCE's own Python modules.

TEST INFRASTRUCTURE.  Needs a checkout of the reference project at oracle/_ref (or at the path in
BALF_REFERENCE):   python -m oracle.make_golden [r2]

What is pinned by these vectors: the seed-0 state_dicts and the forward of the detector
(balf/model) and of HardNet (third_party/hardnet), and every NumPy helper of
balf/utils/test_utils.py that the hot path touches.  The reference is run unmodified except
for two shims, both recorded in the files:

* ``np.argsort`` is forced to ``kind='stable'`` while reference code runs, so that its four
  unstable sorts become deterministic (tie order = input order).  See oracle/postproc.py.
* ``torchgeometry`` (un-vendored) is replaced by ``oracle.thirdparty.spatial_soft_argmax2d``
  and ``kornia`` by an empty stub (only its import is needed by demo_match.detect), so the
  sub-pixel columns of the ``*_subpix`` arrays are NOT reference-pinned (key
  ``unpinned_subpixel`` = 1 in the file).
"""
import hashlib
import os
import sys
import types
import warnings

import numpy as np
import torch
import yaml

REF = os.environ.get("BALF_REFERENCE") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _install_shims():
    from oracle import thirdparty

    class _SoftArgmax:
        def __init__(self, normalized_coordinates=True):
            assert not normalized_coordinates

        def __call__(self, patches):                       # [N,1,ps,ps] -> [N,1,2]
            n, _, ps, _ = patches.shape
            return torch.from_numpy(thirdparty.spatial_soft_argmax2d(patches.reshape(n, ps, ps))).view(n, 1, 2)

    tgm = types.ModuleType("torchgeometry")
    tgm.contrib = types.SimpleNamespace(SpatialSoftArgmax2d=_SoftArgmax)
    sys.modules["torchgeometry"] = tgm
    kornia = types.ModuleType("kornia")
    kornia.feature = types.SimpleNamespace()
    sys.modules["kornia"] = kornia
    sys.modules.setdefault("cv2", types.ModuleType("cv2"))


class stable_argsort:
    def __enter__(self):
        self._orig = np.argsort
        np.argsort = lambda a, *x, **k: self._orig(a, *x, **{**k, "kind": "stable"})

    def __exit__(self, *e):
        np.argsort = self._orig


def ref_modules():
    sys.path.insert(0, REF)
    _install_shims()
    warnings.filterwarnings("ignore")
    from balf.model import get_model
    from balf.utils import test_utils
    from third_party.hardnet.hardnet_pytorch import HardNet
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        from demo import demo_match
    finally:
        os.chdir(cwd)
    cfg = yaml.safe_load(open(os.path.join(REF, "balf/configs/test.yaml")))
    return get_model, test_utils, HardNet, demo_match, cfg


def weight_digest(sd):
    """order-independent digest of a state_dict: (sum, sum of squares) in float64."""
    s = sum(float(v.double().sum()) for v in sd.values())
    q = sum(float((v.double() ** 2).sum()) for v in sd.values())
    return np.array([s, q, float(len(sd))])


def state_dict_fingerprint(sd):
    """key order, shape, dtype and SHA-256 of the bytes of every tensor of a state_dict: pins it bit for bit in a few KB
    (the tensors themselves would take ~10 MB)."""
    return {"keys": np.array(list(sd)),
            "shapes": np.array([",".join(map(str, v.shape)) for v in sd.values()]),
            "dtypes": np.array([str(v.dtype) for v in sd.values()]),
            "sha256": np.array([hashlib.sha256(v.detach().cpu().contiguous().numpy().tobytes()).hexdigest()
                                for v in sd.values()])}


def save_score_planes(path, score):
    """a float32 map as its four little-endian byte planes: planes compress where interleaved floats do not, which keeps
    the 480x640 map under 1 MB (tests/conftest.py: load_score_480x640 rebuilds it bit for bit)."""
    planes = np.ascontiguousarray(score, "<f4").view(np.uint8).reshape(-1, 4).T.copy()
    np.savez_compressed(path, score_480x640_planes=planes)


def synth_image_u8(h, w, seed, channels=1):
    """SURVEY.md section 8d: seeded uint8 image, gray plane replicated to 3 channels."""
    g = torch.Generator().manual_seed(seed)
    u8 = torch.randint(0, 256, (channels, h, w), generator=g, dtype=torch.uint8)
    return u8.permute(1, 2, 0).expand(h, w, 3).contiguous().numpy() if channels == 1 else \
        u8.permute(1, 2, 0).contiguous().numpy()


def main():
    get_model, tu, HardNet, demo_match, cfg = ref_modules()
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)

    # ------------------------------------------------------------------ detector
    torch.manual_seed(0)
    det = get_model.load_model(cfg["model"]).eval()
    sd = det.state_dict()
    x = torch.rand(1, 3, 128, 192, generator=torch.Generator().manual_seed(1234))
    with torch.inference_mode():
        o = det(x)
    # batch-2 non-square case with a different seed (checks per-image SE pooling / grid cells)
    x2 = torch.rand(2, 3, 64, 128, generator=torch.Generator().manual_seed(77))
    with torch.inference_mode():
        o2 = det(x2)
    xb = torch.rand(1, 3, 512, 640, generator=torch.Generator().manual_seed(1234))
    with torch.inference_mode():
        ob = det(xb)
    pb = ob["prob"][0].numpy()
    np.savez(os.path.join(OUT, "detector.npz"),
             weight_digest=weight_digest(sd),
             first_weight=sd["down1.conv.0.weight"].numpy(),
             head_bias=sd["detector_head.dense.bias"].numpy(),
             prob_128x192=o["prob"][0].numpy(), logits_128x192=o["logits"][0].numpy(),
             prob_b2_64x128=o2["prob"].numpy(), logits_b2_64x128=o2["logits"].numpy(),
             prob_512x640_sub8=pb[::8, ::8].copy(), prob_512x640_row255=pb[255].copy(),
             prob_512x640_stats=np.array([pb.astype(np.float64).sum(), pb.min(), pb.max(), pb.mean()]),
             logits_512x640_stats=np.array([ob["logits"].double().sum().item(), ob["logits"].abs().max().item()]))

    # ------------------------------------------------------------------ post-processing on the reference's own score map
    score = pb[16:496].copy()                                  # un-pad crop of a 480x640 image (P1)
    g = {"score_480x640": score, "unpinned_subpixel": np.array(1)}
    with stable_argsort():
        rb = tu.remove_borders(score, 15)
        g["apply_nms15_idx"] = np.flatnonzero(tu.apply_nms(rb, 15)).astype(np.int32)
        g["apply_nms4_idx"] = np.flatnonzero(tu.apply_nms(rb, 4)).astype(np.int32)
        nmsmap = tu.apply_nms(rb, 15)
        for k in (2048, 500, 5000):
            g["kth_topk%d" % k] = tu.get_point_coordinates(nmsmap, num_points=k)
        for name, thr in (("thr001", 0.001), ("thr015", 0.015)):
            g["greedy_" + name] = tu.get_points_direct_from_score_map(rb, thr, 15, False, 4)
        g["greedy_thr001_r4"] = tu.get_points_direct_from_score_map(rb, 0.001, 4, False, 4)
        g["greedy_thr001_subpix4"] = tu.get_points_direct_from_score_map(rb, 0.001, 15, True, 4)
        g["greedy_thr015_subpix5"] = tu.get_points_direct_from_score_map(rb, 0.015, 15, True, 5)
        ys, xs = np.where(rb >= np.float32(0.001))
        pts = np.stack([xs, ys, rb[ys, xs]]).astype(np.float64)
        out, inds = tu.nms_fast(pts, 480, 640, 15)
        g["nms_fast_out"], g["nms_fast_inds"] = out, inds.astype(np.int64)
    save_score_planes(os.path.join(OUT, "postproc_480x640_score.npz"), g.pop("score_480x640"))
    np.savez_compressed(os.path.join(OUT, "postproc_480x640.npz"), **g)

    # ------------------------------------------------------------------ small synthetic maps: ties, plateaus, zeros, edge cases
    rng = np.random.default_rng(7)
    small = {}
    maps = {
        "rand": rng.random((96, 128), dtype=np.float32),
        "quant": (rng.integers(0, 12, (96, 128)) / 16.0).astype(np.float32),          # heavy ties + plateaus
        "sparse": (rng.random((96, 128), dtype=np.float32) * (rng.random((96, 128)) > 0.97)).astype(np.float32),
        "zeros": np.zeros((96, 128), np.float32),
        "odd": rng.random((75, 101), dtype=np.float32),
        "one": np.zeros((64, 64), np.float32),
    }
    maps["one"][40, 21] = 0.5
    with stable_argsort():
        for name, m in maps.items():
            small["map_" + name] = m
            b = 15 if name != "rand" else 4
            rb = tu.remove_borders(m, b)
            small["rb_" + name] = np.array(b)
            for size in (15, 4, 3):
                small["nms%d_%s" % (size, name)] = np.flatnonzero(tu.apply_nms(rb, size)).astype(np.int32)
            nm = tu.apply_nms(rb, 15)
            for k in (1, 50, 2048):
                small["kth%d_%s" % (k, name)] = tu.find_index_higher_scores(nm, num_points=k).astype(np.int32)
                small["kthraw%d_%s" % (k, name)] = tu.find_index_higher_scores(rb, num_points=k).astype(np.int32)
            for r in (15, 4, 1):
                small["greedy%d_%s" % (r, name)] = tu.get_points_direct_from_score_map(rb, 0.015, r, False, 4)
    np.savez(os.path.join(OUT, "postproc_small.npz"), **small)

    # ------------------------------------------------------------------ D0: pad geometry + full detect() of the reference on synthetic u8 images
    d = {}
    args = types.SimpleNamespace(border_size=15, nms_size=15, num_features=2048, s_mult=60, order_coord="xysr",
                                 heatmap_confidence_threshold=0.001, sub_pixel=False, patch_size=4)
    for (h, w, seed) in ((480, 640, 1234), (121, 187, 5), (128, 192, 6)):
        im = synth_image_u8(h, w, seed)
        pad = tu.mod_padding_symmetric(tu.make_shape_even(im / 255.0), 64)
        d["pad_shape_%dx%d" % (h, w)] = np.array(pad.shape)
        d["pad_sum_%dx%d" % (h, w)] = np.array([pad.astype(np.float32).astype(np.float64).sum()])
        if h < 480:
            d["pad_%dx%d" % (h, w)] = pad.astype(np.float32)
            with stable_argsort():
                d["detect_%dx%d" % (h, w)] = demo_match.detect(args, im, det, "cpu")
    np.savez(os.path.join(OUT, "detect.npz"), **d)

    # ------------------------------------------------------------------ HardNet
    torch.manual_seed(0)
    hn = HardNet().eval()
    xh = torch.rand(8, 1, 32, 32, generator=torch.Generator().manual_seed(4321))
    with torch.inference_mode():
        oh = hn(xh)
    np.savez(os.path.join(OUT, "hardnet.npz"), weight_digest=weight_digest(hn.state_dict()),
             first_weight=hn.state_dict()["features.0.weight"].numpy(), out=oh.numpy())
    fingerprints = {"detector": state_dict_fingerprint(sd), "hardnet": state_dict_fingerprint(hn.state_dict())}
    np.savez_compressed(os.path.join(OUT, "state_dict.npz"),
                        **{m + "_" + k: v for m, fp in fingerprints.items() for k, v in fp.items()})
    print("golden vectors written to", OUT)
    for f in sorted(os.listdir(OUT)):
        print("  %-28s %8d bytes" % (f, os.path.getsize(os.path.join(OUT, f))))


def ref_metric_modules():
    """balf/benchmark_test/{repeatability_tools,geometry_tools}.py imported from the reference (they import
    torchvision, which is present, and torchgeometry.core.warp_perspective, which is stubbed: unused by the functions run)."""
    import importlib.util
    tgm = sys.modules.get("torchgeometry") or types.ModuleType("torchgeometry")
    core = types.ModuleType("torchgeometry.core")
    core.warp_perspective = None
    tgm.core = core
    sys.modules["torchgeometry"] = tgm
    sys.modules["torchgeometry.core"] = core
    sys.modules.pop("cv2", None)                     # the real OpenCV (create_common_region_masks needs warpPerspective)
    import cv2  # noqa: F401
    mods = []
    for name in ("repeatability_tools", "geometry_tools"):
        path = os.path.join(REF, "balf/benchmark_test", name + ".py")
        # the metric functions sort with the ndarray METHOD ``x.argsort()`` (repeatability_tools.py:433, :456, :551), which
        # the np.argsort shim cannot reach: the module is executed from its source with exactly that call made stable
        # (same canonical tie rule as everywhere else); nothing else is changed
        src = open(path).read().replace(".argsort()", ".argsort(kind='stable')")
        m = types.ModuleType("ref_" + name)
        m.__file__ = path
        exec(compile(src, path, "exec"), m.__dict__)
        mods.append(m)
    return mods


def metric_inputs():
    """seeded keypoint sets and homographies for the repeatability goldens (also rebuilt by the tests)."""
    rng = np.random.default_rng(2024)
    Hm = np.array([[1.02, 0.03, 5.0], [-0.02, 0.98, -3.0], [1e-5, -2e-5, 1.0]])
    hs, ws = 240, 320
    n1 = 300
    src = np.stack([rng.integers(16, ws - 16, n1), rng.integers(16, hs - 16, n1), np.ones(n1), rng.random(n1)], 1).astype(np.float64)
    # dst image points: 200 true correspondences (src -> dst through H^-1, rounded to the pixel grid) + 80 random ones
    inv = np.linalg.inv(Hm)
    p = (inv @ np.stack([src[:200, 0], src[:200, 1], np.ones(200)], 0)).T
    corr = np.round(p[:, :2] / p[:, 2:]) + rng.integers(-2, 3, (200, 2))
    rnd = np.stack([rng.integers(16, ws - 16, 80), rng.integers(16, hs - 16, 80)], 1)
    dst_xy = np.concatenate([corr, rnd], 0)
    dst = np.concatenate([dst_xy, np.ones((280, 1)), rng.random((280, 1))], 1).astype(np.float64)
    src_ms = src.copy(); src_ms[:, 2] = rng.uniform(0.6, 3.0, n1)
    dst_ms = dst.copy(); dst_ms[:, 2] = rng.uniform(0.6, 3.0, 280)
    return Hm, (hs, ws), src, dst, src_ms, dst_ms


def main_r2():
    """Round-2 vectors (separate files; the round-1 files above stay bit-identical):
    r2_media.npz          media/im1.jpg, im2.jpg decoded by PIL (RGB and convert('L')) and the reference detect() on them
    r2_detector_large.npz reference score maps at 960x1216 (configs[2]) and 1024x1024 (configs[3]) + reference detect()
                          on the two 900x1200 images of configs[2]
    r2_hardnet2048.npz    reference HardNet on 2048 seeded patches
    r2_metrics.npz        reference repeatability metrics / homography helpers on seeded keypoint sets"""
    get_model, tu, HardNet, demo_match, cfg = ref_modules()
    from PIL import Image
    torch.set_num_threads(8)
    torch.manual_seed(0)
    det = get_model.load_model(cfg["model"]).eval()
    args = types.SimpleNamespace(border_size=15, nms_size=15, num_features=2048, s_mult=60, order_coord="xysr",
                                 heatmap_confidence_threshold=0.001, sub_pixel=False, patch_size=4)
    m = {}
    for name in ("im1", "im2"):
        im = Image.open(os.path.join(REF, "media", name + ".jpg"))          # demo_match.load_im (:13-19)
        rgb = np.asarray(im.convert("RGB")).copy()
        gray = np.asarray(im.convert("L")).copy()
        m["rgb_" + name], m["gray_" + name] = rgb, gray
        with stable_argsort():
            m["detect_" + name] = demo_match.detect(args, rgb, det, "cpu")
        pad = tu.mod_padding_symmetric(tu.make_shape_even(rgb / 255.0), 64)
        x = torch.tensor(pad, dtype=torch.float32).permute(2, 0, 1).unsqueeze(0)
        with torch.inference_mode():
            prob = det(x)["prob"][0].numpy()
        hs = prob.shape[0] // 2 - rgb.shape[0] // 2
        ws_ = prob.shape[1] // 2 - rgb.shape[1] // 2
        sc = tu.remove_borders(prob[hs:hs + rgb.shape[0], ws_:ws_ + rgb.shape[1]], 15)
        m["candidates_" + name] = np.array([(sc >= np.float32(0.001)).sum()])
        m["prob_sub8_" + name] = prob[::8, ::8].copy()
        m["prob_stats_" + name] = np.array([prob.astype(np.float64).sum(), prob.min(), prob.max()])
    np.savez_compressed(os.path.join(OUT, "r2_media.npz"), **m)

    d = {}
    for (h, w, seed) in ((900, 1200, 1234), (900, 1200, 1235), (1024, 1024, 1234)):
        im = synth_image_u8(h, w, seed)
        pad = tu.mod_padding_symmetric(tu.make_shape_even(im / 255.0), 64)
        x = torch.tensor(pad, dtype=torch.float32).permute(2, 0, 1).unsqueeze(0)
        with torch.inference_mode():
            prob = det(x)["prob"][0].numpy()
        key = "%dx%d_s%d" % (h, w, seed)
        d["pad_shape_" + key] = np.array(pad.shape)
        d["prob_sub8_" + key] = prob[::8, ::8].copy()
        d["prob_row_" + key] = prob[prob.shape[0] // 2 - 1].copy()
        d["prob_stats_" + key] = np.array([prob.astype(np.float64).sum(), prob.min(), prob.max()])
        if h == 900:
            with stable_argsort():
                d["detect_" + key] = demo_match.detect(args, im, det, "cpu")
    np.savez_compressed(os.path.join(OUT, "r2_detector_large.npz"), **d)

    torch.manual_seed(0)
    hn = HardNet().eval()
    xh = torch.rand(2048, 1, 32, 32, generator=torch.Generator().manual_seed(4321))
    with torch.inference_mode():
        oh = torch.cat([hn(xh[i:i + 256]) for i in range(0, 2048, 256)])
    np.savez_compressed(os.path.join(OUT, "r2_hardnet2048.npz"), out=oh.numpy())

    rt, gt = ref_metric_modules()
    Hm, (hs, ws), src, dst, src_ms, dst_ms = metric_inputs()
    r = {"H": Hm}
    with stable_argsort():
        d2s = gt.apply_homography_to_points(dst, Hm)
        r["dst_to_src"] = d2s
        r["dst_to_src_ms"] = gt.apply_homography_to_points(dst_ms, Hm)
        for tag, a_, b_ in (("unit", src, d2s), ("ms", src_ms, r["dst_to_src_ms"]), ("raw", src, dst)):
            for oe in (0.4, 0.2):
                res = rt.compute_repeatability(a_.copy(), b_.copy(), overlap_err=oe)
                pre = "rep_%s_oe%d_" % (tag, int(oe * 10))
                r[pre + "scalars"] = np.array([res["rep_single_scale"], res["rep_multi_scale"], res["num_points_single_scale"],
                                               res["num_points_multi_scale"], res["error_overlap_single_scale"],
                                               res["error_overlap_multi_scale"], res["total_num_points"], res["possible_matches"]], np.float64)
                r[pre + "corr"] = np.asarray(res["correspondences"], np.int64).reshape(-1, 2)
                r[pre + "corr_m"] = np.asarray(res["correspondences_m"], np.int64).reshape(-1, 2)
        kp = np.stack([src[:, 1], src[:, 0], src[:, 3]], 1)            # (row, col, prob)
        wkp = np.stack([dst[:, 1], dst[:, 0], dst[:, 3]], 1)
        # compute_resize_repeatability maps keypoints (x, y) -> H (x, y): the homography from the first image to the second
        Hs2d = np.linalg.inv(Hm)
        for k, thr in ((1000, 5), (150, 3), (50, 1)):
            res = rt.compute_resize_repeatability(kp.copy(), wkp.copy(), Hs2d, (hs, ws), (hs, ws), keep_k_points=k, distance_thresh=thr)
            r["resize_k%d_t%d" % (k, thr)] = np.array([res["repeatability"], res["localization_err"], res["common_src_num"],
                                                        res["common_dst_num"], res["rep_src_num"], res["rep_dst_num"]], np.float64)
    for i, Hx in enumerate((Hm, np.array([[0.9, -0.1, 30.0], [0.12, 1.05, -12.0], [2e-4, 1e-4, 1.0]]))):
        ms_, md_ = gt.create_common_region_masks(Hx, (hs, ws, 3), (hs + 16, ws - 24, 3))
        r["mask_H%d" % i] = Hx
        r["mask_src_%d" % i] = ms_.astype(np.uint8)
        r["mask_dst_%d" % i] = md_.astype(np.uint8)
    np.savez_compressed(os.path.join(OUT, "r2_metrics.npz"), **r)

    # box_nms (repeatability_tools.py:227-255) with torchvision's CPU nms in place of the hard-coded .cuda() call
    import torchvision
    bx = {}
    rngb = np.random.default_rng(99)
    for name, prob in (("rand", rngb.random((60, 80), dtype=np.float32) * 0.05),
                       ("ref", det(torch.rand(1, 3, 64, 128, generator=torch.Generator().manual_seed(5)))["prob"][0].detach().numpy())):
        for size, iou_, top in ((4, 0.1, -1), (4, 0.1, 40), (6, 0.3, -1)):
            p = torch.from_numpy(prob)
            pts = torch.stack(torch.where(p >= 0.015)).t()
            boxes = torch.cat((pts - size / 2.0, pts + size / 2.0), dim=1).to(torch.float32)
            scores = p[pts[:, 0], pts[:, 1]]
            # stable descending order first so that torchvision's own sort sees the canonical tie order
            order = torch.from_numpy(np.argsort(-scores.numpy(), kind="stable"))
            ind = torchvision.ops.nms(boxes[order], scores[order], iou_)
            ind = order[ind]
            if top > 0:
                ind = ind[:min(top, len(ind))]
            out = torch.zeros_like(p)
            out[pts[ind, 0], pts[ind, 1]] = scores[ind]
            key = "%s_s%d_i%d_k%d" % (name, size, int(iou_ * 10), max(top, 0))
            bx["prob_" + name] = prob
            bx["keep_" + key] = np.flatnonzero(out.numpy()).astype(np.int32)
    np.savez_compressed(os.path.join(OUT, "r2_boxnms.npz"), **bx)
    for f in sorted(os.listdir(OUT)):
        if f.startswith("r2_"):
            print("  %-28s %8d bytes" % (f, os.path.getsize(os.path.join(OUT, f))))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "r2":
        main_r2()
    else:
        main()
