"""The gray-image forward (balf_detector_forward_gray: stage 1 from per-byte tables, a padded byte plane as input) against the
fp32-input forward at precision 'tf32' on preprocess_u8 of the same image.  The tables are built by the same device code that
the fp32-input kernels run per pixel, so the bar is bit equality of prob and logits, not a tolerance."""
import copy

import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def det(detector):
    return copy.deepcopy(detector).to(DEV).eval()


def both(det, u8):
    """u8 [B,H,W,1] uint8 -> ((logits, prob) of the fp32-input forward, (logits, prob) of forward_gray)"""
    import balf_b200._capi as capi
    u8 = u8.to(DEV)
    x, tl = capi.preprocess_u8(u8)
    g, tl_g = capi.pad_gray_u8(u8)
    assert tl == tl_g
    with torch.inference_mode():
        ref = det(x, precision="tf32", want_logits=True)
        got = det.forward_gray(g, precision="tf32", want_logits=True)
    torch.cuda.synchronize()
    return (ref["logits"], ref["prob"]), (got["logits"], got["prob"])


def assert_same(det, u8):
    (rl, rp), (gl, gp) = both(det, u8)
    assert torch.equal(gp, rp), "prob differs: max |d| = %g" % (gp - rp).abs().max().item()
    assert torch.equal(gl, rl), "logits differ: max |d| = %g" % (gl - rl).abs().max().item()


def test_random_bytes_cover_every_value(det):
    gen = torch.Generator().manual_seed(5)
    u8 = torch.randint(0, 256, (2, 128, 192, 1), generator=gen, dtype=torch.uint8)
    u8.view(-1)[:256] = torch.arange(256, dtype=torch.uint8)
    assert torch.unique(u8).numel() == 256
    assert_same(det, u8)


@pytest.mark.parametrize("value", [0, 1, 128, 255])
def test_constant_images(det, value):
    assert_same(det, torch.full((2, 128, 128, 1), value, dtype=torch.uint8))


def test_media_images(det):
    g = load_golden("r2_media.npz")
    u8 = torch.from_numpy(np.stack([g["gray_im1"], g["gray_im2"]])[..., None].copy())
    assert_same(det, u8)


@pytest.mark.parametrize("b,h,w", [(3, 64, 64), (2, 479, 639), (64, 480, 640), (1, 900, 1200), (2, 1024, 1024)])
def test_sizes(det, b, h, w):
    gen = torch.Generator().manual_seed(h * 7 + w)
    assert_same(det, torch.randint(0, 256, (b, h, w, 1), generator=gen, dtype=torch.uint8))


def test_batch_split_over_internal_passes(det):
    import balf_b200._capi as capi
    gen = torch.Generator().manual_seed(11)
    u8 = torch.randint(0, 256, (7, 96, 160, 1), generator=gen, dtype=torch.uint8)
    (_, whole), _ = both(det, u8)
    capi.debug_set(1, 3)                # passes of 3 + 3 + 1 images
    try:
        (rl, rp), (gl, gp) = both(det, u8)
    finally:
        capi.debug_set(1, 0)
    assert torch.equal(gp, rp) and torch.equal(gl, rl)
    assert torch.equal(gp, whole)


def test_weights_modified_in_place(detector):
    d = copy.deepcopy(detector).to(DEV).eval()
    gen = torch.Generator().manual_seed(2)
    u8 = torch.randint(0, 256, (2, 128, 128, 1), generator=gen, dtype=torch.uint8)
    (_, before), _ = both(d, u8)
    with torch.no_grad():               # stage-1 weights the table is built from, and one it is not
        sd = d.state_dict()
        for k in ("down1.conv.0.weight", "down1.residual_split_head_multi_axis_gmlp_layer.grid_gmlp_layer.dense1.bias",
                  "down1.residual_split_head_multi_axis_gmlp_layer.block_gmlp_layer.block_gating_unit.norm.weight",
                  "down1.residual_split_head_multi_axis_gmlp_layer.dense2.weight"):
            sd[k].add_(0.05 * torch.randn(sd[k].shape, generator=gen).to(DEV))
    (rl, rp), (gl, gp) = both(d, u8)
    assert not torch.equal(rp, before)
    assert torch.equal(gp, rp) and torch.equal(gl, rl)


def test_detect_batch_device_records_match_the_fp32_input_path(det):
    import balf_b200._capi as capi
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    args = config.default_test_args(sub_pixel=False, num_features=2048)
    d = copy.deepcopy(det)
    d.precision = "auto"                # resolves to 'tf32' for the windowed extraction
    gen = torch.Generator().manual_seed(9)
    u8 = torch.randint(0, 256, (4, 479, 639, 1), generator=gen, dtype=torch.uint8).to(DEV)
    got = demo_match.detect_batch_device(args, u8, d, "windowed")
    # the fp32-input path from public pieces, and a 3-channel replicated copy of the image (which takes that path)
    x, (top, left) = capi.preprocess_u8(u8)
    with torch.inference_mode():
        prob = d(x, precision="tf32", want_logits=False)["prob"]
    xy, sc, cnt = capi.windowed_nms_topk(prob, args.num_features, border=args.border_size, nms_size=args.nms_size,
                                         crop=(top, left, 479, 639))
    rgb = demo_match.detect_batch_device(args, u8.expand(-1, -1, -1, 3).contiguous(), d, "windowed")
    for want in ((xy, sc, None, cnt), rgb):
        assert torch.equal(got[3], want[3])
        for b in range(4):
            n = int(got[3][b])
            assert n > 0
            assert torch.equal(got[0][b, :n], want[0][b, :n]) and torch.equal(got[1][b, :n], want[1][b, :n])


def test_pad_gray_matches_preprocess_plane(det):
    import balf_b200._capi as capi
    # preprocess_u8's value of every byte (a 16x16 image of the 256 values), then both paths pixel by pixel: x = lut[g]
    x, (top, left) = capi.preprocess_u8(torch.arange(256, dtype=torch.uint8, device=DEV).reshape(1, 16, 16, 1))
    lut = x[0, 0, top:top + 16, left:left + 16].reshape(256)
    assert lut[0] == 0
    gen = torch.Generator().manual_seed(4)
    for h, w in ((64, 64), (479, 639), (120, 186)):
        u8 = torch.randint(0, 256, (2, h, w, 1), generator=gen, dtype=torch.uint8).to(DEV)
        x, tl = capi.preprocess_u8(u8)
        g, tl_g = capi.pad_gray_u8(u8)
        assert tl == tl_g and g.shape == (2,) + tuple(x.shape[2:])
        assert torch.equal(lut[g.long()], x[:, 0])


def test_argument_errors_launch_nothing(det):
    import balf_b200._capi as capi
    u8 = torch.randint(0, 256, (1, 64, 64, 1), dtype=torch.uint8, device=DEV)
    g, _ = capi.pad_gray_u8(u8)
    w = det._weights(torch.device(DEV))
    torch.cuda.synchronize()
    n0 = capi.launch_count()
    bad = [
        lambda: capi.pad_gray_u8(u8.float()),                                           # dtype
        lambda: capi.pad_gray_u8(u8.expand(-1, -1, -1, 3).contiguous()),                # C = 3
        lambda: capi.detector_forward_gray(g.to(torch.int16), w, det.arch, "tf32"),     # dtype
        lambda: capi.detector_forward_gray(g[:, :, :48].contiguous(), w, det.arch, "tf32"),   # Wp not a multiple of 64
        lambda: capi.detector_forward_gray(torch.zeros(1, 96, 64, dtype=torch.uint8, device=DEV), w, det.arch, "tf32"),  # Hp
        lambda: capi.detector_forward_gray(g, w, det.arch, "fp32"),                     # precision 0
        lambda: capi.detector_forward_gray(g, w, det.arch, "f16x3"),                    # precision 2
    ]
    for f in bad:
        with pytest.raises(ValueError):
            f()
    capi.debug_set(0, 0x1E)             # stage 1 sent to the FFMA kernels: not a gray-path configuration
    try:
        with pytest.raises(ValueError):
            capi.detector_forward_gray(g, w, det.arch, "tf32")
    finally:
        capi.debug_set(0, 0x1F)
    assert capi.launch_count() == n0
