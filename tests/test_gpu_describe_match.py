"""Parity of the descriptor stage on the GPU (through the C-ABI) with the oracle:
F1 patch sampling (balf_b200/csrc/patches.cu), H1 HardNet (hardnet.cu), M1 SMNN (match.cu), and the
public demo_match.extract_features / extract_matches chain.

Floating-point stages carry their tolerance here; match indices are bit-exact given the same
distance matrix (tie rule: lower index first).  The modules run on CUDA copies of the session fixtures, which stay on
the CPU for the tests that use them there."""
import contextlib
import copy

import numpy as np
import pytest
import torch

from conftest import load_golden, synth_u8
from oracle import hardnet as ohardnet
from oracle import pipeline, thirdparty

pytestmark = pytest.mark.gpu

PATCH_ATOL = 1e-4        # sample coordinates are fp32 at magnitudes up to ~600 px (ulp 6e-5 px) and noise images have
                         # unit gradients between neighbouring pixels; typical error is < 1e-6 (checked via the mean)
# Descriptor tolerances = 2x the error measured against the REFERENCE's own output on 2048 seeded patches
# (tests/golden/r2_hardnet2048.npz; scripts/measure_parity.py on B200): fp32 FFMA path max |err| 1.0e-6 (mean 1.0e-7); tensor-core
# path (tf32 operands, fp32 accumulate) max |err| 3.1e-4 (mean 5.2e-5) on unit-norm 128-d vectors (typical component 0.09).
DESC_ATOL = 5e-6         # fp32 path: the patch-sampled inputs of the demo chain have a wider dynamic range than rand() patches
DESC_ATOL_TC = 6e-4      # tensor-core (tf32 operand) HardNet path


def dev():
    return torch.device("cuda:0")


def capi():
    import balf_b200._capi as c
    return c


def hn_state(hardnet):
    return {k: v.detach().clone() for k, v in hardnet.state_dict().items()}


def on_gpu(module):
    return copy.deepcopy(module).to(dev())


# ------------------------------------------------------------------------------------------ F1
@pytest.mark.parametrize("h,w,seed", [(480, 640, 3), (481, 643, 4), (900, 1200, 5), (130, 97, 6)])
def test_patches_match_oracle(h, w, seed):
    g = torch.Generator().manual_seed(seed)
    gray = torch.randint(0, 256, (h, w), generator=g, dtype=torch.uint8)
    n = 257
    kp = torch.rand(n, 2, generator=g) * torch.tensor([w - 1.0, h - 1.0])
    kp[:4] = torch.tensor([[0.0, 0.0], [w - 1.0, h - 1.0], [0.0, h - 1.0], [w / 2.0, 0.25]])     # border clamping
    got = capi().extract_patches(gray.to(dev()), kp.to(dev()), 60.0, 32).cpu()
    laf = thirdparty.laf_from_center_scale_ori(kp, 60.0)
    want, level = thirdparty.extract_patches_from_pyramid(gray[None, None].float() / 255.0, laf, 32)
    assert int(level.max()) == int(level.min()) == capi().patch_pyramid_level(h, w, 60.0, 32)
    assert got.shape == want.shape == (n, 1, 32, 32)
    np.testing.assert_allclose(got.numpy(), want.numpy(), atol=PATCH_ATOL, rtol=0)
    assert np.abs(got.numpy() - want.numpy()).mean() < 1e-6


def test_patches_other_levels():
    g = torch.Generator().manual_seed(11)
    gray = torch.randint(0, 256, (300, 400), generator=g, dtype=torch.uint8)
    kp = torch.rand(64, 2, generator=g) * torch.tensor([399.0, 299.0])
    for s_mult in (10.0, 16.0, 130.0):                       # level 0 (no pyramid), 0/1 boundary, level 3
        got = capi().extract_patches(gray.to(dev()), kp.to(dev()), s_mult, 32).cpu()
        laf = thirdparty.laf_from_center_scale_ori(kp, s_mult)
        want, level = thirdparty.extract_patches_from_pyramid(gray[None, None].float() / 255.0, laf, 32)
        assert int(level[0]) == capi().patch_pyramid_level(300, 400, s_mult, 32)
        np.testing.assert_allclose(got.numpy(), want.numpy(), atol=PATCH_ATOL, rtol=0)


def test_patches_batched_counts():
    g = torch.Generator().manual_seed(12)
    gray = torch.randint(0, 256, (3, 200, 264), generator=g, dtype=torch.uint8)
    kp = torch.rand(3, 40, 2, generator=g) * torch.tensor([263.0, 199.0])
    cnt = torch.tensor([40, 0, 17], dtype=torch.int32)
    got = capi().extract_patches_batch(gray.to(dev()), kp.to(dev()), cnt.to(dev()), 60.0, 32).cpu()
    for b in range(3):
        n = int(cnt[b])
        assert torch.count_nonzero(got[b, n:]) == 0
        if n:
            laf = thirdparty.laf_from_center_scale_ori(kp[b, :n], 60.0)
            want, _ = thirdparty.extract_patches_from_pyramid(gray[b][None, None].float() / 255.0, laf, 32)
            np.testing.assert_allclose(got[b, :n].numpy(), want[:, 0].numpy(), atol=PATCH_ATOL, rtol=0)


# ------------------------------------------------------------------------------------------ H1
def test_hardnet_golden(hardnet):
    g = load_golden("hardnet.npz")
    x = torch.rand(8, 1, 32, 32, generator=torch.Generator().manual_seed(4321))
    hn = on_gpu(hardnet)
    with torch.inference_mode():
        got = hn(x.to(dev())).cpu().numpy()
    tol = DESC_ATOL if getattr(hn, "precision", "fp32") == "fp32" else DESC_ATOL_TC
    np.testing.assert_allclose(got, g["out"], atol=tol, rtol=0)                     # the reference's own output
    np.testing.assert_allclose(np.linalg.norm(got, axis=1), 1.0, atol=1e-5)


def test_hardnet_reference_golden_2048(hardnet):
    """the reference's own HardNet output on 2048 seeded patches (two internal passes of the chunked reference loop)"""
    want = load_golden("r2_hardnet2048.npz")["out"]
    x = torch.rand(2048, 1, 32, 32, generator=torch.Generator().manual_seed(4321))
    hn = on_gpu(hardnet)
    with torch.inference_mode():
        got = hn(x.to(dev())).cpu().numpy()
    tc = getattr(hn, "precision", "fp32") != "fp32"
    err = np.abs(got - want)
    assert err.max() <= (DESC_ATOL_TC if tc else 2.5e-6), err.max()
    assert err.mean() <= (1.1e-4 if tc else 2.5e-7), err.mean()
    cos = (got * want).sum(1)
    assert cos.min() > 1 - 2e-6


@pytest.mark.parametrize("n", [1, 7, 1000, 1337])
def test_hardnet_matches_oracle(hardnet, n):
    g = torch.Generator().manual_seed(100 + n)
    x = torch.rand(n, 1, 32, 32, generator=g)
    x[0] = x[0] * 0.01 + 0.5                                                      # low-contrast patch (input_norm)
    hn = on_gpu(hardnet)
    with torch.inference_mode():
        got = hn(x.to(dev())).cpu()
        want = ohardnet.hardnet_forward(hn_state(hardnet), x)
    tol = DESC_ATOL if getattr(hn, "precision", "fp32") == "fp32" else DESC_ATOL_TC
    np.testing.assert_allclose(got.numpy(), want.numpy(), atol=tol, rtol=0)


def test_hardnet_rejects_cpu_and_training(hardnet):
    hn = on_gpu(hardnet)
    with pytest.raises(RuntimeError):
        hn(torch.zeros(2, 1, 32, 32))
    hn.train()
    with pytest.raises(RuntimeError):
        hn(torch.zeros(2, 1, 32, 32, device=dev()))


# ------------------------------------------------------------------------------------------ M1
MATCH_PATHS = {"tc": 0, "ffma": 1}       # the two distance kernels: 3xTF32 tensor cores, fp32 FFMA (balf_debug_set key 3)


@contextlib.contextmanager
def on_match_path(path):
    capi().debug_set(3, MATCH_PATHS[path])
    try:
        yield path
    finally:
        capi().debug_set(3, 0)


@pytest.fixture(params=list(MATCH_PATHS))
def match_path(request):
    """the M1 tests run on both distance kernels"""
    with on_match_path(request.param):
        yield request.param


def unit_rows(n, seed, dup_of=None):
    g = torch.Generator().manual_seed(seed)
    d = torch.randn(n, 128, generator=g)
    if dup_of is not None:                         # correlated sets so that mutual matches exist
        m = min(n, dup_of.shape[0]) // 2
        d[:m] = dup_of[torch.randperm(dup_of.shape[0], generator=g)[:m]] + 0.15 * torch.randn(m, 128, generator=g)
    return d / d.norm(dim=1, keepdim=True)


@pytest.mark.parametrize("n1,n2", [(2048, 2048), (1000, 777), (65, 300), (2, 2), (2, 9)])
def test_smnn_bit_exact_on_same_distance_matrix(match_path, n1, n2):
    d1 = unit_rows(n1, 1)
    d2 = unit_rows(n2, 2, dup_of=d1)
    dist, ids, dm = capi().match_smnn(d1.to(dev()), d2.to(dev()), 0.99, want_dm=True)
    want_dist, want_ids = thirdparty.match_smnn(d1, d2, 0.99, dm=dm.cpu())
    assert len(want_ids) > 0 or min(n1, n2) < 3
    np.testing.assert_array_equal(ids.cpu().numpy(), want_ids.numpy())
    np.testing.assert_array_equal(dist.cpu().numpy(), want_dist.numpy())
    # the distance matrix itself vs torch.cdist (different summation order): tolerance, not bits
    np.testing.assert_allclose(dm.cpu().numpy(), thirdparty.distance_matrix(d1, d2).numpy(), atol=2e-5, rtol=0)


def test_smnn_agreement_with_own_distances():
    d1 = unit_rows(2048, 3)
    d2 = unit_rows(2048, 4, dup_of=d1)
    _, want = thirdparty.match_smnn(d1, d2, 0.99)
    b = set(map(tuple, want.numpy()))
    assert len(b) > 500
    for path in MATCH_PATHS:
        with on_match_path(path):
            _, ids = capi().match_smnn(d1.to(dev()), d2.to(dev()), 0.99)
        a = set(map(tuple, ids.cpu().numpy()))
        assert len(a & b) / len(b) >= 0.99 and len(a & b) / max(len(a), 1) >= 0.99, path


def test_smnn_ties_and_degenerate():
    d = unit_rows(64, 5)
    d1 = torch.cat([d, d[:8]])                     # duplicated rows -> exactly equal distances
    for path in MATCH_PATHS:
        with on_match_path(path):
            dist, ids, dm = capi().match_smnn(d1.to(dev()), d.to(dev()), 0.99, want_dm=True)
            want_dist, want_ids = thirdparty.match_smnn(d1, d, 0.99, dm=dm.cpu())
            np.testing.assert_array_equal(ids.cpu().numpy(), want_ids.numpy())
            for n1, n2 in ((0, 5), (1, 5), (5, 1)):
                dist, ids = capi().match_smnn(torch.zeros(n1, 128, device=dev()), torch.zeros(n2, 128, device=dev()), 0.99)
                assert ids.shape == (0, 2) and dist.shape == (0, 1)


# ------------------------------------------------------------------------------------------ demo chain
def test_extract_features_and_matches(detector, detector_sd, hardnet):
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    args = config.default_test_args()
    det, hn = on_gpu(detector), on_gpu(hardnet)
    rgb1 = synth_u8(200, 264, 21)
    noise = np.random.default_rng(5).integers(-2, 3, rgb1.shape[:2])[..., None]
    rgb2 = np.clip(rgb1.astype(np.int64) + noise, 0, 255).astype(np.uint8)
    gray1, gray2 = rgb1[..., 0].copy(), rgb2[..., 0].copy()
    k1, d1 = demo_match.extract_features(args, rgb1, gray1, det, hn, dev())
    assert k1.shape[1] == 2 and d1.shape == (len(k1), 128)
    # oracle descriptors at the SAME keypoints (isolates F1 + H1 from detector tolerance)
    hn_sd = hn_state(hardnet)
    want_d, _ = pipeline.describe(args, hn_sd, gray1, k1)
    tol = 1e-4 if getattr(hn, "precision", "fp32") == "fp32" else DESC_ATOL_TC
    np.testing.assert_allclose(d1, want_d, atol=tol, rtol=0)
    p1, p2 = demo_match.extract_matches(args, rgb1, gray1, rgb2, gray2, det, hn, dev())
    assert p1.shape == p2.shape and p1.shape[1] == 2
    w1, w2 = pipeline.extract_matches(args, detector_sd, hn_sd, rgb1, gray1, rgb2, gray2)
    got = set(map(tuple, np.round(np.concatenate([p1, p2], 1), 2)))
    want = set(map(tuple, np.round(np.concatenate([w1, w2], 1), 2)))
    assert len(want) > 20
    # measured 1.000 / 1.000 (scripts/measure_parity.py): the demo path runs the detector in its fp32-class default
    assert len(got & want) / len(want) >= 0.99 and len(got & want) / len(got) >= 0.99
