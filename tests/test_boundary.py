"""Host-side contract of the drop-in boundary (CPU only: no compute calls)."""
import os

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle.make_golden import state_dict_fingerprint


def test_library_exports_every_declared_symbol():
    import balf_b200._capi as c
    names = set(c.declared_symbols())
    assert len(names) >= 15
    for n in names:
        assert hasattr(c._lib, n), n
    assert c.abi_version() == 1


def test_debug_set_rejects_unknown_keys():
    import balf_b200._capi as c
    for key in (-1, 4, 8):
        assert c.debug_set(key, 0) == -1, key
        assert "unknown debug key %d" % key in c._last_error().decode()


def test_state_dict_layout(detector, hardnet):
    sd = detector.state_dict()
    assert len(sd) == 167                                            # SURVEY.md appendix A
    assert sum(v.numel() for v in sd.values()) == 1280990
    assert sd["down1.conv.0.weight"].shape == (32, 3)
    assert sd["down4.residual_split_head_multi_axis_gmlp_layer.grid_gmlp_layer.grid_gating_unit.dense.weight"].shape == (64, 64)
    assert sd["down3.residual_channel_attention_block.calayer.excite.0.weight"].shape == (32, 128)
    assert sd["down2.conv2.bias"].shape == (64,)
    assert sd["detector_head.dense.weight"].shape == (65, 256)
    assert sd["detector_head.norm.num_batches_tracked"].dtype == torch.int64
    hs = hardnet.state_dict()
    assert len(hs) == 28 and hs["features.19.weight"].shape == (128, 128, 8, 8)
    assert sum(v.numel() for k, v in hs.items() if k.endswith("weight")) == 1334560


def test_state_dict_identical_to_reference(model_cfg, detector, hardnet):
    """Key order, shapes, dtypes and the bytes of every tensor of the seed-0 state_dicts against the reference's
    (tests/golden/state_dict.npz), and a state_dict of the reference's layout loads strictly."""
    from balf_b200.model import get_model
    g = load_golden("state_dict.npz")
    for name, sd in (("detector", detector.state_dict()), ("hardnet", hardnet.state_dict())):
        for field, got in state_dict_fingerprint(sd).items():
            np.testing.assert_array_equal(got, g[name + "_" + field], err_msg="%s %s" % (name, field))
    ref = {k: torch.zeros([int(n) for n in shape.split(",") if n], dtype=getattr(torch, dtype.split(".")[1]))
           for k, shape, dtype in zip(g["detector_keys"], g["detector_shapes"], g["detector_dtypes"])}
    get_model.load_model(model_cfg).load_state_dict(ref)             # reference checkpoints load strictly


def test_checkpoint_loader_contract(tmp_path, model_cfg):
    from balf_b200.model import get_model
    m = get_model.load_model(model_cfg)
    with pytest.raises(FileNotFoundError):
        get_model.load_test_pretrained_model(m, str(tmp_path / "missing.pth"))
    sd = {k: torch.full_like(v, 0.5) if v.is_floating_point() else v for k, v in m.state_dict().items()}
    path = str(tmp_path / "ckpt.pth")
    torch.save({"epoch": 7, "model_state": sd, "optimizer_state": None, "repeatability": 0.61}, path)
    epoch, rep = get_model.load_test_pretrained_model(m, path, device="cpu")
    assert (epoch, rep) == (7, 0.61)
    assert float(m.state_dict()["down2.conv.0.weight"].mean()) == 0.5
    del sd["down1.conv2.weight"]                                     # incomplete checkpoint -> AssertionError
    torch.save({"model_state": sd}, path)
    with pytest.raises(AssertionError):
        get_model.load_test_pretrained_model(m, path, device="cpu")


def test_unsupported_architecture_is_rejected(model_cfg):
    from balf_b200.model import get_model
    import copy
    cfg = copy.deepcopy(model_cfg)
    cfg["network_architecture"]["grid_size"] = [4, 4]
    with pytest.raises(ValueError):
        get_model.load_model(cfg)


def test_no_cpu_fallback(detector, hardnet):
    with pytest.raises(RuntimeError):
        detector(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError):
        hardnet(torch.zeros(2, 1, 32, 32))
    detector.train()
    with pytest.raises(RuntimeError):
        detector(torch.zeros(1, 3, 64, 64))
    detector.eval()


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dp, _, files in os.walk(os.path.join(root, "balf_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("oracle/", "").replace("the oracle", "").replace("oracle)", ""), os.path.join(dp, f)


def test_pad_geometry_host():
    import balf_b200._capi as c
    from oracle import postproc
    for h, w in ((480, 640), (900, 1200), (121, 187), (128, 192), (1, 1), (63, 65), (1024, 1024)):
        assert c.pad_geometry(h, w) == postproc.padded_geometry(h, w)[:4]
    with pytest.raises(ValueError):
        c.pad_geometry(0, 5)


def test_test_config_defaults():
    from balf_b200.configs import config
    args, cfg = config.parse_test_config([])
    assert (args.border_size, args.nms_size, args.num_features, args.s_mult, args.patch_size) == (15, 15, 2048, 60, 4)
    assert args.heatmap_confidence_threshold == 0.001 and args.sub_pixel is True and args.order_coord == "xysr"
    assert cfg["model"]["network_architecture"]["en_embed_dims"] == [3, 32, 64, 128, 256]


def test_front_end_and_multiscale_host_logic():
    """SURVEY 8(f) rows: level geometry is host arithmetic shared with the oracle; CPU tensors are refused (no fallback);
    the --nms switch rejects what is not built before touching the device."""
    import balf_b200._capi as c
    from balf_b200.utils import train_utils
    from oracle import multiscale as oms
    for n in (1024, 900, 480, 33):
        for s in (0.7, 0.5, 2 ** -0.5):
            for l in range(4):
                assert c.level_size(n, s, l) == oms.level_size(n, s, l)
    assert [c.level_size(1024, 0.7, l) for l in range(3)] == [1024, 717, 502]
    with pytest.raises(RuntimeError):
        c.rgb_to_gray(torch.zeros(4, 4, 3, dtype=torch.uint8))
    with pytest.raises(RuntimeError):
        c.preprocess_f32(torch.zeros(1, 64, 64, 3))
    with pytest.raises(RuntimeError):
        c.resize_preprocess_u8(torch.zeros(1, 64, 64, 1, dtype=torch.uint8), 45, 45)
    with pytest.raises(ValueError):
        train_utils.extract_detections_batch(torch.zeros(1, 64, 64, 1, dtype=torch.uint8), None, nms="bogus")
    assert set(train_utils.NMS_BACKENDS) == {"apply_nms", "nms_fast", "apply_nms_fast", "box_nms"}
