import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session", autouse=True)
def _built_library():
    """The product library must exist before anything imports balf_b200."""
    import __graft_entry__
    __graft_entry__.build()


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name))


def load_score_480x640():
    """The reference's score map of a 480x640 image (tests/golden/postproc_480x640_score.npz), rebuilt bit for bit from
    the four byte planes it is stored as (oracle/make_golden.py: save_score_planes)."""
    planes = load_golden("postproc_480x640_score.npz")["score_480x640_planes"]
    return np.ascontiguousarray(planes.T).view("<f4").reshape(480, 640)


@pytest.fixture(scope="session")
def golden():
    return load_golden


@pytest.fixture(scope="session")
def model_cfg():
    from balf_b200.utils import test_utils
    from balf_b200.configs import config
    return test_utils.get_cfg_from_yaml_file(config.DEFAULT_CFG)["model"]


@pytest.fixture(scope="session")
def detector(model_cfg):
    """drop-in detector with the torch.manual_seed(0) initial weights (== reference init)."""
    from balf_b200.model import get_model
    torch.manual_seed(0)
    return get_model.load_model(model_cfg).eval()


@pytest.fixture(scope="session")
def detector_sd(detector):
    return {k: v.detach().clone() for k, v in detector.state_dict().items()}


@pytest.fixture(scope="session", params=["fp16", "tf32", "fp32"])
def hardnet(request):
    """HardNet with the reference's random init (seed 0), once per precision of balf_hardnet_forward."""
    from balf_b200.third_party.hardnet.hardnet_pytorch import HardNet
    torch.manual_seed(0)
    hn = HardNet().eval()
    hn.precision = request.param
    return hn


def weight_digest(sd):
    s = sum(float(v.double().sum()) for v in sd.values())
    q = sum(float((v.double() ** 2).sum()) for v in sd.values())
    return np.array([s, q, float(len(sd))])


def synth_u8(h, w, seed):
    """SURVEY.md 8d: seeded uint8 gray image replicated to 3 channels, [H,W,3]."""
    g = torch.Generator().manual_seed(seed)
    u8 = torch.randint(0, 256, (1, h, w), generator=g, dtype=torch.uint8)
    return u8.permute(1, 2, 0).expand(h, w, 3).contiguous().numpy()
