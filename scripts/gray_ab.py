"""Same-call A/B of the two stage-1 inputs of a gray batch: the fp32-input forward (preprocess_u8 -> balf_detector_forward) and
the byte-plane forward (pad_gray_u8 -> balf_detector_forward_gray), alternated step by step on the same 64 gray 480x640 images
(bench.py's flagship step: 'tf32' detector, windowed NMS, top-2048).  Reports ms / step of each under CUDA events, the per-kernel
times of each (balf_profile_*), the card and its power limit, and checks that prob and the keypoint records are bit-identical.

    python scripts/gray_ab.py [--rounds 8] [--steps 10] [--out results/gray_ab.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import balf_b200._capi as capi
    from balf_b200.configs import config
    from balf_b200.model import get_model
    from balf_b200.utils import test_utils
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    det = get_model.load_model(test_utils.get_cfg_from_yaml_file(config.DEFAULT_CFG)["model"]).eval().to(dev)
    args = config.default_test_args(sub_pixel=False, num_features=2048)
    gen = torch.Generator().manual_seed(1234)
    u8 = torch.randint(0, 256, (64, 480, 640, 1), generator=gen, dtype=torch.uint8).to(dev)

    def nms(prob, top, left):
        return capi.windowed_nms_topk(prob, args.num_features, border=args.border_size, nms_size=args.nms_size,
                                      crop=(top, left, 480, 640))

    def old():
        x, (top, left) = capi.preprocess_u8(u8)
        with torch.inference_mode():
            prob = det(x, precision="tf32", want_logits=False)["prob"]
        return prob, nms(prob, top, left)

    def new():
        g, (top, left) = capi.pad_gray_u8(u8)
        with torch.inference_mode():
            prob = det.forward_gray(g, precision="tf32")["prob"]
        return prob, nms(prob, top, left)

    po, ro = old()
    pn, rn = new()
    torch.cuda.synchronize()
    same = torch.equal(po, pn) and all(torch.equal(p, q) for p, q in zip(ro, rn))
    for _ in range(3):
        old(), new()
    ms = {"old": [], "new": []}
    prof = {"old": {}, "new": {}}
    capi.profile_enable(True)
    for _ in range(a.rounds):
        for name, fn in (("old", old), ("new", new)):
            capi.profile_report(reset=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / a.steps)
            for k, (n, t) in capi.profile_report(reset=True).items():
                prof[name][k] = prof[name].get(k, 0.0) + t / (a.steps * a.rounds)
    capi.profile_enable(False)
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    res = {"card": card(), "bit_identical": same, "ms_per_step_median": med, "ms_per_step": ms,
           "images_per_s": {k: 64 / (v * 1e-3) for k, v in med.items()}, "speedup": med["old"] / med["new"],
           "kernel_ms_per_step": {k: {"old": prof["old"].get(k), "new": prof["new"].get(k)}
                                  for k in sorted(set(prof["old"]) | set(prof["new"]),
                                                  key=lambda k: -max(prof["old"].get(k, 0), prof["new"].get(k, 0)))}}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    if not same:
        sys.exit("outputs differ between the two paths")


if __name__ == "__main__":
    main()
