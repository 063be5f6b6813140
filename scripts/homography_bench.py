"""RANSAC throughput: balf_find_homography_ransac (--model homography, the default), balf_find_fundamental_ransac
(--model fundamental) or balf_find_essential_ransac + balf_recover_pose (--model essential) on the GPU next to
cv2.findHomography(RANSAC) / cv2.findFundamentalMat(FM_RANSAC) / cv2.findEssentialMat(RANSAC) + cv2.recoverPose on the host.

Workloads: B = 64 synthetic pairs of M = 2048 and M = 8192 matches in a 1200x900 frame with 0.5 px noise, threshold 3 px.
homography: a seeded homography per pair, inlier ratio 0.3, 2000 hypotheses per pair.  fundamental: a seeded two-view
scene per pair (3-D points 4 - 10 units in front of camera 1, the second camera rotated by up to 0.1 rad and moved about
one unit), inlier ratio 0.5, 1000 hypotheses per pair (up to 3 models each).  essential: the same scenes with K given,
threshold 1 px (cv2's default), 1000 hypotheses per pair (up to 10 models each), then the pose of each pair.  GPU: warm-up, then CUDA events around enough calls for a window of at least a
second (ms per call, pairs/s), and the library's per-kernel event timing over a second window (kernel time, point
evaluations B * iters * M per second of kernel time; a fundamental hypothesis counts once although it scores up to 3
models).  CPU: cv2 over the same pairs, once with its default confidence (0.995 for the homography, 0.99 for the
fundamental matrix; adaptive iteration count: what a user calls) and once with confidence 1 - 1e-9 (every iteration at
these inlier ratios: the same work).
Prints one JSON line per workload with the card name and power limit read in the same run.

    python scripts/homography_bench.py [--model {homography,fundamental,essential}] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

W, H = 1200, 900


def synth_pairs(seed, B, M, ratio):
    rng = np.random.default_rng(seed)
    p1 = rng.uniform([0, 0], [W, H], (B, M, 2))
    p2 = np.empty_like(p1)
    k = int(round(ratio * M))
    for b in range(B):
        Hg = np.array([[1 + rng.uniform(-.1, .1), rng.uniform(-.1, .1), rng.uniform(-50, 50)],
                       [rng.uniform(-.1, .1), 1 + rng.uniform(-.1, .1), rng.uniform(-50, 50)],
                       [rng.uniform(-1e-4, 1e-4), rng.uniform(-1e-4, 1e-4), 1.0]])
        q = np.c_[p1[b], np.ones(M)] @ Hg.T
        p2[b] = q[:, :2] / q[:, 2:] + rng.normal(0, 0.5, (M, 2))
        p2[b, k:] = rng.uniform([0, 0], [W, H], (M - k, 2))
    return p1, p2


def synth_two_view(seed, B, M, ratio):
    rng = np.random.default_rng(seed)
    K = np.array([[800.0, 0, W / 2], [0, 800.0, H / 2], [0, 0, 1]])
    p1, p2 = np.empty((B, M, 2)), np.empty((B, M, 2))
    k = int(round(ratio * M))
    for b in range(B):
        X = np.c_[rng.uniform(-3, 3, (M, 2)), rng.uniform(4, 10, M)]
        v = rng.uniform(-0.1, 0.1, 3)
        a = np.linalg.norm(v)
        S = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]]) / a
        R = np.eye(3) + np.sin(a) * S + (1 - np.cos(a)) * S @ S
        t = np.array([1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)])
        q1, q2 = X @ K.T, (X @ R.T + t) @ K.T
        p1[b] = q1[:, :2] / q1[:, 2:]
        p2[b] = q2[:, :2] / q2[:, 2:] + rng.normal(0, 0.5, (M, 2))
        p2[b, k:] = rng.uniform([0, 0], [W, H], (M - k, 2))
    return p1, p2


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def time_calls(fn, min_s):
    """CUDA events around n back-to-back calls, n chosen for a window of at least min_s -> (ms per call, n)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n = max(10, int(min_s * 1e3 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", choices=("homography", "fundamental", "essential"), default="homography")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--min-window", type=float, default=1.0, help="seconds per timed GPU window")
    args = ap.parse_args()
    import cv2
    import balf_b200._capi as c
    dev = torch.device("cuda:0")
    name, power = card()
    fund, ess = args.model == "fundamental", args.model == "essential"
    B, thr = 64, 1.0 if ess else 3.0
    iters, ratio = (1000, 0.5) if fund or ess else (2000, 0.3)
    synth, estimate, prefix = ((synth_two_view, c.find_fundamental_ransac, ("fundamental",)) if fund else
                               (synth_two_view, None, ("essential", "recover_pose")) if ess else
                               (synth_pairs, c.find_homography_ransac, ("ransac",)))
    conf_default = 0.99 if fund else 0.999 if ess else 0.995
    K = np.array([[800.0, 0, W / 2], [0, 800.0, H / 2], [0, 0, 1]])
    lines = []
    for M in (2048, 8192):
        p1, p2 = synth(M, B, M, ratio)
        d1, d2 = torch.from_numpy(p1).to(dev), torch.from_numpy(p2).to(dev)
        cnt = torch.full((B,), M, dtype=torch.int32, device=dev)
        if ess:
            Kd = torch.from_numpy(np.tile(K, (B, 2, 1, 1))).to(dev)

            def call():
                E, mask, n_in = c.find_essential_ransac(d1, d2, cnt, Kd, thr, iters, 0)
                c.recover_pose(E, d1, d2, cnt, Kd, mask)
                return E, mask, n_in
        else:
            call = lambda: estimate(d1, d2, cnt, thr, iters, 0)
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        ms, n = time_calls(call, args.min_window)
        c.profile_enable(True)
        c.profile_report(reset=True)
        time_calls(call, args.min_window)
        torch.cuda.synchronize()
        prof = {k: v for k, v in c.profile_report(reset=True).items() if k.startswith(prefix)}
        c.profile_enable(False)
        kern = {k: v[1] / v[0] for k, v in prof.items()}
        kernel_ms = sum(kern.values())
        _, _, n_in = call()
        cpu = {}
        cpu_pairs = 16 if ess else B        # cv2's 5-point RANSAC takes about a second per pair of 8192 matches
        for arm, conf in (("default_confidence", conf_default), ("all_iterations", 1 - 1e-9)):
            t0 = time.perf_counter()
            if ess:
                inl = []
                for b in range(cpu_pairs):
                    E, m = cv2.findEssentialMat(p1[b], p2[b], K, cv2.RANSAC, conf, thr, maxIters=iters)
                    cv2.recoverPose(E[:3], p1[b], p2[b], K, mask=m)
                    inl.append(int(m.sum()))
            elif fund:
                inl = [int(cv2.findFundamentalMat(p1[b], p2[b], cv2.FM_RANSAC, thr, conf, iters)[1].sum()) for b in range(B)]
            else:
                inl = [int(cv2.findHomography(p1[b], p2[b], cv2.RANSAC, thr, maxIters=iters, confidence=conf)[1].sum())
                       for b in range(B)]
            dt = time.perf_counter() - t0
            cpu[arm] = {"ms_per_batch": dt * 1e3, "pairs_per_s": len(inl) / dt, "mean_inliers": float(np.mean(inl))}
            if ess:
                cpu[arm]["pairs"] = len(inl)
        rec = {"model": args.model, "workload": "B=%d M=%d iters=%d ratio=%.1f" % (B, M, iters, ratio), "card": name, "power_limit": power,
               "gpu_ms_per_call": ms, "gpu_calls_timed": n, "gpu_pairs_per_s": B / (ms * 1e-3),
               "kernel_ms": {k: round(v, 4) for k, v in kern.items()}, "kernel_ms_total": kernel_ms,
               "point_evals_per_s": B * iters * M / (kernel_ms * 1e-3), "gpu_mean_inliers": float(n_in.float().mean()),
               "cpu_cv2": cpu, "cpu_threads": cv2.getNumThreads(), "cpu_count": os.cpu_count()}
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
