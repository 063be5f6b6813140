#!/usr/bin/env python
"""Benchmark of record for the BALF inference hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch 64] [--nms windowed]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input on every rank:
uint8 images -> /255 + pad (D0) -> detector forward (D1-D3) -> border mask + NMS + top-2048
(P1-P8) -> keypoint records (and, for N > 1, one NCCL all-gather of the records).
Workload = BASELINE.json configs[1]: batch 64 synthetic grayscale 640x480 per GPU.

Prints ONE JSON line (rank 0).  ``value`` = whole-job images/s with the uint8 batch already in
HBM; ``e2e`` = the same metric through the public host-buffer API (``demo_match.DetectPipeline``, the streaming ``detect_batch``:
pinned host uint8 in, keypoint records back on the host, copies inside the timed region).
``--impl reference`` times the reference's CPU algorithm (the oracle restatement; the reference
itself cannot travel to the GPU box) on the box's host cores.
``--dump-outputs DIR`` writes what the timed path returned in its last step to DIR/<name>.npy (see dump_outputs):
the inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

import numpy as np
import torch

H, W, K_FEATURES = 480, 640, 2048
DUMP_LIMIT_BYTES = 64 * 10 ** 6 - 4096  # 64 MB of --dump-outputs, less room for the four .npy headers
METRIC = "images/sec detect+NMS+top-k @640x480"
FLOP_PER_PADDED_PIXEL = 119496          # SURVEY.md 8d (Linear / matmul MACs x 2 only)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    p.add_argument("--nms", default="windowed", choices=["windowed", "greedy"])
    p.add_argument("--precision", default=None, help="detector precision (default: the module's)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-extras", action="store_true", help="development / profiling: only the configs[1] workload")
    p.add_argument("--chunk", type=int, default=0, help="development: images per internal detector pass (library default if 0)")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


def workload_name(a):
    return ("configs[1]: batch %d synthetic grayscale 640x480 per GPU, detector + %s NMS + top-%d"
            % (a.batch, a.nms, K_FEATURES))


def config_of(a):
    """the `config` object of the JSON line -- identical for both arms (the reference arm runs the same workload one image
    at a time, the reference's own batching)."""
    return {"workload": workload_name(a), "batch_per_gpu": a.batch, "nms": a.nms, "k": K_FEATURES,
            "padded": "512x640", "weights": "random-init torch.manual_seed(0)",
            "l2": "no explicit flush: each step streams >2 GB of activations per GPU, far above the 126 MB L2"}


def synth_batch(batch, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (batch, H, W, 1), generator=g, dtype=torch.uint8)


def model_cfg():
    from balf_b200.configs import config
    from balf_b200.utils import test_utils
    return test_utils.get_cfg_from_yaml_file(config.DEFAULT_CFG)["model"]


def dump_outputs(path, xy, score, count):
    """The keypoint records the timed path returns (every rank's after the all-gather), as float32 (coordinates and
    counts are exact in it): xy.npy [N,K,2] (x, y), score.npy [N,K], count.npy [N]; rows beyond count are zero.
    image.npy [N] holds the batch index of each row: all images, or, when they would exceed 64 MB, a fixed sample of them
    (seed 0) that fits."""
    per_image = 4 * (xy[0].numel() + score[0].numel() + 2)
    n = len(count)
    image = np.arange(n)
    if n * per_image > DUMP_LIMIT_BYTES:
        image = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // per_image, replace=False))
    rows = torch.from_numpy(image).to(xy.device)
    os.makedirs(path, exist_ok=True)
    for name, t in (("xy", xy), ("score", score), ("count", count)):
        np.save(os.path.join(path, name + ".npy"), t.index_select(0, rows).cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, "image.npy"), image.astype(np.float32))


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_pipeline(a, nms=None, greedy_impl="python"):
    """-> callable(image index) running the reference algorithm (oracle port) on one image.  Imports nothing of the
    product: the weights are the oracle's own seeded replay of the reference constructors (oracle/weights.py)."""
    from oracle import pipeline, postproc, weights                    # the CPU arm only
    sd = weights.detector_state_dict(0)
    args = pipeline.default_args(sub_pixel=False)
    imgs = synth_batch(8, 1234).expand(8, H, W, 3).contiguous().numpy()
    nms = nms or a.nms
    greedy = postproc.greedy_nms                                       # the reference's Python loops (test_utils.py:130-168)
    if greedy_impl == "c":
        from oracle import postproc_c
        greedy = postproc_c.greedy_nms

    def one(i):
        im = imgs[i % len(imgs)]
        score = pipeline.score_map(sd, im)
        if nms == "windowed":
            return postproc.windowed_detect(score, args.border_size, args.nms_size, K_FEATURES)
        return pipeline.detect_from_score_map(args, score, nms=greedy)[0]
    return one


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    one = cpu_pipeline(a)
    per_step = 2
    for i in range(a.warmup):
        one(i)
    t0 = time.perf_counter()
    for s in range(a.steps):
        for j in range(per_step):
            one(s * per_step + j)
    dt = time.perf_counter() - t0
    v = a.steps * per_step / dt
    sample = "%d images per step, batch 1 each (the reference's own batching), %d steps" % (per_step, a.steps)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": config_of(a),
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def cpu_baseline(a, nms=None, greedy_impl="python", budget_s=10.0, max_images=32):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    one = cpu_pipeline(a, nms, greedy_impl)
    one(0)
    n, t0 = 0, time.perf_counter()
    while n < 3 or (time.perf_counter() - t0 < budget_s and n < max_images):
        one(n)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d images of the same workload (%s NMS%s), batch 1 each, %.1f s" %
                      (n, nms or a.nms, ", greedy loop = %s port" % greedy_impl if (nms or a.nms) == "greedy" else "", dt)}


# ------------------------------------------------------------------------------------------ roofline
def level_dims():
    hp, wp = 512, 640
    return [(3, 32, hp * wp), (32, 64, hp * wp // 4), (64, 128, hp * wp // 16), (128, 256, hp * wp // 64)]


def kernel_work(name, images):
    """Algorithmic work of ONE step's launches of kernel `name`: (flops, bytes).
    Detector kernels: Linear / token-mixing MACs x 2 counted once (recomputation is not credited; SURVEY.md 8d) and the
    fp32 tensors each kernel must read and write once (x, u, v, r, q: DESIGN.md section 3).  NMS: 4*H*W bytes per
    image (+ 16*K for the select/sort kernel)."""
    lv = {32: 0, 64: 1, 128: 2, 256: 3}
    if name.startswith("det_"):
        tail = name.rsplit("_c", 1)
        c = int(tail[1]) if len(tail) == 2 and tail[1].isdigit() else None
        if c in lv:
            cin, ch, px = level_dims()[lv[c]]
            n = images * px
            uv = 2 if ch <= 128 else 4                   # bytes per element of u' / v' in HBM (fp16 tiles at stages 1-3)
            rb = 2                                       # ... of r (fp16 at every stage)
            qb = 3 if ch <= 64 else 4                    # ... of q (24-bit planes at stages 1-2, fp32 above)
            xb = 4 if cin < 8 else 2                     # ... of the level input (the network input is fp32, pooled outputs fp16)
            if "branch" in name:                       # half of dense1, branch dense1, token mix, dense2; x in, u' out
                return n * (2 * cin * ch + 2 * ch * ch + 4 * ch * ch + 128 * ch + 2 * ch * ch), n * (xb * cin + uv * ch)
            if "merge" in name:                        # conv.0, dense2 (2C->C), conv1, conv2; x, u', v' in, r, q out
                return n * (2 * cin * ch + 4 * ch * ch + 4 * ch * ch), n * (xb * cin + 2 * uv * ch + rb * ch + qb * ch)
        if name == "det_head":                         # r (fp16), q in; prob out (64 values per 8x8 cell)
            n = images * level_dims()[3][2]
            return n * (2 * 256 * 256 + 2 * 256 * 65), n * (2 * 256 + 4 * 256 + 4 * 64)
        if name == "det_pool":                         # r (fp16), q in, pooled out (fp16, a quarter of the pixels), stages 1-3
            return 0, sum(images * px * (2 * ch + (3 if ch <= 64 else 4) * ch + ch // 2) for _, ch, px in level_dims()[:3])
        return 0, 0
    if name.startswith("nms_windowed"):
        return 0, images * (4 * H * W)
    if name == "nms_select_sort":
        return 0, images * 16 * K_FEATURES
    if name == "preprocess_u8":
        return 0, images * (H * W + 12 * 512 * 640)
    return 0, 0


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm": p["hbm_gbs"], "tensor": p["bf16_tflops_sustained"], "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tensor": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def ncu_traffic(name):
    """dram__bytes_read + dram__bytes_write per launch of kernel `name` from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by scripts/summarize_profiles.py), or None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        return json.load(open(path)).get(name)
    return None


def roofline_of(name, launches, total_ms, steps, images, pk):
    """The bound is the kernel's own: arithmetic intensity (algorithmic flops / algorithmic bytes) against the machine
    balance for tf32 operands (half the bf16 tensor peak / HBM peak) decides between "tensor" and "hbm"."""
    flops, nbytes = kernel_work(name, images)
    per_launch_s = total_ms / max(launches, 1) * 1e-3
    per = steps / max(launches, 1)
    balance = (pk["tensor"] / 2 * 1e12) / (pk["hbm"] * 1e9)
    if flops == 0 and nbytes == 0:
        return {"kernel": name, "bound": "latency", "launch_ms": per_launch_s * 1e3, "launches_per_step": launches / steps}
    kind = "tensor" if nbytes == 0 or (flops and flops / nbytes > balance) else "hbm"
    out = {"kernel": name, "bound": kind, "launch_ms": per_launch_s * 1e3, "launches_per_step": launches / steps,
           "peak_source": pk["src"], "traffic": ncu_traffic(name),
           "algorithmic": {"flops_per_launch": flops * per, "bytes_per_launch": nbytes * per,
                           "intensity_flop_per_byte": (flops / nbytes) if nbytes else None, "tf32_balance": balance}}
    if kind == "tensor":
        ach = flops * per / per_launch_s / 1e12
        out.update({"achieved": ach, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": ach / pk["tensor"],
                    "frac_of_tf32_peak": ach / (pk["tensor"] / 2)})
    else:
        ach = nbytes * per / per_launch_s / 1e9
        out.update({"achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"]})
        if flops:
            out["tensor_tflops"] = flops * per / per_launch_s / 1e12
    return out


def cuda_timed(fn, n=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def kernel_work_nms_greedy(images):
    """greedy path: the score map is read once by the first (threshold) pass; later rounds touch alive pixels only."""
    return images * (4 * H * W + 16 * K_FEATURES)


def extras_greedy(a, dev, pk, det, args, u8):
    """configs[1] with the demo path's NMS (greedy nms_fast, demo/demo_match.py:44-57): the same batch, device-timed, in the
    default precision of that path ('f16x3': fp32-class results on the tensor cores), on the fp32 FFMA kernels and with tf32
    opted in; per-kernel times of the NMS stage and its HBM
    fraction (algorithmic bytes: score map read once + 16 bytes per keypoint)."""
    import copy
    import balf_b200._capi as capi
    from balf_b200.demo import demo_match
    out = {}
    for prec in ("auto", "fp32", "tf32"):
        d = copy.copy(det)
        d.precision = prec
        ms = cuda_timed(lambda: demo_match.detect_batch_device(args, u8, d, "greedy"), n=3 if prec == "fp32" else 5)
        out["detector_%s" % d.resolve_precision("greedy")] = {"ms_per_step": ms, "images_per_s": a.batch / (ms * 1e-3)}
    with torch.inference_mode():
        x, (top, left) = capi.preprocess_u8(u8)
        prob = det(x, precision="tf32")["prob"]
    capi.profile_enable(True)
    capi.profile_report(reset=True)
    n = 10
    for _ in range(n):
        capi.greedy_nms_topk(prob, K_FEATURES, border=args.border_size, thr=args.heatmap_confidence_threshold,
                             radius=args.nms_size, subpixel_ps=0, crop=(top, left, H, W))
    prof = capi.profile_report(reset=True)
    capi.profile_enable(False)
    stage_ms = sum(v[1] for k, v in prof.items() if k.startswith("nms_")) / n
    nbytes = kernel_work_nms_greedy(a.batch)
    out["nms_stage"] = {"ms": stage_ms, "kernels": {k: v[1] / n for k, v in prof.items() if k.startswith("nms_")},
                        "bound": "hbm", "achieved": nbytes / (stage_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                        "frac": nbytes / (stage_ms * 1e-3) / 1e9 / pk["hbm"], "peak_source": pk["src"]}
    return out


def extras_pair(dev, det, n_pairs=4):
    """BASELINE.json configs[2]: HPatches-shaped synthetic pairs 1200x900 through demo_match.extract_matches end to end
    (HOST uint8 images in, matched point arrays out): detector x2, greedy NMS + sub-pixel, level-1 patches, HardNet x2,
    SMNN.  pairs/s over `n_pairs` pairs after one warm-up pair."""
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    from balf_b200.third_party.hardnet.hardnet_pytorch import HardNet
    torch.manual_seed(0)
    hn = HardNet().eval().to(dev)
    args = config.default_test_args()
    rng = np.random.default_rng(0)
    pairs = []
    for i in range(n_pairs + 1):
        g = torch.Generator().manual_seed(1234 + i)
        a_ = torch.randint(0, 256, (900, 1200, 1), generator=g, dtype=torch.uint8).expand(900, 1200, 3).contiguous().numpy()
        b_ = np.clip(a_.astype(np.int64) + rng.integers(-2, 3, (900, 1200, 1)), 0, 255).astype(np.uint8)
        pairs.append((a_, a_[..., 0].copy(), b_, b_[..., 0].copy()))
    res = {}
    for prec in ("auto", "fp32", "tf32"):
        import copy
        d = copy.copy(det)
        d.precision = prec
        demo_match.extract_matches(args, *pairs[0], d, hn, dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        nm = 0
        for pr in pairs[1:]:
            p1, _ = demo_match.extract_matches(args, *pr, d, hn, dev)
            nm += len(p1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        res["detector_%s" % d.resolve_precision("greedy")] = {"pairs_per_s": n_pairs / dt, "ms_per_pair": dt / n_pairs * 1e3,
                                                                 "matches_per_pair": nm / n_pairs}
    res["workload"] = "configs[2]: %d synthetic pairs 1200x900 (second image = first + noise), extract_matches, host buffers" % n_pairs
    res["h2d_bytes_per_pair"] = 2 * (900 * 1200 * 3 + 900 * 1200)
    return res


def extras_cfg3(dev, det, world, rank, gather, total=1024, chunk=64):
    """BASELINE.json configs[3]: `total` synthetic 1024x1024 images STRONG-scaled over the ranks (rank r takes a contiguous
    share), detector + windowed NMS + top-2048, keypoint records all-gathered per chunk through the C-ABI NCCL entry."""
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    from balf_b200.sharding import shard_range
    args = config.default_test_args(sub_pixel=False, num_features=K_FEATURES)
    lo, hi = shard_range(total, rank, world)
    n_local = hi - lo
    g = torch.Generator().manual_seed(1234 + rank)
    u8 = torch.randint(0, 256, (min(n_local, chunk), 1024, 1024, 1), generator=g, dtype=torch.uint8).to(dev)
    e_g0, e_g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run_pass(timed):
        gms = 0.0
        done = 0
        while done < n_local:
            b = min(chunk, n_local - done)
            xy, sc, _, cnt = demo_match.detect_batch_device(args, u8[:b], det, "windowed")
            if gather is not None and b == chunk:
                if timed:
                    e_g0.record()
                gather(xy, sc, cnt)
                if timed:
                    e_g1.record()
                    torch.cuda.synchronize()
                    gms += e_g0.elapsed_time(e_g1)
            done += b
        return gms
    run_pass(False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    gms = run_pass(True)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), gms, n_local


def extras_cfg4(dev, det, world, rank, total=256, chunk=32):
    """BASELINE.json configs[4]: 3-level pyramid (0.7x), 8192 keypoints per image, `total` 1024x1024 images over the ranks."""
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    from balf_b200.sharding import shard_range
    margs = config.default_test_args(sub_pixel=False, num_features=8192)
    lo, hi = shard_range(total, rank, world)
    n_local = hi - lo
    g = torch.Generator().manual_seed(4321 + rank)
    u8 = torch.randint(0, 256, (min(n_local, chunk), 1024, 1024, 1), generator=g, dtype=torch.uint8).to(dev)

    def run_pass():
        done = 0
        while done < n_local:
            b = min(chunk, n_local - done)
            demo_match.detect_multiscale_batch_device(margs, u8[:b], det, scale=0.7, levels=3)
            done += b
    run_pass()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_pass()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), n_local


def extras(dev, pk, det):
    """Secondary rows of the hot path (SURVEY.md 8a H1 / M1 / F1), not part of `value`: HardNet on 4096 patches, SMNN on
    2048 x 2048 descriptors, patch sampling, device-resident, CUDA-event timed."""
    import balf_b200._capi as capi
    from balf_b200.third_party.hardnet.hardnet_pytorch import HardNet
    torch.manual_seed(0)
    hn = HardNet().eval().to(dev)
    x = torch.rand(4096, 1, 32, 32, device=dev)
    out = {}
    with torch.inference_mode():
        ms = cuda_timed(lambda: hn(x))
        tf = 4096 * 78.184e6 / (ms * 1e-3) / 1e12
        out["hardnet"] = {"patches": 4096, "ms": ms, "patches_per_s": 4096 / (ms * 1e-3), "tflops": tf, "dtype": hn.precision,
                          "frac_of_tf32_peak": tf / (pk["tensor"] / 2), "peak": "half of the bf16 figure (%s)" % pk["src"]}
        d1 = torch.nn.functional.normalize(torch.randn(2048, 128, device=dev), dim=1)
        d2 = torch.nn.functional.normalize(d1 + 0.05 * torch.randn(2048, 128, device=dev), dim=1)
        ms = cuda_timed(lambda: capi.match_smnn(d1, d2, 0.99))
        out["smnn"] = {"n1": 2048, "n2": 2048, "ms": ms, "pairs_per_s": 2048 * 2048 / (ms * 1e-3),
                       "note": "includes the device->host read of the match count"}
        # F1: 2048 patches of one 900 x 1200 image (level-1 pyramid build + bilinear gather); algorithmic bytes =
        # source read + level write/read + patches written (SURVEY.md 8d)
        gray = torch.randint(0, 256, (900, 1200), dtype=torch.uint8, device=dev)
        kp = torch.stack([torch.rand(2048, device=dev) * 1100 + 50, torch.rand(2048, device=dev) * 800 + 50], 1)
        ms = cuda_timed(lambda: capi.extract_patches(gray, kp, 60.0, 32))
        nbytes = 900 * 1200 + 2 * 4 * 450 * 600 + 4096 * 2048
        out["patches"] = {"keypoints": 2048, "image": "900x1200", "ms": ms, "bound": "hbm", "achieved_GBs": nbytes / (ms * 1e-3) / 1e9,
                          "frac": nbytes / (ms * 1e-3) / 1e9 / pk["hbm"]}
    return out


# ------------------------------------------------------------------------------------------ main arm
def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    import balf_b200._capi as capi
    from balf_b200.configs import config
    from balf_b200.demo import demo_match
    from balf_b200.model import get_model
    from balf_b200.sharding import KeypointGather

    if a.chunk:
        capi.debug_set(1, a.chunk)
    torch.manual_seed(0)
    det = get_model.load_model(model_cfg()).eval().to(dev)
    if a.precision:
        det.precision = a.precision
    args = config.default_test_args(sub_pixel=False, num_features=K_FEATURES)
    host = synth_batch(a.batch, 1234 + rank).pin_memory()
    u8 = host.to(dev)
    gather = KeypointGather(dev) if world > 1 else None           # the C-ABI collective (balf_gather_keypoints on an ncclComm_t)

    def step_device():
        xy, sc, _, cnt = demo_match.detect_batch_device(args, u8, det, a.nms)
        if gather is not None:
            return gather(xy, sc, cnt)
        return xy, sc, cnt

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(a.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    capi.profile_enable(True)
    capi.profile_report(reset=True)
    l0 = capi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        out = step_device()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = capi.launch_count() - l0
    prof = capi.profile_report(reset=True)
    capi.profile_enable(False)
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, *out)

    # end to end through the host-buffer API: every step's uint8 batch goes pinned host -> device and its keypoint
    # records come back device -> host inside the timed region.  DetectPipeline is the streaming form of
    # demo_match.detect_batch: the copy of step i+1 overlaps the kernels of step i.
    pipe = demo_match.DetectPipeline(args, det, dev, a.nms)
    prev = None
    for _ in range(max(a.warmup, 3) + pipe.depth):      # warm up in the pipelined pattern itself: the staging ring and the
        cur = pipe.submit(host)                          # second in-flight device batch are allocated here, not in the timed passes
        if prev is not None:
            res = pipe.result(prev)
        prev = cur
    res = pipe.result(prev)
    e2e_passes = []
    for _ in range(3):                  # three passes of K steps; the MEDIAN is reported, all are listed
        barrier()
        t0 = time.perf_counter()
        prev = None
        for _ in range(a.steps):
            cur = pipe.submit(host)
            if prev is not None:
                res = pipe.result(prev)
            prev = cur
        res = pipe.result(prev)
        torch.cuda.synchronize()
        e2e_passes.append((time.perf_counter() - t0) * 1e3)
    t_e2e = float(np.median(e2e_passes))
    d2h = sum(int(r.nbytes) for r in res)

    # the other BASELINE.json configs (every rank takes part: cfg3 / cfg4 are sharded over the ranks)
    if a.no_extras:
        c3_ms = c3_gather_ms = c4_ms = float("nan")
        c3_local = c4_local = 0
    else:
        c3_ms, c3_gather_ms, c3_local = extras_cfg3(dev, det, world, rank, gather)
        c4_ms, c4_local = extras_cfg4(dev, det, world, rank)

    t = torch.tensor([ms, t_e2e, c3_ms, c3_gather_ms, c4_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, t_e2e, c3_ms, c3_gather_ms, c4_ms = (float(v) for v in t)
    if rank != 0:
        if gather is not None:
            gather.close()
        if world > 1:
            dist.destroy_process_group()
        return
    images = a.batch * world
    pk = peaks()
    total_kernel_ms = sum(v[1] for v in prof.values())
    kernels = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        r = roofline_of(k, v[0], v[1], a.steps, a.batch, pk)
        kernels[k] = {"launches_per_step": v[0] / a.steps, "ms_per_step": v[1] / a.steps, "share": v[1] / total_kernel_ms,
                      "bound": r["bound"], "achieved": r.get("achieved"), "unit": r.get("unit"), "frac": r.get("frac")}
    top = max(((k, v) for k, v in prof.items() if k.startswith(("det_", "nms_"))), key=lambda kv: kv[1][1])
    roof = roofline_of(top[0], top[1][0], top[1][1], a.steps, a.batch, pk)
    # the NMS + top-k stage the metric names: both kernels of the windowed path against the stage's algorithmic bytes
    nms_keys = [k for k in prof if k.startswith("nms_")]
    roof_nms = None
    if nms_keys:
        stage_ms = sum(prof[k][1] for k in nms_keys) / a.steps
        nbytes = a.batch * (4 * H * W + 16 * K_FEATURES)
        roof_nms = {"kernels": {k: prof[k][1] / a.steps for k in nms_keys}, "bound": "hbm", "stage_ms": stage_ms,
                    "algorithmic_bytes": nbytes, "achieved": nbytes / (stage_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                    "frac": nbytes / (stage_ms * 1e-3) / 1e9 / pk["hbm"], "peak_source": pk["src"],
                    "traffic": sum(filter(None, (ncu_traffic(k) for k in nms_keys))) or None}
    det_ms = sum(v[1] for k, v in prof.items() if k.startswith("det_")) / a.steps
    det_tf = a.batch * 512 * 640 * FLOP_PER_PADDED_PIXEL / (det_ms * 1e-3) / 1e12 if det_ms else None
    line = {
        "metric": METRIC, "value": images * a.steps / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
        "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": {"tf32": "fp16/tf32 operands (11-bit significand), fp32 accumulate",
                  "f16x3": "fp16 hi+lo operand pairs (3 MMAs per product), fp32 accumulate"}.get(det.resolve_precision(a.nms), det.resolve_precision(a.nms)),
        "data": "synthetic",
        "config": config_of(a),
        "clocks": clocks,
        "e2e": {"value": images * a.steps / (t_e2e * 1e-3), "unit": "images/s", "passes_ms": [round(x, 3) for x in e2e_passes],
                "reported": "median of the passes", "h2d_bytes_per_step": int(host.numel()), "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": roof,
        "roofline_nms": roof_nms,
        "detector": {"ms_per_step": det_ms, "tflops": det_tf,
                     "frac_of_tf32_peak": det_tf / (pk["tensor"] / 2) if det_tf else None,
                     "frac_of_f16_peak": det_tf / pk["tensor"] if det_tf else None,
                     "note": "every GEMM and the token mixing run as kind::f16 (fp16 operands); stage-1 conv.0 on the CUDA cores, bias columns as kind::tf32",
                     "peak_source": pk["src"]},
        "kernels": kernels,
        "cfg3": {"workload": "configs[3]: 1024 synthetic 1024x1024 images strong-scaled over %d rank(s), detector + windowed NMS + "
                             "top-2048, records all-gathered per 64-image chunk (balf_gather_keypoints, NCCL)" % world,
                 "images_per_s": 1024 / (c3_ms * 1e-3), "ms": c3_ms, "images_per_rank": c3_local,
                 "gather_ms_total": c3_gather_ms if world > 1 else None},
        "cfg4": {"workload": "configs[4]: 256 synthetic 1024x1024 images over %d rank(s), 3-level pyramid (0.7x), windowed NMS, "
                             "top-8192 merged" % world, "images_per_s": 256 / (c4_ms * 1e-3), "ms": c4_ms, "images_per_rank": c4_local},
    }
    if a.no_extras:
        line.pop("cfg3"), line.pop("cfg4")
    if world == 1 and not a.no_extras:
        line["extras"] = extras(dev, pk, det)
        line["greedy"] = extras_greedy(a, dev, pk, det, config.default_test_args(sub_pixel=False, num_features=K_FEATURES), u8)
        line["pair_cfg2"] = extras_pair(dev, det)
    if world == 1 and not a.no_cpu_baseline and not a.no_extras:
        line["cpu_baseline"] = cpu_baseline(a)
        # the reference's shipped demo path (greedy nms_fast in Python loops) beside the greedy GPU number
        line["greedy"]["cpu_baseline"] = cpu_baseline(a, nms="greedy", greedy_impl="python", budget_s=6.0, max_images=4)
        line["greedy"]["cpu_baseline_c_loop"] = cpu_baseline(a, nms="greedy", greedy_impl="c", budget_s=4.0, max_images=8)
    print(json.dumps(line))
    if gather is not None:
        gather.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
