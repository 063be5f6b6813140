"""Drop-in for the reference's ``demo/demo_match.py`` library functions.

``detect`` (:21-57), ``extract_features`` (:59-95) and ``extract_matches`` (:97-112) keep their
signatures and return layouts.  Each one is a short chain of C-ABI calls on device-resident
buffers; the image goes host->device once as uint8 and only the keypoint / descriptor / match
lists come back (the reference crosses the boundary four times per image with fp32 maps).
``load_im`` / ``draw_matches`` (PIL / cv2 I/O) are out of scope.
"""
import numpy as np
import torch

from .. import _capi
from ..utils import test_utils


def _detect_device(args, im, detector, device):
    """image -> device-resident (xy int32 [K,2], dxdy fp32 [K,2] | None, score [K], K)."""
    dev = torch.device(device)
    if im.dtype == np.uint8:
        u8 = torch.from_numpy(np.ascontiguousarray(im)).to(dev, non_blocking=True)[None]
        x, (top, left) = _capi.preprocess_u8(u8)
    else:                                   # non-uint8 input: the reference's float64 arithmetic, on the host
        pad = test_utils.mod_padding_symmetric(test_utils.make_shape_even(im / 255.), factor=64)
        x = torch.tensor(pad, dtype=torch.float32).permute(2, 0, 1).unsqueeze(0).contiguous().to(dev)
        _, _, top, left = _capi.pad_geometry(im.shape[0], im.shape[1], 64)
    with torch.inference_mode():
        prob = detector(x, precision=detector.resolve_precision("greedy"), want_logits=False)["prob"]
    h, w = im.shape[0], im.shape[1]
    xy, sc, dxdy, cnt = _capi.greedy_nms_topk(
        prob, args.num_features, border=args.border_size, thr=args.heatmap_confidence_threshold,
        radius=args.nms_size, subpixel_ps=args.patch_size if args.sub_pixel else 0, crop=(top, left, h, w))
    return xy[0], (dxdy[0] if dxdy is not None else None), sc[0], int(cnt[0])


def detect_batch_device(args, u8, detector, nms="greedy"):
    """Batched device-resident detect: u8 [B,H,W,C] uint8 CUDA -> (xy int32 [B,K,2], score fp32
    [B,K], dxdy fp32 [B,K,2] | None, count int32 [B]) on the device.  ``nms`` selects the demo
    path ('greedy': demo_match.py:44-57) or the validation path ('windowed':
    balf/utils/train_utils.py:446-452)."""
    B, h, w, _ = u8.shape
    x, (top, left) = _capi.preprocess_u8(u8)
    with torch.inference_mode():
        prob = detector(x, precision=detector.resolve_precision(nms), want_logits=False)["prob"]
    if nms == "windowed":
        xy, sc, cnt = _capi.windowed_nms_topk(prob, args.num_features, border=args.border_size,
                                              nms_size=args.nms_size, crop=(top, left, h, w))
        return xy, sc, None, cnt
    return _capi.greedy_nms_topk(
        prob, args.num_features, border=args.border_size, thr=args.heatmap_confidence_threshold,
        radius=args.nms_size, subpixel_ps=args.patch_size if args.sub_pixel else 0, crop=(top, left, h, w))


def detect_multiscale_batch_device(args, u8, detector, scale=0.7, levels=3, nms="windowed", upsampled_levels=0):
    """Multi-scale pyramid extraction (the mode the reference advertises in balf/configs/config_hpatches.py:50-82 but
    does not implement; semantics defined in include/balf_b200.h and restated in oracle/multiscale.py).
    u8 [B,H,W,C] uint8 CUDA.  Level l (l = -upsampled_levels .. levels - 1, finest first) is the bilinear resize of the
    image to round(H s^l) x round(W s^l) -- l < 0 are the up-sampled levels of the parser's ``--upsampled_levels``; every
    level runs the detector and the per-level extraction with capacity args.num_features, and the lists are merged by score
    into the best args.num_features keypoints in level-0 coordinates.  The parser's defaults (scale_factor_levels sqrt(2),
    pyramid_levels 5, upsampled_levels 1) are ``scale=2 ** -0.5, levels=6, upsampled_levels=1``:
    ``config.multiscale_pyramid(config.default_multiscale_args())``.
    -> (xy fp32 [B,K,2], score fp32 [B,K], level int32 [B,K] (index into the finest-first level list), count int32 [B])
    on the device."""
    B, h, w, _ = u8.shape
    lists, scales = [], []
    for l in range(-int(upsampled_levels), levels):
        hs, ws = _capi.level_size(h, scale, l), _capi.level_size(w, scale, l)
        if l == 0:
            x, (top, left) = _capi.preprocess_u8(u8)
        else:
            x, (top, left) = _capi.resize_preprocess_u8(u8, hs, ws)
        with torch.inference_mode():
            prob = detector(x, precision=detector.resolve_precision(nms), want_logits=False)["prob"]
        if nms == "windowed":
            xy, sc, cnt = _capi.windowed_nms_topk(prob, args.num_features, border=args.border_size,
                                                  nms_size=args.nms_size, crop=(top, left, hs, ws))
        else:
            xy, sc, _, cnt = _capi.greedy_nms_topk(prob, args.num_features, border=args.border_size,
                                                   thr=args.heatmap_confidence_threshold, radius=args.nms_size,
                                                   subpixel_ps=0, crop=(top, left, hs, ws))
        lists.append((xy, sc, cnt))
        scales.append((w / ws, h / hs))
    return _capi.merge_levels_topk(lists, scales, args.num_features)


def detect_batch(args, images, detector, device, nms="greedy"):
    """Batched ``detect`` with HOST buffers in and out: images [B,H,W,C] uint8 (NumPy array or
    torch CPU tensor, pinned for an asynchronous copy) -> (xy int32 [B,K,2], score fp32 [B,K],
    count int32 [B]) NumPy arrays; rows beyond count[b] are zero.  One H2D copy of the uint8
    batch, one D2H copy of the keypoint records."""
    dev = torch.device(device)
    t = images if isinstance(images, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(images))
    xy, sc, dxdy, cnt = detect_batch_device(args, t.to(dev, non_blocking=True), detector, nms)
    return xy.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()


class DetectPipeline:
    """Streaming form of ``detect_batch`` for throughput serving: ``submit`` takes a HOST batch (pinned uint8
    [B,H,W,C]) and returns a ticket, ``result`` returns that batch's (xy, score, count) NumPy arrays.  The host->device
    copy of a batch runs on a copy stream while the kernels of the previous batch run on the compute stream, and the
    keypoint records come back through pinned staging buffers -- every batch still crosses PCIe both ways, the copies
    just no longer sit between the kernels of consecutive batches."""

    def __init__(self, args, detector, device, nms="greedy", depth=4):
        self.args, self.detector, self.nms = args, detector, nms
        self.dev = torch.device(device)
        self.copy_stream = torch.cuda.Stream(self.dev)
        self.compute_stream = torch.cuda.Stream(self.dev)
        self.depth, self._free, self._in_flight = depth, {}, 0

    def _staging(self, outs):
        """a set of pinned host buffers for these output shapes from the free list of that shape (allocated on first use:
        no allocation in the steady state).  A set belongs to its ticket until ``result`` has copied it out and returned
        it -- tickets may be collected in any order and batches of different shapes may interleave."""
        key = tuple((tuple(o.shape), o.dtype) for o in outs)
        free = self._free.setdefault(key, [])
        return key, (free.pop() if free else [torch.empty(o.shape, dtype=o.dtype, pin_memory=True) for o in outs])

    def submit(self, images):
        if self._in_flight >= self.depth:
            raise RuntimeError("DetectPipeline: %d batches in flight, collect a result first" % self._in_flight)
        self._in_flight += 1
        t = images if isinstance(images, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(images))
        with torch.cuda.stream(self.copy_stream):
            u8 = t.to(self.dev, non_blocking=True)
            arrived = torch.cuda.Event()
            arrived.record(self.copy_stream)
        u8.record_stream(self.compute_stream)
        with torch.cuda.stream(self.compute_stream):
            self.compute_stream.wait_event(arrived)
            xy, sc, _, cnt = detect_batch_device(self.args, u8, self.detector, self.nms)
            key, host = self._staging((xy, sc, cnt))
            for h, o in zip(host, (xy, sc, cnt)):
                h.copy_(o, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self.compute_stream)
        return [key, host, done, (xy, sc, cnt)]       # device tensors kept alive until the copies have run

    def result(self, ticket):
        key, host, done, _ = ticket
        if host is None:
            raise RuntimeError("DetectPipeline: this ticket has already been collected")
        done.synchronize()
        self._in_flight -= 1
        out = tuple(h.numpy().copy() for h in host)
        self._free[key].append(host)                  # only now may another submission reuse the staging set
        ticket[1] = ticket[3] = None
        return out


def detect(args, im, detector, device):
    """-> [K,3] float64 rows (x, y, 1.0), score-descending, K <= args.num_features."""
    xy, dxdy, _, n = _detect_device(args, im, detector, device)
    if n == 0:
        return np.zeros([0, 3]), np.zeros([0, 1])          # (sic) the reference returns this pair
    pts = xy[:n].cpu().numpy().astype(np.float64)
    if dxdy is not None:
        pts = pts + dxdy[:n].cpu().numpy().astype(np.float64)
    if args.order_coord == 'yxsr':
        pts = pts[:, ::-1]
    return np.concatenate([pts, np.ones((n, 1))], axis=1)


def extract_features(args, im_rgb, im_gray, detector, descriptor, device):
    """-> (kpts [K,2] float64, descs [K,128] float32)."""
    kpts_np = detect(args, im_rgb, detector, device)
    dev = torch.device(device)
    kp = torch.from_numpy(np.ascontiguousarray(kpts_np[:, 0:2])).float().to(dev)
    gray = torch.from_numpy(np.ascontiguousarray(im_gray)).to(dev)
    patches = _capi.extract_patches(gray, kp, float(args.s_mult), 32)
    if patches.shape[0] == 0:
        return kpts_np[:, 0:2], np.array([])
    with torch.inference_mode():
        descs = descriptor(patches)
    return kpts_np[:, 0:2], descs.cpu().numpy()


_PAIR_STAGING = {}      # (key, device, shape) -> [pinned uint8 staging buffer, event of its last DMA]; the device-resident pair
_PAIR_STAGING_MAX = 4   # path reuses them across calls, at most this many shapes (least recently used first out)


def _pinned_upload(key, arrays, dev):
    """Same-shape uint8 host arrays -> ONE device tensor [len(arrays), ...]: each array is copied into its slice of a cached
    pinned staging buffer and leaves on an asynchronous DMA right away -- the copy of array i+1 into pinned memory runs while
    array i crosses PCIe, and no stacked pageable copy is built first.  The buffer may be rewritten only once its last DMA has
    finished: the event recorded after the copies is waited on at the next use."""
    shape = (len(arrays),) + tuple(arrays[0].shape)
    slot = _PAIR_STAGING.pop((key, dev, shape), None)
    if slot is None:
        while len(_PAIR_STAGING) >= _PAIR_STAGING_MAX:          # images of many sizes (HPatches): do not hoard pinned memory
            _, old_event = _PAIR_STAGING.pop(next(iter(_PAIR_STAGING)))
            if old_event is not None:
                old_event.synchronize()
        slot = [torch.empty(shape, dtype=torch.uint8, pin_memory=True), None]
    _PAIR_STAGING[(key, dev, shape)] = slot                   # (re-)inserted last: dict order = least recently used first
    pin, last = slot
    if last is not None:
        last.synchronize()
    out = torch.empty(shape, dtype=torch.uint8, device=dev)
    view = pin.numpy()
    for i, a in enumerate(arrays):
        np.copyto(view[i], a)
        out[i].copy_(pin[i], non_blocking=True)
    slot[1] = torch.cuda.Event()
    slot[1].record(torch.cuda.current_stream(dev))
    return out


def _features_batch_device(args, rgbs, grays, detector, descriptor, dev):
    """Same-shape uint8 images -> per image (xy int32 [n,2], dxdy fp32 [n,2] | None, descriptors fp32 [n,128]), all on the device:
    ONE batched detector + greedy NMS call, per-image patch sampling, ONE HardNet call over all patches.  Per-image results are
    identical to ``extract_features`` one image at a time (no stage mixes images)."""
    u8 = _pinned_upload("rgb", rgbs, dev)
    xy, _, dxdy, cnt = detect_batch_device(args, u8, detector, "greedy")
    if all(g.dtype == np.uint8 and g.shape == grays[0].shape for g in grays):
        gray_dev = _pinned_upload("gray", grays, dev)                                    # uploads under the detector
    else:
        gray_dev = [torch.from_numpy(np.ascontiguousarray(g)).to(dev, non_blocking=True) for g in grays]
    counts = cnt.cpu().tolist()
    patches = []
    for b, n in enumerate(counts):
        kp = xy[b, :n].float()
        if dxdy is not None:
            kp = kp + dxdy[b, :n]
        patches.append(_capi.extract_patches(gray_dev[b], kp, float(args.s_mult), 32))
    with torch.inference_mode():
        descs = descriptor(torch.cat(patches)) if sum(counts) else torch.zeros(0, 128, device=dev)
    out, o = [], 0
    for b, n in enumerate(counts):
        out.append((xy[b, :n], dxdy[b, :n] if dxdy is not None else None, descs[o:o + n]))
        o += n
    return out


def extract_matches(args, im_rgb1, im_gray1, im_rgb2, im_gray2, detector, descriptor, device):
    """-> (points1 [M,2], points2 [M,2]) of the SMNN(0.99) matches, ordered by the first index."""
    dev = torch.device(device)
    if (im_rgb1.dtype == np.uint8 and im_rgb2.dtype == np.uint8 and im_rgb1.shape == im_rgb2.shape
            and args.order_coord == 'xysr'):
        # device-resident pair: both images through one batched detector / HardNet call, keypoints and descriptors never
        # leave the GPU; only the matched points come back
        (xy1, dx1, d1), (xy2, dx2, d2) = _features_batch_device(args, (im_rgb1, im_rgb2), (im_gray1, im_gray2),
                                                                 detector, descriptor, dev)
        if d1.shape[0] >= 2 and d2.shape[0] >= 2:
            ids = _capi.match_smnn(d1, d2, 0.99)[1].long()
            pts = []
            for xy, dx, col in ((xy1, dx1, 0), (xy2, dx2, 1)):
                # int32 pixel + fp32 offset, added in float64 as the reference does on the host (both convert exactly)
                p = xy[ids[:, col]].double()
                if dx is not None:
                    p = p + dx[ids[:, col]].double()
                pts.append(p)
            both = torch.stack(pts).cpu().numpy()          # one device->host copy of the matched points of both images
            return both[0], both[1]
    kpts1, desc1 = extract_features(args, im_rgb1, im_gray1, detector, descriptor, device)
    kpts2, desc2 = extract_features(args, im_rgb2, im_gray2, detector, descriptor, device)
    ids = _capi.match_smnn(torch.from_numpy(desc1).to(dev), torch.from_numpy(desc2).to(dev), 0.99)[1]
    ids = ids.cpu().numpy()
    return kpts1[ids[:, 0], :2], kpts2[ids[:, 1], :2]


def _ransac_batch(estimate, name, pairs, ransac_thr, max_iters, seed, device):
    """The padded batch of ``find_homography_batch`` / ``find_fundamental_batch``: the lists go to the device as one padded
    float64 buffer, ``estimate`` (a ``_capi`` RANSAC call) runs once, and the 3x3 models and the masks come back in one
    copy -> [(model [3,3] float64 or None, mask uint8 [M_i,1])]; None where the library returned all zeros (no model)."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if not pairs:
        return []
    p = [(np.asarray(a, np.float64).reshape(-1, 2), np.asarray(b, np.float64).reshape(-1, 2)) for a, b in pairs]
    for a, b in p:
        if len(a) != len(b):
            raise ValueError("%s: pts1 and pts2 have %d and %d rows" % (name, len(a), len(b)))
    B, M = len(p), max(max(len(a) for a, _ in p), 1)
    host = np.zeros(2 * B * M * 2 + B)                    # p1 [B,M,2], p2 [B,M,2], then the counts
    pts = host[:4 * B * M].reshape(2, B, M, 2)
    for i, (a, b) in enumerate(p):
        pts[0, i, :len(a)], pts[1, i, :len(b)] = a, b
    host[4 * B * M:] = [len(a) for a, _ in p]
    buf = torch.from_numpy(host).to(dev)
    d = buf[:4 * B * M].view(2, B, M, 2)
    G, mask, _ = estimate(d[0], d[1], buf[4 * B * M:].to(torch.int32), ransac_thr, max_iters, seed)
    out = torch.cat([G.reshape(-1).view(torch.uint8), mask.reshape(-1)]).cpu().numpy()
    Gs = out[:B * 72].view(np.float64).reshape(B, 3, 3)
    masks = out[B * 72:].reshape(B, M)
    return [(Gs[i].copy() if Gs[i].any() else None, masks[i, :len(a)].reshape(-1, 1).copy()) for i, (a, _) in enumerate(p)]


def find_homography_batch(pairs, ransac_thr=3.0, max_iters=2000, seed=0, device=None):
    """RANSAC homographies of many match lists in one library call (semantics: include/balf_b200.h,
    balf_find_homography_ransac).  pairs = [(pts1 [M_i,2], pts2 [M_i,2])] host arrays of any lengths -> [(H [3,3] float64 or
    None, mask uint8 [M_i,1])], each entry in the return layout of ``cv2.findHomography(pts1, pts2, cv2.RANSAC, ransac_thr,
    maxIters=max_iters)``.  H is None when the pair has fewer than 4 matches or no non-degenerate sample.  The lists go to
    the device as one padded float64 buffer, and H and the masks come back in one copy."""
    return _ransac_batch(_capi.find_homography_ransac, "find_homography", pairs, ransac_thr, max_iters, seed, device)


def find_homography(pts1, pts2, ransac_thr=3.0, max_iters=2000, seed=0, device=None):
    """GPU drop-in for ``cv2.findHomography(pts1, pts2, cv2.RANSAC, ransac_thr, maxIters=max_iters)`` on one match list
    (e.g. the output of ``extract_matches``) -> (H [3,3] float64 or None, mask uint8 [M,1]).  The iteration count is fixed
    (no confidence-driven early exit), so the result is a pure function of (points, ransac_thr, max_iters, seed)."""
    return find_homography_batch([(pts1, pts2)], ransac_thr, max_iters, seed, device)[0]


def find_fundamental_batch(pairs, ransac_thr=3.0, max_iters=1000, seed=0, device=None):
    """RANSAC fundamental matrices of many match lists in one library call (semantics: include/balf_b200.h,
    balf_find_fundamental_ransac).  pairs = [(pts1 [M_i,2], pts2 [M_i,2])] host arrays of any lengths -> [(F [3,3] float64
    or None, mask uint8 [M_i,1])], each entry in the return layout of ``cv2.findFundamentalMat(pts1, pts2, cv2.FM_RANSAC,
    ransac_thr, maxIters=max_iters)``, with x2^T F x1 = 0.  F is None when the pair has fewer than 7 matches or no model."""
    return _ransac_batch(_capi.find_fundamental_ransac, "find_fundamental", pairs, ransac_thr, max_iters, seed, device)


def find_fundamental(pts1, pts2, ransac_thr=3.0, max_iters=1000, seed=0, device=None):
    """GPU counterpart of ``cv2.findFundamentalMat(pts1, pts2, cv2.FM_RANSAC, ransac_thr, maxIters=max_iters)`` on one match
    list (e.g. the output of ``extract_matches``) -> (F [3,3] float64 or None, mask uint8 [M,1]).  The differences from
    cv2:
    - F is scaled to unit Frobenius norm with its first largest-magnitude entry positive; cv2 divides by F[2,2] where it
      can.  A fundamental matrix is defined up to scale only, so both describe the same epipolar geometry.
    - The iteration count is fixed (no confidence-driven early exit), so the result is a pure function of (points,
      ransac_thr, max_iters, seed).
    - With exactly 7 matches cv2 returns all (up to 3) 7-point solutions stacked [9,3]; this runs RANSAC as usual and
      returns the best single F.
    Plane degeneracy is not handled: on a planar scene F fits the matches but the epipolar geometry is not determined."""
    return find_fundamental_batch([(pts1, pts2)], ransac_thr, max_iters, seed, device)[0]
