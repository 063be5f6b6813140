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


def _prob_u8(u8, detector, precision):
    """u8 [B,H,W,C] uint8 CUDA -> (prob [B,Hp,Wp], (top, left)).  A gray image at 'tf32' takes the byte-plane forward
    (``forward_gray``: stage 1 from per-byte tables, bit-identical to the fp32-input forward); everything else the fp32 input."""
    with torch.inference_mode():
        if u8.shape[3] == 1 and precision == "tf32":
            g, (top, left) = _capi.pad_gray_u8(u8)
            return detector.forward_gray(g, precision=precision)["prob"], (top, left)
        x, (top, left) = _capi.preprocess_u8(u8)
        return detector(x, precision=precision, want_logits=False)["prob"], (top, left)


def detect_batch_device(args, u8, detector, nms="greedy"):
    """Batched device-resident detect: u8 [B,H,W,C] uint8 CUDA -> (xy int32 [B,K,2], score fp32
    [B,K], dxdy fp32 [B,K,2] | None, count int32 [B]) on the device.  ``nms`` selects the demo
    path ('greedy': demo_match.py:44-57) or the validation path ('windowed':
    balf/utils/train_utils.py:446-452)."""
    B, h, w, _ = u8.shape
    prob, (top, left) = _prob_u8(u8, detector, detector.resolve_precision(nms))
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
            prob, (top, left) = _prob_u8(u8, detector, detector.resolve_precision(nms))
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


def _camera_pairs(name, Ks, n):
    """Ks: n entries, each a 3x3 K (both images) or a pair (K1, K2) -> float64 [n,2,3,3]; ValueError unless every K is
    3x3 and finite with fx, fy > 0 and last row (0, 0, 1)."""
    if len(Ks) != n:
        raise ValueError("%s: %d camera entries for %d pairs" % (name, len(Ks), n))
    out = np.zeros((n, 2, 3, 3))
    for i, k in enumerate(Ks):
        both = isinstance(k, (tuple, list)) and len(k) == 2 and np.ndim(k[0]) == 2
        a = [np.asarray(x, np.float64) for x in (k if both else (k, k))]
        if any(x.shape != (3, 3) for x in a):
            raise ValueError("%s: K of pair %d must be 3x3 or a pair of 3x3" % (name, i))
        a = np.stack(a)
        if not (np.isfinite(a).all() and (a[:, 0, 0] > 0).all() and (a[:, 1, 1] > 0).all()
                and (a[:, 2] == [0.0, 0.0, 1.0]).all()):
            raise ValueError("%s: K of pair %d must be finite with fx, fy > 0 and last row (0, 0, 1)" % (name, i))
        out[i] = a
    return out


def _ransac_batch(estimate, name, pairs, ransac_thr, max_iters, seed, device, Ks=None, pose=False):
    """The padded batch of ``find_homography_batch`` / ``find_fundamental_batch`` / ``find_essential_batch`` /
    ``relative_pose_batch``: the lists (and the camera matrices Ks, validated first) go to the device as one padded float64
    buffer, ``estimate`` (a ``_capi`` RANSAC call) runs once, with pose=True ``_capi.recover_pose`` runs on its output on
    the same stream, and the results come back in one copy -> [(model [3,3] float64 or None, mask uint8 [M_i,1])], with
    pose=True [(R [3,3] or None, t [3,1] or None, E or None, inlier mask [M_i,1], pose mask [M_i,1])]; None where the
    library returned all zeros (no model)."""
    cams = None if Ks is None else _camera_pairs(name, Ks, len(pairs))
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if not pairs:
        return []
    p = [(np.asarray(a, np.float64).reshape(-1, 2), np.asarray(b, np.float64).reshape(-1, 2)) for a, b in pairs]
    for a, b in p:
        if len(a) != len(b):
            raise ValueError("%s: pts1 and pts2 have %d and %d rows" % (name, len(a), len(b)))
    B, M = len(p), max(max(len(a) for a, _ in p), 1)
    nk = 0 if cams is None else 18 * B
    host = np.zeros(2 * B * M * 2 + B + nk)               # p1 [B,M,2], p2 [B,M,2], the counts, then K [B,2,9]
    pts = host[:4 * B * M].reshape(2, B, M, 2)
    for i, (a, b) in enumerate(p):
        pts[0, i, :len(a)], pts[1, i, :len(b)] = a, b
    host[4 * B * M:4 * B * M + B] = [len(a) for a, _ in p]
    if cams is not None:
        host[4 * B * M + B:] = cams.reshape(-1)
    buf = torch.from_numpy(host).to(dev)
    d = buf[:4 * B * M].view(2, B, M, 2)
    cnt = buf[4 * B * M:4 * B * M + B].to(torch.int32)
    kin = () if cams is None else (buf[4 * B * M + B:].view(B, 2, 9),)
    G, mask, _ = estimate(d[0], d[1], cnt, *kin, ransac_thr, max_iters, seed)
    parts = [G.reshape(-1).view(torch.uint8), mask.reshape(-1)]
    if pose:
        R, t, pmask, _ = _capi.recover_pose(G, d[0], d[1], cnt, kin[0], mask)
        parts += [R.reshape(-1).view(torch.uint8), t.reshape(-1).view(torch.uint8), pmask.reshape(-1)]
    out = torch.cat(parts).cpu().numpy()
    Gs = out[:B * 72].view(np.float64).reshape(B, 3, 3)
    masks = out[B * 72:B * 72 + B * M].reshape(B, M)
    if not pose:
        return [(Gs[i].copy() if Gs[i].any() else None, masks[i, :len(a)].reshape(-1, 1).copy())
                for i, (a, _) in enumerate(p)]
    o = B * 72 + B * M
    Rs = out[o:o + B * 72].view(np.float64).reshape(B, 3, 3)
    ts = out[o + B * 72:o + B * 96].view(np.float64).reshape(B, 3, 1)
    pm = out[o + B * 96:].reshape(B, M)
    res = []
    for i, (a, _) in enumerate(p):
        found = Rs[i].any()
        res.append((Rs[i].copy() if found else None, ts[i].copy() if found else None,
                    Gs[i].copy() if Gs[i].any() else None, masks[i, :len(a)].reshape(-1, 1).copy(),
                    pm[i, :len(a)].reshape(-1, 1).copy()))
    return res


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


def find_essential_batch(pairs, Ks, ransac_thr=1.0, max_iters=1000, seed=0, device=None):
    """RANSAC essential matrices of many calibrated match lists in one library call (semantics: include/balf_b200.h,
    balf_find_essential_ransac).  pairs = [(pts1 [M_i,2], pts2 [M_i,2])] undistorted pixel coordinates, Ks = one entry per
    pair, a 3x3 K shared by both images or a pair (K1, K2) -> [(E [3,3] float64 or None, mask uint8 [M_i,1])], each entry
    in the return layout of ``cv2.findEssentialMat(pts1, pts2, K, cv2.RANSAC, threshold=ransac_thr, maxIters=max_iters)``.
    E is None when the pair has fewer than 5 matches or no model.  A K that is not 3x3, not finite, has fx or fy <= 0 or a
    last row other than (0, 0, 1) raises ValueError before anything runs."""
    return _ransac_batch(_capi.find_essential_ransac, "find_essential", pairs, ransac_thr, max_iters, seed, device, Ks=Ks)


def find_essential(pts1, pts2, K1, K2=None, ransac_thr=1.0, max_iters=1000, seed=0, device=None):
    """GPU counterpart of ``cv2.findEssentialMat(pts1, pts2, K1, cv2.RANSAC, threshold=ransac_thr, maxIters=max_iters)``
    (and of its two-camera overload when K2 is given) on one match list -> (E [3,3] float64 or None, mask uint8 [M,1]).
    The differences from cv2:
    - E is scaled to unit Frobenius norm with its first largest-magnitude entry positive.
    - The iteration count is fixed (no confidence-driven early exit), so the result is a pure function of (points, K,
      ransac_thr, max_iters, seed).
    - With exactly 5 matches cv2 returns every 5-point solution stacked [3k,3]; this returns the best single E."""
    return find_essential_batch([(pts1, pts2)], [(K1, K1 if K2 is None else K2)], ransac_thr, max_iters, seed, device)[0]


def recover_pose(E, pts1, pts2, K1, K2=None, mask=None, dist_thresh=50.0, device=None):
    """GPU counterpart of ``cv2.recoverPose(E, pts1, pts2, K1, distanceThresh=dist_thresh, mask=mask)`` on one match list
    -> (n_good, R [3,3], t [3,1], mask uint8 [M,1]), cv2's layout; R, t map camera-1 coordinates to camera 2.  The
    triangulation is closed-form rather than cv2's SVD (include/balf_b200.h, balf_recover_pose), so a match within rounding
    of the depth or distance bounds can be counted differently.  An all-zero E gives zeros."""
    a, b = np.asarray(pts1, np.float64).reshape(-1, 2), np.asarray(pts2, np.float64).reshape(-1, 2)
    if len(a) != len(b):
        raise ValueError("recover_pose: pts1 and pts2 have %d and %d rows" % (len(a), len(b)))
    e = np.asarray(E, np.float64)
    if e.shape != (3, 3):
        raise ValueError("recover_pose: E must be 3x3")
    cams = _camera_pairs("recover_pose", [(K1, K1 if K2 is None else K2)], 1)
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    n, M = len(a), max(len(a), 1)
    host = np.zeros(4 * M + 9 + 18)
    host[:2 * n], host[2 * M:2 * M + 2 * n] = a.reshape(-1), b.reshape(-1)
    host[4 * M:4 * M + 9], host[4 * M + 9:] = e.reshape(-1), cams.reshape(-1)
    buf = torch.from_numpy(host).to(dev)
    m = None
    if mask is not None:
        mk = np.asarray(mask).reshape(-1)
        if len(mk) != n:
            raise ValueError("recover_pose: mask has %d rows for %d matches" % (len(mk), n))
        m = torch.zeros(1, M, dtype=torch.uint8)
        m[0, :n] = torch.from_numpy((mk != 0).astype(np.uint8))
        m = m.to(dev)
    cnt = torch.full((1,), n, dtype=torch.int32, device=dev)
    R, t, pm, ng = _capi.recover_pose(buf[4 * M:4 * M + 9].view(1, 9), buf[:2 * M].view(1, M, 2),
                                      buf[2 * M:4 * M].view(1, M, 2), cnt, buf[4 * M + 9:].view(1, 2, 9), m, dist_thresh)
    out = torch.cat([R.reshape(-1).view(torch.uint8), t.reshape(-1).view(torch.uint8), pm.reshape(-1),
                     ng.view(torch.uint8)]).cpu().numpy()
    return (int(out[96 + M:].view(np.int32)[0]), out[:72].view(np.float64).reshape(3, 3).copy(),
            out[72:96].view(np.float64).reshape(3, 1).copy(), out[96:96 + n].reshape(-1, 1).copy())


def relative_pose_batch(pairs, Ks, ransac_thr=1.0, max_iters=1000, seed=0, device=None):
    """Relative poses of many calibrated match lists: ``find_essential_batch`` then ``recover_pose`` on its inliers, both
    library calls on one stream, with one upload and one download -> [(R [3,3] or None, t [3,1] or None, E [3,3] or None,
    inlier mask uint8 [M_i,1], pose mask uint8 [M_i,1])]; X2 = R X1 + t with |t| = 1.  None where the pair has no model."""
    return _ransac_batch(_capi.find_essential_ransac, "relative_pose", pairs, ransac_thr, max_iters, seed, device, Ks=Ks,
                         pose=True)
