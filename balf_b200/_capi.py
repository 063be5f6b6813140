"""ctypes binding of ``libbalf_b200.so`` (include/balf_b200.h) for the PyTorch-facing modules.

PyTorch is plumbing here: it owns device memory and streams; every computation is a call into
the C-ABI with raw device pointers.  The library must be present -- importing this module
without it raises, and there is no CPU or eager fallback anywhere in the package.
"""
import ctypes
import os
import re

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BALF_B200_LIB") or os.path.join(_HERE, "libbalf_b200.so")   # override: development A/B builds
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "balf_b200.h")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "balf_b200: %s is missing. Build it with `python -c \"import __graft_entry__ as g; g.build()\"` "
        "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
_lib = ctypes.CDLL(LIB_PATH)

c_int, c_void_p, c_size_t, c_float = ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_float


class DetectorArch(ctypes.Structure):
    _fields_ = [("dims", ctypes.c_int32 * 5), ("grid_h", ctypes.c_int32), ("grid_w", ctypes.c_int32),
                ("block_h", ctypes.c_int32), ("block_w", ctypes.c_int32), ("grid_factor", ctypes.c_int32),
                ("block_factor", ctypes.c_int32), ("proj_factor", ctypes.c_int32), ("reduction", ctypes.c_int32),
                ("cell", ctypes.c_int32)]


def _sig(name, restype, *argtypes):
    fn = getattr(_lib, name)
    fn.restype, fn.argtypes = restype, list(argtypes)
    return fn


_P = c_void_p
_arch_p = ctypes.POINTER(DetectorArch)
_last_error = _sig("balf_last_error", ctypes.c_char_p)
abi_version = _sig("balf_abi_version", c_int)
launch_count = _sig("balf_launch_count", ctypes.c_ulonglong)
_check_arch = _sig("balf_detector_check_arch", c_int, _arch_p)
_raw_count = _sig("balf_detector_raw_weight_count", ctypes.c_int64, _arch_p)
_packed_count = _sig("balf_detector_packed_weight_count", ctypes.c_int64, _arch_p)
_pack = _sig("balf_detector_pack_weights", c_int, _arch_p, _P, _P, _P)
_pad_geometry = _sig("balf_pad_geometry", c_int, c_int, c_int, c_int, *([ctypes.POINTER(c_int)] * 4))
_preprocess = _sig("balf_preprocess_u8", c_int, _P, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, _P)
_det_ws = _sig("balf_detector_workspace_bytes", c_size_t, _arch_p, c_int, c_int, c_int)
_det_fwd = _sig("balf_detector_forward", c_int, _arch_p, _P, _P, c_int, c_int, c_int, _P, _P, _P, c_size_t, c_int, _P)
_pad_gray = _sig("balf_pad_gray_u8", c_int, _P, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, _P)
_det_fwd_gray = _sig("balf_detector_forward_gray", c_int, _arch_p, _P, _P, c_int, c_int, c_int, _P, _P, _P, c_size_t, c_int, _P)
_pixel_shuffle = _sig("balf_pixel_shuffle", c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P)
_nms_ws = _sig("balf_nms_workspace_bytes", c_size_t, c_int, c_int, c_int, c_int)
_win_nms = _sig("balf_windowed_nms_topk", c_int, _P, *([c_int] * 10), _P, _P, _P, _P, c_size_t, _P)
_greedy_nms = _sig("balf_greedy_nms_topk", c_int, _P, *([c_int] * 8), c_float, c_int, c_int, c_int, _P, _P, _P, _P, _P,
                   c_size_t, _P)


_prof_enable = _sig("balf_profile_enable", c_int, c_int)
_prof_report = _sig("balf_profile_report", c_int, ctypes.c_char_p, c_size_t, c_int)


def profile_enable(on):
    _ok(_prof_enable(1 if on else 0))


def profile_report(reset=True):
    """host-synchronous -> {kernel name: (launches, total_ms)} since the last reset."""
    buf = ctypes.create_string_buffer(1 << 16)
    _ok(_prof_report(buf, len(buf), 1 if reset else 0))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.split()
        out[name] = (int(n), float(ms))
    return out


debug_set = _sig("balf_debug_set", c_int, c_int, c_int)
debug_set_trace = _sig("balf_debug_set_trace", c_int, c_void_p)


def declared_symbols():
    """Every function the public header declares (tests check that the library exports them all)."""
    return re.findall(r"\b(balf_[a-z0-9_]+)\s*\(", open(HEADER_PATH).read())


class BalfError(RuntimeError):
    pass


def _ok(code):
    if code != 0:
        msg = (_last_error() or b"").decode()
        raise (ValueError if code < 0 else BalfError)("balf_b200: %s (code %d)" % (msg, code))


def _stream(device):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def _need_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError("balf_b200 has no CPU path: %s must be a CUDA tensor" % what)


def _same_device(t, ref, what):
    """t must be a CUDA tensor on ref's device: the C-ABI takes raw pointers and one stream."""
    _need_cuda(t, what)
    if t.device != ref.device:
        raise ValueError("%s is on %s, expected %s" % (what, t.device, ref.device))


_workspaces = {}


def _workspace(device, nbytes):
    """grow-only scratch buffer per (device, stream) -- the C-ABI never allocates.  Keyed by the current stream because
    the kernels of one call use the buffer in stream order: two streams sharing it would race (DetectPipeline runs
    beside default-stream callers)."""
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


# ------------------------------------------------------------------------------------------ detector
def arch_struct(arch):
    a = DetectorArch()
    a.dims[:] = arch["dims"]
    a.grid_h, a.grid_w = arch["grid"]
    a.block_h, a.block_w = arch["block"]
    a.grid_factor, a.block_factor, a.proj_factor = arch["gfac"], arch["bfac"], arch["proj"]
    a.reduction, a.cell = arch["red"], arch["cell"]
    return a


def check_supported_arch(arch):
    _ok(_check_arch(ctypes.byref(arch_struct(arch))))


def detector_pack_weights(raw, arch):
    _need_cuda(raw, "the weight blob")
    a = arch_struct(arch)
    n_raw, n_packed = _raw_count(ctypes.byref(a)), _packed_count(ctypes.byref(a))
    if raw.numel() != n_raw or raw.dtype != torch.float32:
        raise ValueError("weight blob has %d floats, the architecture needs %d" % (raw.numel(), n_raw))
    raw = raw.contiguous()
    packed = torch.empty(n_packed, dtype=torch.float32, device=raw.device)
    with torch.cuda.device(raw.device):
        _ok(_pack(ctypes.byref(a), _ptr(raw), _ptr(packed), _stream(raw.device)))
    return packed


PRECISIONS = {"fp32": 0, "tf32": 1, "f16x3": 2}     # f16x3: tensor cores on fp16 hi + lo operand pairs (three MMAs per product), fp32-class results


def detector_forward(x, packed, arch, precision="fp32", want_logits=True):
    _need_cuda(x, "the input")
    a = arch_struct(arch)
    x = x.contiguous().float()
    B, _, H, W = x.shape
    n_logit = arch["cell"] ** 2 + 1
    logits = torch.empty(B, n_logit, H // arch["cell"], W // arch["cell"], dtype=torch.float32, device=x.device) \
        if want_logits else None
    prob = torch.empty(B, H, W, dtype=torch.float32, device=x.device)
    nbytes = _det_ws(ctypes.byref(a), B, H, W)
    ws = _workspace(x.device, nbytes)
    with torch.cuda.device(x.device):
        _ok(_det_fwd(ctypes.byref(a), _ptr(packed), _ptr(x), B, H, W, _ptr(logits), _ptr(prob), _ptr(ws), nbytes,
                     PRECISIONS[precision], _stream(x.device)))
    return logits, prob


def detector_forward_gray(g, packed, arch, precision="tf32", want_logits=True):
    """``detector_forward`` for a gray image given as its padded byte plane g [B,Hp,Wp] uint8 (``pad_gray_u8``): bit-identical
    to ``detector_forward(preprocess_u8(img)[0])``, stage 1 on per-byte tables (balf_detector_forward_gray).  'tf32' only."""
    _need_cuda(g, "the input")
    if g.dtype != torch.uint8 or g.dim() != 3:
        raise ValueError("expected a padded gray byte plane [B, Hp, Wp] uint8, got %s %s" % (g.dtype, tuple(g.shape)))
    a = arch_struct(arch)
    g = g.contiguous()
    B, H, W = g.shape
    n_logit = arch["cell"] ** 2 + 1
    logits = torch.empty(B, n_logit, H // arch["cell"], W // arch["cell"], dtype=torch.float32, device=g.device) \
        if want_logits else None
    prob = torch.empty(B, H, W, dtype=torch.float32, device=g.device)
    nbytes = _det_ws(ctypes.byref(a), B, H, W)
    ws = _workspace(g.device, nbytes)
    with torch.cuda.device(g.device):
        _ok(_det_fwd_gray(ctypes.byref(a), _ptr(packed), _ptr(g), B, H, W, _ptr(logits), _ptr(prob), _ptr(ws), nbytes,
                          PRECISIONS[precision], _stream(g.device)))
    return logits, prob


def pixel_shuffle(t, r):
    _need_cuda(t, "the input")
    t = t.contiguous().float()
    n, c, h, w = t.shape
    out = torch.empty(n, c // (r * r), h * r, w * r, dtype=torch.float32, device=t.device)
    with torch.cuda.device(t.device):
        _ok(_pixel_shuffle(_ptr(t), _ptr(out), n, c, h, w, r, _stream(t.device)))
    return out


# ------------------------------------------------------------------------------------------ pre / post
def pad_geometry(h, w, factor=64):
    """-> (Hp, Wp, top, left) of make_shape_even + mod_padding_symmetric (pure host arithmetic)."""
    out = [c_int() for _ in range(4)]
    _ok(_pad_geometry(int(h), int(w), int(factor), *[ctypes.byref(o) for o in out]))
    return tuple(o.value for o in out)


def preprocess_u8(img, factor=64):
    """img [B,H,W,C] uint8 CUDA -> (x [B,3,Hp,Wp] fp32, (top, left))."""
    _need_cuda(img, "the image batch")
    img = img.contiguous()
    B, H, W, C = img.shape
    Hp, Wp, top, left = pad_geometry(H, W, factor)
    x = torch.empty(B, 3, Hp, Wp, dtype=torch.float32, device=img.device)
    with torch.cuda.device(img.device):
        _ok(_preprocess(_ptr(img), B, H, W, C, _ptr(x), Hp, Wp, top, left, _stream(img.device)))
    return x, (top, left)


def pad_gray_u8(img, factor=64):
    """img [B,H,W,1] uint8 CUDA (gray) -> (g [B,Hp,Wp] uint8, (top, left)): the image bytes in ``preprocess_u8``'s padded
    geometry, zeros in the padding -- the input of ``detector_forward_gray``."""
    _need_cuda(img, "the image batch")
    if img.dtype != torch.uint8 or img.dim() != 4 or img.shape[3] != 1:
        raise ValueError("expected a gray image batch [B, H, W, 1] uint8, got %s %s" % (img.dtype, tuple(img.shape)))
    img = img.contiguous()
    B, H, W, _ = img.shape
    Hp, Wp, top, left = pad_geometry(H, W, factor)
    g = torch.empty(B, Hp, Wp, dtype=torch.uint8, device=img.device)
    with torch.cuda.device(img.device):
        _ok(_pad_gray(_ptr(img), B, H, W, _ptr(g), Hp, Wp, top, left, _stream(img.device)))
    return g, (top, left)


def _crop_args(score, crop):
    _need_cuda(score, "the score map")
    if score.dim() == 2:
        score = score[None]
    score = score.contiguous().float()
    B, Hs, Ws = score.shape
    top, left, H, W = crop if crop is not None else (0, 0, Hs, Ws)
    return score, B, Hs, Ws, int(top), int(left), int(H), int(W)


def windowed_nms_topk(score, k, border=15, nms_size=15, crop=None):
    """score [B,Hs,Ws] CUDA -> (xy int32 [B,k,2], score fp32 [B,k], count int32 [B])."""
    score, B, Hs, Ws, top, left, H, W = _crop_args(score, crop)
    dev = score.device
    xy = torch.zeros(B, k, 2, dtype=torch.int32, device=dev)
    sc = torch.zeros(B, k, dtype=torch.float32, device=dev)
    cnt = torch.zeros(B, dtype=torch.int32, device=dev)
    nbytes = _nms_ws(B, H, W, k)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        _ok(_win_nms(_ptr(score), B, Hs, Ws, top, left, H, W, int(border), int(nms_size), int(k), _ptr(xy), _ptr(sc),
                     _ptr(cnt), _ptr(ws), nbytes, _stream(dev)))
    return xy, sc, cnt


def greedy_nms_topk(score, k, border=15, thr=0.001, radius=15, subpixel_ps=0, crop=None):
    """score [B,Hs,Ws] CUDA -> (xy int32 [B,k,2], score [B,k], dxdy fp32 [B,k,2] or None, count [B])."""
    score, B, Hs, Ws, top, left, H, W = _crop_args(score, crop)
    dev = score.device
    xy = torch.zeros(B, k, 2, dtype=torch.int32, device=dev)
    sc = torch.zeros(B, k, dtype=torch.float32, device=dev)
    dxdy = torch.zeros(B, k, 2, dtype=torch.float32, device=dev) if subpixel_ps else None
    cnt = torch.zeros(B, dtype=torch.int32, device=dev)
    nbytes = _nms_ws(B, H, W, k)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        _ok(_greedy_nms(_ptr(score), B, Hs, Ws, top, left, H, W, int(border), float(thr), int(radius), int(k),
                        int(subpixel_ps), _ptr(xy), _ptr(sc), _ptr(dxdy), _ptr(cnt), _ptr(ws), nbytes, _stream(dev)))
    return xy, sc, dxdy, cnt


_apply_nms_map = _sig("balf_apply_nms_map", c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P)
_subpixel = _sig("balf_subpixel_refine", c_int, _P, *([c_int] * 8), _P, c_int, c_int, _P, _P)


def apply_nms_map(score, nms_size, border=0):
    """dense apply_nms: score [B,H,W] (or [H,W]) CUDA -> same shape."""
    _need_cuda(score, "the score map")
    squeeze = score.dim() == 2
    s = (score[None] if squeeze else score).contiguous().float()
    out = torch.empty_like(s)
    with torch.cuda.device(s.device):
        _ok(_apply_nms_map(_ptr(s), s.shape[0], s.shape[1], s.shape[2], int(border), int(nms_size), _ptr(out),
                           _stream(s.device)))
    return out[0] if squeeze else out


def subpixel_refine(score, xy, ps, border=0, crop=None):
    """score [B,Hs,Ws], xy int32 [B,n,2] -> dxdy fp32 [B,n,2] (offset to add, includes -ps//2)."""
    score, B, Hs, Ws, top, left, H, W = _crop_args(score, crop)
    xy = xy.contiguous().to(torch.int32)
    n = xy.shape[1]
    dxdy = torch.zeros(B, n, 2, dtype=torch.float32, device=score.device)
    with torch.cuda.device(score.device):
        _ok(_subpixel(_ptr(score), B, Hs, Ws, top, left, H, W, int(border), _ptr(xy), n, int(ps), _ptr(dxdy),
                      _stream(score.device)))
    return dxdy


# ------------------------------------------------------------------------------------------ patches / HardNet / matching
_patch_level = _sig("balf_patch_pyramid_level", c_int, c_int, c_int, c_float, c_int)
_patch_ws = _sig("balf_patches_workspace_bytes", c_size_t, c_int, c_int, c_int)
_patches = _sig("balf_extract_patches_u8", c_int, _P, c_int, c_int, c_int, _P, _P, c_int, c_float, c_int, _P, _P, c_size_t, _P)
_hn_raw = _sig("balf_hardnet_raw_weight_count", ctypes.c_int64)
_hn_packed = _sig("balf_hardnet_packed_weight_count", ctypes.c_int64)
_hn_pack = _sig("balf_hardnet_pack_weights", c_int, _P, _P, _P)
_hn_ws = _sig("balf_hardnet_workspace_bytes", c_size_t, c_int, c_int)
_hn_fwd = _sig("balf_hardnet_forward", c_int, _P, _P, c_int, _P, _P, c_size_t, c_int, _P)
_match_ws = _sig("balf_match_workspace_bytes", c_size_t, c_int, c_int)
_match = _sig("balf_match_smnn", c_int, _P, c_int, _P, c_int, c_int, c_float, _P, _P, _P, _P, _P, c_size_t, _P)


def patch_pyramid_level(h, w, s_mult, ps=32):
    return int(_patch_level(int(h), int(w), float(s_mult), int(ps)))


def extract_patches_batch(gray, kpts, count, s_mult, ps=32):
    """gray [B,H,W] uint8 CUDA, kpts fp32 [B,K,2] (x, y), count int32 [B] or None -> patches fp32 [B,K,ps,ps]
    (rows beyond count[b] are zero)."""
    _need_cuda(gray, "the gray image batch")
    if gray.dtype != torch.uint8:
        raise ValueError("gray images must be uint8 (the /255 is fused into the sampling kernels)")
    if gray.dim() != 3:
        raise ValueError("gray images must be [B,H,W], got %s" % (tuple(gray.shape),))
    _same_device(kpts, gray, "the keypoints")
    B, H, W = gray.shape
    if kpts.dim() != 3 or kpts.shape[0] != B or kpts.shape[2] != 2:
        raise ValueError("keypoints must be [B=%d,K,2], got %s" % (B, tuple(kpts.shape)))
    if count is not None:
        _same_device(count, gray, "the keypoint counts")
        if count.shape != (B,) or count.is_floating_point() or count.is_complex():
            raise ValueError("keypoint counts must be integer [B=%d], got %s %s" % (B, count.dtype, tuple(count.shape)))
        count = count.contiguous().to(torch.int32)
    gray, kpts = gray.contiguous(), kpts.contiguous().float()
    K = kpts.shape[1]
    patches = torch.zeros(B, K, ps, ps, dtype=torch.float32, device=gray.device)
    if K == 0:
        return patches
    nbytes = _patch_ws(B, H, W)
    ws = _workspace(gray.device, nbytes)
    with torch.cuda.device(gray.device):
        _ok(_patches(_ptr(gray), B, H, W, _ptr(kpts), _ptr(count), K, float(s_mult), int(ps), _ptr(patches), _ptr(ws),
                     nbytes, _stream(gray.device)))
    return patches


def extract_patches(gray, kpts, s_mult, ps=32):
    """gray [H,W] uint8 CUDA, kpts fp32 [K,2] -> patches [K,1,ps,ps]  (demo_match.py:62-69)."""
    out = extract_patches_batch(gray[None], kpts[None], None, s_mult, ps)
    return out[0].unsqueeze(1)


def hardnet_pack_weights(raw):
    _need_cuda(raw, "the weight blob")
    if raw.numel() != _hn_raw() or raw.dtype != torch.float32:
        raise ValueError("HardNet weight blob has %d floats, expected %d" % (raw.numel(), _hn_raw()))
    raw = raw.contiguous()
    packed = torch.empty(_hn_packed(), dtype=torch.float32, device=raw.device)
    with torch.cuda.device(raw.device):
        _ok(_hn_pack(_ptr(raw), _ptr(packed), _stream(raw.device)))
    return packed


HARDNET_PRECISIONS = {"fp32": 0, "tf32": 1, "fp16": 2}


def hardnet_forward(patches, packed, precision="tf32"):
    """patches fp32 [N,1,32,32] CUDA -> descriptors fp32 [N,128]."""
    if precision not in HARDNET_PRECISIONS:
        raise ValueError("precision %r is not built (choose from %s)" % (precision, sorted(HARDNET_PRECISIONS)))
    prec = HARDNET_PRECISIONS[precision]
    _need_cuda(patches, "the patches")
    if patches.dim() != 4 or tuple(patches.shape[1:]) != (1, 32, 32):
        raise ValueError("patches must be [N,1,32,32], got %s" % (tuple(patches.shape),))
    patches = patches.contiguous().float()
    n = patches.shape[0]
    desc = torch.empty(n, 128, dtype=torch.float32, device=patches.device)
    if n == 0:
        return desc
    nbytes = _hn_ws(n, prec)
    ws = _workspace(patches.device, nbytes)
    with torch.cuda.device(patches.device):
        _ok(_hn_fwd(_ptr(packed), _ptr(patches), n, _ptr(desc), _ptr(ws), nbytes, prec, _stream(patches.device)))
    return desc


def match_smnn(d1, d2, th=0.99, want_dm=False):
    """d1 [n1,128], d2 [n2,128] CUDA -> (dists fp32 [M,1], ids int64 [M,2]) like kornia.feature.match_smnn
    (ids ascending in the first index).  want_dm=True also returns the fp32 distance matrix used."""
    _need_cuda(d1, "the descriptors d1")
    _same_device(d2, d1, "the descriptors d2")
    # an empty 1-D array stands for "no descriptors" (demo_match.extract_features returns np.array([]) then)
    d1, d2 = [d.reshape(0, 128) if d.dim() == 1 and d.numel() == 0 else d for d in (d1, d2)]
    for name, d in (("d1", d1), ("d2", d2)):
        if d.dim() != 2 or d.shape[1] != 128 or not d.is_floating_point():
            raise ValueError("descriptors %s must be floating-point [n,128], got %s %s" % (name, d.dtype, tuple(d.shape)))
    d1, d2 = d1.contiguous().float(), d2.contiguous().float()
    n1, n2 = d1.shape[0], d2.shape[0]
    dev = d1.device
    ids = torch.zeros(max(n1, 1), 2, dtype=torch.int32, device=dev)
    dist = torch.zeros(max(n1, 1), dtype=torch.float32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    dm = torch.empty(n1, n2, dtype=torch.float32, device=dev) if want_dm else None
    nbytes = _match_ws(n1, n2)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        _ok(_match(_ptr(d1), n1, _ptr(d2), n2, 128, float(th), _ptr(ids), _ptr(dist), _ptr(cnt), _ptr(dm), _ptr(ws),
                   nbytes, _stream(dev)))
    m = int(cnt[0])
    out = (dist[:m].reshape(m, 1), ids[:m].long())
    return out + (dm,) if want_dm else out


# ------------------------------------------------------------------------------------------ front end / multi-scale (SURVEY 8f)
_rgb2gray = _sig("balf_rgb_to_gray_u8", c_int, _P, c_int, c_int, c_int, _P, _P)
_preprocess_f32 = _sig("balf_preprocess_f32", c_int, _P, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, _P)
_resize_pre = _sig("balf_resize_preprocess_u8", c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int,
                   c_int, _P)
_merge_levels = _sig("balf_merge_levels_topk", c_int, c_int, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P)
MAX_LEVELS = 8


def rgb_to_gray(rgb):
    """rgb [B,H,W,3] (or [H,W,3]) uint8 CUDA -> gray uint8, PIL 'L' arithmetic."""
    _need_cuda(rgb, "the image")
    single = rgb.dim() == 3
    t = (rgb[None] if single else rgb).contiguous()
    B, H, W, C = t.shape
    if C != 3 or t.dtype != torch.uint8:
        raise ValueError("rgb_to_gray expects uint8 [.., H, W, 3]")
    gray = torch.empty(B, H, W, dtype=torch.uint8, device=t.device)
    with torch.cuda.device(t.device):
        _ok(_rgb2gray(_ptr(t), B, H, W, _ptr(gray), _stream(t.device)))
    return gray[0] if single else gray


def preprocess_f32(img, factor=64):
    """img [B,H,W,C] float32 CUDA (already normalised) -> (x [B,3,Hp,Wp] fp32, (top, left))."""
    _need_cuda(img, "the image batch")
    img = img.contiguous().float()
    B, H, W, C = img.shape
    Hp, Wp, top, left = pad_geometry(H, W, factor)
    x = torch.empty(B, 3, Hp, Wp, dtype=torch.float32, device=img.device)
    with torch.cuda.device(img.device):
        _ok(_preprocess_f32(_ptr(img), B, H, W, C, _ptr(x), Hp, Wp, top, left, _stream(img.device)))
    return x, (top, left)


def level_size(n, scale, level):
    """pyramid level extent: round-half-up of n * scale**level, at least 32 pixels."""
    return max(int(n * (scale ** level) + 0.5), 32)


def resize_preprocess_u8(img, hs, ws, factor=64):
    """img [B,H,W,C] uint8 CUDA -> bilinear level hs x ws, /255, padded CHW: (x [B,3,Hp,Wp], (top, left))."""
    _need_cuda(img, "the image batch")
    img = img.contiguous()
    B, H, W, C = img.shape
    Hp, Wp, top, left = pad_geometry(hs, ws, factor)
    x = torch.empty(B, 3, Hp, Wp, dtype=torch.float32, device=img.device)
    with torch.cuda.device(img.device):
        _ok(_resize_pre(_ptr(img), B, H, W, C, int(hs), int(ws), _ptr(x), Hp, Wp, top, left, _stream(img.device)))
    return x, (top, left)


def merge_levels_topk(lists, scales, k_out):
    """lists = [(xy int32 [B,K,2], score fp32 [B,K], count int32 [B]) per level] (CUDA), scales = [(sx, sy)] level-0
    pixels per level pixel -> (xy fp32 [B,k_out,2] in the level-0 frame, score [B,k_out], level int32 [B,k_out],
    count int32 [B]), ordered by (score descending, level ascending, rank inside the level)."""
    n = len(lists)
    if not 1 <= n <= MAX_LEVELS:
        raise ValueError("1 .. %d levels" % MAX_LEVELS)
    xy0, sc0, cn0 = lists[0]
    _need_cuda(xy0, "the keypoint lists")
    dev = xy0.device
    B, K = sc0.shape
    keep = [(xy.contiguous(), sc.contiguous(), cn.contiguous()) for xy, sc, cn in lists]
    arr = lambda items: (ctypes.c_void_p * n)(*[t.data_ptr() for t in items])
    fl = lambda items: (c_float * n)(*[float(v) for v in items])
    xy_out = torch.empty(B, k_out, 2, dtype=torch.float32, device=dev)
    sc_out = torch.empty(B, k_out, dtype=torch.float32, device=dev)
    lv_out = torch.empty(B, k_out, dtype=torch.int32, device=dev)
    cnt = torch.empty(B, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _ok(_merge_levels(n, arr([t[0] for t in keep]), arr([t[1] for t in keep]), arr([t[2] for t in keep]),
                          fl([s[0] for s in scales]), fl([s[1] for s in scales]), B, K, int(k_out), _ptr(xy_out),
                          _ptr(sc_out), _ptr(lv_out), _ptr(cnt), _stream(dev)))
    return xy_out, sc_out, lv_out, cnt


# ------------------------------------------------------------------------------------------ repeatability metrics (SURVEY 8 f3)
c_double = ctypes.c_double
_homog_pts = _sig("balf_apply_homography_to_points", c_int, _P, c_int, ctypes.POINTER(c_double), _P, _P)
_common_masks = _sig("balf_common_region_masks", c_int, ctypes.POINTER(c_double), c_int, c_int, c_int, c_int, c_int, _P, _P, _P)
_rep_ws = _sig("balf_repeatability_workspace_bytes", c_size_t, c_int, c_int)
_compute_rep = _sig("balf_compute_repeatability", c_int, _P, c_int, _P, c_int, c_double, c_double, c_double, c_double, _P, _P,
                    _P, _P, _P, c_size_t, _P)
_resize_rep = _sig("balf_resize_repeatability", c_int, _P, c_int, _P, c_int, ctypes.POINTER(c_double), c_int, c_int, c_int,
                   c_int, c_int, c_double, _P, _P, c_size_t, _P)


def _h9(h):
    import numpy as np
    a = np.ascontiguousarray(np.asarray(h, dtype=np.float64).reshape(9))
    return (c_double * 9)(*a.tolist())


def apply_homography_to_points(points, h):
    """points [n,4] float64 CUDA (x, y, radius, score), h 3x3 (host) -> [n,4] float64 CUDA."""
    _need_cuda(points, "the points")
    p = points.contiguous().double()
    out = torch.empty_like(p)
    with torch.cuda.device(p.device):
        _ok(_homog_pts(_ptr(p), p.shape[0], _h9(h), _ptr(out), _stream(p.device)))
    return out


def common_region_masks(h_dst_2_src, shape_src, shape_dst, device, border=15):
    """-> (mask_src uint8 [Hs,Ws], mask_dst uint8 [Hd,Wd]) CUDA."""
    ms = torch.empty(int(shape_src[0]), int(shape_src[1]), dtype=torch.uint8, device=device)
    md = torch.empty(int(shape_dst[0]), int(shape_dst[1]), dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        _ok(_common_masks(_h9(h_dst_2_src), ms.shape[0], ms.shape[1], md.shape[0], md.shape[1], int(border), _ptr(ms), _ptr(md),
                          _stream(device)))
    return ms, md


def compute_repeatability(src, dst, overlap_err=0.4, eps=1e-6, dist_match_thresh=3, radious_size=30.0):
    """src [n1,4], dst [n2,4] float64 CUDA -> (scalars float64 [8] CUDA, corr_s int32 [m,2], corr_m int32 [m,2], overflow int32 [1])
    (see include/balf_b200.h; the first scalars[2] / scalars[3] rows of corr_s / corr_m are valid)."""
    _need_cuda(src, "the points")
    s, d = src.contiguous().double(), dst.contiguous().double()
    n1, n2 = s.shape[0], d.shape[0]
    dev = s.device
    m = max(min(n1, n2), 1)
    scalars = torch.zeros(8, dtype=torch.float64, device=dev)
    cs = torch.zeros(m, 2, dtype=torch.int32, device=dev)
    cm = torch.zeros(m, 2, dtype=torch.int32, device=dev)
    ov = torch.zeros(1, dtype=torch.int32, device=dev)
    nbytes = _rep_ws(n1, n2)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        _ok(_compute_rep(_ptr(s), n1, _ptr(d), n2, float(overlap_err), float(eps), float(dist_match_thresh), float(radious_size),
                         _ptr(scalars), _ptr(cs), _ptr(cm), _ptr(ov), _ptr(ws), nbytes, _stream(dev)))
    return scalars, cs, cm, ov


def resize_repeatability(kp, wkp, h, shape_src, shape_dst, keep_k_points=1000, distance_thresh=5):
    """kp [n1,3], wkp [n2,3] float64 CUDA (row, col, prob) -> float64 [6] CUDA (see include/balf_b200.h)."""
    _need_cuda(kp, "the keypoints")
    a, b = kp.contiguous().double(), wkp.contiguous().double()
    dev = a.device
    out = torch.zeros(6, dtype=torch.float64, device=dev)
    nbytes = _rep_ws(a.shape[0], b.shape[0])
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        _ok(_resize_rep(_ptr(a), a.shape[0], _ptr(b), b.shape[0], _h9(h), int(shape_src[0]), int(shape_src[1]), int(shape_dst[0]),
                        int(shape_dst[1]), int(keep_k_points), float(distance_thresh), _ptr(out), _ptr(ws), nbytes, _stream(dev)))
    return out


_homog_ws = _sig("balf_homography_workspace_bytes", c_size_t, c_int, c_int, c_int)
_homog_ransac = _sig("balf_find_homography_ransac", c_int, _P, _P, _P, c_int, c_int, c_double, c_int, ctypes.c_uint64, _P, _P,
                     _P, _P, c_size_t, _P)


def _pair_inputs(name, p1, p2, count, K):
    """The shared validation of the RANSAC and pose calls -> (p1, p2 float64 [B,M,2], count int32 [B], K float64 [B,2,9]
    or None), all contiguous on p1's device.  CPU tensors raise RuntimeError, bad shapes ValueError."""
    _need_cuda(p1, "the matched points")
    _need_cuda(p2, "the matched points")
    _need_cuda(count, "the match counts")
    if K is not None:
        _need_cuda(K, "the camera matrices")
    a, b = p1.contiguous().double(), p2.contiguous().double()
    cnt = count.contiguous().to(torch.int32)
    if a.dim() != 3 or a.shape[2] != 2 or b.shape != a.shape or cnt.shape != (a.shape[0],):
        raise ValueError("%s: p1, p2 must be [B,M,2] and count [B]" % name)
    if K is not None:
        if K.device != a.device:
            raise ValueError("%s: K is on %s, expected %s" % (name, K.device, a.device))
        if not K.is_floating_point() or tuple(K.shape) not in ((a.shape[0], 2, 3, 3), (a.shape[0], 2, 9)):
            raise ValueError("%s: K must be floating-point [B,2,3,3] or [B,2,9]" % name)
        K = K.contiguous().double().reshape(a.shape[0], 2, 9)
    return a, b, cnt, K


def _ransac(fn_ws, fn, name, p1, p2, count, thr, iters, seed, K=None):
    a, b, cnt, k = _pair_inputs(name, p1, p2, count, K)
    B, M, _ = a.shape
    dev = a.device
    out = torch.empty(B, 3, 3, dtype=torch.float64, device=dev)
    mask = torch.empty(B, M, dtype=torch.uint8, device=dev)
    n_in = torch.empty(B, dtype=torch.int32, device=dev)
    nbytes = fn_ws(B, M, int(iters))                     # 0 for arguments the call itself rejects
    ws = _workspace(dev, nbytes)
    kp = () if K is None else (_ptr(k),)
    with torch.cuda.device(dev):
        _ok(fn(_ptr(a), _ptr(b), _ptr(cnt), *kp, B, M, float(thr), int(iters), int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(out),
               _ptr(mask), _ptr(n_in), _ptr(ws), nbytes, _stream(dev)))
    return out, mask, n_in


def find_homography_ransac(p1, p2, count, thr, iters, seed):
    """p1, p2 float64 [B,M,2] CUDA (x, y) of each pair's matches, count int32 [B] valid rows per pair -> (H float64 [B,3,3],
    inlier mask uint8 [B,M], n_inliers int32 [B]) on the device; RANSAC semantics in include/balf_b200.h."""
    return _ransac(_homog_ws, _homog_ransac, "find_homography_ransac", p1, p2, count, thr, iters, seed)


_fund_ws = _sig("balf_fundamental_workspace_bytes", c_size_t, c_int, c_int, c_int)
_fund_ransac = _sig("balf_find_fundamental_ransac", c_int, _P, _P, _P, c_int, c_int, c_double, c_int, ctypes.c_uint64, _P, _P,
                    _P, _P, c_size_t, _P)


def find_fundamental_ransac(p1, p2, count, thr, iters, seed):
    """p1, p2 float64 [B,M,2] CUDA (x, y) of each pair's matches, count int32 [B] valid rows per pair -> (F float64 [B,3,3]
    with x2^T F x1 = 0, unit Frobenius norm, inlier mask uint8 [B,M], n_inliers int32 [B]) on the device; RANSAC semantics
    in include/balf_b200.h (balf_find_fundamental_ransac)."""
    return _ransac(_fund_ws, _fund_ransac, "find_fundamental_ransac", p1, p2, count, thr, iters, seed)


_ess_ws = _sig("balf_essential_workspace_bytes", c_size_t, c_int, c_int, c_int)
_ess_ransac = _sig("balf_find_essential_ransac", c_int, _P, _P, _P, _P, c_int, c_int, c_double, c_int, ctypes.c_uint64, _P,
                   _P, _P, _P, c_size_t, _P)
_recover_pose = _sig("balf_recover_pose", c_int, _P, _P, _P, _P, _P, _P, c_int, c_int, c_double, _P, _P, _P, _P, _P)


def find_essential_ransac(p1, p2, count, K, thr, iters, seed):
    """p1, p2 float64 [B,M,2] CUDA pixel (x, y) of each pair's matches, count int32 [B] valid rows per pair, K [B,2,3,3]
    (or [B,2,9]) the camera matrices K1, K2 of each pair on the same device -> (E float64 [B,3,3] with x2'^T E x1' = 0 in
    calibrated coordinates, unit Frobenius norm, inlier mask uint8 [B,M], n_inliers int32 [B]) on the device; thr in
    pixels.  RANSAC semantics in include/balf_b200.h (balf_find_essential_ransac)."""
    return _ransac(_ess_ws, _ess_ransac, "find_essential_ransac", p1, p2, count, thr, iters, seed, K=K)


def recover_pose(E, p1, p2, count, K, mask=None, dist_thresh=50.0):
    """E [B,3,3] (or [B,9]), p1, p2 [B,M,2], count [B] and K [B,2,3,3] (or [B,2,9]) on one CUDA device, mask [B,M] (bool or
    uint8; None: every valid row) -> (R float64 [B,3,3], t float64 [B,3], pose mask uint8 [B,M], n_good int32 [B]): the
    pose X2 = R X1 + t of each pair whose candidate puts the most masked matches in front of both cameras
    (include/balf_b200.h, balf_recover_pose)."""
    a, b, cnt, k = _pair_inputs("recover_pose", p1, p2, count, K)
    B, M, _ = a.shape
    dev = a.device
    _need_cuda(E, "E")
    if E.device != dev:
        raise ValueError("recover_pose: E is on %s, expected %s" % (E.device, dev))
    if not E.is_floating_point() or tuple(E.shape) not in ((B, 3, 3), (B, 9)):
        raise ValueError("recover_pose: E must be floating-point [B,3,3] or [B,9]")
    e = E.contiguous().double()
    m = None
    if mask is not None:
        _need_cuda(mask, "the mask")
        if mask.device != dev:
            raise ValueError("recover_pose: mask is on %s, expected %s" % (mask.device, dev))
        if tuple(mask.shape) != (B, M) or mask.dtype not in (torch.bool, torch.uint8):
            raise ValueError("recover_pose: mask must be bool or uint8 [B,M]")
        m = mask.contiguous().to(torch.uint8)
    R = torch.empty(B, 3, 3, dtype=torch.float64, device=dev)
    t = torch.empty(B, 3, dtype=torch.float64, device=dev)
    pmask = torch.empty(B, M, dtype=torch.uint8, device=dev)
    n_good = torch.empty(B, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _ok(_recover_pose(_ptr(e), _ptr(a), _ptr(b), _ptr(cnt), _ptr(k), _ptr(m), B, M, float(dist_thresh), _ptr(R), _ptr(t),
                          _ptr(pmask), _ptr(n_good), _stream(dev)))
    return R, t, pmask, n_good


_box_nms = _sig("balf_box_nms_map", c_int, _P, c_int, c_int, c_int, c_float, c_float, c_float, c_int, _P, _P, c_size_t, _P)


def box_nms_map(prob, size=4, iou=0.1, min_prob=0.015, keep_top_k=-1):
    """prob [B,H,W] float32 CUDA -> [B,H,W]: repeatability_tools.box_nms on every map of the batch."""
    _need_cuda(prob, "the score map")
    p = prob.contiguous().float()
    B, H, W = p.shape
    out = torch.empty_like(p)
    k = int(keep_top_k) if keep_top_k and keep_top_k > 0 else 0
    nbytes = _nms_ws(B, H, W, max(k, 1)) + 12 * B * k + 256
    ws = _workspace(p.device, nbytes)
    with torch.cuda.device(p.device):
        _ok(_box_nms(_ptr(p), B, H, W, float(size), float(iou), float(min_prob), k, _ptr(out), _ptr(ws), nbytes, _stream(p.device)))
    return out


# ------------------------------------------------------------------------------------------ NCCL gather (SURVEY 8e)
_nccl_uid = _sig("balf_nccl_unique_id", c_int, _P)
_nccl_create = _sig("balf_nccl_comm_create", c_int, _P, c_int, c_int, ctypes.POINTER(c_void_p))
_nccl_destroy = _sig("balf_nccl_comm_destroy", c_int, _P)
_gather_ws = _sig("balf_gather_workspace_bytes", c_size_t, c_int, c_int, c_int)
_gather_kp = _sig("balf_gather_keypoints", c_int, _P, c_int, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, c_size_t, _P)


def nccl_unique_id():
    """128-byte ncclUniqueId (bytes); rank 0 creates it and the caller distributes it."""
    buf = ctypes.create_string_buffer(128)
    _ok(_nccl_uid(buf))
    return buf.raw


def nccl_comm_create(uid, world, rank, device):
    comm = c_void_p()
    with torch.cuda.device(device):
        _ok(_nccl_create(ctypes.create_string_buffer(bytes(uid), 128), int(world), int(rank), ctypes.byref(comm)))
    return comm


def nccl_comm_destroy(comm):
    _ok(_nccl_destroy(comm))


def gather_keypoints(comm, world, xy, score, count):
    """this rank's (xy int32 [B,K,2], score fp32 [B,K], count int32 [B]) -> the records of every rank, in rank order."""
    _need_cuda(xy, "the keypoint records")
    xy, score, count = xy.contiguous(), score.contiguous(), count.contiguous()
    B, K, _ = xy.shape
    dev = xy.device
    xy_all = torch.empty(world * B, K, 2, dtype=torch.int32, device=dev)
    sc_all = torch.empty(world * B, K, dtype=torch.float32, device=dev)
    cn_all = torch.empty(world * B, dtype=torch.int32, device=dev)
    nbytes = _gather_ws(world, B, K)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        _ok(_gather_kp(comm, world, _ptr(xy), _ptr(score), _ptr(count), B, K, _ptr(xy_all), _ptr(sc_all), _ptr(cn_all), _ptr(ws),
                       nbytes, _stream(dev)))
    return xy_all, sc_all, cn_all
