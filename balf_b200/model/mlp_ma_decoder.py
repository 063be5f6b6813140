"""B200-native drop-in for the reference's ``balf/model/mlp_ma_decoder.py``.

Same constructor (``MLP_MA_DECODER(model_cfg)`` with the eight keys read at
mlp_ma_decoder.py:249-256), same ``forward(x) -> {'logits', 'prob'}`` contract
(mlp_ma_decoder.py:278-285, decoder.py:16-30) and the same 167-entry ``state_dict`` layout
(SURVEY.md appendix A), but the module owns *parameters only*: the whole forward is one call
into the C-ABI library (``balf_detector_forward``, include/balf_b200.h), which runs
hand-written sm_100a kernels.  There is no eager / CPU path -- a CPU tensor raises.

The parameter tree is created leaf by leaf in the reference's construction order, so
``torch.manual_seed(s); MLP_MA_DECODER(cfg)`` yields bit-identical initial weights to the
reference (checked in tests/test_boundary.py).
"""
import torch
import torch.nn as nn

from .. import _capi
from .decoder import DetectorHead

_P = "residual_split_head_multi_axis_gmlp_layer"
_R = "residual_channel_attention_block"


def down_layout(cin, c, cells, block_px, proj=2, gfac=2, bfac=2, red=4):
    """Leaves of one ``Down`` stage in reference registration order:
    (dotted name, kind, out_features, in_features).  kind 'ln' has (C,) weight and bias."""
    g, b = _P + ".grid_gmlp_layer", _P + ".block_gmlp_layer"
    return (
        ("conv.0", "linear", c, cin),
        (_P + ".norm", "ln", c, c),
        (_P + ".dense1", "linear", c * proj, c),
        (g + ".norm", "ln", c, c),
        (g + ".dense1", "linear", c * gfac, c),
        (g + ".grid_gating_unit.norm", "ln", c, c),
        (g + ".grid_gating_unit.dense", "linear", cells, cells),
        (g + ".dense2", "linear", c, c),
        (b + ".norm", "ln", c, c),
        (b + ".dense1", "linear", c * bfac, c),
        (b + ".block_gating_unit.norm", "ln", c, c),
        (b + ".block_gating_unit.dense", "linear", block_px, block_px),
        (b + ".dense2", "linear", c, c),
        (_P + ".dense2", "linear", c, c * proj),
        (_R + ".norm", "ln", c, c),
        (_R + ".conv1", "linear", c, c),
        (_R + ".conv2", "linear", c, c),
        (_R + ".calayer.excite.0", "linear", c // red, c),
        (_R + ".calayer.excite.2", "linear", c, c // red),
        ("conv2", "linear", c, c),
    )


class _Scope(nn.Module):
    """Pure name-space node of the parameter tree (no behaviour)."""

    def put(self, dotted, leaf):
        node = self
        *path, last = dotted.split(".")
        for name in path:
            if name not in node._modules:
                node.add_module(name, _Scope())
            node = node._modules[name]
        node.add_module(last, leaf)

    def forward(self, *a, **k):
        raise RuntimeError("parameter scope only; the forward lives in balf_detector_forward (CUDA)")


class Down(_Scope):
    """One encoder stage (reference: mlp_ma_decoder.py:201-244) -- parameters only."""

    def __init__(self, in_ch, out_ch, grid_size, block_size, grid_gmlp_factor=2, block_gmlp_factor=2,
                 input_proj_factor=2, channels_reduction=4, downsample=True):
        super().__init__()
        self.downsample = downsample
        self.dims = (in_ch, out_ch)
        for name, kind, n_out, n_in in down_layout(in_ch, out_ch, grid_size[0] * grid_size[1],
                                                   block_size[0] * block_size[1], input_proj_factor,
                                                   grid_gmlp_factor, block_gmlp_factor, channels_reduction):
            self.put(name, nn.LayerNorm(n_out) if kind == "ln" else nn.Linear(n_in, n_out))


class MLP_MA_DECODER(nn.Module):
    def __init__(self, model_cfg):
        super().__init__()
        dims = list(model_cfg["en_embed_dims"])
        self.arch = dict(
            dims=dims, grid=tuple(model_cfg["grid_size"]), block=tuple(model_cfg["block_size"]),
            gfac=model_cfg["grid_gmlp_factor"], bfac=model_cfg["block_gmlp_factor"],
            proj=model_cfg["input_proj_factor"], red=model_cfg["channels_reduction"], cell=model_cfg["cell_size"])
        _capi.check_supported_arch(self.arch)
        for i in range(4):
            self.add_module("down%d" % (i + 1), Down(
                dims[i], dims[i + 1], self.arch["grid"], self.arch["block"], self.arch["gfac"], self.arch["bfac"],
                self.arch["proj"], self.arch["red"], downsample=i < 3))
        self.detector_head = DetectorHead(input_channel=dims[4], cell_size=self.arch["cell"])
        self._packed = None          # (key, device weight blob) cache, see _weights()
        # 'tf32':  tcgen05 tensor-core kernels, fp16 / tf32 operands (11-bit significand, round-to-nearest) with fp32
        #          accumulation -- score maps within rel 1e-3 of the reference (measured max 7e-4, mean 1e-4);
        # 'f16x3': the same kernels in split precision: every operand is an fp16 hi + lo pair, every product runs as three
        #          MMAs (hi*hi + lo*hi + hi*lo) -- fp32-class score maps (measured max rel 5e-6 against the FFMA path, 100 %
        #          greedy keypoint agreement on every tested image) at ~0.7x the 'tf32' throughput, 6x the 'fp32' one;
        # 'fp32':  FFMA kernels, bit-level class of the reference's own fp32 arithmetic (rel ~2e-6);
        # 'auto' (default): what a drop-in user of the reference expects from each call -- 'f16x3' for ``forward`` and for
        #          the demo path (detect / extract_features / extract_matches: the greedy nms_fast amplifies 1e-4 score
        #          perturbations into different suppression chains, 'tf32' measured 98.7-99.8 % keypoint agreement there),
        #          'tf32' for the batched windowed-NMS throughput path (99.8 % agreement).  See DESIGN.md section 4.1.
        self.precision = "auto"

    def resolve_precision(self, nms=None):
        """the arithmetic a call runs in: an explicit ``self.precision`` wins; 'auto' -> 'tf32' for the windowed
        (validation / throughput) extraction, 'f16x3' (fp32-class results on the tensor cores) otherwise."""
        if self.precision != "auto":
            return self.precision
        return "tf32" if nms == "windowed" else "f16x3"

    # -- weight blob: every floating tensor of the state_dict, concatenated in state_dict order
    def _weights(self, device):
        tensors = [t for t in self.state_dict(keep_vars=True).values() if t.is_floating_point()]
        key = (str(device),) + tuple((t.data_ptr(), t._version) for t in tensors)
        if self._packed is None or self._packed[0] != key:
            raw = torch.cat([t.detach().reshape(-1).to(device=device, dtype=torch.float32) for t in tensors])
            self._packed = (key, _capi.detector_pack_weights(raw, self.arch))
        return self._packed[1]

    def forward(self, x, precision=None, want_logits=True):
        """reference contract: {'logits': [B,65,H/8,W/8], 'prob': [B,H,W]}; ``want_logits=False`` (the extraction pipelines of this
        package, which only read 'prob') skips the logits tensor -- 'logits' is then None."""
        if self.training:
            raise RuntimeError("balf_b200 implements the inference path only: call .eval() first")
        if not x.is_cuda:
            raise RuntimeError("balf_b200 has no CPU path: move the model and the input to a CUDA device")
        if x.dim() != 4 or x.shape[1] != self.arch["dims"][0]:
            raise ValueError("expected input [B, %d, H, W], got %s" % (self.arch["dims"][0], tuple(x.shape)))
        precision = precision or self.resolve_precision()
        logits, prob = _capi.detector_forward(x, self._weights(x.device), self.arch, precision, want_logits=want_logits)
        return {"logits": logits, "prob": prob}

    def forward_gray(self, g, precision=None, want_logits=False):
        """``forward`` for a gray uint8 image given as its padded byte plane g [B,Hp,Wp] uint8 (``_capi.pad_gray_u8``): the
        result is bit-identical to ``forward(preprocess_u8(img)[0], 'tf32')``, but stage 1 gathers its pixel-local chain from
        per-byte tables instead of computing it per pixel (balf_detector_forward_gray).  Only 'tf32' exists on this path;
        ``precision=None`` means 'tf32' unless ``self.precision`` names another (which then raises)."""
        if self.training:
            raise RuntimeError("balf_b200 implements the inference path only: call .eval() first")
        if not g.is_cuda:
            raise RuntimeError("balf_b200 has no CPU path: move the model and the input to a CUDA device")
        if self.arch["dims"][0] != 3:
            raise ValueError("forward_gray needs a detector with a 3-channel input, this one has %d" % self.arch["dims"][0])
        precision = precision or ("tf32" if self.precision == "auto" else self.precision)
        logits, prob = _capi.detector_forward_gray(g, self._weights(g.device), self.arch, precision, want_logits=want_logits)
        return {"logits": logits, "prob": prob}
