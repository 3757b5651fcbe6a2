"""Parameter layouts of the three hot-path networks, keyed exactly like the reference's
``state_dict`` so that ``model.load_state_dict(torch.load(...)['model_state_dict'])``
(src/main/tta.py:86-87,168-169) works unchanged.

Only names, shapes and initial values live here; the arithmetic is in ``engine.py`` and
runs on the CUDA kernels.  Key layout: SURVEY.md appendix A.6; constructors mirrored:
``UnetPlusPlusStar.__init__`` (archs/unetplusplusstar.py:400-456),
``deep_supunetplusplus.UnetPlusPlus.__init__`` (:183-249) and smp 0.1.3 ``Unet``.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, List, Tuple

import torch
from torch import nn

DECODER_CHANNELS = (256, 128, 64, 32, 16)


class ParamSpec:
    """Ordered ``key -> tensor`` with a buffer flag and alias groups (shared storage)."""

    def __init__(self, seed_generator: torch.Generator):
        self.tensors: "OrderedDict[str, torch.Tensor]" = OrderedDict()
        self.is_buffer: Dict[str, bool] = {}
        self.alias_of: Dict[str, str] = {}
        self.g = seed_generator

    # -- initialisers (same families as the reference constructors use) --------
    def _kaiming_uniform(self, shape, a=math.sqrt(5.0)):
        fan_in = shape[1] * (shape[2] if len(shape) > 2 else 1) * (shape[3] if len(shape) > 3 else 1)
        gain = math.sqrt(2.0 / (1 + a * a))
        bound = gain * math.sqrt(3.0 / fan_in)
        return (torch.rand(shape, generator=self.g) * 2 - 1) * bound

    def _bias_default(self, cout, fan_in):
        bound = 1.0 / math.sqrt(fan_in)
        return (torch.rand(cout, generator=self.g) * 2 - 1) * bound

    def add(self, key, tensor, buffer=False):
        assert key not in self.tensors, key
        self.tensors[key] = tensor
        self.is_buffer[key] = buffer

    def conv(self, key, cout, cin, k, bias=False, init="default", ndim=2):
        shape = (cout, cin, k, k) if ndim == 2 else (cout, cin, k)
        if init == "decoder":      # kaiming_uniform_(fan_in, relu), bias 0  (unetplusplusstar.py:354-359)
            w = self._kaiming_uniform(shape, a=0.0)
        elif init == "head":       # xavier_uniform_, bias 0 (smp initialize_head)
            fan_in, fan_out = cin * k * k, cout * k * k
            bound = math.sqrt(6.0 / (fan_in + fan_out))
            w = (torch.rand(shape, generator=self.g) * 2 - 1) * bound
        else:                      # nn.Conv default
            w = self._kaiming_uniform(shape)
        self.add(key + ".weight", w)
        if bias:
            fan_in = cin * (k * k if ndim == 2 else k)
            self.add(key + ".bias", torch.zeros(cout) if init in ("decoder", "head") else self._bias_default(cout, fan_in))

    def bn(self, key, c):
        self.add(key + ".weight", torch.ones(c))
        self.add(key + ".bias", torch.zeros(c))
        self.add(key + ".running_mean", torch.zeros(c), buffer=True)
        self.add(key + ".running_var", torch.ones(c), buffer=True)
        self.add(key + ".num_batches_tracked", torch.zeros((), dtype=torch.long), buffer=True)

    def alias_prefix(self, src_prefix: str, dst_prefix: str):
        """Register every key under src_prefix again under dst_prefix, sharing storage
        (encoder.layer4.1 and .2 are one module object, unetplusplusstar.py:323-328)."""
        for key in [k for k in self.tensors if k.startswith(src_prefix + ".")]:
            new = dst_prefix + key[len(src_prefix):]
            self.tensors[new] = self.tensors[key]
            self.is_buffer[new] = self.is_buffer[key]
            self.alias_of[new] = key


# ------------------------------------------------------------------- encoders
def _bottleneck(s: ParamSpec, p, inplanes, planes, downsample, groups=1, base_width=64, se=True):
    """Bottleneck keys: Cadene SEResNetBottleneck / SEResNeXtBottleneck (se=True) or torchvision Bottleneck
    (se=False).  conv2 is the 3x3 with ``groups``; width = floor(planes * base_width / 64) * groups (planes for
    the SE-ResNet and ResNet-50 blocks); the 1x1 downsample (kernel 1, padding 0) follows the block's own modules."""
    width = planes * base_width // 64 * groups
    s.conv(p + ".conv1", width, inplanes, 1)
    s.bn(p + ".bn1", width)
    s.conv(p + ".conv2", width, width // groups, 3)
    s.bn(p + ".bn2", width)
    s.conv(p + ".conv3", planes * 4, width, 1)
    s.bn(p + ".bn3", planes * 4)
    if se:
        s.conv(p + ".se_module.fc1", planes * 4 // 16, planes * 4, 1, bias=True)
        s.conv(p + ".se_module.fc2", planes * 4, planes * 4 // 16, 1, bias=True)
    if downsample:
        s.conv(p + ".downsample.0", planes * 4, inplanes, 1)
        s.bn(p + ".downsample.1", planes * 4)


_LAYERS_50 = ((64, 3), (128, 4), (256, 6), (512, 3))


def _senet_layers(s: ParamSpec, p, n_layers: int, groups=1, base_width=64):
    """Cadene SENet encoder: se_resnet50 (groups 1) or se_resnext50_32x4d (groups 32, base_width 4)."""
    s.conv(p + ".layer0.conv1", 64, 3, 7)
    s.bn(p + ".layer0.bn1", 64)
    inplanes = 64
    for li, (planes, blocks) in enumerate(_LAYERS_50[:n_layers], start=1):
        for b in range(blocks):
            _bottleneck(s, f"{p}.layer{li}.{b}", inplanes, planes, b == 0, groups, base_width)
            inplanes = planes * 4


def _resnet50(s: ParamSpec, p, groups=1, base_width=64):
    """torchvision ResNet-50 / ResNeXt-50 as smp's ResNetEncoder keeps it (no fc)."""
    s.conv(p + ".conv1", 64, 3, 7)
    s.bn(p + ".bn1", 64)
    inplanes = 64
    for li, (planes, blocks) in enumerate(_LAYERS_50, start=1):
        for b in range(blocks):
            _bottleneck(s, f"{p}.layer{li}.{b}", inplanes, planes, b == 0, groups, base_width, se=False)
            inplanes = planes * 4


def _axial_attention(s: ParamSpec, p, dim, in_channels, heads=8, d_kq=8):
    d_v = in_channels // heads
    s.conv(p + ".to_qvk.0", heads * (2 * d_kq + d_v), in_channels, 1, ndim=1)
    s.bn(p + ".to_qvk.1", heads * (2 * d_kq + d_v))
    s.add(p + ".RelativePosEncQKV.relative", torch.randn(2 * d_kq + d_v, 2 * dim - 1, generator=s.g))
    idx = (torch.arange(dim).view(dim, 1) - torch.arange(dim).view(1, dim) + dim - 1).reshape(-1)
    s.add(p + ".RelativePosEncQKV.flatten_index", idx, buffer=True)
    s.bn(p + ".attention_norm", heads * 3)
    s.bn(p + ".out_norm", in_channels * 2)


def _cross_axial_attention(s: ParamSpec, p, dim, in_channels, skip_channels, heads=4, d_kq=8):
    d_v = skip_channels // heads
    s.conv(p + ".to_kq.0", heads * 2 * d_kq, in_channels, 1, ndim=1)
    s.bn(p + ".to_kq.1", heads * 2 * d_kq)
    s.conv(p + ".to_v.0", heads * d_v, skip_channels, 1, ndim=1)
    s.bn(p + ".to_v.1", heads * d_v)
    s.add(p + ".RelativePosEncQKV.relative", torch.randn(2 * d_kq + d_v, 2 * dim - 1, generator=s.g))
    idx = (torch.arange(dim).view(dim, 1) - torch.arange(dim).view(1, dim) + dim - 1).reshape(-1)
    s.add(p + ".RelativePosEncQKV.flatten_index", idx, buffer=True)
    s.bn(p + ".attention_norm", heads * 3)
    s.bn(p + ".out_norm", skip_channels * 2)


def _axial_block(s: ParamSpec, p, in_channels, out_channels, dim, down_sample):
    s.conv(p + ".in_conv1x1.0", 512, in_channels, 1)
    s.bn(p + ".in_conv1x1.1", 512)
    s.conv(p + ".out_conv1x1.0", out_channels, 512, 1)
    s.bn(p + ".out_conv1x1.1", out_channels)
    _axial_attention(s, p + ".height_att", dim, 512)
    _axial_attention(s, p + ".width_att", dim, 512)
    if down_sample:
        s.conv(p + ".shortcut.0", out_channels, in_channels, 3, bias=True)
        s.bn(p + ".shortcut.1", out_channels)
        s.bn(p + ".att_down.1", 512)


def _resnet34(s: ParamSpec, p):
    s.conv(p + ".conv1", 64, 3, 7)
    s.bn(p + ".bn1", 64)
    inplanes = 64
    for li, (planes, blocks, stride) in enumerate(((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)), start=1):
        for b in range(blocks):
            q = f"{p}.layer{li}.{b}"
            s.conv(q + ".conv1", planes, inplanes, 3)
            s.bn(q + ".bn1", planes)
            s.conv(q + ".conv2", planes, planes, 3)
            s.bn(q + ".bn2", planes)
            if b == 0 and (stride != 1 or inplanes != planes):
                s.conv(q + ".downsample.0", planes, inplanes, 1)
                s.bn(q + ".downsample.1", planes)
            inplanes = planes


#: smp 0.1.3 encoder names on the hot path -> parameter layout under "encoder."
SMP_ENCODERS = {
    "resnet34": _resnet34,
    "resnet50": _resnet50,
    "resnext50_32x4d": lambda s, p: _resnet50(s, p, groups=32, base_width=4),
    "se_resnet50": lambda s, p: _senet_layers(s, p, 4),
    "se_resnext50_32x4d": lambda s, p: _senet_layers(s, p, 4, groups=32, base_width=4),
}


# ------------------------------------------------------------------- decoders
def _scse(s: ParamSpec, p, c):
    s.conv(p + ".attention.cSE.1", c // 16, c, 1, bias=True, init="decoder")
    s.conv(p + ".attention.cSE.3", c, c // 16, 1, bias=True, init="decoder")
    s.conv(p + ".attention.sSE.0", 1, c, 1, bias=True, init="decoder")


def dense_decoder_blocks(encoder_channels, decoder_channels=DECODER_CHANNELS) -> List[Tuple[str, int, int, int, int]]:
    """(name, layer_idx, in_ch, skip_ch, out_ch) for every UNet++ decoder block
    (unetplusplusstar.py:202-233 == deep_supunetplusplus.py:85-110)."""
    enc = list(encoder_channels[1:])[::-1]
    in_channels = [enc[0]] + list(decoder_channels[:-1])
    skip_channels = list(enc[1:]) + [0]
    out_channels = list(decoder_channels)
    blocks = []
    for layer_idx in range(len(in_channels) - 1):
        for depth_idx in range(layer_idx + 1):
            if depth_idx == 0:
                in_ch = in_channels[layer_idx]
                skip_ch = skip_channels[layer_idx] * (layer_idx + 1)
                out_ch = out_channels[layer_idx]
            else:
                out_ch = skip_channels[layer_idx]
                skip_ch = skip_channels[layer_idx] * (layer_idx + 1 - depth_idx)
                in_ch = skip_channels[layer_idx - 1]
            blocks.append((f"x_{depth_idx}_{layer_idx}", layer_idx, in_ch, skip_ch, out_ch))
    blocks.append((f"x_0_{len(in_channels) - 1}", 0, in_channels[-1], 0, out_channels[-1]))
    return blocks


def _conv_bn(s: ParamSpec, p, cin, cout, bn_idx, use_bn=True):
    s.conv(p + ".0", cout, cin, 3, bias=not use_bn, init="decoder")
    if use_bn:
        s.bn(f"{p}.{bn_idx}", cout)


def build_unetplusplusstar(s: ParamSpec, base_dim=32, decoder_attention_type="scse", classes=1,
                           decoder_use_batchnorm=True):
    p = "encoder"
    _senet_layers(s, p, 3)
    _axial_block(s, p + ".layer4.0", 1024, 2048, base_dim * 2, True)
    _axial_block(s, p + ".layer4.1", 2048, 2048, base_dim, False)
    s.alias_prefix(p + ".layer4.1", p + ".layer4.2")
    enc_ch = (3, 64, 256, 512, 1024, 2048)
    for name, layer_idx, in_ch, skip_ch, out_ch in dense_decoder_blocks(enc_ch):
        q = f"decoder.blocks.{name}"
        use_catt = layer_idx in (0, 1) and skip_ch > 0          # unetplusplusstar.py:226-231
        _conv_bn(s, q + ".conv1", in_ch + skip_ch, out_ch, 2, decoder_use_batchnorm)
        _conv_bn(s, q + ".conv2", out_ch, out_ch, 2, decoder_use_batchnorm)
        if use_catt:
            dim = base_dim * (2 ** layer_idx)
            cr = skip_ch // 16
            s.conv(q + ".init_conv.1", cr, skip_ch, 1, bias=True, init="decoder")
            s.bn(q + ".init_conv.2", cr)
            _cross_axial_attention(s, q + ".h_catt", dim, in_ch, cr)
            _cross_axial_attention(s, q + ".w_catt", dim, in_ch, cr)
            s.conv(q + ".down_sample", cr, skip_ch, 1, init="decoder")
            s.conv(q + ".up_sample", skip_ch, cr, 1, init="decoder")
        elif decoder_attention_type == "scse":
            if skip_ch > 0:
                _scse(s, q + ".attention1", in_ch + skip_ch)
            _scse(s, q + ".attention2", out_ch)
    s.conv("segmentation_head.0", classes, DECODER_CHANNELS[-1], 3, bias=True, init="head")
    s.add("classification_head.3.weight", torch.randn(classes, 2048, generator=s.g) * 0.02)
    s.add("classification_head.3.bias", torch.zeros(classes))
    for i in range(3):
        s.conv(f"deep_segmentation_head.{i}.0", classes, DECODER_CHANNELS[-3], 3, bias=True, init="head")


def build_smp_style(s: ParamSpec, encoder_name, decoder="unetplusplus", decoder_attention_type=None, classes=1,
                    decoder_use_batchnorm=True, deep_heads=False):
    if encoder_name not in SMP_ENCODERS:
        raise KeyError(f"encoder {encoder_name!r} is outside the B200 hot path ({', '.join(SMP_ENCODERS)})")
    SMP_ENCODERS[encoder_name](s, "encoder")
    enc_ch = (3, 64, 64, 128, 256, 512) if encoder_name == "resnet34" else (3, 64, 256, 512, 1024, 2048)
    if decoder == "unetplusplus":
        blocks = [(n, i, s_, o) for n, _, i, s_, o in dense_decoder_blocks(enc_ch)]
    else:  # smp Unet
        enc = list(enc_ch[1:])[::-1]
        in_ch = [enc[0]] + list(DECODER_CHANNELS[:-1])
        skip_ch = list(enc[1:]) + [0]
        blocks = [(str(i), in_ch[i], skip_ch[i], DECODER_CHANNELS[i]) for i in range(5)]
    for name, in_ch_, skip_ch_, out_ch in blocks:
        q = f"decoder.blocks.{name}"
        _conv_bn(s, q + ".conv1", in_ch_ + skip_ch_, out_ch, 1, decoder_use_batchnorm)
        _conv_bn(s, q + ".conv2", out_ch, out_ch, 1, decoder_use_batchnorm)
        if decoder_attention_type == "scse":
            _scse(s, q + ".attention1", in_ch_ + skip_ch_)
            _scse(s, q + ".attention2", out_ch)
    s.conv("segmentation_head.0", classes, DECODER_CHANNELS[-1], 3, bias=True, init="head")
    if deep_heads:
        for i in range(3):
            s.conv(f"deep_segmentation_head.{i}.0", classes, DECODER_CHANNELS[-3], 3, bias=True, init="head")


def materialise(module: nn.Module, spec: ParamSpec) -> None:
    """Register every tensor of ``spec`` on nested plain ``nn.Module`` containers of
    ``module`` so that ``module.state_dict()`` reproduces the keys (aliases share one
    Parameter object, as in the reference)."""
    made: Dict[str, object] = {}
    for key, tensor in spec.tensors.items():
        *path, leaf = key.split(".")
        node = module
        for part in path:
            child = node._modules.get(part)
            if child is None:
                child = nn.Module()
                node.add_module(part, child)
            node = child
        src = spec.alias_of.get(key)
        if src is not None:
            obj = made[src]
        elif spec.is_buffer[key]:
            obj = tensor
        else:
            obj = nn.Parameter(tensor, requires_grad=tensor.is_floating_point())
        made[key] = obj
        if spec.is_buffer[key]:
            node.register_buffer(leaf, obj)
        else:
            node.register_parameter(leaf, obj)
