"""Test-side restatements of the ResNet-50 family encoders of smp 0.1.3 (resnet50, resnext50_32x4d,
se_resnext50_32x4d), next to the oracle package they extend.

  torchvision ``models.resnet.Bottleneck`` / ``ResNet`` with ``groups`` / ``width_per_group`` (smp's ResNetEncoder
        drops ``fc`` and ``avgpool``): stride on the 3x3 conv2, width = floor(planes * width_per_group / 64) * groups
  pretrainedmodels 0.7.4 ``senet.SEResNeXtBottleneck`` (smp's SENetEncoder over ``se_resnext50_32x4d``): the same
        width, stride on conv2, SE module on conv3's output, 1x1 downsample with padding 0

They are unpinned third-party restatements, written from the published architectures like oracle/shims.py: the
packages cannot be installed offline, so apart from the published parameter totals (tests/test_encoders.py) their
parity with the real packages is not checked.  ``nn.Module`` shims give the key layouts; the functional forwards
(``forward``) are the fp32 references the CUDA path is held to.
"""
from __future__ import annotations

from typing import List

import torch
import torch.nn.functional as F
from torch import nn

from oracle import nets, shims

DECODER_CHANNELS = (256, 128, 64, 32, 16)
NEW_ENCODERS = ("resnet50", "resnext50_32x4d", "se_resnext50_32x4d")
_LAYERS = ((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2))


# ------------------------------------------------------------------ nn.Module shims
class Bottleneck(nn.Module):
    """torchvision Bottleneck (expansion 4)."""
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None, groups=1, base_width=64):
        super().__init__()
        width = int(planes * (base_width / 64.0)) * groups
        self.conv1 = nn.Conv2d(inplanes, width, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(width)
        self.conv2 = nn.Conv2d(width, width, 3, stride=stride, padding=1, groups=groups, bias=False)
        self.bn2 = nn.BatchNorm2d(width)
        self.conv3 = nn.Conv2d(width, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        identity = x if self.downsample is None else self.downsample(x)
        out = self.relu(self.bn1(self.conv1(x)))
        out = self.relu(self.bn2(self.conv2(out)))
        out = self.bn3(self.conv3(out))
        return self.relu(out + identity)


class ResNetEncoder(nn.Module):
    """smp ResNetEncoder over torchvision ResNet(Bottleneck, [3, 4, 6, 3], groups, width_per_group)."""

    def __init__(self, groups=1, width_per_group=64, depth=5):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 64, 7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, stride=2, padding=1)
        self.inplanes = 64
        for li, (planes, blocks, stride) in enumerate(_LAYERS, start=1):
            downsample = nn.Sequential(nn.Conv2d(self.inplanes, planes * 4, 1, stride=stride, bias=False),
                                       nn.BatchNorm2d(planes * 4))
            layers = [Bottleneck(self.inplanes, planes, stride, downsample, groups, width_per_group)]
            self.inplanes = planes * 4
            layers += [Bottleneck(self.inplanes, planes, groups=groups, base_width=width_per_group)
                       for _ in range(1, blocks)]
            setattr(self, f"layer{li}", nn.Sequential(*layers))
        self.out_channels = (3, 64, 256, 512, 1024, 2048)
        self._depth = depth

    def forward(self, x):
        stages = [nn.Identity(), nn.Sequential(self.conv1, self.bn1, self.relu),
                  nn.Sequential(self.maxpool, self.layer1), self.layer2, self.layer3, self.layer4]
        feats = []
        for i in range(self._depth + 1):
            x = stages[i](x)
            feats.append(x)
        return feats


class SEResNeXtBottleneck(nn.Module):
    """pretrainedmodels SEResNeXtBottleneck (expansion 4, base_width 4)."""
    expansion = 4

    def __init__(self, inplanes, planes, groups, reduction, stride=1, downsample=None, base_width=4):
        super().__init__()
        width = (planes * base_width // 64) * groups
        self.conv1 = nn.Conv2d(inplanes, width, kernel_size=1, bias=False, stride=1)
        self.bn1 = nn.BatchNorm2d(width)
        self.conv2 = nn.Conv2d(width, width, kernel_size=3, stride=stride, padding=1, groups=groups, bias=False)
        self.bn2 = nn.BatchNorm2d(width)
        self.conv3 = nn.Conv2d(width, planes * 4, kernel_size=1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.relu = nn.ReLU(inplace=True)
        self.se_module = shims.SEModule(planes * 4, reduction=reduction)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        residual = x if self.downsample is None else self.downsample(x)
        out = self.relu(self.bn1(self.conv1(x)))
        out = self.relu(self.bn2(self.conv2(out)))
        out = self.bn3(self.conv3(out))
        return self.relu(self.se_module(out) + residual)


class SEResNeXtEncoder(shims._SENetEncoder):
    """smp SENetEncoder over se_resnext50_32x4d: SENet(SEResNeXtBottleneck, [3, 4, 6, 3], groups=32,
    reduction=16, inplanes=64, downsample_kernel_size=1, downsample_padding=0)."""

    def __init__(self, depth=5):
        shims.SENet.__init__(self, SEResNeXtBottleneck, [3, 4, 6, 3], groups=32, reduction=16)
        self.out_channels = (3, 64, 256, 512, 1024, 2048)
        self._depth = depth
        del self.last_linear
        del self.avg_pool


def get_encoder(name, in_channels=3, depth=5, weights=None):
    """oracle.shims.get_encoder with the three ResNet-50 family names added."""
    if name == "resnet50":
        return ResNetEncoder(1, 64, depth)
    if name == "resnext50_32x4d":
        return ResNetEncoder(32, 4, depth)
    if name == "se_resnext50_32x4d":
        return SEResNeXtEncoder(depth)
    return shims.get_encoder(name, in_channels, depth, weights)


class Unet(shims.SegmentationModel):
    """smp.Unet (oracle.shims.Unet) built on get_encoder above."""

    def __init__(self, encoder_name="resnet50", decoder_attention_type=None, classes=1):
        super().__init__()
        self.encoder = get_encoder(encoder_name)
        self.decoder = shims._UnetDecoder(self.encoder.out_channels, DECODER_CHANNELS, True, decoder_attention_type)
        self.segmentation_head = shims.SegmentationHead(DECODER_CHANNELS[-1], classes, kernel_size=3)
        self.classification_head = None
        self.initialize()


# ------------------------------------------------------------------ functional fp32 forwards
def _conv(sd, p, x, stride=1, padding=0):
    w = sd[p + ".weight"]
    return F.conv2d(x, w, sd.get(p + ".bias"), stride=stride, padding=padding, groups=x.shape[1] // w.shape[1])


def bottleneck(sd, p, x, stride):
    """torchvision Bottleneck or SEResNeXtBottleneck (SE module when its keys exist): stride and groups on conv2."""
    out = F.relu(nets.bn(sd, p + ".bn1", _conv(sd, p + ".conv1", x)))
    out = F.relu(nets.bn(sd, p + ".bn2", _conv(sd, p + ".conv2", out, stride=stride, padding=1)))
    out = nets.bn(sd, p + ".bn3", _conv(sd, p + ".conv3", out))
    residual = x
    if (p + ".downsample.0.weight") in sd:
        residual = nets.bn(sd, p + ".downsample.1", _conv(sd, p + ".downsample.0", x, stride=stride))
    if (p + ".se_module.fc1.weight") in sd:
        z = F.adaptive_avg_pool2d(out, 1)
        z = torch.sigmoid(nets.conv(sd, p + ".se_module.fc2", F.relu(nets.conv(sd, p + ".se_module.fc1", z))))
        out = out * z
    return F.relu(out + residual)


def encoder(sd, x) -> List[torch.Tensor]:
    """Features [x, f1 .. f5] of the resnet50 / resnext50_32x4d / se_resnext50_32x4d encoders (by key layout)."""
    if "encoder.layer0.conv1.weight" in sd:
        f1 = nets.senet_stem(sd, "encoder.layer0", x)
        y = F.max_pool2d(f1, 3, stride=2, ceil_mode=True)
    else:
        f1 = F.relu(nets.bn(sd, "encoder.bn1", nets.conv(sd, "encoder.conv1", x, stride=2, padding=3)))
        y = F.max_pool2d(f1, 3, stride=2, padding=1)
    feats = [x, f1]
    for li, (_, blocks, stride) in enumerate(_LAYERS, start=1):
        for b in range(blocks):
            y = bottleneck(sd, f"encoder.layer{li}.{b}", y, stride if b == 0 else 1)
        feats.append(y)
    return feats


def unet_forward(sd, x, return_features=False):
    feats = encoder(sd, x)
    rev = feats[1:][::-1]
    y = rev[0]
    for i in range(5):
        y = nets.smp_decoder_block(sd, f"decoder.blocks.{i}", y, rev[i + 1] if i + 1 < len(rev) else None)
    mask = nets.conv(sd, "segmentation_head.0", y, padding=1)
    return (mask, feats) if return_features else mask


def unetplusplus_forward(sd, x, return_features=False):
    feats = encoder(sd, x)
    y = nets._dense_decoder(feats, lambda name, level, xx, skip: nets.smp_decoder_block(sd, f"decoder.blocks.{name}",
                                                                                        xx, skip))
    mask = nets.conv(sd, "segmentation_head.0", y, padding=1)
    return (mask, feats) if return_features else mask


def forward(model_name, sd, x, return_features=False):
    sd = {k: v.detach().float() if v.is_floating_point() else v for k, v in sd.items()}
    with torch.no_grad():
        if model_name == "Unet":
            return unet_forward(sd, x, return_features)
        if model_name == "unetplusplus_deepsup":
            return unetplusplus_forward(sd, x, return_features)
    raise KeyError(model_name)
