"""ResNet-50 family encoders (resnet50, resnext50_32x4d, se_resnext50_32x4d) in Unet and UNet++: key layouts
against the restated third-party modules, published parameter totals, the functional oracle against the modules,
and the host-side block-diagonal packing of the grouped 3x3 weights.  CPU only."""
import pytest
import torch
import torch.nn.functional as F

from eyediseasesegmentation_b200 import archs, kernels as K
from eyediseasesegmentation_b200.archs import spec

import encoder_oracle as eo
from helpers import build_product_model, randomize_bn

CFG_ATT = [None, "scse"]


def _cfg(enc, att):
    cfg = dict(encoder_name=enc, encoder_weights=None, classes=1)
    if att:
        cfg["decoder_attention_type"] = att
    return cfg


def _layout(sd):
    return {k: tuple(v.shape) for k, v in sd.items()}


@pytest.mark.parametrize("att", CFG_ATT)
@pytest.mark.parametrize("enc", eo.NEW_ENCODERS)
def test_unet_state_dict_matches_shim(enc, att):
    product = build_product_model("Unet", _cfg(enc, att))
    torch.manual_seed(0)
    shim = eo.Unet(enc, decoder_attention_type=att).eval()
    assert _layout(product.state_dict()) == _layout(shim.state_dict())
    shim.load_state_dict(product.state_dict(), strict=True)
    product.load_state_dict(shim.state_dict(), strict=True)
    assert all(torch.equal(v, shim.state_dict()[k]) for k, v in product.state_dict().items())


@pytest.mark.parametrize("att", CFG_ATT)
@pytest.mark.parametrize("enc", eo.NEW_ENCODERS)
def test_unetplusplus_state_dict_matches_shim(enc, att):
    """UNet++: the encoder keys are the shim encoder's under 'encoder.', the decoder and heads are exactly those of
    the se_resnet50 model (same encoder channels), and a checkpoint round-trips strictly."""
    cfg = dict(_cfg(enc, att), deep_supervision=True)
    product = build_product_model("unetplusplus_deepsup", cfg).state_dict()
    encoder = {"encoder." + k: v for k, v in eo.get_encoder(enc).state_dict().items()}
    assert _layout({k: v for k, v in product.items() if k.startswith("encoder.")}) == _layout(encoder)
    se50 = build_product_model("unetplusplus_deepsup", dict(cfg, encoder_name="se_resnet50")).state_dict()
    assert _layout({k: v for k, v in product.items() if not k.startswith("encoder.")}) == \
        _layout({k: v for k, v in se50.items() if not k.startswith("encoder.")})
    other = build_product_model("unetplusplus_deepsup", cfg, seed=5)
    other.load_state_dict(product, strict=True)
    assert all(torch.equal(v, product[k]) for k, v in other.state_dict().items())


@pytest.mark.parametrize("enc,total", [("resnet50", 23_508_032), ("resnext50_32x4d", 22_979_904),
                                       ("se_resnext50_32x4d", 25_510_896), ("se_resnet50", 26_039_024)])
def test_encoder_parameter_counts(enc, total):
    """Published ImageNet classifier totals minus the 2048 x 1000 + 1000 classifier."""
    assert sum(p.numel() for p in eo.get_encoder(enc).parameters()) == total
    s = spec.ParamSpec(torch.Generator().manual_seed(0))
    spec.SMP_ENCODERS[enc](s, "encoder")
    assert sum(t.numel() for k, t in s.tensors.items() if not s.is_buffer[k]) == total


@pytest.mark.parametrize("enc", eo.NEW_ENCODERS)
def test_functional_oracle_matches_modules(enc):
    """encoder_oracle.forward (the fp32 reference of the GPU tests) against the shim nn.Module forward."""
    torch.manual_seed(3)
    shim = randomize_bn(eo.Unet(enc, decoder_attention_type="scse"), 4).eval()
    x = torch.randn(1, 3, 64, 64, generator=torch.Generator().manual_seed(7))
    with torch.no_grad():
        want, want_feats = shim(x), shim.encoder(x)
    got, feats = eo.forward("Unet", shim.state_dict(), x, return_features=True)
    for a, b in zip(feats + [got], want_feats + [want]):
        assert (a - b).abs().max().item() <= 1e-5 * max(1.0, b.abs().max().item())


@pytest.mark.parametrize("cpg", [4, 8, 16, 32])
def test_grouped_packing_equals_grouped_conv(cpg):
    """Block-diagonal packing: each 64-channel cout block of the packed filter, convolved densely with its
    64-channel input chunk, equals F.conv2d(groups) on that block."""
    C = 128
    groups = C // cpg
    g = torch.Generator().manual_seed(cpg)
    w = torch.randn(C, cpg, 3, 3, generator=g)
    x = torch.randn(2, C, 9, 11, generator=g)
    want = F.conv2d(x, w, padding=1, groups=groups)
    packed = K.pack_grouped_weights(w.permute(0, 2, 3, 1).contiguous())          # [Cout,3,3,64]
    assert packed.shape == (C, 3, 3, 64)
    dense = packed.permute(0, 3, 1, 2)                                          # [Cout,64,3,3]
    got = torch.cat([F.conv2d(x[:, n * 64:(n + 1) * 64], dense[n * 64:(n + 1) * 64], padding=1)
                     for n in range(C // 64)], dim=1)
    assert (got - want).abs().max().item() <= 1e-6 * want.abs().max().item() * 9 * cpg    # fp32 sums of 9 cpg terms
    assert (packed != 0).sum().item() == w.numel()                              # nothing outside the groups


def test_unsupported_encoder_still_raises_keyerror():
    with pytest.raises(KeyError, match="se_resnext50_32x4d"):
        archs.Unet(encoder_name="efficientnet-b2", encoder_weights=None, classes=1)
    with pytest.raises(KeyError, match="resnet34"):
        archs.get_model("unetplusplus_deepsup", dict(encoder_name="densenet121", encoder_weights=None, classes=1),
                        training=False)
