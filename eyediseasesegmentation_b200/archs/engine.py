"""Execution of the hot-path networks on the libeds_b200 kernels.

``Engine`` takes a reference-layout ``state_dict``, folds every eval-mode BatchNorm into
its convolution, repacks weights for the kernels (``[Cout][R][S][Cin]``, bf16 for the
tensor-core path, head-major attention projections) and evaluates the graph by calling the
C ABI kernel by kernel.  No PyTorch operator touches an activation.

Graphs restated (reference file:line under src/main/archs):
  proposed UNet++*   unetplusplusstar.py:341-352 (encoder), :239-263 (dense decoder),
                     :127-161 (decoder block), axial_attention_v2.py:261-281 (MHSA block)
  baseline UNet++    deep_supunetplusplus.py:116-139, :48-56  (+ smp encoders, 3P)
  smp.Unet           3P (5 decoder blocks)
  encoders (3P)      resnet34 (BasicBlock), resnet50 / resnext50_32x4d (torchvision Bottleneck, stride on the 3x3
                     conv2), se_resnet50 (SEResNetBottleneck, stride on conv1), se_resnext50_32x4d
                     (SEResNeXtBottleneck, stride on conv2); the 32-group 3x3 convolutions run on the grouped kernels
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch

from .. import _lib, kernels as K
from .spec import dense_decoder_blocks

IDENTITY_VIEW = [(1, 0, 0, 0, 1, 0)]
#: on the tensor-core path, SE bottleneck maps of at least this many pixels get the block's tail (scale, residual,
#: ReLU) in conv3's epilogue; smaller ones run conv3 and se_scale_add_relu as separate passes
SE_EPILOGUE_MIN_PIXELS = 256 * 256
BN_EPS = 1e-5


def _bn_affine(sd, p):
    scale = sd[p + ".weight"].float() / torch.sqrt(sd[p + ".running_var"].float() + BN_EPS)
    shift = sd[p + ".bias"].float() - sd[p + ".running_mean"].float() * scale
    return scale, shift


class Gated:
    """A map whose SCSE gate is still pending: value = t * (cgate[n,c] + sgate[n,p])."""
    __slots__ = ("t", "cgate", "sgate")

    def __init__(self, t, cgate, sgate):
        self.t, self.cgate, self.sgate = t, cgate, sgate

    @property
    def shape(self):
        return self.t.shape


def _parts(x):
    return (x.t, x.cgate, x.sgate) if isinstance(x, Gated) else (x, None, None)


def _plain(x):
    """Materialise a pending gate (new tensor; other consumers still hold the ungated map)."""
    return K.apply_gate(x.t, x.cgate, x.sgate) if isinstance(x, Gated) else x


class Engine:
    def __init__(self, arch: str, cfg: dict, sd: Dict[str, torch.Tensor], device: torch.device, precision: str = "bf16"):
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' (tensor cores) or 'fp32' (parity mode)")
        self.arch = arch
        self.cfg = cfg
        self.device = device
        self.act_dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self.conv_impl = "tc" if precision == "bf16" else "simt"
        self.w: Dict[str, object] = {}
        self.groups: Dict[str, int] = {}        # grouped convolutions (ResNeXt conv2) -> groups
        self.features: Optional[Dict[str, torch.Tensor]] = None  # filled when keep_features is set
        self.keep_features = False
        # BatchNorm folding and repacking run on the HOST (IEEE fp32, same results as on the device): weight
        # preparation then costs uploads, not ~800 small elementwise launches per model
        sd = {k: v.detach().cpu() for k, v in sd.items()}
        self.up_mode = _lib.UP_BILINEAR if arch == "unetplusplusstar" else _lib.UP_NEAREST
        self.senet = "encoder.layer0.conv1.weight" in sd
        self._prepare(sd)
        self.w = {k: tuple(t.to(device) if torch.is_tensor(t) else t for t in v) for k, v in self.w.items()}
        if self.act_dtype == torch.bfloat16:      # tensor-core stem: operand packed once
            self.w["stem.packed"] = K.stem_pack_weights(self.w["stem"][0])

    # ------------------------------------------------------------ weight prep
    def _conv(self, sd, name, conv_key, bn_key=None, perm=None, groups=1):
        w = sd[conv_key + ".weight"].float()
        if w.dim() == 3:
            w = w.unsqueeze(-1)
        b = sd.get(conv_key + ".bias")
        b = None if b is None else b.float()
        if bn_key is not None:
            scale, shift = _bn_affine(sd, bn_key)
            w = w * scale.view(-1, 1, 1, 1)
            b = shift if b is None else b * scale + shift
        if perm is not None:
            w = w[perm]
            b = None if b is None else b[perm]
        w = w.permute(0, 2, 3, 1).contiguous()
        if groups > 1:
            self.groups[name] = groups
            if self.conv_impl == "tc":          # block-diagonal 64-channel operand, packed in fp32 before the cast
                w = K.pack_grouped_weights(w)
        self.w[name] = (w.to(self.act_dtype), None if b is None else b.contiguous())

    def _se(self, sd, name, fc1, fc2):
        w1, w2 = sd[fc1 + ".weight"].float(), sd[fc2 + ".weight"].float()
        self.w[name] = (w1.reshape(w1.shape[0], w1.shape[1]).contiguous(), sd[fc1 + ".bias"].float().contiguous(),
                        w2.reshape(w2.shape[0], w2.shape[1]).contiguous(), sd[fc2 + ".bias"].float().contiguous())

    def _scse(self, sd, name, p):
        if (p + ".attention.sSE.0.weight") not in sd:
            return
        self._se(sd, name + ".cse", p + ".attention.cSE.1", p + ".attention.cSE.3")
        self.w[name + ".sse"] = (sd[p + ".attention.sSE.0.weight"].float().reshape(-1).contiguous(),
                                 float(sd[p + ".attention.sSE.0.bias"].float().item()))

    def _attention(self, sd, name, p, heads, d_kq, d_v):
        sim_scale, _ = _bn_affine(sd, p + ".attention_norm")       # shift cancels in the softmax
        osc, osh = _bn_affine(sd, p + ".out_norm")
        self.w[name] = (sd[p + ".RelativePosEncQKV.relative"].float().contiguous(),
                        sim_scale.reshape(heads, 3).contiguous(),
                        osc.reshape(2, heads * d_v).contiguous(), osh.reshape(2, heads * d_v).contiguous())

    @staticmethod
    def _head_major(groups: int, heads: int, device):
        """'(q h)' channel order of the reference projections -> '(h q)' expected by the kernel."""
        return (torch.arange(groups, device=device).view(1, groups) * heads +
                torch.arange(heads, device=device).view(heads, 1)).reshape(-1)

    def _prepare(self, sd):
        dev = torch.device("cpu")
        # stem: [64,3,7,7] -> [7][7][3][64] fp32
        stem_conv, stem_bn = ("encoder.layer0.conv1", "encoder.layer0.bn1") if self.senet else ("encoder.conv1", "encoder.bn1")
        scale, shift = _bn_affine(sd, stem_bn)
        w = sd[stem_conv + ".weight"].float() * scale.view(-1, 1, 1, 1)
        self.w["stem"] = (w.permute(2, 3, 1, 0).contiguous(), shift.contiguous())

        if self.senet:
            n_layers = 3 if self.arch == "unetplusplusstar" else 4
            for li in range(1, n_layers + 1):
                b = 0
                while f"encoder.layer{li}.{b}.conv1.weight" in sd:
                    p = f"encoder.layer{li}.{b}"
                    self._conv(sd, p + ".conv1", p + ".conv1", p + ".bn1")
                    self._conv(sd, p + ".conv2", p + ".conv2", p + ".bn2", groups=self._conv2_groups(sd, p))
                    self._conv(sd, p + ".conv3", p + ".conv3", p + ".bn3")
                    # fp32 copy of the (rounded) conv3 weights as a [Cout][Cin] matrix: the SE squeeze from the
                    # channel means of conv3's input (K.affine_rows)
                    w3 = self.w[p + ".conv3"][0]
                    self.w[p + ".conv3.f32"] = (w3.float().reshape(w3.shape[0], -1).contiguous(),)
                    if (p + ".downsample.0.weight") in sd:
                        self._conv(sd, p + ".downsample", p + ".downsample.0", p + ".downsample.1")
                    self._se(sd, p + ".se", p + ".se_module.fc1", p + ".se_module.fc2")
                    b += 1
        else:
            for li in range(1, 5):
                b = 0
                while f"encoder.layer{li}.{b}.conv1.weight" in sd:
                    p = f"encoder.layer{li}.{b}"
                    self._conv(sd, p + ".conv1", p + ".conv1", p + ".bn1")
                    self._conv(sd, p + ".conv2", p + ".conv2", p + ".bn2", groups=self._conv2_groups(sd, p))
                    if (p + ".conv3.weight") in sd:      # torchvision Bottleneck (resnet50, resnext50_32x4d)
                        self._conv(sd, p + ".conv3", p + ".conv3", p + ".bn3")
                    if (p + ".downsample.0.weight") in sd:
                        self._conv(sd, p + ".downsample", p + ".downsample.0", p + ".downsample.1")
                    b += 1

        if self.arch == "unetplusplusstar":
            for bi in (0, 1):  # layer4.2 aliases layer4.1
                p = f"encoder.layer4.{bi}"
                self._conv(sd, p + ".in", p + ".in_conv1x1.0", p + ".in_conv1x1.1")
                self._conv(sd, p + ".out", p + ".out_conv1x1.0", p + ".out_conv1x1.1")
                for ax in ("height_att", "width_att"):
                    q = f"{p}.{ax}"
                    self._conv(sd, q + ".qkv", q + ".to_qvk.0", q + ".to_qvk.1", perm=self._head_major(80, 8, dev))
                    self._attention(sd, q, q, 8, 8, 64)
                if (p + ".shortcut.0.weight") in sd:
                    self._conv(sd, p + ".shortcut", p + ".shortcut.0", p + ".shortcut.1")
                    sc, sh = _bn_affine(sd, p + ".att_down.1")
                    self.w[p + ".att_down"] = (sc.contiguous(), sh.contiguous())
            enc_ch = (3, 64, 256, 512, 1024, 2048)
            self.blocks = dense_decoder_blocks(enc_ch)
            bn_idx = 2
        else:
            enc_ch = self._encoder_channels(sd)
            if self.arch == "unetplusplus_deepsup":
                self.blocks = dense_decoder_blocks(enc_ch)
            else:
                enc = list(enc_ch[1:])[::-1]
                ins = [enc[0], 256, 128, 64, 32]
                skips = list(enc[1:]) + [0]
                self.blocks = [(str(i), 0, ins[i], skips[i], (256, 128, 64, 32, 16)[i]) for i in range(5)]
            bn_idx = 1

        for name, layer_idx, in_ch, skip_ch, out_ch in self.blocks:
            p = f"decoder.blocks.{name}"
            for cv in ("conv1", "conv2"):
                bn_key = f"{p}.{cv}.{bn_idx}"
                self._conv(sd, f"{p}.{cv}", f"{p}.{cv}.0", bn_key if (bn_key + ".weight") in sd else None)
            if (p + ".down_sample.weight") in sd:  # MHCA block
                cr = skip_ch // 16
                self._conv(sd, p + ".down_sample", p + ".down_sample")
                self._conv(sd, p + ".up_sample", p + ".up_sample")
                self._conv(sd, p + ".init_conv", p + ".init_conv.1", p + ".init_conv.2")
                for ax in ("h_catt", "w_catt"):
                    q = f"{p}.{ax}"
                    self._conv(sd, q + ".kq", q + ".to_kq.0", q + ".to_kq.1", perm=self._head_major(16, 4, dev))
                    self._conv(sd, q + ".v", q + ".to_v.0", q + ".to_v.1", perm=self._head_major(cr // 4, 4, dev))
                    self._attention(sd, q, q, 4, 8, cr // 4)
            else:
                self._scse(sd, p + ".attention1", p + ".attention1")
                self._scse(sd, p + ".attention2", p + ".attention2")
        hw = sd["segmentation_head.0.weight"].float()
        self.w["head"] = (hw.permute(0, 2, 3, 1).contiguous(), sd["segmentation_head.0.bias"].float().contiguous())

    @staticmethod
    def _conv2_groups(sd, p):
        """Groups of a block's 3x3 conv2 (input channels == output channels there): 32 for the ResNeXt blocks."""
        w = sd[p + ".conv2.weight"]
        return int(w.shape[0] // w.shape[1])

    @staticmethod
    def _encoder_channels(sd):
        """(input, stem, layer1 .. layer4) channels of an smp encoder: the last conv of each stage's blocks."""
        ch = [3, 64]
        for li in range(1, 5):
            p = f"encoder.layer{li}.0"
            ch.append(int(sd[p + (".conv3.weight" if (p + ".conv3.weight") in sd else ".conv2.weight")].shape[0]))
        return tuple(ch)

    # ---------------------------------------------------------------- kernels
    def _cv(self, x, name, stride=1, pad=0, relu=False, residual=None):
        w, b = self.w[name]
        if name in self.groups:
            return K.conv2d(x, w, b, stride, pad, relu, residual, impl=self.conv_impl, groups=self.groups[name])
        if isinstance(x, tuple):        # (upsampled part, skip part) of a decoder concat: two-input K loop
            return K.conv2d(x[0], w, b, stride, pad, relu, residual, impl=self.conv_impl, x1=x[1])
        return K.conv2d(x, w, b, stride, pad, relu, residual, impl=self.conv_impl)

    def _split_ok(self, srcs):
        """The tensor-core convolutions can read the concat as two dense maps when both channel counts are
        multiples of 16 (bf16 path only; the fp32 parity path keeps one map)."""
        return (self.conv_impl == "tc" and len(srcs) >= 2 and srcs[0][0].shape[3] % 16 == 0 and
                sum(t[0].shape[3] for t in srcs[1:]) % 16 == 0)

    def _keep(self, name, t):
        if self.keep_features:
            self.features[name] = t

    # SCSE with deferred gates (csrc/scse_gated.cu): a block output keeps its attention2 gate as two
    # side tensors (Gated) until a concat or the head reads it, and attention1 is applied while the
    # concat is written -- no map is written twice.
    def _apply_scse(self, name, x):
        """attention2: statistics of the block output -> (x, cgate, sgate), nothing rewritten."""
        if (name + ".sse") not in self.w:
            return x
        w_sse, b_sse = self.w[name + ".sse"]
        N, H, W, C = x.shape
        mean = torch.empty((N, C), dtype=torch.float32, device=x.device)
        dot = torch.empty((N, H, W), dtype=torch.float32, device=x.device)
        K.gated_stats(x, None, None, w_sse, mean, 0, True, dot, False)
        cgate = K.se_gate(mean, *self.w[name + ".cse"])
        return Gated(x, cgate, K.sse_finalize(None, dot, _lib.UP_NONE, b_sse))

    def _concat_scse(self, name, x, skips, skip_names=None):
        """attention1(cat([up2x(x), *skips])): one statistics pass per source at its own resolution,
        then one pass that writes the gated concat.  A skip source that feeds several blocks of the dense
        decoder is read ONCE for all of them (``_skip_stats``)."""
        w_sse, b_sse = self.w[name + ".sse"]
        srcs = [_parts(x)] + [_parts(s) for s in skips]
        x0 = srcs[0][0]
        N, h, w, _ = x0.shape
        ctot = sum(t[0].shape[3] for t in srcs)
        mean, dot1 = self._consumer_buffers(name, N, ctot, 2 * h, 2 * w, x0.device)
        dot0 = torch.empty((N, h, w), dtype=torch.float32, device=x0.device)
        K.gated_stats(x0, srcs[0][1], srcs[0][2], w_sse[:x0.shape[3]], mean, 0, False, dot0, False)
        off = x0.shape[3]
        for k, (t, cg, sg) in enumerate(srcs[1:]):
            c = t.shape[3]
            key = skip_names[k] if skip_names else None
            if key is None or key not in self._skip_plan:       # a source with this block as its only consumer
                K.gated_stats(t, cg, sg, w_sse[off:off + c], mean, off, False, dot1, True)
            elif key not in self._skip_done:
                self._skip_done.add(key)
                cons = []
                for (cname, coff, cctot) in self._skip_plan[key]:
                    cm, cd = self._consumer_buffers(cname, N, cctot, 2 * h, 2 * w, x0.device)
                    cons.append((self.w[cname + ".sse"][0][coff:coff + c], cm, coff, cd))
                K.gated_stats_multi(t, cg, sg, cons)
            off += c
        cgate = K.se_gate(mean, *self.w[name + ".cse"])
        sgate = K.sse_finalize(dot0, dot1, self.up_mode, b_sse)
        if self._split_ok(srcs):
            return K.concat_gated_split(srcs, self.up_mode, cgate, sgate)
        return K.concat_gated(srcs, self.up_mode, cgate, sgate)

    def _consumer_buffers(self, name, N, ctot, H, W, device):
        """Zero-initialised (channel means [N,ctot], skip dot map [N,H,W]) of one attention1, created the first time
        any of its sources is read."""
        buf = self._stat_bufs.get(name)
        if buf is None:
            buf = (torch.zeros((N, ctot), dtype=torch.float32, device=device),
                   torch.zeros((N, H, W), dtype=torch.float32, device=device))
            self._stat_bufs[name] = buf
        return buf

    def _plan_skip_consumers(self, feats):
        """Static plan of the dense decoder: skip source name -> [(attention1 name, channel offset in that
        block's concat, channels of that concat)] over the SCSE blocks that read it at its own resolution."""
        rev = feats[::-1]
        depth = len(rev) - 1
        ch = {f"f{len(rev) - i}": int(t.shape[3]) for i, t in enumerate(rev)}     # rev[i] = f(5 - i)
        for bname, _layer, _in, _skip, out_ch in self.blocks:
            ch[bname] = int(out_ch)
        plan = {}
        for layer_idx in range(depth):
            for depth_idx in range(depth - layer_idx):
                li = depth_idx + layer_idx
                if layer_idx == 0:
                    bname, xname, snames = f"x_{depth_idx}_{depth_idx}", f"f{len(rev) - depth_idx}", [f"f{len(rev) - depth_idx - 1}"]
                else:
                    bname, xname = f"x_{depth_idx}_{li}", f"x_{depth_idx}_{li - 1}"
                    snames = [f"x_{i}_{li}" for i in range(depth_idx + 1, li + 1)] + [f"f{len(rev) - li - 1}"]
                p = f"decoder.blocks.{bname}.attention1"
                if (p + ".sse") not in self.w:
                    continue
                ctot = ch[xname] + sum(ch[sname] for sname in snames)
                off = ch[xname]
                for sname in snames:
                    plan.setdefault(sname, []).append((p, off, ctot))
                    off += ch[sname]
        return {k: v for k, v in plan.items() if len(v) > 1 and len(v) <= 4}

    # ---------------------------------------------------------------- encoders
    def _se_bottleneck(self, p, x, stride):
        # SEResNetBottleneck strides its 1x1 conv1, SEResNeXtBottleneck (grouped conv2) its 3x3 conv2
        s1, s2 = (1, stride) if (p + ".conv2") in self.groups else (stride, 1)
        out = self._cv(x, p + ".conv1", stride=s1, relu=True)
        out = self._cv(out, p + ".conv2", stride=s2, pad=1, relu=True)
        res = self._cv(x, p + ".downsample", stride=stride) if (p + ".downsample") in self.w else x
        if self.conv_impl == "tc":
            # conv3 (1x1 + folded BN) has no activation, so the channel means its SE module squeezes are an affine
            # function of the channel means of conv3's INPUT (a quarter of the channels): the gate is known before
            # conv3 runs and the squeeze never re-reads the 4x wider map.  On the large maps scale + residual + ReLU
            # then happen on conv3's accumulators (the pre-activation map is never written); on the small ones the
            # epilogue's residual path costs more than the separate pass it replaces (scripts/dev_se_probe.py: 48
            # maps, fused vs conv3 + scale: 1.39 vs 1.44 ms at 256^2, 0.76 vs 0.73 at 128^2, 0.42 vs 0.38 at 64^2)
            w3, b3 = self.w[p + ".conv3"]
            squeeze = K.affine_rows(K.channel_mean(out), self.w[p + ".conv3.f32"][0], b3)
            gate = K.se_gate(squeeze, *self.w[p + ".se"])
            if out.shape[1] * out.shape[2] >= SE_EPILOGUE_MIN_PIXELS:
                return K.conv1x1_se(out, w3, b3, gate, res)
            out = self._cv(out, p + ".conv3")
            return K.se_scale_add_relu(out, gate, res, out=out)
        out = self._cv(out, p + ".conv3")
        gate = K.se_gate(K.channel_mean(out), *self.w[p + ".se"])
        return K.se_scale_add_relu(out, gate, res, out=out)

    def _senet_layer(self, li, x, stride):
        b = 0
        while f"encoder.layer{li}.{b}.conv1" in self.w:
            x = self._se_bottleneck(f"encoder.layer{li}.{b}", x, stride if b == 0 else 1)
            b += 1
        return x

    def _resnet_layer(self, li, x, stride):
        b = 0
        while f"encoder.layer{li}.{b}.conv1" in self.w:
            p = f"encoder.layer{li}.{b}"
            s = stride if b == 0 else 1
            if (p + ".conv3") in self.w:        # torchvision Bottleneck: 1x1, 3x3 (stride, groups), 1x1 + identity
                out = self._cv(x, p + ".conv1", relu=True)
                out = self._cv(out, p + ".conv2", stride=s, pad=1, relu=True)
                idt = self._cv(x, p + ".downsample", stride=s) if (p + ".downsample") in self.w else x
                x = self._cv(out, p + ".conv3", relu=True, residual=idt)
            else:                               # BasicBlock
                out = self._cv(x, p + ".conv1", stride=s, pad=1, relu=True)
                idt = self._cv(x, p + ".downsample", stride=s) if (p + ".downsample") in self.w else x
                x = self._cv(out, p + ".conv2", pad=1, relu=True, residual=idt)
            b += 1
        return x

    def _axial_block(self, p, x_in):
        x = self._cv(x_in, p + ".in", relu=True)
        down = (p + ".shortcut") in self.w
        qkv = self._cv(x, p + ".height_att.qkv")
        x = K.axial_attention(qkv, None, 0, 8, 8, 64, *self.w[p + ".height_att"], relu=False)
        qkv = self._cv(x, p + ".width_att.qkv")
        x = K.axial_attention(qkv, None, 1, 8, 8, 64, *self.w[p + ".width_att"], relu=not down)
        if down:
            x_in = self._cv(x_in, p + ".shortcut", stride=2, pad=1)
            x = K.avgpool2_affine(x, *self.w[p + ".att_down"], relu=True)
        return self._cv(x, p + ".out", relu=True, residual=x_in)

    def _encode(self, x, aug_maps):
        if "stem.packed" in self.w:
            f1 = K.stem_conv_mma(x, aug_maps, self.w["stem.packed"], self.w["stem"][1])
        else:
            f1 = K.stem_conv(x, aug_maps, *self.w["stem"], dtype=self.act_dtype)
        if self.senet:
            y = K.maxpool2d(f1, 3, 2, 0, True)
            f2 = self._senet_layer(1, y, 1)
            f3 = self._senet_layer(2, f2, 2)
            f4 = self._senet_layer(3, f3, 2)
            if self.arch == "unetplusplusstar":
                y = self._axial_block("encoder.layer4.0", f4)
                y = self._axial_block("encoder.layer4.1", y)
                f5 = self._axial_block("encoder.layer4.1", y)  # layer4.2 is the same module object
            else:
                f5 = self._senet_layer(4, f4, 2)
        else:
            y = K.maxpool2d(f1, 3, 2, 1, False)
            f2 = self._resnet_layer(1, y, 1)
            f3 = self._resnet_layer(2, f2, 2)
            f4 = self._resnet_layer(3, f3, 2)
            f5 = self._resnet_layer(4, f4, 2)
        feats = [f1, f2, f3, f4, f5]
        for i, f in enumerate(feats, start=1):
            self._keep(f"f{i}", f)
        return feats

    # ---------------------------------------------------------------- decoders
    def _mhca_skip(self, p, x, skips: Sequence[torch.Tensor]):
        skips = [_plain(t) for t in skips]
        skip = skips[0] if len(skips) == 1 else K.upsample2x_concat(skips[0], list(skips[1:]), _lib.UP_NONE)
        cr = skip.shape[3] // 16
        ori = self._cv(skip, p + ".down_sample")
        s = K.maxpool2d(skip, 2, 2, 0, False)
        s = self._cv(s, p + ".init_conv", relu=True)
        for axis, ax in ((0, "h_catt"), (1, "w_catt")):
            kq = self._cv(x, f"{p}.{ax}.kq")
            v = self._cv(s, f"{p}.{ax}.v")
            s = K.axial_attention(kq, v, axis, 4, 8, cr // 4, *self.w[f"{p}.{ax}"], relu=False)
        return self._cv(K.mhca_gate(ori, s), p + ".up_sample")

    def _decoder_block(self, name, x, skips: Sequence[torch.Tensor], skip_names=None):
        p = f"decoder.blocks.{name}"
        if (p + ".down_sample") in self.w:
            x = _plain(x)
            skip = self._mhca_skip(p, x, skips)
            if self._split_ok([(x, None, None), (skip, None, None)]):
                # the gated skip is already a dense map: only the upsampled half is written
                cat = (K.concat_gated([(x, None, None)], self.up_mode), skip)
            else:
                cat = K.concat_gated([(x, None, None), (skip, None, None)], self.up_mode)
        else:
            if skips and (p + ".attention1.sse") in self.w:
                cat = self._concat_scse(p + ".attention1", x, skips, skip_names)
            else:
                srcs = [_parts(x)] + [_parts(t) for t in skips]
                cat = K.concat_gated_split(srcs, self.up_mode) if self._split_ok(srcs) else \
                    K.concat_gated(srcs, self.up_mode)
        y = self._cv(cat, p + ".conv1", pad=1, relu=True)
        y = self._cv(y, p + ".conv2", pad=1, relu=True)
        if (p + ".down_sample") not in self.w:
            y = self._apply_scse(p + ".attention2", y)
        if self.keep_features:
            self.features[name] = _plain(y)
        return y

    def _decode_dense(self, feats: List[torch.Tensor]):
        rev = feats[::-1]                  # f5, f4, f3, f2, f1
        depth = len(rev) - 1
        nf = len(rev)
        self._skip_plan = self._plan_skip_consumers(feats)
        dense = {}
        for layer_idx in range(depth):
            for depth_idx in range(depth - layer_idx):
                if layer_idx == 0:
                    name = f"x_{depth_idx}_{depth_idx}"
                    dense[name] = self._decoder_block(name, rev[depth_idx], [rev[depth_idx + 1]],
                                                      [f"f{nf - depth_idx - 1}"])
                else:
                    li = depth_idx + layer_idx
                    names = [f"x_{i}_{li}" for i in range(depth_idx + 1, li + 1)]
                    skips = [dense[n] for n in names] + [rev[li + 1]]
                    name = f"x_{depth_idx}_{li}"
                    dense[name] = self._decoder_block(name, dense[f"x_{depth_idx}_{li - 1}"], skips,
                                                      names + [f"f{nf - li - 1}"])
        return self._decoder_block(f"x_0_{depth}", dense[f"x_0_{depth - 1}"], [])

    def _decode_unet(self, feats: List[torch.Tensor]):
        rev = feats[::-1]
        y = rev[0]
        for i in range(5):
            y = self._decoder_block(str(i), y, [rev[i + 1]] if i + 1 < len(rev) else [])
        return y

    # ------------------------------------------------------------------- run
    def run(self, x: torch.Tensor, aug_maps=None) -> torch.Tensor:
        """x [B,3,H,W] fp32 cuda -> logits [V*B, classes, H, W] fp32 (view-major)."""
        if not x.is_cuda:
            raise RuntimeError("the B200 networks only run on a CUDA device (no CPU fallback); got a CPU tensor")
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected [B,3,H,W] input, got {tuple(x.shape)}")
        H, W = x.shape[2:]
        if H % 32 or W % 32:
            raise ValueError(f"input size {H}x{W} must be divisible by 32")
        if self.arch == "unetplusplusstar":
            bd = int(self.cfg.get("base_dim", 32))
            if H != 32 * bd or W != 32 * bd:
                raise ValueError(f"base_dim={bd} fixes the input size to {32 * bd}x{32 * bd}, got {H}x{W} "
                                 "(unetplusplusstar.py:85,296-309)")
        x = x.contiguous().float()
        if self.keep_features:
            self.features = {}
        self._stat_bufs, self._skip_done, self._skip_plan = {}, set(), {}
        feats = self._encode(x, aug_maps or IDENTITY_VIEW)
        y = self._decode_unet(feats) if self.arch == "Unet" else self._decode_dense(feats)
        return K.head_conv3x3(_plain(y), *self.w["head"])
