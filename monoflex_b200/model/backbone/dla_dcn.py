"""DLA-34 + iterative deep aggregation backbone (reference: model/backbone/dla_dcn.py).

The module tree only *holds parameters* under the reference's names so that `state_dict()` keys, checkpoint loading,
optimizer param groups and DDP see exactly what they see in the reference (SURVEY §8b). Execution is not per-module:
`DLASeg.forward` builds (once per input shape) a static plan of fused sm_100a kernels over NHWC fp16 buffers
(monoflex_b200/engine.py) and replays it:

  conv+BN(+residual)+ReLU      -> one tcgen05 implicit GEMM with affine epilogue      (BasicBlock :84-98, Root :195-203)
  torch.cat for Root           -> producers write channel slices of one buffer         (:197)
  MaxPool2d(2)                 -> vectorised NHWC kernel writing its concat slice      (:238)
  DCN (+BN+ReLU)               -> offset/mask conv + fused gather-contract kernel      (DeformConv :384-396)
  ConvTranspose2d + add        -> one HBM-bound kernel                                 (IDAUp :419-425)
"""
import math

import numpy as np
import torch
from torch import nn

from ... import engine
from ..._lib import call, stream
from .DCNv2.dcn_v2 import DCN

BN_MOMENTUM = 0.1


def build_backbone(cfg):
    return DLASeg(base_name=cfg.MODEL.BACKBONE.CONV_BODY, pretrained=cfg.MODEL.PRETRAIN,
                  down_ratio=cfg.MODEL.BACKBONE.DOWN_RATIO, last_level=5)


def _bn(c):
    return nn.BatchNorm2d(c, momentum=BN_MOMENTUM)


class BasicBlock(nn.Module):
    def __init__(self, inplanes, planes, stride=1, dilation=1):
        super(BasicBlock, self).__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 3, stride=stride, padding=dilation, bias=False, dilation=dilation)
        self.bn1 = _bn(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, stride=1, padding=dilation, bias=False, dilation=dilation)
        self.bn2 = _bn(planes)
        self.stride = stride

    def plan(self, P, x, residual, out=None):
        t = P.conv(x, self.conv1.weight, self.stride, 1, self.bn1)
        return P.conv(t, self.conv2.weight, 1, 1, self.bn2, residual=residual if residual is not None else x, out=out)


class Root(nn.Module):
    def __init__(self, in_channels, out_channels, kernel_size, residual):
        super(Root, self).__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, 1, stride=1, bias=False, padding=(kernel_size - 1) // 2)
        self.bn = _bn(out_channels)
        self.residual = residual

    def plan(self, P, children, out=None):
        cat = P.concat(children)
        return P.conv(cat, self.conv.weight, 1, 0, self.bn, residual=children[0] if self.residual else None, out=out)


class Tree(nn.Module):
    def __init__(self, levels, block, in_channels, out_channels, stride=1, level_root=False, root_dim=0,
                 root_kernel_size=1, dilation=1, root_residual=False):
        super(Tree, self).__init__()
        if root_dim == 0:
            root_dim = 2 * out_channels
        if level_root:
            root_dim += in_channels
        if levels == 1:
            self.tree1 = block(in_channels, out_channels, stride, dilation=dilation)
            self.tree2 = block(out_channels, out_channels, 1, dilation=dilation)
            self.root = Root(root_dim, out_channels, root_kernel_size, root_residual)
        else:
            self.tree1 = Tree(levels - 1, block, in_channels, out_channels, stride, root_dim=0,
                              root_kernel_size=root_kernel_size, dilation=dilation, root_residual=root_residual)
            self.tree2 = Tree(levels - 1, block, out_channels, out_channels, root_dim=root_dim + out_channels,
                              root_kernel_size=root_kernel_size, dilation=dilation, root_residual=root_residual)
        self.level_root, self.root_dim, self.levels, self.stride = level_root, root_dim, levels, stride
        self.in_channels, self.out_channels = in_channels, out_channels
        self.downsample = nn.MaxPool2d(stride, stride=stride) if stride > 1 else None
        self.project = None
        if in_channels != out_channels:
            self.project = nn.Sequential(nn.Conv2d(in_channels, out_channels, 1, stride=1, bias=False), _bn(out_channels))

    def plan(self, P, x, children=None):
        """Tree.forward (dla_dcn.py:246-259). For nested trees the reference overwrites the `residual` it was handed
        (:249), so the outer `project` never reaches the output; those parameters exist but are not executed."""
        children = [] if children is None else children
        bottom = P.maxpool2(x) if self.stride > 1 else x
        if self.level_root:
            children.append(bottom)
        if self.levels == 1:
            if self.project is not None:
                residual = P.conv(bottom, self.project[0].weight, 1, 0, self.project[1], act=engine.ACT_NONE)
            else:
                residual = bottom
            x1 = self.tree1.plan(P, x, residual)
            x2 = self.tree2.plan(P, x1, None)
            return self.root.plan(P, [x2, x1] + children)
        x1 = self.tree1.plan(P, x)
        children.append(x1)
        return self.tree2.plan(P, x1, children)


class DLA(nn.Module):
    def __init__(self, levels, channels, block=BasicBlock, residual_root=False):
        super(DLA, self).__init__()
        self.channels = channels
        self.base_layer = nn.Sequential(nn.Conv2d(3, channels[0], 7, stride=1, padding=3, bias=False), _bn(channels[0]),
                                        nn.ReLU(inplace=True))
        self.level0 = self._conv_level(channels[0], channels[0], levels[0])
        self.level1 = self._conv_level(channels[0], channels[1], levels[1], stride=2)
        self.level2 = Tree(levels[2], block, channels[1], channels[2], 2, level_root=False, root_residual=residual_root)
        self.level3 = Tree(levels[3], block, channels[2], channels[3], 2, level_root=True, root_residual=residual_root)
        self.level4 = Tree(levels[4], block, channels[3], channels[4], 2, level_root=True, root_residual=residual_root)
        self.level5 = Tree(levels[5], block, channels[4], channels[5], 2, level_root=True, root_residual=residual_root)

    @staticmethod
    def _conv_level(inplanes, planes, convs, stride=1):
        mods = []
        for i in range(convs):
            mods += [nn.Conv2d(inplanes, planes, 3, stride=stride if i == 0 else 1, padding=1, bias=False), _bn(planes),
                     nn.ReLU(inplace=True)]
            inplanes = planes
        return nn.Sequential(*mods)

    def plan(self, P, x8):
        """DLA.forward (:324-331). x8: image already packed to NHWC fp16 with 8 channels (3 real + 5 zero)."""
        rows_ok = (len(self.level0) == 3 and len(self.level1) == 3 and self.channels[0] == 16 and x8.W % 2 == 0 and
                   self.level1[0].stride[0] == 2 and not P.train)
        y = []
        if P.strict and rows_ok:
            # strict precision on the row-segment kernel: x8 is the image pair plane [hi3 | lo3 | 0 0] (mf_pack_image_pair8);
            # the split products of 7x7, level0 and the stride-2 level1 run as extra MMAs over the same resident row segments;
            # level0 writes column-parity pair planes for level1, level1 hands NHWC pair rows to level2
            x8.npar = 1
            a0 = P.conv_rows_strict(x8, self.base_layer[0].weight, 1, 3, self.base_layer[1], out_planar=True, image=True)
            a1 = P.conv_rows_strict(a0, self.level0[0].weight, 1, 1, self.level0[1], out_planar=True, out_npar=2)
            x = P.conv_rows_strict(a1, self.level1[0].weight, 2, 1, self.level1[1], out_planar=False)
            y += [a1, x]
        elif P.strict:
            # generic fallback: x8 is the 16-channel pair-packed image [hi3 | lo3 | hi3 | 0 x 7] (mf_pack_image_split), so the
            # 7x7 stem is a plain 16-channel conv whose per-tap weights are [W_hi | W_hi | W_lo | 0]: the three split products
            # A_hi W_hi + A_lo W_hi + A_hi W_lo in one pass. Its output and everything after it are hi/lo pairs.
            w = self.base_layer[0].weight.detach().float()
            w_hi = w.half().float()
            w_lo = (w - w_hi).half().float()
            w16 = torch.zeros(w.shape[0], 16, w.shape[2], w.shape[3], dtype=torch.float32, device=w.device)
            w16[:, 0:3], w16[:, 3:6], w16[:, 6:9] = w_hi, w_hi, w_lo
            x = P.conv(x8, w16, 1, 3, self.base_layer[1])
            for seq in (self.level0, self.level1):
                for i in range(0, len(seq), 3):
                    x = P.conv(x, seq[i].weight, seq[i].stride[0], 1, seq[i + 1])
                y.append(x)
        elif rows_ok:
            # full-resolution stem on 16-byte-pixel planes: no im2col copies (csrc/mf_rows.cu)
            x8.npar = 1
            a0 = P.conv_rows(x8, self.base_layer[0].weight, 1, 3, self.base_layer[1], out_planar=True, out_npar=1)
            a1 = P.conv_rows(a0, self.level0[0].weight, 1, 1, self.level0[1], out_planar=True, out_npar=2)
            x = P.conv_rows(a1, self.level1[0].weight, 2, 1, self.level1[1], out_planar=False)
            y += [a1, x]
        else:
            x = P.conv(x8, self.base_layer[0].weight, 1, 3, self.base_layer[1], cin_pad=8)
            for seq in (self.level0, self.level1):
                for i in range(0, len(seq), 3):
                    x = P.conv(x, seq[i].weight, seq[i].stride[0], 1, seq[i + 1])
                y.append(x)
        for i in range(2, 6):
            x = getattr(self, 'level%d' % i).plan(P, x)
            y.append(x)
        return y


def dla34(pretrained=False, **kwargs):
    if pretrained:
        raise RuntimeError("MODEL.PRETRAIN downloads ImageNet weights (dla_dcn.py:333-344); load a checkpoint instead")
    return DLA([1, 1, 1, 2, 2, 1], [16, 32, 64, 128, 256, 512], block=BasicBlock, **kwargs)


def fill_up_weights(up):
    """bilinear kernel init of the depthwise ConvTranspose2d (dla_dcn.py:372-381)."""
    k = up.weight.shape[2]
    f = math.ceil(k / 2)
    c = (2 * f - 1 - f % 2) / (2.0 * f)
    w1 = torch.tensor([1 - abs(i / f - c) for i in range(k)])
    with torch.no_grad():
        up.weight.copy_(torch.outer(w1, w1).expand_as(up.weight))


class DeformConv(nn.Module):
    def __init__(self, chi, cho):
        super(DeformConv, self).__init__()
        self.actf = nn.Sequential(_bn(cho), nn.ReLU(inplace=True))
        self.conv = DCN(chi, cho, kernel_size=(3, 3), stride=1, padding=1, dilation=1, deformable_groups=1)

    def plan(self, P, x):
        return P.dcn(x, self.conv, self.actf[0])


class IDAUp(nn.Module):
    def __init__(self, o, channels, up_f):
        super(IDAUp, self).__init__()
        self.up_f = [int(f) for f in up_f]
        for i in range(1, len(channels)):
            f = self.up_f[i]
            setattr(self, 'proj_%d' % i, DeformConv(channels[i], o))
            up = nn.ConvTranspose2d(o, o, f * 2, stride=f, padding=f // 2, output_padding=0, groups=o, bias=False)
            fill_up_weights(up)
            setattr(self, 'up_%d' % i, up)
            setattr(self, 'node_%d' % i, DeformConv(o, o))

    def plan(self, P, layers, startp, endp):
        """IDAUp.forward (:419-425)."""
        for i in range(startp + 1, endp):
            j = i - startp
            proj = getattr(self, 'proj_%d' % j).plan(P, layers[i])
            summed = P.upsample_add(proj, getattr(self, 'up_%d' % j).weight, layers[i - 1], self.up_f[j])
            layers[i] = getattr(self, 'node_%d' % j).plan(P, summed)


class DLAUp(nn.Module):
    def __init__(self, startp, channels, scales, in_channels=None):
        super(DLAUp, self).__init__()
        self.startp = startp
        in_channels = list(channels) if in_channels is None else in_channels
        self.channels = channels
        channels = list(channels)
        scales = np.array(scales, dtype=int)
        for i in range(len(channels) - 1):
            j = -i - 2
            setattr(self, 'ida_%d' % i, IDAUp(channels[j], in_channels[j:], scales[j:] // scales[j]))
            scales[j + 1:] = scales[j]
            in_channels[j + 1:] = [channels[j] for _ in channels[j + 1:]]

    def plan(self, P, layers):
        """DLAUp.forward (:446-452)."""
        layers = list(layers)
        out = [layers[-1]]
        for i in range(len(layers) - self.startp - 1):
            getattr(self, 'ida_%d' % i).plan(P, layers, len(layers) - i - 2, len(layers))
            out.insert(0, layers[-1])
        return out


class DLASeg(nn.Module):
    def __init__(self, base_name, pretrained, down_ratio, last_level):
        super(DLASeg, self).__init__()
        assert down_ratio in [2, 4, 8, 16]
        self.first_level = int(np.log2(down_ratio))
        self.last_level = last_level
        self.base = globals()[base_name](pretrained=pretrained)
        channels = self.base.channels
        scales = [2 ** i for i in range(len(channels[self.first_level:]))]
        self.dla_up = DLAUp(self.first_level, channels[self.first_level:], scales)
        self.out_channels = channels[self.first_level]
        self.ida_up = IDAUp(self.out_channels, channels[self.first_level:self.last_level],
                            [2 ** i for i in range(self.last_level - self.first_level)])
        self._plans = {}

    # ---- plan construction / execution
    def build_plan(self, B, H, W, device):
        strict = (not self.training) and self._precision() == "strict"
        P = engine.Plan(device, train=self.training, strict=strict)
        self._strict_rows = strict and W % 2 == 0
        x8 = P.act(B, H, W, 8 if (self._strict_rows or not strict) else 16, split=False)
        P.image_pack = "mf_pack_image_pair8" if self._strict_rows else ("mf_pack_image_split" if strict else "mf_pack_image")
        levels = self.base.plan(P, x8)
        ups = self.dla_up.plan(P, levels)
        y = [ups[i] for i in range(self.last_level - self.first_level)]   # the reference's .clone()s are not needed
        self.ida_up.plan(P, y, 0, len(y))
        P.finalize()
        P.input, P.output, P.levels, P.ups = x8, y[-1], levels, ups
        return P

    def _precision(self):
        """'strict' | 'fast' (engine.default_precision unless KeypointDetector.set_precision / self.precision says otherwise)"""
        return getattr(self, "precision", None) or engine.default_precision()

    def _plan_for(self, x):
        key = (tuple(x.shape), engine.fingerprint(self, versions=not self.training), self._precision())
        plan = self._plans.get('plan')
        if plan is None or self._plans.get('key') != key:
            B, _, H, W = x.shape
            plan = self.build_plan(B, H, W, x.device)
            self._plans = {'plan': plan, 'key': key}
        return plan

    def forward(self, x):
        """x: [B,3,H,W] fp32 NCHW (reference signature). Returns the [B,64,H/4,W/4] feature map: fast mode a zero-copy
        channels-last fp16 view of the plan's output buffer; strict mode an fp32 tensor (hi + lo) that remembers its pair
        rows (`_mf_act`) so that the predictor consumes them without a conversion."""
        if self.training:
            # train-mode VALUE (batch statistics); the result carries no grad_fn - gradients reach the parameters through
            # KeypointDetector's tape bridge (model/detector.py), the training entry point
            return self.train_forward(x)
        if not x.is_cuda:
            raise RuntimeError("monoflex_b200 runs on sm_100a GPUs only (input is on %s); no CPU fallback" % x.device)
        x = x.float().contiguous()
        plan = self._plan_for(x)
        self.run_plan(plan, x)
        return plan.output.nchw_view()

    def train_forward(self, x):
        """Train-mode forward of the backbone (batch-statistics BatchNorm, running statistics updated in place) on the
        CUDA kernels; records the tape `tape.backbone_backward` replays (driven by KeypointDetector's tape bridge)."""
        if not self.training:
            raise RuntimeError("train_forward needs module.train()")
        if not x.is_cuda:
            raise RuntimeError("monoflex_b200 runs on sm_100a GPUs only (input is on %s); no CPU fallback" % x.device)
        x = x.float().contiguous()
        plan = self._plan_for(x)
        self.run_plan(plan, x)
        return plan.output.nchw_view()

    def run_plan(self, plan, x):
        B, C, H, W = x.shape
        call(plan.image_pack, x.data_ptr(), plan.input.ptr(), B, C, H, W, stream())
        plan.run()
        self.last_plan = plan
