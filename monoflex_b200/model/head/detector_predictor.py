"""Multi-branch predictor (reference: model/head/detector_predictor.py:19-169), same registry entry, constructor,
parameter names and forward(features, targets) -> {'cls', 'reg'}.

Execution (eval): the 9 shared-input 3x3 convs (class_head.0 + reg_features.i.0, 64->256 each) run as ONE implicit GEMM
with N = 2304 and the InPlaceABN (|gamma|+eps, leaky 0.01) folded into its epilogue; the 1x1 output convs read channel
slices of that buffer and write the fp32 NCHW `cls` / `reg` maps directly; edge fusion = gather kernel + Conv1d-as-GEMM
+ indexed add; sigmoid_hm is one in-place kernel."""
import numpy as np
import torch
from torch import nn

from ... import engine, registry
from ..._lib import call, stream


class InPlaceABN(nn.Module):
    """Parameter container with mapillary/inplace_abn's names (weight, bias, running_mean, running_var); semantics
    y = leaky_relu(BN(x; |weight|+eps, bias), slope) — third-party op, definition unpinned (SURVEY H4)."""

    def __init__(self, num_features, eps=1e-5, momentum=0.1, affine=True, activation="leaky_relu", activation_param=0.01):
        super(InPlaceABN, self).__init__()
        self.num_features, self.eps, self.momentum = num_features, eps, momentum
        self.activation, self.activation_param = activation, activation_param
        self.weight = nn.Parameter(torch.ones(num_features))
        self.bias = nn.Parameter(torch.zeros(num_features))
        self.register_buffer("running_mean", torch.zeros(num_features))
        self.register_buffer("running_var", torch.ones(num_features))


@registry.PREDICTOR.register("Base_Predictor")
class _predictor(nn.Module):
    def __init__(self, cfg, in_channels):
        super(_predictor, self).__init__()
        classes = len(cfg.DATASETS.DETECT_CLASSES)
        self.regression_head_cfg = cfg.MODEL.HEAD.REGRESSION_HEADS
        self.regression_channel_cfg = cfg.MODEL.HEAD.REGRESSION_CHANNELS
        self.output_width = cfg.INPUT.WIDTH_TRAIN // cfg.MODEL.BACKBONE.DOWN_RATIO
        self.output_height = cfg.INPUT.HEIGHT_TRAIN // cfg.MODEL.BACKBONE.DOWN_RATIO
        self.head_conv = hc = cfg.MODEL.HEAD.NUM_CHANNEL
        if not cfg.MODEL.INPLACE_ABN:
            raise NotImplementedError("only the MODEL.INPLACE_ABN=True head of runs/monoflex.yaml:25 is built")
        mom = cfg.MODEL.HEAD.BN_MOMENTUM
        self.class_head = nn.Sequential(nn.Conv2d(in_channels, hc, 3, padding=1, bias=False),
                                        InPlaceABN(hc, momentum=mom), nn.Conv2d(hc, classes, 1, bias=True))
        self.class_head[-1].bias.data.fill_(-np.log(1 / cfg.MODEL.HEAD.INIT_P - 1))
        self.reg_features, self.reg_heads = nn.ModuleList(), nn.ModuleList()
        for idx, keys in enumerate(self.regression_head_cfg):
            self.reg_features.append(nn.Sequential(nn.Conv2d(in_channels, hc, 3, padding=1, bias=False),
                                                   InPlaceABN(hc, momentum=mom)))
            heads = nn.ModuleList()
            for key_index, key in enumerate(keys):
                head = nn.Conv2d(hc, self.regression_channel_cfg[idx][key_index], 1, bias=True)
                if key.find('uncertainty') >= 0 and cfg.MODEL.HEAD.UNCERTAINTY_INIT:
                    nn.init.xavier_normal_(head.weight, gain=0.01)
                if key == '3d_offset':
                    self.offset_index = [idx, key_index]
                nn.init.constant_(head.bias, 0)
                heads.append(head)
            self.reg_heads.append(heads)
        self.enable_edge_fusion = cfg.MODEL.HEAD.ENABLE_EDGE_FUSION
        k = cfg.MODEL.HEAD.EDGE_FUSION_KERNEL_SIZE
        if self.enable_edge_fusion:
            if cfg.MODEL.HEAD.EDGE_FUSION_NORM != 'BN' or cfg.MODEL.HEAD.EDGE_FUSION_RELU or k != 3:
                raise NotImplementedError("edge fusion is built for the runs/monoflex.yaml setting (BN, no ReLU, k=3)")

            def trunc(cout):
                return nn.Sequential(nn.Conv1d(hc, hc, k, padding=k // 2, padding_mode='replicate'),
                                     nn.BatchNorm1d(hc, momentum=mom), nn.Identity(), nn.Conv1d(hc, cout, 1))
            self.trunc_heatmap_conv = trunc(classes)
            self.trunc_offset_conv = trunc(2)
        self.num_classes = classes
        self.num_reg = sum(sum(c) for c in self.regression_channel_cfg)
        self._plans = {}

    # ------------------------------------------------------------------ plan
    def build_plan(self, feat, K_edge):
        """feat: engine.Act-like description of the [B,H,W,64] fp16 feature rows."""
        dev = feat.buf.device
        strict = bool(getattr(feat, "split", False))
        P = engine.Plan(dev, train=self.training, strict=strict)
        B, H, W, hc = feat.B, feat.H, feat.W, self.head_conv
        x = P.act(B, H, W, feat.C)
        x.buf, x.ch_off, x.owner = feat.buf, feat.ch_off, None
        P.acts.remove(x)                                  # externally owned storage
        branches = [self.class_head] + list(self.reg_features)
        w_all = torch.cat([b[0].weight.detach() for b in branches], 0)          # [2304, 64, 3, 3]

        class _ABN(object):
            pass
        abn = _ABN()
        abn.weight = torch.cat([b[1].weight.detach() for b in branches])
        abn.bias = torch.cat([b[1].bias.detach() for b in branches])
        abn.running_mean = torch.cat([b[1].running_mean for b in branches])
        abn.running_var = torch.cat([b[1].running_var for b in branches])
        abn.eps = branches[0][1].eps
        cls = torch.empty(B, self.num_classes, H, W, dtype=torch.float32, device=dev)
        reg = torch.empty(B, self.num_reg, H, W, dtype=torch.float32, device=dev)
        ch0s, ch = [], 0                                    # first `reg` channel of every regression branch
        for heads in self.reg_heads:
            ch0s.append(ch)
            ch += sum(h.weight.shape[0] for h in heads)
        off_ch0 = 0
        if self.enable_edge_fusion:
            off_ch0 = ch0s[self.offset_index[0]] + sum(h.weight.shape[0] for h in
                                                       list(self.reg_heads[self.offset_index[0]])[:self.offset_index[1]])
        # strict precision runs the generic split GEMMs: the nine 3x3 convs as one N = 2304 layer whose hi/lo hidden map goes
        # through HBM once (2.3 GB at B = 8), then the 1x1 heads on its channel slices
        fused = not P.train and not strict and hc == 256 and feat.C % 64 == 0 and \
            all(sum(h.weight.shape[0] for h in heads) <= 32 for heads in self.reg_heads) and self.num_classes <= 32
        head2 = not P.train and strict and hc == 256 and feat.C % 64 == 0 and \
            (H * W) % 4 == 0 and len(branches) <= 12 and self.num_classes <= 32 and \
            all(sum(h.weight.shape[0] for h in heads) <= 32 for heads in self.reg_heads)
        if head2:
            # ---- strict precision: the N = 2304 pair GEMM contracts the 1x1 heads in its epilogue from the fp32 accumulators
            # (csrc/mf_igemm2.cu EPI == 2); the 2.3 GB hidden map never reaches HBM, only its border pixels for the edge fusion
            import ctypes
            nb = len(branches)
            w3, n_pad, k_pad = P.pack_weight(w_all, split=True)
            scale, shift = P.affine(nb * hc, n_pad, abn, None, abs_weight=True)
            ntot = self.num_classes + self.num_reg
            head_w = torch.zeros(nb, 32, hc, dtype=torch.float32, device=dev)
            head_bias = torch.zeros(ntot, dtype=torch.float32, device=dev)
            out_nch, out_ch0, hid_col = [], [], []
            head_lists = [[self.class_head[2]]] + [list(h) for h in self.reg_heads]
            for i, heads in enumerate(head_lists):
                wcat = torch.cat([h.weight.detach().float().reshape(h.weight.shape[0], hc) for h in heads], 0)
                c0 = 0 if i == 0 else self.num_classes + ch0s[i - 1]
                head_w[i, :wcat.shape[0]] = wcat
                head_bias[c0:c0 + wcat.shape[0]] = torch.cat([h.bias.detach().float() for h in heads])
                out_nch.append(wcat.shape[0]); out_ch0.append(c0); hid_col.append(-1)
            part = torch.empty(8, B, ntot, H * W, dtype=torch.float32, device=dev)
            P.edge_idx = torch.zeros(B, K_edge, 2, dtype=torch.long, device=dev)
            hid_buf = hid_mask = None
            if self.enable_edge_fusion:
                hid_col[0], hid_col[self.offset_index[0] + 1] = 0, hc
                hid_buf = torch.zeros(B * H * W, 4 * hc, dtype=torch.half, device=dev)     # [cls hi | off hi | cls lo | off lo]
                hid_mask = torch.zeros(B * H * W, dtype=torch.uint8, device=dev)
                ow_, oh_ = self.output_width, self.output_height
                P.add("mf_edge_mask", lambda: (P.edge_idx.data_ptr(), hid_mask.data_ptr(), B, K_edge, H, W, ow_, oh_))
            arr_nc, arr_c0, arr_hc = (ctypes.c_int * nb)(*out_nch), (ctypes.c_int * nb)(*out_ch0), (ctypes.c_int * nb)(*hid_col)
            P.keep.extend([head_w, head_bias, part, hid_buf, hid_mask, arr_nc, arr_c0, arr_hc, cls, reg])
            cin = feat.C
            P.add("mf_head_conv_f16x2", lambda: (
                x.ptr(), x.ld, x.lo, B, H, W, cin, w3.data_ptr(), n_pad, k_pad, nb, scale.data_ptr(), shift.data_ptr(),
                engine.ACT_LEAKY, head_w.data_ptr(), part.data_ptr(), ntot, ctypes.cast(arr_nc, ctypes.c_void_p),
                ctypes.cast(arr_c0, ctypes.c_void_p), ctypes.cast(arr_hc, ctypes.c_void_p),
                hid_buf.data_ptr() if hid_buf is not None else None, 4 * hc, 2 * hc,
                hid_mask.data_ptr() if hid_mask is not None else None))
            ncls_, nreg_, hw_ = self.num_classes, self.num_reg, H * W
            P.add("mf_head2_reduce", lambda: (part.data_ptr(), head_bias.data_ptr(), cls.data_ptr(), reg.data_ptr(), B, ncls_,
                                              nreg_, hw_))

            class _Hid(object):
                pass
            hid = _Hid()
            hid.ptr = lambda: hid_buf.data_ptr()
            hid.ld, hid.lo = 4 * hc, 2 * hc
            edge_cols = (0, hc)
        elif fused:
            # ---- one kernel: 9 x (3x3 conv + IABN) + every 1x1 head; hidden activations stay on chip (csrc/mf_head.cu)
            nb = len(branches)
            w3, n_pad, k_pad = P.pack_weight(w_all)
            scale, shift = P.affine(nb * hc, n_pad, abn, None, abs_weight=True)
            head_w = torch.zeros(nb * 32, hc, dtype=torch.float32, device=dev)
            head_bias = torch.zeros(nb * 32, dtype=torch.float32, device=dev)
            out_ptrs, out_ctot, out_nch, hid_col = [], [], [], []
            head_lists = [[self.class_head[2]]] + [list(h) for h in self.reg_heads]
            for i, heads in enumerate(head_lists):
                wcat = torch.cat([h.weight.detach().float().reshape(h.weight.shape[0], hc) for h in heads], 0)
                bcat = torch.cat([h.bias.detach().float() for h in heads])
                head_w[i * 32:i * 32 + wcat.shape[0]] = wcat
                head_bias[i * 32:i * 32 + bcat.shape[0]] = bcat
                out_nch.append(wcat.shape[0])
                if i == 0:
                    out_ptrs.append(cls.data_ptr()); out_ctot.append(self.num_classes)
                else:
                    out_ptrs.append(reg.data_ptr() + 4 * ch0s[i - 1] * H * W); out_ctot.append(self.num_reg)
                hid_col.append(-1)
            hid_ld = 2 * hc
            hid_buf = torch.zeros(B * H * W, hid_ld, dtype=torch.half, device=dev)
            if self.enable_edge_fusion:
                hid_col[0] = 0                               # edge fusion reads the cls branch ...
                hid_col[self.offset_index[0] + 1] = hc       # ... and the 3d_offset branch
            w2h = head_w.half().contiguous()
            import ctypes
            arr_p = (ctypes.c_void_p * nb)(*out_ptrs)
            arr_ct, arr_nc, arr_hc = (ctypes.c_int * nb)(*out_ctot), (ctypes.c_int * nb)(*out_nch), (ctypes.c_int * nb)(*hid_col)
            P.edge_idx = torch.zeros(B, K_edge, 2, dtype=torch.long, device=dev)
            hid_mask = None
            if self.enable_edge_fusion:
                # only the border pixels the edge fusion gathers need their hidden activations in HBM
                hid_mask = torch.zeros(B * H * W, dtype=torch.uint8, device=dev)
                ow_, oh_ = self.output_width, self.output_height
                P.add("mf_edge_mask", lambda: (P.edge_idx.data_ptr(), hid_mask.data_ptr(), B, K_edge, H, W, ow_, oh_))
            P.keep.extend([w2h, head_bias, hid_buf, hid_mask, arr_p, arr_ct, arr_nc, arr_hc, cls, reg])
            cin = feat.C
            mask_ptr = hid_mask.data_ptr() if hid_mask is not None else None
            P.add("mf_head_fused", lambda: (
                x.ptr(), x.ld, B, H, W, cin, w3.data_ptr(), w2h.data_ptr(), scale.data_ptr(), shift.data_ptr(), head_bias.data_ptr(),
                nb, ctypes.cast(arr_p, ctypes.c_void_p), ctypes.cast(arr_ct, ctypes.c_void_p),
                ctypes.cast(arr_nc, ctypes.c_void_p), ctypes.cast(arr_hc, ctypes.c_void_p), hid_buf.data_ptr(), hid_ld,
                mask_ptr))

            class _Hid(object):
                pass
            hid = _Hid()
            hid.ptr = lambda: hid_buf.data_ptr()
            hid.ld = hid_ld
            edge_cols = (0, hc)
        else:
            # train mode: every branch normalises with its own InPlaceABN module (batch statistics, running-stat update)
            norm = [(b[1], i * hc, hc) for i, b in enumerate(branches)] if P.train else abn
            # train mode: the nine branch weights are re-packed from their live parameters on every run (static plan)
            w_head = [b[0].weight for b in branches] if P.train else w_all
            hid = P.conv(x, w_head, 1, 1, norm, act=engine.ACT_LEAKY, abs_weight=True)   # [B,H,W,2304]

            def slice_of(i):
                sl = P.act(B, H, W, hc)
                sl.owner, sl.ch_off = hid, i * hc
                return sl
            P.conv_to_f32(slice_of(0), self.class_head[2].weight, self.class_head[2].bias, cls, engine.OUT_F32_NCHW,
                          engine.ACT_NONE, self.num_classes)
            ch = 0
            for i, heads in enumerate(self.reg_heads):
                src = slice_of(i + 1)
                for head in heads:
                    P.conv_to_f32(src, head.weight, head.bias, reg[:, ch:], engine.OUT_F32_NCHW, engine.ACT_NONE,
                                  self.num_reg)
                    ch += head.weight.shape[0]
            edge_cols = (0, (self.offset_index[0] + 1) * hc)
        if not hasattr(P, "edge_idx"):
            P.edge_idx = torch.zeros(B, K_edge, 2, dtype=torch.long, device=dev)
        P.edge_len = torch.zeros(B, dtype=torch.long, device=dev)
        if self.enable_edge_fusion:
            ea = P.act(B, 1, K_edge + 2, hc)
            eb = P.act(B, 1, K_edge + 2, hc)
            ow, oh = self.output_width, self.output_height
            if strict:
                P.add("mf_edge_gather_split", lambda: (hid.ptr(), hid.ld, hid.lo, edge_cols[0], edge_cols[1],
                                                        P.edge_idx.data_ptr(), ea.ptr(), eb.ptr(), B, H, W, K_edge, ow, oh))
            else:
                P.add("mf_edge_gather", lambda: (hid.ptr(), hid.ld, edge_cols[0], edge_cols[1], P.edge_idx.data_ptr(), ea.ptr(),
                                                  eb.ptr(), B, H, W, K_edge, ow, oh))
            for src, seq, dst, ch0, ctot in ((ea, self.trunc_heatmap_conv, cls, 0, self.num_classes),
                                             (eb, self.trunc_offset_conv, reg, off_ch0, self.num_reg)):
                t = P.conv(src, seq[0].weight, 1, 0, seq[1], bias=seq[0].bias, act=engine.ACT_NONE)   # [B,1,K,256]
                w2 = seq[3].weight.detach().float().reshape(seq[3].weight.shape[0], hc).contiguous()
                b2 = seq[3].bias.detach().float().contiguous()
                P.keep.extend([w2, b2])
                n_out = w2.shape[0]
                if strict:
                    P.add("mf_edge_head_add_split", lambda t=t, w2=w2, b2=b2, n_out=n_out, dst=dst, ch0=ch0, ctot=ctot: (
                        t.ptr(), t.ld, t.lo, w2.data_ptr(), b2.data_ptr(), n_out, P.edge_idx.data_ptr(), P.edge_len.data_ptr(),
                        dst.data_ptr(), ctot, ch0, B, K_edge, H, W))
                else:
                    P.add("mf_edge_head_add", lambda t=t, w2=w2, b2=b2, n_out=n_out, dst=dst, ch0=ch0, ctot=ctot: (
                        t.ptr(), w2.data_ptr(), b2.data_ptr(), n_out, P.edge_idx.data_ptr(), P.edge_len.data_ptr(),
                        dst.data_ptr(), ctot, ch0, B, K_edge, H, W))
        n_cls = cls.numel()
        P.add("mf_sigmoid_clamp", lambda: (cls.data_ptr(), n_cls))
        P.finalize()
        P.cls, P.reg, P.hidden = cls, reg, hid
        if P.train:       # what head_backward.predictor_backward needs: activations kept by the train-mode forward
            P.ctx = dict(x=x, hid=hid, ea=ea if self.enable_edge_fusion else None, eb=eb if self.enable_edge_fusion else None,
                         bn={id(m): (raw, y, st, c0, cc) for (m, raw, y, st, c0, cc) in P.bn_saved}, K_edge=K_edge,
                         off_ch0=off_ch0, ch0s=ch0s)
        return P

    def plan_for(self, features, K_edge):
        feat = _as_rows(features)
        key = (feat.buf.data_ptr(), feat.ch_off, feat.B, feat.H, feat.W, feat.buf.shape[1], K_edge,
               engine.fingerprint(self, versions=not self.training), bool(getattr(feat, "split", False)))
        plan = self._plans.get('plan')
        if plan is None or self._plans.get('key') != key:
            plan = self.build_plan(feat, K_edge)
            self._plans = {'plan': plan, 'key': key}
        self.last_plan = plan
        return plan

    @staticmethod
    def load_targets(plan, targets):
        """edge_indices [B,K,2] / edge_len [B] of the batch into the plan's static device buffers (:138-139)."""
        plan.edge_idx.copy_(torch.stack([t.get_field("edge_indices") for t in targets]), non_blocking=True)
        plan.edge_len.copy_(torch.stack([t.get_field("edge_len") for t in targets]).view(-1), non_blocking=True)

    def forward(self, features, targets):
        return self._run(features, targets)      # training mode: train-mode value, see train_forward

    def train_forward(self, features, targets):
        """Train-mode forward (InPlaceABN / BatchNorm1d on batch statistics); keeps the activations
        head_backward.predictor_backward needs (driven by KeypointDetector's tape bridge)."""
        if not self.training:
            raise RuntimeError("train_forward needs module.train()")
        return self._run(features, targets)

    def _run(self, features, targets):
        plan = self.plan_for(features, targets[0].get_field("edge_indices").shape[0])
        if not getattr(self, "_targets_preloaded", False):     # a captured training step loads them before the replay
            self.load_targets(plan, targets)
        plan.run()
        return {'cls': plan.cls, 'reg': plan.reg}


class _Rows(object):
    pass


def _as_rows(features):
    """Accept the backbone's zero-copy channels-last fp16 view, or any [B,C,H,W] CUDA tensor (converted by a kernel)."""
    act = features if isinstance(features, engine.Act) else getattr(features, "_mf_act", None)
    if act is not None:                          # the backbone plan's own output rows (strict precision: hi/lo pairs)
        r = _Rows()
        r.B, r.H, r.W, r.C, r.ch_off, r.buf, r.split = act.B, act.H, act.W, act.C, act.ch_off, act.buf, act.split
        return r
    if not features.is_cuda:
        raise RuntimeError("monoflex_b200 runs on sm_100a GPUs only; no CPU fallback")
    B, C, H, W = features.shape
    r = _Rows()
    r.B, r.H, r.W, r.C, r.ch_off, r.split = B, H, W, C, 0, False
    if features.dtype == torch.half and features.stride(1) == 1 and features.stride(3) % 8 == 0 and \
            features.stride(2) == W * features.stride(3) and features.stride(0) == H * features.stride(2):
        ld = features.stride(3)
        base = features.permute(0, 2, 3, 1)                     # [B,H,W,C] view
        r.ch_off = base.storage_offset() % ld
        rows = torch.as_strided(base, (B * H * W, ld), (ld, 1), storage_offset=base.storage_offset() - r.ch_off)
        r.buf = rows
        return r
    x = features.float().contiguous()
    buf = torch.empty(B * H * W, C, dtype=torch.half, device=x.device)
    call("mf_nchw_f32_to_nhwc_f16", x.data_ptr(), buf.data_ptr(), B, C, H * W, C, stream())
    r.buf = buf
    return r


def make_predictor(cfg, in_channels):
    return registry.PREDICTOR[cfg.MODEL.HEAD.PREDICTOR](cfg, in_channels)
