"""TEST TOOLING — generates tests/golden/*.npz by executing the UNMODIFIED reference (/root/reference, via
oracle/ref_shims.py) on the deterministic synthetic workload. Run in the build container only:

    python -m oracle.make_golden

The fixtures pin oracle/monoflex_oracle.py (tests/test_oracle_golden.py) and, through it, the CUDA path. Inputs are not
stored: they are regenerated from monoflex_b200/synthetic.py seeds, so a fixture also pins the generator.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims as rs            # noqa: E402
from monoflex_b200 import synthetic as syn    # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def ref_targets(tg):
    from structures.params_3d import ParamsList
    from data.datasets.kitti_utils import Calibration
    out = []
    for b in range(len(tg['calib_P'])):
        t = ParamsList(tg['size'][b], is_train=False)
        c = Calibration.__new__(Calibration)
        P = np.array(tg['calib_P'][b])
        c.P = P
        c.c_u, c.c_v, c.f_u, c.f_v = P[0, 2], P[1, 2], P[0, 0], P[1, 1]
        c.b_x, c.b_y = P[0, 3] / (-c.f_u), P[1, 3] / (-c.f_v)
        t.add_field('calib', c)
        t.add_field('pad_size', tg['pad_size'][b])
        t.add_field('edge_indices', tg['edge_indices'][b])
        t.add_field('edge_len', tg['edge_len'][b])
        out.append(t)
    return out


def dcn_columns():
    """The reference's modulated_deformable_im2col_cpu columns of the dcn_op.npz inputs -> dcn_cols.npz, so the sampling
    step of oracle.dcn_columns stays pinned to the reference's C loops without the compiled library."""
    lib = rs._load_ref_so()
    with np.load(os.path.join(OUT, "dcn_op.npz")) as z:
        x, off, mask = (np.ascontiguousarray(z[k]) for k in ("x", "offset", "mask"))
    B, C, H, W = x.shape
    cols = np.empty((B, C * 9, H * W), np.float32)
    for b in range(B):
        lib.modulated_deformable_im2col_cpu(x[b].ctypes.data, off[b].ctypes.data, mask[b].ctypes.data, 1, C, H, W, H, W,
                                            3, 3, 1, 1, 1, 1, 1, 1, 1, cols[b].ctypes.data)
    np.savez_compressed(os.path.join(OUT, "dcn_cols.npz"), cols=cols)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    # ---------------------------------------------------------------- 1. DCNv2 operator (reference C loops via _ext shim)
    rs.install()
    import _ext
    g = np.random.Generator(np.random.PCG64(11))
    B, C, H, W, Co = 2, 8, 6, 7, 5
    x = torch.from_numpy(g.standard_normal((B, C, H, W)).astype(np.float32))
    off = torch.from_numpy((g.standard_normal((B, 18, H, W)) * 1.5).astype(np.float32))
    mask = torch.from_numpy(g.uniform(0, 1, (B, 9, H, W)).astype(np.float32))
    w = torch.from_numpy((g.standard_normal((Co, C, 3, 3)) * 0.2).astype(np.float32))
    bias = torch.from_numpy(g.standard_normal(Co).astype(np.float32))
    y = _ext.dcn_v2_forward(x, w, bias, off, mask, 3, 3, 1, 1, 1, 1, 1, 1, 1)
    np.savez_compressed(os.path.join(OUT, "dcn_op.npz"), x=x.numpy(), offset=off.numpy(), mask=mask.numpy(), weight=w.numpy(),
                        bias=bias.numpy(), y=y.numpy())
    dcn_columns()

    # ---------------------------------------------------------------- 2. whole detector, eval, 1x3x128x256
    Hh, Ww, Bb = 128, 256, 1
    cfg = rs.reference_cfg(width=Ww, height=Hh)
    model = rs.build_reference_model(cfg).eval()
    sd = syn.make_state_dict(0)
    model.load_state_dict(sd)
    images = syn.make_images(Bb, Hh, Ww)
    tg = syn.make_targets(Bb, Ww // 4, Hh // 4)
    targets = ref_targets(tg)
    taps = {}
    with torch.no_grad():
        levels = model.backbone.base(images)
        feats = model.backbone(images)
        pred = model.heads.predictor(feats, targets)
        out = {'features': feats.numpy(), 'cls': pred['cls'].numpy(), 'reg': pred['reg'].numpy()}
        for i in (2, 5):
            out['level%d' % i] = levels[i].numpy()
        for thr in (0.0, 0.2):
            model.heads.post_processor.det_threshold = thr
            res, _, _ = model.heads.post_processor({k: v.clone() for k, v in pred.items()}, targets, test=True)
            out['result_thr%s' % thr] = res.numpy()
    np.savez_compressed(os.path.join(OUT, "detector_128x256.npz"), **out)

    # ---------------------------------------------------------------- 3. decode only (bit-exact integer indices)
    import model.layers.utils as lu
    cl, rgm = syn.make_head_logits(2, 80, 24)
    tg2 = syn.make_targets(2, 80, 24)
    targets2 = ref_targets(tg2)
    cfg2 = rs.reference_cfg(width=320, height=96)
    pp = rs.build_reference_model(cfg2).eval().heads.post_processor
    heat = torch.sigmoid(cl).clamp(1e-4, 1 - 1e-4)
    out = {}
    with torch.no_grad():
        sc, inds, cls_, ys, xs = lu.select_topk(lu.nms_hm(heat), 50)
        out.update(scores=sc.numpy(), inds=inds.numpy(), clses=cls_.numpy(), ys=ys.numpy(), xs=xs.numpy())
        for thr in (0.0, 0.2):
            pp.det_threshold = thr
            for b in range(2):
                res, _, _ = pp({'cls': heat[b:b + 1].clone(), 'reg': rgm[b:b + 1].clone()}, targets2[b:b + 1], test=True)
                out['result_b%d_thr%s' % (b, thr)] = res.numpy()
    np.savez_compressed(os.path.join(OUT, "decode_24x80.npz"), **out)

    # ---------------------------------------------------------------- 4. focal loss
    from model.layers.focal_loss import FocalLoss
    g = np.random.Generator(np.random.PCG64(12))
    pred = torch.from_numpy(g.uniform(1e-4, 1 - 1e-4, (2, 3, 24, 80)).astype(np.float32))
    tgt = torch.from_numpy((g.uniform(0, 1, (2, 3, 24, 80)) ** 8).astype(np.float32))
    tgt.view(-1)[::97] = 1.0
    loss, npos = FocalLoss(2, 4)(pred, tgt)
    np.savez_compressed(os.path.join(OUT, "focal.npz"), loss=np.float32(loss.item()), num_pos=np.float32(npos.item()))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
