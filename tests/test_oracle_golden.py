"""CPU: pin the oracle (oracle/monoflex_oracle.py) against the golden vectors recorded from the UNMODIFIED reference
(oracle/make_golden.py). fp32-vs-fp32 on possibly different CPUs: 2e-4 relative; integer outputs bit-exact."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err
from monoflex_b200 import synthetic as syn
from oracle import monoflex_oracle as mo


def load(name):
    with np.load(os.path.join(GOLDEN, name)) as z:
        return {k: torch.from_numpy(z[k]) for k in z.files}


def test_dcn_op_matches_reference_c_loops():
    g = load("dcn_op.npz")
    y = mo.dcn_v2_forward(g['x'], g['weight'], g['bias'], g['offset'], g['mask'])
    assert rel_err(y, g['y']) < 1e-5


def test_dcn_zero_offset_known_answer():
    """testcuda.py:32-67 check_zero_offset: zero offsets, mask 0.5, identity weight => 2*out == input."""
    x = torch.randn(2, 2, 4, 4)
    w = torch.zeros(2, 2, 3, 3)
    w[0, 0, 1, 1] = w[1, 1, 1, 1] = 1.0
    y = mo.dcn_v2_forward(x, w, torch.zeros(2), torch.zeros(2, 18, 4, 4), torch.full((2, 9, 4, 4), 0.5))
    assert (x - 2 * y).abs().max() < 1e-10


@pytest.fixture(scope="module")
def detector_run():
    sd = syn.make_state_dict(0)
    x = syn.make_images(1, 128, 256)
    tg = syn.make_targets(1, 64, 32)
    taps = {}
    with torch.no_grad():
        out = {}
        for thr in (0.0, 0.2):
            res, _ = mo.detector_eval(sd, x, tg['edge_indices'], tg['edge_len'], tg['calib_P'], tg['pad_size'], tg['size'],
                                      thr, taps)
            out[thr] = res[0]
    return taps, out


def test_backbone_and_heads_match_reference(detector_run):
    taps, _ = detector_run
    g = load("detector_128x256.npz")
    for k in ("level2", "level5", "features", "cls", "reg"):
        assert rel_err(taps[k], g[k]) < 2e-4, k


def test_results_match_reference(detector_run):
    _, out = detector_run
    g = load("detector_128x256.npz")
    for thr in (0.0, 0.2):
        ref = g['result_thr%s' % thr]
        assert out[thr].shape == ref.shape
        if ref.numel():
            assert torch.equal(out[thr][:, 0], ref[:, 0])             # class ids
            assert (out[thr] - ref).abs().max() < 2e-3 * max(1.0, ref.abs().max().item())


def test_decode_bit_exact_indices():
    g = load("decode_24x80.npz")
    cl, rgm = syn.make_head_logits(2, 80, 24)
    tg = syn.make_targets(2, 80, 24)
    heat = torch.sigmoid(cl).clamp(1e-4, 1 - 1e-4)
    for thr in (0.0, 0.2):
        res, topk = mo.post_process({'cls': heat, 'reg': rgm}, tg['calib_P'], tg['pad_size'], tg['size'], thr)
        assert torch.equal(topk[1], g['inds'])                         # int64 flat indices, bit exact
        assert torch.equal(topk[2], g['clses']) and torch.equal(topk[3], g['ys']) and torch.equal(topk[4], g['xs'])
        assert torch.equal(topk[0], g['scores'])
        for b in range(2):
            ref = g['result_b%d_thr%s' % (b, thr)]
            assert res[b].shape == ref.shape
            assert (res[b] - ref).abs().max() <= 1e-4 * max(1.0, ref.abs().max().item())


def test_focal_loss():
    g = load("focal.npz")
    gen = np.random.Generator(np.random.PCG64(12))
    pred = torch.from_numpy(gen.uniform(1e-4, 1 - 1e-4, (2, 3, 24, 80)).astype(np.float32))
    tgt = torch.from_numpy((gen.uniform(0, 1, (2, 3, 24, 80)) ** 8).astype(np.float32))
    tgt.view(-1)[::97] = 1.0
    loss, npos = mo.focal_loss(pred, tgt)
    assert abs(loss.item() - g['loss'].item()) < 1e-4 * abs(g['loss'].item())
    assert npos.item() == g['num_pos'].item()


def test_topk_tie_rule():
    """Documented tie rule: (score desc, flat index asc) — torch.topk leaves it unspecified (SURVEY H5)."""
    heat = torch.full((1, 3, 8, 8), 1e-4)
    sc, inds, cls, ys, xs = mo.select_topk(mo.nms_hm(heat), 5)
    assert inds.tolist() == [[0, 1, 2, 3, 4]] and cls.tolist() == [[0.0] * 5]


def test_oracle_ref_library_if_present():
    """The torch restatement of the DCNv2 sampling columns agrees bit-for-bit-ish with the columns the reference's own C
    loops (modulated_deformable_im2col_cpu, oracle/make_golden.py) produced for the same inputs."""
    g = load("dcn_op.npz")
    cols = load("dcn_cols.npz")['cols']
    x, off, mask = g['x'].contiguous(), g['offset'].contiguous(), g['mask'].contiguous()
    B, C, H, W = x.shape
    ours = mo.dcn_columns(x, off, mask).reshape(B, C * 9, H * W)
    for b in range(B):
        assert (ours[b] - cols[b]).abs().max() < 1e-6


def test_loss_oracle_matches_reference_loss_computation():
    """oracle.loss_computation vs the UNMODIFIED reference Loss_Computation (oracle/make_golden_loss.py): the 11 loss
    terms, the logged metrics and the autograd gradient of the summed loss w.r.t. both head outputs."""
    import torch
    from monoflex_b200 import synthetic as syn
    gold = np.load(os.path.join(GOLDEN, "loss_4x96x320.npz"))
    fields = syn.make_train_targets(4)
    cls, reg = syn.make_train_predictions(4, fields)
    cls.requires_grad_(True)
    reg.requires_grad_(True)
    loss, log = mo.loss_computation(cls, reg, fields, [syn.KITTI_P2] * 4)
    assert set(loss) == set(mo.LOSS_NAMES)
    for k, v in loss.items():
        assert abs(v.item() - gold["loss_" + k]) <= 2e-6 * max(1.0, abs(gold["loss_" + k])), k
    for k, v in log.items():
        assert abs(v.item() - gold["log_" + k]) <= 2e-6 * max(1.0, abs(gold["log_" + k])), k
    total = sum(loss.values())
    total.backward()
    centers = np.stack([f["target_centers"] for f in fields])
    mask = np.stack([f["reg_mask"] for f in fields]).astype(bool)
    g = reg.grad.numpy()
    rows = np.stack([g[b, :, centers[b, i, 1], centers[b, i, 0]] for b in range(4) for i in range(mask.shape[1]) if mask[b, i]])
    ref = gold["grad_reg_at_centers"]
    assert np.abs(rows - ref).max() <= 1e-5 * np.abs(ref).max()
    assert abs(np.abs(g).sum() - gold["grad_reg_abs_sum"]) <= 1e-5 * gold["grad_reg_abs_sum"]
    gc = cls.grad.numpy().reshape(-1)
    assert np.abs(gc[::97] - gold["grad_cls_sample"]).max() <= 1e-5 * np.abs(gold["grad_cls_sample"]).max()


def test_train_step_oracle_matches_reference_train_mode():
    """oracle.detector_train_losses (train-mode BN / IABN, predictor with edge fusion, 11-term loss) + autograd vs the UNMODIFIED
    reference model in train() mode (oracle/make_golden_train.py): losses, every parameter's gradient norm, three gradients in
    full. This pins the oracle for the training rows (R2-R6, R11-R12 backward)."""
    import torch
    from monoflex_b200 import synthetic as syn
    gold = np.load(os.path.join(GOLDEN, "train_step_2x384x1280.npz"))
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v)
          for k, v in syn.make_state_dict(seed=0).items()}
    fields = syn.make_train_targets(2, empty_image=0)
    images = syn.make_images(2, 384, 1280, seed=1)
    idx, n, _ = syn.edge_indices()
    loss, _ = mo.detector_train_losses(sd, images, fields, idx.unsqueeze(0).repeat(2, 1, 1), torch.tensor([n, n]),
                                       [syn.KITTI_P2] * 2)
    for k, v in loss.items():
        assert abs(v.item() - gold["loss_" + k]) <= 2e-4 * max(1.0, abs(gold["loss_" + k])), (k, v.item(), gold["loss_" + k])
    sum(loss.values()).backward()
    names, norms = list(gold["grad_names"]), gold["grad_norms"]
    checked = 0
    for k, ref in zip(names, norms):
        g = sd[k].grad
        got = 0.0 if g is None else float(g.double().norm())
        assert abs(got - ref) <= 2e-3 * ref + 2e-5, (k, got, ref)      # conv biases in front of a train-mode BN have ~0 (noise) gradients
        checked += ref > 0
    assert checked >= 260
    for k in ("backbone.base.base_layer.0.weight", "backbone.base.level2.tree1.bn1.weight", "heads.predictor.class_head.2.bias"):
        ref = gold["grad_" + k]
        assert np.abs(sd[k].grad.numpy() - ref).max() <= 2e-3 * np.abs(ref).max(), k


def test_input_pipeline_oracle_vs_reference_golden():
    """N4: pad_image + ToTensor + Normalize and the heat-map drawing restated in oracle/input_oracle.py reproduce the unmodified
    reference functions (oracle/make_golden_input.py) bit for bit."""
    from oracle import input_oracle as io
    from monoflex_b200.data import gaussian_radius
    with np.load(os.path.join(GOLDEN, "input_pipeline.npz")) as z:
        g = {k: z[k] for k in z.files}
    imgs, obj = io.synthetic_case(seed=0)
    assert np.array_equal(obj, g["obj"])
    for b, im in enumerate(imgs):
        padded, pad = io.pad_image(im, 384, 1280)
        t = io.to_tensor_normalize(padded, [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]).numpy()
        assert np.array_equal(pad, g["pads"][b])
        assert np.array_equal(t[:, ::7, ::11], g["image_samples"][b])
        assert t.astype(np.float64).sum() == g["image_sums"][b]
    assert np.array_equal(io.draw_heatmaps(obj, 3, 96, 320), g["hm"])
    got = np.array([gaussian_radius(h, w) for h, w in ((10.0, 20.0), (3.5, 7.25), (40.0, 12.0), (1.0, 1.0), (96.0, 300.0))])
    assert np.array_equal(got, g["radii"])
