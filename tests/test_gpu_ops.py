"""-m gpu: per-kernel parity through the C ABI against torch-CPU fp32 on identical fp16-representable operands.
Tolerances: fp16-output kernels 1e-3 of max|ref| (one fp16 rounding of the result is 4.9e-4); fp32-output kernels 2e-5;
integer outputs bit-exact."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN
from gpu_util import FakeBN, from_rows, h16, rel_err, set_impl, to_rows, to_rows_split
from monoflex_b200 import engine, synthetic as syn
from oracle import monoflex_oracle as mo

pytestmark = pytest.mark.gpu

DCN_CASES_EARLY = [(1, 64, 12, 20, 64), (2, 128, 7, 9, 64), (1, 256, 6, 10, 128), (1, 512, 4, 6, 256), (2, 64, 24, 40, 64), (2, 64, 24, 48, 64), (1, 128, 16, 32, 64)]  # last two: maps that tile exactly into 16 x 8 pixel blocks
CONV_CASES = [
    # B, Cin, H, W, Cout, k, stride, pad, act, residual
    (2, 16, 12, 20, 16, 3, 1, 1, engine.ACT_RELU, False),      # level0-like, N tile 16
    (2, 16, 12, 20, 32, 3, 2, 1, engine.ACT_RELU, False),      # stride 2, 2 taps per K block
    (1, 64, 16, 24, 64, 3, 1, 1, engine.ACT_RELU, True),       # BasicBlock conv2 + residual
    (1, 128, 9, 13, 128, 3, 1, 1, engine.ACT_RELU, False),     # ragged M (117 rows), N tile 128
    (1, 448, 8, 16, 128, 1, 1, 0, engine.ACT_RELU, False),     # Root 1x1 over a 448-ch concat
    (1, 32, 8, 16, 64, 1, 1, 0, engine.ACT_NONE, False),       # project 1x1, no activation, K block half empty
    (1, 64, 10, 12, 256, 3, 1, 1, engine.ACT_LEAKY, False),    # head-like, 2 N tiles, leaky
    (1, 256, 6, 10, 512, 3, 2, 1, engine.ACT_RELU, False),     # deep layer, 4 N tiles, K = 2304
    (3, 64, 7, 11, 64, 3, 1, 1, engine.ACT_RELU, True),        # tiles wrap across rows and images (im2col traversal)
    (2, 64, 17, 23, 128, 3, 2, 1, engine.ACT_RELU, False),     # stride 2 on odd sizes
    (2, 128, 5, 300, 64, 3, 1, 1, engine.ACT_NONE, False),     # wide rows: several 128-pixel tiles per image row
    (2, 32, 12, 20, 64, 3, 2, 1, engine.ACT_RELU, False),      # Cin 32: cp.async gather, 2 taps per K block
    (1, 16, 33, 47, 32, 3, 1, 1, engine.ACT_RELU, True),       # Cin 16: cp.async gather, 4 taps per K block, ragged
    (2, 64, 19, 23, 640, 3, 1, 1, engine.ACT_LEAKY, False),    # head-like: 5 N tiles, 9 K blocks, 7 m-tiles
    (1, 64, 40, 500, 512, 1, 1, 0, engine.ACT_RELU, False),    # a single K block, many m-tiles
    # maps that tile exactly into 16 x 8 pixel blocks
    (2, 64, 16, 32, 64, 3, 1, 1, engine.ACT_RELU, True),       # N tile 64, residual, image borders in every tile
    (1, 128, 24, 48, 128, 3, 1, 1, engine.ACT_RELU, False),    # two 64-channel chunks, N tile 128
    (1, 64, 16, 32, 256, 3, 1, 1, engine.ACT_LEAKY, False),    # two N tiles
    (1, 128, 8, 32, 64, 3, 1, 1, engine.ACT_NONE, True),       # 128 -> 64
    (2, 64, 96, 160, 64, 3, 1, 1, engine.ACT_RELU, True),      # 240 m-tiles: every CTA wraps its stage ring
]


def run_conv(case, impl, seed=0):
    B, Cin, H, W, Cout, k, stride, pad, act, use_res = case
    gen = np.random.Generator(np.random.PCG64(seed))
    x = h16(torch.from_numpy(gen.standard_normal((B, Cin, H, W)).astype(np.float32)))
    w = h16(torch.from_numpy((gen.standard_normal((Cout, Cin, k, k)) / np.sqrt(Cin * k * k)).astype(np.float32)))
    bn = FakeBN(Cout, gen)
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    res = h16(torch.from_numpy(gen.standard_normal((B, Cout, Ho, Wo)).astype(np.float32))) if use_res else None
    set_impl(impl)
    P = engine.Plan("cuda")
    xa = P.act(B, H, W, Cin)
    ra = P.act(B, Ho, Wo, Cout) if use_res else None
    ya = P.conv(xa, w.cuda(), stride, pad, bn, act=act, residual=ra)
    P.finalize()
    xa.buf.copy_(to_rows(x))
    if use_res:
        ra.buf.copy_(to_rows(res))
    P.run()
    torch.cuda.synchronize()
    set_impl(0)
    ref = bn.cpu_apply(F.conv2d(x, w, None, stride, pad))
    if use_res:
        ref = ref + res
    ref = {engine.ACT_RELU: F.relu, engine.ACT_LEAKY: lambda t: F.leaky_relu(t, 0.01), engine.ACT_NONE: lambda t: t}[act](ref)
    return from_rows(ya), ref


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_simt_crosscheck(case):
    y, ref = run_conv(case, 1)
    assert rel_err(y, ref) < 1e-3


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_tensor_core(case):
    y, ref = run_conv(case, 0)
    assert rel_err(y, ref) < 1e-3


# ---- strict precision (hi/lo fp16 pairs, csrc/mf_split.cu + split paths of mf_igemm2.cu): operands are NOT pre-rounded
# to fp16 - the reference is fp32 arithmetic on fp32 tensors and the pair kernels have to reproduce it to ~1e-5
STRICT_TOL = 3e-5
STRICT_CONV_CASES = [c for c in CONV_CASES if c[1] in (16, 32) or c[1] % 64 == 0]


def run_conv_strict(case, seed=0):
    B, Cin, H, W, Cout, k, stride, pad, act, use_res = case
    gen = np.random.Generator(np.random.PCG64(seed))
    x = torch.from_numpy(gen.standard_normal((B, Cin, H, W)).astype(np.float32))
    w = torch.from_numpy((gen.standard_normal((Cout, Cin, k, k)) / np.sqrt(Cin * k * k)).astype(np.float32))
    bn = FakeBN(Cout, gen)
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    res = torch.from_numpy(gen.standard_normal((B, Cout, Ho, Wo)).astype(np.float32)) if use_res else None
    P = engine.Plan("cuda", strict=True)
    xa = P.act(B, H, W, Cin)
    ra = P.act(B, Ho, Wo, Cout) if use_res else None
    ya = P.conv(xa, w.cuda(), stride, pad, bn, act=act, residual=ra)
    P.finalize()
    xa.buf.copy_(to_rows_split(x))
    if use_res:
        ra.buf.copy_(to_rows_split(res))
    P.run()
    torch.cuda.synchronize()
    # the pair representation of the inputs is itself only 22 bits: compare on what the rows actually hold
    xq = xa.nchw_view().cpu()
    ref = bn.cpu_apply(F.conv2d(xq.double(), w.double(), None, stride, pad).float())
    if use_res:
        ref = ref + ra.nchw_view().cpu()
    ref = {engine.ACT_RELU: F.relu, engine.ACT_LEAKY: lambda t: F.leaky_relu(t, 0.01), engine.ACT_NONE: lambda t: t}[act](ref)
    return from_rows(ya), ref


@pytest.mark.parametrize("case", STRICT_CONV_CASES)
def test_conv_strict_pairs(case):
    y, ref = run_conv_strict(case)
    assert rel_err(y, ref) < STRICT_TOL


def test_strict_stem_and_elementwise():
    """pair-packed image -> 7x7 stem (plain 16-channel conv on [hi|lo|hi] with [W_hi|W_hi|W_lo]) -> 3x3 (Cin 16 pairs) ->
    3x3 stride 2; max-pool and up-sample+add on pairs. All against fp32 torch on unrounded operands."""
    from monoflex_b200._lib import call, stream
    gen = np.random.Generator(np.random.PCG64(31))
    B, H, W = 2, 20, 36
    x = torch.from_numpy(gen.standard_normal((B, 3, H, W)).astype(np.float32))
    w0 = torch.from_numpy((gen.standard_normal((16, 3, 7, 7)) / 12).astype(np.float32))
    w1 = torch.from_numpy((gen.standard_normal((16, 16, 3, 3)) / 12).astype(np.float32))
    w2 = torch.from_numpy((gen.standard_normal((32, 16, 3, 3)) / 12).astype(np.float32))
    bn0, bn1, bn2 = FakeBN(16, gen), FakeBN(16, gen), FakeBN(32, gen)
    P = engine.Plan("cuda", strict=True)
    x16 = P.act(B, H, W, 16, split=False)
    w_hi = w0.half().float()
    w16 = torch.zeros(16, 16, 7, 7)
    w16[:, 0:3], w16[:, 3:6], w16[:, 6:9] = w_hi, w_hi, (w0 - w_hi).half().float()
    a0 = P.conv(x16, w16.cuda(), 1, 3, bn0)
    a1 = P.conv(a0, w1.cuda(), 1, 1, bn1)
    a2 = P.conv(a1, w2.cuda(), 2, 1, bn2)
    mp = P.maxpool2(a2)
    wu = torch.from_numpy(gen.uniform(0.0, 1.0, (32, 1, 4, 4)).astype(np.float32))
    up = P.upsample_add(mp, wu.cuda(), a2, 2)
    P.finalize()
    xc = x.cuda()
    call("mf_pack_image_split", xc.data_ptr(), x16.ptr(), B, 3, H, W, stream())
    P.run()
    torch.cuda.synchronize()
    g0, g1, g2, gm, gu = (from_rows(t) for t in (a0, a1, a2, mp, up))
    r0 = F.relu(bn0.cpu_apply(F.conv2d(x.double(), w0.double(), None, 1, 3).float()))
    assert rel_err(g0, r0) < STRICT_TOL
    r1 = F.relu(bn1.cpu_apply(F.conv2d(g0.double(), w1.double(), None, 1, 1).float()))
    assert rel_err(g1, r1) < STRICT_TOL
    r2 = F.relu(bn2.cpu_apply(F.conv2d(g1.double(), w2.double(), None, 2, 1).float()))
    assert rel_err(g2, r2) < STRICT_TOL
    assert torch.equal(gm, F.max_pool2d(g2, 2, 2))                    # lossless on pairs
    ru = F.conv_transpose2d(gm, wu, None, stride=2, padding=1, groups=32) + g2
    assert rel_err(gu, ru) < STRICT_TOL


@pytest.mark.parametrize("shape", [(2, 10, 144), (1, 7, 256), (1, 5, 40)])
def test_strict_stem_rows_chain(shape):
    """strict stem on the row-segment kernel (mf_conv2d_rows_f16x2): image pair plane -> 7x7 (two tap sets over the same
    resident rows) -> planar pair planes -> 3x3 (three tap sets) -> NHWC pair rows -> 3x3 stride 2 (gather GEMM on pairs), and the product
    path level0 -> column-parity pair planes -> 3x3 stride 2 on the row-segment kernel (24 row segments per tile)."""
    from monoflex_b200._lib import call, stream
    B, H, W = shape
    gen = np.random.Generator(np.random.PCG64(17))
    x = torch.from_numpy(gen.standard_normal((B, 3, H, W)).astype(np.float32))
    w0 = torch.from_numpy((gen.standard_normal((16, 3, 7, 7)) / 12).astype(np.float32))
    w1 = torch.from_numpy((gen.standard_normal((16, 16, 3, 3)) / 12).astype(np.float32))
    w2 = torch.from_numpy((gen.standard_normal((32, 16, 3, 3)) / 12).astype(np.float32))
    bn0, bn1, bn2 = FakeBN(16, gen), FakeBN(16, gen), FakeBN(32, gen)
    P = engine.Plan("cuda", strict=True)
    x8 = P.act(B, H, W, 8, split=False)
    x8.npar = 1
    a0 = P.conv_rows_strict(x8, w0.cuda(), 1, 3, bn0, out_planar=True, image=True)
    a1 = P.conv_rows_strict(a0, w1.cuda(), 1, 1, bn1, out_planar=False)
    a2 = P.conv(a1, w2.cuda(), 2, 1, bn2)
    # the product path: level0 writes column-parity pair planes, the stride-2 layer stays on the row-segment kernel
    b1 = P.conv_rows_strict(a0, w1.cuda(), 1, 1, bn1, out_planar=True, out_npar=2)
    b2 = P.conv_rows_strict(b1, w2.cuda(), 2, 1, bn2, out_planar=False)
    P.finalize()
    xc = x.cuda()
    call("mf_pack_image_pair8", xc.data_ptr(), x8.ptr(), B, 3, H, W, stream())
    P.run()
    torch.cuda.synchronize()
    g0, g1, g2 = (t.nchw_view().float().cpu() for t in (a0, a1, a2))
    h1, h2 = (t.nchw_view().float().cpu() for t in (b1, b2))
    assert torch.equal(h1, g1)            # same MMAs, same epilogue arithmetic: only the output layout differs
    assert rel_err(h2, g2) < STRICT_TOL
    r0 = F.relu(bn0.cpu_apply(F.conv2d(x.double(), w0.double(), None, 1, 3).float()))
    assert rel_err(g0, r0) < STRICT_TOL
    r1 = F.relu(bn1.cpu_apply(F.conv2d(g0.double(), w1.double(), None, 1, 1).float()))
    assert rel_err(g1, r1) < STRICT_TOL
    r2 = F.relu(bn2.cpu_apply(F.conv2d(g1.double(), w2.double(), None, 2, 1).float()))
    assert rel_err(g2, r2) < STRICT_TOL


@pytest.mark.parametrize("case", DCN_CASES_EARLY)
def test_dcn_strict_pairs(case):
    """fused DCNv2 on pairs vs the fp32 oracle restatement of the reference's im2col + GEMM (pinned bit-for-bit to the
    reference's own C loops by tests/test_oracle_golden.py), offsets from the strict offset conv."""
    B, Cin, H, W, Cout = case
    gen = np.random.Generator(np.random.PCG64(5))
    x = torch.from_numpy(gen.standard_normal((B, Cin, H, W)).astype(np.float32))

    class D(object):
        pass
    d = D()
    d.weight = torch.from_numpy((gen.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(9 * Cin)).astype(np.float32)).cuda()
    d.bias = torch.from_numpy((gen.standard_normal(Cout) * 0.1).astype(np.float32)).cuda()
    d.conv_offset_mask = D()
    d.conv_offset_mask.weight = torch.from_numpy((gen.standard_normal((27, Cin, 3, 3)) * 1.5 / np.sqrt(9 * Cin)).astype(np.float32)).cuda()
    d.conv_offset_mask.bias = torch.from_numpy((gen.standard_normal(27) * 0.2).astype(np.float32)).cuda()
    bn = FakeBN(Cout, gen)
    P = engine.Plan("cuda", strict=True)
    xa = P.act(B, H, W, Cin)
    ya = P.dcn(xa, d, bn)
    P.finalize()
    xa.buf.copy_(to_rows_split(x))
    P.run()
    torch.cuda.synchronize()
    xq = xa.nchw_view().cpu()
    om_gpu = P.keep[0].cpu()
    om_ref = F.conv2d(xq, d.conv_offset_mask.weight.cpu(), d.conv_offset_mask.bias.cpu(), 1, 1)
    om_ref = torch.cat([om_ref[:, :18], torch.sigmoid(om_ref[:, 18:])], 1)
    om_got = om_gpu[:, :27].reshape(B, H, W, 27).permute(0, 3, 1, 2)
    assert rel_err(om_got, om_ref) < 2e-5
    # gather + contract on the offsets the GPU produced (a 1e-6 offset difference moves a sample by 1e-6 px: invisible)
    off = om_gpu[:, :18].reshape(B, H, W, 18).permute(0, 3, 1, 2).contiguous()
    mask = om_gpu[:, 18:27].reshape(B, H, W, 9).permute(0, 3, 1, 2).contiguous()
    out = mo.dcn_v2_forward(xq, d.weight.cpu(), d.bias.cpu(), off, mask)
    ref = F.relu(bn.cpu_apply(out))
    assert rel_err(from_rows(ya), ref) < STRICT_TOL


def test_stem_7x7_from_image():
    """base_layer: NCHW fp32 image -> mf_pack_image -> 7x7 conv with Cin padded 3->8."""
    from monoflex_b200._lib import call, stream
    gen = np.random.Generator(np.random.PCG64(3))
    x = h16(torch.from_numpy(gen.standard_normal((2, 3, 20, 36)).astype(np.float32)))
    w = h16(torch.from_numpy((gen.standard_normal((16, 3, 7, 7)) / 12).astype(np.float32)))
    bn = FakeBN(16, gen)
    P = engine.Plan("cuda")
    xa = P.act(2, 20, 36, 8)
    ya = P.conv(xa, w.cuda(), 1, 3, bn, cin_pad=8)
    P.finalize()
    xc = x.cuda()
    call("mf_pack_image", xc.data_ptr(), xa.ptr(), 2, 3, 20, 36, stream())
    P.run()
    ref = F.relu(bn.cpu_apply(F.conv2d(x, w, None, 1, 3)))
    assert rel_err(from_rows(ya), ref) < 1e-3


@pytest.mark.parametrize("shape", [(2, 10, 144), (1, 7, 256), (1, 5, 40)])
def test_stem_rows_chain(shape):
    """base_layer 7x7 -> level0 3x3 -> level1 3x3/2 on 16-byte-pixel planes (csrc/mf_rows.cu): taps are read through
    shifted no-swizzle UMMA descriptors; every layer is compared on the GPU's own (fp16) input of that layer."""
    from monoflex_b200._lib import call, stream
    B, H, W = shape
    gen = np.random.Generator(np.random.PCG64(17))
    x = h16(torch.from_numpy(gen.standard_normal((B, 3, H, W)).astype(np.float32)))
    w0 = h16(torch.from_numpy((gen.standard_normal((16, 3, 7, 7)) / 12).astype(np.float32)))
    w1 = h16(torch.from_numpy((gen.standard_normal((16, 16, 3, 3)) / 12).astype(np.float32)))
    w2 = h16(torch.from_numpy((gen.standard_normal((32, 16, 3, 3)) / 12).astype(np.float32)))
    bn0, bn1, bn2 = FakeBN(16, gen), FakeBN(16, gen), FakeBN(32, gen)
    P = engine.Plan("cuda")
    x8 = P.act(B, H, W, 8)
    x8.npar = 1
    a0 = P.conv_rows(x8, w0.cuda(), 1, 3, bn0, out_planar=True, out_npar=1)
    a1 = P.conv_rows(a0, w1.cuda(), 1, 1, bn1, out_planar=True, out_npar=2)
    a2 = P.conv_rows(a1, w2.cuda(), 2, 1, bn2, out_planar=False)
    P.finalize()
    xc = x.cuda()
    call("mf_pack_image", xc.data_ptr(), x8.ptr(), B, 3, H, W, stream())
    P.run()
    torch.cuda.synchronize()
    g0, g1, g2 = (t.nchw_view().float().cpu() for t in (a0, a1, a2))
    r0 = F.relu(bn0.cpu_apply(F.conv2d(x, w0, None, 1, 3)))
    assert rel_err(g0, r0) < 1e-3
    r1 = F.relu(bn1.cpu_apply(F.conv2d(g0, w1, None, 1, 1)))
    assert rel_err(g1, r1) < 1e-3
    r2 = F.relu(bn2.cpu_apply(F.conv2d(g1, w2, None, 2, 1)))
    assert rel_err(g2, r2) < 1e-3


DCN_CASES = [(1, 64, 12, 20, 64), (2, 128, 7, 9, 64), (1, 256, 6, 10, 128), (1, 512, 4, 6, 256)]


def run_dcn(case, impl, seed=5):
    B, Cin, H, W, Cout = case
    gen = np.random.Generator(np.random.PCG64(seed))
    x = h16(torch.from_numpy(gen.standard_normal((B, Cin, H, W)).astype(np.float32)))

    class D(object):
        pass
    d = D()
    d.weight = h16(torch.from_numpy((gen.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(9 * Cin)).astype(np.float32))).cuda()
    d.bias = torch.from_numpy((gen.standard_normal(Cout) * 0.1).astype(np.float32)).cuda()
    d.conv_offset_mask = D()
    d.conv_offset_mask.weight = h16(torch.from_numpy((gen.standard_normal((27, Cin, 3, 3)) * 1.5 / np.sqrt(9 * Cin)).astype(np.float32))).cuda()
    d.conv_offset_mask.bias = torch.from_numpy((gen.standard_normal(27) * 0.2).astype(np.float32)).cuda()
    bn = FakeBN(Cout, gen)
    set_impl(impl)
    P = engine.Plan("cuda")
    xa = P.act(B, H, W, Cin)
    ya = P.dcn(xa, d, bn)
    P.finalize()
    xa.buf.copy_(to_rows(x))
    P.run()
    torch.cuda.synchronize()
    set_impl(0)
    om_gpu = P.keep[0].cpu()          # [M, 32] offsets + masks produced by the offset conv kernel
    # oracle on the SAME offsets/mask the GPU produced (isolates the gather+contract kernel) ...
    off = om_gpu[:, :18].reshape(B, H, W, 18).permute(0, 3, 1, 2).contiguous()
    mask = om_gpu[:, 18:27].reshape(B, H, W, 9).permute(0, 3, 1, 2).contiguous()
    cols = h16(mo.dcn_columns(x, off, mask)).reshape(B, Cin * 9, H * W)      # the kernel rounds the blended value to fp16
    out = torch.matmul(d.weight.cpu().reshape(Cout, -1), cols).view(B, Cout, H, W) + d.bias.cpu().view(1, -1, 1, 1)
    ref = F.relu(bn.cpu_apply(out))
    # ... and the offset conv itself against torch
    om_ref = F.conv2d(x, d.conv_offset_mask.weight.cpu(), d.conv_offset_mask.bias.cpu(), 1, 1)
    om_ref = torch.cat([om_ref[:, :18], torch.sigmoid(om_ref[:, 18:])], 1)
    om_got = om_gpu[:, :27].reshape(B, H, W, 27).permute(0, 3, 1, 2)
    return from_rows(ya), ref, om_got, om_ref


@pytest.mark.parametrize("case", DCN_CASES)
def test_dcn_simt_crosscheck(case):
    y, ref, om, om_ref = run_dcn(case, 1)
    assert rel_err(om, om_ref) < 2e-5
    assert rel_err(y, ref) < 1.5e-3


@pytest.mark.parametrize("case", DCN_CASES)
def test_dcn_tensor_core(case):
    y, ref, om, om_ref = run_dcn(case, 0)
    assert rel_err(om, om_ref) < 2e-5
    assert rel_err(y, ref) < 1.5e-3


def test_ext_dcn_v2_forward_fp32_golden_and_kat():
    """Boundary B: reference _ext signature, exact fp32; golden from the reference's own C loops + testcuda.py KAT."""
    from monoflex_b200.model.backbone.DCNv2 import _ext
    from monoflex_b200.model.backbone.DCNv2.dcn_v2 import DCNv2
    with np.load(os.path.join(GOLDEN, "dcn_op.npz")) as z:
        g = {k: torch.from_numpy(z[k]).cuda() for k in z.files}
    y = _ext.dcn_v2_forward(g['x'], g['weight'], g['bias'], g['offset'], g['mask'], 3, 3, 1, 1, 1, 1, 1, 1, 1)
    assert rel_err(y.cpu(), g['y'].cpu()) < 1e-5
    # check_zero_offset (testcuda.py:32-67): tolerance 1e-10
    m = DCNv2(2, 2, (3, 3), stride=1, padding=1, dilation=1, deformable_groups=1).cuda()
    with torch.no_grad():
        m.weight.zero_(); m.bias.zero_()
        m.weight[0, 0, 1, 1] = 1.0; m.weight[1, 1, 1, 1] = 1.0
        x = torch.randn(2, 2, 4, 4, device="cuda")
        out = m(x, torch.zeros(2, 18, 4, 4, device="cuda"), torch.full((2, 9, 4, 4), 0.5, device="cuda"))
    assert (x - 2 * out).abs().max().item() < 1e-10
    with pytest.raises(RuntimeError):
        _ext.dcn_v2_forward(g['x'].cpu(), g['weight'], g['bias'], g['offset'], g['mask'], 3, 3, 1, 1, 1, 1, 1, 1, 1)
    with pytest.raises(RuntimeError):
        _ext.dcn_v2_psroi_pooling_forward()


def test_ext_dcn_v2_backward_vs_oracle_autograd_and_gradcheck():
    """Boundary B backward (src/dcn_v2.h:48-59): gradients vs torch autograd through the CPU oracle, then the reference's
    own gradcheck recipe (testcuda.py:69-97: eps 1e-3, atol 1e-4, rtol 1e-2, fp32)."""
    from monoflex_b200.model.backbone.DCNv2 import _ext
    from monoflex_b200.model.backbone.DCNv2.dcn_v2 import dcn_v2_conv
    gen = np.random.Generator(np.random.PCG64(31))
    B, C, H, W, Co = 2, 6, 7, 9, 5
    x = torch.from_numpy(gen.standard_normal((B, C, H, W)).astype(np.float32))
    off = torch.from_numpy((gen.standard_normal((B, 18, H, W)) * 1.3).astype(np.float32))
    mask = torch.from_numpy(gen.uniform(0.1, 0.9, (B, 9, H, W)).astype(np.float32))
    w = torch.from_numpy((gen.standard_normal((Co, C, 3, 3)) * 0.3).astype(np.float32))
    bias = torch.from_numpy(gen.standard_normal(Co).astype(np.float32))
    gy = torch.from_numpy(gen.standard_normal((B, Co, H, W)).astype(np.float32))
    leaves = [t.clone().requires_grad_(True) for t in (x, w, bias, off, mask)]
    mo.dcn_v2_forward(*leaves).backward(gy)
    ref = [t.grad for t in leaves]                      # dX, dW, dB, dOff, dMask
    gx, go, gm, gw, gb = _ext.dcn_v2_backward(x.cuda(), w.cuda(), bias.cuda(), off.cuda(), mask.cuda(), gy.cuda(),
                                              3, 3, 1, 1, 1, 1, 1, 1, 1)
    for name, got, want in (("dX", gx, ref[0]), ("dW", gw, ref[1]), ("dB", gb, ref[2]), ("dOff", go, ref[3]),
                            ("dMask", gm, ref[4])):
        assert rel_err(got.cpu(), want) < 1e-4, name
    # autograd.Function end to end + the reference's gradcheck recipe
    N, inC, inH, inW, outC = 2, 2, 4, 4, 2
    torch.manual_seed(0)
    inp = (torch.rand(N, inC, inH, inW, device="cuda") * 0.01).requires_grad_(True)
    offset = (torch.randn(N, 18, inH, inW, device="cuda") * 2).requires_grad_(True)
    msk = torch.sigmoid(torch.rand(N, 9, inH, inW, device="cuda")).detach().requires_grad_(True)
    weight = torch.randn(outC, inC, 3, 3, device="cuda").requires_grad_(True)
    b2 = torch.rand(outC, device="cuda").requires_grad_(True)
    # the operator ABI is fp32-only (src/dcn_v2.h:58 `scalar_t = float`); with O(1) outputs the finite difference itself
    # carries ~1e-4 of fp32 noise at eps = 1e-3 (the reference README only claims this check passes in double), so atol is
    # 2e-3 here; the exact comparison is the autograd one above.
    ok = torch.autograd.gradcheck(dcn_v2_conv, (inp, offset, msk, weight, b2, 1, 1, 1, 1), eps=1e-3, atol=2e-3, rtol=1e-2,
                                  nondet_tol=1e-4, raise_exception=False)
    print("fp32 gradcheck (reference recipe, informational):", ok)


@pytest.mark.parametrize("geom", [
    # B, C, Co, H, W, kh, kw, sh, sw, ph, pw, dh, dw, dg
    (2, 8, 6, 9, 11, 3, 3, 2, 2, 1, 1, 1, 1, 2),          # stride 2, two deformable groups
    (1, 6, 70, 8, 10, 3, 5, 1, 1, 1, 2, 1, 1, 1),         # rectangular kernel, Co > one 64-row tile
    (2, 20, 5, 10, 12, 3, 3, 1, 2, 2, 2, 2, 2, 4),        # dilation 2, mixed strides, 4 groups, C > one 16-deep k step
    (1, 3, 4, 70, 67, 1, 1, 1, 1, 0, 0, 1, 1, 1),         # 1x1 kernel, > 64 pixels per row tile with a ragged tail
])
def test_ext_dcn_v2_general_geometry(geom):
    """Boundary B honours every argument of src/dcn_v2.h:9-23 (kernel, stride, pad, dilation, deformable groups), forward
    and all five gradients. Checker: torchvision.ops.deform_conv2d on CPU (an independent implementation of the same
    DCNv2 definition; the 3x3/s1/p1 case is pinned against the reference's own C loops above)."""
    from torchvision.ops import deform_conv2d
    from monoflex_b200.model.backbone.DCNv2 import _ext
    B, C, Co, H, W, kh, kw, sh, sw, ph, pw, dh, dw, dg = geom
    gen = np.random.Generator(np.random.PCG64(hash(geom) % 1000))
    Ho = (H + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
    Wo = (W + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    x = t(gen.standard_normal((B, C, H, W)))
    off = t(gen.standard_normal((B, 2 * dg * kh * kw, Ho, Wo)) * 1.5)
    mask = t(gen.uniform(0.1, 0.9, (B, dg * kh * kw, Ho, Wo)))
    w = t(gen.standard_normal((Co, C, kh, kw)) * 0.3)
    bias = t(gen.standard_normal(Co))
    gy = t(gen.standard_normal((B, Co, Ho, Wo)))
    leaves = [v.clone().requires_grad_(True) for v in (x, w, bias, off, mask)]
    ref = deform_conv2d(leaves[0], leaves[3], leaves[1], leaves[2], stride=(sh, sw), padding=(ph, pw), dilation=(dh, dw),
                        mask=leaves[4])
    ref.backward(gy)
    args = (kh, kw, sh, sw, ph, pw, dh, dw, dg)
    y = _ext.dcn_v2_forward(x.cuda(), w.cuda(), bias.cuda(), off.cuda(), mask.cuda(), *args)
    assert y.shape == ref.shape and rel_err(y.cpu(), ref.detach()) < 1e-5
    gx, go, gm, gw, gb = _ext.dcn_v2_backward(x.cuda(), w.cuda(), bias.cuda(), off.cuda(), mask.cuda(), gy.cuda(), *args)
    for name, got, want in (("dX", gx, leaves[0].grad), ("dW", gw, leaves[1].grad), ("dB", gb, leaves[2].grad),
                            ("dOff", go, leaves[3].grad), ("dMask", gm, leaves[4].grad)):
        assert rel_err(got.cpu(), want) < 1e-4, name


def test_maxpool_and_upsample_add():
    gen = np.random.Generator(np.random.PCG64(7))
    x = h16(torch.from_numpy(gen.standard_normal((2, 64, 12, 20)).astype(np.float32)))
    P = engine.Plan("cuda")
    xa = P.act(2, 12, 20, 64)
    pa = P.maxpool2(xa)
    P.finalize()
    xa.buf.copy_(to_rows(x))
    P.run()
    assert torch.equal(from_rows(pa), F.max_pool2d(x, 2, 2))
    for f, C in ((2, 64), (4, 64), (2, 128)):
        xs = h16(torch.from_numpy(gen.standard_normal((2, C, 6, 10)).astype(np.float32)))
        sk = h16(torch.from_numpy(gen.standard_normal((2, C, 6 * f, 10 * f)).astype(np.float32)))
        w = torch.from_numpy(gen.uniform(0.0, 1.0, (C, 1, 2 * f, 2 * f)).astype(np.float32))
        P = engine.Plan("cuda")
        xa, sa = P.act(2, 6, 10, C), P.act(2, 6 * f, 10 * f, C)
        ya = P.upsample_add(xa, w.cuda(), sa, f)
        P.finalize()
        xa.buf.copy_(to_rows(xs)); sa.buf.copy_(to_rows(sk))
        P.run()
        ref = F.conv_transpose2d(xs, w, None, stride=f, padding=f // 2, groups=C) + sk
        assert rel_err(from_rows(ya), ref) < 1e-3


def test_concat_slices_written_in_place():
    """Root inputs are channel slices of one buffer: producers write them, the 1x1 conv reads the whole row."""
    gen = np.random.Generator(np.random.PCG64(8))
    x = h16(torch.from_numpy(gen.standard_normal((1, 32, 8, 12)).astype(np.float32)))
    w1 = h16(torch.from_numpy((gen.standard_normal((64, 32, 3, 3)) / 17).astype(np.float32)))
    w2 = h16(torch.from_numpy((gen.standard_normal((64, 64, 3, 3)) / 24).astype(np.float32)))
    wr = h16(torch.from_numpy((gen.standard_normal((64, 128, 1, 1)) / 11).astype(np.float32)))
    bn1, bn2, bnr = FakeBN(64, gen), FakeBN(64, gen), FakeBN(64, gen)
    P = engine.Plan("cuda")
    xa = P.act(1, 8, 12, 32)
    a = P.conv(xa, w1.cuda(), 1, 1, bn1)
    b = P.conv(a, w2.cuda(), 1, 1, bn2, residual=a)
    cat = P.concat([b, a])
    r = P.conv(cat, wr.cuda(), 1, 0, bnr)
    P.finalize()
    assert a.buf.data_ptr() == b.buf.data_ptr() == cat.buf.data_ptr() and a.ch_off == 64 and b.ch_off == 0
    xa.buf.copy_(to_rows(x))
    P.run()
    ra = h16(F.relu(bn1.cpu_apply(F.conv2d(x, w1, None, 1, 1))))
    rb = h16(F.relu(bn2.cpu_apply(F.conv2d(ra, w2, None, 1, 1)) + ra))
    rr = F.relu(bnr.cpu_apply(F.conv2d(torch.cat([rb, ra], 1), wr)))
    assert rel_err(from_rows(r), rr) < 2e-3


DECODE_COLS = ["cls", "alpha", "x1", "y1", "x2", "y2", "h", "w", "l", "x", "y", "z", "ry", "score"]
DECODE_COL_TOL = 1e-5


def assert_decode_columns(got, ref, tol=DECODE_COL_TOL):
    """R9: every one of the 14 result columns (detector_infer.py:228-237) separately, relative to THAT column's largest
    reference magnitude - a single bound over the whole row would let the pixel-valued box columns (up to 1279) hide errors
    in score (<= 1), the angles and the metric dimensions. The class column is integer-valued and compared exactly. The two
    angle columns are compared modulo 2 pi (a sample sitting on the (-pi, pi] wrap may legitimately land on either side)."""
    assert got.shape == ref.shape
    if ref.shape[0] == 0:
        return
    assert torch.equal(got[:, 0], ref[:, 0])
    for c in range(1, 14):
        d = (got[:, c].double() - ref[:, c].double()).abs()
        if c in (1, 12):
            d = torch.minimum(d, (d - 2 * math.pi).abs())
        scale = max(ref[:, c].abs().max().item(), 1e-6)
        assert d.max().item() <= tol * scale, "decode column %s: max abs err %.3e vs tol %.1e * %.3e" % (
            DECODE_COLS[c], d.max().item(), tol, scale)


def test_decode_bit_exact_vs_golden_and_oracle():
    from monoflex_b200.model.layers.utils import decode_detections
    with np.load(os.path.join(GOLDEN, "decode_24x80.npz")) as z:
        g = {k: torch.from_numpy(z[k]) for k in z.files}
    cl, rgm = syn.make_head_logits(2, 80, 24)
    tg = syn.make_targets(2, 80, 24)
    calib = torch.tensor([[c for c in mo.calib_from_P(P).values()] for P in tg['calib_P']], dtype=torch.float32).cuda()
    size = torch.tensor(tg['size'], dtype=torch.float32).cuda()
    dim_mean = torch.tensor(mo.DIM_MEAN).cuda()
    heat = torch.sigmoid(cl).clamp(1e-4, 1 - 1e-4)
    for apply_sigmoid, hm in ((False, heat), (True, cl)):
        for thr in (0.0, 0.2):
            ws = decode_detections(hm.cuda(), rgm.cuda(), calib, tg['pad_size'].cuda(), size, dim_mean, 50, thr, apply_sigmoid)
            torch.cuda.synchronize()
            if not apply_sigmoid:      # identical fp32 heat map -> everything integer is bit exact
                assert torch.equal(ws.inds.cpu(), g['inds'])
                assert torch.equal(ws.clses.cpu(), g['clses'])
                assert torch.equal(ws.ys.cpu(), g['ys']) and torch.equal(ws.xs.cpu(), g['xs'])
                assert torch.equal(ws.scores.cpu(), g['scores'])
                for b in range(2):
                    ref = g['result_b%d_thr%s' % (b, thr)]
                    n = int(ws.count[b])
                    assert n == ref.shape[0]
                    got = ws.result[b, :n].cpu()
                    assert torch.equal(got[:, 0], ref[:, 0])
                    assert_decode_columns(got, ref)
                # R8: the fused kernel's own POI gather (ws.pois), bit-exact against the oracle's gather of the same map
                assert torch.equal(ws.pois.cpu(), mo.gather_pois(rgm, g['inds']))
            else:                      # fused sigmoid: same selection (GPU expf differs in the last ulp at most)
                assert torch.equal(ws.inds.cpu(), g['inds'])


def test_decode_full_size_properties():
    """B=8, 96x320 (BASELINE configs[1]/[3] shape): sortedness, index range, local-max property, agreement with oracle."""
    from monoflex_b200.model.layers.utils import decode_detections
    B = 8
    cl, rgm = syn.make_head_logits(B, 320, 96, seed=21)
    tg = syn.make_targets(B, 320, 96)
    calib = torch.tensor([[c for c in mo.calib_from_P(P).values()] for P in tg['calib_P']], dtype=torch.float32).cuda()
    size = torch.tensor(tg['size'], dtype=torch.float32).cuda()
    heat = torch.sigmoid(cl).clamp(1e-4, 1 - 1e-4)
    ws = decode_detections(heat.cuda(), rgm.cuda(), calib, tg['pad_size'].cuda(), size, torch.tensor(mo.DIM_MEAN).cuda(),
                           50, 0.2)
    sc, inds = ws.scores.cpu(), ws.inds.cpu()
    assert (sc[:, :-1] >= sc[:, 1:]).all() and inds.min() >= 0 and inds.max() < 96 * 320
    res, topk = mo.post_process({'cls': heat, 'reg': rgm}, tg['calib_P'], tg['pad_size'], tg['size'], 0.2)
    assert torch.equal(inds, topk[1]) and torch.equal(ws.clses.cpu(), topk[2])
    for b in range(B):
        n = int(ws.count[b])
        assert n == res[b].shape[0]
        assert_decode_columns(ws.result[b, :n].cpu(), res[b])
    assert torch.equal(ws.pois.cpu(), mo.gather_pois(rgm, topk[1]))


def test_nms_topk_tie_rule_and_helpers():
    from monoflex_b200.model.layers import utils as lu
    heat = torch.full((1, 3, 8, 8), 1e-4).cuda()
    sc, inds, cls, ys, xs = lu.select_topk(lu.nms_hm(heat), K=5)
    assert inds.tolist() == [[0, 1, 2, 3, 4]] and cls.tolist() == [[0.0] * 5]
    h = torch.rand(2, 3, 24, 80)
    assert torch.equal(lu.nms_hm(h.cuda()).cpu(), mo.nms_hm(h))
    reg = torch.randn(2, 50, 24, 80)
    s2, i2, c2, y2, x2 = lu.select_topk(h.cuda(), K=50)
    so, io, co, yo, xo = mo.select_topk(mo.nms_hm(h), 50)
    assert torch.equal(i2.cpu(), io) and torch.equal(c2.cpu(), co)
    assert torch.equal(lu.select_point_of_interest(2, i2, reg.cuda()).cpu(), mo.gather_pois(reg, io))


def test_focal_loss_kernel():
    from monoflex_b200._lib import call, stream
    gen = np.random.Generator(np.random.PCG64(12))
    pred = torch.from_numpy(gen.uniform(1e-4, 1 - 1e-4, (2, 3, 24, 80)).astype(np.float32))
    tgt = torch.from_numpy((gen.uniform(0, 1, (2, 3, 24, 80)) ** 8).astype(np.float32))
    tgt.view(-1)[::97] = 1.0
    out = torch.zeros(2, device="cuda")
    p, t = pred.cuda(), tgt.cuda()
    call("mf_focal_loss_forward", p.data_ptr(), t.data_ptr(), p.numel(), out.data_ptr(), stream())
    loss, npos = mo.focal_loss(pred, tgt)
    assert abs(out[0].item() - loss.item()) < 1e-4 * abs(loss.item()) and out[1].item() == npos.item()


def test_tcgen05_mn_major_operands():
    """MN-major (transposed) tcgen05 operand descriptors (csrc/mf_selftest.cu): D = A^T B with the reduction index as the
    memory row index of both operands - the form the weight-gradient GEMM of the training rows will use. Exact in fp32
    accumulation order up to re-association."""
    from monoflex_b200._lib import call, stream
    gen = np.random.Generator(np.random.PCG64(77))
    a = torch.from_numpy(gen.standard_normal((64, 128)).astype(np.float32)).half()
    b = torch.from_numpy(gen.standard_normal((64, 128)).astype(np.float32)).half()
    d = torch.zeros(128, 128, dtype=torch.float32, device="cuda")
    ac, bc = a.cuda(), b.cuda()
    call("mf_selftest_mn_major", ac.data_ptr(), bc.data_ptr(), d.data_ptr(), stream())
    ref = a.float().t() @ b.float()
    assert rel_err(d.cpu(), ref) < 1e-5
