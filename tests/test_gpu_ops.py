"""Kernel-level parity on the GPU, through the C ABI: the convolution operator (tcgen05 implicit GEMM in both
precision modes, and the SIMT reference conv) against torch fp32 F.conv2d on the CPU, and the standalone
depthwise cross-correlation against the oracle."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN, assert_close
import siammask_b200 as smb
from oracle.siammask_oracle import Oracle, xcorr_depthwise_loops

pytestmark = pytest.mark.gpu

# (name, B, Cin, H, Cout, k, stride, pad, dil)   — the geometries that occur on the hot path (SURVEY App. A)
CONV_CASES = [
    ("1x1_64_256", 2, 64, 63, 256, 1, 1, 0, 1),          # layer1 conv3 / downsample (tiled-TMA path)
    ("1x1_1024_256", 1, 1024, 31, 256, 1, 1, 0, 1),      # layer3 conv1 / ResDownS
    ("1x1_256_64", 2, 256, 17, 64, 1, 1, 0, 1),
    ("3x3_p1", 2, 64, 63, 64, 3, 1, 1, 1),               # layer1 conv2 (im2col TMA, zero padding)
    ("3x3_s2_p0", 2, 128, 63, 128, 3, 2, 0, 1),          # layer2.0 conv2 (stride 2)
    ("3x3_s2_p0_ds", 1, 256, 63, 512, 3, 2, 0, 1),       # layer2.0 downsample
    ("3x3_d2_p2", 2, 256, 31, 256, 3, 1, 2, 2),          # layer3.1-5 conv2 (dilation 2)
    ("3x3_p1_ds3", 1, 512, 31, 1024, 3, 1, 1, 1),        # layer3.0 downsample (the 4.5 GMAC conv)
    ("3x3_p0_search", 2, 256, 31, 256, 3, 1, 0, 1),      # conv_search 31 -> 29
    ("3x3_p0_kernel", 3, 256, 7, 256, 3, 1, 0, 1),       # conv_kernel 7 -> 5 (M = 75 < one tile)
    ("1x1_head10", 2, 256, 25, 10, 1, 1, 0, 1),          # head.3 cls (N tail, NCHW epilogue)
    ("1x1_head20", 1, 256, 25, 20, 1, 1, 0, 1),
    ("1x1_mask3969", 1, 256, 25, 3969, 1, 1, 0, 1),      # mask head.3 (16 N tiles, last one ragged)
    ("3x3_v2", 2, 512, 15, 128, 3, 1, 1, 1),             # refine v2.0
    ("3x3_v22", 2, 128, 15, 32, 3, 1, 1, 1),             # refine v2.2 (N = 32)
    ("3x3_v0", 1, 64, 61, 16, 3, 1, 1, 1),               # refine v0.0 (N = 16)
    # resident-patch kernel (conv3x3_patch_sm100.cu): every (channels, size) pair the engine sends there
    ("3x3_p1_128_31", 3, 128, 31, 128, 3, 1, 1, 1),      # layer2.1-3 conv2 @255 (two k-blocks, PW 32, 4 rows per tile)
    ("3x3_p1_64_31", 2, 64, 31, 64, 3, 1, 1, 1),         # layer1 conv2 @127 (template)
    ("3x3_p1_128_15", 2, 128, 15, 128, 3, 1, 1, 1),      # layer2.1-3 conv2 @127 (PW 16, 8 rows per tile, ragged last tile)
    ("3x3_p1_64_63_b5", 5, 64, 63, 64, 3, 1, 1, 1),      # > 148 tiles: persistent CTAs take a second tile
]


def _case(c, seed=0):
    name, B, Cin, H, Cout, k, s, p, d = c
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, Cin, H, H, generator=g)
    w = torch.randn(Cout, Cin, k, k, generator=g) * (2.0 / (Cin * k * k)) ** 0.5
    scale = torch.rand(Cout, generator=g) + 0.5
    shift = torch.randn(Cout, generator=g)
    ref = F.conv2d(x, w, None, s, p, d) * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)
    return x, w, scale, shift, ref, (s, p, d)


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv_tensor_exact(case):
    x, w, scale, shift, ref, (s, p, d) = _case(case)
    out = smb.conv2d(x.cuda(), w, scale, shift, s, p, d, relu=False, backend="tensor", precision="exact")
    assert_close(out, ref, 2e-5, "tcgen05 exact " + case[0])
    out = smb.conv2d(x.cuda(), w, scale, shift, s, p, d, relu=True, backend="tensor", precision="exact")
    assert_close(out, ref.relu(), 2e-5, "tcgen05 exact+relu " + case[0])


@pytest.mark.parametrize("case", CONV_CASES[:8], ids=[c[0] for c in CONV_CASES[:8]])
def test_conv_tensor_fast(case):
    x, w, scale, shift, ref, (s, p, d) = _case(case, seed=1)
    out = smb.conv2d(x.cuda(), w, scale, shift, s, p, d, backend="tensor", precision="fast")
    assert_close(out, ref, 3e-3, "tcgen05 fast " + case[0])     # single fp16 pass: ~2^-11 per operand


@pytest.mark.parametrize("case", [CONV_CASES[0], CONV_CASES[3], CONV_CASES[4], CONV_CASES[6], CONV_CASES[10]],
                         ids=lambda c: c[0])
def test_conv_simt_reference(case):
    x, w, scale, shift, ref, (s, p, d) = _case(case, seed=2)
    out = smb.conv2d(x.cuda(), w, scale, shift, s, p, d, backend="simt", precision="exact")
    assert_close(out, ref, 2e-5, "simt " + case[0])


def test_conv_small_channels_simt_only():
    # Cin not a multiple of 64 has no tensor-core path: the operator must say so, not fall back silently
    x = torch.randn(1, 16, 9, 9).cuda()
    w = torch.randn(4, 16, 3, 3)
    with pytest.raises(RuntimeError):
        smb.conv2d(x, w, None, None, 1, 1, 1, backend="tensor")


# 256 / 150 planes @29: 8 resp. 4 whole tiles of the bulk-copy pipeline (+ a 22-plane remainder on the one-warp-per-plane
# kernel); 48 / 35 planes @45: 6 resp. 4 tiles of 8 (+3); the small ones never reach the bulk path
@pytest.mark.parametrize("shape", [(2, 8, 29, 29, 5), (1, 256, 29, 29, 5), (3, 50, 29, 29, 5), (3, 16, 45, 45, 5),
                                   (1, 35, 45, 45, 5), (2, 4, 12, 12, 3), (1, 3, 7, 7, 7)], ids=str)
def test_xcorr_depthwise_matches_oracle(shape):
    B, Cn, H, W, k = shape
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, Cn, H, W, generator=g)
    ker = torch.randn(B, Cn, k, k, generator=g)
    out = smb.conv2d_dw_group(x.cuda(), ker.cuda())
    assert_close(out, Oracle.xcorr_depthwise(x, ker), 2e-6, f"xcorr {shape}")
    loops = torch.from_numpy(xcorr_depthwise_loops(x.numpy(), ker.numpy())).float()
    assert_close(out, loops, 2e-6, f"xcorr {shape} vs loops")


def test_xcorr_misaligned_view_takes_the_fallback():
    """cp.async.bulk needs 16-byte aligned operands: a view that starts one 3364-byte plane into its storage is only
    4-byte aligned and must still give the right answer (one-warp-per-plane kernel)."""
    g = torch.Generator().manual_seed(6)
    xb = torch.randn(65, 1, 29, 29, generator=g).cuda()
    kb = torch.randn(65, 1, 5, 5, generator=g).cuda()
    x, ker = xb[1:], kb[1:]
    assert x.data_ptr() % 16 != 0 and x.is_contiguous()
    assert_close(smb.conv2d_dw_group(x, ker), Oracle.xcorr_depthwise(x.cpu(), ker.cpu()), 2e-6, "xcorr misaligned view")


def test_xcorr_golden_and_properties():
    g = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, "xcorr_small.npz")).items()}
    out = smb.conv2d_dw_group(g["x"].cuda(), g["k"].cuda())
    assert_close(out, g["out"], 2e-6, "xcorr vs reference golden")
    # size-independent properties at the benchmark size (B*C = 64*256 planes): linearity in x and in k
    gen = torch.Generator().manual_seed(9)
    x1 = torch.randn(64, 256, 29, 29, generator=gen).cuda()
    x2 = torch.randn(64, 256, 29, 29, generator=gen).cuda()
    k1 = torch.randn(64, 256, 5, 5, generator=gen).cuda()
    a = smb.conv2d_dw_group(x1 + 2 * x2, k1)
    b = smb.conv2d_dw_group(x1, k1) + 2 * smb.conv2d_dw_group(x2, k1)
    assert_close(a, b, 1e-5, "xcorr linearity @ 64x256 planes")
    # delta kernel picks a shifted window
    kd = torch.zeros(64, 256, 5, 5).cuda()
    kd[:, :, 1, 3] = 1.0
    assert torch.equal(smb.conv2d_dw_group(x1, kd), x1[:, :, 1:26, 3:28])
    with pytest.raises(RuntimeError):
        smb.conv2d_dw_group(x1[:1], k1)          # paired batches only, like the reference
