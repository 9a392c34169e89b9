"""Shared convolution cases.  Names follow the reference's own tests
(src/caffe/test/test_convolution_layer.cpp) and the BASELINE.json configs (SURVEY Appendix A)."""
import hashlib
import os


# (name, dict(N, Cin, H, W, O, k, s, p, d, G, bias))
REF_TEST_CASES = [
    ("TestSimpleConvolution", dict(N=2, Cin=3, H=6, W=4, O=4, k=3, s=2, p=0, d=1, G=1, bias=True)),     # :228
    ("TestDilatedConvolution", dict(N=2, Cin=3, H=17, W=13, O=4, k=3, s=1, p=0, d=2, G=1, bias=True)),   # :266 (shape 2x3x17x13? kept small)
    ("Test1x1Convolution", dict(N=2, Cin=3, H=6, W=4, O=4, k=1, s=1, p=0, d=1, G=1, bias=True)),        # :452
    ("TestSimpleConvolutionGroup", dict(N=2, Cin=6, H=6, W=4, O=3, k=3, s=2, p=0, d=1, G=3, bias=True)), # :481
    ("TestGradient", dict(N=2, Cin=3, H=6, W=4, O=2, k=3, s=2, p=0, d=1, G=1, bias=True)),              # :730
    ("TestGradientGroup", dict(N=2, Cin=6, H=6, W=4, O=3, k=3, s=2, p=0, d=1, G=3, bias=True)),         # :826
]

# edge cases: ragged windows (truncating division), rectangular kernels/strides/pads, pad > kernel/2,
# single pixel outputs, batch 1, stride > kernel
EDGE_CASES = [
    ("ragged_trunc", dict(N=1, Cin=2, H=8, W=9, O=3, k=3, s=2, p=0, d=1, G=1, bias=False)),
    ("rect_kernel", dict(N=2, Cin=4, H=9, W=11, O=5, k=(3, 5), s=(2, 1), p=(1, 2), d=(1, 1), G=1, bias=True)),
    ("big_pad", dict(N=1, Cin=3, H=5, W=5, O=2, k=3, s=1, p=3, d=1, G=1, bias=True)),
    ("one_pixel_out", dict(N=3, Cin=5, H=3, W=3, O=7, k=3, s=1, p=0, d=1, G=1, bias=True)),
    ("stride_gt_kernel", dict(N=2, Cin=3, H=10, W=10, O=4, k=2, s=3, p=0, d=1, G=1, bias=False)),
    ("dil_rect", dict(N=1, Cin=2, H=12, W=10, O=3, k=3, s=(1, 2), p=(2, 1), d=(2, 3), G=1, bias=True)),
    ("g2_5x5", dict(N=2, Cin=8, H=9, W=9, O=6, k=5, s=1, p=2, d=1, G=2, bias=True)),
    ("1x1_s2", dict(N=2, Cin=16, H=8, W=8, O=8, k=1, s=2, p=0, d=1, G=1, bias=False)),
    ("k7_s2_p3", dict(N=1, Cin=3, H=20, W=20, O=8, k=7, s=2, p=3, d=1, G=1, bias=False)),
    ("k11_s4", dict(N=1, Cin=3, H=35, W=35, O=6, k=11, s=4, p=0, d=1, G=1, bias=True)),
]

# scaled-down layers of the BASELINE configs (same k/s/p/g structure, N small so the oracle is fast)
MODEL_CASES = [
    ("lenet_conv1", dict(N=4, Cin=1, H=28, W=28, O=20, k=5, s=1, p=0, d=1, G=1, bias=True)),
    ("lenet_conv2", dict(N=4, Cin=20, H=12, W=12, O=50, k=5, s=1, p=0, d=1, G=1, bias=True)),
    ("alexnet_conv2_g2", dict(N=2, Cin=96, H=27, W=27, O=256, k=5, s=1, p=2, d=1, G=2, bias=True)),
    ("alexnet_conv4_g2", dict(N=2, Cin=384, H=13, W=13, O=384, k=3, s=1, p=1, d=1, G=2, bias=True)),
    ("resnet_stem", dict(N=2, Cin=3, H=64, W=64, O=64, k=7, s=2, p=3, d=1, G=1, bias=False)),
    ("resnet_res2_3x3", dict(N=2, Cin=64, H=56, W=56, O=64, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet_res2_1x1_expand", dict(N=2, Cin=64, H=56, W=56, O=256, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("resnet_res3_1x1_s2", dict(N=2, Cin=256, H=56, W=56, O=128, k=1, s=2, p=0, d=1, G=1, bias=False)),
    ("resnet_res4_3x3", dict(N=2, Cin=256, H=14, W=14, O=256, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet_res5_3x3", dict(N=3, Cin=512, H=7, W=7, O=512, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet_res5_1x1", dict(N=3, Cin=512, H=7, W=7, O=2048, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("vgg_conv1_1", dict(N=1, Cin=3, H=64, W=64, O=64, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("googlenet_5x5", dict(N=2, Cin=16, H=28, W=28, O=32, k=5, s=1, p=2, d=1, G=1, bias=True)),
    ("googlenet_aux_4x4", dict(N=4, Cin=512, H=4, W=4, O=128, k=1, s=1, p=0, d=1, G=1, bias=True)),
    # 1x1 / stride 1 layers whose H*W is a multiple of 4: the TMA-fed weight-gradient kernel (zero-filled K tail at
    # 14x14 = 196, ragged O and C against the 128 x N_TILE tile, split-K with several CTAs per tile, bias)
    ("resnet_res4_1x1_expand", dict(N=8, Cin=256, H=14, W=14, O=1024, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("resnet_res4_1x1_reduce", dict(N=2, Cin=1024, H=14, W=14, O=256, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("ragged_1x1_14", dict(N=3, Cin=96, H=14, W=14, O=72, k=1, s=1, p=0, d=1, G=1, bias=True)),
    ("ragged_1x1_rect", dict(N=2, Cin=40, H=6, W=10, O=200, k=1, s=1, p=0, d=1, G=1, bias=True)),
    ("resnet_res3_1x1_reduce", dict(N=2, Cin=512, H=28, W=28, O=128, k=1, s=1, p=0, d=1, G=1, bias=False)),
]

# 3x3 / stride 1 / pad 1 with C % 32 == 0 and H*W % 4 == 0, ragged against the 128-pixel tile and the image borders:
# the shapes the bulk-copy-staged forward / dgrad kernel (conv_tc_stg.cu) takes, next to the ResNet ones above
MODEL_CASES += [
    ("resnet_res3_3x3", dict(N=2, Cin=128, H=28, W=28, O=128, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("ragged_3x3_rect", dict(N=3, Cin=32, H=12, W=20, O=40, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("staged_5x5_c32", dict(N=5, Cin=32, H=10, W=14, O=48, k=5, s=1, p=2, d=1, G=1, bias=True)),         # 140-pixel images: most tiles span two
    ("staged_1x1_small_maps", dict(N=7, Cin=96, H=12, W=11, O=160, k=1, s=1, p=0, d=1, G=1, bias=True)), # 132-pixel images, ragged O
    ("staged_3x3_c96_odd_halfblocks", dict(N=2, Cin=96, H=8, W=16, O=64, k=3, s=1, p=1, d=1, G=1, bias=False)),   # 27 half blocks: K padding
    ("staged_rect_1x3", dict(N=2, Cin=64, H=12, W=12, O=32, k=(1, 3), s=1, p=(0, 1), d=1, G=1, bias=True)),
    ("gather_1x1_tiny_maps", dict(N=37, Cin=96, H=4, W=4, O=160, k=1, s=1, p=0, d=1, G=1, bias=True)),   # H*W < 128: stays on the gather kernel
    # staged weight gradient: a map wide enough that only ONE X stage fits (W = 80), and an odd width (unaligned tap windows)
    ("wstg_wide_3x3", dict(N=2, Cin=32, H=8, W=80, O=32, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("wstg_oddw_3x3", dict(N=5, Cin=32, H=8, W=13, O=40, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("strided_1x1_to_7x7", dict(N=5, Cin=64, H=14, W=14, O=96, k=1, s=2, p=0, d=1, G=1, bias=False)),   # wgrad: subsample, then plane mode
    # 7x7 maps: the staged kernel's plane mode (whole image planes staged, up to 4 images per 128-row tile)
    ("plane_3x3_7x7", dict(N=9, Cin=64, H=7, W=7, O=72, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("plane_1x1_7x7", dict(N=11, Cin=96, H=7, W=7, O=160, k=1, s=1, p=0, d=1, G=1, bias=True)),
    ("plane_5x5_7x7", dict(N=6, Cin=32, H=7, W=7, O=128, k=5, s=1, p=2, d=1, G=1, bias=True)),
]

ALL_CASES = REF_TEST_CASES + EDGE_CASES + MODEL_CASES


def make(mod, c):
    """Build mod.ConvParams (oracle's or capi's) from a case dict."""
    return mod.ConvParams.make(c["N"], c["Cin"], c["H"], c["W"], c["O"], c["k"], c["s"], c["p"], c["d"], c["G"], c["bias"])


def tensors(rng, prm, scale_w=None):
    import numpy as np
    x = rng.standard_normal(prm.x_shape()).astype(np.float32)
    fan_in = prm.Kd
    w = (rng.standard_normal(prm.w_shape()) * (scale_w if scale_w else (2.0 / fan_in) ** 0.5)).astype(np.float32)
    b = (rng.standard_normal((prm.O,)) * 0.1).astype(np.float32) if prm.has_bias else None
    dy = rng.standard_normal(prm.y_shape()).astype(np.float32)
    return x, w, b, dy


def rel_err(a, ref):
    """max|a-ref| / max|ref| -- the blob-level relative error the 1e-3 bar is stated in (DESIGN.md)."""
    import numpy as np
    den = float(np.abs(ref).max())
    return float(np.abs(a.astype(np.float64) - ref.astype(np.float64)).max()) / (den if den > 0 else 1.0)


# BASELINE.json configurations at FULL size (the batch sizes the benchmark runs): the persistent multi-tile path of the
# forward / dgrad kernel (several tiles per CTA, accumulator ping-pong, mbarrier phase wrap) and the N-dependent split-K
# plans of the weight-gradient kernels.  Checked against what the reference's im2col + OpenBLAS loop (oracle.ref_conv_fwd_bwd)
# computed for them (tests/golden/full_size_ref_golden.npz).  Mirrors test_convolution_layer.cpp:228-264,481-509 at benchmark scale.
FULL_SIZE_CASES = [
    ("resnet50_res2_1x1_expand_n64", dict(N=64, Cin=64, H=56, W=56, O=256, k=1, s=1, p=0, d=1, G=1, bias=False)),   # 3136 tiles
    ("resnet50_res2_1x1_reduce_n64", dict(N=64, Cin=256, H=56, W=56, O=64, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("resnet50_res2_3x3_n64", dict(N=64, Cin=64, H=56, W=56, O=64, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet50_res3_3x3_n64", dict(N=64, Cin=128, H=28, W=28, O=128, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet50_res4_3x3_n64", dict(N=64, Cin=256, H=14, W=14, O=256, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet50_res4_1x1_expand_n64", dict(N=64, Cin=256, H=14, W=14, O=1024, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("resnet50_res5_3x3_n64", dict(N=64, Cin=512, H=7, W=7, O=512, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("resnet50_res5_1x1_reduce_n64", dict(N=64, Cin=2048, H=7, W=7, O=512, k=1, s=1, p=0, d=1, G=1, bias=False)),
    ("resnet50_res3_1x1_s2_n64", dict(N=64, Cin=256, H=56, W=56, O=512, k=1, s=2, p=0, d=1, G=1, bias=False)),
    ("resnet50_stem_7x7_n64", dict(N=64, Cin=3, H=224, W=224, O=64, k=7, s=2, p=3, d=1, G=1, bias=False)),
    ("alexnet_conv2_g2_n256", dict(N=256, Cin=96, H=27, W=27, O=256, k=5, s=1, p=2, d=1, G=2, bias=True)),
    ("alexnet_conv3_n256", dict(N=256, Cin=256, H=13, W=13, O=384, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("vgg16_conv1_2_n32", dict(N=32, Cin=64, H=224, W=224, O=64, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("vgg16_conv5_n32", dict(N=32, Cin=512, H=14, W=14, O=512, k=3, s=1, p=1, d=1, G=1, bias=True)),
    ("googlenet_3a_5x5_n128", dict(N=128, Cin=16, H=28, W=28, O=32, k=5, s=1, p=2, d=1, G=1, bias=True)),
    ("googlenet_3a_3x3_n128", dict(N=128, Cin=96, H=28, W=28, O=128, k=3, s=1, p=1, d=1, G=1, bias=True)),
]


def full_size_inputs(rng, prm):
    """x, w, b, dy and the pre-existing weight diff dw0 (accumulated into) of a FULL_SIZE_CASES layer, in draw order."""
    import numpy as np
    x = rng.standard_normal(prm.x_shape(), dtype=np.float32)
    w = rng.standard_normal(prm.w_shape(), dtype=np.float32) * np.float32((2.0 / prm.Kd) ** 0.5)
    b = (rng.standard_normal(prm.O, dtype=np.float32) * np.float32(0.1)) if prm.has_bias else None
    dy = rng.standard_normal(prm.y_shape(), dtype=np.float32)
    dw0 = rng.standard_normal(prm.w_shape(), dtype=np.float32) * np.float32(0.1)
    return x, w, b, dy, dw0


def sample_index(n, k=512):
    """The fixed positions (seeded, repeats allowed) at which tests/golden/full_size_ref_golden.npz keeps an output of n
    elements: the full outputs (up to 400 MB each) are too large to store."""
    import numpy as np
    return np.random.default_rng(1701).integers(0, n, k)


# im2col / col2im shapes (C, H, W, k, s, p, d) compared bit for bit with the reference's im2col.cpp; the first row is
# test_im2col_kernel.cu's 500x15x15, k3 s2 d3 p0 (test_im2col_kernel.cu:102-212)
REF_IM2COL_SHAPES = [
    (500, 15, 15, (3, 3), (2, 2), (0, 0), (3, 3)),
    (3, 6, 5, (3, 3), (2, 2), (0, 0), (1, 1)),
    (4, 9, 11, (3, 5), (2, 1), (1, 2), (1, 1)),
    (2, 12, 10, (3, 3), (1, 2), (2, 1), (2, 3)),
    (3, 20, 20, (7, 7), (2, 2), (3, 3), (1, 1)),
    (1, 5, 5, (3, 3), (1, 1), (3, 3), (1, 1)),
]


def digest(a):
    """sha256 of an array's float32 bytes: how tests/golden/im2col_ref_digests.json records outputs that must match bit for bit."""
    import numpy as np
    return hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest()
