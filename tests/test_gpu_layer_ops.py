"""Per-kernel parity of the layers the Isensee, batch-normalised, deconvolution and 2D models add, one op at a time
through the C ABI against float64 references (bounds and case helpers: tests/gpu_cases.py).

- bf16 outputs (y, dx): close_bf16 per element (its max|ref| term per channel where channels differ in scale);
- fp32 reductions (dgamma, dbeta, db, head sums and weights, norm and moving statistics): |got - ref| <= 1e-5 * sum|term|
  per channel;
- conv / deconv weight gradients (bf16 products): whole-tensor relative error <= 2e-3;
- data movement (zero insertion, depth <-> space without bias, seg_upsample_add, sumpool_f32): exact.
"""
import pytest

from tests import gpu_cases as gc

pytestmark = pytest.mark.gpu


def ids(cases):
    return [c[0] for c in cases]


NORM_ALL = gc.NORM_CASES + [gc.NORM_BIG]
NORM_BWD = [c for c in NORM_ALL if c[2] > 1]   # one voxel: zero variance, the float64 reference has no gradient there


# ---- instance norm + LeakyReLU: fm_op_instnorm_lrelu, fm_op_instnorm_lrelu_bwd ----------------------------------
@pytest.mark.parametrize("with_add,with_scale", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["plain", "add", "dropout", "add+dropout"])
@pytest.mark.parametrize("case", gc.NORM_CASES, ids=ids(gc.NORM_CASES))
def test_instnorm_lrelu_fwd(ctx, case, with_add, with_scale):
    ok, worst = gc.instnorm_fwd_case(ctx, case, with_add, with_scale)
    assert ok, "worst error / tolerance = %.3f" % worst


def test_instnorm_lrelu_fwd_cfg3_level0(ctx):
    ok, worst = gc.instnorm_fwd_case(ctx, gc.NORM_BIG, True, False)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("with_gy2,with_scale", [(False, False), (True, False), (False, True)],
                         ids=["gy", "gy+gy2", "dropout"])
@pytest.mark.parametrize("case", NORM_BWD, ids=ids(NORM_BWD))
def test_instnorm_lrelu_bwd(ctx, case, with_gy2, with_scale):
    ok, worst = gc.instnorm_bwd_case(ctx, case, with_gy2, with_scale)
    assert ok, "worst error / tolerance = %.3f" % worst


# ---- batch norm + ReLU: fm_op_batchnorm_relu, fm_op_batchnorm_relu_bwd ------------------------------------------
@pytest.mark.parametrize("training", [True, False], ids=["training", "inference"])
@pytest.mark.parametrize("case", NORM_ALL, ids=ids(NORM_ALL))
def test_batchnorm_relu_fwd(ctx, case, training):
    ok, worst = gc.batchnorm_fwd_case(ctx, case, training)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("with_gy2", [False, True], ids=["gy", "gy+gy2"])
@pytest.mark.parametrize("case", NORM_ALL, ids=ids(NORM_ALL))
def test_batchnorm_relu_bwd(ctx, case, with_gy2):
    ok, worst = gc.batchnorm_bwd_case(ctx, case, with_gy2)
    assert ok, "worst error / tolerance = %.3f" % worst


# ---- stride-2 in-convs: fprop, zero insertion, stride-1 dgrad / wgrad: fm_op_conv_strided, fm_op_zero_insert -----
@pytest.mark.parametrize("case", gc.STRIDED_CASES, ids=ids(gc.STRIDED_CASES))
def test_conv_strided_fwd_bwd(ctx, case):
    ok, worst = gc.conv_strided_case(ctx, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("shape,pz", [((2, 3, 5, 2, 16), 2), ((1, 4, 4, 4, 64), 2), ((2, 5, 3, 1, 32), 1)],
                         ids=["3d_ragged", "3d_c64", "2d"])
def test_zero_insert(ctx, shape, pz):
    assert gc.zero_insert_case(ctx, shape, pz)


# ---- deconvolution: 1x1x1 conv + depth_to_space, and back: fm_op_deconv, fm_op_depth_space ----------------------
@pytest.mark.parametrize("relu_mask", [1, 0], ids=["unet", "unet_bn"])
@pytest.mark.parametrize("case", gc.DECONV_CASES, ids=ids(gc.DECONV_CASES))
def test_deconv_fwd_bwd(ctx, case, relu_mask):
    ok, worst = gc.deconv_case(ctx, case, relu_mask)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("shape,pz", [((2, 3, 5, 2, 16), 2), ((1, 2, 2, 2, 256), 2), ((2, 5, 3, 1, 128), 1)],
                         ids=["3d_ragged", "3d_c256", "2d_c128"])
def test_depth_space_shuffles(ctx, shape, pz):
    assert gc.depth_space_case(ctx, shape, pz)


# ---- the 2D family, kernel code 31 on Z = 1: fm_op_conv3d_fprop, fm_op_conv_dgrad, fm_op_conv_wgrad; pz = 1:
#      fm_op_maxpool(_bwd), fm_op_upsample(_bwd) -------------------------------------------------------------------------------------
C2D_SINGLE = [c for c in gc.CONV2D_CASES if c[6] == 0]


@pytest.mark.parametrize("impl", [0, 1], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("case", gc.CONV2D_CASES, ids=ids(gc.CONV2D_CASES))
def test_conv2d_fprop(ctx, case, impl):
    ok, worst = gc.conv_fprop_case(ctx, impl, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("impl", [0, 1], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("case", C2D_SINGLE, ids=ids(C2D_SINGLE))
def test_conv2d_dgrad(ctx, case, impl):
    ok, worst = gc.conv_dgrad_case(ctx, impl, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("impl", [0, 1], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("case", C2D_SINGLE, ids=ids(C2D_SINGLE))
def test_conv2d_wgrad(ctx, case, impl):
    ok, worst = gc.conv_wgrad_case(ctx, impl, case)
    assert ok, "rel. error / 2e-3 = %.3f" % worst


@pytest.mark.parametrize("shape", [(2, 8, 12, 1, 32), (1, 6, 10, 1, 256)], ids=["c32", "c256"])
def test_maxpool2d_fwd_bwd(ctx, shape):
    ok, worst = gc.maxpool_case(ctx, shape=shape, pz=1)
    assert ok, worst


@pytest.mark.parametrize("shape", [(2, 4, 6, 1, 64), (1, 3, 5, 1, 128)], ids=["c64", "c128"])
def test_upsample2d_fwd_bwd(ctx, shape):
    ok, worst = gc.upsample_case(ctx, shape=shape, pz=1)
    assert ok, worst


# ---- existing conv cases without the ReLU (the Isensee and batch-norm blocks call the same kernels with relu = 0) ------
@pytest.mark.parametrize("case", gc.CONV_CASES, ids=ids(gc.CONV_CASES))
def test_conv3d_fprop_tcgen05_no_relu(ctx, case):
    ok, worst = gc.conv_fprop_case(ctx, 0, case, relu=0)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", gc.CONV_CASES[:9], ids=ids(gc.CONV_CASES[:9]))
def test_conv3d_fprop_simt_no_relu(ctx, case):
    ok, worst = gc.conv_fprop_case(ctx, 1, case, relu=0)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("impl", [2, 3], ids=["reproducible", "shared-acc"])
@pytest.mark.parametrize("case", gc.MARCH_CASES, ids=ids(gc.MARCH_CASES))
def test_conv3d_fprop_march_no_relu(ctx, case, impl):
    ok, worst = gc.conv_fprop_case(ctx, impl, case, relu=0)
    assert ok, "worst error / tolerance = %.3f" % worst


# ---- 1x1x1 heads: fm_op_head (k_head_fwd, k_head_fwd_dice, k_head_bwd) ------------------------------------------
@pytest.mark.parametrize("sigmoid", [1, 0], ids=["sigmoid", "logit"])
@pytest.mark.parametrize("case", gc.HEAD_CASES, ids=ids(gc.HEAD_CASES))
def test_head_fwd(ctx, case, sigmoid):
    ok, worst = gc.head_fwd_case(ctx, case, sigmoid)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", gc.HEAD_CASES, ids=ids(gc.HEAD_CASES))
def test_head_fwd_dice(ctx, case):
    ok, worst = gc.head_fwd_dice_case(ctx, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("mode", [0, 1, 2], ids=["relu_mask", "plain", "accumulate"])
@pytest.mark.parametrize("case", gc.HEAD_CASES, ids=ids(gc.HEAD_CASES))
def test_head_bwd(ctx, case, mode):
    ok, worst = gc.head_bwd_case(ctx, case, mode)
    assert ok, "worst error / tolerance = %.3f" % worst


# ---- deep-supervision plumbing: fm_op_seg_upsample_add, fm_op_sumpool_f32 ---------------------------------------
@pytest.mark.parametrize("shape,pz", [((2, 8, 6, 4), 2), ((1, 16, 16, 16), 2), ((2, 10, 6, 1), 1)],
                         ids=["3d", "3d_cube", "2d"])
def test_seg_upsample_add(ctx, shape, pz):
    assert gc.seg_upsample_add_case(ctx, shape, pz)


@pytest.mark.parametrize("shape,pz", [((2, 4, 3, 2), 2), ((1, 8, 8, 8), 2), ((2, 5, 3, 1), 1)],
                         ids=["3d", "3d_cube", "2d"])
def test_sumpool_f32(ctx, shape, pz):
    assert gc.sumpool_case(ctx, shape, pz)
