"""Per-kernel parity on the GPU, through the C ABI (see tests/gpu_cases.py for the stated tolerance)."""
import numpy as np
import pytest

from tests import gpu_cases as gc

pytestmark = pytest.mark.gpu

IDS = [c[0] for c in gc.CONV_CASES]
SINGLE = [c for c in gc.CONV_CASES if c[6] == 0 and c[8] == 3]


@pytest.mark.parametrize("case", gc.CONV_CASES, ids=IDS)
def test_conv3d_fprop_tcgen05(ctx, case):
    ok, worst = gc.conv_fprop_case(ctx, 0, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", gc.CONV_CASES[:9], ids=IDS[:9])
def test_conv3d_fprop_simt(ctx, case):
    ok, worst = gc.conv_fprop_case(ctx, 1, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_conv3d_dgrad_tcgen05(ctx, case):
    ok, worst = gc.conv_dgrad_case(ctx, 0, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_conv3d_wgrad_tcgen05(ctx, case):
    ok, worst = gc.conv_wgrad_case(ctx, 0, case)
    assert ok, "rel. error / 2e-3 = %.3f" % worst


@pytest.mark.parametrize("case", SINGLE[:5], ids=[c[0] for c in SINGLE[:5]])
def test_conv3d_wgrad_simt(ctx, case):
    ok, worst = gc.conv_wgrad_case(ctx, 1, case)
    assert ok, "rel. error / 2e-3 = %.3f" % worst


MIDS = [c[0] for c in gc.MARCH_CASES]
MSINGLE = [c for c in gc.MARCH_CASES if c[6] == 0]


@pytest.mark.parametrize("impl", [2, 3], ids=["reproducible", "shared-acc"])
@pytest.mark.parametrize("case", gc.MARCH_CASES, ids=MIDS)
def test_conv3d_fprop_march(ctx, case, impl):
    ok, worst = gc.conv_fprop_case(ctx, impl, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", [gc.MARCH_CASES[1], gc.MARCH_CASES[4], gc.MARCH_CASES[7]],
                         ids=[gc.MARCH_CASES[i][0] for i in (1, 4, 7)])
def test_conv3d_march_bit_reproducible(ctx, case):
    """impl 2 is the kernel behind predict / evaluate / patch_wise_prediction: three issuing warps take turns plane by
    plane under a token, so the fp32 summation order is fixed - the output must be identical run to run."""
    first = gc.conv_fprop_raw(ctx, 2, case)
    for _ in range(4):
        assert np.array_equal(gc.conv_fprop_raw(ctx, 2, case), first)


@pytest.mark.parametrize("case", MSINGLE, ids=[c[0] for c in MSINGLE])
def test_conv3d_dgrad_march(ctx, case):
    # dgrad runs the marching kernel with Cout input channels and C1 output channels
    if case[7] > 64 or case[5] > 64:
        pytest.skip("filter bank not resident")
    for impl in (2, 3):
        ok, worst = gc.conv_dgrad_case(ctx, impl, case)
        assert ok, "impl %d: worst error / tolerance = %.3f" % (impl, worst)


@pytest.mark.parametrize("case", gc.WGRAD_MARCH_CASES, ids=[c[0] for c in gc.WGRAD_MARCH_CASES])
def test_conv3d_wgrad_march(ctx, case):
    ok, worst = gc.conv_wgrad_case(ctx, 2, case)
    assert ok, "rel. error / 2e-3 = %.3f" % worst


@pytest.mark.parametrize("case", gc.UP_CASES, ids=[c[0] for c in gc.UP_CASES])
def test_conv3d_up_fprop(ctx, case):
    """Decoder conv over concatenate([UpSampling3D(coarse), skip]) computed at coarse resolution == the conv over the
    materialised upsampled tensor (torch fp64)."""
    ok, worst = gc.conv_up_fprop_case(ctx, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", gc.UP_CASES, ids=[c[0] for c in gc.UP_CASES])
def test_conv3d_up_bwd(ctx, case):
    ok, worst = gc.conv_up_bwd_case(ctx, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", gc.FIRST_CASES, ids=[c[0] for c in gc.FIRST_CASES])
def test_conv3d_first_layer(ctx, case):
    ok, worst = gc.conv_first_case(ctx, case)
    assert ok, "worst error / tolerance = %.3f" % worst


def test_maxpool3d_fwd_bwd(ctx):
    ok, worst = gc.maxpool_case(ctx)
    assert ok, worst


def test_upsample3d_fwd_bwd(ctx):
    ok, worst = gc.upsample_case(ctx)
    assert ok, worst


def test_dice_sums_and_gradient(ctx):
    ok, worst = gc.dice_case(ctx)
    assert ok, worst


@pytest.mark.parametrize("with_mask", [False, True])
def test_dice_and_xent_sums_and_gradient(ctx, with_mask):
    ok, worst = gc.dice_xent_case(ctx, with_mask)
    assert ok, worst


def test_keras_adam(ctx):
    ok, worst = gc.adam_case(ctx)
    assert ok, worst

