"""Post-processing on the GPU (fm_postprocess, fm_patchwise_segment, fm_op_gaussian3d): every comparison is BIT-EXACT
against scipy through oracle/postprocess_oracle.py."""
import ctypes

import numpy as np
import pytest

from oracle import postprocess_oracle as ppo
from oracle import unet_oracle as uo

pytestmark = pytest.mark.gpu

SHAPES = [(256, 256, 64), (96, 80, 40), (7, 5, 3), (1, 9, 2)]
SIGMAS = [0, 0.5, 1, 2]
FLAGS = [(True, True), (True, False), (False, True), (False, False)]


def device_gaussian(x, sigma):
    from fetal_net import _lib
    from fetal_net.device_postprocess import gaussian_weights
    w = gaussian_weights(sigma)
    out = np.empty_like(x)
    _lib.check(_lib.load().fm_op_gaussian3d(_lib.get_context().handle, x.ctypes.data_as(_lib.c_vp),
                                            0 if x.dtype == np.float32 else 1, _lib.i32ptr(_lib.i32x(x.shape)),
                                            (len(w) - 1) // 2, _lib.dptr(w), out.ctypes.data_as(_lib.c_vp)))
    return out


def raw_postprocess(pred, sigma=1, threshold=0.5, fill_holes=True, connected_component=True):
    """fm_postprocess through the C ABI: (uint8 mask, number of components, return code)."""
    from fetal_net import _lib
    from fetal_net.device_postprocess import _spec
    spec, _w = _spec(sigma, threshold, fill_holes, connected_component)
    mask = np.empty(pred.shape, np.uint8)
    n = _lib.c_i64(0)
    rc = _lib.load().fm_postprocess(_lib.get_context().handle, pred.ctypes.data_as(_lib.c_vp),
                                    0 if pred.dtype == np.float32 else 1, _lib.i32ptr(_lib.i32x(pred.shape)),
                                    ctypes.byref(spec), mask.ctypes.data_as(_lib.c_u8p), ctypes.byref(n))
    return mask, n.value, rc


def assert_same(pred, **kw):
    """device postprocess_prediction == oracle, including the ValueError of an empty component list."""
    from fetal_net.device_postprocess import postprocess_prediction
    try:
        ref = ppo.postprocess_prediction(pred, **kw)
    except ValueError:
        with pytest.raises(ValueError):
            postprocess_prediction(pred, **kw)
        return None
    got = postprocess_prediction(pred, **kw)
    assert got.dtype == np.bool_ and got.shape == ref.shape
    assert np.array_equal(got, ref), (pred.shape, pred.dtype, kw, int((got != ref).sum()))
    return got


def field(shape, seed=0):
    return np.random.default_rng(seed).random(shape)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", SHAPES)
def test_gaussian_bit_exact(shape, dtype, ctx):
    x = field(shape).astype(dtype)
    for s in SIGMAS:
        from scipy import ndimage
        ref = ndimage.gaussian_filter(x, s)
        got = device_gaussian(x, s)
        assert np.array_equal(got, ref), (shape, dtype, s, float(np.abs(got.astype(float) - ref).max()))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", SHAPES)
def test_postprocess_bit_exact(shape, dtype, ctx):
    x = field(shape, 1).astype(dtype)
    for s in SIGMAS:
        for fill, cc in FLAGS:
            assert_same(x, gaussian_std=s, threshold=0.5, fill_holes=fill, connected_component=cc)


def ball(shape, centre, radius):
    g = np.indices(shape).astype(np.float64)
    return sum((g[a] - centre[a]) ** 2 for a in range(3)) <= radius ** 2


def test_hollow_sphere_is_filled(ctx):
    shape = (40, 40, 40)
    shell = ball(shape, (20, 20, 20), 12) & ~ball(shape, (20, 20, 20), 9)
    got = assert_same(shell.astype(np.float64), gaussian_std=0)
    assert np.array_equal(got, ball(shape, (20, 20, 20), 12))


def test_cavity_open_to_the_border_is_not_filled(ctx):
    shape = (30, 30, 30)
    box = np.zeros(shape, bool)
    box[5:25, 5:25, 5:25] = True
    box[8:22, 8:22, 8:22] = False
    box[14:16, 14:16, 22:] = False         # tunnel from the cavity through the wall to the z border
    got = assert_same(box.astype(np.float32), gaussian_std=0)
    assert np.array_equal(got, box)


def test_diagonal_blobs_stay_separate(ctx):
    v = np.zeros((12, 12, 12), np.float64)
    v[1:4, 1:4, 1:4] = 1                   # 27 voxels
    v[4:8, 4:8, 4:8] = 1                   # 64 voxels, touches the first only at a corner
    v[8:10, 8:10, 4:8] = 1                 # 16 voxels, touches the second only along an edge
    mask, n, rc = raw_postprocess(v, sigma=0)
    assert rc == 0 and n == 3
    got = assert_same(v, gaussian_std=0)
    assert got.sum() == 64 and got[4:8, 4:8, 4:8].all()


def test_equal_largest_components_keep_the_raster_first(ctx):
    v = np.zeros((10, 10, 10), np.float64)
    v[6:9, 0:3, 0:3] = 1                   # later in x, earlier in z
    v[1:4, 6:9, 6:9] = 1                   # first voxel (1, 6, 6) comes first in C order
    got = assert_same(v, gaussian_std=0)
    assert got[1:4, 6:9, 6:9].all() and got.sum() == 27


def test_values_exactly_at_the_threshold(ctx):
    rng = np.random.default_rng(4)
    for dtype, thr in [(np.float64, 0.5), (np.float32, 0.5), (np.float32, 0.1), (np.float64, 0.1)]:
        t = dtype(thr)
        v = rng.choice(np.array([np.nextafter(t, dtype(0)), t, np.nextafter(t, dtype(1))], dtype), (20, 18, 16))
        for fill, cc in FLAGS:
            assert_same(v, gaussian_std=0, threshold=thr, fill_holes=fill, connected_component=cc)


def test_empty_and_full_foreground(ctx):
    from fetal_net.device_postprocess import postprocess_prediction
    empty = np.zeros((16, 12, 8))
    with pytest.raises(ValueError):
        postprocess_prediction(empty)
    assert not postprocess_prediction(empty, connected_component=False).any()
    full = np.ones((16, 12, 8), np.float32)
    for fill, cc in FLAGS:
        assert postprocess_prediction(full, fill_holes=fill, connected_component=cc).all()
    assert raw_postprocess(full)[1:] == (1, 0)


def test_checkerboard_every_voxel_its_own_component(ctx):
    from scipy import ndimage
    shape = (64, 48, 32)
    v = (np.indices(shape).sum(axis=0) % 2 == 0).astype(np.float64)
    mask, n, rc = raw_postprocess(v, sigma=0, fill_holes=False)
    assert rc == 0 and n == ndimage.label(v > 0.5)[1] == v.size // 2
    for fill, cc in FLAGS:
        assert_same(v, gaussian_std=0, fill_holes=fill, connected_component=cc)


def test_serpentine_deep_union_chains(ctx):
    """One path that winds through the whole volume: unions chain over hundreds of thousands of voxels."""
    X, Y, Z = 48, 64, 64
    v = np.zeros((X, Y, Z), np.float64)
    for x in range(0, X, 2):
        v[x, 0::2, :] = 1                                   # rows along z
        for y in range(1, Y - 1, 2):
            v[x, y, Z - 1 if (y // 2) % 2 == 0 else 0] = 1  # alternate row ends
        if x + 1 < X:
            v[x + 1, 0 if (x // 2) % 2 else Y - 2, 0 if (x // 2) % 2 else Z - 1] = 1   # hop to the next slice
    comb = np.zeros((X, Y, Z), np.float64)                  # a comb: one spine, teeth along z
    comb[:, 0, :] = 1
    comb[::2, :, 0] = 1
    for arr in (v, comb):
        for fill, cc in FLAGS:
            assert_same(arr, gaussian_std=0, fill_holes=fill, connected_component=cc)


def test_two_runs_identical(ctx):
    from fetal_net.device_postprocess import postprocess_prediction
    x = field((256, 256, 64), 5)
    a = postprocess_prediction(x, gaussian_std=0, fill_holes=True, connected_component=True)
    b = postprocess_prediction(x, gaussian_std=0, fill_holes=True, connected_component=True)
    assert np.array_equal(a, b)
    ma, na, _ = raw_postprocess(x, sigma=1)
    mb, nb, _ = raw_postprocess(x, sigma=1)
    assert na == nb and np.array_equal(ma, mb)


def test_volume_over_int32_voxels_refused(ctx):
    from fetal_net import _lib
    from fetal_net.device_postprocess import _spec, postprocess_prediction
    spec, _w = _spec(1, 0.5, True, True)
    dummy = np.zeros(8, np.float64)
    mask = np.zeros(8, np.uint8)
    rc = _lib.load().fm_postprocess(ctx.handle, dummy.ctypes.data_as(_lib.c_vp), 1,
                                    _lib.i32ptr(_lib.i32x((2048, 1024, 1024))), ctypes.byref(spec),
                                    mask.ctypes.data_as(_lib.c_u8p), None)
    assert rc == -1                       # FM_EINVAL, before anything is read
    with pytest.raises(ValueError):
        postprocess_prediction(np.broadcast_to(np.float32(0), (2048, 1024, 1024)))


# ---- patch_wise_segmentation ---------------------------------------------------------------------

def check_segmentation(model, vol, patch, overlap, batch, **kw):
    """fm_patchwise_segment == oracle(patch_wise_prediction(...).squeeze()), its map == patch_wise_prediction's."""
    from fetal_net.device_postprocess import patch_wise_segmentation
    from fetal_net.prediction import patch_wise_prediction
    prob = patch_wise_prediction(model, vol, patch, overlap_factor=overlap, batch_size=batch, **kw)
    thr = float(np.median(prob))          # a decisive threshold for whatever the network predicts
    for fill, cc in FLAGS:
        pp = dict(threshold=thr, fill_holes=fill, connected_component=cc)
        ref = ppo.postprocess_prediction(prob.squeeze(), **pp)
        mask, p2 = patch_wise_segmentation(model, vol, patch, overlap_factor=overlap, batch_size=batch,
                                           return_prediction=True, **kw, **pp)
        assert np.array_equal(p2, prob)
        assert mask.dtype == np.bool_ and np.array_equal(mask, ref), (fill, cc, int((mask != ref).sum()))
        assert np.array_equal(patch_wise_segmentation(model, vol, patch, overlap_factor=overlap, batch_size=batch,
                                                      **kw, **pp), ref)
    return prob


@pytest.fixture(scope="module")
def native64():
    from fetal_net.model import unet_model_3d
    from tests.test_gpu_model import decisive_weights
    m = unet_model_3d(input_shape=(1, 64, 64, 64), n_base_filters=16, depth=4)
    m.set_named_weights(decisive_weights(uo.unet3d_layers(4, 16), seed=3))
    return m


def test_segmentation_configs0_geometry(native64):
    vol = np.random.default_rng(0).standard_normal((1, 256, 256, 64)).astype(np.float32)
    check_segmentation(native64, vol, (64, 64, 64), 0.5, 49)


def test_segmentation_volume_smaller_than_patch(native64):
    """pad_for_fit on every axis: the crop of the padded map precedes the filter."""
    vol = np.random.default_rng(1).standard_normal((1, 50, 41, 60)).astype(np.float32)
    check_segmentation(native64, vol, (64, 64, 64), 0.5, 5)


def test_segmentation_2d_model_with_truth():
    from fetal_net.model import unet_model_2d
    layers = uo.unet2d_layers(4, 32, 6)
    w = uo.glorot_uniform_weights(layers, seed=4, ndim=2)
    rng = np.random.default_rng(5)
    for k in w:
        w[k] = (w[k] * np.sqrt(2.0) * 1.15).astype(np.float32) if k.endswith("/kernel") else \
            (0.05 * rng.standard_normal(w[k].shape)).astype(np.float32)
    model = unet_model_2d(input_shape=(32, 32, 6), n_base_filters=32, depth=4)
    model.set_named_weights(w)
    vol = rng.standard_normal((1, 48, 32, 10)).astype(np.float32)
    truth = (rng.random(vol.shape) < 0.4).astype(np.float32)
    check_segmentation(model, vol, (32, 32, 5), 0.5, 7, truth_data=truth, prev_truth_index=1, prev_truth_size=1)


def test_segmentation_generic_model_route(ctx):
    """A non-native model goes through patch_wise_prediction + the device postprocess_prediction."""
    from oracle.ref_harness import FunctionModel
    from tests.golden.make_golden import ramp_model
    fn, oshape = ramp_model((8, 8, 8), 1)
    vol = np.random.default_rng(6).standard_normal((1, 20, 16, 12)).astype(np.float32)
    check_segmentation(FunctionModel(fn, oshape), vol, (8, 8, 8), 0.5, 4)
