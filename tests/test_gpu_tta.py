"""Flip test-time augmentation on the GPU (fm_patchwise_predict_flips, fm_op_median_passes, fetal_net.device_tta): every
comparison is BIT-EXACT against the host composition - a host loop of np.flip -> patch_wise_prediction -> np.flip,
np.median over its stack, and scipy post-processing through oracle/postprocess_oracle.py."""
import ctypes
import warnings

import numpy as np
import pytest

from oracle import postprocess_oracle as ppo
from oracle import unet_oracle as uo

pytestmark = pytest.mark.gpu

FLAGS = [(True, True), (True, False), (False, True), (False, False)]
AXES = [(), (0,), (1,), (2,), (0, 1), (0, 2), (1, 2), (0, 1, 2)]


def host_flips(model, data, config, overlap):
    """predict_flips restated with np.flip: the input flip acts on the axes of `data` as given (so on (C, X, Y) of a
    [1,X,Y,Z] volume), the un-flip on the [X,Y,Z] prediction."""
    from fetal_net.prediction import patch_wise_prediction
    patch = tuple(config["patch_shape"]) + (config["patch_depth"],)
    maps = []
    for axes in AXES:
        d = np.flip(data, axes) if axes else data
        p = patch_wise_prediction(model, np.expand_dims(np.squeeze(d), 0), patch, overlap_factor=overlap).squeeze()
        maps.append(np.flip(p, axes) if axes else p)
    return maps


def check_tta(model, data, config, overlap, batch):
    """predict_flips, flip_tta_prediction and flip_tta_segmentation == the host composition, for all four flag pairs."""
    from fetal_net.device_tta import flip_tta_prediction, flip_tta_segmentation
    from fetal_net.prediction import predict_flips
    ref_maps = host_flips(model, data, config, overlap)
    ref_med = np.median(np.stack(ref_maps), axis=0)
    maps = predict_flips(data, model, overlap, config)
    assert len(maps) == 8
    for k, (got, ref) in enumerate(zip(maps, ref_maps)):
        assert got.dtype == np.float64 and got.shape == ref.shape and np.array_equal(got, ref), (AXES[k],)
    med, maps2 = flip_tta_prediction(data, model, overlap, config, batch_size=batch, return_maps=True)
    assert med.shape == ref_med.shape and np.array_equal(med, ref_med)
    assert all(np.array_equal(a, b) for a, b in zip(maps2, ref_maps))
    assert np.array_equal(flip_tta_prediction(data, model, overlap, config, batch_size=batch), ref_med)
    thr = float(np.median(ref_med))       # a decisive threshold for whatever the network predicts
    for fill, cc in FLAGS:
        pp = dict(threshold=thr, fill_holes=fill, connected_component=cc)
        ref = ppo.postprocess_prediction(ref_med, **pp)
        mask, m2 = flip_tta_segmentation(data, model, overlap, config, batch_size=batch, return_prediction=True, **pp)
        assert np.array_equal(m2, ref_med)
        assert mask.dtype == np.bool_ and np.array_equal(mask, ref), (fill, cc, int((mask != ref).sum()))
        assert np.array_equal(flip_tta_segmentation(data, model, overlap, config, batch_size=batch, **pp), ref)
    return ref_maps, ref_med


def raw_flips(model, data, config, overlap, batch, passes=8, in_flip=None, out_flip=None, maps=None, median=None):
    """fm_patchwise_predict_flips through the C ABI with caller-chosen output arrays; returns the return code."""
    from fetal_net import _lib
    from fetal_net.device_tta import _flip_masks
    from fetal_net.prediction import _geometry, patch_plan
    data4 = np.expand_dims(np.squeeze(data), 0)
    g = _geometry(model, data4, list(config["patch_shape"]) + [config["patch_depth"]], overlap)
    idx = patch_plan(g["padded"], g["patch_shape"], g["prediction_shape"], overlap)
    vol = _lib.f32c(data4[0])
    mi, mo = _flip_masks(np.ndim(data))
    in_flip = mi if in_flip is None else _lib.i32x(in_flip)
    out_flip = mo if out_flip is None else _lib.i32x(out_flip)
    return _lib.load().fm_patchwise_predict_flips(
        model._h, _lib.fptr(vol), _lib.i32ptr(_lib.i32x(vol.shape)), _lib.i32ptr(_lib.i32x(g["halo"])),
        _lib.i32ptr(_lib.i32x(g["fit"])), _lib.dptr(np.asarray(g["pad"], np.float64)), _lib.i32ptr(idx), len(idx),
        batch, passes, _lib.i32ptr(in_flip), _lib.i32ptr(out_flip), _lib.dptr(maps), _lib.dptr(median), None, None,
        None)


@pytest.fixture(scope="module")
def native64():
    from fetal_net.model import unet_model_3d
    from tests.test_gpu_model import decisive_weights
    m = unet_model_3d(input_shape=(1, 64, 64, 64), n_base_filters=16, depth=4)
    m.set_named_weights(decisive_weights(uo.unet3d_layers(4, 16), seed=3))
    return m


CFG64 = {"patch_shape": [64, 64], "patch_depth": 64}


def test_flips_configs0_geometry(native64):
    """1 x 256 x 256 x 64, 64^3 patches, overlap 0.5: maps, median and masks; maps and median also into pageable
    arrays, and in sub-batches of 5 and of 49 patches."""
    data = np.random.default_rng(0).standard_normal((256, 256, 64)).astype(np.float32)
    ref_maps, ref_med = check_tta(native64, data, CFG64, 0.5, 49)
    for batch in (5, 49):
        maps = np.empty((8, 256, 256, 64))
        med = np.empty((256, 256, 64))
        assert raw_flips(native64, data, CFG64, 0.5, batch, maps=maps, median=med) == 0
        assert np.array_equal(maps, np.stack(ref_maps)) and np.array_equal(med, ref_med)


def test_flips_volume_smaller_than_patch(native64):
    """pad_for_fit on every axis, with odd totals: the crop of each padded map precedes the un-flip."""
    data = np.random.default_rng(1).standard_normal((50, 41, 60)).astype(np.float32)
    check_tta(native64, data, CFG64, 0.5, 5)


def test_flips_4d_input(native64):
    """[1,X,Y,Z]: the input flips act on (C, X, Y), the un-flips on (X, Y, Z), as in the reference."""
    from fetal_net.device_tta import flip_tta_prediction
    data = np.random.default_rng(2).standard_normal((1, 96, 80, 64)).astype(np.float32)
    _, ref_med = check_tta(native64, data, CFG64, 0.5, 5)
    # the quirk changes the result: the same volume as [X,Y,Z] flips input and map along the same axes
    assert not np.array_equal(ref_med, flip_tta_prediction(data[0], native64, 0.5, CFG64))


def test_flips_2d_model():
    """2.5D unet_model_2d: 5-slice patches through config['patch_depth'], prediction (H, W, 1), z halo (2, 2)."""
    from fetal_net.model import unet_model_2d
    w = uo.glorot_uniform_weights(uo.unet2d_layers(4, 32, 5), seed=4, ndim=2)
    rng = np.random.default_rng(5)
    for k in w:
        w[k] = (w[k] * np.sqrt(2.0) * 1.15).astype(np.float32) if k.endswith("/kernel") else \
            (0.05 * rng.standard_normal(w[k].shape)).astype(np.float32)
    model = unet_model_2d(input_shape=(32, 32, 5), n_base_filters=32, depth=4)
    model.set_named_weights(w)
    data = rng.standard_normal((1, 48, 32, 10)).astype(np.float32)
    check_tta(model, data, {"patch_shape": [32, 32], "patch_depth": 5}, 0.5, 7)


def test_flips_generic_model_route(ctx):
    """A non-native model takes the host composition: predict_flips -> np.median -> device postprocess_prediction."""
    from oracle.ref_harness import FunctionModel
    from tests.golden.make_golden import ramp_model
    fn, oshape = ramp_model((8, 8, 8), 1)
    data = np.random.default_rng(6).standard_normal((20, 16, 12)).astype(np.float32)
    check_tta(FunctionModel(fn, oshape), data, {"patch_shape": [8, 8], "patch_depth": 8}, 0.5, 4)


def device_median(x):
    from fetal_net import _lib
    x = np.ascontiguousarray(x, np.float64)
    out = np.empty(x.shape[1:])
    _lib.check(_lib.load().fm_op_median_passes(_lib.get_context().handle, _lib.dptr(x), x.shape[0], out.size,
                                               _lib.dptr(out)))
    return out


@pytest.mark.parametrize("passes", [1, 2, 3, 4, 5, 6, 7, 8])
def test_median_hook_crafted(passes, ctx):
    """np.median over `passes` values: ties, +-inf (inf + -inf is NaN), NaN in one pass, voxel counts that are not a
    multiple of the 4-voxel vector."""
    rng = np.random.default_rng(passes)
    for nvox in (1, 3, 5, 4099, 1 << 16):
        x = rng.integers(0, 4, (passes, nvox)) / 4.0                                  # many ties
        x[rng.random(x.shape) < 0.1] = np.inf
        x[rng.random(x.shape) < 0.1] = -np.inf
        x[rng.integers(passes), rng.random(nvox) < 0.05] = np.nan
        if nvox > 4:
            x[:, 0] = [np.inf if k % 2 else -np.inf for k in range(passes)]           # +-inf in the middle pair
            x[:, 1] = rng.standard_normal(passes)                                     # distinct values
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            ref = np.median(x, axis=0)
        got = device_median(x)
        assert np.array_equal(got, ref, equal_nan=True), (passes, nvox, np.flatnonzero(~((got == ref) |
                                                                                      (np.isnan(got) & np.isnan(ref)))))
    # a large random field: the median of continuous values is one of them (odd) or the exact mean of two (even)
    x = rng.standard_normal((passes, 256 * 256 * 64 // 8 + 3))
    assert np.array_equal(device_median(x), np.median(x, axis=0))


def test_refusals_before_anything_is_read(native64, ctx):
    from fetal_net import _lib
    data = np.zeros((64, 64, 64), np.float32)
    nine = np.zeros(9, np.int32)
    for passes in (0, 9):
        assert raw_flips(native64, data, CFG64, 0.5, 5, passes=passes, in_flip=nine, out_flip=nine) == -1
    for bad in (-1, 8):
        masks = np.zeros(8, np.int32)
        masks[5] = bad
        assert raw_flips(native64, data, CFG64, 0.5, 5, in_flip=masks) == -1
        assert raw_flips(native64, data, CFG64, 0.5, 5, out_flip=masks) == -1
    x = np.zeros((9, 4))
    out = np.empty(4)
    for passes in (0, 9):
        assert _lib.load().fm_op_median_passes(ctx.handle, _lib.dptr(x), passes, 4, _lib.dptr(out)) == -1
    # post-processing of a volume over 2^31 - 1 voxels is refused up front, like fm_postprocess
    from fetal_net.device_postprocess import _spec
    spec, _w = _spec(1, 0.5, True, True)
    mask = np.zeros(8, np.uint8)
    rc = _lib.load().fm_patchwise_predict_flips(
        native64._h, _lib.fptr(data), _lib.i32ptr(_lib.i32x((2048, 1024, 1024))), _lib.i32ptr(_lib.i32x([0] * 6)),
        _lib.i32ptr(_lib.i32x([0] * 6)), _lib.dptr(np.zeros(2)), _lib.i32ptr(_lib.i32x([0, 0, 0])), 1, 5, 8,
        _lib.i32ptr(nine), _lib.i32ptr(nine), None, None, ctypes.byref(spec), mask.ctypes.data_as(_lib.c_u8p), None)
    assert rc == -1
