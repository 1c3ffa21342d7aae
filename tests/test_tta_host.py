"""Host side of the device flip TTA (fetal_net.device_tta): the per-pass flip masks handed to fm_patchwise_predict_flips
must reproduce the reference's flip_it on the input and on the prediction for every axis subset of predict_flips."""
import numpy as np
import pytest


def apply_mask(a, mask):
    for axis in range(3):
        if mask >> axis & 1:
            a = np.flip(a, axis)
    return a


@pytest.mark.parametrize("ndim", [3, 4])
def test_flip_masks_reproduce_flip_it(ndim):
    from fetal_net.device_tta import _AXES_SETS, _flip_masks
    from fetal_net.prediction import flip_it
    rng = np.random.default_rng(0)
    data = rng.standard_normal((1, 5, 4, 3) if ndim == 4 else (5, 4, 3))
    pred = rng.standard_normal((5, 4, 3))
    in_flip, out_flip = _flip_masks(ndim)
    assert len(_AXES_SETS) == len(in_flip) == len(out_flip) == 8
    assert _AXES_SETS == [(), (0,), (1,), (2,), (0, 1), (0, 2), (1, 2), (0, 1, 2)]
    for axes, mi, mo in zip(_AXES_SETS, in_flip, out_flip):
        assert 0 <= mi <= 7 and 0 <= mo <= 7
        # predict_flips: patch_wise_prediction(np.expand_dims(np.squeeze(flip_it(data, axes)), 0)) ...
        assert np.array_equal(apply_mask(np.squeeze(data), int(mi)), np.squeeze(flip_it(data, axes))), (ndim, axes)
        # ... then flip_it(prediction.squeeze(), axes)
        assert np.array_equal(apply_mask(pred, int(mo)), flip_it(pred, axes)), (ndim, axes)


def test_flip_masks_refuse_other_ranks():
    from fetal_net.device_tta import _flip_masks
    for ndim in (2, 5):
        with pytest.raises(ValueError):
            _flip_masks(ndim)


def test_native_route_only_for_shapes_predict_flips_keeps():
    from fetal_net.device_tta import _native_route
    from fetal_net.model.unet3d import Model
    native = Model.__new__(Model)          # only the type and the label count are looked at
    native.n_labels = 1
    assert _native_route(native, np.zeros((4, 3, 2)))
    assert _native_route(native, np.zeros((1, 4, 3, 2)))
    assert not _native_route(native, np.zeros((4, 1, 2)))       # squeeze would drop the unit axis
    assert not _native_route(native, np.zeros((2, 4, 3, 2)))
    assert not _native_route(object(), np.zeros((4, 3, 2)))
    native.n_labels = 2                                          # the maps would be [X,Y,Z,2]
    assert not _native_route(native, np.zeros((4, 3, 2)))
