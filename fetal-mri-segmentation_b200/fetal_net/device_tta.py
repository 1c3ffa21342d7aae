"""Flip test-time augmentation on the device: the reference's predict_flips (fetal_net/prediction.py:65-85), the
per-voxel median its callers take (predict_nifti2.py:86-87) and postprocess_prediction, in one call.

`flip_tta_prediction(data, model, overlap_factor, config)` returns np.median(np.stack(predict_flips(...)), axis=0),
`flip_tta_segmentation(...)` that median post-processed like fetal_net.device_postprocess.postprocess_prediction. With a
native Model the eight sliding-window passes, the un-flips, the median and the post-processing all run in
fm_patchwise_predict_flips: the volume goes up once, and only what the caller asks for comes back. Any other model takes
the host composition predict_flips -> np.median -> postprocess_prediction. Both routes give the same bits.
"""
import ctypes
import itertools

import numpy as np

from . import _lib
from .device_postprocess import _finish, _spec, postprocess_prediction
from .model.unet3d import Model
from .prediction import _geometry, _native_truth, patch_plan, predict_flips

# the 8 axis subsets of predict_flips, powerset order () (0,) (1,) (2,) (0,1) (0,2) (1,2) (0,1,2)
_AXES_SETS = list(itertools.chain.from_iterable(itertools.combinations([0, 1, 2], r) for r in range(4)))


def _flip_masks(ndim):
    """(input masks, output masks) of the 8 passes of predict_flips, int32 with bit a = volume axis a. flip_it flips
    the axes of whatever it is given: a [X,Y,Z] input and the [X,Y,Z] prediction alike, but of a [1,X,Y,Z] input axis
    0 is the channel (a no-op) and axes 1, 2 are X, Y, while the un-flip still acts on the prediction's X, Y, Z."""
    out = [sum(1 << a for a in axes) for axes in _AXES_SETS]
    if ndim == 3:
        inp = out
    elif ndim == 4:
        inp = [sum(1 << (a - 1) for a in axes if a > 0) for axes in _AXES_SETS]
    else:
        raise ValueError("flip TTA takes a [X,Y,Z] or [1,X,Y,Z] volume, got %d dimensions" % ndim)
    return _lib.i32x(inp), _lib.i32x(out)


def _native_route(model, data):
    """True when fm_patchwise_predict_flips computes exactly what predict_flips does: a native one-label Model and a
    [X,Y,Z] or [1,X,Y,Z] volume none of whose extents is 1 (the reference's squeeze would drop it)."""
    shape = np.shape(data)
    spatial = shape if len(shape) == 3 else (shape[1:] if len(shape) == 4 and shape[0] == 1 else None)
    return isinstance(model, Model) and model.n_labels == 1 and spatial is not None and all(s > 1 for s in spatial)


def _device_flips(data, model, overlap_factor, config, batch_size, maps=False, median=False, pp=None):
    """One fm_patchwise_predict_flips call over the 8 passes: (maps [8,X,Y,Z] | None, median [X,Y,Z] | None,
    uint8 mask | None, number of components). Results are page-locked arrays; `pp` = _spec(...) or None."""
    data = np.asarray(data)
    in_flip, out_flip = _flip_masks(data.ndim)
    vol4 = np.expand_dims(np.squeeze(data), 0)            # what predict_flips hands patch_wise_prediction
    patch_shape = list(config["patch_shape"]) + [config["patch_depth"]]
    g = _geometry(model, vol4, patch_shape, overlap_factor)
    vol = _lib.f32c(vol4[0])
    _native_truth(model, g, vol, None, None)
    idx = patch_plan(g["padded"], g["patch_shape"], g["prediction_shape"], overlap_factor)
    maps_out = _lib.pinned_empty((len(_AXES_SETS),) + vol.shape, np.float64) if maps else None
    median_out = _lib.pinned_empty(vol.shape, np.float64) if median else None
    spec = pp[0] if pp is not None else None
    mask = np.empty(vol.shape, np.uint8) if pp is not None else None
    ncomp = _lib.c_i64(0)
    _lib.check(_lib.load().fm_patchwise_predict_flips(
        model._h, _lib.fptr(vol), _lib.i32ptr(_lib.i32x(vol.shape)), _lib.i32ptr(_lib.i32x(g["halo"])),
        _lib.i32ptr(_lib.i32x(g["fit"])), _lib.dptr(np.asarray(g["pad"], np.float64)), _lib.i32ptr(idx), len(idx),
        int(batch_size), len(_AXES_SETS), _lib.i32ptr(in_flip), _lib.i32ptr(out_flip), _lib.dptr(maps_out),
        _lib.dptr(median_out), ctypes.byref(spec) if spec is not None else None,
        mask.ctypes.data_as(_lib.c_u8p) if mask is not None else None, ctypes.byref(ncomp)))
    return maps_out, median_out, mask, ncomp.value


def flip_tta_prediction(data, model, overlap_factor, config, batch_size=5, return_maps=False):
    """np.median(np.stack(predict_flips(data, model, overlap_factor, config)), axis=0): the float64 [X,Y,Z] median, and
    with return_maps also the list of the 8 maps. `batch_size` is the native model's patches per launch (the result
    does not depend on it); other models run predict_flips as it is."""
    if _native_route(model, data):
        maps, median, _, _ = _device_flips(data, model, overlap_factor, config, batch_size, maps=return_maps,
                                           median=True)
        return (median, list(maps)) if return_maps else median
    maps = predict_flips(data, model, overlap_factor, config)
    median = np.median(np.stack(maps), axis=0)
    return (median, maps) if return_maps else median


def flip_tta_segmentation(data, model, overlap_factor, config, gaussian_std=1, threshold=0.5, fill_holes=True,
                          connected_component=True, batch_size=5, return_prediction=False):
    """postprocess_prediction(flip_tta_prediction(...), gaussian_std, threshold, fill_holes, connected_component): the
    bool [X,Y,Z] mask, and with return_prediction also the median."""
    if not _native_route(model, data):
        median = flip_tta_prediction(data, model, overlap_factor, config, batch_size)
        mask = postprocess_prediction(median, gaussian_std, threshold, fill_holes, connected_component)
        return (mask, median) if return_prediction else mask
    pp = _spec(gaussian_std, threshold, fill_holes, connected_component)
    _, median, mask, ncomp = _device_flips(data, model, overlap_factor, config, batch_size, median=return_prediction,
                                           pp=pp)
    mask = _finish(mask, ncomp, connected_component)
    return (mask, median) if return_prediction else mask
