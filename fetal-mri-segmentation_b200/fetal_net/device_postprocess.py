"""The reference's post-processing (fetal_net/postprocess.py:13 `postprocess_prediction`) on the device.

`postprocess_prediction(pred, gaussian_std=1, threshold=0.5, fill_holes=True, connected_component=True)` keeps the
reference signature and returns the same bool [X,Y,Z] mask as scipy, bit for bit: Gaussian filter (mode 'reflect',
truncate 4), `> threshold` in the input dtype, binary_fill_holes, largest 6-connected component.
`patch_wise_segmentation(...)` is patch_wise_prediction followed by that post-processing; with a native Model the
float64 probability map never leaves the device (fm_patchwise_segment).

This module deliberately has its own name: under the overlay `fetal_net.postprocess` keeps resolving to the
reference's file (INTEGRATION.md shows how a caller routes postprocess_prediction here).
"""
import ctypes

import numpy as np

from . import _lib
from .model.unet3d import Model
from .prediction import _crop_fit, _geometry, _native_truth, patch_plan, patch_wise_prediction

_DTYPES = {np.dtype(np.float32): 0, np.dtype(np.float64): 1}


def gaussian_weights(sigma, truncate=4.0):
    """The 2r + 1 weights of scipy.ndimage.gaussian_filter1d (r = int(truncate * sigma + 0.5)), computed with
    numpy.exp exactly as scipy does. sigma <= 1e-15, an axis gaussian_filter skips, gives the identity [1.0]."""
    sigma = float(sigma)
    if sigma <= 1e-15:
        return np.ones(1, np.float64)
    radius = int(truncate * sigma + 0.5)
    x = np.arange(-radius, radius + 1)
    phi_x = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return phi_x / phi_x.sum()


def _spec(gaussian_std, threshold, fill_holes, connected_component):
    if not np.isscalar(gaussian_std) or not float(gaussian_std) >= 0:
        raise ValueError("gaussian_std must be a non-negative number, got %r" % (gaussian_std,))
    w = np.ascontiguousarray(gaussian_weights(gaussian_std), np.float64)
    spec = _lib.PostprocessSpec(radius=(len(w) - 1) // 2, weights=_lib.dptr(w), threshold=float(threshold),
                                fill_holes=1 if fill_holes else 0, connected_component=1 if connected_component else 0)
    return spec, w          # the weights array must outlive the call


def _finish(mask, n_components, connected_component):
    if connected_component and n_components == 0:
        # the reference's np.argmax over an empty list of component sizes
        raise ValueError("postprocess_prediction: no connected component above the threshold")
    return mask.view(np.bool_)


def postprocess_prediction(pred, gaussian_std=1, threshold=0.5, fill_holes=True, connected_component=True):
    """Drop-in for fetal_net/postprocess.py:13 on a float32 / float64 [X,Y,Z] array; returns a bool [X,Y,Z] mask."""
    pred = np.asarray(pred)
    if pred.ndim != 3:
        raise ValueError("postprocess_prediction expects a 3-D array, got shape %s" % (pred.shape,))
    if pred.dtype not in _DTYPES:
        raise ValueError("postprocess_prediction supports float32 and float64, got %s" % pred.dtype)
    spec, _w = _spec(gaussian_std, threshold, fill_holes, connected_component)
    if pred.size > np.iinfo(np.int32).max:
        raise ValueError("postprocess_prediction: %d voxels exceed 2^31 - 1" % pred.size)
    pred = np.ascontiguousarray(pred)
    mask = np.empty(pred.shape, np.uint8)
    ncomp = _lib.c_i64(0)
    ctx = _lib.get_context()
    _lib.check(_lib.load().fm_postprocess(ctx.handle, pred.ctypes.data_as(_lib.c_vp), _DTYPES[pred.dtype],
                                          _lib.i32ptr(_lib.i32x(pred.shape)), ctypes.byref(spec),
                                          mask.ctypes.data_as(_lib.c_u8p), ctypes.byref(ncomp)))
    return _finish(mask, ncomp.value, connected_component)


def patch_wise_segmentation(model, data, patch_shape, overlap_factor=0, batch_size=5, truth_data=None,
                            prev_truth_index=None, prev_truth_size=None, gaussian_std=1, threshold=0.5, fill_holes=True,
                            connected_component=True, return_prediction=False):
    """postprocess_prediction(patch_wise_prediction(model, data, ...).squeeze(), ...) for a one-label model: the bool
    [X,Y,Z] mask, and with return_prediction also the [X,Y,Z,1] float64 map patch_wise_prediction returns."""
    if getattr(model, "n_labels", 1) != 1:
        raise NotImplementedError("patch_wise_segmentation post-processes one probability map; the model has %d labels "
                                  "(segment each label of patch_wise_prediction with postprocess_prediction)"
                                  % model.n_labels)
    if not isinstance(model, Model):
        prob = patch_wise_prediction(model, data, patch_shape, overlap_factor=overlap_factor, batch_size=batch_size,
                                     truth_data=truth_data, prev_truth_index=prev_truth_index,
                                     prev_truth_size=prev_truth_size)
        mask = postprocess_prediction(prob.reshape(prob.shape[:3]), gaussian_std, threshold, fill_holes,
                                      connected_component)
        return (mask, prob) if return_prediction else mask
    lib = _lib.load()
    data = np.asarray(data)
    assert data.ndim == 4 and data.shape[0] == 1, "data must be [1,X,Y,Z] (prediction.py:296)"
    spec, _w = _spec(gaussian_std, threshold, fill_holes, connected_component)
    g = _geometry(model, data, patch_shape, overlap_factor)
    assert g["channels"] == 1, "post-processing needs a one-label model"
    idx = patch_plan(g["padded"], g["patch_shape"], g["prediction_shape"], overlap_factor)
    vol = _lib.f32c(data[0])
    truth = _native_truth(model, g, vol, truth_data, prev_truth_size)
    prob = _lib.pinned_empty(g["out_dims"] + (1,), np.float64) if return_prediction else None
    mask = np.empty(vol.shape, np.uint8)
    ncomp = _lib.c_i64(0)
    _lib.check(lib.fm_patchwise_segment(model._h, _lib.fptr(vol), _lib.i32ptr(_lib.i32x(vol.shape)),
                                        _lib.i32ptr(_lib.i32x(g["halo"])), _lib.i32ptr(_lib.i32x(g["fit"])),
                                        _lib.dptr(np.asarray(g["pad"], np.float64)), _lib.i32ptr(idx), len(idx),
                                        int(batch_size), _lib.fptr(truth), int(prev_truth_index or 0),
                                        int(prev_truth_size or 0), ctypes.byref(spec),
                                        mask.ctypes.data_as(_lib.c_u8p), _lib.dptr(prob), ctypes.byref(ncomp)))
    mask = _finish(mask, ncomp.value, connected_component)
    return (mask, _crop_fit(prob, g["fit"])) if return_prediction else mask
