"""Host side of the device post-processing (fetal_net.device_postprocess): the oracle and the Gaussian weights it hands
to the library are pinned to scipy here; the device kernels are compared to the oracle in test_gpu_postprocess.py."""
import importlib.util
import os

import numpy as np
import pytest
from scipy import ndimage

from oracle import postprocess_oracle as ppo
from oracle.ref_harness import REFERENCE_ROOT, reference_available

SHAPES = [(7, 5, 3), (2, 9, 1), (1, 9, 2), (33, 20, 17)]
SIGMAS = [0, 0.1, 0.5, 1, 1.7, 2]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_restated_filter_order_equals_scipy(dtype):
    """scipy's correlate1d sum order (centre first, then the symmetric pairs from the outermost in), reflect indexing
    that also covers lines shorter than the radius, and rounding to the input dtype after every axis."""
    rng = np.random.default_rng(0)
    for shape in SHAPES:
        x = rng.random(shape).astype(dtype)
        for s in SIGMAS:
            ref = ndimage.gaussian_filter(x, s)
            got = ppo.gaussian_filter_restated(x, s)
            assert got.dtype == ref.dtype and np.array_equal(got, ref), (shape, s)


@pytest.mark.parametrize("sigma", [0.1, 0.5, 1, 2])
def test_weights_equal_scipy_impulse_response(sigma):
    from fetal_net.device_postprocess import gaussian_weights
    w = gaussian_weights(sigma)
    r = (len(w) - 1) // 2
    assert r == int(4.0 * sigma + 0.5)
    impulse = np.zeros(2 * r + 11)
    impulse[r + 5] = 1.0
    assert np.array_equal(ndimage.gaussian_filter1d(impulse, sigma)[5:5 + 2 * r + 1], w)
    assert np.array_equal(w, ppo.gaussian_weights(sigma))


def test_sigma_zero_is_identity():
    from fetal_net.device_postprocess import gaussian_weights
    assert np.array_equal(gaussian_weights(0), [1.0])
    x = np.random.default_rng(1).random((6, 5, 4))
    assert np.array_equal(ndimage.gaussian_filter(x, 0), x)
    assert np.array_equal(ppo.gaussian_filter_restated(x, 0), x)


@pytest.mark.parametrize("pred, kwargs", [
    (np.zeros((4, 4)), {}),                                       # not 3-D
    (np.zeros((2, 4, 4, 4)), {}),
    (np.zeros((4, 4, 4), np.int32), {}),                          # dtype
    (np.zeros((4, 4, 4), np.float16), {}),
    (np.zeros((4, 4, 4)), dict(gaussian_std=-1)),                 # sigma
    (np.zeros((4, 4, 4)), dict(gaussian_std=float("nan"))),
])
def test_argument_checks_raise_before_any_device_call(pred, kwargs):
    from fetal_net.device_postprocess import postprocess_prediction
    with pytest.raises(ValueError):
        postprocess_prediction(pred, **kwargs)


def test_oracle_largest_component_tie_and_empty():
    seg = np.zeros((6, 6, 6), bool)
    seg[0, 0, 3:5] = True          # first in C order
    seg[4, 4, 0:2] = True          # same size, starts earlier in z but later in x
    assert np.array_equal(ppo.largest_component(seg), seg & (np.arange(6)[:, None, None] == 0))
    with pytest.raises(ValueError):
        ppo.postprocess_prediction(np.zeros((5, 5, 5)))


def _load_reference_postprocess():
    spec = importlib.util.spec_from_file_location("reference_postprocess",
                                                  os.path.join(REFERENCE_ROOT, "fetal_net", "postprocess.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)          # imports numpy and scipy only
    return mod


@pytest.mark.skipif(not reference_available(), reason="reference tree only exists in the build container")
def test_oracle_matches_live_reference_postprocess():
    ref = _load_reference_postprocess()
    rng = np.random.default_rng(2)
    field = ndimage.gaussian_filter(rng.random((40, 36, 24)), 2)
    field = (field - field.min()) / (field.max() - field.min())
    for dtype in (np.float32, np.float64):
        for flags in [(True, True), (True, False), (False, True), (False, False)]:
            kw = dict(gaussian_std=1, threshold=0.5, fill_holes=flags[0], connected_component=flags[1])
            assert np.array_equal(ppo.postprocess_prediction(field.astype(dtype), **kw),
                                  ref.postprocess_prediction(field.astype(dtype), **kw)), (dtype, flags)
