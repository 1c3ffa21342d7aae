"""Host side of n_labels > 1: the label-wise Dice restatement, the checkpoint flag, the refusals of the paths that take
one-label models only, and the C ABI declaration of fm_model_label_dice. No GPU needed."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def label_dice(t, p, i, axis=1):
    ti = np.take(t, i, axis=axis).astype(np.float64)
    pi = np.take(p, i, axis=axis).astype(np.float64)
    return (2.0 * (ti * pi).sum() + 1.0) / (ti.sum() + pi.sum() + 1.0)


def test_label_dice_against_loops():
    rng = np.random.default_rng(0)
    t = (rng.random((2, 3, 4, 5, 6)) > 0.5).astype(np.float32)
    p = rng.random((2, 3, 4, 5, 6)).astype(np.float32)
    for i in range(3):
        inter = st = sp = 0.0
        for b in range(2):
            for v in np.ndindex(4, 5, 6):
                inter += float(t[(b, i) + v]) * float(p[(b, i) + v])
                st += float(t[(b, i) + v])
                sp += float(p[(b, i) + v])
        assert label_dice(t, p, i) == pytest.approx((2 * inter + 1) / (st + sp + 1), rel=1e-12)
        # the 2D models carry the label axis last
        assert label_dice(np.moveaxis(t, 1, -1), np.moveaxis(p, 1, -1), i, axis=-1) == \
            pytest.approx(label_dice(t, p, i), rel=1e-12)


def test_device_sums_layout_gives_label_dice():
    """The device keeps (sum t p, sum t, sum p) per label over the [voxel][label] layout; the label of element e is
    e mod L. Restated here: the per-label sums of the label-fastest flattening equal the channels-first Dice."""
    rng = np.random.default_rng(1)
    L = 4
    t = (rng.random((2, L, 3, 4, 5)) > 0.5).astype(np.float32)
    p = rng.random((2, L, 3, 4, 5)).astype(np.float32)
    flat_t = np.moveaxis(t, 1, -1).reshape(-1).astype(np.float64)
    flat_p = np.moveaxis(p, 1, -1).reshape(-1).astype(np.float64)
    lab = np.arange(flat_t.size) % L
    for i in range(L):
        m = lab == i
        d = (2 * (flat_t[m] * flat_p[m]).sum() + 1) / (flat_t[m].sum() + flat_p[m].sum() + 1)
        assert d == pytest.approx(label_dice(t, p, i), rel=1e-12)


def test_header_declares_label_dice():
    from fetal_net import _lib
    text = open(os.path.join(ROOT, "include", "fetal_b200.h")).read()
    assert "int fm_model_label_dice(fm_model* m, float* out, int n);" in text
    assert "fm_model_label_dice" in _lib.SIGNATURES


class _FakeModel:
    n_labels = 3
    ndim = 3
    output_shape = (None, 3, 32, 32, 32)


def test_patch_wise_segmentation_refuses_multi_label():
    from fetal_net.device_postprocess import patch_wise_segmentation
    with pytest.raises(NotImplementedError, match="3 labels"):
        patch_wise_segmentation(_FakeModel(), np.zeros((1, 8, 8, 8), np.float32), patch_shape=(8, 8, 8))


def test_device_sampler_refuses_multi_label():
    from fetal_net.device_sampler import DeviceSampler, _check_one_label
    with pytest.raises(NotImplementedError, match="one target channel"):
        _check_one_label(_FakeModel())

    class _S:
        pass
    with pytest.raises(NotImplementedError, match="one target channel"):
        DeviceSampler.train_on_next_batch(_S(), _FakeModel())


def test_geometry_of_multi_label_2d_model():
    """A [H, W, n_labels] output is 2D even when n_labels > 1 (the reference's shape rule alone would call it 3D)."""
    from fetal_net.prediction import _geometry

    class _M2:
        n_labels, ndim, output_shape = 3, 2, (None, 32, 32, 3)

    g = _geometry(_M2(), np.zeros((1, 40, 40, 10), np.float32), (32, 32, 5), 0.5)
    assert not g["is3d"] and g["channels"] == 3 and g["prediction_shape"] == (32, 32, 1)
    g3 = _geometry(_FakeModel(), np.zeros((1, 40, 40, 40), np.float32), (32, 32, 32), 0.5)
    assert g3["is3d"] and g3["channels"] == 3 and g3["prediction_shape"] == (32, 32, 32)


def test_load_old_model_restores_labels_and_label_wise_flag(tmp_path, monkeypatch):
    from fetal_net import training
    seen = {}

    class _Rebuilt:
        def load_weights(self, path):
            pass

        def load_optimizer_state(self, path):
            return False

    def fake_builder(**kw):
        seen.update(kw)
        return _Rebuilt()

    monkeypatch.setattr(training._model_ns, "unet_model_3d", fake_builder)
    path = str(tmp_path / "m.h5")
    with open(path, "wb") as f:
        np.savez(f, __config__=np.array([1, 32, 32, 32, 4, 16, 3]), __builder__=np.array("unet_model_3d"),
                 __isensee_levels__=np.array(0), __deconvolution__=np.array(0), __batch_normalization__=np.array(0),
                 __label_wise__=np.array(1))
    training.load_old_model(path, verbose=False)
    assert seen["n_labels"] == 3 and seen["include_label_wise_dice_coefficients"] is True
    seen.clear()
    with open(path, "wb") as f:   # archives written before the flag existed
        np.savez(f, __config__=np.array([1, 32, 32, 32, 4, 16, 2]), __builder__=np.array("unet_model_3d"))
    training.load_old_model(path, verbose=False)
    assert seen["n_labels"] == 2 and "include_label_wise_dice_coefficients" not in seen


def test_keras_h5_names_multi_label_head():
    """A (1,1,1,C,L) final kernel bridges under the same conv3d_<n> key, shape intact, as a one-label head does."""
    from fetal_net import keras_h5
    rng = np.random.default_rng(2)
    body = rng.standard_normal((3, 3, 3, 1, 16)).astype(np.float32)
    head = rng.standard_normal((1, 1, 1, 32, 3)).astype(np.float32)
    arrays = keras_h5.to_npz_arrays([("conv", "conv3d_1", body, np.zeros(16, np.float32)),
                                     ("conv", "conv3d_2", head, np.arange(3, dtype=np.float32))])
    assert arrays["conv3d_2/kernel:0"].shape == (1, 1, 1, 32, 3)
    assert np.array_equal(arrays["conv3d_2/kernel:0"], head)
    assert np.array_equal(arrays["conv3d_2/bias:0"], np.arange(3, dtype=np.float32))
