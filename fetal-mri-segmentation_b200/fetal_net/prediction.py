"""Sliding-window inference — same entry points as the reference's fetal_net/prediction.py.

`patch_wise_prediction(model, data, patch_shape, overlap_factor=0, batch_size=5, permute=False,
truth_data=None, prev_truth_index=None, prev_truth_size=None)` keeps the reference signature,
return dtype (float64) and layout ([X,Y,Z,C], prediction.py:118-119,210). The host side here only
does what the reference does with integers and one percentile (pad arithmetic, prediction.py:129-146);
gather, network, overlap-add and the divide run on the device through the C ABI:

  native Model  -> fm_patchwise_predict: upload volume once, gather -> U-Net -> fp64 overlap-add -> download
  other models  -> fm_gather_patches, model.predict(batch) on whatever backend it has, fm_reassemble
"""
import itertools

import numpy as np

from . import _lib
from .model.unet3d import Model


def get_set_of_patch_indices_full(start, stop, step):
    """Corner grid of prediction.py:88-95: per axis start, start+step, ... <= stop, plus `stop` itself when it is not a
    multiple of the step (the reference tests `stop % step`, not `(stop - start) % step`); Cartesian product with the
    first axis slowest. Host twin of fm_patch_plan."""
    per_axis = []
    for lo, hi, stride in zip(start, stop, step):
        corners = list(range(lo, hi + 1, stride))
        if hi % stride > 0:
            corners.append(hi)
        per_axis.append(corners)
    return np.array(list(itertools.product(*per_axis)))


def patch_plan(padded_shape, patch_shape, prediction_shape, overlap_factor):
    """Patch corners through the C ABI (fm_patch_plan) — (n,3) int32, x-major product order."""
    lib = _lib.load()
    padded, patch, pred = _lib.i32x(padded_shape), _lib.i32x(patch_shape), _lib.i32x(prediction_shape)
    n = _lib.c_i64(0)
    import ctypes
    _lib.check(lib.fm_patch_plan(_lib.i32ptr(padded), _lib.i32ptr(patch), _lib.i32ptr(pred),
                                 float(overlap_factor), None, 0, ctypes.byref(n)))
    idx = np.empty((n.value, 3), np.int32)
    _lib.check(lib.fm_patch_plan(_lib.i32ptr(padded), _lib.i32ptr(patch), _lib.i32ptr(pred),
                                 float(overlap_factor), _lib.i32ptr(idx), n.value, ctypes.byref(n)))
    return idx


def _pad_pairs(diff):
    # [(ceil(d/2), floor(d/2))] — prediction.py:139-140,142-143
    return [(int(np.ceil(d / 2)), int(np.floor(d / 2))) for d in diff]


def _geometry(model, data, patch_shape, overlap_factor):
    """Integer/percentile host logic of prediction.py:129-146,161-163,169-173."""
    out_shape = tuple(model.output_shape)
    is3d = int(np.sum(np.array(out_shape[1:]) > 1)) > 2
    if getattr(model, "n_labels", 1) > 1 and getattr(model, "ndim", None) in (2, 3):
        # the reference's shape rule (prediction.py:129) takes a [H, W, n_labels > 1] output for a 3D one
        is3d = model.ndim == 3
    prediction_shape = tuple(out_shape[-3:]) if is3d else tuple(out_shape[-3:-1]) + (1,)
    patch_shape = tuple(int(v) for v in patch_shape)
    vol = data[0]
    halo = _pad_pairs(np.subtract(patch_shape, prediction_shape))
    halo_dims = tuple(int(s + a + b) for s, (a, b) in zip(vol.shape, halo))
    fit = _pad_pairs(np.maximum(np.subtract(patch_shape, halo_dims), 0))
    # the 1st-percentile pad value (prediction.py:141,146) is only needed where something is padded
    needs_pad = any(a + b for a, b in halo) or any(a + b for a, b in fit)
    pad0 = float(np.percentile(vol, q=1)) if needs_pad else 0.0
    if any(a + b for a, b in fit):
        # second percentile is taken over the already halo-padded array (prediction.py:144-146)
        padded_once = np.pad(vol, halo, mode='constant', constant_values=pad0) if any(a + b for a, b in halo) else vol
        pad1 = float(np.percentile(padded_once, q=1))
    else:
        pad1 = pad0
    padded = tuple(int(s + a + b) for s, (a, b) in zip(halo_dims, fit))
    n_channels = out_shape[1] if is3d else out_shape[-1]
    out_dims = tuple(int(s + a + b) for s, (a, b) in zip(vol.shape, fit))   # prediction.py:169
    return dict(is3d=is3d, prediction_shape=prediction_shape, patch_shape=patch_shape, halo=halo, fit=fit,
                pad=(pad0, pad1), padded=padded, out_dims=out_dims, channels=int(n_channels))


def _crop_fit(arr, fit):
    # prediction.py:198-207
    if sum(a + b for a, b in fit) > 0:
        sl = tuple(slice(a or None, -b if b else None) for a, b in fit)
        arr = arr[sl]
    return arr


def _native_truth(model, g, vol, truth_data, prev_truth_size):
    """Checks the patch shape against a native Model's input; returns the float32 previous-truth volume of the 2.5D
    path (or None)."""
    if g["is3d"]:
        assert tuple(g["patch_shape"]) == tuple(model.input_shape[2:]), \
            "patch_shape %s != model input %s" % (g["patch_shape"], model.input_shape[2:])
        assert truth_data is None, "truth_data conditions the 2.5D model only"
        return None
    n_truth = int(prev_truth_size) if truth_data is not None else 0
    assert tuple(g["patch_shape"][:2]) == tuple(model.input_shape[1:3]) and \
        g["patch_shape"][2] + n_truth == model.input_shape[3], \
        "patch_shape %s (+%d truth slices) != model input %s" % (g["patch_shape"], n_truth, model.input_shape[1:])
    if truth_data is None:
        return None
    truth = _lib.f32c(np.asarray(truth_data)[0])
    assert truth.shape == vol.shape
    return truth


def patch_wise_prediction(model, data, patch_shape, overlap_factor=0, batch_size=5,
                          permute=False, truth_data=None, prev_truth_index=None, prev_truth_size=None,
                          shard=None, reduce_root=None):
    """Drop-in for fetal_net/prediction.py:118-210. `shard=(rank, count)` (extension) makes this call
    process only its contiguous share of the patch list and return (partial float64 sums, int16 counts)
    for the caller to reduce; with `reduce_root` (native models, ranks = the library's NCCL communicator) the partial
    sums are reduced on the GPUs and the call returns the finished volume on that rank and None elsewhere — see
    fetal_net.distributed.sharded_patch_wise_prediction."""
    lib = _lib.load()
    data = np.asarray(data)
    assert data.ndim == 4 and data.shape[0] == 1, "data must be [1,X,Y,Z] (prediction.py:296)"
    g = _geometry(model, data, patch_shape, overlap_factor)
    if permute:
        # prediction.py:185 routes every batch through predict(..., permute=True): the per-patch average over the
        # flip/rotation keys. The fused native pipeline has no such hook, so take the generic route with a model
        # wrapper whose predict() does the averaging — same patches, same order, same reassembly.
        assert g["is3d"], "permute=True needs [B,C,x,y,z] patches (augment.py:407-434)"
        assert shard is None, "permute=True is not sharded"
        return patch_wise_prediction(_PermutingModel(model), data, patch_shape, overlap_factor, batch_size,
                                     False, truth_data, prev_truth_index, prev_truth_size)
    idx = patch_plan(g["padded"], g["patch_shape"], g["prediction_shape"], overlap_factor)
    vol = _lib.f32c(data[0])                      # Keras casts the float64 feed to float32
    vol_dims = _lib.i32x(vol.shape)
    halo = _lib.i32x(g["halo"])
    fit = _lib.i32x(g["fit"])
    padv = np.asarray(g["pad"], np.float64)
    # the float64 result lives in page-locked memory from a small pool (an ordinary ndarray to the caller): the
    # device->host slabs land in it directly, without a staging copy or the first-touch faults of a fresh 33 MB array
    out = (_lib.pinned_empty if isinstance(model, Model) else np.empty)(g["out_dims"] + (g["channels"],), np.float64)
    rank, count = (0, 1) if shard is None else (int(shard[0]), int(shard[1]))
    # counts are analytic: the library rejects an uncovered voxel itself ('Found zeros in count'), so the
    # int16 map only travels back when the caller has to divide after a cross-rank reduce
    cnt = np.empty(g["out_dims"], np.int16) if count > 1 else None

    if isinstance(model, Model):
        truth = _native_truth(model, g, vol, truth_data, prev_truth_size)
        if reduce_root is not None and count > 1:
            is_root = rank == int(reduce_root)
            _lib.check(lib.fm_patchwise_predict_dp(model._h, _lib.fptr(vol), _lib.i32ptr(vol_dims), _lib.i32ptr(halo),
                                                   _lib.i32ptr(fit), _lib.dptr(padv), _lib.i32ptr(idx), len(idx),
                                                   int(batch_size), int(reduce_root), _lib.fptr(truth),
                                                   int(prev_truth_index or 0), int(prev_truth_size or 0),
                                                   _lib.dptr(out) if is_root else None, None))
            if not is_root:
                return None
            out = _crop_fit(out, g["fit"])
            assert np.array_equal(out.shape[:-1], data[0].shape), 'prediction shape wrong'
            return out
        _lib.check(lib.fm_patchwise_predict(model._h, _lib.fptr(vol), _lib.i32ptr(vol_dims), _lib.i32ptr(halo),
                                            _lib.i32ptr(fit), _lib.dptr(padv), _lib.i32ptr(idx), len(idx),
                                            int(batch_size), rank, count, _lib.fptr(truth),
                                            int(prev_truth_index or 0), int(prev_truth_size or 0),
                                            _lib.dptr(out), _lib.i16ptr(cnt)))
    else:
        # any other Keras-like model: patches are gathered on the device, the model predicts wherever it
        # lives, the overlap-add / average runs on the device again
        ctx = _lib.get_context()
        lo, hi = len(idx) * rank // count, len(idx) * (rank + 1) // count
        ps = g["patch_shape"]
        preds = np.empty((hi - lo,) + tuple(g["prediction_shape"]) + (g["channels"],), np.float32)
        patch_i32 = _lib.i32x(ps)
        truth = None if truth_data is None else _lib.f32c(np.asarray(truth_data)[0])
        zero_pad = np.zeros(2, np.float64)
        for b0 in range(lo, hi, batch_size):
            bi = np.ascontiguousarray(idx[b0:min(b0 + batch_size, hi)])
            batch = np.empty((len(bi),) + tuple(ps), np.float32)
            _lib.check(lib.fm_gather_patches(ctx.handle, _lib.fptr(vol), _lib.i32ptr(vol_dims), _lib.i32ptr(halo),
                                             _lib.i32ptr(fit), _lib.dptr(padv), _lib.i32ptr(bi), len(bi),
                                             _lib.i32ptr(patch_i32), _lib.fptr(batch)))
            if truth is not None:
                # prediction.py:106-110: truth slices [z + prev_truth_index, +prev_truth_size) as extra channels
                ti = bi.copy()
                ti[:, 2] += int(prev_truth_index)
                tps = _lib.i32x(list(ps[:2]) + [int(prev_truth_size)])
                tb = np.empty((len(bi),) + tuple(ps[:2]) + (int(prev_truth_size),), np.float32)
                _lib.check(lib.fm_gather_patches(ctx.handle, _lib.fptr(truth), _lib.i32ptr(vol_dims), _lib.i32ptr(halo),
                                                 _lib.i32ptr(fit), _lib.dptr(zero_pad), _lib.i32ptr(ti), len(ti),
                                                 _lib.i32ptr(tps), _lib.fptr(tb)))
                batch = np.concatenate([batch, tb], axis=-1)
            if g["is3d"]:
                p = predict(model, batch[:, None], permute=False)          # [B,C,x,y,z]
                preds[b0 - lo:b0 - lo + len(bi)] = np.asarray(p, np.float32).transpose(0, 2, 3, 4, 1)
            else:
                p = predict(model, batch, permute=False)                   # [B,H,W,C]
                preds[b0 - lo:b0 - lo + len(bi)] = np.expand_dims(np.asarray(p, np.float32), -2)   # prediction.py:184
        if count == 1:
            _lib.check(lib.fm_reassemble(ctx.handle, _lib.fptr(preds), _lib.i32ptr(idx), len(idx),
                                         _lib.i32ptr(_lib.i32x(g["prediction_shape"])), g["channels"],
                                         _lib.i32ptr(_lib.i32x(g["out_dims"])), _lib.dptr(out), None))
        else:
            raise NotImplementedError("sharded inference needs a native Model")

    if shard is not None and count > 1:
        return _crop_fit(out, g["fit"]), _crop_fit(cnt, g["fit"])
    # prediction.py:196 'Found zeros in count' is raised by the library (fm_reassemble) for an uncovered voxel
    out = _crop_fit(out, g["fit"])
    assert np.array_equal(out.shape[:-1], data[0].shape), 'prediction shape wrong'  # prediction.py:209
    return out


def predict(model, data, permute=False):
    # prediction.py:354-361
    if permute:
        return np.asarray([predict_with_permutations(model, data[i]) for i in range(data.shape[0])])
    return model.predict(data)


# ---------------------------------------------------------------------------------------------
# test-time augmentation wrappers (prediction.py:19-85,364-369; augment.py:380-469). They only
# re-index the volume on the host; every prediction inside is the device pipeline above.
# ---------------------------------------------------------------------------------------------
class _PermutingModel:
    """Keras-Model duck type whose predict() averages over the permutation keys (prediction.py:356-359)."""

    def __init__(self, model):
        self._model = model
        self.output_shape = model.output_shape

    def predict(self, data):
        return predict(self._model, np.asarray(data), permute=True)


def flip_it(data_, axes):
    # prediction.py:19-22
    for ax in axes:
        data_ = np.flip(data_, ax)
    return data_


def generate_permutation_keys():
    """augment.py:380-396: keys ((rotate_y, rotate_z), flip_x, flip_y, flip_z, transpose) — 3*2*2*2*2 = 48 tuples.
    Kept as a set like the reference so the float32 mean below adds the terms in the same order."""
    return set(itertools.product(itertools.combinations_with_replacement(range(2), 2),
                                 range(2), range(2), range(2), range(2)))


def permute_data(data, key):
    """augment.py:407-434 as it actually behaves: rot90 by rotate_y in the (x,y) plane, then the three flips;
    rotate_z and transpose are carried in the key but unused (commented out in the reference)."""
    data = np.copy(data)
    (rotate_y, _rotate_z), flip_x, flip_y, flip_z, _transpose = key
    if rotate_y != 0:
        data = np.rot90(data, rotate_y, axes=(1, 2))
    if flip_x:
        data = data[:, ::-1]
    if flip_y:
        data = data[:, :, ::-1]
    if flip_z:
        data = data[:, :, :, ::-1]
    return data


def reverse_permutation_key(key):
    # augment.py:467-469
    return tuple(-r for r in key[0]), key[1], key[2], key[3], key[4]


def reverse_permute_data(data, key):
    # augment.py:448-464: undo in the opposite order with the rotation negated
    (rotate_y, _rotate_z), flip_x, flip_y, flip_z, _transpose = reverse_permutation_key(key)
    data = np.copy(data)
    if flip_z:
        data = data[:, :, :, ::-1]
    if flip_y:
        data = data[:, :, ::-1]
    if flip_x:
        data = data[:, ::-1]
    if rotate_y != 0:
        data = np.rot90(data, rotate_y, axes=(1, 2))
    return data


def predict_with_permutations(model, data):
    """prediction.py:364-369: data [C,x,y,z]; mean over all keys of the un-permuted prediction of the permuted
    patch. All 48 permuted copies go to the device as ONE predict() batch when the patch is square in (x,y)
    (rot90 keeps the shape); otherwise key by key like the reference."""
    keys = list(generate_permutation_keys())
    permuted = [permute_data(data, k) for k in keys]
    if all(p.shape == permuted[0].shape for p in permuted):
        stack = np.ascontiguousarray(np.stack(permuted))
        # native model: 8 patches per launch, so the activation workspace is sized for 8 (not 32) full patches - the
        # reference runs one patch at a time and never holds more
        outs = np.asarray(model.predict(stack, batch_size=8) if isinstance(model, Model) else model.predict(stack))
        predictions = [reverse_permute_data(outs[i], k) for i, k in enumerate(keys)]
    else:
        predictions = [reverse_permute_data(model.predict(np.ascontiguousarray(p[np.newaxis]))[0], k)
                       for p, k in zip(permuted, keys)]
    return np.mean(predictions, axis=0)


def predict_flips(data, model, overlap_factor, config):
    """prediction.py:65-85: the 8 axis-flip subsets in powerset order () (0,) (1,) (2,) (0,1) (0,2) (1,2) (0,1,2);
    returns the list of un-flipped predictions [X,Y,Z] (the caller takes the median, predict_nifti2.py:86-87).
    A native Model with a [X,Y,Z] or [1,X,Y,Z] volume runs all 8 passes in one device call (fetal_net.device_tta); its
    entries are then views of one page-locked [8,X,Y,Z] array."""
    from .device_tta import _device_flips, _native_route
    if _native_route(model, data):
        return list(_device_flips(data, model, overlap_factor, config, 5, maps=True)[0])
    patch_shape = list(config["patch_shape"]) + [config["patch_depth"]]
    axes_sets = itertools.chain.from_iterable(itertools.combinations([0, 1, 2], r) for r in range(4))
    predictions = []
    for axes in axes_sets:
        data_ = flip_it(data, axes)
        curr = patch_wise_prediction(model=model, data=np.expand_dims(np.squeeze(data_), 0),
                                     overlap_factor=overlap_factor, patch_shape=patch_shape).squeeze()
        predictions.append(flip_it(curr, axes).squeeze())
    return predictions


def rescale_intensity_to_image_range(data, in_min, in_max):
    """What augment.py:123-126 `contrast_augment` asks of skimage.exposure.rescale_intensity(data,
    in_range=(lo, hi), out_range='image'): clip to [lo, hi], map linearly onto the image's own [min, max]."""
    data = np.asarray(data)
    omin, omax = data.min(), data.max()
    scaled = (np.clip(data, in_min, in_max) - in_min) / (in_max - in_min)
    return (scaled * (omax - omin) + omin).astype(data.dtype)


def predict_augment(data, model, overlap_factor, patch_shape, num_augments=32):
    """prediction.py:25-62: random contrast window, flips, (x,y) transpose and an in-plane rotation of up to
    +-30 degrees (scipy.ndimage.rotate, order 2, reshape=False), predict, undo; returns [num_augments,X,Y,Z].
    Draws from np.random in the reference's order, so a seeded run reproduces the reference's augmentations."""
    from scipy import ndimage
    data_max, data_min = data.max(), data.min()
    data = np.squeeze(data)
    predictions = []
    for _ in range(num_augments):
        val_range = data_max - data_min
        lo = data_min + 0.10 * np.random.uniform(-1, 1) * val_range
        hi = data_max + 0.10 * np.random.uniform(-1, 1) * val_range
        curr = rescale_intensity_to_image_range(data, lo, hi)
        rotate_factor = np.random.uniform(-30, 30)
        to_flip = np.arange(0, 3)[np.random.choice([True, False], size=3)]
        to_transpose = np.random.choice([True, False])
        curr = flip_it(curr, to_flip)
        if to_transpose:
            curr = curr.transpose([1, 0, 2])
        curr = ndimage.rotate(curr, rotate_factor, order=2, reshape=False)
        pred = patch_wise_prediction(model=model, data=curr[np.newaxis, ...], overlap_factor=overlap_factor,
                                     patch_shape=patch_shape).squeeze()
        pred = ndimage.rotate(pred, -rotate_factor)     # default order 3, reshape=True — as the reference
        if to_transpose:
            pred = pred.transpose([1, 0, 2])
        predictions.append(flip_it(pred, to_flip).squeeze())
    return np.stack(predictions, axis=0)


# ---------------------------------------------------------------------------------------------
# the callers of the hot path inside the reference's own prediction module (prediction.py:277-351): host I/O glue
# (PyTables in, NIfTI out) around predict / patch_wise_prediction. The I/O helpers are the reference's own, reached
# through the overlay (fetal_net.utils.utils: get_image, pickle_load); they need nibabel / tables like the reference.
# ---------------------------------------------------------------------------------------------
def _reference_utils():
    try:
        from .utils import utils as ref_utils          # resolves to <FETAL_REFERENCE_ROOT>/fetal_net/utils/utils.py
    except ImportError as e:
        raise ImportError("run_validation_case(s) writes NIfTI images with the reference's own helpers "
                          "(fetal_net/utils/utils.py: get_image, pickle_load): set FETAL_REFERENCE_ROOT to a checkout "
                          "of the reference (and install nibabel / tables as it requires)") from e
    return ref_utils


def run_validation_case(data_index, output_dir, model, data_file, training_modalities, patch_shape,
                        overlap_factor=0, permute=False, prev_truth_index=None, prev_truth_size=None,
                        use_augmentations=False):
    """prediction.py:277-330 with the same signature: writes data_<modality>.nii.gz, truth.nii.gz and prediction.nii.gz
    of one case; the prediction itself is predict() (volume == patch) or patch_wise_prediction() on the device."""
    import os
    get_image = _reference_utils().get_image
    if not os.path.exists(output_dir):
        os.makedirs(output_dir)
    test_data = np.asarray([data_file.root.data[data_index]])
    test_truth_data = np.asarray([data_file.root.truth[data_index]]) if prev_truth_index is not None else None
    for i, modality in enumerate(training_modalities):
        get_image(test_data[i]).to_filename(os.path.join(output_dir, "data_{0}.nii.gz".format(modality)))
    get_image(data_file.root.truth[data_index]).to_filename(os.path.join(output_dir, "truth.nii.gz"))
    if tuple(patch_shape) == tuple(test_data.shape[-3:]):
        prediction = predict(model, test_data, permute=permute)
    elif use_augmentations:
        prediction = predict_augment(data=test_data, model=model, overlap_factor=overlap_factor, patch_shape=patch_shape)
    else:
        prediction = patch_wise_prediction(model=model, data=test_data, overlap_factor=overlap_factor,
                                           patch_shape=patch_shape, truth_data=test_truth_data,
                                           prev_truth_index=prev_truth_index, prev_truth_size=prev_truth_size)[np.newaxis]
    prediction = prediction.squeeze()
    prediction_image = get_image(prediction)
    if isinstance(prediction_image, list):
        for i, image in enumerate(prediction_image):
            filename = os.path.join(output_dir, "prediction_{0}.nii.gz".format(i + 1))
            image.to_filename(filename)
    else:
        filename = os.path.join(output_dir, "prediction.nii.gz")
        prediction_image.to_filename(filename)
    return filename


def run_validation_cases(validation_keys_file, model_file, training_modalities, hdf5_file, patch_shape,
                         output_dir=".", overlap_factor=0, permute=False,
                         prev_truth_index=None, prev_truth_size=None, use_augmentations=False):
    """prediction.py:333-351 with the same signature (the entry point of fetal/predict.py:5,22-30)."""
    import os
    import tables                                        # the reference's data files are PyTables HDF5
    from .training import get_last_model_path, load_old_model
    file_names = []
    validation_indices = _reference_utils().pickle_load(validation_keys_file)
    model = load_old_model(get_last_model_path(model_file))
    data_file = tables.open_file(hdf5_file, "r")
    try:
        for index in validation_indices:
            if 'subject_ids' in data_file.root:
                case_directory = os.path.join(output_dir, data_file.root.subject_ids[index].decode('utf-8'))
            else:
                case_directory = os.path.join(output_dir, "validation_case_{}".format(index))
            file_names.append(
                run_validation_case(data_index=index, output_dir=case_directory, model=model, data_file=data_file,
                                    training_modalities=training_modalities, overlap_factor=overlap_factor,
                                    permute=permute, patch_shape=patch_shape, prev_truth_index=prev_truth_index,
                                    prev_truth_size=prev_truth_size, use_augmentations=use_augmentations))
    finally:
        data_file.close()
    return file_names
