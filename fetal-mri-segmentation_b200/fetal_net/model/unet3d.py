"""`unet_model_3d` — the reference builder (fetal_net/model/unet3d/unet.py:17-86) over libfetalb200.

Returns a `Model` with the Keras-Model members the reference's callers use (SURVEY.md §8b):
predict / output_shape (prediction.py:129-134,361), fit_generator (training.py:110-124),
train_on_batch / evaluate / metrics_names / optimizer.lr (experiments/train_adv.py:227,257,220,285),
summary (train_fetal.py:44), load_weights / save / save_weights (train_fetal.py:43, training.py:83).
"""
import ctypes
import os

import numpy as np

from .. import _lib
from ..metrics import dice_coefficient_loss, device_loss_spec


class _Optimizer:
    """`model.optimizer.lr` as used by Keras callbacks (ReduceLROnPlateau sets it)."""

    def __init__(self, lr):
        self.lr = float(lr)
        self.beta_1, self.beta_2, self.epsilon = 0.9, 0.999, 1e-7


def _slot_keys(l):
    """Suffixes of a layer's two arrays in a checkpoint: kernel/bias, gamma/beta or moving_mean/moving_variance."""
    return l.get("keys") or (("/gamma:0", "/beta:0") if l["is_norm"] else ("/kernel:0", "/bias:0"))


class Model:
    """Keras-Model duck type whose numerics run in libfetalb200 (one fm_model handle)."""

    def __init__(self, input_shape, depth, n_base_filters, n_labels, initial_learning_rate, loss_function,
                 device=None, ndim=3, isensee_levels=None, dropout_rate=0.0, dropout_seed=0x5EED, mask_shape=None,
                 deconvolution=False, batch_normalization=False, label_wise_dice=False):
        lib = _lib.load()
        self._ctx = _lib.get_context(device)
        self.ndim = int(ndim)
        h = _lib.c_vp()
        self.trainable = True
        if isensee_levels is not None and self.ndim == 2:
            H, W, in_ch = [int(v) for v in input_shape]             # slices-as-channels (unet/isensee.py:38-39)
            spec = _lib.Isensee2DSpec(H, W, in_ch, int(depth), int(n_base_filters), int(isensee_levels), int(n_labels))
            _lib.check(lib.fm_model_create_isensee2d(self._ctx.handle, ctypes.byref(spec), ctypes.byref(h)))
            _lib.check(lib.fm_model_set_dropout(h, float(dropout_rate), int(dropout_seed)))
            self.input_shape = (None, H, W, in_ch)
            self.output_shape = (None, H, W, int(n_labels))
        elif isensee_levels is not None:
            in_ch, X, Y, Z = [int(v) for v in input_shape]
            spec = _lib.Isensee3DSpec(in_ch, X, Y, Z, int(depth), int(n_base_filters), int(isensee_levels), int(n_labels))
            _lib.check(lib.fm_model_create_isensee3d(self._ctx.handle, ctypes.byref(spec), ctypes.byref(h)))
            _lib.check(lib.fm_model_set_dropout(h, float(dropout_rate), int(dropout_seed)))
            self.input_shape = (None, in_ch, X, Y, Z)
            self.output_shape = (None, int(n_labels), X, Y, Z)
        elif self.ndim == 3:
            in_ch, X, Y, Z = [int(v) for v in input_shape]          # channels-first (unet3d/unet.py:9)
            spec = _lib.UNet3DSpec(in_ch, X, Y, Z, int(depth), int(n_base_filters), int(n_labels))
            _lib.check(lib.fm_model_create_unet3d_ex(self._ctx.handle, ctypes.byref(spec), (1 if deconvolution else 0) |
                                                     (2 if batch_normalization else 0), ctypes.byref(h)))
            self.input_shape = (None, in_ch, X, Y, Z)
            self.output_shape = (None, int(n_labels), X, Y, Z)
        else:
            H, W, in_ch = [int(v) for v in input_shape]             # slices-as-channels (unet/unet.py:49-50)
            spec = _lib.UNet2DSpec(H, W, in_ch, int(depth), int(n_base_filters), int(n_labels))
            _lib.check(lib.fm_model_create_unet2d_ex(self._ctx.handle, ctypes.byref(spec), (1 if deconvolution else 0) |
                                                     (2 if batch_normalization else 0), ctypes.byref(h)))
            if dropout_rate:                                         # SpatialDropout2D (unet/unet.py:60-61,76-77)
                _lib.check(lib.fm_model_set_dropout(h, float(dropout_rate), int(dropout_seed)))
            self.input_shape = (None, H, W, in_ch)
            self.output_shape = (None, H, W, int(n_labels))
        self._h = h
        self._lib = lib
        self.depth = int(depth)
        self.n_base_filters = int(n_base_filters)
        self.n_labels = int(n_labels)
        self.optimizer = _Optimizer(initial_learning_rate)
        # the second (weight mask) input of isensee2017.py:85-88: the loss argument is then the closure FACTORY
        self.mask_shape = None if mask_shape is None else tuple(int(v) for v in mask_shape)
        self.loss = loss_function
        self._loss_spec = device_loss_spec(loss_function, has_mask_input=self.mask_shape is not None)
        if self._loss_spec is not None:
            _lib.check(lib.fm_model_set_loss(h, int(self._loss_spec[0]), float(self._loss_spec[1]),
                                             float(self._loss_spec[2])))
        self.metrics = ['binary_accuracy', 'vod_coefficient']
        self.metrics_names = ['loss', 'binary_accuracy', 'vod_coefficient']
        if loss_function is not dice_coefficient_loss:
            self.metrics_names.append('dice_coefficient')
        # include_label_wise_dice_coefficients (unet3d/unet.py:71-75): one dice_coefficient per label channel, after the
        # others; 2D models take the label axis last ([B,H,W,n_labels]) - see label_dice_coefficient
        self.label_wise_dice = bool(label_wise_dice) and self.n_labels > 1
        if self.label_wise_dice:
            self.metrics_names += ['label_%d_dice_coef' % i for i in range(self.n_labels)]
        self.stop_training = False
        self.deconvolution = bool(deconvolution)
        self.batch_normalization = bool(batch_normalization)
        self.isensee_levels = isensee_levels
        self.name = ('isensee2017_model_3d' if self.ndim == 3 else 'isensee2017_model') if isensee_levels is not None \
            else ('unet_model_3d' if self.ndim == 3 else 'unet_model_2d')
        # layer table (Keras creation order; Keras would name them conv3d_1..conv3d_N)
        self.layers = []
        for i in range(lib.fm_model_num_layers(h)):
            name = ctypes.create_string_buffer(32)
            info = (ctypes.c_int64 * 5)()
            _lib.check(lib.fm_model_layer_info(h, i, name, info))
            code = int(info[2])                                      # 33 / 31, 22 / 21, 11; 0 norm; -1 BN moving statistics
            k = max(code, 0) // 10                                   # 33 / 31 -> 3, 22 / 21 -> 2, 11 -> 1, norm -> 0
            is_norm = code <= 0
            is_moving = code < 0                                     # (moving_mean, moving_variance) of the layer before
            is_deconv = k == 2                                       # Keras names them conv3d_transpose_<n>
            n_same = sum(1 for l in self.layers if (l["is_norm"], l["is_deconv"], l["is_moving"]) ==
                         (is_norm, is_deconv, is_moving)) + 1
            norm_name = "batch_normalization_%d" if batch_normalization else "instance_normalization_%d"
            self.layers.append(dict(index=i, name=name.value.decode(), is_norm=is_norm, is_deconv=is_deconv,
                                    is_moving=is_moving,
                                    keys=("/moving_mean:0", "/moving_variance:0") if is_moving else
                                    (("/gamma:0", "/beta:0") if is_norm else ("/kernel:0", "/bias:0")),
                                    keras_name=(norm_name if is_norm else
                                                ("conv%dd_transpose_%%d" if is_deconv else "conv%dd_%%d") % self.ndim) % n_same,
                                    cin=int(info[0]), cout=int(info[1]), k=k,
                                    kshape=(int(info[1]),) if is_norm else
                                    (k,) * self.ndim + (int(info[0]), int(info[1]))))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.fm_model_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ---- weights ---------------------------------------------------------------------------
    def count_params(self):
        return int(self._lib.fm_model_num_params(self._h))

    def get_weights(self):
        """[kernel_1, bias_1, kernel_2, ...] in Keras layout (k,k,k,Cin,Cout) / (Cout,)."""
        out = []
        for l in self.layers:
            k = np.empty(l["kshape"], np.float32)
            b = np.empty((l["cout"],), np.float32)
            _lib.check(self._lib.fm_model_get_weights(self._h, l["index"], _lib.fptr(k), _lib.fptr(b)))
            out += [k, b]
        return out

    def set_weights(self, weights):
        assert len(weights) == 2 * len(self.layers), "expected %d arrays" % (2 * len(self.layers))
        for l in self.layers:
            k = _lib.f32c(weights[2 * l["index"]])
            b = _lib.f32c(weights[2 * l["index"] + 1])
            assert k.shape == l["kshape"], (l["name"], k.shape)
            assert b.shape == (l["cout"],), (l["name"], b.shape)
            _lib.check(self._lib.fm_model_set_weights(self._h, l["index"], _lib.fptr(k), _lib.fptr(b)))

    def get_gradients(self):
        """Gradients of the last train step (Keras layout) - test hook."""
        out = []
        for l in self.layers:
            k = np.empty(l["kshape"], np.float32)
            b = np.empty((l["cout"],), np.float32)
            _lib.check(self._lib.fm_model_get_grads(self._h, l["index"], _lib.fptr(k), _lib.fptr(b)))
            out += [k, b]
        return out

    def set_named_weights(self, named):
        """`named`: {'<layer>/kernel': ..., '<layer>/bias': ...} keyed by our layer names (enc0a ...)."""
        ws = []
        for l in self.layers:
            if l.get("is_moving"):  # '<conv>_moving' pseudo-layer of a BatchNormalization
                base = l["name"][:-len("_moving")]
                ws += [named[base + "/moving_mean"], named[base + "/moving_variance"]]
            elif l["is_norm"]:      # '<conv>_norm' pseudo-layer: kernel slot = gamma, bias slot = beta
                base = l["name"][:-len("_norm")]
                ws += [named[base + "/gamma"], named[base + "/beta"]]
            else:
                ws += [named[l["name"] + "/kernel"], named[l["name"] + "/bias"]]
        self.set_weights(ws)

    def init_glorot_uniform(self, seed=0):
        """Keras default initialisation (glorot_uniform kernels, zero biases; SURVEY.md App. A.2)."""
        rng = np.random.default_rng(seed)
        ws = []
        for l in self.layers:
            if l.get("is_moving"):                                  # moving_mean = 0, moving_variance = 1
                ws += [np.zeros((l["cout"],), np.float32), np.ones((l["cout"],), np.float32)]
                continue
            if l["is_norm"]:                                        # gamma = 1, beta = 0 (SURVEY.md App. A.6)
                ws += [np.ones((l["cout"],), np.float32), np.zeros((l["cout"],), np.float32)]
                continue
            rf = l["k"] ** self.ndim
            limit = np.sqrt(6.0 / (rf * l["cin"] + rf * l["cout"]))
            ws.append(rng.uniform(-limit, limit, size=l["kshape"]).astype(np.float32))
            ws.append(np.zeros((l["cout"],), np.float32))
        self.set_weights(ws)

    def _weight_arrays(self):
        arrays = {}
        for l, (k, b) in zip(self.layers, zip(*[iter(self.get_weights())] * 2)):
            arrays[l["keras_name"] + _slot_keys(l)[0]] = k
            arrays[l["keras_name"] + _slot_keys(l)[1]] = b
        arrays["__config__"] = np.array(list(self.input_shape[1:]) + [self.depth, self.n_base_filters, self.n_labels])
        # builder name + its extra arguments, so that load_old_model can rebuild the right family
        arrays["__builder__"] = np.array(getattr(self, "name", "unet_model_3d"))
        arrays["__isensee_levels__"] = np.array(int(getattr(self, "isensee_levels", 0) or 0))
        arrays["__deconvolution__"] = np.array(int(getattr(self, "deconvolution", False)))
        arrays["__batch_normalization__"] = np.array(int(getattr(self, "batch_normalization", False)))
        arrays["__label_wise__"] = np.array(int(getattr(self, "label_wise_dice", False)))
        return arrays

    def save_weights(self, path):
        """HDF5 is absent in this image (SURVEY.md §5): weights go to an .npz keyed by Keras layer names."""
        with open(path, "wb") as f:   # keep the caller's file name (e.g. '...-epoch01-loss-0.5.h5')
            np.savez(f, **self._weight_arrays())

    def get_optimizer_state(self):
        """(iterations, lr, [m_kernel, m_bias, v_kernel, v_bias] per layer in Keras layout) - what Keras'
        model.save() stores besides the weights."""
        moments = []
        for l in self.layers:
            mk, vk = np.empty(l["kshape"], np.float32), np.empty(l["kshape"], np.float32)
            mb, vb = np.empty((l["cout"],), np.float32), np.empty((l["cout"],), np.float32)
            _lib.check(self._lib.fm_model_get_adam_state(self._h, l["index"], _lib.fptr(mk), _lib.fptr(mb),
                                                         _lib.fptr(vk), _lib.fptr(vb)))
            moments.append((mk, mb, vk, vb))
        return int(self._lib.fm_model_get_iterations(self._h)), float(self.optimizer.lr), moments

    def set_optimizer_state(self, iterations, lr, moments):
        assert len(moments) == len(self.layers)
        for l, (mk, mb, vk, vb) in zip(self.layers, moments):
            mk, mb, vk, vb = (_lib.f32c(a) for a in (mk, mb, vk, vb))
            assert mk.shape == l["kshape"] == vk.shape and mb.shape == (l["cout"],) == vb.shape, l["name"]
            _lib.check(self._lib.fm_model_set_adam_state(self._h, l["index"], _lib.fptr(mk), _lib.fptr(mb),
                                                         _lib.fptr(vk), _lib.fptr(vb)))
        _lib.check(self._lib.fm_model_set_iterations(self._h, int(iterations)))
        self.optimizer.lr = float(lr)

    def save(self, path):
        """Keras' model.save(): weights AND optimizer state (Adam moments, iteration count, the current - possibly
        plateau-reduced - learning rate), so that load_old_model(...) + train_model(...) resumes like the reference's
        load_model() path (fetal/train_fetal.py:25-28, fetal_net/training.py:45-65). save_weights stays weights-only."""
        arrays = self._weight_arrays()
        it, lr, moments = self.get_optimizer_state()
        arrays["__iterations__"] = np.array(it)
        arrays["__lr__"] = np.array(lr)
        for l, (mk, mb, vk, vb) in zip(self.layers, moments):
            arrays["__adam_m__/" + l["keras_name"] + "/kernel"] = mk
            arrays["__adam_m__/" + l["keras_name"] + "/bias"] = mb
            arrays["__adam_v__/" + l["keras_name"] + "/kernel"] = vk
            arrays["__adam_v__/" + l["keras_name"] + "/bias"] = vb
        with open(path, "wb") as f:
            np.savez(f, **arrays)

    def load_optimizer_state(self, path):
        """Restores what save() wrote; returns False for a weights-only file (the optimizer then starts fresh)."""
        from .. import keras_h5
        if keras_h5.is_hdf5(path):
            return False
        with np.load(path) as z:
            if "__iterations__" not in z.files:
                return False
            moments = [tuple(np.asarray(z["__adam_%s__/%s/%s" % (mv, l["keras_name"], kb)])
                             for mv, kb in (("m", "kernel"), ("m", "bias"), ("v", "kernel"), ("v", "bias")))
                       for l in self.layers]
            self.set_optimizer_state(int(z["__iterations__"]), float(z["__lr__"]), moments)
        return True

    def load_weights(self, path):
        """Reads the .npz written by save_weights (whatever the file is called), or - where h5py is installed - a
        Keras .h5 checkpoint of the reference directly (fetal_net.keras_h5; layers matched by creation order)."""
        from .. import keras_h5
        if keras_h5.is_hdf5(path):
            z = keras_h5.to_npz_arrays(keras_h5.read_keras_h5_weights(path))
            ws = self._weights_from_mapping(z)
        else:
            with np.load(path) as z:
                ws = self._weights_from_mapping(z)
        self.set_weights(ws)

    def _weights_from_mapping(self, z):
        ws = []
        for l in self.layers:
            ws += [np.asarray(z[l["keras_name"] + _slot_keys(l)[0]]), np.asarray(z[l["keras_name"] + _slot_keys(l)[1]])]
        return ws

    def set_fast_inference(self, fast=True):
        """predict / evaluate / patch_wise_prediction on the three-issuer conv mode of the training passes: about a quarter
        more conv throughput, results no longer bit-identical from run to run (default: reproducible)."""
        _lib.check(self._lib.fm_model_set_inference_mode(self._h, 1 if fast else 0))

    def reset_optimizer(self):
        _lib.check(self._lib.fm_model_reset_optimizer(self._h))

    # ---- inference -------------------------------------------------------------------------
    def predict(self, x, batch_size=32, verbose=0):
        if self.mask_shape is not None and isinstance(x, (list, tuple)):
            x = x[0]                                               # the mask input only feeds the loss
        x = _lib.f32c(x)
        assert x.shape[1:] == self.input_shape[1:], "expected [B,%s], got %s" % (self.input_shape[1:], x.shape)
        out = np.empty((x.shape[0],) + self.output_shape[1:], np.float32)
        for b0 in range(0, x.shape[0], batch_size):
            xb = x[b0:b0 + batch_size]
            yb = out[b0:b0 + batch_size]
            _lib.check(self._lib.fm_predict(self._h, _lib.fptr(xb), int(xb.shape[0]), _lib.fptr(yb)))
        return out

    # ---- training --------------------------------------------------------------------------
    def _check_loss(self):
        if not self.trainable:
            raise NotImplementedError("%s: training is on the §8 'next' list (forward / inference is built)" % self.name)
        if self._loss_spec is None:
            raise NotImplementedError("loss %r: dice_coefficient_loss, dice_and_xent and dice_and_xent_mask (with "
                                      "mask_shape) are built on the device path" % (self.loss,))

    def _split_mask(self, x):
        """`[x, mask]` -> x after handing the weight mask to the device (two-input model, isensee2017.py:85-88)."""
        if self.mask_shape is None:
            return x
        assert isinstance(x, (list, tuple)) and len(x) == 2, "this model takes [x, weight_mask] (mask_shape was given)"
        x, mask = x
        mask = _lib.f32c(mask)
        assert mask.shape[1:] == self.mask_shape and mask.shape[0] == len(x), (mask.shape, self.mask_shape)
        assert int(np.prod(self.mask_shape)) == int(np.prod(self.output_shape[1:])), "one weight per output voxel"
        _lib.check(self._lib.fm_model_set_weight_mask(self._h, _lib.fptr(mask), int(mask.shape[0])))
        return x

    def train_on_batch(self, x, y, **kw):
        self._check_loss()
        x = self._split_mask(x)
        x, y = _lib.f32c(x), _lib.f32c(y)
        assert x.shape[1:] == self.input_shape[1:] and y.shape == (x.shape[0],) + self.output_shape[1:], (x.shape, y.shape)
        m = np.zeros(4, np.float32)
        _lib.check(self._lib.fm_train_step(self._h, _lib.fptr(x), _lib.fptr(y), int(x.shape[0]),
                                           float(self.optimizer.lr), _lib.fptr(m)))
        return self._metrics(m)

    def label_dice(self):
        """Dice of each label over the batch of the last training step / evaluation (fm_model_label_dice)."""
        d = np.zeros(self.n_labels, np.float32)
        _lib.check(self._lib.fm_model_label_dice(self._h, _lib.fptr(d), self.n_labels))
        return d

    def _metrics(self, m):
        """metrics_names' values from the four device metrics (+ the label-wise Dice)."""
        out = [float(v) for v in m[:len(self.metrics_names) - (self.n_labels if self.label_wise_dice else 0)]]
        return out + ([float(v) for v in self.label_dice()] if self.label_wise_dice else [])

    def train_on_sampled_batch(self, sampler, cases, corners, aug=None, warp=None):
        """One training step on samples cut on the device by a `fetal_net.device_sampler.DeviceSampler`
        (next(generator) + train_on_batch of fetal_net/training.py:110-124 with no host batch): fm_train_step_sampled.
        aug / warp: per-sample fm_sample_aug / fm_sample_warp arrays (a data-parallel rank passes its slice); with both
        None the sampler draws them from its `device_augment`."""
        from ..device_sampler import _c_array, _check_one_label
        self._check_loss()
        _check_one_label(self)
        cases, corners = _lib.i32x(cases), _lib.i32x(corners)
        if aug is None and warp is None:
            aug, warp = sampler.draw_augment(cases.size)
        ti, ts, pi, ps = sampler._args()
        m = np.zeros(4, np.float32)
        _lib.check(self._lib.fm_train_step_sampled_warp(
            self._h, sampler._handle, _lib.i32ptr(cases), _lib.i32ptr(corners), _c_array(_lib.SampleAug, aug),
            _c_array(_lib.SampleWarp, warp), int(cases.size), ti, ts, pi, ps, float(self.optimizer.lr), _lib.fptr(m)))
        return [float(v) for v in m[:len(self.metrics_names)]]

    def test_on_batch(self, x, y, **kw):
        if not self.trainable:                                      # metrics on the host from .predict
            from .. import metrics as _m
            p = self.predict(x)
            return [_m.dice_coefficient_loss(y, p), _m.binary_accuracy(y, p), _m.vod_coefficient(y, p)]
        self._check_loss()
        x = self._split_mask(x)
        x, y = _lib.f32c(x), _lib.f32c(y)
        m = np.zeros(4, np.float32)
        _lib.check(self._lib.fm_evaluate(self._h, _lib.fptr(x), _lib.fptr(y), int(x.shape[0]), _lib.fptr(m)))
        return self._metrics(m)

    def evaluate(self, x, y, batch_size=32, verbose=0):
        """Keras semantics: per-batch metrics averaged with batch-size weights."""
        tot, n = np.zeros(len(self.metrics_names)), 0
        two = getattr(self, "mask_shape", None) is not None and isinstance(x, (list, tuple))
        for b0 in range(0, len(y), batch_size):
            xb = [a[b0:b0 + batch_size] for a in x] if two else x[b0:b0 + batch_size]
            r = self.test_on_batch(xb, y[b0:b0 + batch_size])
            nb = len(y[b0:b0 + batch_size])
            tot += np.asarray(r) * nb
            n += nb
        return list(tot / max(n, 1))

    def fit_generator(self, generator, steps_per_epoch, epochs=1, validation_data=None, validation_steps=None,
                      max_queue_size=10, workers=1, use_multiprocessing=False, callbacks=None, verbose=1,
                      initial_epoch=0, **kw):
        """The training driver of fetal_net/training.py:110-124 (main-thread train_on_batch loop, per-epoch
        validation, Keras callback protocol: on_train_begin / on_epoch_begin / on_epoch_end / on_train_end)."""
        callbacks = list(callbacks or [])
        history = {}
        for cb in callbacks:
            cb.set_model(self)
            cb.on_train_begin()
        self.stop_training = False
        for epoch in range(initial_epoch, epochs):
            for cb in callbacks:
                cb.on_epoch_begin(epoch)
            tot, n = np.zeros(len(self.metrics_names)), 0
            on_device = hasattr(generator, "train_on_next_batch")   # DeviceSampler: the batch never visits the host
            for _ in range(int(steps_per_epoch)):
                if on_device:
                    r, nb = generator.train_on_next_batch(self), generator.batch_size
                else:
                    x, y = next(generator)[:2]
                    r, nb = self.train_on_batch(x, y), len(y)
                tot += np.asarray(r) * nb
                n += nb
            logs = {k: float(v) for k, v in zip(self.metrics_names, tot / max(n, 1))}
            if validation_data is not None and validation_steps:
                vt, vn = np.zeros(len(self.metrics_names)), 0
                for _ in range(int(validation_steps)):
                    x, y = next(validation_data)[:2]
                    r = self.test_on_batch(x, y)
                    vt += np.asarray(r) * len(y)
                    vn += len(y)
                logs.update({"val_" + k: float(v) for k, v in zip(self.metrics_names, vt / max(vn, 1))})
            logs["lr"] = float(self.optimizer.lr)
            for k, v in logs.items():
                history.setdefault(k, []).append(v)
            if verbose:
                print("Epoch %d/%d - " % (epoch + 1, epochs) + " - ".join("%s: %.4f" % kv for kv in logs.items()))
            for cb in callbacks:
                cb.on_epoch_end(epoch, logs)
            if self.stop_training:
                break
        for cb in callbacks:
            cb.on_train_end()
        return history

    def summary(self, print_fn=print):
        print_fn("%-10s %-12s %6s %6s %3s %10s" % ("layer", "keras name", "Cin", "Cout", "k", "params"))
        for l in self.layers:
            print_fn("%-14s %-26s %6d %6d %3d %10d" % (l["name"], l["keras_name"], l["cin"], l["cout"], l["k"],
                                                       2 * l["cout"] if l["is_norm"] else
                                                       l["k"] ** self.ndim * l["cin"] * l["cout"] + l["cout"]))
        print_fn("Total params: %d" % self.count_params())

    def to_json(self):
        import json
        return json.dumps(dict(class_name=self.name, input_shape=self.input_shape[1:], depth=self.depth,
                               n_base_filters=self.n_base_filters, n_labels=self.n_labels))


def unet_model_3d(input_shape, pool_size=(2, 2, 2), n_labels=1, initial_learning_rate=0.00001, deconvolution=False,
                  depth=4, n_base_filters=32, include_label_wise_dice_coefficients=False,
                  batch_normalization=False, activation_name="sigmoid", loss_function=dice_coefficient_loss,
                  **kargs):
    """Same signature and defaults as the reference builder (unet3d/unet.py:17-20); unknown kwargs
    (dropout_rate, mask_shape, old_model_path, ... — train_fetal.py:33-39) are swallowed like there."""
    if tuple(pool_size) != (2, 2, 2):
        raise NotImplementedError("pool_size %r: the B200 path builds the reference default (2,2,2)" % (pool_size,))
    if activation_name != "sigmoid":
        raise NotImplementedError("activation_name %r: only 'sigmoid' is built" % activation_name)
    return Model(input_shape=input_shape, depth=depth, n_base_filters=n_base_filters, n_labels=n_labels,
                 initial_learning_rate=initial_learning_rate, loss_function=loss_function,
                 device=kargs.get("device"), deconvolution=deconvolution, batch_normalization=batch_normalization,
                 label_wise_dice=include_label_wise_dice_coefficients)


def unet_model_2d(input_shape, pool_size=(2, 2), n_labels=1, initial_learning_rate=0.00001, deconvolution=False,
                  depth=4, n_base_filters=32, include_label_wise_dice_coefficients=False,
                  batch_normalization=False, activation_name="sigmoid", loss_function=dice_coefficient_loss,
                  dropout_rate=0, **kargs):
    """Same signature and defaults as the reference 2D / 2.5D builder (fetal_net/model/unet/unet.py:22-25):
    `input_shape=(H, W, D)` with the slices (and previous-slice truth) as channels. `dropout_rate` > 0 puts a
    SpatialDropout2D behind the first conv block of every level in training steps (unet/unet.py:60-61,76-77; keep
    masks from the library's counter-based hash, `dropout_seed` kwarg)."""
    if tuple(pool_size) != (2, 2):
        raise NotImplementedError("pool_size %r: the B200 path builds the reference default (2,2)" % (pool_size,))
    if activation_name != "sigmoid":
        raise NotImplementedError("activation_name %r: only 'sigmoid' is built" % activation_name)
    if batch_normalization and dropout_rate:
        raise NotImplementedError("batch_normalization=True together with dropout_rate > 0 is not built")
    return Model(input_shape=input_shape, depth=depth, n_base_filters=n_base_filters, n_labels=n_labels,
                 initial_learning_rate=initial_learning_rate, loss_function=loss_function,
                 device=kargs.get("device"), ndim=2, dropout_rate=dropout_rate or 0.0,
                 dropout_seed=kargs.get("dropout_seed", 0x5EED), deconvolution=deconvolution,
                 batch_normalization=batch_normalization, label_wise_dice=include_label_wise_dice_coefficients)


def isensee2017_model_3d(input_shape=(1, 128, 128, 128), n_base_filters=16, depth=5, dropout_rate=0.3,
                         n_segmentation_levels=1, n_labels=1, optimizer=None, initial_learning_rate=5e-4,
                         loss_function=dice_coefficient_loss, activation_name="sigmoid", mask_shape=None, **kargs):
    """Same signature and defaults as the reference builder (fetal_net/model/unet3d/isensee2017.py:15-18).
    `dropout_rate` drives SpatialDropout3D between the two convs of each context module in training steps
    (identity at inference); the keep masks come from a counter-based hash (`dropout_seed` kwarg), not TF's RNG."""
    if activation_name != "sigmoid":
        raise NotImplementedError("activation_name %r: only 'sigmoid' is built" % activation_name)
    return Model(input_shape=input_shape, depth=depth, n_base_filters=n_base_filters, n_labels=n_labels,
                 initial_learning_rate=initial_learning_rate, loss_function=loss_function,
                 device=kargs.get("device"), ndim=3, isensee_levels=n_segmentation_levels,
                 dropout_rate=dropout_rate or 0.0, dropout_seed=kargs.get("dropout_seed", 0x5EED),
                 mask_shape=mask_shape)


def isensee2017_model(input_shape=(4, 128, 128, 128), n_base_filters=16, depth=5, dropout_rate=0.3,
                      n_segmentation_levels=3, n_labels=1, optimizer=None, initial_learning_rate=5e-4,
                      loss_function=dice_coefficient_loss, activation_name="sigmoid", summation=False, **kargs):
    """Same signature and defaults as the reference 2D builder (fetal_net/model/unet/isensee.py:14-16):
    `input_shape=(H, W, D)` with the slices as channels. With `summation=False` (the reference default) only the finest
    1x1 head reaches the output (isensee.py:81-82) - Keras drops the coarser, unconnected heads from the model, so they
    hold no weights here either; `summation=True` sums the `n_segmentation_levels` heads coarse to fine through
    UpSampling2D (isensee.py:69-80)."""
    if activation_name != "sigmoid":
        raise NotImplementedError("activation_name %r: only 'sigmoid' is built" % activation_name)
    if len(input_shape) != 3:
        raise ValueError("isensee2017_model takes input_shape=(H, W, slices); got %r" % (input_shape,))
    return Model(input_shape=input_shape, depth=depth, n_base_filters=n_base_filters, n_labels=n_labels,
                 initial_learning_rate=initial_learning_rate, loss_function=loss_function,
                 device=kargs.get("device"), ndim=2, isensee_levels=n_segmentation_levels if summation else 1,
                 dropout_rate=dropout_rate or 0.0, dropout_seed=kargs.get("dropout_seed", 0x5EED))
