"""Training driver with the reference's names (fetal_net/training.py): get_callbacks, load_old_model,
train_model, step_decay. The callbacks are small host-side re-expressions of the Keras ones the
reference wires up (training.py:26-42); the step itself is Model.train_on_batch -> fm_train_step."""
import csv
import glob
import math
import os
from functools import partial

import numpy as np

from . import metrics as _metrics
from . import model as _model_ns


def step_decay(epoch, initial_lrate, drop, epochs_drop):
    # training.py:22-23
    return initial_lrate * math.pow(drop, math.floor((1 + epoch) / float(epochs_drop)))


class Callback:
    def set_model(self, model):
        self.model = model

    def on_train_begin(self, logs=None):
        pass

    def on_train_end(self, logs=None):
        pass

    def on_epoch_begin(self, epoch, logs=None):
        pass

    def on_epoch_end(self, epoch, logs=None):
        pass


class ModelCheckpoint(Callback):
    """Keras ModelCheckpoint(save_best_only=True, monitor='val_loss') with the reference's file pattern
    (training.py:30-32, SURVEY.md App. A.12)."""

    def __init__(self, filepath, monitor='val_loss', save_best_only=True, verbose=0):
        self.filepath, self.monitor, self.save_best_only, self.verbose = filepath, monitor, save_best_only, verbose
        self.best = np.inf

    def on_epoch_end(self, epoch, logs=None):
        logs = logs or {}
        cur = logs.get(self.monitor)
        if self.save_best_only and (cur is None or not cur < self.best):
            return
        if cur is not None:
            self.best = cur
        path = self.filepath.format(epoch=epoch + 1, **logs)
        self.model.save(path)
        if self.verbose:
            print("Epoch %05d: saving model to %s" % (epoch + 1, path))


class CSVLogger(Callback):
    def __init__(self, filename, append=False):
        self.filename, self.append, self.keys = filename, append, None

    def on_epoch_end(self, epoch, logs=None):
        logs = logs or {}
        new = not (self.append and os.path.exists(self.filename)) and self.keys is None
        if self.keys is None:
            self.keys = sorted(logs.keys())
        with open(self.filename, "w" if new else "a", newline="") as f:
            w = csv.writer(f)
            if new:
                w.writerow(["epoch"] + self.keys)
            w.writerow([epoch] + [logs.get(k) for k in self.keys])


class LearningRateScheduler(Callback):
    def __init__(self, schedule):
        self.schedule = schedule

    def on_epoch_begin(self, epoch, logs=None):
        self.model.optimizer.lr = float(self.schedule(epoch))


class ReduceLROnPlateau(Callback):
    def __init__(self, monitor='val_loss', factor=0.1, patience=10, verbose=0, min_delta=1e-4, min_lr=0):
        self.monitor, self.factor, self.patience, self.verbose = monitor, factor, patience, verbose
        self.min_delta, self.min_lr = min_delta, min_lr
        self.best, self.wait = np.inf, 0

    def on_epoch_end(self, epoch, logs=None):
        cur = (logs or {}).get(self.monitor)
        if cur is None:
            return
        if cur < self.best - self.min_delta:
            self.best, self.wait = cur, 0
            return
        self.wait += 1
        if self.wait >= self.patience:
            new_lr = max(self.model.optimizer.lr * self.factor, self.min_lr)
            if self.verbose:
                print("Epoch %05d: ReduceLROnPlateau reducing learning rate to %g" % (epoch + 1, new_lr))
            self.model.optimizer.lr = new_lr
            self.wait = 0


class EarlyStopping(Callback):
    def __init__(self, monitor='val_loss', patience=0, verbose=0):
        self.monitor, self.patience, self.verbose = monitor, patience, verbose
        self.best, self.wait = np.inf, 0

    def on_epoch_end(self, epoch, logs=None):
        cur = (logs or {}).get(self.monitor)
        if cur is None:
            return
        if cur < self.best:
            self.best, self.wait = cur, 0
        else:
            self.wait += 1
            if self.wait >= self.patience:
                self.model.stop_training = True


def get_callbacks(model_file, initial_learning_rate=0.0001, learning_rate_drop=0.5, learning_rate_epochs=None,
                  learning_rate_patience=50, logging_file="training.log", verbosity=1,
                  early_stopping_patience=None):
    # training.py:26-42 — same order: checkpoint, csv, lr schedule | plateau, early stopping
    callbacks = list()
    callbacks.append(ModelCheckpoint(model_file + '-epoch{epoch:02d}-loss{val_loss:.3f}-acc{val_binary_accuracy:.3f}.h5',
                                     save_best_only=True, verbose=verbosity, monitor='val_loss'))
    callbacks.append(CSVLogger(logging_file, append=True))
    if learning_rate_epochs:
        callbacks.append(LearningRateScheduler(partial(step_decay, initial_lrate=initial_learning_rate,
                                                       drop=learning_rate_drop, epochs_drop=learning_rate_epochs)))
    else:
        callbacks.append(ReduceLROnPlateau(factor=learning_rate_drop, patience=learning_rate_patience,
                                           verbose=verbosity))
    if early_stopping_patience:
        callbacks.append(EarlyStopping(verbose=verbosity, patience=early_stopping_patience))
    return callbacks


def get_last_model_path(model_file_path):
    # fetal/utils.py:42-43 — newest mtime among <model_file>*.h5
    return sorted(glob.glob(model_file_path + '*.h5'), key=os.path.getmtime)[-1]


def load_old_model(model_file, verbose=True, config=None):
    """training.py:45-86: Keras could rebuild a model from the HDF5 alone; our container stores weights +
    the builder arguments, so the model is rebuilt from the stored config (or from `config`)."""
    if verbose:
        print("Loading pre-trained model")
    from . import keras_h5
    if keras_h5.is_hdf5(model_file):
        # a genuine Keras .h5 of the reference: the architecture comes from the config (the reference's manual-build
        # fallback, training.py:72-84), the weights through the h5py bridge
        if config is None:
            raise ValueError("load_old_model(%r): a Keras HDF5 checkpoint needs `config` (model_name, input_shape) to "
                             "rebuild the architecture" % (model_file,))
        loss = getattr(_metrics, config.get('loss', 'dice_coefficient_loss'))
        m = getattr(_model_ns, config['model_name'])(input_shape=config['input_shape'],
                                                     initial_learning_rate=config.get('initial_learning_rate', 1e-5),
                                                     loss_function=loss,
                                                     **({'dropout_rate': config['dropout_rate']}
                                                        if 'dropout_rate' in config else {}))
        m.load_weights(model_file)
        return m
    with np.load(model_file) as z:
        cfg = [int(v) for v in z["__config__"]]
        builder_name = str(z["__builder__"]) if "__builder__" in z.files else None
        levels = int(z["__isensee_levels__"]) if "__isensee_levels__" in z.files else 0
        deconv = bool(int(z["__deconvolution__"])) if "__deconvolution__" in z.files else False
        bnorm = bool(int(z["__batch_normalization__"])) if "__batch_normalization__" in z.files else False
        label_wise = bool(int(z["__label_wise__"])) if "__label_wise__" in z.files else False
    loss = _metrics.dice_coefficient_loss
    lr = 1e-5
    if config is not None:
        loss = getattr(_metrics, config.get('loss', 'dice_coefficient_loss'))
        lr = config.get('initial_learning_rate', lr)
    if builder_name is None:                        # archives written before the builder name was stored
        builder_name = 'unet_model_3d' if len(cfg) == 7 else 'unet_model_2d'   # (C,X,Y,Z) vs (H,W,D)
    kwargs = dict(input_shape=tuple(cfg[:-3]), depth=cfg[-3], n_base_filters=cfg[-2], n_labels=cfg[-1],
                  initial_learning_rate=lr, loss_function=loss)
    if deconv:
        kwargs['deconvolution'] = True
    if bnorm:
        kwargs['batch_normalization'] = True
    if label_wise:
        kwargs['include_label_wise_dice_coefficients'] = True
    if builder_name in ('isensee2017_model_3d', 'isensee2017_model'):
        kwargs['n_segmentation_levels'] = levels
        if builder_name == 'isensee2017_model':     # the 2D builder: `levels` heads reach the output only when summed
            kwargs['summation'] = levels > 1
    if builder_name != 'unet_model_3d' and config is not None and 'dropout_rate' in config:
        kwargs['dropout_rate'] = config['dropout_rate']
    m = getattr(_model_ns, builder_name)(**kwargs)
    m.load_weights(model_file)
    # Keras' load_model also restores the optimizer (Adam moments, iterations, the current learning rate): a resumed
    # run continues where the checkpoint stopped. Weights-only archives start a fresh optimizer.
    m.load_optimizer_state(model_file)
    return m


def train_model(model, model_file, training_generator, validation_generator, steps_per_epoch, validation_steps,
                initial_learning_rate=0.001, learning_rate_drop=0.5, learning_rate_epochs=None, n_epochs=500,
                learning_rate_patience=20, early_stopping_patience=None, output_folder='.'):
    # training.py:89-124
    return model.fit_generator(generator=training_generator, steps_per_epoch=steps_per_epoch, epochs=n_epochs,
                               validation_data=validation_generator, validation_steps=validation_steps,
                               max_queue_size=15, workers=1, use_multiprocessing=False,
                               callbacks=get_callbacks(model_file, initial_learning_rate=initial_learning_rate,
                                                       learning_rate_drop=learning_rate_drop,
                                                       learning_rate_epochs=learning_rate_epochs,
                                                       learning_rate_patience=learning_rate_patience,
                                                       early_stopping_patience=early_stopping_patience,
                                                       logging_file=os.path.join(output_folder, 'training')))
