"""Training batches cut on the device (SURVEY.md §8f rank 3).

Device-resident counterpart of the reference's training generator (`data_generator` -> `add_data` -> `extract_patch` ->
`get_patch_from_3d_data`, `convert_data`; fetal_net/generator.py:222-348,380-401) for the `augment=None` path: the cases
are uploaded once (`fm_volset_set_case`), the HOST keeps making every random decision with the reference's own call
sequence on the global `random` / `np.random` generators -

    index  = next(index_generator)                  # random.sample per epoch (np.random.seed() first), or in order
    corner = [np.random.randint(0, high) for high in truth.shape - patch_shape]          # generator.py:266-269
    drop_easy_patches: np.random.random() against 1 - |mean(truth[16:-16, 16:-16, :]) - 0.5|      # :307-310
    skip_blank: keep the sample only if np.any(truth != 0)                                        # :323

- and the device cuts the whole batch with one kernel (`sample_patches_kernel`, csrc/sampler.cu): the data patch, the
target slice(s) at `truth_index`, the previous-truth slice(s) at `prev_truth_index` appended as extra input channels
(generator.py:305-306), slices that stick out of the volume completed with the nearest edge sample
(utils/patches.py:75-91). Same seeds => the same (case, corner) sequence and bit-identical float32 batches as the
reference generator (tests/golden/sampler_golden.npz is frozen from the unmodified reference).

`DeviceSampler` is an iterator yielding `(x, y)` like the reference generator (so `fit_generator` takes it unchanged);
`train_on_next_batch(model)` skips the host round trip altogether (`fm_train_step_sampled`: the batch goes straight
into the model's input buffers; 32 bytes of arguments per sample cross the bus, 68 more with a warp).

Not covered here, by design: the reference's nilearn / imgaug augmentation pipeline (`augment_data`,
generator.py:271-295), `truth_downsample`, masks and `categorical=True` - those stay on the reference's host generator
(reachable through the overlay, see fetal_net/__init__.py). The device offers its OWN augmentations instead, off by
default, parameters drawn per sample on the host (`device_augment`):

    flip=True               one of the 8 axis-flip combinations (data, previous truth and target alike)
    intensity=(lo, hi)      data *= uniform(lo, hi)
    noise_sigma=s           data += s * N(0, 1) (counter-based hash on the device)
    rotate=(sx, sy, sz)     degrees, one normal draw per axis
    scale=(sx, sy, sz)      factor 1 + N(0, s) per axis, clipped to [0.5, 2] (above 1 enlarges structures)
    translate=(sx, sy, sz)  voxels, one normal draw per axis
    elastic=dict(alpha=a or (ax, ay, az), grid=G)   smooth random displacement of up to alpha voxels per axis,
                            trilinear between G x G x G hashed control points (G in 2..8)

The last four form a warp (`sample_patches_warp_kernel`, fm_sample_warp in include/fetal_b200.h): every element of the
sample reads the volume at s = c + t + M (q + d(q) - c), q the position the unwarped cut reads, c the centre of the data
box, M = Rz Ry Rx diag(1/sx, 1/sy, 1/sz), t the offset and d the elastic displacement; data channels are interpolated
trilinearly, target and previous-truth channels take the nearest sample, both with edge replication. This is the
library's own augmentation, not the reference's nilearn / imgaug pipeline; oracle/sampler_oracle.py states it in NumPy.
`skip_blank` and `drop_easy_patches` still decide on the UNWARPED truth patch, on the host, in the reference's draw
order. The draws per batch: the flip / intensity / noise-seed draws of every sample first (the same np.random calls as
without a warp), then per sample three angles, three scale factors, three offsets and the elastic seed, each only when
its key is present; without the warp keys the np.random stream is that of the unwarped sampler.
"""
import ctypes
import math
import random

import numpy as np

from . import _lib


def random_list_generator(index_list):
    """generator.py:201-204, including its np.random.seed() at the start of every pass."""
    while True:
        np.random.seed()
        yield from random.sample(index_list, len(index_list))


def list_generator(index_list):
    """generator.py:207-209."""
    while True:
        yield from index_list


class PatchDraws:
    """The host half: which (case, corner) samples make up the next batch. No device needed."""

    def __init__(self, truth_list, index_list, batch_size=1, patch_shape=None, shuffle_index_list=True,
                 skip_blank=True, truth_index=-1, truth_size=1, prev_truth_index=None, prev_truth_size=None,
                 drop_easy_patches=False, is3d=False, categorical=False, augment=None, truth_downsample=None):
        if augment is not None:
            raise NotImplementedError("DeviceSampler covers the augment=None path; the nilearn/imgaug pipeline of "
                                      "generator.py:271-295 stays on the reference's host generator. The on-device "
                                      "route is DeviceSampler(device_augment=...): flips, intensity, noise, rotate, "
                                      "scale, translate and elastic, the library's own augmentation")
        if categorical:
            raise NotImplementedError("categorical=True (to_categorical targets) is not part of the soft-Dice path")
        if truth_downsample is not None and truth_downsample > 1:
            raise NotImplementedError("truth_downsample is not supported by the device sampler")
        if patch_shape is None:
            raise ValueError("patch_shape is required")
        self.patch_shape = tuple(int(v) for v in patch_shape)
        self.batch_size = int(batch_size)
        self.skip_blank = bool(skip_blank)
        self.truth_index, self.truth_size = int(truth_index), int(truth_size)
        self.prev_truth_index = None if prev_truth_index is None else int(prev_truth_index)
        self.prev_truth_size = 0 if prev_truth_index is None else int(1 if prev_truth_size is None else prev_truth_size)
        self.drop_easy_patches = bool(drop_easy_patches)
        self.is3d = bool(is3d)
        self._index_generator = (random_list_generator if shuffle_index_list else list_generator)(list(index_list))
        # host copies of the truth volumes: the skip_blank / drop_easy_patches decisions are host decisions
        self._truth = [np.asarray(t) for t in truth_list]
        self._shapes = [t.shape[-3:] for t in self._truth]

    # ---- the host decisions, in the reference's order --------------------------------------------------------------
    def _truth_patch(self, case, corner, index, size):
        """get_patch_from_3d_data(truth, patch_shape[:-1] + (size,), corner + (0, 0, index)) by clamped indices."""
        t = self._truth[case]
        lo = (corner[0], corner[1], corner[2] + index)
        hi = (lo[0] + self.patch_shape[0], lo[1] + self.patch_shape[1], lo[2] + size)
        if min(lo) >= 0 and all(h <= n for h, n in zip(hi, t.shape)):
            return t[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]]        # inside the volume: a view, no gather
        ix = np.clip(np.arange(corner[0], corner[0] + self.patch_shape[0]), 0, t.shape[0] - 1)
        iy = np.clip(np.arange(corner[1], corner[1] + self.patch_shape[1]), 0, t.shape[1] - 1)
        iz = np.clip(np.arange(corner[2] + index, corner[2] + index + size), 0, t.shape[2] - 1)
        return t[np.ix_(ix, iy, iz)]

    def draw(self):
        """One batch worth of accepted samples: (cases int32 [B], corners int32 [B, 3])."""
        cases, corners = [], []
        while len(cases) < self.batch_size:
            index = next(self._index_generator)
            shape = self._shapes[index]
            corner = [np.random.randint(low=0, high=high) for high in np.subtract(shape, self.patch_shape)]
            if self.drop_easy_patches or self.skip_blank:
                truth = self._truth_patch(index, corner, self.truth_index, self.truth_size)
                if self.drop_easy_patches:
                    truth_mean = np.mean(truth[16:-16, 16:-16, :])
                    if 1 - np.abs(truth_mean - 0.5) < np.random.random():
                        continue
                if self.skip_blank and not np.any(truth != 0):
                    continue
            cases.append(index)
            corners.append(corner)
        return np.asarray(cases, np.int32), np.asarray(corners, np.int32).reshape(-1, 3)

    def _args(self):
        return (self.truth_index, self.truth_size, self.prev_truth_index if self.prev_truth_size else 0,
                self.prev_truth_size)


_WARP_KEYS = ("rotate", "scale", "translate", "elastic")


def _three(name, v):
    """Three finite, non-negative numbers (one per axis) or ValueError."""
    try:
        t = tuple(float(e) for e in v)
    except TypeError:
        raise ValueError("device_augment[%r] must be three numbers (x, y, z), got %r" % (name, v))
    if len(t) != 3 or not all(math.isfinite(e) and e >= 0 for e in t):
        raise ValueError("device_augment[%r] must be three finite numbers >= 0, got %r" % (name, v))
    return t


def warp_spec(device_augment):
    """The validated warp keys of `device_augment`: {key: value} with rotate / scale / translate as (x, y, z) sigmas
    and elastic as (alpha (x, y, z), grid); {} when there is no warp."""
    a = device_augment or {}
    spec = {}
    for k in ("rotate", "scale", "translate"):
        if k in a:
            spec[k] = _three(k, a[k])
    if "elastic" in a:
        e = a["elastic"]
        if not isinstance(e, dict) or set(e) != {"alpha", "grid"}:
            raise ValueError("device_augment['elastic'] must be dict(alpha=a or (ax, ay, az), grid=G), got %r" % (e,))
        alpha = e["alpha"]
        alpha = _three("elastic.alpha", (alpha,) * 3 if isinstance(alpha, (int, float)) else alpha)
        g = e["grid"]
        if isinstance(g, bool) or not isinstance(g, (int, np.integer)) or not 2 <= g <= 8:
            raise ValueError("device_augment['elastic']['grid'] must be an integer in 2..8, got %r" % (g,))
        spec["elastic"] = (alpha, int(g))
    return spec


def warp_matrix(angles_deg, scales):
    """M = Rz Ry Rx diag(1/sx, 1/sy, 1/sz) in float64 (Rotation.from_euler('xyz', angles, degrees=True) times the
    inverse scale: the source position of an output voxel, so a factor above 1 enlarges structures)."""
    ax, ay, az = np.deg2rad(np.asarray(angles_deg, np.float64))
    rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    ry = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
    rz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
    return rz @ ry @ rx @ np.diag(1.0 / np.asarray(scales, np.float64))


def _c_array(cls, v):
    """None, a ctypes array of `cls`, or a sequence of `cls` (e.g. a slice of one) -> what the C call takes."""
    if v is None or (isinstance(v, ctypes.Array) and v._type_ is cls):
        return v
    v = list(v)
    return (cls * len(v))(*v) if v else None


def _check_one_label(model):
    """The sampler cuts one target channel; expanding integer truth into label channels (the reference generator's
    `labels` / `categorical` handling) is not built, so multi-label models train through train_on_batch."""
    if getattr(model, "n_labels", 1) != 1:
        raise NotImplementedError("the device sampler cuts one target channel; a model with %d labels trains through "
                                  "train_on_batch with label-channel targets" % model.n_labels)


class DeviceSampler(PatchDraws):
    """data_generator(data_file, index_list, ...) with the cases resident in HBM.

    data_list / truth_list: per-case arrays [X, Y, Z] (what `data_file.root.data[i]` / `.truth[i]` return after
    DataFileDummy / pad_samples). Arguments carry the reference's names and defaults (generator.py:222-226).
    """

    def __init__(self, data_list, truth_list, index_list, device_augment=None, device=None, **kw):
        if len(data_list) != len(truth_list):
            raise ValueError("data_list and truth_list differ in length")
        PatchDraws.__init__(self, truth_list, index_list, **kw)
        warp_spec(device_augment)
        self.device_augment = device_augment
        self._lib = _lib.load()
        self._ctx = _lib.get_context(device)
        h = _lib.c_vp()
        _lib.check(self._lib.fm_volset_create(self._ctx.handle, len(data_list), ctypes.byref(h)))
        self._handle = h
        for i, (d, t) in enumerate(zip(data_list, truth_list)):
            d32, t32 = _lib.f32c(d), _lib.f32c(t)
            if d32.shape != t32.shape or d32.ndim != 3:
                raise ValueError("case %d: data %s / truth %s must be equal-shaped 3-D volumes" % (i, d32.shape, t32.shape))
            _lib.check(self._lib.fm_volset_set_case(h, i, _lib.fptr(d32), _lib.fptr(t32), _lib.i32ptr(_lib.i32x(d32.shape))))

    def __del__(self):
        h, self._handle = getattr(self, "_handle", None), None
        if h is not None:
            try:
                self._lib.fm_volset_destroy(h)
            except Exception:
                pass

    def _aug_array(self, n):
        """fm_sample_aug[n] from `device_augment` = dict(flip=bool, intensity=(lo, hi), noise_sigma=float) or None."""
        a = self.device_augment
        if not a:
            return None
        arr = (_lib.SampleAug * n)()
        for b in range(n):
            arr[b].flip = int(np.random.randint(0, 8)) if a.get("flip") else 0
            lo, hi = a.get("intensity", (1.0, 1.0))
            arr[b].intensity_scale = float(np.random.uniform(lo, hi))
            arr[b].noise_sigma = float(a.get("noise_sigma", 0.0))
            arr[b].noise_seed = int(np.random.randint(0, 2 ** 31 - 1))
        return arr

    def _warp_array(self, n):
        """fm_sample_warp[n] from the rotate / scale / translate / elastic keys of `device_augment`, or None without
        them. Per sample: three angles, three scale factors, three offsets, the elastic seed (present keys only)."""
        spec = warp_spec(self.device_augment)
        if not spec:
            return None
        arr = (_lib.SampleWarp * n)()
        for b in range(n):
            angles = [np.random.normal(0.0, s) for s in spec["rotate"]] if "rotate" in spec else [0.0] * 3
            scales = ([float(np.clip(1.0 + np.random.normal(0.0, s), 0.5, 2.0)) for s in spec["scale"]]
                      if "scale" in spec else [1.0] * 3)
            offset = [np.random.normal(0.0, s) for s in spec["translate"]] if "translate" in spec else [0.0] * 3
            arr[b].matrix[:] = [float(v) for v in warp_matrix(angles, scales).astype(np.float32).ravel()]
            arr[b].offset[:] = [float(np.float32(v)) for v in offset]
            if "elastic" in spec:
                alpha, grid = spec["elastic"]
                arr[b].elastic_alpha[:] = alpha
                arr[b].elastic_grid = grid
                arr[b].elastic_seed = int(np.random.randint(0, 2 ** 31 - 1))
        return arr

    def draw_augment(self, n):
        """The per-sample augmentation arguments of the next n samples, drawn from np.random: (fm_sample_aug array or
        None, fm_sample_warp array or None)."""
        aug = self._aug_array(n)
        return aug, self._warp_array(n)

    def gather(self, cases, corners, aug=None, warp=None):
        """The batch of the given (case, corner) samples, cut on the device and copied back: x, y shaped like
        convert_data's output (generator.py:380-401). With aug and warp both None the augmentations are drawn from
        `device_augment`; otherwise exactly the given per-sample arrays are applied (None: none of that kind)."""
        cases, corners = _lib.i32x(cases), _lib.i32x(corners)
        n = cases.size
        if aug is None and warp is None:
            aug, warp = self.draw_augment(n)
        p0, p1, p2 = self.patch_shape
        x = np.empty((n, p0, p1, p2 + self.prev_truth_size), np.float32)
        y = np.empty((n, p0, p1, self.truth_size), np.float32)
        ti, ts, pi, ps = self._args()
        _lib.check(self._lib.fm_volset_gather_warp(self._handle, _lib.i32ptr(cases), _lib.i32ptr(corners),
                                                   _c_array(_lib.SampleAug, aug), _c_array(_lib.SampleWarp, warp), n,
                                                   _lib.i32ptr(_lib.i32x(self.patch_shape)), ti, ts, pi, ps,
                                                   _lib.fptr(x), _lib.fptr(y)))
        if self.is3d:
            x, y = np.expand_dims(x, 1), np.expand_dims(y, 1)
        return x, y

    def __iter__(self):
        return self

    def __next__(self):
        cases, corners = self.draw()
        return self.gather(cases, corners)

    def train_on_next_batch(self, model):
        """next(generator) + model.train_on_batch(x, y) without the batch ever visiting the host. Returns the
        metrics of Model.train_on_batch ([loss, dice_coefficient, vod_coefficient, binary_accuracy])."""
        _check_one_label(model)
        cases, corners = self.draw()
        aug, warp = self.draw_augment(len(cases))
        return model.train_on_sampled_batch(self, cases, corners, aug=aug, warp=warp)
