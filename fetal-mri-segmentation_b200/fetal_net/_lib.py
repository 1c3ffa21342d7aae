"""ctypes binding of libfetalb200.so (C ABI declared in include/fetal_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfetalb200.so")

c_int = ctypes.c_int
c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64 = ctypes.c_int64
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_u64 = ctypes.c_uint64
c_u64p = ctypes.POINTER(ctypes.c_uint64)
c_f = ctypes.c_float
c_fp = ctypes.POINTER(ctypes.c_float)
c_d = ctypes.c_double
c_dp = ctypes.POINTER(ctypes.c_double)
c_i16p = ctypes.POINTER(ctypes.c_int16)
c_u8p = ctypes.POINTER(ctypes.c_uint8)
c_vp = ctypes.c_void_p


class UNet3DSpec(ctypes.Structure):
    _fields_ = [("in_channels", ctypes.c_int32), ("X", ctypes.c_int32), ("Y", ctypes.c_int32),
                ("Z", ctypes.c_int32), ("depth", ctypes.c_int32), ("n_base_filters", ctypes.c_int32),
                ("n_labels", ctypes.c_int32)]


class Isensee3DSpec(ctypes.Structure):
    _fields_ = [("in_channels", ctypes.c_int32), ("X", ctypes.c_int32), ("Y", ctypes.c_int32), ("Z", ctypes.c_int32),
                ("depth", ctypes.c_int32), ("n_base_filters", ctypes.c_int32),
                ("n_segmentation_levels", ctypes.c_int32), ("n_labels", ctypes.c_int32)]


class SampleAug(ctypes.Structure):
    """fm_sample_aug: per-sample cheap augmentations of the device sampler."""
    _fields_ = [("flip", ctypes.c_uint32), ("intensity_scale", ctypes.c_float), ("noise_sigma", ctypes.c_float),
                ("noise_seed", ctypes.c_uint32)]


class Isensee2DSpec(ctypes.Structure):
    _fields_ = [("H", ctypes.c_int32), ("W", ctypes.c_int32), ("in_channels", ctypes.c_int32),
                ("depth", ctypes.c_int32), ("n_base_filters", ctypes.c_int32),
                ("n_segmentation_levels", ctypes.c_int32), ("n_labels", ctypes.c_int32)]


class UNet2DSpec(ctypes.Structure):
    _fields_ = [("H", ctypes.c_int32), ("W", ctypes.c_int32), ("in_channels", ctypes.c_int32),
                ("depth", ctypes.c_int32), ("n_base_filters", ctypes.c_int32), ("n_labels", ctypes.c_int32)]


class PostprocessSpec(ctypes.Structure):
    """fm_postprocess_spec: Gaussian weights (2 radius + 1), threshold and the two flags of postprocess_prediction."""
    _fields_ = [("radius", ctypes.c_int32), ("weights", ctypes.POINTER(ctypes.c_double)), ("threshold", ctypes.c_double),
                ("fill_holes", ctypes.c_int32), ("connected_component", ctypes.c_int32)]


# name -> (restype, argtypes); exactly the symbols include/fetal_b200.h declares
SIGNATURES = {
    "fm_ctx_create": (c_int, [c_int, ctypes.POINTER(c_vp)]),
    "fm_ctx_destroy": (c_int, [c_vp]),
    "fm_last_error": (ctypes.c_char_p, []),
    "fm_ctx_device_info": (c_int, [c_vp, ctypes.POINTER(c_int)]),
    "fm_ctx_stream": (c_u64, [c_vp]),
    "fm_ctx_synchronize": (c_int, [c_vp]),
    "fm_ctx_launch_count": (c_i64, [c_vp]),
    "fm_ctx_profile_enable": (c_int, [c_vp, c_int]),
    "fm_ctx_profile_count": (c_int, [c_vp]),
    "fm_ctx_profile_get": (c_int, [c_vp, c_int, ctypes.c_char_p, c_dp]),
    "fm_model_create_unet3d": (c_int, [c_vp, ctypes.POINTER(UNet3DSpec), ctypes.POINTER(c_vp)]),
    "fm_model_create_unet2d": (c_int, [c_vp, ctypes.POINTER(UNet2DSpec), ctypes.POINTER(c_vp)]),
    "fm_model_create_unet3d_ex": (c_int, [c_vp, ctypes.POINTER(UNet3DSpec), c_int, ctypes.POINTER(c_vp)]),
    "fm_model_create_unet2d_ex": (c_int, [c_vp, ctypes.POINTER(UNet2DSpec), c_int, ctypes.POINTER(c_vp)]),
    "fm_model_create_isensee3d": (c_int, [c_vp, ctypes.POINTER(Isensee3DSpec), ctypes.POINTER(c_vp)]),
    "fm_model_create_isensee2d": (c_int, [c_vp, ctypes.POINTER(Isensee2DSpec), ctypes.POINTER(c_vp)]),
    "fm_model_destroy": (c_int, [c_vp]),
    "fm_model_num_layers": (c_int, [c_vp]),
    "fm_model_layer_info": (c_int, [c_vp, c_int, ctypes.c_char_p, c_i64p]),
    "fm_model_num_params": (c_i64, [c_vp]),
    "fm_model_set_weights": (c_int, [c_vp, c_int, c_fp, c_fp]),
    "fm_model_get_weights": (c_int, [c_vp, c_int, c_fp, c_fp]),
    "fm_model_get_grads": (c_int, [c_vp, c_int, c_fp, c_fp]),
    "fm_model_reset_optimizer": (c_int, [c_vp]),
    "fm_model_set_dropout": (c_int, [c_vp, ctypes.c_float, ctypes.c_uint64]),
    "fm_model_set_loss": (c_int, [c_vp, c_int, ctypes.c_float, ctypes.c_float]),
    "fm_model_set_inference_mode": (c_int, [c_vp, c_int]),
    "fm_model_set_weight_mask": (c_int, [c_vp, c_fp, c_int]),
    "fm_train_metrics_async": (c_int, [c_vp]),
    "fm_train_metrics_wait": (c_int, [c_vp, c_fp]),
    "fm_host_alloc": (c_int, [ctypes.c_size_t, ctypes.POINTER(c_vp)]),
    "fm_host_free": (c_int, [c_vp]),
    "fm_predict": (c_int, [c_vp, c_fp, c_int, c_fp]),
    "fm_patch_plan": (c_int, [c_i32p, c_i32p, c_i32p, c_d, c_i32p, c_i64, c_i64p]),
    "fm_patchwise_predict": (c_int, [c_vp, c_fp, c_i32p, c_i32p, c_i32p, c_dp, c_i32p, c_i64, c_int,
                                     c_int, c_int, c_fp, c_int, c_int, c_dp, c_i16p]),
    "fm_reassemble": (c_int, [c_vp, c_fp, c_i32p, c_i64, c_i32p, c_int, c_i32p, c_dp, c_i16p]),
    "fm_gather_patches": (c_int, [c_vp, c_fp, c_i32p, c_i32p, c_i32p, c_dp, c_i32p, c_i64, c_i32p, c_fp]),
    "fm_postprocess": (c_int, [c_vp, c_vp, c_int, c_i32p, ctypes.POINTER(PostprocessSpec), c_u8p, c_i64p]),
    "fm_patchwise_segment": (c_int, [c_vp, c_fp, c_i32p, c_i32p, c_i32p, c_dp, c_i32p, c_i64, c_int, c_fp, c_int, c_int,
                                     ctypes.POINTER(PostprocessSpec), c_u8p, c_dp, c_i64p]),
    "fm_op_gaussian3d": (c_int, [c_vp, c_vp, c_int, c_i32p, c_int, c_dp, c_vp]),
    "fm_patchwise_predict_flips": (c_int, [c_vp, c_fp, c_i32p, c_i32p, c_i32p, c_dp, c_i32p, c_i64, c_int, c_int, c_i32p,
                                           c_i32p, c_dp, c_dp, ctypes.POINTER(PostprocessSpec), c_u8p, c_i64p]),
    "fm_op_median_passes": (c_int, [c_vp, c_dp, c_int, c_i64, c_dp]),
    "fm_train_step": (c_int, [c_vp, c_fp, c_fp, c_int, c_f, c_fp]),
    "fm_train_forward": (c_int, [c_vp, c_fp, c_fp, c_int]),
    "fm_train_backward": (c_int, [c_vp]),
    "fm_train_apply": (c_int, [c_vp, c_f, c_u64, c_fp]),
    "fm_model_loss_sums": (c_int, [c_vp, c_u64p]),
    "fm_model_grad_buffer": (c_int, [c_vp, c_u64p, c_i64p]),
    "fm_model_num_buckets": (c_int, [c_vp]),
    "fm_model_bucket_range": (c_int, [c_vp, c_int, c_i64p, c_i64p]),
    "fm_stream_wait_bucket": (c_int, [c_vp, c_u64, c_int]),
    "fm_train_step_device": (c_int, [c_vp, c_u64, c_u64, c_int, c_f, c_fp]),
    "fm_predict_device": (c_int, [c_vp, c_u64, c_int, c_u64]),
    "fm_evaluate": (c_int, [c_vp, c_fp, c_fp, c_int, c_fp]),
    "fm_model_get_adam_state": (c_int, [c_vp, c_int, c_fp, c_fp, c_fp, c_fp]),
    "fm_model_set_adam_state": (c_int, [c_vp, c_int, c_fp, c_fp, c_fp, c_fp]),
    "fm_model_get_iterations": (c_int, [c_vp]),
    "fm_model_set_iterations": (c_int, [c_vp, c_int]),
    "fm_volset_create": (c_int, [c_vp, c_int, ctypes.POINTER(c_vp)]),
    "fm_volset_destroy": (c_int, [c_vp]),
    "fm_volset_set_case": (c_int, [c_vp, c_int, c_fp, c_fp, c_i32p]),
    "fm_volset_gather": (c_int, [c_vp, c_i32p, c_i32p, ctypes.POINTER(SampleAug), c_int, c_i32p, c_int, c_int, c_int,
                                 c_int, c_fp, c_fp]),
    "fm_train_step_sampled": (c_int, [c_vp, c_vp, c_i32p, c_i32p, ctypes.POINTER(SampleAug), c_int, c_int, c_int,
                                      c_int, c_int, c_f, c_fp]),
    "fm_comm_unique_id": (c_int, [c_u8p]),
    "fm_comm_init": (c_int, [c_vp, c_int, c_int, c_u8p]),
    "fm_comm_destroy": (c_int, [c_vp]),
    "fm_comm_info": (c_int, [c_vp, ctypes.POINTER(c_int)]),
    "fm_comm_enable": (c_int, [c_vp, c_int]),
    "fm_comm_stream": (c_u64, [c_vp]),
    "fm_comm_allreduce_bench": (c_int, [c_vp, c_i64, c_int, c_fp]),
    "fm_comm_broadcast_params": (c_int, [c_vp, c_int]),
    "fm_train_step_dp": (c_int, [c_vp, c_fp, c_fp, c_int, c_f, c_fp]),
    "fm_patchwise_predict_dp": (c_int, [c_vp, c_fp, c_i32p, c_i32p, c_i32p, c_dp, c_i32p, c_i64, c_int,
                                        c_int, c_fp, c_int, c_int, c_dp, c_i16p]),
    "fm_op_conv3d_fprop": (c_int, [c_vp, c_int, c_fp, c_fp, c_fp, c_fp] + [c_int] * 9 + [c_fp]),
    "fm_op_conv3d_dgrad": (c_int, [c_vp, c_int, c_fp, c_fp, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_conv3d_wgrad": (c_int, [c_vp, c_int, c_fp, c_fp] + [c_int] * 6 + [c_fp, c_fp]),
    "fm_op_conv_dgrad": (c_int, [c_vp, c_int, c_fp, c_fp, c_fp] + [c_int] * 7 + [c_fp]),
    "fm_op_conv_wgrad": (c_int, [c_vp, c_int, c_fp, c_fp] + [c_int] * 7 + [c_fp, c_fp]),
    "fm_op_conv3d_first": (c_int, [c_vp, c_fp, c_fp, c_fp] + [c_int] * 6 + [c_fp, c_fp, c_fp]),
    "fm_op_conv3d_up_fprop": (c_int, [c_vp, c_fp, c_fp, c_fp, c_fp] + [c_int] * 8 + [c_fp]),
    "fm_op_conv3d_up_bwd": (c_int, [c_vp, c_fp, c_fp, c_fp] + [c_int] * 8 + [c_fp, c_fp]),
    "fm_op_maxpool3d": (c_int, [c_vp, c_fp] + [c_int] * 5 + [c_fp]),
    "fm_op_maxpool3d_bwd": (c_int, [c_vp, c_fp, c_fp, c_fp] + [c_int] * 5 + [c_fp]),
    "fm_op_upsample3d": (c_int, [c_vp, c_fp] + [c_int] * 5 + [c_fp]),
    "fm_op_upsample3d_bwd": (c_int, [c_vp, c_fp, c_fp] + [c_int] * 5 + [c_fp]),
    "fm_op_maxpool": (c_int, [c_vp, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_maxpool_bwd": (c_int, [c_vp, c_fp, c_fp, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_upsample": (c_int, [c_vp, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_upsample_bwd": (c_int, [c_vp, c_fp, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_dice": (c_int, [c_vp, c_fp, c_fp, c_i64, c_dp, c_fp]),
    "fm_op_dice_xent": (c_int, [c_vp, c_fp, c_fp, c_fp, c_i64, ctypes.c_float, ctypes.c_float, c_dp, c_fp]),
    "fm_op_adam": (c_int, [c_vp, c_fp, c_fp, c_fp, c_fp, c_i64, c_int, c_f]),
    "fm_op_instnorm_lrelu": (c_int, [c_vp, c_fp, c_fp, c_fp, c_fp, c_fp, c_int, c_i64, c_int, c_fp, c_fp]),
    "fm_op_instnorm_lrelu_bwd": (c_int, [c_vp, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, c_int, c_i64, c_int, c_fp, c_fp,
                                         c_fp]),
    "fm_op_batchnorm_relu": (c_int, [c_vp, c_int, c_fp, c_fp, c_fp, c_fp, c_fp, c_int, c_i64, c_int, c_fp]),
    "fm_op_batchnorm_relu_bwd": (c_int, [c_vp, c_fp, c_fp, c_fp, c_fp, c_fp, c_int, c_i64, c_int, c_fp, c_fp, c_fp]),
    "fm_op_conv_strided": (c_int, [c_vp, c_fp, c_fp, c_fp] + [c_int] * 7 + [c_fp, c_fp, c_fp, c_fp]),
    "fm_op_deconv": (c_int, [c_vp, c_fp, c_fp, c_fp] + [c_int] * 6 + [c_fp, c_fp, c_int, c_fp, c_fp, c_fp]),
    "fm_op_depth_space": (c_int, [c_vp, c_int, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_zero_insert": (c_int, [c_vp, c_fp] + [c_int] * 6 + [c_fp]),
    "fm_op_head": (c_int, [c_vp, c_fp, c_fp, c_fp, c_i64, c_int, c_int, c_fp, c_fp, c_dp, c_fp, c_int, c_fp, c_fp,
                           c_fp]),
    "fm_op_seg_upsample_add": (c_int, [c_vp, c_fp, c_fp] + [c_int] * 5 + [c_fp]),
    "fm_op_sumpool_f32": (c_int, [c_vp, c_fp] + [c_int] * 5 + [c_fp]),
}

_lib = None


class FetalB200Error(RuntimeError):
    pass


def load():
    """Loads the shared library (once) and types every entry point. Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FetalB200Error(
            "libfetalb200.so not found at %s - build it with `python fetal-mri-segmentation_b200/build.py` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().fm_last_error()
        raise FetalB200Error("libfetalb200 error %d: %s" % (rc, msg.decode("utf-8", "replace") if msg else "?"))


def fptr(a):
    return a.ctypes.data_as(c_fp) if a is not None else None


def dptr(a):
    return a.ctypes.data_as(c_dp) if a is not None else None


def i32ptr(a):
    return a.ctypes.data_as(c_i32p) if a is not None else None


def i16ptr(a):
    return a.ctypes.data_as(c_i16p) if a is not None else None


def f32c(a):
    """float32, C-contiguous view/copy of `a` (the reference feeds float64, Keras casts to float32)."""
    return np.ascontiguousarray(a, dtype=np.float32)


def i32x(vals):
    return np.ascontiguousarray(np.asarray(vals, dtype=np.int32).reshape(-1))


class _PinnedBlock:
    """One page-locked allocation; goes back to the pool when the last NumPy view of it dies."""

    def __init__(self, nbytes):
        p = c_vp()
        check(load().fm_host_alloc(nbytes, ctypes.byref(p)))
        self.ptr, self.nbytes = p.value, nbytes

    def release(self):
        if self.ptr:
            load().fm_host_free(c_vp(self.ptr))
            self.ptr = None


_pinned_pool = {}       # nbytes -> [free _PinnedBlock]
_PINNED_POOL_MAX = 4    # free blocks kept per size


class _PinnedLease:
    """Owner object behind a pooled array: returns the block to the pool on garbage collection."""

    def __init__(self, block):
        self.block = block

    def __del__(self):
        try:
            free = _pinned_pool.setdefault(self.block.nbytes, [])
            if len(free) < _PINNED_POOL_MAX:
                free.append(self.block)
            else:
                self.block.release()
        except Exception:
            pass


def pinned_empty(shape, dtype):
    """np.empty(shape, dtype) in page-locked memory from a small pool: what fm_patchwise_predict writes its result
    into. The array owns its block (through .base) until it and all its views are collected."""
    dtype = np.dtype(dtype)
    nbytes = max(int(np.prod(shape)) * dtype.itemsize, 1)
    free = _pinned_pool.get(nbytes)
    block = free.pop() if free else _PinnedBlock(nbytes)
    buf = (ctypes.c_byte * nbytes).from_address(block.ptr)
    buf._lease = _PinnedLease(block)            # keeps the block out of the pool while any view is alive
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


_contexts = {}


class Context:
    """One fm_ctx per (process, device)."""

    def __init__(self, device=0):
        lib = load()
        h = c_vp()
        check(lib.fm_ctx_create(int(device), ctypes.byref(h)))
        self.handle = h
        self.device = int(device)

    @property
    def stream(self):
        return int(load().fm_ctx_stream(self.handle))

    def synchronize(self):
        check(load().fm_ctx_synchronize(self.handle))

    def launch_count(self):
        return int(load().fm_ctx_launch_count(self.handle))

    def profile(self, on):
        check(load().fm_ctx_profile_enable(self.handle, 1 if on else 0))

    def profile_records(self):
        """[(kernel name, ms, algorithmic flops, algorithmic bytes)] since profile(True)."""
        lib = load()
        out = []
        for i in range(lib.fm_ctx_profile_count(self.handle)):
            name = ctypes.create_string_buffer(48)
            v = (c_d * 3)()
            check(lib.fm_ctx_profile_get(self.handle, i, name, v))
            out.append((name.value.decode(), float(v[0]), float(v[1]), float(v[2])))
        return out

    def device_info(self):
        out = (c_int * 3)()
        check(load().fm_ctx_device_info(self.handle, out))
        return tuple(out)

    def comm_info(self):
        """(rank, ranks, NCCL version code) of the native data-parallel communicator (ranks = 1 without one)."""
        out = (c_int * 3)()
        check(load().fm_comm_info(self.handle, out))
        return tuple(out)


def default_device():
    return int(os.environ.get("LOCAL_RANK", os.environ.get("FETAL_B200_DEVICE", "0")))


def get_context(device=None):
    device = default_device() if device is None else int(device)
    if device not in _contexts:
        _contexts[device] = Context(device)
    return _contexts[device]
