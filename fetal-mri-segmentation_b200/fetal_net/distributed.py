"""Data-parallel extension of the hot path (the reference is single-process: training.py:115-117).

One process per GPU. The collectives run on raw NCCL inside libfetalb200 (csrc/comm.cu: fm_comm_init,
fm_train_step_dp, fm_patchwise_predict_dp) - no device pointer leaves the library. `torch.distributed` (any backend,
gloo is enough) is only the CONTROL plane: it carries the 128-byte NCCL id from rank 0 to the other ranks.

  training   batch sharded over ranks, weights replicated. Soft Dice is a WHOLE-batch statistic
             (metrics.py:11-15 flattens the batch axis), so the forward all-reduces the 8 loss sums and
             every rank back-propagates the global Dice; the gradient of that one global scalar is the
             SUM (not the mean) of the ranks' local gradients. The flat fp32 gradient buffer is
             all-reduced bucket by bucket on a side stream while the rest of backward still runs,
             then every rank applies the identical Adam step. batch_normalization=True U-Nets take every
             layer's batch statistics over the global batch: one float64 all-reduce of the per-channel
             (sum, sum of squares, count) per layer in forward and of the gradient sums in backward, so
             the step equals the single-process step on the concatenated batch (uneven shards too) and
             the moving statistics stay identical on every rank. The gradient buckets then start after
             backward's last statistics all-reduce instead of overlapping backward.
  inference  the patch list of patch_wise_prediction is split contiguously over ranks; each rank
             overlap-adds its patches into a private float64 partial sum on its GPU, one ncclReduce, then
             sum / count on the root. Counts are analytic (identical on every rank) and never communicated.
"""
import os

import numpy as np

from . import _lib


def shard_range(n, rank, count):
    """Contiguous share [lo, hi) of n patches for `rank` of `count` (same rule as fm_patchwise_predict)."""
    return n * rank // count, n * (rank + 1) // count


def init_comm(ctx=None, rank=None, world=None):
    """Creates the native NCCL communicator of `ctx` (idempotent). The id travels through the default
    torch.distributed process group when one is initialised, otherwise through a TCPStore on
    MASTER_ADDR:MASTER_PORT+1 (env, as set by torchrun). Returns (rank, world)."""
    import torch.distributed as dist
    ctx = ctx or _lib.get_context()
    lib = _lib.load()
    r, w, _ = ctx.comm_info()
    if w > 1:
        return r, w
    if dist.is_available() and dist.is_initialized():
        rank = dist.get_rank() if rank is None else rank
        world = dist.get_world_size() if world is None else world
    else:
        rank = int(os.environ.get("RANK", "0")) if rank is None else rank
        world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else world
    if world == 1:
        return 0, 1
    uid = np.zeros(128, np.uint8)
    if rank == 0:
        _lib.check(lib.fm_comm_unique_id(uid.ctypes.data_as(_lib.c_u8p)))
    if dist.is_available() and dist.is_initialized():
        box = [uid.tobytes()]
        dist.broadcast_object_list(box, src=0)
        uid = np.frombuffer(box[0], np.uint8).copy()
    else:
        store = dist.TCPStore(os.environ.get("MASTER_ADDR", "127.0.0.1"), int(os.environ["MASTER_PORT"]) + 1, world,
                              is_master=(rank == 0))
        if rank == 0:
            store.set("fetal_b200_nccl_uid", uid.tobytes())
        uid = np.frombuffer(store.get("fetal_b200_nccl_uid"), np.uint8).copy()
    _lib.check(lib.fm_comm_init(ctx.handle, int(rank), int(world), uid.ctypes.data_as(_lib.c_u8p)))
    return rank, world


class DataParallelTrainer:
    """Wraps a native Model for multi-GPU training: `train_on_batch` on this rank's shard of the global batch."""

    def __init__(self, model, overlap=True):
        self.model = model
        self.lib = _lib.load()
        self.ctx = model._ctx
        self.device = model._ctx.device
        self.rank, self.world = init_comm(self.ctx)

    def broadcast_weights(self, src=0):
        """Rank `src`'s weights and Adam state to every replica."""
        _lib.check(self.lib.fm_comm_broadcast_params(self.model._h, int(src)))

    def train_on_batch(self, x, y):
        """x, y: this rank's shard of the global batch ([x, weight_mask] for a two-input model). Returns the GLOBAL
        [loss, acc, vod(, dice)(, label-wise Dice)]."""
        self.model._check_loss()
        x = self.model._split_mask(x)
        x, y = _lib.f32c(x), _lib.f32c(y)
        m = np.zeros(4, np.float32)
        _lib.check(self.lib.fm_train_step_dp(self.model._h, _lib.fptr(x), _lib.fptr(y), int(x.shape[0]),
                                             float(self.model.optimizer.lr), _lib.fptr(m)))
        return self.model._metrics(m)

    def allreduce_bench(self, nbytes, iters=20):
        """(ms per all-reduce, bus GB/s = 2 (n-1)/n * bytes / t) of an in-place fp32 SUM all-reduce of `nbytes`."""
        ms = np.zeros(1, np.float32)
        _lib.check(self.lib.fm_comm_allreduce_bench(self.ctx.handle, int(nbytes), int(iters), _lib.fptr(ms)))
        t = float(ms[0]) * 1e-3
        return float(ms[0]), 2.0 * (self.world - 1) / self.world * nbytes / t / 1e9

    def set_comm_enabled(self, on):
        _lib.check(self.lib.fm_comm_enable(self.ctx.handle, 1 if on else 0))


def sharded_patch_wise_prediction(model, data, patch_shape, overlap_factor=0, batch_size=5, dst=0):
    """patch_wise_prediction with the patch list sharded over the ranks. Returns the float64 [X,Y,Z,C] volume on
    rank `dst` (None elsewhere). Native models reduce the partial sums on the GPUs (fm_patchwise_predict_dp); any
    other Keras-like model goes through torch.distributed (used by the gloo tests on CPU)."""
    from .prediction import patch_wise_prediction
    if hasattr(model, "_h"):
        rank, count = init_comm(model._ctx)
        if count == 1:
            return patch_wise_prediction(model, data, patch_shape, overlap_factor, batch_size)
        return patch_wise_prediction(model, data, patch_shape, overlap_factor, batch_size, shard=(rank, count),
                                     reduce_root=dst)
    import torch
    import torch.distributed as dist
    rank, count = dist.get_rank(), dist.get_world_size()
    if count == 1:
        return patch_wise_prediction(model, data, patch_shape, overlap_factor, batch_size)
    part, cnt = patch_wise_prediction(model, data, patch_shape, overlap_factor, batch_size, shard=(rank, count))
    t = torch.as_tensor(part)
    dist.reduce(t, dst)                                                  # float64 partial sums
    if rank != dst:
        return None
    assert np.all(cnt > 0), 'Found zeros in count'
    return t.numpy() / cnt[..., None]
