"""2-GPU test of fetal_net.distributed at n_labels = 3: the data-parallel step equals the single-GPU step on the global
batch (loss, label-wise Dice, gradients), and patch-sharded inference equals patch_wise_prediction with its label axis.
Skipped on boxes with fewer than 2 GPUs."""
import os

import numpy as np
import pytest
import torch

from tests.test_gpu_distributed import _free_port

pytestmark = pytest.mark.gpu

L = 3


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    os.environ["FETAL_B200_DETERMINISTIC"] = "1"      # per-sample activations identical in the 2 x 2 and 1 x 4 runs
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda:%d" % rank))
    from fetal_net.distributed import DataParallelTrainer, sharded_patch_wise_prediction
    from fetal_net.model import unet_model_3d
    from fetal_net.prediction import patch_wise_prediction
    from oracle import unet_oracle as uo
    from tests.test_gpu_multilabel import blob_targets, decisive_weights

    w = decisive_weights(uo.unet3d_layers(4, 16, n_labels=L), seed=2)
    rng = np.random.default_rng(9)
    x = rng.standard_normal((4, 1, 32, 32, 32)).astype(np.float32)
    t = blob_targets((4, L, 32, 32, 32), rng)
    build = lambda dev: unet_model_3d(input_shape=(1, 32, 32, 32), n_base_filters=16, n_labels=L,
                                      include_label_wise_dice_coefficients=True, initial_learning_rate=1e-4, device=dev)
    model = build(rank)
    model.set_named_weights(w)
    dp = DataParallelTrainer(model)
    lo, hi = 4 * rank // world, 4 * (rank + 1) // world
    res = dp.train_on_batch(x[lo:hi], t[lo:hi])
    grads = model.get_gradients()
    vol = rng.standard_normal((1, 72, 40, 32)).astype(np.float32)
    sharded = sharded_patch_wise_prediction(model, vol, (32, 32, 32), overlap_factor=0.5)
    if rank == 0:
        ref_model = build(0)
        ref_model.set_named_weights(w)
        ref = ref_model.train_on_batch(x, t)
        cos = []
        for g, r in zip(grads, ref_model.get_gradients()):
            g, r = g.astype(np.float64).ravel(), r.astype(np.float64).ravel()
            cos.append(float(g @ r / max(np.linalg.norm(g) * np.linalg.norm(r), 1e-300)))
        single = patch_wise_prediction(model, vol, (32, 32, 32), overlap_factor=0.5)
        out.put(dict(res=res, ref=ref, min_cos=min(cos), shape=single.shape,
                     infer_equal=bool(np.array_equal(sharded, single))))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_step_and_sharded_inference_with_labels():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    r = q.get(timeout=300)
    [p.join(timeout=120) for p in procs]
    assert len(r["res"]) == len(r["ref"]) == 3 + L, r
    assert r["res"][0] == pytest.approx(r["ref"][0], abs=1e-6), r
    for i in range(3, 3 + L):                           # label-wise Dice from the all-reduced per-label sums
        assert r["res"][i] == pytest.approx(r["ref"][i], abs=1e-6), r
    assert r["min_cos"] >= 0.9999, r
    assert r["shape"] == (72, 40, 32, L) and r["infer_equal"], r
