"""2-GPU tests of data-parallel training of batch-normalised U-Nets (NCCL): the statistics of every BatchNormalization
span the global batch, so a data-parallel step on shards equals the single-process step on the whole batch, including
uneven shards, and the replicas' moving statistics and parameters stay bit-identical. Covers unet_model_3d with and
without deconvolution and unet_model_2d, through DataParallelTrainer.train_on_batch and train_on_sampled_batch.
Skipped on boxes with fewer than 2 GPUs."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GLOBAL_BATCH = 4
SPLITS = [(2, 2), (3, 1)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _cos(g, r):
    g, r = g.astype(np.float64).ravel(), r.astype(np.float64).ravel()
    return float(g @ r / max(np.linalg.norm(g) * np.linalg.norm(r), 1e-300))


def _build(kind, rank):
    from fetal_net.model import unet_model_2d, unet_model_3d
    from oracle import unet_oracle as uo
    from tests.test_gpu_model import _bn_weights
    if kind == "2d":
        model = unet_model_2d(input_shape=(32, 32, 6), n_base_filters=16, depth=3, initial_learning_rate=1e-3,
                              batch_normalization=True, device=rank)
        w = _bn_weights(uo.unet2d_layers(3, 16, 6), 2, seed=31)
    else:
        deconv = kind == "3d_deconv"
        model = unet_model_3d(input_shape=(1, 32, 32, 16), n_base_filters=16, depth=3, initial_learning_rate=1e-3,
                              batch_normalization=True, deconvolution=deconv, device=rank)
        w = _bn_weights(uo.unet3d_layers(3, 16, deconvolution=deconv), 3, seed=21)
    model.set_named_weights(w)
    return model


def _checked_grads(model):
    """(name, array) of the gradients that carry signal: not the moving statistics (non-trainable, zero) and not the
    bias of a conv in front of a BatchNormalization (analytically zero: rounding noise)."""
    names = {l["name"] for l in model.layers}
    out = []
    for l, gk, gb in zip(model.layers, model.get_gradients()[0::2], model.get_gradients()[1::2]):
        if l["is_moving"]:
            continue
        out.append((l["name"] + "/kernel", gk))
        if l["name"] + "_norm" not in names:
            out.append((l["name"] + "/bias", gb))
    return out


def _moving(model):
    ws = model.get_weights()
    return [(ws[2 * i], ws[2 * i + 1]) for i, l in enumerate(model.layers) if l["is_moving"]]


def _compare(res, ref, grads, ref_grads, moving, ref_moving):
    cos = [_cos(g, r) for (_, g), (_, r) in zip(grads, ref_grads)]
    rel = max(float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-30))
              for pair, rpair in zip(moving, ref_moving) for a, b in zip(pair, rpair))
    return dict(res=res, ref=ref, min_cos=min(cos), argmin=grads[int(np.argmin(cos))][0], moving_rel=rel)


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    os.environ["FETAL_B200_DETERMINISTIC"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda:%d" % rank))
    from fetal_net.device_sampler import DeviceSampler
    from fetal_net.distributed import DataParallelTrainer
    from tests.test_gpu_model import _blob_truth

    results = {}
    for kind in ("3d", "3d_deconv", "2d"):
        rng = np.random.default_rng(5)
        shape = (32, 32, 6) if kind == "2d" else (1, 32, 32, 16)
        x = rng.standard_normal((GLOBAL_BATCH,) + shape).astype(np.float32)
        x2 = rng.standard_normal((GLOBAL_BATCH,) + shape).astype(np.float32)
        if kind == "2d":
            t = (rng.random((GLOBAL_BATCH, 32, 32, 1)) < 0.3).astype(np.float32)
            t2 = (rng.random((GLOBAL_BATCH, 32, 32, 1)) < 0.3).astype(np.float32)
        else:
            t, t2 = _blob_truth(x), _blob_truth(x2)
        for split in SPLITS:
            lo = sum(split[:rank])
            hi = lo + split[rank]
            model = _build(kind, rank)
            dp = DataParallelTrainer(model)
            res = dp.train_on_batch(x[lo:hi], t[lo:hi])
            grads, moving = _checked_grads(model), _moving(model)
            dp.train_on_batch(x2[lo:hi], t2[lo:hi])
            ws2 = model.get_weights()
            box = [None, None]
            dist.all_gather_object(box, (moving, ws2))
            if rank == 0:
                ref_model = _build(kind, 0)
                ref = ref_model.train_on_batch(x, t)
                r = _compare(res, ref, grads, _checked_grads(ref_model), moving, _moving(ref_model))
                r["moving_equal"] = all(np.array_equal(a, b) for pa, pb in zip(box[0][0], box[1][0])
                                        for a, b in zip(pa, pb))
                r["params_equal"] = all(np.array_equal(a, b) for a, b in zip(box[0][1], box[1][1]))
                results["%s %s" % (kind, split)] = r
    # the sampled step: (cases, corners) per rank, against train_on_batch on the gather of both ranks' samples
    data = [np.random.default_rng(7 + i).standard_normal((48, 48, 12)).astype(np.float32) for i in range(2)]
    truth = [(np.random.default_rng(9 + i).random((48, 48, 12)) > 0.6).astype(np.float32) for i in range(2)]
    kw = dict(batch_size=2, patch_shape=(32, 32, 5), shuffle_index_list=False, truth_index=2, truth_size=1,
              prev_truth_index=1, prev_truth_size=1, skip_blank=False)
    sampler = DeviceSampler(data, truth, [0, 1], device=rank, **kw)
    cases = np.array([0, 1, 1, 0], np.int32)
    corners = np.array([[0, 3, 1], [16, 5, 7], [9, 16, 2], [4, 11, 6]], np.int32)
    for split in SPLITS:
        lo = sum(split[:rank])
        hi = lo + split[rank]
        model = _build("2d", rank)
        DataParallelTrainer(model)
        res = model.train_on_sampled_batch(sampler, cases[lo:hi], corners[lo:hi])
        grads, moving = _checked_grads(model), _moving(model)
        box = [None, None]
        dist.all_gather_object(box, moving)
        if rank == 0:
            xs, ys = sampler.gather(cases, corners)
            ref_model = _build("2d", 0)
            ref = ref_model.train_on_batch(xs, ys)
            r = _compare(res, ref, grads, _checked_grads(ref_model), moving, _moving(ref_model))
            r["moving_equal"] = all(np.array_equal(a, b) for pa, pb in zip(box[0], box[1]) for a, b in zip(pa, pb))
            r["params_equal"] = True
            results["sampled 2d %s" % (split,)] = r
    if rank == 0:
        out.put(results)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_batch_norm_step():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    results = q.get(timeout=600)
    [p.join(timeout=120) for p in procs]
    assert len(results) == 3 * len(SPLITS) + len(SPLITS), sorted(results)
    for name, r in results.items():
        # global Dice loss / metrics of the whole batch (FETAL_B200_DETERMINISTIC=1 in the workers)
        assert np.allclose(r["res"], r["ref"], rtol=0, atol=1e-6), (name, r)
        # summed gradients == full-batch gradients (the fp32 summation order of the weight gradients differs)
        assert r["min_cos"] >= 0.9999, (name, r)
        # every rank holds the same moving statistics: those of the single-process step
        assert r["moving_equal"] and r["moving_rel"] <= 1e-6, (name, r)
        # after a second step the replicas' parameters are still identical
        assert r["params_equal"], (name, r)
