"""Data-parallel training of the batch-normalised U-Net (batch statistics over the global batch): unet_model_3d(depth 4,
16 base filters, batch_normalization=True) at 8 x 64^3 per GPU, and the same U-Net without batch normalisation for
comparison. Run one process per GPU:
    python -m torch.distributed.run --nproc_per_node N tools/bench_bn_dp.py --out FILE [--steps K] [--warmup W]
Rank 0 adds the record of this world size to FILE (JSON, one entry per GPU count): step ms and voxels/s with the
collectives on, the step with them switched off (fm_comm_enable: every rank then normalises with its own batch) and the
difference = exposed communication, the number of statistics all-reduces per step, the latency of one all-reduce of
the largest statistics message, and dp_parity: one data-parallel step against one single-GPU step on the whole global
batch (loss difference, minimum gradient cosine). Also the GPU name, power limit and max SM clock. Steps are timed with
CUDA events on the library's stream, --steps after --warmup untimed ones, max over the ranks."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "fetal-mri-segmentation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

DEPTH, NF, PATCH, BATCH = 4, 16, (64, 64, 64), 8


def gpu_identity(device):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(device)], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def make_batch(rank, batch=BATCH):
    rng = np.random.default_rng(100 + rank)
    x = rng.standard_normal((batch, 1) + PATCH).astype(np.float32)
    t = (rng.random(x.shape) < 0.3).astype(np.float32)
    return x, t


def build(bn, device):
    from fetal_net.model import unet_model_3d
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, initial_learning_rate=1e-4,
                          batch_normalization=bn, device=device)
    model.init_glorot_uniform(seed=0)
    return model


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from fetal_net import _lib
    from fetal_net.distributed import DataParallelTrainer
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")))
    assert torch.cuda.is_available(), "bench_bn_dp.py needs a GPU"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda:%d" % local))
    ctx = _lib.get_context(local)
    stream = torch.cuda.ExternalStream(ctx.stream, device="cuda:%d" % local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return float(v)
        t = torch.tensor([float(v)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / args.steps

    x, t = make_batch(rank)
    xp, tp = torch.as_tensor(x).pin_memory().numpy(), torch.as_tensor(t).pin_memory().numpy()
    rec = dict(world=world, per_gpu_batch=BATCH, global_batch=BATCH * world)
    for bn in (True, False):
        model = build(bn, local)
        dp = DataParallelTrainer(model)
        r = {}
        r["norm_layers"] = sum(1 for l in model.layers if l["is_norm"])
        r["stats_allreduces_per_step"] = 2 * r["norm_layers"] if world > 1 else 0
        r["buckets"] = int(_lib.load().fm_model_num_buckets(model._h))
        r["step_ms"] = timed(lambda: dp.train_on_batch(xp, tp))
        r["voxels_per_s"] = BATCH * world * float(np.prod(PATCH)) / (r["step_ms"] * 1e-3)
        if world > 1:
            dp.set_comm_enabled(False)
            r["step_ms_without_comm"] = timed(lambda: dp.train_on_batch(xp, tp))
            dp.set_comm_enabled(True)
            r["exposed_comm_ms"] = r["step_ms"] - r["step_ms_without_comm"]
            cmax = max(l["cout"] for l in model.layers if l["is_norm"])
            nbytes = (2 * cmax + 1) * 8
            ms, _ = dp.allreduce_bench(nbytes, iters=50)
            r["stats_message_bytes_max"] = nbytes
            r["small_allreduce_ms"] = max_over_ranks(ms)
        # parity: a fresh replica set, one data-parallel step, against one single-GPU step on the global batch
        del dp, model
        barrier()
        model = build(bn, local)
        res = DataParallelTrainer(model).train_on_batch(x, t)
        moving = [w for l, w in zip(model.layers, model.get_weights()[0::2]) if l["is_moving"]]
        barrier()
        if rank == 0 and world > 1:
            grads = model.get_gradients()
            ref = build(bn, local)
            shards = [make_batch(q) for q in range(world)]
            rres = ref.train_on_batch(np.concatenate([s[0] for s in shards]), np.concatenate([s[1] for s in shards]))
            names = {l["name"] for l in model.layers}
            cos = []
            rgrads = ref.get_gradients()
            for l, g, q, gb, qb in zip(model.layers, grads[0::2], rgrads[0::2], grads[1::2], rgrads[1::2]):
                if l["is_moving"]:
                    continue
                pairs = [(g, q)] + ([] if l["name"] + "_norm" in names else [(gb, qb)])   # pre-BN conv bias: noise
                for a, b in pairs:
                    a, b = a.astype(np.float64).ravel(), b.astype(np.float64).ravel()
                    cos.append(float(a @ b / max(np.linalg.norm(a) * np.linalg.norm(b), 1e-300)))
            rmov = [w for l, w in zip(ref.layers, ref.get_weights()[0::2]) if l["is_moving"]]
            mrel = max([float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-30))
                        for a, b in zip(moving, rmov)] or [0.0])
            r["dp_parity"] = dict(loss_dp=float(res[0]), loss_single_gpu_global_batch=float(rres[0]),
                                  loss_abs_diff=abs(float(res[0]) - float(rres[0])), min_grad_cos=min(cos),
                                  moving_mean_max_rel_diff=mrel,
                                  kernels="default (order-dependent fp32 accumulation in training passes)")
            del ref
        del model
        barrier()
        rec["bn_unet" if bn else "plain_unet"] = r
    if rank == 0:
        rec["gpu"] = gpu_identity(local)
        rec["steps"], rec["warmup"] = args.steps, args.warmup
        out = {}
        if os.path.exists(args.out):
            with open(args.out) as f:
                out = json.load(f)
        out.setdefault("config", dict(model="unet_model_3d", depth=DEPTH, n_base_filters=NF, patch=list(PATCH),
                                      per_gpu_batch=BATCH, timing="CUDA events on the library stream, max over ranks"))
        out.setdefault("runs", {})["%d_gpu" % world] = rec
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps(rec))
    barrier()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
