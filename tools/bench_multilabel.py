"""Cost of several labels (n_labels > 1) in the U-Net training step and in sliding-window inference.

    python tools/bench_multilabel.py --out DIR [--steps K] [--rounds R] [--warmup W]

Training: configs[1] (unet_model_3d depth 4 / 16 base filters, batch 8 x 1x64^3, soft-Dice loss) at n_labels 1, 2
and 4, one model each, alternated in one process: R rounds of K Model.train_on_batch steps per setting (host float32
inputs, the targets [8, n_labels, 64, 64, 64]), wall clock with a device synchronise at the end of every round, median
over the rounds. Inference: configs[0] (patch_wise_prediction of one 1x256x256x64 volume, patch 64^3, overlap_factor
0.5, batch 5) at n_labels 1 and 4, alternated the same way. Then a separate pass with the library's CUDA-event profiler
on gives the head / loss kernel times of a training step and their achieved bytes/s from the algorithmic bytes each
launcher states (head forward in training: C V 2 + L V 4 (t) + L V 4 (p)). Writes DIR/bench_multilabel.json with the
GPU name, power limit and max SM clock."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "fetal-mri-segmentation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

DEPTH, NF, PATCH, BATCH = 4, 16, (64, 64, 64), 8
TRAIN_LABELS, INFER_LABELS = (1, 2, 4), (1, 4)
VOLUME, INFER_BATCH = (1, 256, 256, 64), 5
PREFIXES = ("head_", "dice_", "label_transpose")


def gpu_identity(device):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(device)], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    from fetal_net import _lib
    from fetal_net.model import unet_model_3d
    from fetal_net.prediction import patch_wise_prediction
    assert torch.cuda.is_available(), "bench_multilabel.py needs a GPU"
    ctx = _lib.get_context(0)
    rng = np.random.default_rng(7)
    x = rng.standard_normal((BATCH, 1) + PATCH).astype(np.float32)
    models, targets = {}, {}
    for n in sorted(set(TRAIN_LABELS) | set(INFER_LABELS)):
        m = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, n_labels=n,
                          initial_learning_rate=1e-5)
        m.init_glorot_uniform(seed=0)
        models[n] = m
        targets[n] = (rng.random((BATCH, n) + PATCH) < 0.3).astype(np.float32)
    vol = rng.standard_normal(VOLUME).astype(np.float32)

    def train(n, steps):
        ctx.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            models[n].train_on_batch(x, targets[n])
        ctx.synchronize()
        return (time.perf_counter() - t0) / steps

    def infer(n, calls):
        ctx.synchronize()
        t0 = time.perf_counter()
        for _ in range(calls):
            patch_wise_prediction(models[n], vol, patch_shape=PATCH, overlap_factor=0.5, batch_size=INFER_BATCH)
        ctx.synchronize()
        return (time.perf_counter() - t0) / calls

    for n in TRAIN_LABELS:
        train(n, args.warmup)
    for n in INFER_LABELS:
        infer(n, args.warmup)
    tr = {n: [] for n in TRAIN_LABELS}
    inf = {n: [] for n in INFER_LABELS}
    for _ in range(args.rounds):
        for n in TRAIN_LABELS:
            tr[n].append(train(n, args.steps) * 1e3)
        for n in INFER_LABELS:
            inf[n].append(infer(n, max(1, args.steps // 4)) * 1e3)
    base_t, base_i = float(np.median(tr[1])), float(np.median(inf[1]))
    rec = dict(gpu=gpu_identity(0),
               train=dict(workload="configs[1]: unet_model_3d depth %d / %d base filters, batch %d x 1x%s, "
                          "Model.train_on_batch with host float32 inputs" % (DEPTH, NF, BATCH, "x".join(map(str, PATCH))),
                          timing="wall clock, %d rounds x %d steps per setting, settings alternated, median over rounds"
                          % (args.rounds, args.steps), n_labels={}),
               infer=dict(workload="configs[0]: patch_wise_prediction of one %s volume, patch %s, overlap_factor 0.5, "
                          "batch %d" % ("x".join(map(str, VOLUME)), "x".join(map(str, PATCH)), INFER_BATCH),
                          timing="wall clock, %d rounds x %d calls per setting, alternated, median over rounds"
                          % (args.rounds, max(1, args.steps // 4)), n_labels={}))
    for n in TRAIN_LABELS:
        ms = float(np.median(tr[n]))
        rec["train"]["n_labels"][str(n)] = dict(ms_per_step=ms, ms_rounds=tr[n], time_vs_one_label=ms / base_t)
    for n in INFER_LABELS:
        ms = float(np.median(inf[n]))
        rec["infer"]["n_labels"][str(n)] = dict(ms_per_call=ms, ms_rounds=inf[n], time_vs_one_label=ms / base_i)

    # head / loss kernels of a training step: a separate pass with the library's profiler on
    kernels = {}
    for n in TRAIN_LABELS:
        ctx.synchronize()
        ctx.profile(True)
        for _ in range(args.steps):
            models[n].train_on_batch(x, targets[n])
        ctx.synchronize()
        recs = [r for r in ctx.profile_records() if r[0].startswith(PREFIXES)]
        ctx.profile(False)
        per = {}
        for r in recs:
            per.setdefault(r[0], []).append(r)
        kernels[str(n)] = {k: dict(launches_per_step=len(v) / args.steps, us_median=1e3 * float(np.median([r[1] for r in v])),
                                   algorithmic_bytes=v[0][3],
                                   gb_per_s=v[0][3] / (float(np.median([r[1] for r in v])) * 1e-3) / 1e9)
                           for k, v in sorted(per.items())}
    rec["train_head_loss_kernels"] = kernels
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_multilabel.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"train": {k: v["ms_per_step"] for k, v in rec["train"]["n_labels"].items()},
                      "infer": {k: v["ms_per_call"] for k, v in rec["infer"]["n_labels"].items()}}))
    print(json.dumps(kernels))


if __name__ == "__main__":
    main()
