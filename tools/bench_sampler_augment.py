"""Cost of the device sampler's augmentations in the sampled training step (bench.py's train_sampled workload: 6
resident cases of 160x160x96, batch 8 x 64^3 cut on the device, unet_model_3d depth 4 / 16 base filters).

    python tools/bench_sampler_augment.py --out DIR [--steps K] [--rounds R] [--warmup W]

Four `device_augment` settings, alternated in one process (R rounds of K steps each, wall clock around
DeviceSampler.train_on_next_batch with a device synchronise at the end of every round; median over the rounds):
none; flip + intensity + noise; plus rotate / scale / translate; plus elastic. Then, in a separate profiled pass, the
sample_patches / sample_patches_warp kernel times from the library's CUDA-event profiler with their algorithmic bytes
(8 per output element), and the host time of scipy.ndimage.map_coordinates resampling the same batch (data trilinear,
truth nearest) through a warp. Writes DIR/bench_sampler_augment.json with the GPU name, power limit and max SM clock."""
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

DEPTH, NF, PATCH, BATCH, SHAPE, NCASES = 4, 16, (64, 64, 64), 8, (160, 160, 96), 6
BASIC = dict(flip=True, intensity=(0.9, 1.1), noise_sigma=0.05)
AFFINE = dict(BASIC, rotate=(15.0, 15.0, 15.0), scale=(0.1, 0.1, 0.1), translate=(5.0, 5.0, 5.0))
SETTINGS = [("none", None), ("flip_intensity_noise", BASIC), ("plus_rotate_scale_translate", AFFINE),
            ("plus_elastic", dict(AFFINE, elastic=dict(alpha=3.0, grid=4)))]


def gpu_identity(device):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(device)], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def host_resample_seconds(data, truth, cases, corners, warps):
    """scipy.ndimage.map_coordinates of the batch's data (order 1) and truth (order 0) patches through the warps."""
    from scipy import ndimage
    from oracle import sampler_oracle as so
    t0 = time.perf_counter()
    for c, corner, w in zip(cases, corners, warps):
        s = so.source_coords(corner, PATCH, 0, PATCH[2], w)
        ndimage.map_coordinates(data[c], s, order=1, mode="nearest")
        ndimage.map_coordinates(truth[c], s, order=0, mode="nearest")
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    from fetal_net import _lib
    from fetal_net.device_sampler import DeviceSampler, warp_matrix
    from fetal_net.model import unet_model_3d
    assert torch.cuda.is_available(), "bench_sampler_augment.py needs a GPU"
    ctx = _lib.get_context(0)
    rng = np.random.default_rng(7)
    data = [rng.standard_normal(SHAPE).astype(np.float32) for _ in range(NCASES)]
    truth = [(rng.random(SHAPE) < 0.3).astype(np.float32) for _ in range(NCASES)]
    np.random.seed(1)
    sampler = DeviceSampler(data, truth, list(range(NCASES)), batch_size=BATCH, patch_shape=PATCH,
                            shuffle_index_list=True, skip_blank=True, truth_index=0, truth_size=PATCH[2], is3d=True)
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, initial_learning_rate=1e-4)
    model.init_glorot_uniform(seed=0)

    def run(setting, steps):
        sampler.device_augment = setting
        ctx.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            sampler.train_on_next_batch(model)
        ctx.synchronize()
        return (time.perf_counter() - t0) / steps

    for _, setting in SETTINGS:
        run(setting, args.warmup)
    per = {name: [] for name, _ in SETTINGS}
    for _ in range(args.rounds):
        for name, setting in SETTINGS:
            per[name].append(run(setting, args.steps) * 1e3)
    base = float(np.median(per["none"]))
    rec = dict(gpu=gpu_identity(0), workload="DeviceSampler.train_on_next_batch: %d resident cases of %s, batch %d x "
               "%s, unet_model_3d depth %d / %d base filters" % (NCASES, "x".join(map(str, SHAPE)), BATCH,
                                                               "x".join(map(str, PATCH)), DEPTH, NF),
               timing="wall clock, %d rounds x %d steps per setting, settings alternated, median over rounds" %
               (args.rounds, args.steps), settings={})
    for name, setting in SETTINGS:
        ms = float(np.median(per[name]))
        rec["settings"][name] = dict(device_augment=setting, ms_per_step=ms, ms_rounds=per[name],
                                     voxels_per_s=BATCH * float(np.prod(PATCH)) / (ms * 1e-3),
                                     rate_vs_unaugmented=base / ms)

    # kernel times: a separate pass with the library's profiler on
    kernels = {}
    for name, setting in SETTINGS:
        sampler.device_augment = setting
        ctx.synchronize()
        ctx.profile(True)
        for _ in range(args.steps):
            sampler.train_on_next_batch(model)
        ctx.synchronize()
        recs = [r for r in ctx.profile_records() if r[0] in ("sample_patches", "sample_patches_warp")]
        ctx.profile(False)
        ms = [r[1] for r in recs]
        nbytes = recs[0][3]
        kernels[name] = dict(kernel=recs[0][0], launches=len(recs), us_mean=1e3 * float(np.mean(ms)),
                             us_median=1e3 * float(np.median(ms)), algorithmic_bytes=nbytes,
                             gb_per_s=nbytes / (float(np.median(ms)) * 1e-3) / 1e9)
    rec["sampler_kernels"] = kernels

    # the same batch resampled on the host (scipy, one thread)
    cases, corners = sampler.draw()
    r = np.random.default_rng(11)
    warps = [dict(matrix=warp_matrix(r.normal(0, 15, 3), np.clip(1 + r.normal(0, 0.1, 3), 0.5, 2)).astype(np.float32),
                  offset=r.normal(0, 5, 3).astype(np.float32), alpha=np.zeros(3, np.float32), seed=0, grid=0)
             for _ in range(BATCH)]
    sec = host_resample_seconds(data, truth, cases, corners, warps)
    rec["host_map_coordinates"] = dict(seconds_per_batch=sec, device_steps_equivalent=sec / (base * 1e-3),
                                       note="scipy.ndimage.map_coordinates order 1 (data) + order 0 (truth) of %d "
                                            "patches of %s through a rotate/scale/translate warp, single-threaded, "
                                            "on the GPU host's CPU" % (BATCH, "x".join(map(str, PATCH))))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_sampler_augment.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: (v["ms_per_step"], v["rate_vs_unaugmented"]) for k, v in rec["settings"].items()}))
    print(json.dumps(kernels))
    print("host map_coordinates %.3f s per batch" % sec)


if __name__ == "__main__":
    main()
