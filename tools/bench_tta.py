"""Flip test-time augmentation benchmark on BASELINE configs[0]: the reference's predict_flips (8 sliding-window passes
over the axis-flipped volume), the per-voxel median of the 8 maps and postprocess_prediction, for bench.py's seeded
256x256x64 volume and Glorot seed-0 model at overlap 0.5, on the host route and on the device route.
    python tools/bench_tta.py --out DIR [--steps K] [--warmup W] [--host-runs R]
Writes DIR/bench_tta.json with the GPU name, power limit and max SM clock, bit-exact flags of the device maps, median and
mask against the host composition, the wall times of the host route (host flip loop around patch_wise_prediction +
np.median + scipy post-processing) and of flip_tta_prediction / flip_tta_segmentation at batch 5 and 49, and the
per-kernel device times of the three TTA kernels with their algorithmic bytes. Every timed device loop runs --steps
iterations after --warmup untimed ones; the host route runs --host-runs times after one untimed run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "fetal-mri-segmentation_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

from bench_postprocess import DEPTH, NF, OVERLAP, PATCH, VOLUME, gpu_identity, timed  # noqa: E402

CONFIG = {"patch_shape": list(PATCH[:2]), "patch_depth": PATCH[2]}
TTA_KERNELS = ("flip_volume", "flip_crop", "median_passes")


def host_flips(model, data, batch):
    """predict_flips (prediction.py:65-85) as the reference runs it: flip on the host, one device sliding window per
    pass, un-flip on the host."""
    from fetal_net.device_tta import _AXES_SETS
    from fetal_net.prediction import flip_it, patch_wise_prediction
    maps = []
    for axes in _AXES_SETS:
        d = flip_it(data, axes)
        p = patch_wise_prediction(model, np.expand_dims(np.squeeze(d), 0), PATCH, overlap_factor=OVERLAP,
                                  batch_size=batch).squeeze()
        maps.append(flip_it(p, axes).squeeze())
    return maps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-runs", type=int, default=3)
    args = ap.parse_args()

    import torch
    from fetal_net import _lib
    from fetal_net.device_tta import flip_tta_prediction, flip_tta_segmentation
    from fetal_net.model import unet_model_3d
    from fetal_net.prediction import patch_wise_prediction, predict_flips
    from oracle import postprocess_oracle as ppo
    assert torch.cuda.is_available(), "bench_tta needs a GPU"

    ctx = _lib.get_context(0)
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH)
    model.init_glorot_uniform(seed=0)
    data = np.random.default_rng(0).standard_normal((1,) + VOLUME).astype(np.float32)

    ref_maps = host_flips(model, data, 5)
    ref_med = np.median(np.stack(ref_maps), axis=0)
    pp = dict(gaussian_std=1, threshold=0.5, fill_holes=True, connected_component=True)
    try:
        ref_mask = ppo.postprocess_prediction(ref_med, **pp)
    except ValueError:
        # the seeded network may leave nothing above 0.5: threshold at the median instead, so that every stage works
        pp["threshold"] = float(np.median(ref_med))
        ref_mask = ppo.postprocess_prediction(ref_med, **pp)

    nvox = int(np.prod(VOLUME))
    res = dict(gpu=gpu_identity(), workload=dict(volume=VOLUME, input="[1,X,Y,Z] float32", patch=PATCH,
                                                 overlap_factor=OVERLAP, patches_per_pass=49, passes=8, **pp),
               steps=args.steps, warmup=args.warmup)
    maps = predict_flips(data, model, OVERLAP, CONFIG)
    mask, med = flip_tta_segmentation(data, model, OVERLAP, CONFIG, batch_size=49, return_prediction=True, **pp)
    res["bit_exact"] = dict(maps=all(np.array_equal(a, b) for a, b in zip(maps, ref_maps)),
                            median=bool(np.array_equal(med, ref_med)),
                            median_of_prediction=bool(np.array_equal(flip_tta_prediction(data, model, OVERLAP, CONFIG,
                                                                                         batch_size=5), ref_med)),
                            mask=bool(np.array_equal(mask, ref_mask)))
    res["mask_voxels"] = int(ref_mask.sum())
    del maps

    def host_route(batch):
        m = host_flips(model, data, batch)
        return ppo.postprocess_prediction(np.median(np.stack(m), axis=0), **pp)

    res["host_route"] = {}
    for batch in (5, 49):
        r = timed(lambda: host_route(batch), args.host_runs, 1)
        r["what"] = "host flip loop around patch_wise_prediction (device) + np.median + scipy post-processing"
        res["host_route"]["batch%d" % batch] = r
    # the host route's parts, once each at batch 49
    t0 = time.perf_counter()
    m = host_flips(model, data, 49)
    t1 = time.perf_counter()
    stack = np.stack(m)
    med_h = np.median(stack, axis=0)
    t2 = time.perf_counter()
    ppo.postprocess_prediction(med_h, **pp)
    t3 = time.perf_counter()
    res["host_route_parts_batch49_ms"] = dict(flip_loop=(t1 - t0) * 1e3, stack_and_median=(t2 - t1) * 1e3,
                                              scipy_postprocess=(t3 - t2) * 1e3, cpu_count=os.cpu_count())
    del m, stack

    res["device_route"] = {}
    for batch in (5, 49):
        res["device_route"]["flip_tta_prediction_batch%d" % batch] = timed(
            lambda: flip_tta_prediction(data, model, OVERLAP, CONFIG, batch_size=batch), args.steps, args.warmup)
        res["device_route"]["flip_tta_segmentation_batch%d" % batch] = timed(
            lambda: flip_tta_segmentation(data, model, OVERLAP, CONFIG, batch_size=batch, **pp), args.steps,
            args.warmup)
    res["device_route"]["predict_flips_maps_batch5"] = timed(lambda: predict_flips(data, model, OVERLAP, CONFIG),
                                                             args.steps, args.warmup)
    res["patch_wise_prediction_batch49"] = timed(
        lambda: patch_wise_prediction(model, data, PATCH, overlap_factor=OVERLAP, batch_size=49), args.steps,
        args.warmup)

    # per-kernel device times: CUDA events around every launch, averaged over --steps calls
    ctx.profile(True)
    for _ in range(args.steps):
        flip_tta_segmentation(data, model, OVERLAP, CONFIG, batch_size=49, **pp)
    recs = ctx.profile_records()
    ctx.profile(False)
    kernels, total = {}, 0.0
    for name, ms, flops, nbytes in recs:
        total += ms / args.steps
        if name not in TTA_KERNELS:
            continue
        k = kernels.setdefault(name, dict(ms=0.0, bytes=0.0, launches=0))
        k["ms"] += ms / args.steps
        k["bytes"] += nbytes / args.steps
        k["launches"] += 1
    for k in kernels.values():
        k["launches"] //= args.steps
        k["implied_gbs"] = k["bytes"] / (k["ms"] * 1e-3) / 1e9 if k["ms"] > 0 else None
    res["tta_kernels_per_call"] = kernels
    res["device_ms_all_kernels_per_call"] = total
    res["tta_kernels_note"] = (
        "algorithmic bytes per call (each array read / written once): flip_volume 8 B/voxel for each pass with a "
        "nonzero input mask, 6 of 8 for this [1,X,Y,Z] input (the 16.8 MB float32 volume and its flipped copy fit the "
        "126 MB L2), flip_crop 16 B/voxel for 8 passes (reads the 33.5 MB "
        "padded map the overlap-add has just written, L2-resident; writes a 33.5 MB stack slot), median_passes "
        "72 B/voxel once (the 268 MB stack exceeds L2, so it is read from HBM except for the most recent slots). "
        "%d voxels." % nvox)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_tta.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
