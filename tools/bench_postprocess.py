"""Post-processing benchmark on BASELINE configs[0]: the reference's postprocess_prediction (gaussian 1, threshold 0.5,
fill holes, largest connected component) of the 256x256x64 float64 map that patch_wise_prediction returns for bench.py's
seeded volume and model, on the host with scipy and on the device.
    python tools/bench_postprocess.py --out DIR [--steps K] [--warmup W] [--scipy-runs R]
Writes DIR/bench_postprocess.json with the GPU name and power limit, scipy's median time, the wall time of fm_postprocess
(host map -> host mask), the per-kernel device times with their algorithmic bytes, and patch_wise_segmentation against
patch_wise_prediction + scipy end to end. Every timed loop runs --steps iterations after --warmup untimed ones."""
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

PATCH, VOLUME, OVERLAP, DEPTH, NF = (64, 64, 64), (256, 256, 64), 0.5, 4, 16     # bench.py's configs[0]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return dict(ms_median=float(np.median(ts)) * 1e3, ms_min=float(np.min(ts)) * 1e3, ms_mean=float(np.mean(ts)) * 1e3,
                runs=steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scipy-runs", type=int, default=5)
    args = ap.parse_args()

    import torch
    from fetal_net import _lib
    from fetal_net.device_postprocess import patch_wise_segmentation, postprocess_prediction
    from fetal_net.model import unet_model_3d
    from fetal_net.prediction import patch_wise_prediction
    from oracle import postprocess_oracle as ppo
    assert torch.cuda.is_available(), "bench_postprocess needs a GPU"

    ctx = _lib.get_context(0)
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH)
    model.init_glorot_uniform(seed=0)
    vol = np.random.default_rng(0).standard_normal((1,) + VOLUME).astype(np.float32)
    prob = patch_wise_prediction(model, vol, PATCH, overlap_factor=OVERLAP, batch_size=49)
    pred = np.ascontiguousarray(prob.squeeze())
    pp = dict(gaussian_std=1, threshold=0.5, fill_holes=True, connected_component=True)
    try:
        ref = ppo.postprocess_prediction(pred, **pp)
    except ValueError:
        # the seeded network may leave nothing above 0.5: threshold at the median instead, so that every stage works
        pp["threshold"] = float(np.median(pred))
        ref = ppo.postprocess_prediction(pred, **pp)

    res = dict(gpu=gpu_identity(), workload=dict(volume=VOLUME, map_dtype="float64", map_bytes=int(pred.nbytes),
                                                 patch=PATCH, overlap_factor=OVERLAP, patches=49, **pp),
               steps=args.steps, warmup=args.warmup)
    dev = postprocess_prediction(pred, **pp)
    res["bit_exact_vs_scipy"] = bool(np.array_equal(dev, ref))
    res["mask_voxels"] = int(ref.sum())

    ts = []
    for _ in range(args.scipy_runs):
        t0 = time.perf_counter()
        ppo.postprocess_prediction(pred, **pp)
        ts.append(time.perf_counter() - t0)
    res["scipy_postprocess"] = dict(ms_median=float(np.median(ts)) * 1e3, runs=args.scipy_runs, cpu_count=os.cpu_count(),
                                    note="oracle/postprocess_oracle.py: scipy.ndimage with np.bincount for the sizes")
    res["fm_postprocess_wall"] = timed(lambda: postprocess_prediction(pred, **pp), args.steps, args.warmup)
    res["fm_postprocess_wall"]["what"] = "host float64 map -> H2D -> kernels -> D2H -> host bool mask"

    # per-kernel device times: CUDA events around every launch, averaged over --steps calls
    ctx.profile(True)
    for _ in range(args.steps):
        postprocess_prediction(pred, **pp)
    recs = ctx.profile_records()
    ctx.profile(False)
    kernels = {}
    for name, ms, flops, nbytes in recs:
        k = kernels.setdefault(name, dict(ms=0.0, bytes=nbytes, launches=0))
        k["ms"] += ms / args.steps
        k["launches"] += 1
    for k in kernels.values():
        k["launches"] //= args.steps
        k["implied_gbs"] = k["bytes"] / (k["ms"] * 1e-3) / 1e9 if k["ms"] > 0 else None
    res["device_kernels"] = kernels
    res["device_ms_total"] = sum(k["ms"] for k in kernels.values())
    res["device_note"] = ("algorithmic bytes (each array read / written once); the 33.5 MB map and the 4 MB mask and "
                          "16 MB label arrays stay in the 126 MB L2 between kernels, so the implied bandwidth is not an "
                          "HBM share")

    seg = lambda: patch_wise_segmentation(model, vol, PATCH, overlap_factor=OVERLAP, batch_size=49, **pp)
    host = lambda: ppo.postprocess_prediction(patch_wise_prediction(model, vol, PATCH, overlap_factor=OVERLAP,
                                                                    batch_size=49).squeeze(), **pp)
    res["bit_exact_segmentation"] = bool(np.array_equal(seg(), ref))
    res["patch_wise_segmentation"] = timed(seg, args.steps, args.warmup)
    res["patch_wise_prediction"] = timed(lambda: patch_wise_prediction(model, vol, PATCH, overlap_factor=OVERLAP,
                                                                       batch_size=49), args.steps, args.warmup)
    res["patch_wise_prediction_plus_scipy"] = timed(host, args.scipy_runs, 1)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_postprocess.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
