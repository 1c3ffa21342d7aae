#!/usr/bin/env python
"""bench.py — throughput of the hot path on B200 (and the reference's CPU path beside it).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload all|train|infer]
                    [--dump-outputs DIR]

ONE JSON line (rank 0). The top-level record is BASELINE.json's metric on configs[1]: one "step" = one soft-Dice
training step (fwd + loss + bwd + Keras-Adam) of the depth-4 / 16-filter 3D U-Net on a batch of 8 synthetic 64^3
patches per GPU (weak scaling: global batch 8 N, Dice-sum + bucketed gradient all-reduce on the library's own NCCL
communicator). Nested records cover the rest of the metric:

  infer          configs[0]: patch_wise_prediction of one 1x256x256x64 volume, patch 64^3, overlap_factor 0.5 (49
                 patches): device time, e2e with PAGEABLE and with pinned host buffers, conv / HBM rooflines.
  train_sampled  (N = 1) the same step fed by the on-device patch sampler (DeviceSampler.train_on_next_batch).
  families       (N = 1) configs[2] (Isensee-2017, 2 x 128x128x64) and configs[3] (2.5D U-Net, 8 x 256x256x6): step,
                 e2e, predict, roofline of their dominant kernel.
  train_cfg5     (N > 1) configs[4]'s patch shape: batch 8 x 1x128x128x64 per GPU, same data-parallel step.
  infer_sharded  (N > 1) sharded_patch_wise_prediction of one 1x512x512x128 volume, patch 128x128x64 (147 patches).
  allreduce      (N > 1) gradient all-reduce: bytes, standalone ms and bus GB/s = 2 (n-1)/n * bytes / t, and the
                 EXPOSED communication time per step (step with collectives on minus step with them switched off).
  dp_parity      (N > 1) one data-parallel step on the default kernels vs a single-GPU step on the full global batch.

`value` is timed with CUDA events on the stream the kernels are launched on, inputs already resident in HBM; `e2e` goes
through the reference-facing Python API (Model.train_on_batch / patch_wise_prediction) with host buffers, H2D + D2H inside
the timed region. `--impl reference` times the oracle port of the reference's CPU path on the host cores. Every timed
loop of every record runs exactly `--steps` iterations (reported as `steps`); the warm-up calls before it are untimed.

`--dump-outputs DIR` writes, after the timed steps, what the caller of each timed path received from its last step as
DIR/<name>.npy: train_metrics (loss, binary_accuracy, vod_coefficient, dice_coefficient as fm_train_step_device returns
them) and infer_prediction (the float64 patch_wise_prediction result of the last timed call, bit for bit). The inputs
are seeded, so two builds can be compared output for output. The model's weights are not dumped: a training pass is not
bit-reproducible (fp32 red.add of the weight gradients, three-issuer marching kernels; DESIGN.md §5), and Adam turns a
last-bit difference of a near-zero gradient into an update of the size of the learning rate, so after a few steps the
weights of two runs differ far beyond rounding while the metrics agree to it.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "fetal-mri-segmentation_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
# the benchmark leaves the source tree as it found it (it may be read-only): no bytecode caches next to the modules
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

PATCH = (64, 64, 64)
PATCH5 = (128, 128, 64)
BATCH = 8
DEPTH, NF = 4, 16
VOLUME = (256, 256, 64)
VOLUME5 = (512, 512, 128)
OVERLAP = 0.5
METRIC = "U-Net train voxels/sec"
UNIT = "voxels/s"

# algorithmic FLOPs (SURVEY.md §8d / App. B): 3D U-Net d4 nf16
FWD_GF_PER_PATCH = 118.472          # 64^3
FIRST_CONV_GF = 0.226
FWD_GF_PER_PATCH5 = 473.889         # 128x128x64
FIRST_CONV_GF5 = 0.906
NPARAMS = 4079713


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]),
                    tf_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


DUMP_LIMIT_BYTES = 64 << 20


def write_dump(path, arrays):
    """Writes {name: array} as path/<name>.npy (float64 stays float64, everything else becomes float32)."""
    out = {k: np.ascontiguousarray(a, dtype=np.float64 if np.asarray(a).dtype == np.float64 else np.float32)
           for k, a in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT_BYTES, "dump of %d bytes exceeds %d" % (total, DUMP_LIMIT_BYTES)
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


def ncu_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, averaged over the kernel's launches of one
    step / one call) from the committed `ncu --set full` capture (profiles/r2_dram_traffic.json, written by
    tools/summarize_profiles_r2.py from the capture of tools/r2_step13.sh)."""
    out = {}
    path = os.path.join(ROOT, "profiles", "r2_dram_traffic.json")
    if os.path.exists(path):
        for k, v in json.load(open(path)).items():
            out[k] = (float(v["avg_bytes_per_launch"]), "r2_dram_traffic.json")
    return out


# bench kernel name (ctx.profile) -> key in profiles/r2_dram_traffic.json, per workload
TRAFFIC_KEYS = {
    "train": {"conv3d_wgrad_march": "bwd/conv3d_wgrad_march_kernel", "conv3d_march_fprop": "fwd/conv3d_march2_kernel<1, 32>",
              "conv3d_march_dgrad": "bwd/conv3d_march2_kernel<1, 32>", "maxpool3d_bwd": "bwd/maxpool3d_bwd_kernel<2>",
              "maxpool3d_fwd": "fwd/maxpool3d_fwd_kernel<2>", "head_fwd_dice": "fwd/head_fwd_tpv_kernel<32, 1>",
              "head_bwd_dice": "bwd/head_bwd_kernel", "upsample3d_fwd": "fwd/upsample3d_fwd_kernel<2>",
              "adam": "bwd/adam_kernel"},
    "infer": {"conv3d_march_fprop": "infer/conv3d_march2_kernel<2, 32>", "conv3d_tc_fprop": "infer/conv3d_tc_fprop_kernel",
              "reassemble": "infer/reassemble4_kernel", "gather_patches": "infer/gather_patches4_kernel",
              "maxpool3d_fwd": "infer/maxpool3d_fwd_kernel<2>", "upsample3d_fwd": "infer/upsample3d_fwd_kernel<2>",
              "head_fwd": "infer/head_fwd_tpv_kernel<32, 0>"},
}


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe). NVML is polled from a thread
    every few ms (nvidia-smi -lms cannot deliver a sample inside a 50 ms region); the fields are the ones
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*` prints."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device):
        self.device, self.rows, self.thread, self.run = device, [], None, False
        self.max_mhz = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(int(self.device))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.run = True
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        nv = self.nv
        while self.run:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        if self.nv is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvml unavailable"], samples=0)
        self.run = False
        self.thread.join(timeout=1)
        sm = [r[0] for r in self.rows]
        reasons = sorted({nm for _, rs in self.rows for bit, nm in self.REASONS.items() if rs & bit})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=self.max_mhz, reasons=reasons,
                    samples=len(sm))


def tensor_peak(pk, clocks):
    """The denominator for a tensor-bound kernel: the burst cuBLAS figure when the timed region ran at the maximum SM
    clock with no power cap active (a short region), else the sustained one. Both fractions are printed anyway."""
    burst = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and
                 clocks["sm_mhz"] >= 0.97 * clocks["sm_max_mhz"] and "sw_power_cap" not in (clocks.get("reasons") or []))
    return (pk["tf_burst"], "burst") if burst else (pk["tf_sustained"], "sustained")


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle (PyTorch-CPU fp32 restatement of the Keras/TF path) on the
# host cores. The reference itself cannot run here (no TensorFlow/Keras in the image; SURVEY.md §8c).
# ------------------------------------------------------------------------------------------------
def cpu_train_steps(batch, steps, warmup, budget_s=None):
    """Times `steps` full oracle training steps (after `warmup`) on `batch` 64^3 patches; stops early only when a
    budget is given and exceeded. Returns (list of seconds per timed step, torch thread count)."""
    import torch
    from oracle import unet_oracle as uo
    torch.set_num_threads(os.cpu_count())
    rng = np.random.default_rng(1)
    w = uo.glorot_uniform_weights(uo.unet3d_layers(DEPTH, NF), seed=0)
    x = rng.standard_normal((batch, 1) + PATCH).astype(np.float32)
    t = (np.random.default_rng(2).random(x.shape) < 0.3).astype(np.float32)
    state, times = {}, []
    t_start = time.time()
    for i in range(warmup + steps):
        t0 = time.time()
        uo.unet3d_train_step(x, t, w, state, 1e-4)
        if i >= warmup:
            times.append(time.time() - t0)
        if budget_s is not None and time.time() - t_start > budget_s and len(times) >= 1:
            break
    return times, torch.get_num_threads()


def cpu_infer_sample():
    """A bounded sample of configs[0] on the host cores: the oracle network driven through the reference's own
    sliding-window control flow on a 97x97x64 sub-volume (4 patches of 64^3 at overlap_factor 0.5)."""
    import torch
    from oracle import prediction_oracle as po
    from oracle import unet_oracle as uo
    torch.set_num_threads(os.cpu_count())
    w = uo.glorot_uniform_weights(uo.unet3d_layers(DEPTH, NF), seed=0)
    vol = np.random.default_rng(0).standard_normal((1, 97, 97, 64)).astype(np.float32)
    model = uo.OracleModel(w, (1,) + PATCH)
    po.patch_wise_prediction(model, vol[:, :64, :64], PATCH, overlap_factor=OVERLAP)      # warm-up: one patch
    t0 = time.time()
    po.patch_wise_prediction(model, vol, PATCH, overlap_factor=OVERLAP)
    sec = time.time() - t0
    return dict(value=97 * 97 * 64 / sec, unit=UNIT, cores=os.cpu_count(), kind="port",
                sample="oracle network through the reference's patch_wise_prediction control flow on a 97x97x64 "
                       "sub-volume (4 patches of 64^3), one timed call, %d threads; patch-voxels/s = %.3g" % (
                           torch.get_num_threads(), 4 * 64 ** 3 / sec))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the full configs[1] step (8 patches), exactly --steps timed steps after --warmup untimed ones
    times, threads = cpu_train_steps(BATCH, args.steps, args.warmup)
    sec = float(np.mean(times))
    vps = BATCH * int(np.prod(PATCH)) / sec
    sample = "oracle (PyTorch-CPU fp32 restatement of the Keras/TF path) full train step on 8 x 64^3, %d timed steps " \
             "after %d warm-up, %d threads" % (len(times), args.warmup, threads)
    line = dict(impl="reference", metric=METRIC, value=vps, unit=UNIT, n_gpus=args.gpus, steps=len(times),
                warmup=args.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", config=workload_config(args.gpus),
                cpu_baseline=dict(value=vps, unit=UNIT, cores=os.cpu_count(), kind="port", sample=sample),
                e2e=dict(value=vps, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def workload_config(n_gpus):
    return dict(workload="unet_model_3d(depth=4,n_base_filters=16) soft-Dice train step, batch 8 x 1x64x64x64 per GPU "
                         "(BASELINE configs[1])",
                global_batch=BATCH * n_gpus, patch=list(PATCH), parallelism="dp%d" % n_gpus,
                l2="working set ~1.9 GB of activations+gradients per step >> 126 MB L2 (no explicit flush needed)")


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
class Env:
    pass


def setup_env(need_dist):
    import torch
    import torch.distributed as dist
    from fetal_net import _lib
    e = Env()
    e.torch, e.dist, e._lib = torch, dist, _lib
    e.world = int(os.environ.get("WORLD_SIZE", "1"))
    e.rank = int(os.environ.get("RANK", "0"))
    e.local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(e.local)
    if e.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda:%d" % e.local))   # control plane only
    e.ctx = _lib.get_context(e.local)
    e.lib = _lib.load()
    e.stream = torch.cuda.ExternalStream(e.ctx.stream, device="cuda:%d" % e.local)
    return e


def barrier(e):
    if e.world > 1:
        e.dist.barrier()
    e.torch.cuda.synchronize()
    e.ctx.synchronize()


def max_over_ranks(e, v):
    if e.world == 1:
        return float(v)
    tt = e.torch.tensor([float(v)], device="cuda", dtype=e.torch.float64)
    e.dist.all_reduce(tt, op=e.dist.ReduceOp.MAX)
    return float(tt.item())


def timed_device(e, fn, steps):
    """ms for `steps` calls, CUDA events on the library's stream, barrier + sync on both sides, max over ranks."""
    torch = e.torch
    barrier(e)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(e.stream)
    for _ in range(steps):
        fn()
    e1.record(e.stream)
    barrier(e)
    return max_over_ranks(e, e0.elapsed_time(e1))


def timed_wall(e, fn, steps):
    barrier(e)
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    barrier(e)
    return max_over_ranks(e, (time.perf_counter() - t0) / steps)


def aggregate(recs):
    agg = {}
    for name, kms, fl, by in recs:
        a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
        a[0] += 1
        a[1] += kms
        a[2] += fl
        a[3] += by
    return agg


def roofline_of(name, a, nrep, total_ms, pk, clocks, traffic, workload="train"):
    cnt, kms, fl, by = a
    tkey = TRAFFIC_KEYS.get(workload, {}).get(name)
    tr = traffic.get(tkey) if tkey else None
    if fl > 0:
        ach = fl / kms / 1e9        # TFLOP/s: algorithmic flops per launch / avg launch duration
        peak, which = tensor_peak(pk, clocks)
        return dict(kernel=name, bound="tensor", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak,
                    frac_burst=ach / pk["tf_burst"], frac_sustained=ach / pk["tf_sustained"],
                    peak_source="%s (%s)" % (pk["src"], which), traffic=tr[0] if tr else None,
                    traffic_note=("ncu --set full capture, profiles/%s" % tr[1]) if tr else None,
                    launches_per_step=cnt // nrep, avg_launch_ms=kms / cnt, algorithmic_flops_per_launch=fl / cnt,
                    share_of_step=kms / total_ms)
    ach = by / kms / 1e6
    return dict(kernel=name, bound="hbm", achieved=ach, peak=pk["hbm"], unit="GB/s", frac=ach / pk["hbm"],
                peak_source=pk["src"], traffic=tr[0] if tr else None,
                traffic_note=("ncu --set full capture, profiles/%s" % tr[1]) if tr else None,
                launches_per_step=cnt // nrep, avg_launch_ms=kms / cnt, algorithmic_bytes_per_launch=by / cnt,
                share_of_step=kms / total_ms)


def make_batch(rank, shape, batch=BATCH):
    rng = np.random.default_rng(1 + rank)
    x = rng.standard_normal((batch, 1) + tuple(shape)).astype(np.float32)
    t = (np.random.default_rng(2 + rank).random(x.shape) < 0.3).astype(np.float32)
    return x, t


def bench_train(e, args, patch, fwd_gf, first_gf, steps, warmup, with_profile, dump=None):
    """The data-parallel (or single-GPU) training step on `patch`; returns the record dict (rank 0) or None. With a
    `dump` dict, rank 0 puts the metrics of the last timed step into it."""
    torch, _lib, lib, ctx = e.torch, e._lib, e.lib, e.ctx
    from fetal_net.distributed import DataParallelTrainer
    from fetal_net.model import unet_model_3d
    model = unet_model_3d(input_shape=(1,) + tuple(patch), n_base_filters=NF, depth=DEPTH, initial_learning_rate=1e-4,
                          device=e.local)
    model.init_glorot_uniform(seed=0)
    x, t = make_batch(e.rank, patch)
    xd, td = torch.as_tensor(x).cuda(), torch.as_tensor(t).cuda()
    xp, tp = torch.as_tensor(x).pin_memory(), torch.as_tensor(t).pin_memory()
    dp = DataParallelTrainer(model) if e.world > 1 else None
    m4 = np.zeros(4, np.float32)
    lr = 1e-4
    last = {}

    def step_device():
        if dp is None:
            _lib.check(lib.fm_train_step_device(model._h, xd.data_ptr(), td.data_ptr(), BATCH, lr, _lib.fptr(m4)))
        else:
            # the data-parallel entry point takes host buffers (pinned: staged on the copy stream while the previous
            # step's backward still runs); the collective structure is the real one
            last["m"] = dp.train_on_batch(xp.numpy(), tp.numpy())

    def step_e2e(xa, ta):
        r = (model if dp is None else dp).train_on_batch(xa, ta)
        last["m"] = r
        return r

    for _ in range(max(warmup, 3)):
        step_device()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(e.local)
    if e.rank == 0:
        sampler.start()
    ms = timed_device(e, step_device, steps)
    clocks = sampler.stop() if e.rank == 0 else None
    launches = ctx.launch_count() - launches0
    if dump is not None and e.rank == 0:
        dump["train_metrics"] = np.asarray(last["m"] if dp is not None else m4, np.float32).copy()
    ms_step = ms / steps
    vox_step = BATCH * int(np.prod(patch)) * e.world
    rec = dict(value=vox_step / (ms_step * 1e-3), ms_per_step=ms_step, clocks=clocks, gpu_launches=int(launches))

    # e2e through the public API: pinned host buffers (the contract's figure) and pageable ones (what a caller that
    # feeds plain NumPy batches from the reference's generator gets)
    for _ in range(2):
        step_e2e(xp.numpy(), tp.numpy())
    s_pin = timed_wall(e, lambda: step_e2e(xp.numpy(), tp.numpy()), steps)
    for _ in range(2):
        step_e2e(x, t)
    s_page = timed_wall(e, lambda: step_e2e(x, t), steps)
    nbytes = int(x.nbytes + t.nbytes)
    rec["e2e"] = dict(value=vox_step / s_pin, unit=UNIT, h2d_bytes_per_step=nbytes, d2h_bytes_per_step=64,
                      ms_per_step=s_pin * 1e3, host_buffers="pinned")
    rec["e2e_pageable"] = dict(value=vox_step / s_page, unit=UNIT, h2d_bytes_per_step=nbytes, d2h_bytes_per_step=64,
                               ms_per_step=s_page * 1e3, host_buffers="pageable numpy")
    rec["loss"] = float(last["m"][0]) if "m" in last else float(m4[0])
    rec["conv_tflops_whole_step"] = e.world * BATCH * (3 * fwd_gf - first_gf) / ms_step

    if with_profile and e.rank == 0:
        # roofline leg: two extra steps with per-launch CUDA events (rank 0 only, no collectives inside)
        pk = peaks()
        ctx.profile(True)
        nprof = 2
        for _ in range(nprof):
            if dp is None:
                _lib.check(lib.fm_train_step_device(model._h, xd.data_ptr(), td.data_ptr(), BATCH, lr, _lib.fptr(m4)))
            else:
                _lib.check(lib.fm_train_forward(model._h, _lib.fptr(x), _lib.fptr(t), BATCH))
                _lib.check(lib.fm_train_backward(model._h))
        agg = aggregate(ctx.profile_records())
        ctx.profile(False)
        total_ms = sum(a[1] for a in agg.values())
        traffic = ncu_traffic()
        rec["kernel_breakdown"] = {
            k: dict(launches=a[0] // nprof, ms_per_step=a[1] / nprof, share=a[1] / total_ms,
                    tflops=(a[2] / a[1] / 1e9) if a[1] > 0 and a[2] > 0 else None,
                    gbs=(a[3] / a[1] / 1e6) if a[1] > 0 and a[3] > 0 else None,
                    frac_of_peak=((a[2] / a[1] / 1e9) / tensor_peak(pk, clocks)[0]) if a[2] > 0 else
                    ((a[3] / a[1] / 1e6) / pk["hbm"] if a[3] > 0 else None))
            for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])}
        top = max(agg.items(), key=lambda kv: kv[1][1])
        rec["roofline"] = roofline_of(top[0], top[1], nprof, total_ms, pk, clocks, traffic)
        rec["rooflines"] = {k: roofline_of(k, agg[k], nprof, total_ms, pk, clocks, traffic)
                            for k in TRAFFIC_KEYS["train"] if k in agg}
    rec["_model"], rec["_dp"] = model, dp
    return rec


def bench_train_sampled(e, steps, plain_ms):
    """fit_generator's inner loop fed by the on-device sampler (fetal_net.device_sampler, the generator.py:243-348
    counterpart): per step the host draws (case, corner) with the reference generator's RNG call sequence, 32 bytes per
    sample cross the bus, the patches are cut from the resident volume set straight into the network's input buffers.
    Wall clock around DeviceSampler.train_on_next_batch at the configs[1] shape, beside the plain device step."""
    from fetal_net.device_sampler import DeviceSampler
    from fetal_net.model import unet_model_3d
    rng = np.random.default_rng(7)
    shape = (160, 160, 96)
    data = [rng.standard_normal(shape).astype(np.float32) for _ in range(6)]
    truth = [(rng.random(shape) < 0.3).astype(np.float32) for _ in range(6)]
    np.random.seed(1)
    sampler = DeviceSampler(data, truth, list(range(6)), batch_size=BATCH, patch_shape=PATCH, shuffle_index_list=True,
                            skip_blank=True, truth_index=0, truth_size=PATCH[2], is3d=True, device=e.local)
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, initial_learning_rate=1e-4,
                          device=e.local)
    model.init_glorot_uniform(seed=0)
    for _ in range(3):
        sampler.train_on_next_batch(model)
    sec = timed_wall(e, lambda: sampler.train_on_next_batch(model), steps)
    vox = BATCH * int(np.prod(PATCH))
    return dict(value=vox / sec, unit=UNIT, ms_per_step=sec * 1e3, fraction_of_device_step_rate=plain_ms / (sec * 1e3),
                config=dict(workload="DeviceSampler.train_on_next_batch: 6 resident cases of 160x160x96, batch 8 x 64^3 "
                                     "cut on the device (skip_blank=True, shuffled index list), same model as the "
                                     "headline step", host_bytes_per_step=32 * BATCH), steps=steps)


def bench_allreduce(e, rec_train, steps):
    """Gradient all-reduce: standalone bus bandwidth, and the exposed time per step (collectives on vs off)."""
    dp, model = rec_train["_dp"], rec_train["_model"]
    torch = e.torch
    nbytes = ((NPARAMS + 3) // 4 * 4 + 64) * 4
    ms, bus = dp.allreduce_bench(nbytes, iters=20)
    ms = max_over_ranks(e, ms)
    x, t = make_batch(e.rank, PATCH)
    xp, tp = torch.as_tensor(x).pin_memory(), torch.as_tensor(t).pin_memory()

    def step():
        dp.train_on_batch(xp.numpy(), tp.numpy())
    for _ in range(3):
        step()
    on = timed_device(e, step, steps) / steps
    dp.set_comm_enabled(False)
    for _ in range(2):
        step()
    off = timed_device(e, step, steps) / steps
    dp.set_comm_enabled(True)
    dp.broadcast_weights(0)                  # the replicas drifted apart while the collectives were off
    n = e.world
    return dict(steps=steps, bytes=int(nbytes), buckets=int(e.lib.fm_model_num_buckets(model._h)), standalone_ms=ms,
                bus_gbs=2.0 * (n - 1) / n * nbytes / (ms * 1e-3) / 1e9, bus_peak_gbs=900.0,
                frac_of_nvlink=2.0 * (n - 1) / n * nbytes / (ms * 1e-3) / 1e9 / 900.0,
                step_ms_with_comm=on, step_ms_without_comm=off, exposed_ms=max(on - off, 0.0),
                note="16.3 MB fp32 in %d buckets + 72 B of loss sums per step: latency-bound message sizes; "
                     "exposed = step with collectives minus the same step with them switched off (fm_comm_enable)" %
                     int(e.lib.fm_model_num_buckets(model._h)))


def bench_dp_parity(e):
    """One data-parallel step on the DEFAULT kernels against a single-GPU step on the full global batch."""
    from fetal_net.distributed import DataParallelTrainer
    from fetal_net.model import unet_model_3d
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, initial_learning_rate=1e-4,
                          device=e.local)
    model.init_glorot_uniform(seed=0)
    dp = DataParallelTrainer(model)
    x, t = make_batch(e.rank, PATCH)
    res = dp.train_on_batch(x, t)
    barrier(e)
    out = None
    if e.rank == 0:
        grads = model.get_gradients()
        ref = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, initial_learning_rate=1e-4,
                            device=e.local)
        ref.init_glorot_uniform(seed=0)
        shards = [make_batch(r, PATCH) for r in range(e.world)]
        xa = np.concatenate([s[0] for s in shards])
        ta = np.concatenate([s[1] for s in shards])
        rres = ref.train_on_batch(xa, ta)
        rgrads = ref.get_gradients()
        cos = []
        for g, r in zip(grads, rgrads):
            g, r = g.astype(np.float64).ravel(), r.astype(np.float64).ravel()
            cos.append(float(g @ r / max(np.linalg.norm(g) * np.linalg.norm(r), 1e-300)))
        out = dict(loss_dp=float(res[0]), loss_single_gpu_full_batch=float(rres[0]),
                   loss_abs_diff=abs(float(res[0]) - float(rres[0])), min_grad_cos=min(cos),
                   global_batch=int(xa.shape[0]), kernels="default (order-dependent fp32 accumulation in training passes)")
        del ref
    barrier(e)
    return out


def bench_infer(e, args, steps, warmup, dump=None):
    """configs[0]: patch_wise_prediction of one 256x256x64 volume (49 patches), single GPU. With a `dump` dict, the
    result of the last timed call goes into it."""
    torch, ctx = e.torch, e.ctx
    from fetal_net.model import unet_model_3d
    from fetal_net.prediction import patch_wise_prediction
    model = unet_model_3d(input_shape=(1,) + PATCH, n_base_filters=NF, depth=DEPTH, device=e.local)
    model.init_glorot_uniform(seed=0)
    vol = np.random.default_rng(0).standard_normal((1,) + VOLUME).astype(np.float32)
    volp = torch.as_tensor(vol).pin_memory().numpy()
    call = lambda v: patch_wise_prediction(model, v, PATCH, overlap_factor=OVERLAP, batch_size=49)
    for _ in range(max(warmup, 3)):
        out = call(vol)
    l0 = ctx.launch_count()
    sampler = ClockSampler(e.local)
    sampler.start()

    def timed_calls(v):
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            r = call(v)
            ts.append(time.perf_counter() - t0)
        return r, ts
    out, t_page = timed_calls(vol)
    clocks = sampler.stop()
    if dump is not None:
        dump["infer_prediction"] = np.array(out, np.float64)
    launches = int((ctx.launch_count() - l0) // steps)
    for _ in range(2):
        call(volp)
    _, t_pin = timed_calls(volp)
    # the same call with the inference passes on the three-issuer conv mode (Model.set_fast_inference: results are no
    # longer bit-identical run to run; the default above is the reproducible mode)
    model.set_fast_inference(True)
    for _ in range(2):
        out_fast = call(vol)
    _, t_fast = timed_calls(vol)
    model.set_fast_inference(False)
    fast_dev = float(np.abs(out_fast - out).max())
    # the calls are 10 ms of wall clock each on a shared host: the median over the timed calls is the figure, the mean
    # (which a single descheduled call can double) is printed beside it
    s_page, s_pin = float(np.median(t_page)), float(np.median(t_pin))
    nvox = int(np.prod(VOLUME))
    # device leg: the same call with per-launch CUDA events (gather + network + overlap-add, no host copies)
    ctx.profile(True)
    call(vol)
    agg = aggregate(ctx.profile_records())
    ctx.profile(False)
    dev_ms = sum(a[1] for a in agg.values())
    pk = peaks()
    traffic = ncu_traffic()
    breakdown = {k: dict(launches=a[0], ms=a[1], tflops=(a[2] / a[1] / 1e9 if a[2] else None),
                         gbs=(a[3] / a[1] / 1e6 if a[3] else None),
                         frac_of_peak=((a[2] / a[1] / 1e9) / tensor_peak(pk, clocks)[0]) if a[2] > 0 else
                         ((a[3] / a[1] / 1e6) / pk["hbm"] if a[3] > 0 else None))
                 for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])}
    roofs = {}
    for name in ("conv3d_march_fprop", "conv3d_tc_fprop", "reassemble", "gather_patches", "maxpool3d_fwd",
                 "upsample3d_fwd", "head_fwd"):
        if name in agg:
            roofs[name] = roofline_of(name, agg[name], 1, dev_ms, pk, clocks, traffic, "infer")
    return dict(metric="U-Net infer voxels/sec", value=nvox / (dev_ms * 1e-3), unit=UNIT, ms_per_step=dev_ms,
                value_is="output voxels / summed kernel time of one call (volume resident in HBM)",
                config=dict(workload="patch_wise_prediction 1x256x256x64, patch 64^3, overlap_factor 0.5, 49 patches "
                                     "(BASELINE configs[0])", patches=49, batch_size=49,
                            l2="49 patches x 64^3 x up to 96 channels of activations per call >> 126 MB L2"),
                steps=steps, clocks=clocks,
                e2e=dict(value=nvox / s_page, unit=UNIT, h2d_bytes_per_step=int(vol.nbytes),
                         d2h_bytes_per_step=int(out.nbytes), ms_per_step=s_page * 1e3, host_buffers="pageable numpy",
                         ms_per_step_mean=float(np.mean(t_page)) * 1e3, ms_per_step_min=float(np.min(t_page)) * 1e3,
                         statistic="median of %d timed calls" % steps),
                e2e_pinned=dict(value=nvox / s_pin, unit=UNIT, h2d_bytes_per_step=int(vol.nbytes),
                                d2h_bytes_per_step=int(out.nbytes), ms_per_step=s_pin * 1e3,
                                ms_per_step_mean=float(np.mean(t_pin)) * 1e3,
                                host_buffers="pinned input, pageable output"),
                e2e_fast_inference=dict(value=nvox / float(np.median(t_fast)), unit=UNIT,
                                        ms_per_step=float(np.median(t_fast)) * 1e3, host_buffers="pageable numpy",
                                        max_abs_diff_vs_reproducible=fast_dev,
                                        note="Model.set_fast_inference(True): three-issuer MMA order, not bit-reproducible "
                                             "run to run"),
                gpu_launches=launches, roofline=roofs.get("conv3d_march_fprop"), rooflines=roofs,
                patch_voxels_per_s=49 * int(np.prod(PATCH)) / s_page,
                conv_tflops=49 * FWD_GF_PER_PATCH / dev_ms, out_mean=float(out.mean()), kernel_breakdown=breakdown)


def bench_infer_sharded(e, steps):
    """configs[4] inference: one 512x512x128 volume, patch 128x128x64, overlap_factor 0.5 -> 147 patches, sharded."""
    from fetal_net.distributed import sharded_patch_wise_prediction
    from fetal_net.model import unet_model_3d
    model = unet_model_3d(input_shape=(1,) + PATCH5, n_base_filters=NF, depth=DEPTH, device=e.local)
    model.init_glorot_uniform(seed=0)
    vol = np.random.default_rng(0).standard_normal((1,) + VOLUME5).astype(np.float32)
    call = lambda: sharded_patch_wise_prediction(model, vol, PATCH5, overlap_factor=OVERLAP, batch_size=7)
    out = None
    for _ in range(2):
        out = call()
    sec = timed_wall(e, call, steps)
    nvox = int(np.prod(VOLUME5))
    if e.rank != 0:
        return None
    return dict(metric="U-Net sharded infer voxels/sec", steps=steps, value=nvox / sec, unit=UNIT, ms_per_volume=sec * 1e3,
                config=dict(workload="sharded_patch_wise_prediction 1x512x512x128, patch 128x128x64, overlap_factor 0.5, "
                                     "147 patches split contiguously over the ranks, one ncclReduce of the float64 "
                                     "partial sums (BASELINE configs[4])", patches=147, ranks=e.world),
                timed="wall clock around the public call incl. H2D of the volume on every rank, the reduce and the D2H "
                      "of the 268 MB float64 result on rank 0; max over ranks",
                conv_tflops=147 * FWD_GF_PER_PATCH5 / (sec * 1e3), out_mean=float(out.mean()) if out is not None else None)


def bench_family(e, kind, steps):
    """configs[2] (Isensee-2017 residual 3D U-Net, 128x128x64) and configs[3] (2.5D U-Net on 5 slices + previous-truth
    channel, 256x256): training step and predict through the same entry points, single GPU."""
    torch, _lib, lib, ctx = e.torch, e._lib, e.lib, e.ctx
    from fetal_net.model import isensee2017_model_3d, unet_model_2d
    rng = np.random.default_rng(3)
    if kind == "isensee":
        B, shape = 2, (1, 128, 128, 64)
        model = isensee2017_model_3d(input_shape=shape, n_base_filters=16, depth=5, n_segmentation_levels=3,
                                     dropout_rate=0.3, initial_learning_rate=5e-4, device=e.local)
        x = rng.standard_normal((B,) + shape).astype(np.float32)
        t = (rng.random((B,) + shape) < 0.3).astype(np.float32)
        fwd_gf, first_gf, units = 173.638, 0.906, B * 128 * 128 * 64
        name = "isensee2017_model_3d(depth=5,n_base_filters=16,n_segmentation_levels=3,dropout_rate=0.3), batch 2 x " \
               "1x128x128x64 (BASELINE configs[2])"
    else:
        B, shape = 8, (256, 256, 6)
        model = unet_model_2d(input_shape=shape, n_base_filters=32, depth=4, initial_learning_rate=1e-4, device=e.local)
        x = rng.standard_normal((B,) + shape).astype(np.float32)
        x[..., 5] = rng.random((B, 256, 256)) < 0.3
        t = (rng.random((B, 256, 256, 1)) < 0.3).astype(np.float32)
        fwd_gf, first_gf, units = 71.504, 2 * 9 * 6 * 32 * 65536 / 1e9, B * 256 * 256
        name = "unet_model_2d(depth=4,n_base_filters=32) on 5 slices + 1 previous-truth channel, batch 8 x 256x256x6 " \
               "(BASELINE configs[3])"
    model.init_glorot_uniform(seed=0)
    xd, td = torch.as_tensor(x).cuda(), torch.as_tensor(t).cuda()
    xp, tp = torch.as_tensor(x).pin_memory(), torch.as_tensor(t).pin_memory()
    m4 = np.zeros(4, np.float32)

    def step():
        _lib.check(lib.fm_train_step_device(model._h, xd.data_ptr(), td.data_ptr(), B, 1e-4, _lib.fptr(m4)))
    for _ in range(3):
        step()
    sampler = ClockSampler(e.local)
    sampler.start()
    ms = timed_device(e, step, steps) / steps
    clocks = sampler.stop()
    for _ in range(2):
        model.train_on_batch(xp.numpy(), tp.numpy())
    s_e2e = timed_wall(e, lambda: model.train_on_batch(xp.numpy(), tp.numpy()), steps)
    for _ in range(2):
        model.predict(xp.numpy())
    s_pred = timed_wall(e, lambda: model.predict(xp.numpy()), steps)
    pk = peaks()
    ctx.profile(True)
    for _ in range(2):
        step()
    agg = aggregate(ctx.profile_records())
    ctx.profile(False)
    total_ms = sum(a[1] for a in agg.values())
    top = max(agg.items(), key=lambda kv: kv[1][1])
    breakdown = {k: dict(launches=a[0] // 2, ms_per_step=a[1] / 2, share=a[1] / total_ms,
                         tflops=(a[2] / a[1] / 1e9) if a[1] > 0 and a[2] > 0 else None,
                         gbs=(a[3] / a[1] / 1e6) if a[1] > 0 and a[3] > 0 else None)
                 for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])[:12]}
    train_gf = B * (3 * fwd_gf - first_gf)
    return dict(metric="train voxels/sec" if kind == "isensee" else "train pixels/sec", value=units / (ms * 1e-3),
                unit="voxels/s" if kind == "isensee" else "pixels/s", ms_per_step=ms, config=dict(workload=name, batch=B),
                clocks=clocks, conv_tflops_whole_step=train_gf / ms,
                e2e=dict(value=units / s_e2e, ms_per_step=s_e2e * 1e3, host_buffers="pinned",
                         h2d_bytes_per_step=int(x.nbytes + t.nbytes), d2h_bytes_per_step=64),
                predict=dict(value=units / s_pred, ms_per_call=s_pred * 1e3, conv_tflops=B * fwd_gf / (s_pred * 1e3),
                             note="Model.predict with host buffers (H2D + forward + D2H)"),
                roofline=roofline_of(top[0], top[1], 2, total_ms, pk, clocks, {}, kind), kernel_breakdown=breakdown,
                loss=float(m4[0]), steps=steps)


def run_b200(args):
    e = setup_env(True)
    want_train = args.workload in ("all", "train")
    want_infer = args.workload in ("all", "infer")
    line = None
    dump = {} if args.dump_outputs else None
    if want_train:
        rec = bench_train(e, args, PATCH, FWD_GF_PER_PATCH, FIRST_CONV_GF, args.steps, args.warmup, True, dump)
        cpu_base = None
        if e.rank == 0 and e.world == 1 and not args.no_cpu_baseline:
            times, threads = cpu_train_steps(BATCH, 3, 1, budget_s=40)
            sec = float(np.mean(times))
            cpu_base = dict(value=BATCH * int(np.prod(PATCH)) / sec, unit=UNIT, cores=os.cpu_count(), kind="port",
                            sample="oracle (PyTorch-CPU fp32 restatement) full train step on 8 x 64^3, %d timed steps "
                                   "after 1 warm-up, %d threads" % (len(times), threads))
        extra = {}
        if e.world > 1:
            extra["allreduce"] = bench_allreduce(e, rec, args.steps)
        model, dp = rec.pop("_model"), rec.pop("_dp")
        del model, dp
        if e.world > 1:
            r5 = bench_train(e, args, PATCH5, FWD_GF_PER_PATCH5, FIRST_CONV_GF5, args.steps, 3, False)
            r5.pop("_model"), r5.pop("_dp")
            r5["config"] = dict(workload="same step on BASELINE configs[4]'s patch shape: batch 8 x 1x128x128x64 per GPU",
                                global_batch=BATCH * e.world, patch=list(PATCH5))
            r5["unit"] = UNIT
            r5["steps"] = args.steps
            extra["train_cfg5"] = r5
            extra["infer_sharded"] = bench_infer_sharded(e, args.steps)
            extra["dp_parity"] = bench_dp_parity(e)
        if e.rank == 0:
            line = dict(metric=METRIC, value=rec["value"], unit=UNIT, n_gpus=e.world, steps=args.steps,
                        warmup=max(args.warmup, 3), ms_per_step=rec["ms_per_step"], higher_is_better=True,
                        scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                        config=workload_config(e.world), clocks=rec["clocks"], e2e=rec["e2e"],
                        e2e_pageable=rec["e2e_pageable"], gpu_launches=rec["gpu_launches"],
                        roofline=rec.get("roofline"), rooflines=rec.get("rooflines"), cpu_baseline=cpu_base,
                        conv_tflops_whole_step=rec["conv_tflops_whole_step"],
                        kernel_breakdown=rec.get("kernel_breakdown"), loss=rec["loss"],
                        collective=("libfetalb200 NCCL communicator (fm_train_step_dp), NCCL %s" %
                                    (e.ctx.comm_info()[2],)) if e.world > 1 else None)
            line.update(extra)
    if args.workload == "all" and e.rank == 0 and e.world == 1 and line is not None:
        line["train_sampled"] = bench_train_sampled(e, args.steps, line["ms_per_step"])
        line["families"] = dict(isensee=bench_family(e, "isensee", args.steps),
                                unet2d=bench_family(e, "unet2d", args.steps))
    if want_infer and e.rank == 0:
        inf = bench_infer(e, args, args.steps, 3, dump)
        if not args.no_cpu_baseline and e.world == 1:
            inf["cpu_baseline"] = cpu_infer_sample()
        if line is None:
            line = dict(inf, n_gpus=1, warmup=3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
                        data="synthetic")
        else:
            line["infer"] = inf
    barrier(e)
    if e.rank == 0:
        if dump is not None:
            write_dump(args.dump_outputs, dump)
        print(json.dumps(line))
    if e.world > 1:
        e.lib.fm_comm_destroy(e.ctx.handle)
        e.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "train", "infer"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of each workload as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the outputs of --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
