"""The sampler's warp augmentation on the device (`sample_patches_warp_kernel`, fm_volset_gather_warp,
fm_train_step_sampled_warp): bit-exact against the unwarped cut where the warp maps voxels onto voxels, against the
NumPy oracle (oracle/sampler_oracle.py) within the float32-coordinate bound for random rotate / scale / translate /
elastic warps, and the sampled training step with warps against train_on_batch on the gathered batch."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import sampler_oracle as so
from tests.test_sampler import CONFIGS, cases

pytestmark = pytest.mark.gpu

QUARTER = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float32)


@pytest.fixture(scope="module")
def samplers():
    """One DeviceSampler over the golden cases per sampler config."""
    from fetal_net.device_sampler import DeviceSampler
    data, truth = cases()
    out = {}
    for name, (patch, kw) in CONFIGS.items():
        kw = {k: v for k, v in kw.items() if k != "is3d"}
        out[name] = DeviceSampler(data, truth, [0], batch_size=1, patch_shape=patch, shuffle_index_list=False, **kw)
    return out


def _warp(matrix=None, offset=(0, 0, 0), alpha=(0, 0, 0), seed=0, grid=0):
    from fetal_net import _lib
    w = _lib.SampleWarp()
    w.matrix[:] = [float(v) for v in (np.eye(3) if matrix is None else np.asarray(matrix)).ravel()]
    w.offset[:] = [float(v) for v in offset]
    w.elastic_alpha[:] = [float(v) for v in alpha]
    w.elastic_seed, w.elastic_grid = int(seed), int(grid)
    return w


def _as_oracle(w):
    return dict(matrix=np.asarray(w.matrix, np.float32).reshape(3, 3), offset=np.asarray(w.offset, np.float32),
                alpha=np.asarray(w.elastic_alpha, np.float32), seed=int(w.elastic_seed), grid=int(w.elastic_grid))


def _aug(flips, scale=1.0):
    from fetal_net import _lib
    arr = (_lib.SampleAug * len(flips))()
    for b, f in enumerate(flips):
        arr[b].flip, arr[b].intensity_scale, arr[b].noise_sigma, arr[b].noise_seed = f, scale, 0.0, 0
    return arr


def _edge_corners(patch, rng, n):
    """(case, corner) of n samples over the golden cases, corners anywhere from sticking out below to sticking out
    above the volume; the first two stick out on every axis."""
    data, _ = cases()
    cs = [b % len(data) for b in range(n)]
    out = [[int(rng.integers(-(p // 2), d - p // 2 + 1)) for d, p in zip(data[c].shape, patch)] for c in cs]
    out[0] = [-4, -3, -2]
    out[1] = [d - p + 3 for d, p in zip(data[cs[1]].shape, patch)]
    return np.array(cs, np.int32), np.array(out, np.int32)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_null_warp_equals_gather(name, samplers):
    from fetal_net import _lib
    s = samplers[name]
    rng = np.random.default_rng(1)
    cs, corners = _edge_corners(s.patch_shape, rng, 9)
    aug = _aug([int(v) for v in rng.integers(0, 8, 9)], 1.25)
    p0, p1, p2 = s.patch_shape
    ti, ts, pi, ps = s._args()
    out = []
    for fn in ("fm_volset_gather", "fm_volset_gather_warp"):
        x = np.empty((9, p0, p1, p2 + ps), np.float32)
        y = np.empty((9, p0, p1, ts), np.float32)
        extra = (aug,) if fn == "fm_volset_gather" else (aug, None)
        _lib.check(getattr(s._lib, fn)(s._handle, _lib.i32ptr(cs), _lib.i32ptr(corners.ravel()), *extra, 9,
                                       _lib.i32ptr(_lib.i32x(s.patch_shape)), ti, ts, pi, ps, _lib.fptr(x),
                                       _lib.fptr(y)))
        out.append((x, y))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_exact_warps_equal_the_unwarped_cut(name, samplers):
    """Identity, integer offsets and the quarter turn map voxel centres onto voxel centres: bit for bit the unwarped
    cut at corner + t (the quarter turn: rot90 of the cut), corners at the volume edges included."""
    s = samplers[name]
    rng = np.random.default_rng(2)
    n = 8
    cs, corners = _edge_corners(s.patch_shape, rng, n)
    x0, y0 = s.gather(cs, corners, aug=None, warp=[_warp() for _ in range(n)])
    xr, yr = s.gather(cs, corners, aug=_aug([0] * n))
    assert np.array_equal(x0, xr) and np.array_equal(y0, yr), "identity"
    offs = rng.integers(-6, 7, (n, 3))
    x, y = s.gather(cs, corners, warp=[_warp(offset=t) for t in offs])
    xr, yr = s.gather(cs, corners + offs.astype(np.int32), aug=_aug([0] * n))
    assert np.array_equal(x, xr) and np.array_equal(y, yr), "integer offsets"
    x, y = s.gather(cs, corners, warp=[_warp(matrix=QUARTER) for _ in range(n)])
    assert np.array_equal(x, np.rot90(x0, k=-1, axes=(1, 2))), "quarter turn, x"
    assert np.array_equal(y, np.rot90(y0, k=-1, axes=(1, 2))), "quarter turn, y"


def test_warps_of_large_batches_travel_through_the_staging_area(samplers):
    """Beyond the inline limit (64 samples) the arguments and the warps go through pinned staging memory."""
    s = samplers["u25d"]
    rng = np.random.default_rng(6)
    n = 70
    cs, corners = _edge_corners(s.patch_shape, rng, n)
    offs = rng.integers(-6, 7, (n, 3))
    flips = [int(v) for v in rng.integers(0, 8, n)]
    x, y = s.gather(cs, corners, aug=_aug(flips, 1.25), warp=[_warp(offset=t) for t in offs])
    xr, yr = s.gather(cs, corners + offs.astype(np.int32), aug=_aug(flips, 1.25))
    assert np.array_equal(x, xr) and np.array_equal(y, yr)


def _random_warps(rng, n):
    from fetal_net.device_sampler import warp_matrix
    ws = []
    for _ in range(n):
        m = warp_matrix(rng.uniform(-30, 30, 3), rng.uniform(0.8, 1.2, 3)).astype(np.float32)
        ws.append(_warp(matrix=m, offset=rng.uniform(-5, 5, 3).astype(np.float32), alpha=(3, 3, 3),
                        seed=int(rng.integers(0, 2 ** 31 - 1)), grid=4))
    return ws


@pytest.mark.parametrize("name", ["u3d", "u25d"])
def test_random_warps_against_oracle(name, samplers):
    s = samplers[name]
    patch, kw = CONFIGS[name]
    data, truth = cases()
    rng = np.random.default_rng(3)
    n = 12
    cs, corners = _edge_corners(patch, rng, n)
    ws = _random_warps(rng, n)
    flips = [int(v) for v in rng.integers(0, 8, n)]
    x, y = s.gather(cs, corners, aug=_aug(flips, 1.5), warp=ws)
    excluded = total = 0
    for b in range(n):
        c = int(cs[b])
        ex, ey, mx, my = so.sample(data[c], truth[c], corners[b], patch, kw["truth_index"], kw["truth_size"],
                                   kw.get("prev_truth_index"), kw.get("prev_truth_size") or 0, flips[b], 1.5,
                                   _as_oracle(ws[b]))
        p2 = patch[2]
        bound = 2.0 ** -12 * float(data[c].max() - data[c].min()) * 1.5
        err = float(np.max(np.abs(x[b, ..., :p2].astype(np.float64) - ex[..., :p2])))
        assert err <= bound, (b, err, bound)
        for got, ref, margin in ((x[b, ..., p2:], ex[..., p2:], mx[..., p2:]), (y[b], ey, my)):
            keep = margin >= 1e-3
            assert np.array_equal(got[keep], ref[keep]), (b, int(np.sum(got[keep] != ref[keep])))
            excluded += int(np.sum(~keep))
            total += keep.size
    assert excluded < 0.01 * total, (excluded, total)


def test_flip_of_warp_is_warp_then_flip(samplers):
    s = samplers["u25d"]
    p2 = s.patch_shape[2]
    rng = np.random.default_rng(4)
    cs, corners = _edge_corners(s.patch_shape, rng, 4)
    ws = _random_warps(rng, 4)
    x0, y0 = s.gather(cs, corners, aug=_aug([0] * 4, 0.75), warp=ws)
    for flip in range(8):
        x, y = s.gather(cs, corners, aug=_aug([flip] * 4, 0.75), warp=ws)
        ex, ey = x0, y0
        if flip & 1:
            ex, ey = ex[:, ::-1], ey[:, ::-1]
        if flip & 2:
            ex, ey = ex[:, :, ::-1], ey[:, :, ::-1]
        if flip & 4:
            ex = np.concatenate([ex[..., :p2][..., ::-1], ex[..., p2:][..., ::-1]], -1)
            ey = ey[..., ::-1]
        assert np.array_equal(x, ex) and np.array_equal(y, ey), flip


AUGMENT = dict(flip=True, intensity=(0.9, 1.1), rotate=(15.0, 15.0, 15.0), scale=(0.1, 0.1, 0.1),
               translate=(3.0, 3.0, 1.0), elastic=dict(alpha=3.0, grid=4))


@pytest.mark.parametrize("kind", ["2d", "3d"])
def test_sampled_step_with_warps_equals_train_on_batch(kind):
    """fm_train_step_sampled_warp == fm_volset_gather_warp + train_on_batch, step after step (the bound of
    test_train_on_sampled_batch_equals_train_on_batch: the run-to-run spread)."""
    from fetal_net.device_sampler import DeviceSampler
    from fetal_net.model import unet_model_2d, unet_model_3d
    rng = np.random.default_rng(5)
    shape = (48, 48, 12) if kind == "2d" else (48, 48, 24)
    data = [rng.standard_normal(shape).astype(np.float32) for _ in range(2)]
    truth = [(rng.random(shape) > 0.6).astype(np.float32) for _ in range(2)]
    if kind == "2d":
        kw = dict(patch_shape=(32, 32, 5), truth_index=2, truth_size=1, prev_truth_index=1, prev_truth_size=1)
    else:
        kw = dict(patch_shape=(32, 32, 16), truth_index=0, truth_size=16, is3d=True)
    losses = []
    for on_device in (False, True):
        np.random.seed(3)
        s = DeviceSampler(data, truth, [0, 1], batch_size=4, shuffle_index_list=False, skip_blank=False,
                          device_augment=AUGMENT, **kw)
        if kind == "2d":
            model = unet_model_2d(input_shape=(32, 32, 6), n_base_filters=16, depth=3, initial_learning_rate=1e-3)
        else:
            model = unet_model_3d(input_shape=(1, 32, 32, 16), n_base_filters=16, depth=3, initial_learning_rate=1e-3)
        model.init_glorot_uniform(seed=11)
        ls = []
        for _ in range(4):
            if on_device:
                ls.append(s.train_on_next_batch(model)[0])
            else:
                x, y = next(s)
                ls.append(model.train_on_batch(x, y)[0])
        losses.append(ls)
    assert np.allclose(losses[0], losses[1], atol=2e-3), losses
    assert losses[0][-1] < losses[0][0]


def test_library_rejects_bad_warps(samplers):
    from fetal_net import _lib
    s = samplers["u25d"]
    cs, corners = np.array([0, 1], np.int32), np.array([[2, 3, 4], [5, 6, 7]], np.int32)
    bad_matrix = np.eye(3)
    bad_matrix[1, 2] = np.nan
    for bad in (_warp(matrix=bad_matrix), _warp(offset=(0, np.inf, 0)), _warp(alpha=(1, -0.5, 1), grid=4),
                _warp(grid=9), _warp(grid=1)):
        with pytest.raises(_lib.FetalB200Error):
            s.gather(cs, corners, warp=[_warp(), bad])
    x, y = s.gather(cs, corners, warp=[_warp(), _warp()])    # the library is still usable
    xr, yr = s.gather(cs, corners, aug=_aug([0, 0]))
    assert np.array_equal(x, xr) and np.array_equal(y, yr)


# ---- two ranks --------------------------------------------------------------------------------------------------------

def _free_port():
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    p = sk.getsockname()[1]
    sk.close()
    return p


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    os.environ["FETAL_B200_DETERMINISTIC"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda:%d" % rank))
    from fetal_net.device_sampler import DeviceSampler
    from fetal_net.distributed import DataParallelTrainer
    from tests.test_gpu_distributed_batchnorm import _build, _checked_grads, _cos

    data = [np.random.default_rng(7 + i).standard_normal((48, 48, 12)).astype(np.float32) for i in range(2)]
    truth = [(np.random.default_rng(9 + i).random((48, 48, 12)) > 0.6).astype(np.float32) for i in range(2)]
    kw = dict(batch_size=2, patch_shape=(32, 32, 5), shuffle_index_list=False, truth_index=2, truth_size=1,
              prev_truth_index=1, prev_truth_size=1, skip_blank=False)
    sampler = DeviceSampler(data, truth, [0, 1], device=rank, **kw)
    cases_ = np.array([0, 1, 1, 0], np.int32)
    corners = np.array([[0, 3, 1], [16, 5, 7], [9, 16, 2], [4, 11, 6]], np.int32)
    rng = np.random.default_rng(13)
    ws = _random_warps(rng, 4)
    aug = _aug([1, 6, 0, 3], 1.1)
    lo, hi = 2 * rank, 2 * rank + 2
    model = _build("2d", rank)
    DataParallelTrainer(model)
    res = model.train_on_sampled_batch(sampler, cases_[lo:hi], corners[lo:hi], aug=aug[lo:hi], warp=ws[lo:hi])
    grads = _checked_grads(model)
    if rank == 0:
        xs, ys = sampler.gather(cases_, corners, aug=aug, warp=ws)
        ref_model = _build("2d", 0)
        ref = ref_model.train_on_batch(xs, ys)
        cos = [_cos(g, r) for (_, g), (_, r) in zip(grads, _checked_grads(ref_model))]
        out.put(dict(res=res, ref=ref, min_cos=min(cos)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_sampled_step_with_warps():
    """Two ranks, each with its slice of the samples and their warps, equal the single-process step on the whole
    batch (FETAL_B200_DETERMINISTIC=1 in the workers; the bounds of the data-parallel batch-norm test)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    r = q.get(timeout=600)
    [p.join(timeout=120) for p in procs]
    assert np.allclose(r["res"], r["ref"], rtol=0, atol=1e-6), r
    assert r["min_cos"] >= 0.9999, r
