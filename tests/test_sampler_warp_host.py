"""Host side of the sampler's warp augmentation (fetal_net.device_sampler `rotate` / `scale` / `translate` /
`elastic`): the NumPy oracle (oracle/sampler_oracle.py) pinned to independent statements, the warp matrix to scipy's
rotations, the np.random draw order and the validation of the new keys. The device kernel is compared to the oracle in
test_gpu_sampler_warp.py."""
import ctypes

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from oracle import sampler_oracle as so
from tests.test_sampler import CONFIGS, cases, host_cut


def _kw(kw):
    return dict(truth_index=kw["truth_index"], truth_size=kw["truth_size"],
                prev_truth_index=kw.get("prev_truth_index"), prev_truth_size=kw.get("prev_truth_size") or 0)


def _corners(shape, patch):
    """Interior corners and corners sticking out of the volume on either side."""
    hi = [n - p for n, p in zip(shape, patch)]
    return [[0, 0, 0], [hi[0], hi[1], hi[2]], [-3, 2, -2], [hi[0] + 4, -5, hi[2] + 3], [1, hi[1] + 2, 1]]


def _oracle_cut(data, truth, case, corner, patch, kw, warp=None):
    x, y, _, _ = so.sample(data[case], truth[case], corner, patch, warp=warp, **_kw(kw))
    return x, y


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_identity_warp_is_the_edge_padded_cut(name):
    data, truth = cases()
    patch, kw = CONFIGS[name]
    for case in range(len(data)):
        for corner in _corners(data[case].shape, patch):
            x, y = _oracle_cut(data, truth, case, corner, patch, kw)
            ex, ey = host_cut(data, truth, case, corner, patch, **dict(kw, is3d=False))
            assert np.array_equal(x, ex) and np.array_equal(y, ey), (name, case, corner)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_integer_offset_is_the_cut_at_the_shifted_corner(name):
    data, truth = cases()
    patch, kw = CONFIGS[name]
    for t in ([3, -2, 1], [-7, 5, -4], [0, 0, 9]):
        warp = dict(so.identity_warp(), offset=np.asarray(t, np.float32))
        for corner in _corners(data[0].shape, patch):
            x, y = _oracle_cut(data, truth, 0, corner, patch, kw, warp)
            ex, ey = host_cut(data, truth, 0, np.add(corner, t), patch, **dict(kw, is3d=False))
            assert np.array_equal(x, ex) and np.array_equal(y, ey), (name, t, corner)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_quarter_turn_is_rot90_of_the_cut(name):
    """M = [[0,-1,0],[1,0,0],[0,0,1]] about the centre of a square patch: output[i, j] = cut[P - 1 - j, i]."""
    data, truth = cases()
    patch, kw = CONFIGS[name]
    assert patch[0] == patch[1]
    warp = dict(so.identity_warp(), matrix=np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float32))
    for corner in _corners(data[1].shape, patch):
        x, y = _oracle_cut(data, truth, 1, corner, patch, kw, warp)
        ex, ey = host_cut(data, truth, 1, corner, patch, **dict(kw, is3d=False))
        assert np.array_equal(x, np.rot90(ex, k=-1, axes=(0, 1))), (name, corner)
        assert np.array_equal(y, np.rot90(ey, k=-1, axes=(0, 1))), (name, corner)


def test_numpy_hash_equals_integer_statement():
    def mix(x):
        m = 0xFFFFFFFF
        x ^= x >> 16
        x = (x * 0x7FEB352D) & m
        x ^= x >> 15
        x = (x * 0x846CA68B) & m
        x ^= x >> 16
        return x
    vals = [0, 1, 2, 3, 255, 65535, 65536, 0x7FFFFFFF, 0x80000000, 0xDEADBEEF, 0xFFFFFFFF]
    vals += [int(v) for v in np.random.default_rng(0).integers(0, 2 ** 32, 1000, dtype=np.uint64)]
    got = so.hash32(np.asarray(vals, np.uint64).astype(np.uint32))
    assert [int(v) for v in got] == [mix(v) for v in vals]
    # control values: x-major point g, axis a <- hash32(hash32(seed) ^ (3 g + a)), exact in float32
    g = so.control_grids(12345, 3)
    hs = mix(12345)
    for gx, gy, gz, a in [(0, 0, 0, 0), (2, 1, 0, 1), (1, 2, 2, 2), (2, 2, 2, 0)]:
        idx = (gx * 3 + gy) * 3 + gz
        ref = (mix(hs ^ (3 * idx + a)) >> 8) * 2.0 ** -23 - 1.0
        assert g[a, gx, gy, gz] == ref and np.float64(np.float32(ref)) == ref
    assert g.min() >= -1 and g.max() < 1


def test_warp_matrix_equals_scipy_rotation_times_inverse_scale():
    from fetal_net.device_sampler import warp_matrix
    rng = np.random.default_rng(1)
    for _ in range(20):
        ang = rng.normal(0, 20, 3)
        sc = rng.uniform(0.6, 1.6, 3)
        ref = Rotation.from_euler("xyz", ang, degrees=True).as_matrix() @ np.diag(1.0 / sc)
        assert np.allclose(warp_matrix(ang, sc), ref, rtol=0, atol=1e-12)


def _bare_sampler(device_augment):
    """A DeviceSampler without a volume set: only the host draws are exercised."""
    from fetal_net.device_sampler import DeviceSampler
    s = object.__new__(DeviceSampler)
    s.device_augment = device_augment
    return s


def _parent_draws(a, n):
    """The draw sequence of the sampler before the warp keys existed."""
    for _ in range(n):
        if a.get("flip"):
            np.random.randint(0, 8)
        lo, hi = a.get("intensity", (1.0, 1.0))
        np.random.uniform(lo, hi)
        np.random.randint(0, 2 ** 31 - 1)


@pytest.mark.parametrize("a", [dict(flip=True), dict(flip=True, intensity=(0.9, 1.1), noise_sigma=0.1),
                               dict(intensity=(0.5, 2.0))])
def test_without_warp_keys_the_random_stream_is_unchanged(a):
    s = _bare_sampler(a)
    np.random.seed(4)
    _parent_draws(a, 5)
    ref = np.random.random()
    np.random.seed(4)
    s._aug_array(5)
    assert np.random.random() == ref
    np.random.seed(4)
    aug, warp = s.draw_augment(5)
    assert aug is not None and warp is None and np.random.random() == ref


@pytest.mark.parametrize("keys", [("rotate",), ("scale",), ("translate",), ("elastic",),
                                  ("rotate", "scale", "translate", "elastic"), ("rotate", "elastic")])
def test_warp_draw_order(keys):
    """The flip / intensity / noise-seed draws of every sample first, then per sample three angles, three scales,
    three offsets and the elastic seed, each only when its key is present."""
    from fetal_net.device_sampler import warp_matrix
    full = dict(rotate=(10.0, 5.0, 20.0), scale=(0.1, 0.2, 0.05), translate=(3.0, 0.0, 2.0),
                elastic=dict(alpha=(3.0, 2.0, 1.0), grid=4))
    a = dict(flip=True, intensity=(0.9, 1.1), **{k: full[k] for k in keys})
    n = 4
    np.random.seed(9)
    aug, warp = _bare_sampler(a).draw_augment(n)
    after = np.random.random()
    np.random.seed(9)
    _parent_draws(a, n)
    for b in range(n):
        ang = [np.random.normal(0, s) for s in full["rotate"]] if "rotate" in a else [0.0] * 3
        sc = ([float(np.clip(1 + np.random.normal(0, s), 0.5, 2.0)) for s in full["scale"]] if "scale" in a
              else [1.0] * 3)
        off = [np.random.normal(0, s) for s in full["translate"]] if "translate" in a else [0.0] * 3
        seed = np.random.randint(0, 2 ** 31 - 1) if "elastic" in a else 0
        assert np.array_equal(np.asarray(warp[b].matrix, np.float32),
                              warp_matrix(ang, sc).astype(np.float32).ravel()), (keys, b)
        assert np.array_equal(np.asarray(warp[b].offset, np.float32), np.asarray(off, np.float32)), (keys, b)
        assert warp[b].elastic_seed == seed
        assert warp[b].elastic_grid == (4 if "elastic" in a else 0)
        assert list(warp[b].elastic_alpha) == ([3.0, 2.0, 1.0] if "elastic" in a else [0.0] * 3)
    assert after == np.random.random()
    assert aug is not None and len(aug) == n and ctypes.sizeof(warp[0]) == 68


@pytest.mark.parametrize("bad", [
    dict(rotate=10), dict(rotate=(1, 2)), dict(rotate=(1, 2, float("nan"))), dict(rotate=(1, -2, 3)),
    dict(scale=(0.1, 0.1)), dict(scale="abc"), dict(scale=(0.1, float("inf"), 0.1)),
    dict(translate=(1, 2, 3, 4)), dict(translate=(-1, 0, 0)),
    dict(elastic=3), dict(elastic=dict(alpha=3)), dict(elastic=dict(grid=4)), dict(elastic=dict(alpha=3, grid=1)),
    dict(elastic=dict(alpha=3, grid=9)), dict(elastic=dict(alpha=3, grid=4.0)), dict(elastic=dict(alpha=-1, grid=4)),
    dict(elastic=dict(alpha=(1, 2), grid=4)), dict(elastic=dict(alpha=float("nan"), grid=4)),
    dict(elastic=dict(alpha=3, grid=4, sigma=2)),
])
def test_bad_warp_keys_raise_value_error(bad):
    from fetal_net.device_sampler import DeviceSampler, warp_spec
    with pytest.raises(ValueError):
        warp_spec(bad)
    data, truth = cases()
    with pytest.raises(ValueError):
        DeviceSampler(data, truth, [0], device_augment=bad, patch_shape=(8, 8, 4))


def test_good_warp_keys_are_accepted():
    from fetal_net.device_sampler import warp_spec
    spec = warp_spec(dict(flip=True, rotate=(10, 0, 5), scale=[0.1] * 3, translate=np.array([1.0, 2.0, 0.0]),
                          elastic=dict(alpha=3, grid=np.int64(2))))
    assert spec["rotate"] == (10.0, 0.0, 5.0) and spec["elastic"] == ((3.0, 3.0, 3.0), 2)
    assert warp_spec(dict(flip=True)) == {} and warp_spec(None) == {}
