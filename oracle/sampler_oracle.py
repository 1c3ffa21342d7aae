"""TEST INFRASTRUCTURE ONLY — NumPy / scipy statement of one training sample cut by the device sampler with a warp
(fetal_net.device_sampler, `sample_patches_warp_kernel` in csrc/sampler.cu, fm_sample_warp in include/fetal_b200.h).

The warp is the library's own augmentation, not the reference's nilearn / imgaug pipeline. An element of the assembled
sample that the unwarped cut reads at volume position q reads

    s = c + t + M (q + d(q) - c),   c = corner + (P - 1) / 2,
    d(q)[a] = alpha[a] * trilinear(G_a, (q - corner) / spacing),   spacing = (P - 1) / (G - 1)

with q = corner + (i, j, z0 + k) for the data patch (z0 = 0), the target slices (z0 = truth_index) and the
previous-truth slices (z0 = prev_truth_index). The control values of G_a come from the sampler's integer hash. Data
channels: map_coordinates(order=1, mode='nearest'); target and previous truth: map_coordinates(order=0,
mode='nearest') = floor(s + 0.5) on the clamped coordinate. Everything here is float64 from the float32 warp
parameters; the intensity scale multiplies the float32 interpolated data, and the flips act on the assembled arrays.
"""
import numpy as np
from scipy import ndimage


def hash32(x):
    """The sampler's integer mixer on NumPy uint32 (wrap-around multiplication)."""
    x = np.asarray(x, dtype=np.uint32)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint32(16))
        x = x * np.uint32(0x7FEB352D)
        x = x ^ (x >> np.uint32(15))
        x = x * np.uint32(0x846CA68B)
        x = x ^ (x >> np.uint32(16))
    return x


def control_grids(seed, grid):
    """[3, G, G, G] float64: the value of axis a at x-major control point g is ((h >> 8) 2^-23) - 1 with
    h = hash32(hash32(seed) ^ (3 g + a))."""
    g3 = grid ** 3
    t = np.arange(3 * g3, dtype=np.uint32)                 # t = 3 g + a
    h = hash32(hash32(np.uint32(seed)) ^ t)
    v = (h >> np.uint32(8)).astype(np.float64) * 2.0 ** -23 - 1.0
    return v.reshape(g3, 3).T.reshape(3, grid, grid, grid)


def identity_warp():
    return dict(matrix=np.eye(3, dtype=np.float32), offset=np.zeros(3, np.float32), alpha=np.zeros(3, np.float32),
                seed=0, grid=0)


def source_coords(corner, patch, z0, nz, warp):
    """float64 [3, P0, P1, nz]: the source position of every element of a slab of nz slices at patch-local z0."""
    m = np.asarray(warp["matrix"], np.float32).astype(np.float64).reshape(3, 3)
    t = np.asarray(warp["offset"], np.float32).astype(np.float64)
    corner = np.asarray(corner, np.float64)
    patch = np.asarray(patch, np.int64)
    c = corner + (patch - 1) / 2.0
    p = np.stack(np.meshgrid(np.arange(patch[0]), np.arange(patch[1]), z0 + np.arange(nz), indexing="ij")).astype(
        np.float64)                                        # q - corner
    if warp["grid"]:
        grid = int(warp["grid"])
        alpha = np.asarray(warp["alpha"], np.float32).astype(np.float64)
        u = np.empty_like(p)
        for a in range(3):
            u[a] = 0.0 if patch[a] == 1 else p[a] / ((patch[a] - 1) / (grid - 1))
        u = np.clip(u, 0, grid - 1)
        ctrl = control_grids(warp["seed"], grid)
        d = np.stack([alpha[a] * ndimage.map_coordinates(ctrl[a], u, order=1, mode="nearest") for a in range(3)])
        p = p + d
    r = p - ((patch - 1) / 2.0)[:, None, None, None]      # q + d(q) - c
    return (c + t)[:, None, None, None] + np.einsum("ab,bxyz->axyz", m, r)


def rounding_margin(coords, shape):
    """Distance of every clamped coordinate from a rounding boundary k + 1/2 (min over the axes)."""
    s = np.clip(coords, 0, np.asarray(shape, np.float64)[:, None, None, None] - 1)
    return np.min(np.abs(s - np.floor(s) - 0.5), axis=0)


def sample(data, truth, corner, patch, truth_index, truth_size, prev_truth_index=None, prev_truth_size=0, flip=0,
           scale=1.0, warp=None):
    """One sample as the device assembles it: x float32 [P0, P1, P2 + prev_truth_size], y float32 [P0, P1,
    truth_size], and the rounding margins of the truth elements (x_margin with +inf on the data channels, y_margin)."""
    warp = identity_warp() if warp is None else warp
    data = np.asarray(data, np.float64)
    truth = np.asarray(truth, np.float64)
    s = source_coords(corner, patch, 0, patch[2], warp)
    x = ndimage.map_coordinates(data, s, order=1, mode="nearest").astype(np.float32) * np.float32(scale)
    x_margin = np.full(x.shape, np.inf)
    s = source_coords(corner, patch, truth_index, truth_size, warp)
    y = ndimage.map_coordinates(truth, s, order=0, mode="nearest").astype(np.float32)
    y_margin = rounding_margin(s, truth.shape)
    if prev_truth_index is not None and prev_truth_size:
        s = source_coords(corner, patch, prev_truth_index, prev_truth_size, warp)
        xp = ndimage.map_coordinates(truth, s, order=0, mode="nearest").astype(np.float32)
        x = np.concatenate([x, xp], axis=-1)
        x_margin = np.concatenate([x_margin, rounding_margin(s, truth.shape)], axis=-1)
    p2 = patch[2]
    if flip & 1:
        x, y, x_margin, y_margin = x[::-1], y[::-1], x_margin[::-1], y_margin[::-1]
    if flip & 2:
        x, y, x_margin, y_margin = x[:, ::-1], y[:, ::-1], x_margin[:, ::-1], y_margin[:, ::-1]
    if flip & 4:
        zf = lambda a: np.concatenate([a[..., :p2][..., ::-1], a[..., p2:][..., ::-1]], axis=-1)
        x, y, x_margin, y_margin = zf(x), y[..., ::-1], zf(x_margin), y_margin[..., ::-1]
    return (np.ascontiguousarray(x), np.ascontiguousarray(y), np.ascontiguousarray(x_margin),
            np.ascontiguousarray(y_margin))
