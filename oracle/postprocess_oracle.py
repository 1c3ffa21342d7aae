"""TEST INFRASTRUCTURE ONLY — restatement of the reference's fetal_net/postprocess.py:13 `postprocess_prediction`.

The reference file is 19 lines of numpy / scipy; read as:

    pred = gaussian_filter(pred, gaussian_std)
    seg = pred > threshold
    if fill_holes:           seg = binary_fill_holes(seg)
    if connected_component:  seg = <largest 6-connected component of seg>   (np.argmax over label sizes)

`postprocess_prediction` below runs exactly that on scipy, so it is the oracle the device path is compared to bit for
bit. `gaussian_filter_restated` spells out the summation order scipy's correlate1d uses for the symmetric Gaussian
kernel (mode 'reflect', axes 0, 1, 2, output rounded to the input dtype after each axis) in plain NumPy: the device
kernel follows the same order, and a CPU test pins the restatement to scipy.
"""
import numpy as np
from scipy import ndimage


def gaussian_weights(sigma, truncate=4.0):
    """scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, int(truncate * sigma + 0.5)): 2r + 1 float64 weights.
    sigma <= 1e-15 (which gaussian_filter skips) gives radius 0 and the single weight 1.0, i.e. the identity."""
    sigma = float(sigma)
    if sigma <= 1e-15:
        return np.ones(1, np.float64)
    radius = int(truncate * sigma + 0.5)
    x = np.arange(-radius, radius + 1)
    phi_x = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return phi_x / phi_x.sum()


def reflect_index(j, n):
    """scipy mode 'reflect' (d c b a | a b c d | d c b a) for any line length n >= 1, also shorter than the radius."""
    m = np.mod(j, 2 * n)
    return np.where(m < n, m, 2 * n - 1 - m)


def gaussian_filter_restated(pred, sigma):
    """gaussian_filter(pred, sigma) for float32 / float64 input, in the device kernel's order:
    acc = x[i] * w[0]; acc += (x[i - l] + x[i + l]) * w[l] for l = r .. 1, in float64, then rounded to the input dtype."""
    w = gaussian_weights(sigma)
    r = (len(w) - 1) // 2
    out = np.asarray(pred)
    dtype = out.dtype
    for axis in range(out.ndim):
        x = np.moveaxis(out, axis, -1).astype(np.float64)
        n = x.shape[-1]
        i = np.arange(n)
        acc = x * w[r]
        for l in range(r, 0, -1):
            acc = acc + (x[..., reflect_index(i - l, n)] + x[..., reflect_index(i + l, n)]) * w[r + l]
        out = np.moveaxis(acc.astype(dtype), -1, axis)
    return np.ascontiguousarray(out)


def largest_component(seg):
    """Largest 6-connected component of a bool volume; ties go to the lowest label, i.e. the component whose first
    voxel in C order comes first. Raises ValueError without any component (the reference's np.argmax([]))."""
    labeled, n = ndimage.label(seg)
    sizes = np.bincount(labeled.ravel(), minlength=n + 1)[1:]
    return labeled == int(np.argmax(sizes)) + 1


def postprocess_prediction(pred, gaussian_std=1, threshold=0.5, fill_holes=True, connected_component=True):
    pred = ndimage.gaussian_filter(pred, gaussian_std)
    seg = pred > threshold
    if fill_holes:
        seg = ndimage.binary_fill_holes(seg)
    if connected_component:
        seg = largest_component(seg)
    return seg
