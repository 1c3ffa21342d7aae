"""Per-op parity cases shared by tests/test_gpu_ops.py and tools/gpu_diag.py.

Each case runs ONE kernel through the C ABI (fm_op_* hooks, host fp32 channels-last in/out) and
compares with a plain PyTorch-CPU fp32/fp64 reference of the same op on the same bf16-rounded
inputs. Tolerance (stated once): device tensors are bf16 with fp32 accumulation, so an output
element may differ from the exact result by one bf16 rounding of itself plus accumulation-order
noise:  |got - ref| <= 2^-7 * |ref| + 2^-8 * max|ref|   (bf16 has 8 significand bits).
Gradients w.r.t. weights are fp32 end to end: rel. error of the whole tensor <= 2e-3.
"""
import ctypes

import numpy as np
import torch
import torch.nn.functional as F

from fetal_net import _lib


def bf16_round(a):
    return torch.as_tensor(np.asarray(a, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def close_bf16(got, ref):
    ref = np.asarray(ref, np.float64)
    got = np.asarray(got, np.float64)
    tol = 2.0 ** -7 * np.abs(ref) + 2.0 ** -8 * max(np.abs(ref).max(), 1e-30)
    err = np.abs(got - ref)
    worst = float((err / tol).max())
    return worst <= 1.0, worst


def rel_err(got, ref):
    ref = np.asarray(ref, np.float64)
    got = np.asarray(got, np.float64)
    return float(np.linalg.norm(got - ref) / max(np.linalg.norm(ref), 1e-30))


def cl_to_cf(x):  # [N,X,Y,Z,C] -> [N,C,X,Y,Z]
    return torch.as_tensor(x).permute(0, 4, 1, 2, 3).contiguous()


def cf_to_cl(x):
    return x.permute(0, 2, 3, 4, 1).contiguous().numpy()


def keras_to_torch_w(w):  # (k,k,k,Cin,Cout) -> (Cout,Cin,k,k,k); a 2D kernel (3,3,Cin,Cout) -> (Cout,Cin,3,3,1)
    w = torch.as_tensor(w)
    if w.dim() == 4:
        w = w[:, :, None]
    return w.permute(4, 3, 0, 1, 2).contiguous()


def kshape(k):  # spatial extent of a Keras kernel for kernel code k (31 = 3x3 Conv2D on a Z = 1 volume)
    return (3, 3) if k == 31 else (k, k, k)


def kpad(k):  # 'same' padding of the equivalent conv3d
    return (1, 1, 0) if k == 31 else k // 2


def ktaps(k):
    return int(np.prod(kshape(k)))


CONV_CASES = [
    # name, N, X, Y, Z, C1, C2, Cout, k
    ("c16_32_8cube", 2, 8, 8, 8, 16, 0, 32, 3),         # SW32 operands (enc0b shape class)
    ("c32_32_16cube", 1, 16, 16, 16, 32, 0, 32, 3),     # SW64
    ("c64_64", 2, 8, 8, 8, 64, 0, 64, 3),               # SW128
    ("c128_256", 1, 8, 8, 8, 128, 0, 256, 3),           # 2 K chunks, 2 N tiles
    ("cat64_32_to32", 1, 16, 16, 16, 64, 32, 32, 3),    # dec0a: two sources, mixed swizzle
    ("cat256_128_to128", 1, 8, 8, 8, 256, 128, 128, 3), # dec2a
    ("ragged_12x10x6", 2, 12, 10, 6, 32, 0, 64, 3),     # partial tiles / clipping
    ("tiny_4cube", 3, 4, 4, 4, 16, 0, 16, 3),           # box larger than the tensor
    ("k1_64_32", 2, 8, 8, 8, 64, 0, 32, 1),             # 1x1x1 (Isensee localisation shape)
    ("cfg_64cube_16_32", 1, 64, 64, 64, 16, 0, 32, 3),  # enc0b at the real patch size
]

# shapes the plane-marching kernel covers (Y % 16 == 0, Z % 8 == 0, filter bank resident in smem)
MARCH_CASES = [
    ("m32_32_16cube", 1, 16, 16, 16, 32, 0, 32, 3),
    ("m16_32_32cube", 2, 32, 32, 32, 16, 0, 32, 3),     # SW32 slabs, ring wrap (X > 16 blocks)
    ("m32_64_16x32x16", 1, 16, 32, 16, 32, 0, 64, 3),   # N = 64 (ring of 8 blocks)
    ("m_oddx_10x16x8", 3, 10, 16, 8, 32, 0, 32, 3),     # X not a multiple of the x-chunk
    ("m_cat64_32_32cube", 2, 32, 32, 32, 64, 32, 32, 3),  # dec0a: two sources, mixed swizzle
    ("m64_16_32cube", 1, 32, 32, 32, 64, 0, 16, 3),     # N = 16 blocks
    ("m_x2", 2, 2, 16, 8, 16, 0, 16, 3),                # only two planes
    ("m_cfg_64cube_32_32", 1, 64, 64, 64, 32, 0, 32, 3),  # dec0b at the real patch size
    # equal plane ranges per CTA that cross column boundaries: segments of 1-4 planes (7 planes per column, 4 per CTA)
    ("m_ragged_7x32x16", 2, 7, 32, 16, 32, 0, 32, 3),
    ("m_ragged_cat_13x32x32", 1, 13, 32, 32, 64, 32, 32, 3),
]


# shapes for the marching wgrad kernel (Cin, Cout multiples of 32)
WGRAD_MARCH_CASES = [
    ("w32_32_16cube", 1, 16, 16, 16, 32, 0, 32, 3),
    ("w32_32_32cube", 2, 32, 32, 32, 32, 0, 32, 3),      # dY ring wrap (X > 8)
    ("w64_32_16x32x16", 1, 16, 32, 16, 64, 0, 32, 3),    # two ci chunks
    ("w32_64_oddx", 3, 10, 16, 8, 32, 0, 64, 3),         # two co chunks, X not multiple of chunk
    ("w128_64_x2", 2, 2, 16, 16, 128, 0, 64, 3),         # 8 pairs, two planes
    ("w_cfg_64cube_32_32", 1, 64, 64, 64, 32, 0, 32, 3),
    ("w16_32_32cube", 2, 32, 32, 32, 16, 0, 32, 3),      # enc0b: Cin = 16 (SWIZZLE_32B X operand, 8 M blocks)
    ("w16_16_32cube", 2, 32, 32, 32, 16, 0, 16, 3),      # Isensee level 0: Cout = 16 (SWIZZLE_32B dY, N = 48)
    ("w32_16_16x16x24", 1, 16, 16, 24, 32, 0, 16, 3),    # Isensee u0_up: 32 -> 16
    ("w_ragged_7x32x16", 2, 7, 32, 16, 32, 0, 32, 3),    # plane ranges crossing column boundaries, 1-plane segments
    ("w_ragged_13x32x32", 1, 13, 32, 32, 64, 0, 32, 3),
]


def conv_fprop_case(ctx, impl, case, seed=0, relu=1):
    name, N, X, Y, Z, C1, C2, Cout, k = case
    rng = np.random.default_rng(seed)
    x1 = bf16_round(rng.standard_normal((N, X, Y, Z, C1)))
    x2 = bf16_round(rng.standard_normal((N, X, Y, Z, C2))) if C2 else None
    w = bf16_round(rng.standard_normal(kshape(k) + (C1 + C2, Cout)) / np.sqrt(ktaps(k) * (C1 + C2)))
    b = rng.standard_normal(Cout).astype(np.float32)
    y = np.empty((N, X, Y, Z, Cout), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv3d_fprop(ctx.handle, impl, _lib.fptr(x1), _lib.fptr(x2), _lib.fptr(w), _lib.fptr(b),
                                      N, X, Y, Z, C1, C2, Cout, k, relu, _lib.fptr(y)))
    xin = torch.as_tensor(x1 if x2 is None else np.concatenate([x1, x2], -1))
    ref = F.conv3d(cl_to_cf(xin).double(), keras_to_torch_w(w).double(), torch.as_tensor(b).double(), padding=kpad(k))
    return close_bf16(y, cf_to_cl(F.relu(ref) if relu else ref))


def conv_fprop_raw(ctx, impl, case, seed=0):
    """The raw output of one fprop launch (for run-to-run bit-reproducibility checks)."""
    name, N, X, Y, Z, C1, C2, Cout, k = case
    rng = np.random.default_rng(seed)
    x1 = bf16_round(rng.standard_normal((N, X, Y, Z, C1)))
    x2 = bf16_round(rng.standard_normal((N, X, Y, Z, C2))) if C2 else None
    w = bf16_round(rng.standard_normal((k, k, k, C1 + C2, Cout)) / np.sqrt(k ** 3 * (C1 + C2)))
    b = rng.standard_normal(Cout).astype(np.float32)
    y = np.empty((N, X, Y, Z, Cout), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv3d_fprop(ctx.handle, impl, _lib.fptr(x1), _lib.fptr(x2), _lib.fptr(w), _lib.fptr(b),
                                      N, X, Y, Z, C1, C2, Cout, k, 1, _lib.fptr(y)))
    return y


def conv_dgrad_case(ctx, impl, case, seed=1):
    name, N, X, Y, Z, C1, C2, Cout, k = case
    Cin = C1  # single source
    rng = np.random.default_rng(seed)
    dy = bf16_round(rng.standard_normal((N, X, Y, Z, Cout)))
    w = bf16_round(rng.standard_normal(kshape(k) + (Cin, Cout)) / np.sqrt(ktaps(k) * Cout))
    act = bf16_round(rng.standard_normal((N, X, Y, Z, Cin)))       # ReLU mask source (act > 0)
    dx = np.empty((N, X, Y, Z, Cin), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv_dgrad(ctx.handle, impl, _lib.fptr(dy), _lib.fptr(w), _lib.fptr(act),
                                      N, X, Y, Z, Cin, Cout, k, _lib.fptr(dx)))
    ref = F.conv_transpose3d(cl_to_cf(dy).double(), keras_to_torch_w(w).double(), padding=kpad(k))
    ref = cf_to_cl(ref) * (act > 0)
    return close_bf16(dx, ref)


def conv_wgrad_case(ctx, impl, case, seed=2):
    name, N, X, Y, Z, C1, C2, Cout, k = case
    Cin = C1
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((N, X, Y, Z, Cin)))
    dy = bf16_round(rng.standard_normal((N, X, Y, Z, Cout)))
    dw = np.empty(kshape(k) + (Cin, Cout), np.float32)
    db = np.empty((Cout,), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv_wgrad(ctx.handle, impl, _lib.fptr(x), _lib.fptr(dy), N, X, Y, Z, Cin, Cout, k,
                                      _lib.fptr(dw), _lib.fptr(db)))
    xt = cl_to_cf(x).double().requires_grad_(False)
    wt = torch.zeros((Cout, Cin) + (kshape(k) + (1,))[:3], dtype=torch.float64, requires_grad=True)
    out = F.conv3d(xt, wt, padding=kpad(k))
    out.backward(cl_to_cf(dy).double())
    ref_w = wt.grad.permute(2, 3, 4, 1, 0).numpy().reshape(dw.shape)
    ref_b = dy.reshape(-1, Cout).astype(np.float64).sum(0)
    e = max(rel_err(dw, ref_w), rel_err(db, ref_b))
    return e <= 2e-3, e / 2e-3


# decoder convolutions at coarse resolution: name, N, X, Y, Z (fine), Cc (coarse / up source), Cs (skip), Cout
UP_CASES = [
    ("up_dec2a_16cube", 1, 16, 16, 16, 256, 128, 128),   # dec2a of the depth-4 / 16-filter U-Net (2 N tiles in dgrad)
    ("up_dec1a_32cube", 1, 32, 32, 32, 128, 64, 64),     # dec1a
    ("up_dec0a_16cube", 2, 16, 16, 16, 64, 32, 32),      # dec0a channel mix (mixed swizzle widths)
    ("up_ragged_12x20x8", 2, 12, 20, 8, 64, 64, 64),     # coarse extents 6x10x4: partial boxes / clipping
    ("up_small_4cube", 3, 4, 4, 4, 32, 16, 16),          # coarse box larger than the tensor
]


def _up_reference(coarse, skip, w, b, dy=None):
    """torch fp64: conv3d(concatenate([nearest-upsample x2 (coarse), skip])) and its gradients."""
    ct = cl_to_cf(coarse).double().requires_grad_(True)
    up = F.interpolate(ct, scale_factor=2, mode="nearest")
    wt = keras_to_torch_w(w).double().requires_grad_(True)
    out = F.conv3d(torch.cat([up, cl_to_cf(skip).double()], 1), wt, None if b is None else torch.as_tensor(b).double(),
                   padding=1)
    if dy is None:
        return out
    out.backward(cl_to_cf(dy).double())
    return cf_to_cl(ct.grad), wt.grad.permute(2, 3, 4, 1, 0).numpy()


def conv_up_fprop_case(ctx, case, seed=7):
    name, N, X, Y, Z, Cc, Cs, Cout = case
    rng = np.random.default_rng(seed)
    coarse = bf16_round(rng.standard_normal((N, X // 2, Y // 2, Z // 2, Cc)))
    skip = bf16_round(rng.standard_normal((N, X, Y, Z, Cs)))
    w = bf16_round(rng.standard_normal((3, 3, 3, Cc + Cs, Cout)) / np.sqrt(27 * (Cc + Cs)))
    b = rng.standard_normal(Cout).astype(np.float32)
    y = np.empty((N, X, Y, Z, Cout), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv3d_up_fprop(ctx.handle, _lib.fptr(coarse), _lib.fptr(skip), _lib.fptr(w), _lib.fptr(b),
                                         N, X, Y, Z, Cc, Cs, Cout, 1, _lib.fptr(y)))
    ref = F.relu(_up_reference(coarse, skip, w, b)).detach()
    return close_bf16(y, cf_to_cl(ref))


def conv_up_bwd_case(ctx, case, seed=8):
    """Gradient towards the coarse tensor (ReLU-masked) within the bf16 bound, weight gradient of the up-source
    channels within 2e-3 (fp32 accumulation end to end)."""
    name, N, X, Y, Z, Cc, Cs, Cout = case
    rng = np.random.default_rng(seed)
    coarse = bf16_round(rng.standard_normal((N, X // 2, Y // 2, Z // 2, Cc)))
    skip = np.zeros((N, X, Y, Z, Cs), np.float32)
    dy = bf16_round(rng.standard_normal((N, X, Y, Z, Cout)))
    w = bf16_round(rng.standard_normal((3, 3, 3, Cc + Cs, Cout)) / np.sqrt(27 * Cout))
    dc = np.empty_like(coarse)
    dw = np.empty((3, 3, 3, Cc, Cout), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv3d_up_bwd(ctx.handle, _lib.fptr(coarse), _lib.fptr(dy), _lib.fptr(w), N, X, Y, Z, Cc, Cs,
                                       Cout, 1, _lib.fptr(dc), _lib.fptr(dw)))
    ref_dc, ref_dw = _up_reference(coarse, skip, w, None, dy)
    ok, worst = close_bf16(dc, ref_dc * (coarse > 0))
    e = rel_err(dw, ref_dw[:, :, :, :Cc, :])
    return ok and e <= 2e-3, max(worst, e / 2e-3)


FIRST_CASES = [  # name, N, X, Y, Z, Cout : shapes the im2col + tcgen05 first-layer kernels cover (Y % 16 == 0, Z % 8 == 0)
    ("first16_32cube", 2, 32, 32, 32, 16),
    ("first32_16x32x8", 3, 5, 32, 8, 32),      # Isensee / 32-filter variants; single z tile, odd x
    ("first16_64cube", 1, 64, 64, 64, 16),     # the BASELINE patch
    ("first16_ragged_9x12x6", 2, 9, 12, 6, 16),  # not covered by the tensor-core kernel: SIMT route
]


def conv_first_case(ctx, case, seed=9):
    """First conv (fp32 single-channel input) forward within the bf16 bound (the tensor-core route rounds the volume to
    bf16, so the reference does too) and its weight gradient within 2e-3."""
    name, N, X, Y, Z, Cout = case
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((N, X, Y, Z)))
    w = bf16_round(rng.standard_normal((3, 3, 3, 1, Cout)) / np.sqrt(27.0))
    b = rng.standard_normal(Cout).astype(np.float32)
    dy = bf16_round(rng.standard_normal((N, X, Y, Z, Cout)))
    y = np.empty((N, X, Y, Z, Cout), np.float32)
    dw = np.empty((3, 3, 3, 1, Cout), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv3d_first(ctx.handle, _lib.fptr(x), _lib.fptr(w), _lib.fptr(b), N, X, Y, Z, Cout, 1,
                                      _lib.fptr(y), _lib.fptr(dy), _lib.fptr(dw)))
    xt = torch.as_tensor(x)[:, None].double()
    wt = keras_to_torch_w(w).double().requires_grad_(True)
    out = F.conv3d(xt, wt, torch.as_tensor(b).double(), padding=1)
    ok, worst = close_bf16(y, cf_to_cl(F.relu(out).detach()))
    out.backward(cl_to_cf(dy).double())
    e = rel_err(dw, wt.grad.permute(2, 3, 4, 1, 0).numpy())
    return ok and e <= 2e-3, max(worst, e / 2e-3)


def maxpool_case(ctx, seed=3, shape=(2, 8, 12, 16, 32), pz=2):
    N, X, Y, Z, C = shape
    pool = (2, 2, pz)
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((N, X, Y, Z, C)))
    y = np.empty((N, X // 2, Y // 2, Z // pz, C), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_maxpool(ctx.handle, _lib.fptr(x), N, X, Y, Z, C, pz, _lib.fptr(y)))
    ref = cf_to_cl(F.max_pool3d(cl_to_cf(x), pool))
    ok = np.array_equal(y, ref)                                    # exact: max of bf16 values
    # backward with skip-gradient add and ReLU mask
    dy = bf16_round(rng.standard_normal(y.shape))
    dskip = bf16_round(rng.standard_normal(x.shape))
    dx = np.empty_like(x)
    _lib.check(lib.fm_op_maxpool_bwd(ctx.handle, _lib.fptr(x), _lib.fptr(dy), _lib.fptr(dskip), N, X, Y, Z, C, pz,
                                       _lib.fptr(dx)))
    xt = cl_to_cf(x).double().requires_grad_(True)
    F.max_pool3d(xt, pool).backward(cl_to_cf(dy).double())
    refb = (cf_to_cl(xt.grad) + dskip) * (x > 0)
    ok2, worst = close_bf16(dx, refb)
    return ok and ok2, worst if ok else float("inf")


def upsample_case(ctx, seed=4, shape=(2, 4, 6, 8, 64), pz=2):
    N, X, Y, Z, C = shape
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((N, X, Y, Z, C)))
    y = np.empty((N, 2 * X, 2 * Y, pz * Z, C), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_upsample(ctx.handle, _lib.fptr(x), N, X, Y, Z, C, pz, _lib.fptr(y)))
    ref = np.repeat(np.repeat(np.repeat(x, 2, 1), 2, 2), pz, 3)
    ok = np.array_equal(y, ref)
    dy = bf16_round(rng.standard_normal(y.shape))
    act = bf16_round(rng.standard_normal(x.shape))
    dx = np.empty_like(x)
    _lib.check(lib.fm_op_upsample_bwd(ctx.handle, _lib.fptr(dy), _lib.fptr(act), N, X, Y, Z, C, pz, _lib.fptr(dx)))
    refb = dy.astype(np.float64).reshape(N, X, 2, Y, 2, Z, pz, C).sum((2, 4, 6)) * (act > 0)
    ok2, worst = close_bf16(dx, refb)
    return ok and ok2, worst if ok else float("inf")


def dice_case(ctx, seed=5):
    n = 8 * 16 ** 3 + 3           # not a multiple of 4: exercises the scalar tail
    rng = np.random.default_rng(seed)
    p = rng.random(n).astype(np.float32)
    t = (rng.random(n) < 0.3).astype(np.float32)
    sums = np.zeros(8, np.float64)
    g = np.empty(n, np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_dice(ctx.handle, _lib.fptr(p), _lib.fptr(t), n, _lib.dptr(sums), _lib.fptr(g)))
    pb, tb = (p > 0.5), (t > 0.5)
    ref = np.array([(t.astype(np.float64) * p).sum(), t.sum(dtype=np.float64), p.sum(dtype=np.float64),
                    (tb & pb).sum(), tb.sum(), pb.sum(), (t == pb.astype(np.float32)).sum(), n], np.float64)
    e1 = float(np.max(np.abs(sums - ref) / np.maximum(np.abs(ref), 1)))
    I, S = ref[0], ref[1] + ref[2] + 1.0
    gref = -(2.0 * t * S - (2.0 * I + 1.0)) / (S * S)
    e2 = rel_err(g, gref)
    # float32 per-thread partial sums over <= n/151552 elements each, then float64: 1e-6 is ample
    return e1 <= 1e-6 and e2 <= 1e-5, max(e1 / 1e-6, e2 / 1e-5)


def dice_xent_case(ctx, with_mask, seed=15):
    """fm_op_dice_xent (dice_and_xent / dice_and_xent_mask, metrics.py:68-95) against torch autograd in fp64: the ninth
    statistic (sum w * bce) and d(loss)/d(logit) through the sigmoid. Probabilities include saturated ones (the Keras
    clip at 1e-7 is active there: zero cross-entropy gradient)."""
    import torch
    from oracle import unet_oracle as uo
    n = 4 * 16 ** 3 + 2
    rng = np.random.default_rng(seed)
    z = (4.0 * rng.standard_normal(n)).astype(np.float32)
    z[:64] = 40.0 * np.sign(z[:64])                        # saturated: p == 1 or ~4e-18 in fp32
    p = (1.0 / (1.0 + np.exp(-z.astype(np.float64)))).astype(np.float32)
    t = (rng.random(n) < 0.3).astype(np.float32)
    mask = (6.0 * rng.random(n)).astype(np.float32) if with_mask else None
    xw, sigma = 0.7, 3.0
    sums = np.zeros(9, np.float64)
    g = np.empty(n, np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_dice_xent(ctx.handle, _lib.fptr(p), _lib.fptr(t), _lib.fptr(mask) if with_mask else None, n,
                                   xw, sigma, _lib.dptr(sums), _lib.fptr(g)))
    # reference: the loss as a function of the logit, with p fixed to the SAME fp32 probabilities the kernel saw
    pt = torch.tensor(p.astype(np.float64), requires_grad=True)
    tt = torch.tensor(t.astype(np.float64))
    mt = torch.tensor(mask.astype(np.float64)) if with_mask else None
    loss = uo.dice_and_xent(tt, pt, xw, mt, sigma if with_mask else None)
    loss.backward()
    gref = (pt.grad * pt.detach() * (1 - pt.detach())).numpy()       # chain through the sigmoid
    w = np.exp(-mask.astype(np.float64) / sigma) if with_mask else np.ones(n)
    xent_ref = float((torch.as_tensor(w) * uo.binary_crossentropy(tt, pt.detach())).sum())
    e1 = abs(sums[8] - xent_ref) / abs(xent_ref)
    lref = float(loss.detach())
    e2 = abs((-(2 * sums[0] + 1) / (sums[1] + sums[2] + 1) + xw * sums[8] / sums[7]) - lref) / abs(lref)
    e3 = rel_err(g, gref)
    # fp32 log / exp per voxel, fp32 partial sums then fp64: 2e-6 on the sums; 2e-5 on the gradient
    return e1 <= 2e-6 and e2 <= 2e-6 and e3 <= 2e-5, max(e1 / 2e-6, e2 / 2e-6, e3 / 2e-5)


def adam_case(ctx, seed=6):
    from oracle.unet_oracle import keras_adam_step
    n = 100003
    rng = np.random.default_rng(seed)
    p = rng.standard_normal(n).astype(np.float32)
    m = np.zeros(n, np.float32)
    v = np.zeros(n, np.float32)
    p2, m2, v2 = p.copy(), m.copy(), v.copy()
    lib = _lib.load()
    worst = 0.0
    for it in range(3):
        g = rng.standard_normal(n).astype(np.float32) * 1e-3
        _lib.check(lib.fm_op_adam(ctx.handle, _lib.fptr(p), _lib.fptr(g), _lib.fptr(m), _lib.fptr(v), n, it, 1e-3))
        keras_adam_step(p2, g, m2, v2, it, 1e-3)
        worst = max(worst, float(np.max(np.abs(p - p2))), float(np.max(np.abs(m - m2))))
    return worst <= 2e-6, worst / 2e-6


# ---------------------------------------------------------------------------------------------------------------------
# Layer kernels of the Isensee, batch-normalised, deconvolution and 2D models (tests/test_gpu_layer_ops.py). References
# are float64 torch on the same bf16-rounded inputs; backward references come from autograd on the Keras-form forward.
# Bounds (stated once):
#   bf16 outputs (y, dx): close_bf16 per element, taken per channel where a channel's scale differs from the others';
#   fp32 reductions (dgamma, dbeta, db, head sums and weights, moving statistics, norm statistics): per channel
#     |got - ref| <= 1e-5 * sum |term|  (the sums cancel, so the bound follows the terms, not the result);
#   weight gradients from bf16 products (conv / deconv dw): whole-tensor relative error <= 2e-3, as for wgrad;
#   pure data movement (zero insertion, depth <-> space without bias, seg_upsample_add, sumpool_f32): exact.
# ---------------------------------------------------------------------------------------------------------------------
RED_TOL = 1e-5


def close_bf16_per_channel(got, ref):
    """close_bf16 with the max|ref| term taken per channel (last axis)."""
    ref = np.asarray(ref, np.float64)
    got = np.asarray(got, np.float64)
    C = ref.shape[-1]
    r, g = ref.reshape(-1, C), got.reshape(-1, C)
    tol = 2.0 ** -7 * np.abs(r) + 2.0 ** -8 * np.maximum(np.abs(r).max(0), 1e-30)
    worst = float((np.abs(g - r) / tol).max())
    return worst <= 1.0, worst


def close_sum(got, ref, abs_terms, extra=0.0):
    """fp32 reduction bound: |got - ref| <= RED_TOL * sum|term| (+ `extra`, e.g. the fp32 rounding of the stored
    result), element-wise."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    tol = RED_TOL * np.asarray(abs_terms, np.float64) + extra + 1e-30
    worst = float((np.abs(got - ref) / tol).max())
    return worst <= 1.0, worst


# name, N, voxels per sample, C. Channel-group folds: shuffles for C < 256, shared memory for C >= 256, C = 8 = one group
# of 256 lanes. Blocks per sample: 1 below 1024 voxels, capped at 1024 above 524288; 1000, 1023, 4097 and 7 leave partial
# blocks that neither the block size nor the backward's 2-voxel stride divides; 32^3 gives N * blocks > 32 (the batch-norm
# fold wraps its lanes).
NORM_CASES = [
    ("n1_v1_c64", 1, 1, 64),
    ("n3_v1_c16", 3, 1, 16),
    ("n3_v7_c16", 3, 7, 16),
    ("n1_v511_c32", 1, 511, 32),
    ("n3_v1000_c64", 3, 1000, 64),
    ("n1_v1023_c128", 1, 1023, 128),
    ("n3_v1024_c256", 3, 1024, 256),
    ("n1_v4097_c512", 1, 4097, 512),
    ("n3_v4097_c8", 3, 4097, 8),
    ("n3_v1000_c512", 3, 1000, 512),
    ("n1_v1023_c256", 1, 1023, 256),
    ("n3_v32k_c8", 3, 32 ** 3, 8),
    ("n1_v32k_c128", 1, 32 ** 3, 128),
    ("n2_v32k_c32", 2, 32 ** 3, 32),
]
NORM_BIG = ("n1_cfg3_l0_c16", 1, 128 * 128 * 64, 16)   # the cfg3 level-0 shape (more blocks than the 1024 cap)


def norm_inputs(N, vox, C, seed):
    """x [N, vox, C] bf16 with two numerical edges: channel 0 has mean 8 x its std (fp32 E[x^2] - mean^2), channel 1 a
    std of about eps = 1e-3 (largest s / sigma term of the backward)."""
    rng = np.random.default_rng(seed)
    x = 0.5 + rng.standard_normal((N, vox, C))
    x[..., 0] = 8.0 + rng.standard_normal((N, vox))
    x[..., 1] = 1e-3 * rng.standard_normal((N, vox)) - 2e-3
    gamma = (1.0 + 0.5 * rng.standard_normal(C)).astype(np.float32)
    beta = (0.3 * rng.standard_normal(C)).astype(np.float32)
    return bf16_round(x), gamma, beta, rng


def _norm_cf(a):  # [N, vox, C] -> [N, C, vox] float64 tensor
    return torch.as_tensor(np.asarray(a, np.float64)).permute(0, 2, 1).contiguous()


def _norm_cl(t):
    return t.detach().permute(0, 2, 1).numpy()


def drop_scales(rng, N, C, rate=0.3):
    """SpatialDropout keep / scale factors: some channels 0, the rest 1 / (1 - rate)."""
    keep = rng.random((N, C)) >= rate
    keep[:, 0] = True
    return np.where(keep, 1.0 / (1.0 - rate), 0.0).astype(np.float32)


def instnorm_fwd_case(ctx, case, with_add, with_scale, seed=20):
    from oracle.unet_oracle import _instance_norm
    name, N, vox, C = case
    x, gamma, beta, rng = norm_inputs(N, vox, C, seed)
    add = bf16_round(rng.standard_normal((N, vox, C))) if with_add else None
    cs = drop_scales(rng, N, C) if with_scale else None
    y = np.empty((N, vox, C), np.float32)
    stats = np.empty((N, C, 2), np.float32)
    _lib.check(_lib.load().fm_op_instnorm_lrelu(ctx.handle, _lib.fptr(x), _lib.fptr(gamma), _lib.fptr(beta),
                                                _lib.fptr(add), _lib.fptr(cs), N, vox, C, _lib.fptr(y),
                                                _lib.fptr(stats)))
    xt = _norm_cf(x)
    ref = F.leaky_relu(_instance_norm(xt, torch.as_tensor(gamma).double(), torch.as_tensor(beta).double()), 0.3)
    if cs is not None:
        ref = ref * torch.as_tensor(cs).double()[:, :, None]
    if add is not None:
        ref = ref + _norm_cf(add)
    ok, worst = close_bf16_per_channel(y, _norm_cl(ref))
    # statistics: mean = sum x / n and var = sum x^2 / n - mean^2 are fp32 partial sums
    x64 = np.asarray(x, np.float64)
    mean = x64.mean(1)
    var = x64.var(1)
    ok1, w1 = close_sum(stats[..., 0], mean, np.abs(x64).mean(1), 1e-7 * np.abs(mean))
    var_got = np.maximum(1.0 / stats[..., 1].astype(np.float64) - float(np.float32(1e-3)), 0.0) ** 2  # eps = 1e-3f
    ok2, w2 = close_sum(var_got, var, (x64 ** 2).mean(1) + mean ** 2, 1e-6 * var)
    return ok and ok1 and ok2, max(worst, w1, w2)


def instnorm_bwd_case(ctx, case, with_gy2, with_scale, seed=21):
    from oracle.unet_oracle import _instance_norm
    name, N, vox, C = case
    x, gamma, beta, rng = norm_inputs(N, vox, C, seed)
    gy = bf16_round(rng.standard_normal((N, vox, C)))
    gy2 = bf16_round(rng.standard_normal((N, vox, C))) if with_gy2 else None
    cs = drop_scales(rng, N, C) if with_scale else None
    dx = np.empty((N, vox, C), np.float32)
    dg = np.empty(C, np.float32)
    db = np.empty(C, np.float32)
    _lib.check(_lib.load().fm_op_instnorm_lrelu_bwd(ctx.handle, _lib.fptr(x), _lib.fptr(gamma), _lib.fptr(beta),
                                                    _lib.fptr(gy), _lib.fptr(gy2), _lib.fptr(cs), N, vox, C,
                                                    _lib.fptr(dx), _lib.fptr(dg), _lib.fptr(db)))
    xt = _norm_cf(x).requires_grad_(True)
    gt = torch.as_tensor(gamma).double().requires_grad_(True)
    bt = torch.as_tensor(beta).double().requires_grad_(True)
    y = F.leaky_relu(_instance_norm(xt, gt, bt), 0.3)
    if cs is not None:
        y = y * torch.as_tensor(cs).double()[:, :, None]
    g = _norm_cf(gy) + (_norm_cf(gy2) if gy2 is not None else 0.0)
    y.backward(g)
    ok, worst = close_bf16_per_channel(dx, _norm_cl(xt.grad))
    # terms of dgamma / dbeta: g_z * xh and g_z with g_z = dL/dz at the norm output
    with torch.no_grad():
        z = _instance_norm(xt, gt, bt)
        xh = (z - bt[None, :, None]) / gt[None, :, None]
        gz = g * torch.where(z > 0, 1.0, 0.3) * (torch.as_tensor(cs).double()[:, :, None] if cs is not None else 1.0)
        tg = (gz * xh).abs().sum((0, 2)).numpy()
        tb = gz.abs().sum((0, 2)).numpy()
    ok1, w1 = close_sum(dg, gt.grad.numpy(), tg)
    ok2, w2 = close_sum(db, bt.grad.numpy(), tb)
    return ok and ok1 and ok2, max(worst, w1, w2)


def _bn_weights(gamma, beta, mm, mv):
    return {"bn/gamma": gamma, "bn/beta": beta, "bn/moving_mean": mm, "bn/moving_variance": mv}


def batchnorm_fwd_case(ctx, case, training, seed=22):
    from oracle.unet_oracle import _batch_norm
    name, N, vox, C = case
    x, gamma, beta, rng = norm_inputs(N, vox, C, seed)
    mm = (0.5 * rng.standard_normal(C)).astype(np.float32)
    mv = (0.5 + rng.random(C)).astype(np.float32)
    mm_got, mv_got = mm.copy(), mv.copy()
    y = np.empty((N, vox, C), np.float32)
    _lib.check(_lib.load().fm_op_batchnorm_relu(ctx.handle, int(training), _lib.fptr(x), _lib.fptr(gamma),
                                                _lib.fptr(beta), _lib.fptr(mm_got), _lib.fptr(mv_got), N, vox, C,
                                                _lib.fptr(y)))
    upd = {}
    ref = F.relu(_batch_norm(_norm_cf(x), _bn_weights(gamma, beta, mm, mv), "bn", training, upd))
    ok, worst = close_bf16_per_channel(y, _norm_cl(ref))
    if not training:
        return ok and np.array_equal(mm_got, mm) and np.array_equal(mv_got, mv), worst
    # the moving-average step (Keras: momentum 0.99, variance times n / (n - (1 + eps))) on fp32 batch sums
    x64 = np.asarray(x, np.float64).reshape(-1, C)
    n = x64.shape[0]
    m = x64.mean(0)
    ok1, w1 = close_sum(mm_got, upd["bn/moving_mean"], 0.01 * np.abs(x64).mean(0), 1e-7 * np.abs(mm_got))
    ok2, w2 = close_sum(mv_got, upd["bn/moving_variance"], 0.01 * ((x64 ** 2).mean(0) + m ** 2) * n / (n - 1.001),
                        1e-7 * np.abs(mv_got))
    return ok and ok1 and ok2, max(worst, w1, w2)


def batchnorm_bwd_case(ctx, case, with_gy2, seed=23):
    from oracle.unet_oracle import _batch_norm
    name, N, vox, C = case
    x, gamma, beta, rng = norm_inputs(N, vox, C, seed)
    gy = bf16_round(rng.standard_normal((N, vox, C)))
    gy2 = bf16_round(rng.standard_normal((N, vox, C))) if with_gy2 else None
    dx = np.empty((N, vox, C), np.float32)
    dg = np.empty(C, np.float32)
    db = np.empty(C, np.float32)
    _lib.check(_lib.load().fm_op_batchnorm_relu_bwd(ctx.handle, _lib.fptr(x), _lib.fptr(gamma), _lib.fptr(beta),
                                                    _lib.fptr(gy), _lib.fptr(gy2), N, vox, C, _lib.fptr(dx),
                                                    _lib.fptr(dg), _lib.fptr(db)))
    xt = _norm_cf(x).requires_grad_(True)
    gt = torch.as_tensor(gamma).double().requires_grad_(True)
    bt = torch.as_tensor(beta).double().requires_grad_(True)
    w = {"bn/gamma": gt, "bn/beta": bt, "bn/moving_mean": np.zeros(C), "bn/moving_variance": np.ones(C)}
    z = _batch_norm(xt, w, "bn", True, None)
    g = _norm_cf(gy) + (_norm_cf(gy2) if gy2 is not None else 0.0)
    F.relu(z).backward(g)
    ok, worst = close_bf16_per_channel(dx, _norm_cl(xt.grad))
    with torch.no_grad():
        xh = (z - bt[None, :, None]) / gt[None, :, None]
        gz = g * (z > 0)
        tg = (gz * xh).abs().sum((0, 2)).numpy()
        tb = gz.abs().sum((0, 2)).numpy()
    ok1, w1 = close_sum(dg, gt.grad.numpy(), tg)
    ok2, w2 = close_sum(db, bt.grad.numpy(), tb)
    return ok and ok1 and ok2, max(worst, w1, w2)


# name, N, Xin, Yin, Zin, Cin, Cout, k: the Isensee in-convs (stride 2, TF 'SAME': pad 0 before, 1 after)
STRIDED_CASES = [
    ("s16_32_16cube", 2, 16, 16, 16, 16, 32, 3),
    ("s32_64_16cube", 1, 16, 16, 16, 32, 64, 3),
    ("s64_128_8cube", 2, 8, 8, 8, 64, 128, 3),
    ("s128_256_8cube", 1, 8, 8, 8, 128, 256, 3),
    ("s_ragged_14x20x6", 2, 14, 20, 6, 16, 32, 3),     # output 7 x 10 x 3: no tile multiple
    ("s_one_voxel", 1, 2, 2, 2, 32, 64, 3),            # 1-voxel output
    ("s2d_16_32", 2, 32, 32, 1, 16, 32, 31),           # isensee2d: z is not strided
    ("s2d_64_128_ragged", 1, 14, 10, 1, 64, 128, 31),
    ("s2d_128_256", 1, 8, 8, 1, 128, 256, 31),
]


def conv_strided_case(ctx, case, seed=24):
    name, N, Xin, Yin, Zin, Cin, Cout, k = case
    pz = 1 if k == 31 else 2
    X, Y, Z = Xin // 2, Yin // 2, Zin // pz
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((N, Xin, Yin, Zin, Cin)))
    w = bf16_round(rng.standard_normal(kshape(k) + (Cin, Cout)) / np.sqrt(ktaps(k) * Cin))
    b = rng.standard_normal(Cout).astype(np.float32)
    dy = bf16_round(rng.standard_normal((N, X, Y, Z, Cout)))
    y = np.empty((N, X, Y, Z, Cout), np.float32)
    dx = np.empty_like(x)
    dw = np.empty_like(w)
    _lib.check(_lib.load().fm_op_conv_strided(ctx.handle, _lib.fptr(x), _lib.fptr(w), _lib.fptr(b), N, Xin, Yin, Zin,
                                              Cin, Cout, k, _lib.fptr(y), _lib.fptr(dy), _lib.fptr(dx),
                                              _lib.fptr(dw)))
    xt = cl_to_cf(x).double().requires_grad_(True)
    wt = keras_to_torch_w(w).double().requires_grad_(True)
    pad = (0, 0, 0, 1, 0, 1) if k == 31 else (0, 1) * 3
    out = F.conv3d(F.pad(xt, pad), wt, torch.as_tensor(b).double(), stride=(2, 2, pz))
    ok, worst = close_bf16(y, cf_to_cl(out.detach()))
    out.backward(cl_to_cf(dy).double())
    ok1, w1 = close_bf16(dx, cf_to_cl(xt.grad))
    e = rel_err(dw, wt.grad.permute(2, 3, 4, 1, 0).numpy().reshape(dw.shape))
    return ok and ok1 and e <= 2e-3, max(worst, w1, e / 2e-3)


# name, N, X, Y, Z (coarse), C, pz: Deconvolution3D (pz = 2) / Deconvolution2D (pz = 1, Z = 1), C -> C channels
DECONV_CASES = [
    ("d3_16_4cube", 2, 4, 4, 4, 16, 2),
    ("d3_64_4cube", 1, 4, 4, 4, 64, 2),
    ("d3_256_2cube", 2, 2, 2, 2, 256, 2),
    ("d3_ragged_3x5x2", 2, 3, 5, 2, 32, 2),
    ("d2_128_8x8", 2, 8, 8, 1, 128, 1),
    ("d2_ragged_5x3", 1, 5, 3, 1, 32, 1),
]


def deconv_case(ctx, case, relu_mask, seed=25):
    name, N, X, Y, Z, C, pz = case
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((N, X, Y, Z, C)))
    ks = (2, 2, 2) if pz == 2 else (2, 2)
    w = bf16_round(rng.standard_normal(ks + (C, C)) / np.sqrt(C))      # (..., Cout, Cin): not symmetric
    b = (0.1 * rng.standard_normal(C)).astype(np.float32)
    fine = (N, 2 * X, 2 * Y, pz * Z, C)
    dy = bf16_round(rng.standard_normal(fine))
    y = np.empty(fine, np.float32)
    dx = np.empty_like(x)
    dw = np.empty_like(w)
    db = np.empty(C, np.float32)
    _lib.check(_lib.load().fm_op_deconv(ctx.handle, _lib.fptr(x), _lib.fptr(w), _lib.fptr(b), N, X, Y, Z, C, pz,
                                        _lib.fptr(y), _lib.fptr(dy), int(relu_mask), _lib.fptr(dx), _lib.fptr(dw),
                                        _lib.fptr(db)))
    wk = torch.as_tensor(w).double()
    if pz == 1:
        wk = wk[:, :, None]                              # (2,2,1,Cout,Cin)
    wt = wk.permute(4, 3, 0, 1, 2).contiguous().requires_grad_(True)   # conv_transpose weight (Cin, Cout, kx, ky, kz)
    xt = cl_to_cf(x).double().requires_grad_(True)
    out = F.conv_transpose3d(xt, wt, torch.as_tensor(b).double(), stride=(2, 2, pz))
    ok, worst = close_bf16(y, cf_to_cl(out.detach()))
    out.backward(cl_to_cf(dy).double())
    ref_dx = cf_to_cl(xt.grad) * ((x > 0) if relu_mask else 1.0)
    ok1, w1 = close_bf16(dx, ref_dx)
    e = rel_err(dw, wt.grad.permute(2, 3, 4, 1, 0).numpy().reshape(w.shape))
    dy64 = dy.reshape(-1, C).astype(np.float64)
    ok2, w2 = close_sum(db, dy64.sum(0), np.abs(dy64).sum(0))
    return ok and ok1 and ok2 and e <= 2e-3, max(worst, w1, w2, e / 2e-3)


def depth_space_case(ctx, shape, pz, seed=26):
    """Both shuffles without bias, exact: fine[n][2x+a][2y+b][pz*z+c][co] = z8[n][x][y][z][((a*2+b)*pz+c)*C + co]."""
    N, X, Y, Z, C = shape
    rng = np.random.default_rng(seed)
    z8 = bf16_round(rng.standard_normal((N, X, Y, Z, 4 * pz * C)))
    ref = z8.reshape(N, X, Y, Z, 2, 2, pz, C).transpose(0, 1, 4, 2, 5, 3, 6, 7).reshape(N, 2 * X, 2 * Y, pz * Z, C)
    fine = np.empty_like(ref)
    back = np.empty_like(z8)
    lib = _lib.load()
    _lib.check(lib.fm_op_depth_space(ctx.handle, 1, _lib.fptr(z8), N, X, Y, Z, C, pz, _lib.fptr(fine)))
    _lib.check(lib.fm_op_depth_space(ctx.handle, 0, _lib.fptr(ref), N, X, Y, Z, C, pz, _lib.fptr(back)))
    return np.array_equal(fine, ref) and np.array_equal(back, z8)


def zero_insert_case(ctx, shape, pz, seed=27):
    N, X, Y, Z, C = shape
    rng = np.random.default_rng(seed)
    c = bf16_round(rng.standard_normal(shape))
    ref = np.zeros((N, 2 * X, 2 * Y, pz * Z, C), np.float32)
    if pz == 2:
        ref[:, 1::2, 1::2, 1::2] = c
    else:
        ref[:, 1::2, 1::2, :] = c
    fine = np.full_like(ref, np.nan)
    _lib.check(_lib.load().fm_op_zero_insert(ctx.handle, _lib.fptr(c), N, X, Y, Z, C, pz, _lib.fptr(fine)))
    return np.array_equal(fine, ref)


def seg_upsample_add_case(ctx, shape, pz, seed=28):
    """out = fine + upsample(coarse), the same single fp32 addition per voxel: exact."""
    N, X, Y, Z = shape      # fine extents
    rng = np.random.default_rng(seed)
    fine = rng.standard_normal(shape).astype(np.float32)
    coarse = rng.standard_normal((N, X // 2, Y // 2, Z // pz)).astype(np.float32)
    ref = fine + np.repeat(np.repeat(np.repeat(coarse, 2, 1), 2, 2), pz, 3)
    out = np.empty_like(fine)
    _lib.check(_lib.load().fm_op_seg_upsample_add(ctx.handle, _lib.fptr(fine), _lib.fptr(coarse), N, X, Y, Z, pz,
                                                  _lib.fptr(out)))
    return np.array_equal(out, ref)


def sumpool_case(ctx, shape, pz, seed=29):
    """coarse = sum of the 2 x 2 (x pz) children in the kernel's fp32 order (x-major pairs, z pair first): exact."""
    N, X, Y, Z = shape      # coarse extents
    rng = np.random.default_rng(seed)
    fine = rng.standard_normal((N, 2 * X, 2 * Y, pz * Z)).astype(np.float32)
    f = fine.reshape(N, X, 2, Y, 2, Z, pz)
    ref = np.zeros((N, X, Y, Z), np.float32)
    for a in range(2):
        for b in range(2):
            pair = f[:, :, a, :, b, :, 0] + f[:, :, a, :, b, :, 1] if pz == 2 else f[:, :, a, :, b, :, 0]
            ref = ref + pair
    out = np.empty((N, X, Y, Z), np.float32)
    _lib.check(_lib.load().fm_op_sumpool_f32(ctx.handle, _lib.fptr(fine), N, X, Y, Z, pz, _lib.fptr(out)))
    return np.array_equal(out, ref)


# name, voxels, C: C in {16, 32, 64} takes the thread-per-voxel kernels, 8 / 128 / 256 the lanes-per-voxel ones;
# voxel counts are not multiples of 256 or of a block's voxels
HEAD_CASES = [
    ("h8", 4099, 8),
    ("h16", 5003, 16),
    ("h32", 777, 32),
    ("h64", 4097, 64),
    ("h128", 3001, 128),
    ("h256", 1031, 256),
    ("h16_big", 2 * 32 ** 3 + 5, 16),
    ("h256_big", 32 ** 3 + 9, 256),
]


def _head_inputs(voxels, C, seed):
    rng = np.random.default_rng(seed)
    x = bf16_round(rng.standard_normal((voxels, C)))
    w = (rng.standard_normal(C) / np.sqrt(C)).astype(np.float32)
    b = np.array([0.2], np.float32)
    # saturated logits: |z| >= 30 * sum|w| (p == 1 or ~1e-18 in fp32)
    x[:32] = 30.0 * np.sign(w)
    x[32:64] = -30.0 * np.sign(w)
    return x, w, b, rng


def head_fwd_case(ctx, case, sigmoid, seed=30):
    name, voxels, C = case
    x, w, b, rng = _head_inputs(voxels, C, seed)
    p = np.empty(voxels, np.float32)
    _lib.check(_lib.load().fm_op_head(ctx.handle, _lib.fptr(x), _lib.fptr(w), _lib.fptr(b), voxels, C, int(sigmoid),
                                      None, _lib.fptr(p), None, None, 0, None, None, None))
    x64 = x.astype(np.float64)
    z = x64 @ w.astype(np.float64) + float(b[0])
    dz = RED_TOL * (np.abs(x64) @ np.abs(w.astype(np.float64)) + abs(float(b[0])))
    if not sigmoid:
        return close_sum(p, z, dz / RED_TOL, 1e-7 * np.abs(z))
    ref = 1.0 / (1.0 + np.exp(-z))
    # fp32 logit within the reduction bound, then the fp32 sigmoid (fast exp: a few ulp)
    tol = ref * (1 - ref) * dz + 1e-6 * ref
    worst = float((np.abs(p - ref) / (tol + 1e-30)).max())
    return worst <= 1.0, worst


def head_fwd_dice_case(ctx, case, seed=31):
    """The training forward: p as in head_fwd_case, and the 8 statistics of its own p (fp32 per-thread sums, fp64
    fold): sums of p within the reduction bound, the counts exact."""
    name, voxels, C = case
    x, w, b, rng = _head_inputs(voxels, C, seed)
    t = (rng.random(voxels) < 0.3).astype(np.float32)
    p = np.empty(voxels, np.float32)
    sums = np.zeros(8, np.float64)
    _lib.check(_lib.load().fm_op_head(ctx.handle, _lib.fptr(x), _lib.fptr(w), _lib.fptr(b), voxels, C, 1,
                                      _lib.fptr(t), _lib.fptr(p), _lib.dptr(sums), None, 0, None, None, None))
    z = x.astype(np.float64) @ w.astype(np.float64) + float(b[0])
    ref = 1.0 / (1.0 + np.exp(-z))
    tol = ref * (1 - ref) * RED_TOL * (np.abs(x.astype(np.float64)) @ np.abs(w.astype(np.float64)) + 0.2) + 1e-6 * ref
    w0 = float((np.abs(p - ref) / (tol + 1e-30)).max())
    p64, t64 = p.astype(np.float64), t.astype(np.float64)
    pb, tb = p > 0.5, t > 0.5
    ok1, w1 = close_sum(sums[:3], [(t64 * p64).sum(), t64.sum(), p64.sum()], [(t64 * p64).sum(), t64.sum(), p64.sum()])
    counts = np.array([(tb & pb).sum(), tb.sum(), pb.sum(), (t == pb.astype(np.float32)).sum(), voxels], np.float64)
    ok2 = np.array_equal(sums[3:8], counts)
    return w0 <= 1.0 and ok1 and ok2, max(w0, w1, 0.0 if ok2 else float("inf"))


def head_bwd_case(ctx, case, mode, seed=32):
    """dx = dz * w (mode 0: masked by x > 0; mode 2: added to the incoming dx), dw = sum dz x, db = sum dz."""
    name, voxels, C = case
    x, w, b, rng = _head_inputs(voxels, C, seed)
    dz = rng.standard_normal(voxels).astype(np.float32)
    dx0 = bf16_round(rng.standard_normal((voxels, C)))
    dx = dx0.copy()
    dw = np.empty(C, np.float32)
    db = np.empty(1, np.float32)
    _lib.check(_lib.load().fm_op_head(ctx.handle, _lib.fptr(x), _lib.fptr(w), _lib.fptr(b), voxels, C, 1, None, None,
                                      None, _lib.fptr(dz), mode, _lib.fptr(dx), _lib.fptr(dw), _lib.fptr(db)))
    x64, dz64 = x.astype(np.float64), dz.astype(np.float64)
    ref = dz64[:, None] * w.astype(np.float64)[None, :]
    if mode == 0:
        ref = ref * (x > 0)
    elif mode == 2:
        ref = ref + dx0
    ok, worst = close_bf16(dx, ref)
    ok1, w1 = close_sum(dw, dz64 @ x64, np.abs(dz64) @ np.abs(x64))
    ok2, w2 = close_sum(db, [dz64.sum()], [np.abs(dz64).sum()])
    return ok and ok1 and ok2, max(worst, w1, w2)


# the 2D family (kernel code 31 on Z = 1 volumes): unet2d_layers (depth 4, 32 filters, 6 input slices padded to 16)
# and isensee2d_layers (16 filters; localisation concat [skip, up])
CONV2D_CASES = [
    ("u2d_enc0a_16_32", 2, 32, 32, 1, 16, 0, 32, 31),
    ("u2d_enc1b_64_64", 2, 16, 16, 1, 64, 0, 64, 31),
    ("u2d_enc3a_128_256", 1, 4, 4, 1, 128, 0, 256, 31),
    ("u2d_dec2a_cat256_128", 1, 8, 8, 1, 256, 128, 128, 31),
    ("u2d_dec0a_cat64_32", 2, 32, 32, 1, 64, 32, 32, 31),
    ("i2d_ctx_16_16", 2, 32, 32, 1, 16, 0, 16, 31),
    ("i2d_loc1_cat16_16", 1, 32, 32, 1, 16, 16, 16, 31),
    ("i2d_up_64_32", 1, 16, 16, 1, 64, 0, 32, 31),
    ("ragged2d_12x10", 3, 12, 10, 1, 32, 0, 64, 31),
]
