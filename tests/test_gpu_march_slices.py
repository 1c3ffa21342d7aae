"""The marching fprop / dgrad on layers whose filter bank only fits in shared memory as 32-wide Cout slices (64 -> 64 and
64 -> 128 convolutions: dec1b, enc2a, enc2b of the U-Net): parity with the float64 reference (tolerance of
tests/gpu_cases.py), bit-reproducibility of the ordered issue mode, and the output of single-slice layers pinned to
what they computed before slicing existed."""
import hashlib

import numpy as np
import pytest
import torch.nn.functional as F

from fetal_net import _lib
from tests import gpu_cases as gc

pytestmark = pytest.mark.gpu

# name, N, X, Y, Z, C1, C2, Cout, k
SLICED_FPROP = [
    ("s64_64_32cube", 1, 32, 32, 32, 64, 0, 64, 3),      # dec1b: 2 slices
    ("s64_128_32cube", 1, 32, 32, 32, 64, 0, 128, 3),    # 4 slices
    ("s64_64_16x32x64", 2, 16, 32, 64, 64, 0, 64, 3),    # 16 x 8 columns in y and z
    ("s64_64_16cube", 4, 16, 16, 16, 64, 0, 64, 3),      # enc2a
    ("s64_128_16cube", 4, 16, 16, 16, 64, 0, 128, 3),    # enc2b
    # two sources: a 64 + 64 -> 64 slice (221 KB) leaves no room for the slab rings, so 64 + 32 and 32 + 32
    ("s_cat64_32_to64", 1, 32, 32, 32, 64, 32, 64, 3),
    ("s_cat32_32_to64", 1, 32, 32, 32, 32, 32, 64, 3),
    ("s_oddx_37x32x32", 1, 37, 32, 32, 64, 0, 64, 3),    # X not a multiple of the x-chunk
]
# dgrad: dY has Cout channels, dX has C1
SLICED_DGRAD = [
    ("d64_64_32cube", 1, 32, 32, 32, 64, 0, 64, 3),
    ("d128_from64_32cube", 1, 32, 32, 32, 128, 0, 64, 3),  # 4 slices of dX
    ("d64_64_16cube", 4, 16, 16, 16, 64, 0, 64, 3),      # enc2a
    ("d_oddx_10x16x8", 3, 10, 16, 8, 64, 0, 64, 3),      # X not a multiple of the x-chunk, few planes per CTA
    ("d_oddx_37x32x32", 1, 37, 32, 32, 64, 0, 64, 3),
]


def ids(cases):
    return [c[0] for c in cases]


def dgrad_run(ctx, impl, case, masked, seed=1):
    name, N, X, Y, Z, Cin, _, Cout, k = case
    rng = np.random.default_rng(seed)
    dy = gc.bf16_round(rng.standard_normal((N, X, Y, Z, Cout)))
    w = gc.bf16_round(rng.standard_normal((3, 3, 3, Cin, Cout)) / np.sqrt(27 * Cout))
    act = gc.bf16_round(rng.standard_normal((N, X, Y, Z, Cin))) if masked else None
    dx = np.empty((N, X, Y, Z, Cin), np.float32)
    lib = _lib.load()
    _lib.check(lib.fm_op_conv_dgrad(ctx.handle, impl, _lib.fptr(dy), _lib.fptr(w), _lib.fptr(act), N, X, Y, Z, Cin,
                                    Cout, k, _lib.fptr(dx)))
    return dx, dy, w, act


@pytest.mark.parametrize("impl", [2, 3], ids=["reproducible", "shared-acc"])
@pytest.mark.parametrize("case", SLICED_FPROP, ids=ids(SLICED_FPROP))
def test_sliced_fprop(ctx, case, impl):
    ok, worst = gc.conv_fprop_case(ctx, impl, case)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", SLICED_FPROP[:2] + SLICED_FPROP[3:4], ids=ids(SLICED_FPROP[:2] + SLICED_FPROP[3:4]))
def test_sliced_fprop_no_relu(ctx, case):
    ok, worst = gc.conv_fprop_case(ctx, 2, case, relu=0)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("masked", [True, False], ids=["mask", "no-mask"])
@pytest.mark.parametrize("impl", [2, 3], ids=["reproducible", "shared-acc"])
@pytest.mark.parametrize("case", SLICED_DGRAD, ids=ids(SLICED_DGRAD))
def test_sliced_dgrad(ctx, case, impl, masked):
    dx, dy, w, act = dgrad_run(ctx, impl, case, masked)
    ref = gc.cf_to_cl(F.conv_transpose3d(gc.cl_to_cf(dy).double(), gc.keras_to_torch_w(w).double(), padding=1))
    if masked:
        ref = ref * (act > 0)
    ok, worst = gc.close_bf16(dx, ref)
    assert ok, "worst error / tolerance = %.3f" % worst


@pytest.mark.parametrize("case", SLICED_FPROP, ids=ids(SLICED_FPROP))
def test_sliced_fprop_bit_reproducible(ctx, case):
    first = gc.conv_fprop_raw(ctx, 2, case)
    for _ in range(2):
        assert np.array_equal(gc.conv_fprop_raw(ctx, 2, case), first)


@pytest.mark.parametrize("case", SLICED_DGRAD, ids=ids(SLICED_DGRAD))
def test_sliced_dgrad_bit_reproducible(ctx, case):
    first = dgrad_run(ctx, 2, case, True)[0]
    for _ in range(2):
        assert np.array_equal(dgrad_run(ctx, 2, case, True)[0], first)


# Layers whose whole bank fits run as one slice with the pack layout they always had: their ordered-issue outputs are
# pinned (sha-256 of the float32 output bytes) to those of the library before Cout slices existed.
SINGLE_SLICE_PINS = [
    # two sources 64 + 32 -> 32 (K chunks of 64 and 32)
    ("fprop", gc.MARCH_CASES[4], "adcf052522ecfc9e738a35af1dc0a91ea21a46a69e09cb3f6291e22cb9b7cdae"),
    # 32 -> 64 (the Cout = 64 issue mode)
    ("fprop", gc.MARCH_CASES[2], "bf7ee76367014c774f3d34d2931480a4f207ebe45a6c073f07fdd85274c3fdaf"),
    # dY 64 -> dX 32, masked, K chunks of 64
    ("dgrad", ("p64_to32", 2, 16, 32, 16, 32, 0, 64, 3),
     "ca7d88bb5f56d7d77c20f96ccc9be8a625e6d7eac1356ea837b83810b587c689"),
]


@pytest.mark.parametrize("kind,case,digest", SINGLE_SLICE_PINS, ids=[p[1][0] for p in SINGLE_SLICE_PINS])
def test_single_slice_output_unchanged(ctx, kind, case, digest):
    out = gc.conv_fprop_raw(ctx, 2, case) if kind == "fprop" else dgrad_run(ctx, 2, case, True)[0]
    assert hashlib.sha256(np.ascontiguousarray(out, np.float32).tobytes()).hexdigest() == digest
