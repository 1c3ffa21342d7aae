"""Pins the oracle (oracle/prediction_oracle.py) against (a) the goldens frozen from the unmodified
reference code and (b) the reference itself where /root/reference is present (build container only).
Also pins the closed forms of the network oracle (dice, Adam) against independent derivations."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import prediction_oracle as po
from oracle import unet_oracle as uo
from oracle.ref_harness import FunctionModel, reference_available

from tests.golden.make_golden import ramp_model, ramp_model_2d


def sha16(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def plan_names(golden):
    return sorted({k.split("/")[1] for k in golden if k.startswith("plan/")})


def run_names(golden):
    return sorted({k.split("/")[1] for k in golden if k.startswith("run/")})


def test_plans_match_golden(golden):
    for name in plan_names(golden):
        a = golden["plan/%s/args" % name]
        padded, patch, pshape = tuple(a[0:3]), tuple(a[3:6]), tuple(a[6:9])
        idx = po.patch_plan(padded, patch, pshape, float(golden["plan/%s/f" % name]))
        assert len(idx) == int(golden["plan/%s/n" % name]), name
        assert sha16(idx.astype(np.int32)) == str(golden["plan/%s/sha" % name]), name
        if "plan/%s/idx" % name in golden:
            assert np.array_equal(idx, golden["plan/%s/idx" % name]), name


def test_survey_known_answers(golden):
    # SURVEY.md §8c goldens (4) and (5)
    idx = po.patch_plan((256, 256, 64), (64, 64, 64), (64, 64, 64), 0.5)
    assert idx[:9].tolist() == [[0, 0, 0], [0, 33, 0], [0, 66, 0], [0, 99, 0], [0, 132, 0], [0, 165, 0],
                                [0, 192, 0], [33, 0, 0], [33, 33, 0]]
    assert len(idx) == 49
    cnt = po.count_map((256, 256, 64), (64, 64, 64), idx)
    assert sha16(cnt) == "ba96762db2430b62" == str(golden["count/cfg1/sha"])
    hist = dict(zip(*[v.tolist() for v in golden["count/cfg1/hist"]]))
    assert hist == {1: 295936, 2: 1601536, 3: 34816, 4: 2166784, 6: 94208, 9: 1024}
    assert int(cnt.astype(np.int64).sum()) == 49 * 64 ** 3
    assert np.array_equal(cnt[:, 0, 0], golden["count/cfg1/axis_x"])


def test_patchwise_oracle_matches_golden(golden):
    for name in run_names(golden):
        vol = golden["run/%s/vol" % name]
        patch = tuple(int(v) for v in golden["run/%s/patch" % name])
        fn, oshape = ramp_model(patch, int(golden["run/%s/channels" % name]))
        out = po.patch_wise_prediction(FunctionModel(fn, oshape), vol, patch,
                                       overlap_factor=float(golden["run/%s/f" % name]),
                                       batch_size=int(golden["run/%s/batch" % name]))
        ref = golden["run/%s/out" % name]
        assert out.dtype == np.float64 and out.shape == ref.shape, name
        assert np.array_equal(out, ref), name      # bit-exact


def test_patchwise_oracle_2d_and_truth_conditioning_matches_golden(golden):
    names = sorted({k.split("/")[1] for k in golden if k.startswith("run2d/")})
    assert len(names) == 4
    for name in names:
        vol = golden["run2d/%s/vol" % name]
        patch = tuple(int(v) for v in golden["run2d/%s/patch" % name])
        pti, pts = [int(v) for v in golden["run2d/%s/prev" % name]]
        truth = golden.get("run2d/%s/truth" % name)
        fn, oshape = ramp_model_2d(patch[:2], patch[2] + pts)
        out = po.patch_wise_prediction(FunctionModel(fn, oshape), vol, patch,
                                       overlap_factor=float(golden["run2d/%s/f" % name]),
                                       batch_size=int(golden["run2d/%s/batch" % name]), truth_data=truth,
                                       prev_truth_index=pti if truth is not None else None,
                                       prev_truth_size=pts if truth is not None else None)
        assert np.array_equal(out, golden["run2d/%s/out" % name]), name


def test_extract_patch_matches_golden(golden):
    data = golden["patch/data"]
    shape = tuple(int(v) for v in golden["patch/shape"])
    for i, c in enumerate(golden["patch/corners"]):
        assert np.array_equal(po.extract_patch(data, shape, c), golden["patch/out%d" % i]), i


@pytest.mark.skipif(not reference_available(), reason="reference tree only exists in the build container")
def test_oracle_matches_live_reference():
    from oracle.ref_harness import load_reference_prediction
    pred = load_reference_prediction()
    rng = np.random.default_rng(3)
    for vshape, patch, f, bs in [((1, 33, 20, 18), (16, 8, 8), 0.5, 5), ((1, 10, 30, 9), (16, 16, 8), 0.7, 2)]:
        vol = rng.standard_normal(vshape).astype(np.float32)
        fn, oshape = ramp_model(patch, 1)
        ref = pred.patch_wise_prediction(FunctionModel(fn, oshape), vol, patch_shape=patch, overlap_factor=f,
                                         batch_size=bs)
        out = po.patch_wise_prediction(FunctionModel(fn, oshape), vol, patch, overlap_factor=f, batch_size=bs)
        assert np.array_equal(out, ref)


def test_oracle_identity_model_returns_the_volume():
    # identity-model goldens of SURVEY.md §8c (1)-(2)
    for vshape in [(1, 96, 80, 40), (1, 70, 70, 20)]:
        vol = np.random.default_rng(0).standard_normal(vshape).astype(np.float32)
        m = FunctionModel(lambda x: x.astype(np.float32), (None, 1, 32, 32, 32))
        out = po.patch_wise_prediction(m, vol, (32, 32, 32), overlap_factor=0.5)
        assert np.array_equal(out[..., 0], vol[0])


# ---- network oracle: closed forms ------------------------------------------------------------

def test_dice_known_answers():
    # the test_metrics tensor of the reference (test/test_metrics.py:13-17): a 3-channel block pattern
    d = np.zeros((1, 3, 10, 10, 10), np.float32)
    d[0, 0, :5] = 1
    d[0, 1, 5:] = 1
    d[0, 2, :, :5] = 1
    t = torch.tensor(d)
    assert float(uo.dice_coefficient(t, t)) == pytest.approx(1.0)
    assert float(uo.dice_coefficient(t, torch.zeros_like(t))) == pytest.approx(1.0 / (d.sum() + 1.0))
    assert float(uo.dice_coefficient(torch.zeros_like(t), torch.zeros_like(t))) == pytest.approx(1.0)


def test_dice_closed_form_gradient_matches_autograd():
    g = torch.Generator().manual_seed(0)
    p = torch.rand(2, 1, 6, 5, 4, generator=g, dtype=torch.float64, requires_grad=True)
    t = (torch.rand(2, 1, 6, 5, 4, generator=g) < 0.3).double()
    uo.dice_coefficient_loss(t, p).backward()
    assert torch.allclose(p.grad, uo.dice_grad_closed_form(t, p.detach()), rtol=1e-12, atol=1e-14)


def test_keras_adam_first_steps():
    # Keras-2 Adam, step 1: m = (1-b1) g, v = (1-b2) g^2, lr_t = lr*sqrt(1-b2)/(1-b1)
    p = np.array([1.0, -2.0], np.float32)
    g = np.array([0.5, -0.25], np.float32)
    m, v = np.zeros(2, np.float32), np.zeros(2, np.float32)
    uo.keras_adam_step(p, g, m, v, 0, 1e-3)
    lr_t = 1e-3 * np.sqrt(1 - 0.999) / (1 - 0.9)
    exp = np.array([1.0, -2.0]) - lr_t * (0.1 * g) / (np.sqrt(0.001 * g * g) + 1e-7)
    assert np.allclose(p, exp, rtol=1e-6)


def test_param_counts_match_survey():
    # SURVEY.md §8a: 4 079 713 / 16 315 585 / 8 263 619 / 5 441 569
    n = lambda L: sum(k ** (3 if len(L[0]) and True else 3) * ci * co + co for _, ci, co, k in L)
    assert n(uo.unet3d_layers(4, 16)) == 4079713
    assert n(uo.unet3d_layers(4, 32)) == 16315585
    assert n(uo.isensee3d_layers(5, 16, 3)) == 8263619
    assert sum(k ** 2 * ci * co + co for _, ci, co, k in uo.unet2d_layers(4, 32, 6)) == 5441569


def test_instance_norm_backward_closed_form_matches_autograd():
    """The closed form behind the instnorm_bwd_* kernels (eps on the STD, LeakyReLU slope and dropout scale folded in)
    equals autograd through the oracle's own forward restatement (keras_contrib InstanceNormalization semantics)."""
    import torch
    import torch.nn.functional as F
    from oracle import unet_oracle as uo
    rng = np.random.default_rng(5)
    N, C = 2, 8
    x = rng.standard_normal((N, C, 6, 5, 4))
    x[:, 3] *= 1e-3                                   # a low-variance channel: eps / sigma is not negligible there
    gy = rng.standard_normal(x.shape)
    gamma = 1.0 + 0.3 * rng.standard_normal(C)
    beta = 0.2 * rng.standard_normal(C)
    cs = (rng.random((N, C)) > 0.3) / 0.7
    xt = torch.tensor(x, requires_grad=True)
    gt = torch.tensor(gamma, requires_grad=True)
    bt = torch.tensor(beta, requires_grad=True)
    y = F.leaky_relu(uo._instance_norm(xt, gt, bt), 0.3) * torch.tensor(cs).reshape(N, C, 1, 1, 1)
    y.backward(torch.tensor(gy))
    dx, dg, db = uo.instance_norm_lrelu_backward_closed_form(x, gy, gamma, beta, chan_scale=cs)
    np.testing.assert_allclose(dx, xt.grad.numpy(), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(dg, gt.grad.numpy(), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(db, bt.grad.numpy(), rtol=1e-9, atol=1e-10)


def test_strided_conv_backward_as_zero_inserted_stride1_backward():
    """The identity behind the Isensee stride-2 backward (csrc/api.cu backward_isensee, k_zero_insert): for
    y = conv3d(pad(x, after=1), w, stride=2) (TF 'SAME', even extents, k = 3), placing dy[v] at the ODD fine position
    2v + 1 of an otherwise zero tensor dz makes the stride-1 'same' dgrad / wgrad of dz equal the strided conv's own
    gradients:  dx[u] = sum_t w[t]^T dz[u + 1 - t],   dw[t] = sum_u x[u + t - 1] dz[u]."""
    import torch
    import torch.nn.functional as F
    torch.manual_seed(0)
    x = torch.randn(2, 3, 8, 6, 4, dtype=torch.float64, requires_grad=True)
    w = torch.randn(5, 3, 3, 3, 3, dtype=torch.float64, requires_grad=True)
    y = F.conv3d(F.pad(x, (0, 1, 0, 1, 0, 1)), w, stride=2)
    dy = torch.randn_like(y)
    y.backward(dy)
    dz = torch.zeros(2, 5, 8, 6, 4, dtype=torch.float64)
    dz[:, :, 1::2, 1::2, 1::2] = dy
    # stride-1 'same' conv z = conv3d(x, w, padding=1) has dgrad = conv_transpose and wgrad = correlation with x
    xs = x.detach().clone().requires_grad_(True)
    ws = w.detach().clone().requires_grad_(True)
    F.conv3d(xs, ws, padding=1).backward(dz)
    np.testing.assert_allclose(xs.grad.numpy(), x.grad.numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(ws.grad.numpy(), w.grad.numpy(), rtol=1e-12, atol=1e-12)


def test_upsampled_source_conv_equals_parity_class_convs_at_coarse_resolution():
    """3x3x3 'same' conv over UpSampling3D(2)(x) == eight 2x2x2-support convs over x, one per output parity class
    (oracle.unet_oracle.upsampled_conv_parity_weights) - 8 x 8 = 64 tap-voxel products per coarse voxel instead of
    8 x 27 = 216. Exact in float64, borders included."""
    import torch
    import torch.nn.functional as F
    from oracle import unet_oracle as uo
    torch.manual_seed(1)
    x = torch.randn(2, 4, 5, 3, 4, dtype=torch.float64)
    w = torch.randn(6, 4, 3, 3, 3, dtype=torch.float64)
    up = x.repeat_interleave(2, 2).repeat_interleave(2, 3).repeat_interleave(2, 4)
    ref = F.conv3d(up, w, padding=1)
    wc = uo.upsampled_conv_parity_weights(w.numpy())
    out = torch.zeros_like(ref)
    nonzero = 0
    for px in range(2):
        for py in range(2):
            for pz in range(2):
                k = torch.as_tensor(wc[px, py, pz])
                nonzero += int((k.abs().sum(dim=(0, 1)) > 0).sum())
                out[:, :, px::2, py::2, pz::2] = F.conv3d(x, k, padding=1)
    assert nonzero == 64
    np.testing.assert_allclose(out.numpy(), ref.numpy(), rtol=1e-12, atol=1e-12)


# ----------------------------------------------------------------------------------------------
# the pin against REAL Keras: tools/export_keras_fixture.py writes tests/golden/keras_fixture.npz
# where Keras/TensorFlow exist (not in this image). The reader is exercised on a synthetic file.
# ----------------------------------------------------------------------------------------------
KERAS_CASES = {
    "unet3d_d4_nf16": dict(layers=lambda: uo.unet3d_layers(4, 16), fwd=lambda x, w: uo.unet3d_forward(x, w, depth=4)),
    "isensee3d_d3_nf8_seg2": dict(layers=lambda: uo.isensee3d_layers(3, 8, 2),
                                  fwd=lambda x, w: uo.isensee3d_forward(x, w, depth=3, n_segmentation_levels=2)),
    "unet2d_d3_nf16": dict(layers=lambda: uo.unet2d_layers(3, 16, 6), fwd=lambda x, w: uo.unet2d_forward(x, w, depth=3)),
}


def test_keras_fixture_reader_on_synthetic_file():
    """Keras-style variable names, numbered from an arbitrary session offset and listed in graph-depth order (the
    coarse segmentation head AFTER later-created decoder layers), must map back onto the oracle's layer table."""
    from oracle import keras_fixture as kf
    layers = uo.isensee3d_layers(3, 8, 2)
    w = uo.glorot_uniform_weights(layers, seed=3)
    w.update({k: v + 0.25 for k, v in uo.isensee3d_norm_params(layers).items()})
    z, names, ci, ni = {}, [], 40, 17
    for lname, cin, cout, k in layers:
        ci += 1
        names += ["conv3d_%d/kernel:0" % ci, "conv3d_%d/bias:0" % ci]
        z["t/w/conv3d_%d/kernel:0" % ci], z["t/w/conv3d_%d/bias:0" % ci] = w[lname + "/kernel"], w[lname + "/bias"]
        if not lname.endswith("_seg"):
            ni += 1
            names += ["instance_normalization_%d/gamma:0" % ni, "instance_normalization_%d/beta:0" % ni]
            z["t/w/instance_normalization_%d/gamma:0" % ni] = w[lname + "/gamma"]
            z["t/w/instance_normalization_%d/beta:0" % ni] = w[lname + "/beta"]
    rng = np.random.default_rng(0)
    z["t/names"] = np.array([names[i] for i in rng.permutation(len(names))])
    got = kf.named_weights(z, "t", layers)
    assert set(got) == set(w)
    for k in w:
        assert np.array_equal(got[k], w[k]), k


@pytest.mark.parametrize("tag", sorted(KERAS_CASES))
def test_oracle_matches_keras_fixture(tag):
    """The network oracle against real Keras output (predict, loss of one train_on_batch, the Adam-updated weights).
    Tolerances: both sides are fp32 on a CPU with different summation orders -> 2e-4 on probabilities, 1e-5 on the
    loss, 2e-6 on the updated weights (one Adam step moves every weight by ~lr)."""
    from oracle import keras_fixture as kf
    z = kf.load()
    if z is None or tag + "/names" not in z.files:
        pytest.skip("tests/golden/keras_fixture.npz absent (needs Keras/TF: tools/export_keras_fixture.py)")
    case = KERAS_CASES[tag]
    layers = case["layers"]()
    w = kf.named_weights(z, tag, layers)
    x, t = z[tag + "/x"], z[tag + "/t"]
    with torch.no_grad():
        p = case["fwd"](torch.as_tensor(x), w).numpy()
    assert np.abs(p - z[tag + "/predict"]).max() <= 2e-4
    res = uo.train_step(case["fwd"], x, t, w, {}, float(z[tag + "/lr"]))
    assert abs(res["loss"] - float(z[tag + "/train_metrics"][0])) <= 1e-5
    after = kf.named_weights(z, tag, layers, which="w_after")
    for k in w:
        assert np.abs(w[k] - after[k]).max() <= 2e-6, k


# ----------------------------------------------------------------------------------------------
# independent cross-checks of the network oracle's building blocks (explicit NumPy loops, no torch)
# ----------------------------------------------------------------------------------------------
def _naive_conv3d_same(x, kern, bias):
    """Keras Conv3D(padding='same', strides 1) on channels-first x [C,X,Y,Z] with kernel (k0,k1,k2,Cin,Cout):
    y[co, p] = b[co] + sum_{t, ci} x[ci, p + t - 1] * kern[t0, t1, t2, ci, co] (cross-correlation, zero padding)."""
    C, X, Y, Z = x.shape
    k = kern.shape[0]
    r = k // 2
    xp = np.zeros((C, X + 2 * r, Y + 2 * r, Z + 2 * r))
    xp[:, r:r + X, r:r + Y, r:r + Z] = x
    y = np.zeros((kern.shape[-1], X, Y, Z))
    for a in range(k):
        for b in range(k):
            for c in range(k):
                y += np.einsum("cxyz,co->oxyz", xp[:, a:a + X, b:b + Y, c:c + Z], kern[a, b, c])
    return y + bias[:, None, None, None]


def test_unet3d_forward_matches_explicit_numpy_on_a_tiny_network():
    """depth-2 U-Net on a 4x4x2 volume: conv 'same' with the Keras kernel layout, ReLU, 2^3 max-pool, nearest upsampling,
    concat order [up, skip] (unet3d/unet.py:61), 1x1x1 head + sigmoid - written out with NumPy loops."""
    layers = uo.unet3d_layers(2, 2)
    w = uo.glorot_uniform_weights(layers, seed=3)
    rng = np.random.default_rng(4)
    for k_ in w:
        if k_.endswith("/bias"):
            w[k_] = rng.standard_normal(w[k_].shape).astype(np.float32) * 0.1
    x = rng.standard_normal((1, 1, 4, 4, 2))
    relu = lambda a: np.maximum(a, 0)
    cb = lambda a, name: relu(_naive_conv3d_same(a, w[name + "/kernel"].astype(np.float64), w[name + "/bias"].astype(np.float64)))
    e0 = cb(cb(x[0], "enc0a"), "enc0b")
    pooled = e0.reshape(e0.shape[0], 2, 2, 2, 2, 1, 2).max(axis=(2, 4, 6))
    e1 = cb(cb(pooled, "enc1a"), "enc1b")
    up = e1.repeat(2, 1).repeat(2, 2).repeat(2, 3)
    d0 = cb(cb(np.concatenate([up, e0], axis=0), "dec0a"), "dec0b")
    logits = np.einsum("cxyz,co->oxyz", d0, w["final/kernel"][0, 0, 0].astype(np.float64)) + w["final/bias"].astype(np.float64)[:, None, None, None]
    want = 1 / (1 + np.exp(-logits))
    with torch.no_grad():
        got = uo.unet3d_forward(torch.as_tensor(x), w, depth=2).numpy()[0]
    assert np.abs(got - want).max() <= 1e-10


def test_deconvolution_and_batch_norm_blocks_match_explicit_numpy():
    """Deconvolution3D(kernel 2, strides 2) with the Keras Conv3DTranspose kernel (2,2,2,Cout,Cin):
    y[co, 2i+a, 2j+b, 2k+c] = bias[co] + sum_ci x[ci,i,j,k] K[a,b,c,co,ci]; BatchNormalization(axis=1) in training mode:
    biased batch variance, eps 1e-3 under the root, moving statistics with momentum 0.99 and Keras' sample-size factor."""
    rng = np.random.default_rng(5)
    C = 3
    x = rng.standard_normal((2, C, 2, 3, 2))
    kern = rng.standard_normal((2, 2, 2, C, C))
    bias = rng.standard_normal(C)
    want = np.zeros((2, C, 4, 6, 4))
    for a in range(2):
        for b in range(2):
            for c in range(2):
                want[:, :, a::2, b::2, c::2] = np.einsum("ncxyz,oc->noxyz", x, kern[a, b, c])
    want += bias[None, :, None, None, None]
    layers = [("enc0a", 1, C, 3)]      # (only the 'up0' entries below are read)
    w = {"up0/kernel": kern, "up0/bias": bias}
    kt = torch.as_tensor(kern).permute(4, 3, 0, 1, 2).contiguous()
    got = torch.nn.functional.conv_transpose3d(torch.as_tensor(x), kt, torch.as_tensor(bias), stride=2).numpy()
    assert np.abs(got - want).max() <= 1e-12 and layers and w             # the permutation unet3d_forward applies
    # batch norm
    y = torch.as_tensor(rng.standard_normal((3, 2, 4, 2, 2)) * 2 + 1)
    wb = {"b/gamma": np.array([1.5, 0.5]), "b/beta": np.array([0.1, -0.2]), "b/moving_mean": np.array([0.3, 0.0]),
          "b/moving_variance": np.array([2.0, 1.0])}
    upd = {}
    out = uo._batch_norm(y, wb, "b", True, upd).numpy()
    yn = y.numpy()
    mean = yn.mean(axis=(0, 2, 3, 4))
    var = yn.var(axis=(0, 2, 3, 4))
    ref = (yn - mean[None, :, None, None, None]) / np.sqrt(var + 1e-3)[None, :, None, None, None] * \
        wb["b/gamma"][None, :, None, None, None] + wb["b/beta"][None, :, None, None, None]
    assert np.abs(out - ref).max() <= 1e-12
    n = yn.size // 2
    assert np.allclose(upd["b/moving_mean"], 0.99 * wb["b/moving_mean"] + 0.01 * mean, rtol=0, atol=1e-12)
    assert np.allclose(upd["b/moving_variance"], 0.99 * wb["b/moving_variance"] + 0.01 * var * n / (n - 1.001), rtol=0, atol=1e-12)
    inf = uo._batch_norm(y, wb, "b", False, None).numpy()
    ref_inf = (yn - wb["b/moving_mean"][None, :, None, None, None]) / np.sqrt(wb["b/moving_variance"] + 1e-3)[None, :, None, None, None] * \
        wb["b/gamma"][None, :, None, None, None] + wb["b/beta"][None, :, None, None, None]
    assert np.abs(inf - ref_inf).max() <= 1e-12
