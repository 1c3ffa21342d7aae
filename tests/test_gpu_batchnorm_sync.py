"""Batch normalisation over a global batch split into shards, one stage at a time on one GPU: what every rank of a
data-parallel step does (fm_op_batchnorm_sums -> all-reduce -> fm_op_batchnorm_relu_global, and the same for the
backward). The all-reduce is emulated by adding the shards' float64 sums on the host.

- one shard: y, the moving statistics, dx, dgamma and dbeta are bit-identical to fm_op_batchnorm_relu(_bwd) on the
  same batch;
- several shards, against the float64 full-batch reference below: concat(y) and concat(dx) within the per-element bf16
  bound, the moving statistics within 1e-6 of the sum of their terms' magnitudes (and bit-identical across shards),
  dgamma / dbeta summed over the shards within 1e-5 * sum|term| per channel.
"""
import numpy as np
import pytest

from fetal_net import _lib
from tests import gpu_cases as gc

pytestmark = pytest.mark.gpu

EPS, MOMENTUM = 1e-3, 0.99
CASES = gc.NORM_CASES + [gc.NORM_BIG]
SPLITS = [None, (2, 2), (3, 1, 1), (1, 1, 1, 1, 1)]   # None: the case's own batch as one shard


def split_id(s):
    return "whole" if s is None else "+".join(map(str, s))


def _params():
    return [pytest.param(c, s, id="%s-%s" % (c[0], split_id(s))) for c in CASES for s in SPLITS
            if c is not gc.NORM_BIG or s in (None, (2, 2))]    # the 1M-voxel case: one split is enough


def bn_reference(x, gamma, beta, mm, mv, gy):
    """Keras BatchNormalization(axis=-1) + ReLU over the whole batch x [N, vox, C] in float64: y, the moving
    statistics after one training step, dx, dgamma, dbeta, and the magnitudes of the terms of each sum."""
    x = np.asarray(x, np.float64)
    C = x.shape[-1]
    n = x.size // C
    mean = x.mean((0, 1))
    var = x.var((0, 1))
    rstd = 1.0 / np.sqrt(var + EPS)
    xh = (x - mean) * rstd
    z = xh * gamma + beta
    y = np.maximum(z, 0.0)
    corr = n / (n - (1.0 + EPS))
    mm_new = mm * MOMENTUM + mean * (1 - MOMENTUM)
    mv_new = mv * MOMENTUM + var * corr * (1 - MOMENTUM)
    mm_terms = np.abs(mm) * MOMENTUM + np.abs(x).mean((0, 1)) * (1 - MOMENTUM)
    # magnitudes: the correction is negative for a single voxel (n = 1 < 1 + eps)
    mv_terms = np.abs(mv) * MOMENTUM + ((x ** 2).mean((0, 1)) + mean ** 2) * abs(corr) * (1 - MOMENTUM)
    out = dict(y=y, mm=mm_new, mv=mv_new, mm_terms=mm_terms, mv_terms=mv_terms)
    if gy is not None:
        g = np.asarray(gy, np.float64) * (z > 0)
        out.update(dbeta=g.sum((0, 1)), dgamma=(g * xh).sum((0, 1)), tb=np.abs(g).sum((0, 1)),
                   tg=np.abs(g * xh).sum((0, 1)),
                   dx=gamma * rstd * (g - g.mean((0, 1)) - xh * (g * xh).mean((0, 1))))
    return out


def shards(a, sizes):
    bounds = np.cumsum([0] + list(sizes))
    return [np.ascontiguousarray(a[lo:hi]) for lo, hi in zip(bounds[:-1], bounds[1:])]


def split_forward(ctx, xs, gamma, beta, mm, mv):
    """Per shard (y, moving_mean, moving_var, stats) with the global forward sums."""
    lib = _lib.load()
    vox, C = xs[0].shape[1:]
    total = np.zeros(2 * C + 1)
    for x in xs:
        s = np.empty(2 * C + 1)
        _lib.check(lib.fm_op_batchnorm_sums(ctx.handle, _lib.fptr(x), len(x), vox, C, _lib.dptr(s)))
        assert s[2 * C] == len(x) * vox
        total = total + s
    out = []
    for x in xs:
        y = np.empty(x.shape, np.float32)
        m, v = mm.copy(), mv.copy()
        st = np.empty((C, 2), np.float32)
        _lib.check(lib.fm_op_batchnorm_relu_global(ctx.handle, _lib.fptr(x), _lib.fptr(gamma), _lib.fptr(beta),
                                                   _lib.fptr(m), _lib.fptr(v), len(x), vox, C, _lib.dptr(total),
                                                   _lib.fptr(y), _lib.fptr(st)))
        out.append((y, m, v, st))
    return out


def split_backward(ctx, xs, gys, stats, gamma, beta):
    """Per shard (dx, dgamma, dbeta) with the global backward sums."""
    lib = _lib.load()
    vox, C = xs[0].shape[1:]
    total = np.zeros(2 * C + 1)
    local = []
    for x, gy in zip(xs, gys):
        s = np.empty(2 * C + 1)
        dg, db = np.empty(C, np.float32), np.empty(C, np.float32)
        _lib.check(lib.fm_op_batchnorm_bwd_sums(ctx.handle, _lib.fptr(x), _lib.fptr(stats), _lib.fptr(gamma),
                                                _lib.fptr(beta), _lib.fptr(gy), None, len(x), vox, C, _lib.dptr(s),
                                                _lib.fptr(dg), _lib.fptr(db)))
        total = total + s
        local.append((dg, db))
    out = []
    for (x, gy), (dg, db) in zip(zip(xs, gys), local):
        dx = np.empty(x.shape, np.float32)
        _lib.check(lib.fm_op_batchnorm_relu_bwd_global(ctx.handle, _lib.fptr(x), _lib.fptr(stats), _lib.fptr(gamma),
                                                       _lib.fptr(beta), _lib.fptr(gy), None, len(x), vox, C,
                                                       _lib.dptr(total), _lib.fptr(dx)))
        out.append((dx, dg, db))
    return out


def inputs(case, split, seed):
    name, N, vox, C = case
    if split is not None:
        N = sum(split)
    x, gamma, beta, rng = gc.norm_inputs(N, vox, C, seed)
    x = x.astype(np.float32)
    mm = (0.5 * rng.standard_normal(C)).astype(np.float32)
    mv = (0.5 + rng.random(C)).astype(np.float32)
    gy = gc.bf16_round(rng.standard_normal((N, vox, C))).astype(np.float32)
    return x, gamma, beta, mm, mv, gy, [N] if split is None else list(split)


@pytest.mark.parametrize("case,split", _params())
def test_batchnorm_global_forward(ctx, case, split):
    x, gamma, beta, mm, mv, _, sizes = inputs(case, split, seed=40)
    res = split_forward(ctx, shards(x, sizes), gamma, beta, mm, mv)
    for _, m, v, st in res[1:]:      # every rank computes the same statistics and moving averages
        assert np.array_equal(m, res[0][1]) and np.array_equal(v, res[0][2]) and np.array_equal(st, res[0][3])
    y = np.concatenate([r[0] for r in res])
    m, v = res[0][1], res[0][2]
    if len(sizes) == 1:
        y1, m1, v1 = np.empty_like(x), mm.copy(), mv.copy()
        _lib.check(_lib.load().fm_op_batchnorm_relu(ctx.handle, 1, _lib.fptr(x), _lib.fptr(gamma), _lib.fptr(beta),
                                                    _lib.fptr(m1), _lib.fptr(v1), len(x), x.shape[1], x.shape[2],
                                                    _lib.fptr(y1)))
        assert np.array_equal(y, y1) and np.array_equal(m, m1) and np.array_equal(v, v1)
    ref = bn_reference(x, gamma, beta, mm, mv, None)
    ok, worst = gc.close_bf16_per_channel(y, ref["y"])
    ok1 = np.all(np.abs(m - ref["mm"]) <= 1e-6 * ref["mm_terms"])
    ok2 = np.all(np.abs(v - ref["mv"]) <= 1e-6 * ref["mv_terms"])
    assert ok and ok1 and ok2, (worst, float(np.max(np.abs(m - ref["mm"]) / ref["mm_terms"])),
                                float(np.max(np.abs(v - ref["mv"]) / ref["mv_terms"])))


@pytest.mark.parametrize("case,split", _params())
def test_batchnorm_global_backward(ctx, case, split):
    x, gamma, beta, mm, mv, gy, sizes = inputs(case, split, seed=41)
    xs, gys = shards(x, sizes), shards(gy, sizes)
    stats = split_forward(ctx, xs, gamma, beta, mm, mv)[0][3]
    res = split_backward(ctx, xs, gys, stats, gamma, beta)
    dx = np.concatenate([r[0] for r in res])
    dg = np.sum([r[1].astype(np.float64) for r in res], 0)
    db = np.sum([r[2].astype(np.float64) for r in res], 0)
    if len(sizes) == 1:
        dx1, dg1, db1 = np.empty_like(x), np.empty_like(gamma), np.empty_like(beta)
        _lib.check(_lib.load().fm_op_batchnorm_relu_bwd(ctx.handle, _lib.fptr(x), _lib.fptr(gamma), _lib.fptr(beta),
                                                        _lib.fptr(gy), None, len(x), x.shape[1], x.shape[2],
                                                        _lib.fptr(dx1), _lib.fptr(dg1), _lib.fptr(db1)))
        assert np.array_equal(dx, dx1) and np.array_equal(res[0][1], dg1) and np.array_equal(res[0][2], db1)
    ref = bn_reference(x, gamma, beta, mm, mv, gy)
    ok, worst = gc.close_bf16_per_channel(dx, ref["dx"])
    ok1, w1 = gc.close_sum(dg, ref["dgamma"], ref["tg"])
    ok2, w2 = gc.close_sum(db, ref["dbeta"], ref["tb"])
    assert ok and ok1 and ok2, (worst, w1, w2)
