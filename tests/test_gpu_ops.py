"""Op-level parity of the HBM-bound kernels (norm, pool, ReLU, stem/logits convs, losses, masks,
counts, optimizer) against the numpy oracle, through the C ABI."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from boxsegliver_b200.device import bf16_bits_to_f32, f32_to_bf16_bits, round_bf16
from oracle import tf_ops as O
from tests.gpu_util import TOL_BF16, bf16_randn, padded, rel

pytestmark = pytest.mark.gpu


def _norm_forward(ctx, mode, n, h, w, c, relu, is_training, pool, x_ld=None, y_ld=None, seed=0):
    rng = np.random.default_rng(seed)
    x_ld, y_ld = x_ld or c, y_ld or c
    y = bf16_randn(rng, (n, h, w, c), 1.3) + round_bf16(rng.standard_normal(c).astype(np.float32))
    y = round_bf16(y)
    gamma = rng.uniform(0.5, 1.5, c).astype(np.float32)
    beta = rng.normal(0, 0.3, c).astype(np.float32)
    mm = rng.normal(0, 0.2, c).astype(np.float32)
    mv = rng.uniform(0.5, 1.5, c).astype(np.float32)
    groups = n if mode else 1
    eps = 1e-6 if mode else 1e-3
    d = _lib.NormDesc(mode, n, h * w, c, x_ld, y_ld, eps, 0.999, relu, 1, 1)
    dev = dict(y=ctx.bf16_from_f32(padded(y, x_ld)), gamma=ctx.from_numpy(gamma), beta=ctx.from_numpy(beta),
               mm=ctx.from_numpy(mm), mv=ctx.from_numpy(mv), sums=ctx.alloc(groups * c * 16),
               a=ctx.alloc(n * h * w * y_ld * 2).zero(), pooled=ctx.alloc(max(n * h * w * c // 2, 16)).zero())
    for k in ("mean", "rstd", "scale", "shift", "c1", "c2"):
        dev[k] = ctx.alloc(groups * c * 4)
    if mode == 1 or is_training:
        ctx.call("bsl_norm_stats", C.byref(d), dev["y"].p, dev["sums"].p, ctx.stream)
    ctx.call("bsl_norm_finalize", C.byref(d), C.c_int(is_training), dev["sums"].p, dev["gamma"].p, dev["beta"].p,
             dev["mm"].p if mode == 0 else None, dev["mv"].p if mode == 0 else None, dev["mean"].p, dev["rstd"].p,
             dev["scale"].p, dev["shift"].p, ctx.stream)
    if pool:
        ctx.call("bsl_norm_apply_pool", C.byref(d), C.c_int(h), C.c_int(w), dev["y"].p, dev["scale"].p, dev["shift"].p,
                 dev["a"].p, dev["pooled"].p, C.c_int(c), ctx.stream)
    else:
        ctx.call("bsl_norm_apply", C.byref(d), dev["y"].p, dev["scale"].p, dev["shift"].p, dev["a"].p, ctx.stream)
    ctx.check_device()
    return d, dev, dict(y=y, gamma=gamma, beta=beta, mm=mm, mv=mv, eps=eps)


@pytest.mark.parametrize("mode,n,h,w,c,relu,train,pool", [
    (0, 4, 16, 16, 64, 1, 1, False), (0, 2, 8, 8, 128, 1, 1, True), (0, 3, 8, 8, 64, 1, 0, False),
    (1, 3, 16, 16, 64, 1, 1, True), (1, 2, 8, 12, 256, 0, 1, False), (0, 2, 2, 2, 1024, 1, 1, False)])
def test_norm_forward(ctx, mode, n, h, w, c, relu, train, pool):
    d, dev, host = _norm_forward(ctx, mode, n, h, w, c, relu, train, pool)
    y64 = host["y"].astype(np.float64)
    g, b = host["gamma"].astype(np.float64), host["beta"].astype(np.float64)
    if mode == 0 and train:
        z, _, nmm, nmv = O.batch_norm_train(y64, g, b, host["mm"].astype(np.float64), host["mv"].astype(np.float64))
        assert rel(dev["mm"].download(np.float32, (c,)), nmm) < 1e-5
        assert rel(dev["mv"].download(np.float32, (c,)), nmv) < 1e-5
    elif mode == 0:
        z = O.batch_norm_infer(y64, g, b, host["mm"].astype(np.float64), host["mv"].astype(np.float64))
        assert np.array_equal(dev["mm"].download(np.float32, (c,)), host["mm"])   # untouched in eval
    else:
        z, _ = O.instance_norm(y64, g, b, 1e-6)
    ref = O.relu(z) if relu else z
    got = ctx.bf16_to_f32(dev["a"], (n, h, w, c))
    assert rel(got, ref) < 5e-3
    if pool:
        gp = ctx.bf16_to_f32(dev["pooled"], (n, h // 2, w // 2, c))
        assert np.array_equal(gp, O.max_pool_2x2(got)), "pooled tensor must be the exact max of the stored activations"
    for v in dev.values():
        v.free()


@pytest.mark.parametrize("mode,n,h,w,c", [(0, 4, 16, 16, 64), (1, 3, 8, 8, 128), (0, 2, 4, 4, 512)])
def test_norm_backward(ctx, mode, n, h, w, c):
    d, dev, host = _norm_forward(ctx, mode, n, h, w, c, 1, 1, False, seed=5)
    rng = np.random.default_rng(9)
    da = bf16_randn(rng, (n, h, w, c))
    dda = ctx.bf16_from_f32(da)
    dyo = ctx.alloc(n * h * w * c * 2)
    dg, db = ctx.alloc(c * 4), ctx.alloc(c * 4)
    ctx.call("bsl_norm_bwd_reduce", C.byref(d), dev["y"].p, dda.p, C.c_int(c), dev["mean"].p, dev["rstd"].p,
             dev["scale"].p, dev["shift"].p, dev["sums"].p, ctx.stream)
    ctx.call("bsl_norm_bwd_finalize", C.byref(d), dev["sums"].p, dev["c1"].p, dev["c2"].p, dg.p, db.p, ctx.stream)
    ctx.call("bsl_norm_bwd_apply", C.byref(d), dev["y"].p, dda.p, C.c_int(c), dev["mean"].p, dev["rstd"].p,
             dev["scale"].p, dev["shift"].p, dev["c1"].p, dev["c2"].p, dyo.p, C.c_int(c), ctx.stream)
    ctx.check_device()
    y64 = host["y"].astype(np.float64)
    g, b = host["gamma"].astype(np.float64), host["beta"].astype(np.float64)
    if mode == 0:
        z, cache, _, _ = O.batch_norm_train(y64, g, b, 0 * g, 1 + 0 * g)
        fn = O.batch_norm_grad
    else:
        z, cache = O.instance_norm(y64, g, b, 1e-6)
        fn = O.instance_norm_grad
    dz = O.relu_grad(da.astype(np.float64), z)
    rdx, rdg, rdb = fn(dz, cache)
    assert rel(ctx.bf16_to_f32(dyo, (n, h, w, c)), rdx) < 5e-3
    assert rel(dg.download(np.float32, (c,)), rdg) < 1e-4
    assert rel(db.download(np.float32, (c,)), rdb) < 1e-4
    for v in list(dev.values()) + [dda, dyo, dg, db]:
        v.free()


def test_maxpool_backward_ties_and_skip_add(ctx):
    n, h, w, c = 2, 8, 8, 64
    rng = np.random.default_rng(2)
    act = np.maximum(bf16_randn(rng, (n, h, w, c)), 0)            # many exact-zero ties, as after ReLU
    act[0, :2, :2, :] = round_bf16(np.float32(0.75))              # a positive all-equal window
    dpool = bf16_randn(rng, (n, h // 2, w // 2, c))
    dskip = bf16_randn(rng, (n, h, w, 2 * c))                     # lower half of a concat gradient buffer
    da, dp, ds = ctx.bf16_from_f32(act), ctx.bf16_from_f32(dpool), ctx.bf16_from_f32(dskip)
    out = ctx.alloc(n * h * w * c * 2)
    ctx.call("bsl_maxpool2x2_bwd_add", C.c_int(n), C.c_int(h), C.c_int(w), C.c_int(c), da.p, C.c_int(c), dp.p, C.c_int(c),
             ds.p, C.c_int(2 * c), out.p, C.c_int(c), ctx.stream)
    ctx.check_device()
    ref = round_bf16((O.max_pool_2x2_grad(act, dpool) + dskip[..., :c]).astype(np.float32))
    assert np.array_equal(ctx.bf16_to_f32(out, (n, h, w, c)), ref)
    ctx.call("bsl_maxpool2x2_bwd_add", C.c_int(n), C.c_int(h), C.c_int(w), C.c_int(c), da.p, C.c_int(c), dp.p, C.c_int(c),
             None, C.c_int(0), out.p, C.c_int(c), ctx.stream)
    assert np.array_equal(ctx.bf16_to_f32(out, (n, h, w, c)), O.max_pool_2x2_grad(act, dpool))
    for b in (da, dp, ds, out):
        b.free()


def test_relu_backward_in_place_view(ctx):
    n, h, w, c = 2, 4, 4, 64
    rng = np.random.default_rng(3)
    y = np.maximum(bf16_randn(rng, (n, h, w, 2 * c)), 0)
    dy = bf16_randn(rng, (n, h, w, 2 * c))
    dy_dev, y_dev = ctx.bf16_from_f32(dy), ctx.bf16_from_f32(y)
    up = C.c_void_p(dy_dev.ptr + c * 2)
    ctx.call("bsl_relu_bwd", C.c_longlong(n * h * w), C.c_int(c), C.c_void_p(y_dev.ptr + c * 2), C.c_int(2 * c), up,
             C.c_int(2 * c), up, C.c_int(2 * c), ctx.stream)
    got = ctx.bf16_to_f32(dy_dev, (n, h, w, 2 * c))
    assert np.array_equal(got[..., c:], O.relu_grad(dy[..., c:], y[..., c:]))
    assert np.array_equal(got[..., :c], dy[..., :c]), "lower channel half must be untouched"
    dy_dev.free(); y_dev.free()


@pytest.mark.parametrize("cin", [1, 3])
def test_stem_conv(ctx, cin):
    n, h, w, cout = 2, 12, 20, 64
    rng = np.random.default_rng(cin)
    x = rng.uniform(0, 1, (n, h, w, cin)).astype(np.float32)
    wt = (rng.standard_normal((3, 3, cin, cout)) * 0.2).astype(np.float32)
    dy = bf16_randn(rng, (n, h, w, cout))
    dx_, dw_, ddy = ctx.from_numpy(x), ctx.from_numpy(wt), ctx.bf16_from_f32(dy)
    yo, dwo = ctx.alloc(n * h * w * cout * 2), ctx.alloc(9 * cin * cout * 4)
    d = _lib.Conv2dDesc(n, h, w, cin, cout, 3, 3, cin, cout)
    ctx.call("bsl_conv2d_stem_fprop", C.byref(d), dx_.p, dw_.p, yo.p, ctx.stream)
    ctx.call("bsl_conv2d_stem_wgrad", C.byref(d), dx_.p, ddy.p, dwo.p, ctx.stream)
    ctx.check_device()
    assert rel(ctx.bf16_to_f32(yo, (n, h, w, cout)), O.conv2d(x.astype(np.float64), wt.astype(np.float64))) < 3e-3
    assert rel(dwo.download(np.float32, (3, 3, cin, cout)),
               O.conv2d_backprop_filter(x.astype(np.float64), wt.shape, dy.astype(np.float64))) < 1e-5
    for b in (dx_, dw_, ddy, yo, dwo):
        b.free()


@pytest.mark.parametrize("n,h,w,cin,ld", [(2, 12, 20, 3, 64), (1, 5, 300, 1, 64), (3, 16, 128, 5, 64), (2, 7, 131, 7, 64),
                                          (2, 12, 20, 3, 32), (1, 5, 300, 1, 32), (2, 16, 131, 2, 32)])
def test_stem_im2col_bit_exact(ctx, n, h, w, cin, ld):
    """col[p, t*cin+ci] = bf16(x[p + tap t, ci]) with zero SAME padding; columns >= 9*cin are zero. Row pitch 64
    (bsl_stem_im2col) or 32 columns (bsl_stem_im2col_ld)."""
    rng = np.random.default_rng(w)
    x = rng.uniform(-1, 1, (n, h, w, cin)).astype(np.float32)
    dx_ = ctx.from_numpy(x)
    col = ctx.alloc(n * h * w * ld * 2)
    ctx.call("bsl_memset", col.p, C.c_int(0xff), C.c_size_t(col.nbytes), ctx.stream)
    d = _lib.Conv2dDesc(n, h, w, cin, 64, 3, 3, cin, 64)
    if ld == 64:
        ctx.call("bsl_stem_im2col", C.byref(d), dx_.p, col.p, ctx.stream)
    else:
        ctx.call("bsl_stem_im2col_ld", C.byref(d), dx_.p, col.p, C.c_int(ld), ctx.stream)
    ctx.check_device()
    got = col.download(np.uint16, (n, h, w, ld))
    xp = np.zeros((n, h + 2, w + 2, cin), np.float32)
    xp[:, 1:-1, 1:-1] = x
    ref = np.zeros((n, h, w, ld), np.float32)
    for t in range(9):
        ref[..., t * cin:(t + 1) * cin] = xp[:, t // 3:t // 3 + h, t % 3:t % 3 + w]
    from boxsegliver_b200.device import f32_to_bf16_bits
    assert np.array_equal(got, f32_to_bf16_bits(ref).reshape(ref.shape))
    dx_.free()
    col.free()


@pytest.mark.parametrize("classes", [2, 3])
def test_logits_conv(ctx, classes):
    n, h, w, cin = 2, 10, 12, 64
    rng = np.random.default_rng(classes)
    x = bf16_randn(rng, (n, h, w, cin))
    wt = (rng.standard_normal((1, 1, cin, classes)) * 0.2).astype(np.float32)
    bias = rng.standard_normal(classes).astype(np.float32)
    dl = rng.standard_normal((n, h, w, classes)).astype(np.float32)
    dx_, dw_, db_, ddl = ctx.bf16_from_f32(x), ctx.from_numpy(wt), ctx.from_numpy(bias), ctx.from_numpy(dl)
    lo, dxo = ctx.alloc(n * h * w * classes * 4), ctx.alloc(n * h * w * cin * 2)
    dwo, dbo = ctx.alloc(cin * classes * 4), ctx.alloc(classes * 4)
    d = _lib.Conv2dDesc(n, h, w, cin, classes, 1, 1, cin, classes)
    ctx.call("bsl_conv2d_head_fprop", C.byref(d), dx_.p, dw_.p, db_.p, lo.p, ctx.stream)
    ctx.call("bsl_conv2d_head_dgrad", C.byref(d), ddl.p, dw_.p, dxo.p, ctx.stream)
    ctx.call("bsl_conv2d_head_wgrad", C.byref(d), dx_.p, ddl.p, dwo.p, dbo.p, ctx.stream)
    ctx.check_device()
    x64, w64, dl64 = x.astype(np.float64), wt.astype(np.float64), dl.astype(np.float64)
    assert rel(lo.download(np.float32, (n, h, w, classes)), O.conv2d(x64, w64) + bias) < 1e-5
    assert rel(ctx.bf16_to_f32(dxo, (n, h, w, cin)), O.conv2d_backprop_input(x.shape, w64, dl64)) < 3e-3
    assert rel(dwo.download(np.float32, (1, 1, cin, classes)), O.conv2d_backprop_filter(x64, wt.shape, dl64)) < 1e-5
    assert rel(dbo.download(np.float32, (classes,)), dl64.sum(axis=(0, 1, 2))) < 1e-5
    for b in (dx_, dw_, db_, ddl, lo, dxo, dwo, dbo):
        b.free()


def _loss_desc(n, hw, classes, wtype, numeric=(), decay=1000.0, scale=1.0):
    nw = (C.c_float * 8)(*(list(numeric) + [0.0] * (8 - len(numeric))))
    return _lib.LossDesc(n, hw, classes, {"none": 0, "numerical": 1, "proportion": 2}[wtype], nw, decay, scale)


@pytest.mark.parametrize("wtype,classes", [("none", 3), ("numerical", 3), ("proportion", 3), ("numerical", 2)])
def test_weighted_xent(ctx, wtype, classes):
    n, h, w = 4, 16, 24
    rng = np.random.default_rng(classes)
    logits = (rng.standard_normal((n, h, w, classes)) * 2).astype(np.float32)
    labels = rng.integers(0, classes, (n, h, w)).astype(np.int32)
    labels[1] = 0                      # an all-background image
    labels[2][labels[2] == classes - 1] = 0   # an image with one class absent
    numeric = (0.2, 0.4, 4.4)[:classes]
    d = _loss_desc(n, h * w, classes, wtype, numeric if wtype == "numerical" else (), scale=0.5)
    dl_, dlab = ctx.from_numpy(logits), ctx.from_numpy(labels)
    counts, loss, dlo = ctx.alloc(n * classes * 4), ctx.alloc(16), ctx.alloc(logits.nbytes)
    wsb = ctx.lib.bsl_loss_workspace(ctx.h, C.byref(d))
    ws = ctx.alloc(wsb)
    ctx.call("bsl_label_counts", C.byref(d), dlab.p, counts.p, ctx.stream)
    ctx.call("bsl_wxent_fwd_bwd", C.byref(d), dl_.p, dlab.p, counts.p, loss.p, dlo.p, ws.p, C.c_size_t(wsb), ctx.stream)
    ctx.check_device()
    cnt = counts.download(np.int32, (n, classes))
    assert np.array_equal(cnt, np.stack([np.bincount(labels[i].ravel(), minlength=classes) for i in range(n)]))
    kw = {}
    if wtype == "numerical":
        kw["numeric_w"] = numeric
    if wtype == "proportion":
        kw["proportion_decay"] = 1000.0
    rl, rdl = O.weighted_sparse_softmax_cross_entropy(logits.astype(np.float64), labels, wtype, **kw)
    assert abs(float(loss.download(np.float32, (1,))[0]) - float(rl)) < 1e-5 * max(1.0, abs(float(rl)))
    assert rel(dlo.download(np.float32, logits.shape), 0.5 * rdl) < 1e-5
    for b in (dl_, dlab, counts, loss, dlo, ws):
        b.free()


def test_dice_loss(ctx):
    n, h, w, classes = 3, 16, 16, 3
    rng = np.random.default_rng(4)
    logits = (rng.standard_normal((n, h, w, classes)) * 2).astype(np.float32)
    labels = rng.integers(0, classes, (n, h, w)).astype(np.int32)
    labels[0] = 0
    d = _loss_desc(n, h * w, classes, "none")
    dl_, dlab, loss, dlo = ctx.from_numpy(logits), ctx.from_numpy(labels), ctx.alloc(16), ctx.alloc(logits.nbytes)
    wsb = ctx.lib.bsl_loss_workspace(ctx.h, C.byref(d))
    ws = ctx.alloc(wsb)
    ctx.call("bsl_dice_fwd_bwd", C.byref(d), dl_.p, dlab.p, loss.p, dlo.p, C.c_int(0), ws.p, C.c_size_t(wsb), ctx.stream)
    ctx.check_device()
    l64 = logits.astype(np.float64)
    prob = O.softmax(l64)
    rl, dp = O.sparse_dice_loss(prob, labels)
    assert abs(float(loss.download(np.float32, (1,))[0]) - float(rl)) < 1e-5
    assert rel(dlo.download(np.float32, logits.shape), O.softmax_grad(dp, prob)) < 1e-4
    for b in (dl_, dlab, loss, dlo, ws):
        b.free()


def test_softmax_masks_argmax_counts_bit_exact(ctx):
    n, h, w, classes = 3, 20, 36, 3      # hw = 720: warps straddle image boundaries
    rng = np.random.default_rng(8)
    logits = (rng.standard_normal((n, h, w, classes)) * 3).astype(np.float32)
    labels = rng.integers(0, classes, (n, h, w)).astype(np.int32)
    d = _loss_desc(n, h * w, classes, "none")
    dl_, dlab = ctx.from_numpy(logits), ctx.from_numpy(labels)
    prob, masks = ctx.alloc(logits.nbytes), ctx.alloc((classes - 1) * n * h * w)
    am, ilr = ctx.alloc(n * h * w), ctx.alloc(n * (classes - 1) * 3 * 4)
    ctx.call("bsl_softmax_threshold", C.byref(d), dl_.p, dlab.p, prob.p, masks.p, am.p, ilr.p, ctx.stream)
    ctx.check_device()
    p = prob.download(np.float32, logits.shape)
    assert rel(p, O.softmax(logits.astype(np.float64))) < 1e-6
    m = masks.download(np.uint8, (classes - 1, n, h, w))
    ref_m = np.stack([(p[..., c] > 0.5).astype(np.uint8) for c in range(1, classes)])
    assert np.array_equal(m, ref_m), "threshold masks must be bit-exact w.r.t. the emitted probabilities"
    assert np.array_equal(am.download(np.uint8, (n, h, w)), np.argmax(p, axis=-1).astype(np.uint8))
    got = ilr.download(np.uint32, (n, classes - 1, 3))
    for c in range(1, classes):
        i_, l_, r_ = O.seg_counts(m[c - 1][..., None], labels, c)
        assert np.array_equal(got[:, c - 1, 0], i_) and np.array_equal(got[:, c - 1, 1], l_)
        assert np.array_equal(got[:, c - 1, 2], r_)
    for b in (dl_, dlab, prob, masks, am, ilr):
        b.free()


def test_adam_and_momentum_steps(ctx):
    nel = 100_003
    rng = np.random.default_rng(6)
    w = rng.standard_normal(nel).astype(np.float32)
    g = rng.standard_normal(nel).astype(np.float32)
    m0 = (rng.standard_normal(nel) * 0.1).astype(np.float32)
    v0 = rng.uniform(0, 0.1, nel).astype(np.float32)
    dw, dg, dm, dv = (ctx.from_numpy(a) for a in (w, g, m0, v0))
    shadow, sq = ctx.alloc(nel * 2), ctx.alloc(8)
    d = _lib.AdamDesc(1e-3, 0.9, 0.99, 1e-8, 1e-5, 0.5, 7, 0.0)
    ctx.call("bsl_adam_step", C.byref(d), dw.p, dg.p, dm.p, dv.p, shadow.p, C.c_size_t(nel), sq.p, ctx.stream)
    ctx.check_device()
    geff = 0.5 * g.astype(np.float64) + 1e-5 * w
    rw, rm, rv = O.adam_step(w.astype(np.float64), geff, m0.astype(np.float64), v0.astype(np.float64), 7, 1e-3)
    got_w = dw.download(np.float32, (nel,))
    assert rel(got_w - w, rw - w) < 1e-4
    assert rel(dm.download(np.float32, (nel,)), rm) < 1e-6 and rel(dv.download(np.float32, (nel,)), rv) < 1e-6
    assert np.array_equal(ctx.bf16_to_f32(shadow, (nel,)), round_bf16(got_w))
    assert abs(sq.download(np.float64, (1,))[0] - float((w.astype(np.float64) ** 2).sum())) < 1e-6 * nel
    acc = ctx.from_numpy(m0)
    dw2 = ctx.from_numpy(w)
    ctx.call("bsl_momentum_step", C.c_float(0.01), C.c_float(0.9), C.c_int(0), C.c_float(0.0), C.c_float(1.0), dw2.p,
             dg.p, acc.p, None, C.c_size_t(nel), None, ctx.stream)
    rw2, racc = O.momentum_step(w.astype(np.float64), g.astype(np.float64), m0.astype(np.float64), 0.01)
    assert rel(dw2.download(np.float32, (nel,)), rw2) < 1e-6
    for b in (dw, dg, dm, dv, shadow, sq, acc, dw2):
        b.free()


def test_optimizer_flag_variants(ctx):
    """--adam_beta1/2/eps, AdamW's decoupled decay, --mm_mm / --mm_nesterov (/root/reference/core/solver.py:86-97,
    204-219) against oracle.tf_ops in fp64."""
    nel = 50_001
    rng = np.random.default_rng(16)
    w = rng.standard_normal(nel).astype(np.float32)
    g = rng.standard_normal(nel).astype(np.float32)
    m0 = (rng.standard_normal(nel) * 0.1).astype(np.float32)
    v0 = rng.uniform(0, 0.1, nel).astype(np.float32)
    f8 = lambda a: a.astype(np.float64)  # noqa: E731
    for b1, b2, eps, decay in ((0.5, 0.999, 1e-8, 0.0), (0.9, 0.99, 1e-3, 0.0), (0.9, 0.99, 1e-8, 3e-2)):
        dw, dg, dm, dv = (ctx.from_numpy(a) for a in (w, g, m0, v0))
        d = _lib.AdamDesc(2e-3, b1, b2, eps, 0.0, 1.0, 3, decay)
        ctx.call("bsl_adam_step", C.byref(d), dw.p, dg.p, dm.p, dv.p, None, C.c_size_t(nel), None, ctx.stream)
        rw, rm, rv = O.adam_step(f8(w), f8(g), f8(m0), f8(v0), 3, 2e-3, b1, b2, eps, decoupled_decay=decay)
        assert rel(dw.download(np.float32, (nel,)) - w, rw - w) < 1e-4, (b1, b2, eps, decay)
        assert rel(dm.download(np.float32, (nel,)), rm) < 1e-6 and rel(dv.download(np.float32, (nel,)), rv) < 1e-6
        if decay:    # the decay really is decoupled: it differs from folding wd * w into the gradient
            rw_l2, _, _ = O.adam_step(f8(w), f8(g) + decay * f8(w), f8(m0), f8(v0), 3, 2e-3, b1, b2, eps)
            assert rel(rw - w, rw_l2 - w) > 1e-2
        for b in (dw, dg, dm, dv):
            b.free()
    for mom, nesterov in ((0.5, 0), (0.9, 1), (0.7, 1)):
        dw, dg, acc = (ctx.from_numpy(a) for a in (w, g, m0))
        ctx.call("bsl_momentum_step", C.c_float(0.01), C.c_float(mom), C.c_int(nesterov), C.c_float(1e-4),
                 C.c_float(1.0), dw.p, dg.p, acc.p, None, C.c_size_t(nel), None, ctx.stream)
        rw, racc = O.momentum_step(f8(w), f8(g) + 1e-4 * f8(w), f8(m0), 0.01, mom, bool(nesterov))
        assert rel(dw.download(np.float32, (nel,)) - w, rw - w) < 1e-5, (mom, nesterov)
        assert rel(acc.download(np.float32, (nel,)), racc) < 1e-6
        for b in (dw, dg, acc):
            b.free()


def test_casts_roundtrip(ctx):
    rng = np.random.default_rng(1)
    a = rng.standard_normal(10_001).astype(np.float32)
    src, mid, dst = ctx.from_numpy(a), ctx.alloc(a.size * 2), ctx.alloc(a.nbytes)
    ctx.call("bsl_cast_f32_to_bf16", src.p, mid.p, C.c_size_t(a.size), ctx.stream)
    ctx.call("bsl_cast_bf16_to_f32", mid.p, dst.p, C.c_size_t(a.size), ctx.stream)
    assert np.array_equal(dst.download(np.float32, a.shape), round_bf16(a))
    for b in (src, mid, dst):
        b.free()


def test_relu_bwd_bias_matches_two_passes(ctx):
    """bsl_relu_bwd_bias == bsl_relu_bwd followed by the bias-gradient reduction of bsl_convT2d_bwd_filter: the masked
    gradient bit for bit (also in place, with channel windows of a wider buffer), the bias gradient to fp32 rounding
    of the same fixed-order sums."""
    rng = np.random.default_rng(31)
    for pixels, c, ld in ((2 * 32 * 32, 64, 128), (5 * 16 * 16, 256, 256), (1000, 8, 24)):
        yh = np.maximum(rng.standard_normal((pixels, ld)), 0).astype(np.float32)
        dyh = rng.standard_normal((pixels, ld)).astype(np.float32)
        y, dy = ctx.from_numpy(f32_to_bf16_bits(yh)), ctx.from_numpy(f32_to_bf16_bits(dyh))
        a, b = ctx.alloc(pixels * ld * 2).zero(), ctx.from_numpy(f32_to_bf16_bits(dyh))
        db = ctx.alloc(c * 4)
        c0 = ld - c                                            # upper channel window, like the concat buffer
        win = lambda buf: C.c_void_p(buf.ptr + c0 * 2)         # noqa: E731
        ctx.call("bsl_relu_bwd", C.c_longlong(pixels), C.c_int(c), win(y), C.c_int(ld), win(dy), C.c_int(ld), win(a),
                 C.c_int(ld), ctx.stream)
        ctx.call("bsl_relu_bwd_bias", C.c_longlong(pixels), C.c_int(c), win(y), C.c_int(ld), win(b), C.c_int(ld), win(b),
                 C.c_int(ld), db.p, ctx.stream)               # in place
        ctx.check_device()
        ra = a.download(np.uint16, (pixels, ld))[:, c0:]
        rb = b.download(np.uint16, (pixels, ld))[:, c0:]
        assert np.array_equal(ra, rb)
        if c0:
            assert np.array_equal(b.download(np.uint16, (pixels, ld))[:, :c0], f32_to_bf16_bits(dyh)[:, :c0])  # untouched
        ref = bf16_bits_to_f32(ra).astype(np.float64).sum(axis=0)
        got = db.download(np.float32, (c,))
        assert np.allclose(got, ref, rtol=2e-6, atol=1e-4), np.abs(got - ref).max()
        for buf in (y, dy, a, b, db):
            buf.free()
