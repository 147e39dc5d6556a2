"""Op-level parity of the kernels downstream of the logits (csrc/loss.cu, csrc/infer.cu) at the shapes the engines train
and evaluate on, through the C ABI the engines call (engine.py / unet3d_engine.py loss_backward and predict_outputs,
inference.py). References: oracle.tf_ops in fp64 on the same fp32 logits the device reads (tests/test_loss_ref.py pins
those functions to torch autograd), np.bincount for the label counts, numpy's fp32 arithmetic for the inference passes.

Gates: loss values 1e-6 relative; dlogits 5e-6 relative L2 per (image, class) slice; probabilities 1e-6 relative L2
per (image, class) slice. Measured worst on a B200: 5.3e-8, 4.0e-7 and 1.3e-7, the size of fp32 rounding. Integer outputs, masks, argmax, flips and TTA averages are exact. Every output sits in front
of a guard region, starts as a NaN byte pattern where the kernel must overwrite it, and the loss workspace is filled
with the same pattern before every call, so a partial or a weight row a kernel leaves unwritten shows up as NaN. Every
case runs twice and must be bit-identical: all reductions here are fixed-order or integer.

Grid arithmetic in the comments is for 148 SMs: the per-pixel loss passes cap at 8 * 148 = 1184 blocks of 256 threads
(303 104 threads; the vector cross-entropy path takes 4 pixels per thread), the label counts and the Dice reduction at
64 blocks per image (16 384 pixels), and the inference passes at 16 * 148 = 2368 blocks (606 208 elements)."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from oracle import tf_ops as O
from tests.gpu_util import report

pytestmark = pytest.mark.gpu

BSL_EINVAL, BSL_EUNSUPPORTED, BSL_EWORKSPACE = -1, -2, -3
GUARD = 256          # canary bytes after every output
POISON = 0xFF        # every fp32 / fp64 lane NaN, int32 -1, uint8 255
TOL_LOSS, TOL_DL, TOL_PROB = 1e-6, 5e-6, 1e-6
WTYPE = {"none": 0, "numerical": 1, "proportion": 2}


class Out:
    """An output of `shape` x `dtype` followed by GUARD bytes; it starts as `init` (or the poison pattern) and the
    guard as poison."""

    def __init__(self, ctx, dtype, shape, init=None):
        self.dtype, self.shape = np.dtype(dtype), tuple(shape)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        host = np.full(self.nbytes + GUARD, POISON, np.uint8)
        if init is not None:
            host[:self.nbytes] = np.ascontiguousarray(init, self.dtype).view(np.uint8).ravel()
        self.buf = ctx.from_numpy(host)

    @property
    def p(self):
        return self.buf.p

    def get(self):
        raw = self.buf.download(np.uint8, (self.nbytes + GUARD,))
        assert (raw[self.nbytes:] == POISON).all(), "a store past the end of an output"
        return raw[:self.nbytes].view(self.dtype).reshape(self.shape)

    def free(self):
        self.buf.free()


def _bits(a):
    return np.ascontiguousarray(a).view({1: np.uint8, 4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def _slice_rel(got, ref, n, classes):
    """Largest relative L2 error over the (image, class) slices of [n * hw, classes] tensors."""
    g = np.asarray(got, np.float64).reshape(n, -1, classes)
    r = np.asarray(ref, np.float64).reshape(n, -1, classes)
    num = np.sqrt(((g - r) ** 2).sum(axis=1))
    den = np.maximum(np.sqrt((r ** 2).sum(axis=1)), 1e-30)
    return float((num / den).max())


def _loss_desc(n, hw, classes, wtype="none", numeric=(), decay=0.0, scale=1.0):
    nw = (C.c_float * 8)(*(list(numeric) + [0.0] * (8 - len(numeric))))
    return _lib.LossDesc(n, hw, classes, WTYPE[wtype], nw, decay, scale)


# ------------------------------------------------------------------ weighted cross entropy, Dice, label counts
def _lc(cid, n, hw, classes, wtype, numeric=(), decay=0.0, scale=1.0, dice=False, accumulate=False, labels="mixed",
        null_dlogits=False):
    numeric = tuple(float(np.float32(v)) for v in numeric)      # the reference uses the fp32 weights the device reads
    return pytest.param(dict(cid=cid, n=n, hw=hw, classes=classes, wtype=wtype, numeric=numeric, decay=decay,
                             scale=scale, dice=dice, accumulate=accumulate, labels=labels,
                             null_dlogits=null_dlogits), id=cid)


LOSS_CASES = [
    # cfg2 (UNet 256^2, batch 64). VEC path: 1 048 576 quads over 303 104 threads, 3.5 trips of the grid stride; the
    # weight table's lanes take images i and i + 32; label counts want 256 blocks per image -> 64, 4 trips each
    _lc("L1", 64, 256 * 256, 3, "numerical", numeric=(0.2, 0.4, 4.4)),
    # cfg3 (GUNet 512^2, batch 32, xentropy+dice): xent, then Dice accumulating into its dlogits. dice_final runs
    # 1024 threads (32 warps, one image each); dice_reduce wants 1024 blocks per image -> 64, 16 trips
    _lc("L2", 32, 512 * 512, 3, "numerical", numeric=(0.2, 0.4, 4.4), dice=True, accumulate=True),
    # cfg4 (UNet3D 64 x 128 x 128, batch 4 per GPU, 8 GPUs -> loss_scale 1/8): VEC path with 2 classes, 3.5 trips
    _lc("L3", 4, 64 * 128 * 128, 2, "numerical", numeric=(0.6, 2.4), scale=0.125, dice=True),
    # hw = 97 x 61 = 5917, not a multiple of 4 -> the scalar path; 4 classes; dice_final: 256 threads = 8 warps for
    # 9 images, warp 0 takes images 0 and 8
    _lc("L4", 9, 97 * 61, 4, "proportion", decay=1000.0, dice=True),
    # 33 images of 5 x 6 px: the weight table's lane 0 takes images 0 and 32; dice_final's 32 warps, warp 0 takes
    # images 0 and 32; warps straddle images. Proportion without decay divides by the class count, so every class is
    # in every image (an absent class is 1/0, NaN in the reference as on the device)
    _lc("L5", 33, 5 * 6, 3, "proportion", decay=0.0, dice=True, labels="every"),
    # one image of 16 385 px: label counts and dice_reduce want 65 blocks -> 64, the last pixel takes a second trip;
    # odd hw -> scalar path. Both losses with and without dlogits
    _lc("L6", 1, 16385, 2, "none", dice=True, null_dlogits=True),
    # no label in [0, classes): nz = 0 takes the safe division -- loss 0, dlogits 0
    _lc("L7", 3, 32 * 32, 3, "none", labels="all_ignored"),
    # labels 255 and -1 mixed in: ignored by the cross entropy and the counts, background for Dice
    _lc("L8", 4, 24 * 40, 3, "none", dice=True, labels="ignored"),
]


def _loss_inputs(cs):
    n, hw, k = cs["n"], cs["hw"], cs["classes"]
    rng = np.random.default_rng(n * 1000 + k)
    logits = rng.standard_normal((n, hw, k), dtype=np.float32) * np.float32(2)
    logits += rng.normal(0, 1.5, (n, 1, k)).astype(np.float32)            # per image and per class
    labels = rng.integers(0, k, (n, hw), dtype=np.int32)
    kind = cs["labels"]
    if kind == "every":
        labels[:, :k] = np.arange(k)
    elif kind == "all_ignored":
        labels[:] = 255
    elif n >= 3:
        labels[0] = 0                                                    # all background
        missing = k - 1 if k > 2 else 0                                  # with 2 classes: all foreground
        labels[1][labels[1] == missing] = (missing + 1) % k
        if cs["dice"]:
            # background, foreground probabilities 0 in fp32: U = 0 and the Dice eps keeps 2I / (U + eps) at 0
            labels[n - 1] = 0
            logits[n - 1, :, 1:] -= np.float32(200)
    if kind == "ignored":
        r = rng.random((n, hw))
        labels[r < 0.1] = 255
        labels[(r >= 0.1) & (r < 0.15)] = -1
    return logits, labels


def _xent_ref(logits, labels, cs, step=4):
    """(loss, dlogits * loss_scale) in fp64, in slices of `step` images (SUM_BY_NONZERO_WEIGHTS recombined)."""
    n, k = cs["n"], cs["classes"]
    kw = {"numeric_w": cs["numeric"]} if cs["wtype"] == "numerical" else {}
    if cs["wtype"] == "proportion":
        kw["proportion_decay"] = cs["decay"]
    dl = np.zeros(logits.shape, np.float64)
    if cs["labels"] in ("ignored", "all_ignored"):
        # The device's own contract for labels outside [0, classes): weight 0, outside nz and the counts, a zero
        # gradient row. The reference's "none" weighting would count them in nz, so the oracle runs on the in-range
        # pixels only (no per-image renormalisation with "none").
        assert cs["wtype"] == "none"
        ok = (labels >= 0) & (labels < k)
        if not ok.any():
            return 0.0, dl
        loss, d = O.weighted_sparse_softmax_cross_entropy(logits[ok].astype(np.float64)[None, :, None],
                                                          labels[ok][None, :, None], "none")
        dl[ok] = d[0, :, 0]
        return float(loss), dl * cs["scale"]
    total, nz = 0.0, 0.0
    for s in range(0, n, step):
        lg, lb = logits[s:s + step].astype(np.float64)[:, :, None], labels[s:s + step][:, :, None]
        loss, d = O.weighted_sparse_softmax_cross_entropy(lg, lb, cs["wtype"], **kw)
        w = O.compute_weights(cs["wtype"], O.one_hot(lb, k, np.float64), **kw)
        m = float((np.broadcast_to(w, lb.shape) != 0).sum())
        total += float(loss) * m
        nz += m
        dl[s:s + step] = d[:, :, 0] * m
    return total / nz, dl * (cs["scale"] / nz)


def _dice_ref(logits, labels, cs, step=4):
    """(loss, dlogits * loss_scale) in fp64, in slices of `step` images (the 1/n of the mean recombined)."""
    n = cs["n"]
    dl = np.zeros(logits.shape, np.float64)
    terms = 0.0
    for s in range(0, n, step):
        prob = O.softmax(logits[s:s + step].astype(np.float64))[:, :, None]
        m = prob.shape[0]
        loss, dprob = O.sparse_dice_loss(prob, labels[s:s + step][:, :, None])
        terms += (1.0 - float(loss)) * m
        dl[s:s + step] = O.softmax_grad(dprob, prob)[:, :, 0] * (m / n)
    return 1.0 - terms / n, dl * cs["scale"]


def _run_loss(ctx, cs, logits, labels):
    """label counts, xent (with dlogits, and without it when asked), Dice (into a poisoned buffer, or accumulating
    into the xent gradient as the xentropy+dice step does) -- every output downloaded."""
    n, hw, k = cs["n"], cs["hw"], cs["classes"]
    d = _loss_desc(n, hw, k, cs["wtype"], cs["numeric"], cs["decay"], cs["scale"])
    dlg, dlab = ctx.from_numpy(logits), ctx.from_numpy(labels)
    wsb = ctx.lib.bsl_loss_workspace(ctx.h, C.byref(d))
    ws = ctx.alloc(wsb)
    res, outs = {}, []

    def out(*a, **kw):
        outs.append(Out(ctx, *a, **kw))
        return outs[-1]

    def poison():
        ctx.call("bsl_memset", ws.p, C.c_int(POISON), C.c_size_t(wsb), ctx.stream)

    counts = out(np.int32, (n, k))
    ctx.call("bsl_label_counts", C.byref(d), dlab.p, counts.p, ctx.stream)
    res["counts"] = counts.get()
    loss, dl = out(np.float32, (1,)), out(np.float32, logits.shape)
    poison()
    ctx.call("bsl_wxent_fwd_bwd", C.byref(d), dlg.p, dlab.p, counts.p, loss.p, dl.p, ws.p, C.c_size_t(wsb),
             ctx.stream)
    res["xent"], res["dl_xent"] = loss.get(), dl.get()
    if cs["null_dlogits"]:
        loss = out(np.float32, (1,))
        poison()
        ctx.call("bsl_wxent_fwd_bwd", C.byref(d), dlg.p, dlab.p, counts.p, loss.p, None, ws.p, C.c_size_t(wsb),
                 ctx.stream)
        res["xent_nodl"] = loss.get()
    if cs["dice"]:
        acc = cs["accumulate"]
        loss, dl = out(np.float32, (1,)), out(np.float32, logits.shape, init=res["dl_xent"] if acc else None)
        poison()
        ctx.call("bsl_dice_fwd_bwd", C.byref(d), dlg.p, dlab.p, loss.p, dl.p, C.c_int(int(acc)), ws.p,
                 C.c_size_t(wsb), ctx.stream)
        res["dice"], res["dl_dice"] = loss.get(), dl.get()
        if cs["null_dlogits"]:
            loss = out(np.float32, (1,))
            poison()
            ctx.call("bsl_dice_fwd_bwd", C.byref(d), dlg.p, dlab.p, loss.p, None, C.c_int(0), ws.p, C.c_size_t(wsb),
                     ctx.stream)
            res["dice_nodl"] = loss.get()
    ctx.check_device()
    for b in outs + [dlg, dlab, ws]:
        b.free()
    return res


@pytest.mark.parametrize("cs", LOSS_CASES)
def test_loss_op_parity(ctx, cs):
    n, k = cs["n"], cs["classes"]
    logits, labels = _loss_inputs(cs)
    r1 = _run_loss(ctx, cs, logits, labels)
    want_counts = np.stack([(labels == c).sum(axis=1) for c in range(k)], axis=1)
    assert np.array_equal(r1["counts"], want_counts)
    errs = {}
    loss, dl = _xent_ref(logits, labels, cs)
    got = float(r1["xent"][0])
    if cs["labels"] == "all_ignored":
        assert got == 0.0 and not r1["dl_xent"].any(), "nz = 0: loss and dlogits must be exactly 0"
    errs["xent"] = abs(got - loss) / abs(loss) if loss else abs(got)
    errs["dl_xent"] = _slice_rel(r1["dl_xent"], dl, n, k)
    del dl
    if cs["null_dlogits"]:
        assert _bits(r1["xent_nodl"]) == _bits(r1["xent"]), "xent without dlogits must give the same loss bits"
    if cs["dice"]:
        loss, dl = _dice_ref(logits, labels, cs)
        errs["dice"] = abs(float(r1["dice"][0]) - loss) / abs(loss)
        if cs["accumulate"]:
            dl += r1["dl_xent"]          # the xent gradient the Dice pass accumulates into
        errs["dl_dice"] = _slice_rel(r1["dl_dice"], dl, n, k)
        del dl
        if cs["null_dlogits"]:
            assert _bits(r1["dice_nodl"]) == _bits(r1["dice"]), "dice without dlogits must give the same loss bits"
    report(f"loss {cs['cid']} n{n} hw{cs['hw']} c{k} {cs['wtype']}", **errs)
    gates = dict(xent=TOL_LOSS, dice=TOL_LOSS, dl_xent=TOL_DL, dl_dice=TOL_DL)
    bad = {key: v for key, v in errs.items() if not v <= gates[key]}
    assert not bad, f"over the gate: {bad}"
    r2 = _run_loss(ctx, cs, logits, labels)
    assert r1.keys() == r2.keys()
    for key in r1:
        assert np.array_equal(_bits(r1[key]), _bits(r2[key])), f"{key} not bit-reproducible"


# ------------------------------------------------------------------ softmax, threshold masks, argmax, I / L / R counts
SOFTMAX = [
    pytest.param(64, 256 * 256, 3, id="cfg2"),            # warp-uniform counts; 4.2 M px over 303 104 threads
    pytest.param(4, 64 * 128 * 128, 2, id="cfg4"),        # 2 classes, 4.2 M px
    pytest.param(5, 97 * 61, 4, id="c4-odd"),             # 4 classes, odd hw: warps straddle images
    pytest.param(3, 20 * 36, 3, id="hw720"),              # 720 = 22.5 warps: straddling warps
    pytest.param(37, 7, 2, id="hw7"),                     # hw < 32: every warp spans several images
    pytest.param(33, 5 * 6, 4, id="hw30-c4"),
]
OUTPUTS = ("prob", "masks", "argmax", "ilr")


def _softmax_inputs(n, hw, k):
    """Logits with per-image / per-class offsets, a few labels outside [0, k), and exact ties: rows of equal logits,
    rows whose two largest entries are equal, and rows with two equal maxima and the rest 200 below (p = 0.5 exactly
    there). Returns the tie rows and the class argmax must pick (the first of the equal maxima)."""
    rng = np.random.default_rng(n * 31 + hw + k)
    P = n * hw
    logits = (rng.standard_normal((n, hw, k), dtype=np.float32) * np.float32(3)
              + rng.normal(0, 1.5, (n, 1, k)).astype(np.float32)).reshape(P, k)
    labels = rng.integers(0, k, P, dtype=np.int32)
    labels[rng.random(P) < 0.02] = 255
    labels[rng.random(P) < 0.02] = -1
    nt = min(max(P // 64, 6), 3000)
    rows = rng.choice(P, nt, replace=False)
    first = np.zeros(nt, np.int64)
    half = np.zeros(nt, bool)
    for j, p in enumerate(rows):
        v = np.float32(rng.normal(0, 2))
        kind = j % 3
        if kind == 0:
            logits[p] = v
            half[j] = k == 2
        else:
            a, b = np.sort(rng.choice(k, 2, replace=False))
            logits[p] = v - np.float32(200) if kind == 2 else v - rng.uniform(0.5, 3, k).astype(np.float32)
            logits[p, a] = logits[p, b] = v
            first[j], half[j] = a, kind == 2
    return logits, labels, rows, first, half


def _run_softmax(ctx, n, hw, k, dlg, dlab, which):
    P = n * hw
    d = _loss_desc(n, hw, k)
    o = dict(prob=Out(ctx, np.float32, (P, k)), masks=Out(ctx, np.uint8, (k - 1, P)),
             argmax=Out(ctx, np.uint8, (P,)), ilr=Out(ctx, np.uint32, (n, k - 1, 3)))
    ptr = {key: (o[key].p if key in which else None) for key in OUTPUTS}
    ctx.call("bsl_softmax_threshold", C.byref(d), dlg.p, dlab.p if "ilr" in which else None, ptr["prob"],
             ptr["masks"], ptr["argmax"], ptr["ilr"], ctx.stream)
    ctx.check_device()
    res = {key: o[key].get() for key in which}
    for key in OUTPUTS:
        if key not in which:
            raw = o[key].buf.download(np.uint8, (o[key].nbytes + GUARD,))
            assert (raw == POISON).all(), f"{key} written although it was not requested"
        o[key].free()
    return res


@pytest.mark.parametrize("n,hw,k", SOFTMAX)
def test_softmax_threshold_parity(ctx, n, hw, k):
    P = n * hw
    logits, labels, rows, first, half = _softmax_inputs(n, hw, k)
    dlg, dlab = ctx.from_numpy(logits), ctx.from_numpy(labels)
    full = _run_softmax(ctx, n, hw, k, dlg, dlab, OUTPUTS)
    p = full["prob"]
    err = _slice_rel(p, O.softmax(logits.astype(np.float64)), n, k)
    report(f"softmax n{n} hw{hw} c{k}", prob=err)
    assert err <= TOL_PROB
    # masks, argmax and the counts are exact functions of the emitted probabilities
    masks = full["masks"]
    assert np.array_equal(masks, np.stack([(p[:, c] > 0.5).astype(np.uint8) for c in range(1, k)]))
    assert np.array_equal(full["argmax"], np.argmax(p, axis=-1).astype(np.uint8))
    for c in range(1, k):
        i_, l_, r_ = O.seg_counts(masks[c - 1].reshape(n, hw, 1), labels.reshape(n, hw), c)
        assert np.array_equal(full["ilr"][:, c - 1], np.stack([i_, l_, r_], axis=1).astype(np.uint32)), c
    # ties: the first maximum wins; p = 0.5 exactly is not above the threshold
    assert np.array_equal(full["argmax"][rows], first.astype(np.uint8))
    assert half.any() and ((p[rows[half]] == 0.5).sum(axis=1) == 2).all()
    assert not masks[:, rows[half]].any()
    # every non-empty subset of the outputs gives the bits of the full call (the full set once more: a rerun)
    for bitset in range(1, 16):
        which = tuple(key for j, key in enumerate(OUTPUTS) if bitset >> j & 1)
        sub = _run_softmax(ctx, n, hw, k, dlg, dlab, which)
        for key in which:
            assert np.array_equal(_bits(sub[key]), _bits(full[key])), (which, key)
    dlg.free()
    dlab.free()


# ------------------------------------------------------------------ test-time mirroring, TTA average, confusion counts
AX = ((1, 3), (2, 2), (4, 1))        # axes bit -> numpy axis of [n, d, h, w, c]


@pytest.mark.parametrize("shape", [pytest.param((2, 5, 7, 9, 3), id="odd"),
                                   pytest.param((1, 64, 128, 128, 2), id="cfg4-grid-stride")])
def test_flip_f32_bit_exact(ctx, shape):
    rng = np.random.default_rng(sum(shape))
    src = rng.standard_normal(shape, dtype=np.float32)
    base = rng.standard_normal(shape, dtype=np.float32)
    dsrc = ctx.from_numpy(src)
    for axes in range(8):
        flipped = np.flip(src, tuple(ax for bit, ax in AX if axes & bit))
        for acc in (0, 1):
            dst = Out(ctx, np.float32, shape, init=base if acc else None)
            ctx.call("bsl_flip_f32", C.c_longlong(shape[0]), *(C.c_int(v) for v in shape[1:]), C.c_int(axes),
                     C.c_int(acc), dsrc.p, dst.p, ctx.stream)
            want = base + flipped if acc else flipped
            assert np.array_equal(_bits(dst.get()), _bits(want)), (axes, acc)
            dst.free()
    dsrc.free()


@pytest.mark.parametrize("k", [2, 3, 4])
def test_tta_finalize_bit_exact(ctx, k):
    pixels = 700_001                                   # > 606 208: the grid-stride loop runs
    rng = np.random.default_rng(k)
    for count in (1, 3, 8):
        acc = rng.uniform(0, count, (pixels, k)).astype(np.float32)
        t = rng.choice(pixels, 3000, replace=False)
        acc[t[:1000]] = acc[t[:1000], :1]                              # all classes equal
        a = rng.integers(0, k - 1, 2000)
        hi = acc[t[1000:], :].max(axis=1) + np.float32(0.5)
        acc[t[1000:], a] = hi                                          # an exact tie of the two largest
        acc[t[1000:2000], a[:1000] + 1] = hi[:1000]
        # one ulp apart: the division may or may not make them equal
        acc[t[2000:], a[1000:] + 1] = np.nextafter(hi[1000:], np.float32(np.inf))
        want_avg = acc / np.float32(count)
        want_pred = np.argmax(want_avg, axis=-1).astype(np.uint8)
        assert (want_pred[t[1000:2000]] == a[:1000]).all()
        dacc = ctx.from_numpy(acc)
        for with_avg in (True, False):
            avg, pred = Out(ctx, np.float32, (pixels, k)), Out(ctx, np.uint8, (pixels,))
            ctx.call("bsl_tta_finalize", C.c_longlong(pixels), C.c_int(k), C.c_int(count), dacc.p,
                     avg.p if with_avg else None, pred.p, ctx.stream)
            if with_avg:
                assert np.array_equal(_bits(avg.get()), _bits(want_avg)), count
            else:
                raw = avg.buf.download(np.uint8, (avg.nbytes + GUARD,))
                assert (raw == POISON).all(), "avg_prob written although it is NULL"
            assert np.array_equal(pred.get(), want_pred), (count, with_avg)
            avg.free()
            pred.free()
        dacc.free()


@pytest.mark.parametrize("n", [pytest.param(1000, id="1000"), pytest.param(4 * 64 * 128 * 128, id="cfg4")])
def test_confusion_counts_exact(ctx, n):
    rng = np.random.default_rng(n % 977)
    label_map = rng.integers(0, 4, n, dtype=np.uint8)                  # argmax prediction, classes 0..3
    mask = rng.integers(0, 3, n, dtype=np.uint8)                       # a <Cls>Pred mask; any non-zero counts
    labels = rng.integers(0, 4, n, dtype=np.int32)
    labels[rng.random(n) < 0.05] = 255
    labels[rng.random(n) < 0.02] = -1
    start = np.array([10**12 + 3, 17, 5, 1], np.uint64)                # counts accumulate over batches
    dmap, dmask, dlab = ctx.from_numpy(label_map), ctx.from_numpy(mask), ctx.from_numpy(labels)
    for test_value, ref_value, t, dt in ((-1, 1, mask, dmask), (-1, 2, mask, dmask), (1, 1, label_map, dmap),
                                         (2, 2, label_map, dmap), (3, 3, label_map, dmap), (2, 1, label_map, dmap)):
        cnt = Out(ctx, np.uint64, (4,), init=start)
        ctx.call("bsl_confusion_counts", C.c_longlong(n), dt.p, C.c_int(test_value), dlab.p, C.c_int(ref_value),
                 cnt.p, ctx.stream)
        a = t != 0 if test_value < 0 else t == test_value
        b = labels == ref_value
        want = start + np.array([(a & b).sum(), (a & ~b).sum(), (~a & ~b).sum(), (~a & b).sum()], np.uint64)
        assert np.array_equal(cnt.get(), want), (test_value, ref_value)
        cnt.free()
    for b_ in (dmap, dmask, dlab):
        b_.free()


# ------------------------------------------------------------------ refusals
def test_loss_and_inference_refusals(ctx):
    """Return codes of include/bsl_b200.h for arguments outside what the kernels cover; every refusal comes before any
    launch, so the buffers are never read."""
    lib, h, s = ctx.lib, ctx.h, ctx.stream
    buf = ctx.alloc(1 << 16)
    p = buf.p
    for classes, wtype in ((1, "none"), (5, "none")):
        d = _loss_desc(2, 64, classes, wtype)
        assert lib.bsl_label_counts(h, C.byref(d), p, p, s) == BSL_EUNSUPPORTED, classes
        assert lib.bsl_wxent_fwd_bwd(h, C.byref(d), p, p, p, p, p, p, C.c_size_t(1 << 16), s) == BSL_EUNSUPPORTED
        assert lib.bsl_dice_fwd_bwd(h, C.byref(d), p, p, p, p, C.c_int(0), p, C.c_size_t(1 << 16), s) == \
            BSL_EUNSUPPORTED
        assert lib.bsl_softmax_threshold(h, C.byref(d), p, p, p, p, p, p, s) == BSL_EUNSUPPORTED
    d = _loss_desc(2, 64, 3)
    d.weight_type = 3
    assert lib.bsl_wxent_fwd_bwd(h, C.byref(d), p, p, p, p, p, p, C.c_size_t(1 << 16), s) == BSL_EUNSUPPORTED
    assert lib.bsl_label_counts(h, C.byref(d), p, p, s) == BSL_EUNSUPPORTED
    d = _loss_desc(2, 64, 3)
    short = C.c_size_t(lib.bsl_loss_workspace(h, C.byref(d)) - 1)
    assert lib.bsl_wxent_fwd_bwd(h, C.byref(d), p, p, p, p, p, p, short, s) == BSL_EWORKSPACE
    assert lib.bsl_dice_fwd_bwd(h, C.byref(d), p, p, p, p, C.c_int(0), p, short, s) == BSL_EWORKSPACE
    assert lib.bsl_softmax_threshold(h, C.byref(d), p, None, p, p, p, p, s) == BSL_EINVAL     # ilr needs labels
    dims = (C.c_longlong(1), C.c_int(2), C.c_int(3), C.c_int(4), C.c_int(2))
    assert lib.bsl_flip_f32(h, *dims, C.c_int(1), C.c_int(0), p, p, s) == BSL_EINVAL          # src == dst
    assert lib.bsl_flip_f32(h, *dims, C.c_int(8), C.c_int(0), p, C.c_void_p(buf.ptr + 4096), s) == BSL_EINVAL
    assert lib.bsl_tta_finalize(h, C.c_longlong(16), C.c_int(5), C.c_int(2), p, p, p, s) == BSL_EUNSUPPORTED
    assert lib.bsl_tta_finalize(h, C.c_longlong(16), C.c_int(3), C.c_int(0), p, p, p, s) == BSL_EINVAL
    assert lib.bsl_confusion_counts(h, C.c_longlong(0), p, C.c_int(1), p, C.c_int(1), p, s) == BSL_EINVAL
    ctx.check_device()
    buf.free()
