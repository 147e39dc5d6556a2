"""Op-level parity of the small kernels around the convolutions, at the shapes the engines run them, through the C ABI
the engines call:

  * the pixel-pair packing helpers of UNet3D's full-resolution level (unet3d_engine.py): bsl_gather_f32_bf16 and
    bsl_gather_add2_f32 with the engine's own index tables, bsl_fold_pair_sums, and bsl_add_bf16 (the AddN of L.fork,
    pair view and generic);
  * the logits head bsl_conv2d_head_fprop / _dgrad / _wgrad at UNet's, GUNet's and UNet3D's channel and class counts;
  * GUNet's context MLP (bsl_fc_fwd / _bwd, 200 -> 256 -> 256 -> n_modulator_param with dropout on the hidden layers),
    the guide pyramid (bsl_avgpool2x2_f32), --img_grad (bsl_image_gradients_pack), the in-place backbone dropout
    (bsl_dropout_bf16) and UNetInter --mid_cat's guide pooling (bsl_maxpool2x2_f32_bf16);
  * bsl_scale_f32 (the cross-replica mean of the batch-norm moving statistics) and the refusals of all of them.

Gates are per element. Where numpy's fp32 (or fp64) arithmetic reproduces the kernel's exactly -- gathers, folds,
bf16 additions, poolings, image gradients, dropout, scaling -- the output must be bit-identical. Where the kernel sums
many products in fp32 (head, MLP) the gate is |got - ref64| <= k * ulp(ref64) + m * 2^-24 * sum|terms|, ref64 the fp64
value on the device's own fp32 / bf16 inputs, sum|terms| the fp64 sum of the magnitudes of the summed terms and m at
least the longest chain of fp32 additions the kernel runs for that element; each case reports its worst element as
err_u = max |got - ref64| / (2^-24 * sum|terms|) (for the head's bf16 dx: err_ulp, in bf16 ulps of ref64) and
frac = the largest fraction of the bound used. Every output sits in front of a guard region and, where it is a strided
view, between lanes that must keep a canary; bf16 inputs read through a stride hold NaN in the lanes outside them.

Grid arithmetic in the comments is for 148 SMs: the guide, pooling and head kernels cap at 16 * 148 = 2368 blocks of
256 threads (606 208 threads), the gathers and the scaling at 8 * 148 = 1184 blocks (303 104 threads), the head's
filter-gradient reduction at 4 * 148 = 592 blocks and its bias column sums at 2 * 148 = 296 blocks."""
import ctypes as C
from types import SimpleNamespace as NS

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from boxsegliver_b200.device import bf16_bits_to_f32, f32_to_bf16_bits, round_bf16
from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine
from boxsegliver_b200.unet3d_engine import UNet3DEngine
from oracle import tf_ops as O
from tests.gpu_util import report
from tests.test_gpu_norm_ops import Out, _bf16_strided

pytestmark = pytest.mark.gpu

BSL_EINVAL, BSL_EUNSUPPORTED = -1, -2
U32 = 2.0 ** -24                # unit roundoff of fp32


def _free(*bufs):
    for b in bufs:
        getattr(b, "buf", b).free()            # an Out or a DeviceBuffer


def _ulp32(ref):
    return np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)


def _ulp_bf16(ref):
    return _ulp32(ref) * 65536.0


class Worst:
    """Per-element gate |got - ref| <= k_ulp * ulp(ref) + m * 2^-24 * absum, checked chunk by chunk; keeps the worst
    element's error in units of 2^-24 * absum (err_u), or with ulp=_ulp_bf16 in bf16 ulps of ref (err_ulp)."""

    def __init__(self, tag):
        self.tag, self.err_u, self.frac, self.unit = tag, 0.0, 0.0, "err_u"

    def check(self, got, ref, absum, m, k_ulp=2.0, ulp=_ulp32):
        got = np.asarray(got, np.float64)
        assert got.shape == ref.shape, (self.tag, got.shape, ref.shape)
        assert np.isfinite(got).all(), f"{self.tag}: non-finite output"
        err = np.abs(got - ref)
        bound = k_ulp * ulp(ref) + m * U32 * absum
        frac = err / np.maximum(bound, 1e-300)
        i = int(np.argmax(frac))
        assert frac.flat[i] <= 1.0, (f"{self.tag}: element {np.unravel_index(i, ref.shape)}: got {got.flat[i]!r}, "
                                     f"fp64 {ref.flat[i]!r}, bound {bound.flat[i]:.3e}")
        self.frac = max(self.frac, float(frac.flat[i]))
        if ulp is _ulp_bf16:
            self.unit = "err_ulp"
            self.err_u = max(self.err_u, float((err / ulp(ref)).max()))
        else:
            self.err_u = max(self.err_u, float((err / np.maximum(U32 * absum, 1e-300)).max()))

    def numbers(self):
        return {f"{self.tag}_{self.unit}": self.err_u, f"{self.tag}_frac": self.frac}


# ------------------------------------------------------------------ pixel-pair packing: gathers, engine tables
# The level-0 layers of UNet3D's pixel-pair packed level (unet3d_engine.py _build_layers, cpb): 30 channels stored in 32
# lanes, master filters (3, 3, cinp, coutp) / (cinp, coutp) for the stem.
PAIR_LAYERS = {
    "conv": NS(pair="conv", cinp=32, coutp=32),                    # conv_e0/conv2, conv_d0/conv2
    "catpair": NS(pair="conv", catpair=True, cinp=64, coutp=32),   # conv_d0/conv1 over the [enc | up] concat buffer
    "strided": NS(pair="strided", cinp=32, coutp=64),              # conv_e1/conv1, leaving the packed level
    "stem": NS(pair="stem", cinp=32, coutp=32),                    # the im2col GEMM of conv_e0/conv1
}


def _pair_table(name):
    """(idx, msize): the engine's super-filter index table and the master filter size. "grid" is no engine layer: every
    element of a 150 001-element master copied twice among 400 002 entries, more than the 303 104 threads of the
    capped grid, so the grid-stride loops of both gathers turn."""
    if name == "grid":
        msize = 150001
        rng = np.random.default_rng(11)
        idx = rng.permutation(np.concatenate((np.arange(msize), np.arange(msize), np.full(100000, -1))))
        return idx, msize
    L = PAIR_LAYERS[name]
    msize = L.cinp * L.coutp * (1 if L.pair == "stem" else 9)
    return UNet3DEngine._super_index(L).ravel(), msize


@pytest.mark.parametrize("name", list(PAIR_LAYERS) + ["grid"])
def test_pair_packing_gathers(ctx, name):
    """bsl_gather_f32_bf16 == bf16(w[idx]) (0 where idx < 0) and bsl_gather_add2_f32 == g[a] + g[b] in fp32, bit for
    bit, with the tables unet3d_engine builds; and in fp64 the fold is the adjoint of the gather,
    <gather(w), G> == <w, fold(G)> to the fp32 rounding of the fold."""
    idx, msize = _pair_table(name)
    fold = UNet3DEngine._fold_table(idx, msize)
    rng = np.random.default_rng(len(name) * 7 + msize)
    w = rng.standard_normal(msize, dtype=np.float32) * np.float32(0.05)      # full fp32 mantissas: rounding matters
    g = rng.standard_normal(idx.size, dtype=np.float32)                      # super-filter gradient, every element
    bw, bg = ctx.from_numpy(w), ctx.from_numpy(g)
    bidx, bfold = ctx.from_numpy(idx.astype(np.int32)), ctx.from_numpy(fold)
    sup, red = Out(ctx, 1, idx.size, esize=2), Out(ctx, 1, msize, esize=4)
    ctx.call("bsl_gather_f32_bf16", bw.p, bidx.p, C.c_size_t(idx.size), sup.p, ctx.stream)
    ctx.call("bsl_gather_add2_f32", bg.p, bfold.p, C.c_size_t(msize), red.p, ctx.stream)
    got_sup, got_red = sup.raw().ravel(), red.raw().ravel()
    want_sup = f32_to_bf16_bits(np.where(idx >= 0, w[np.maximum(idx, 0)], np.float32(0)))
    assert np.array_equal(got_sup, want_sup), f"{name}: {int((got_sup != want_sup).sum())} super-filter elements differ"
    gz = np.append(g, np.float32(0))                                         # index -1 -> the appended zero
    want_red = (gz[fold[:, 0]] + gz[fold[:, 1]]).astype(np.float32)
    assert np.array_equal(got_red, want_red.view(np.uint32)), \
        f"{name}: {int((got_red != want_red.view(np.uint32)).sum())} folded gradient elements differ"
    sup64 = bf16_bits_to_f32(got_sup).astype(np.float64)
    red64 = got_red.view(np.float32).astype(np.float64)
    wb = round_bf16(w).astype(np.float64)
    lhs, rhs = float(sup64 @ g.astype(np.float64)), float(wb @ red64)
    bound = U32 * float(np.abs(wb) @ np.abs(red64)) + 1e-12 * float(np.abs(sup64) @ np.abs(g.astype(np.float64)))
    assert abs(lhs - rhs) <= bound, (name, lhs, rhs, bound)
    report(f"pair gathers {name}", entries=int(idx.size), master=int(msize), adjoint_gap=abs(lhs - rhs), bound=bound)
    _free(bw, bg, bidx, bfold, sup, red)


@pytest.mark.parametrize("groups,c", [(1, 32), (1, 64), (4, 32), (4, 64)])
def test_fold_pair_sums(ctx, groups, c):
    """fp64 [groups][2][2c] -> [groups][2][c], dst = src[.., ch] + src[.., c + ch]: batch norm (one group) and instance
    norm (one group per volume, 4 volumes as UNet3D's batch) at the 32 lanes of the packed level and 64 lanes. One
    fp64 addition per element, so bit for bit."""
    rng = np.random.default_rng(groups * 100 + c)
    src = rng.standard_normal((groups, 2, 2 * c)) * np.exp(rng.uniform(-3, 12, (groups, 2, 2 * c)))
    bs = ctx.from_numpy(src)
    out = Out(ctx, groups * 2, c, esize=8)
    ctx.call("bsl_fold_pair_sums", bs.p, C.c_int(groups), C.c_int(c), out.p, ctx.stream)
    want = (src[..., :c] + src[..., c:]).reshape(groups * 2, c)
    assert np.array_equal(out.raw(), want.view(np.uint64))
    _free(bs, out)


# ------------------------------------------------------------------ AddN of the skip and strided-conv gradients
# ew_plan: threads = 256 // (c / 8) rows of c / 8 channel groups, want = pixels / (2 rows) blocks, cap 2368; the grid
# stride is blocks * rows pixels and no pixel count below is a multiple of it.
ADD_CASES = [
    # UNet3D level 0 (L.fork with a PairView, 3 x 24 x 80 x 96 voxels): 276 480 voxel pairs, 64 dense lanes + the
    # encoder half of the 128-lane concat gradient. 32 rows x 2368 blocks = 75 776 pixels per trip, 3.6 trips
    pytest.param(dict(pixels=3 * 24 * 80 * 96 // 2, c=64, a_ld=64, b_ld=128, out_ld=64), id="pair-view"),
    # the generic call, b = the concat gradient of pitch 2c
    pytest.param(dict(pixels=3 * 24 * 80 * 96, c=64, a_ld=64, b_ld=128, out_ld=64), id="c64"),       # 7.3 trips
    pytest.param(dict(pixels=3 * 24 * 40 * 48, c=128, a_ld=128, b_ld=256, out_ld=128), id="c128"),   # 16 rows, 3.6
    pytest.param(dict(pixels=3 * 24 * 40 * 48, c=256, a_ld=256, b_ld=512, out_ld=256), id="c256"),   # 8 rows, 7.3
    # c = 320: 40 channel groups -> 6 rows, 240-thread blocks; 14 208 pixels per trip, 2.2 trips
    pytest.param(dict(pixels=2 * 9 * 40 * 44, c=320, a_ld=320, b_ld=640, out_ld=320), id="c320"),
    # strided a and out: lanes [c, out_ld) of out must keep their canary
    pytest.param(dict(pixels=2 * 9 * 40 * 44, c=320, a_ld=328, b_ld=640, out_ld=384), id="c320-strided"),
]


@pytest.mark.parametrize("cs", ADD_CASES)
def test_add_bf16(ctx, cs):
    """out = bf16(fp32(a) + fp32(b)) bit for bit over channel-strided views; nothing outside lanes [0, c) of out."""
    P, c = cs["pixels"], cs["c"]
    rng = np.random.default_rng(P + c)
    scale = np.exp2(rng.integers(-6, 3, (P, 1))).astype(np.float32)         # per-pixel magnitudes 2^-6 .. 2^2
    a = round_bf16(rng.standard_normal((P, c), dtype=np.float32) * scale)
    b = round_bf16(rng.standard_normal((P, c), dtype=np.float32))
    ba, bb = _bf16_strided(ctx, a, cs["a_ld"], np.nan), _bf16_strided(ctx, b, cs["b_ld"], np.nan)
    out = Out(ctx, P, c, ld=cs["out_ld"], esize=2)
    ctx.call("bsl_add_bf16", C.c_longlong(P), C.c_int(c), ba.p, C.c_int(cs["a_ld"]), bb.p, C.c_int(cs["b_ld"]), out.p,
             C.c_int(cs["out_ld"]), ctx.stream)
    got, want = out.raw(), f32_to_bf16_bits(a + b).reshape(P, c)
    assert np.array_equal(got, want), f"{int((got != want).sum())} of {got.size} sums differ"
    _free(ba, bb, out)


# ------------------------------------------------------------------ GUNet --img_grad input
@pytest.mark.parametrize("n,h,w,c", [(4, 512, 512, 1), (4, 512, 512, 3), (3, 37, 53, 3)])
def test_image_gradients_pack(ctx, n, h, w, c):
    """Lanes [0, 3c) of 64-lane rows = bf16(x), bf16(x[y + 1] - x[y]), bf16(x[x + 1] - x[x]) with the differences in
    fp32 and zero in the last row / column (tf.image.image_gradients); lanes [3c, 64) untouched. 4 x 512 x 512 is
    GUNet's training size (3.1 M elements at c = 3: 5.2 trips of the capped grid); 37 x 53 is ragged."""
    rng = np.random.default_rng(n * h * w + c)
    x = rng.standard_normal((n, h, w, c), dtype=np.float32)
    bx = ctx.from_numpy(x)
    out = Out(ctx, n * h * w, 3 * c, ld=64, esize=2)
    ctx.call("bsl_image_gradients_pack", C.c_int(n), C.c_int(h), C.c_int(w), C.c_int(c), bx.p, out.p, C.c_int(64),
             ctx.stream)
    dy, dx = O.image_gradients(x)           # numpy fp32 subtractions, as the kernel's
    assert dy.dtype == np.float32 and dx.dtype == np.float32
    want = f32_to_bf16_bits(np.concatenate((x, dy, dx), axis=-1)).reshape(n * h * w, 3 * c)
    got = out.raw()
    assert np.array_equal(got, want), f"{int((got != want).sum())} of {got.size} lanes differ"
    _free(bx, out)


# ------------------------------------------------------------------ UNetInter --mid_cat guide pooling
@pytest.mark.parametrize("g", [1, 2])
def test_maxpool_guide_into_pooled_lanes(ctx, g):
    """The guide's lanes [64, 64 + g) of the 128-lane pooled buffer of UNetInter's first block (64 activation channels +
    g guide channels, padded to 128): bf16(max of the 2x2 window), every other lane keeps its canary. 20 x 256 x 256
    (655 360 outputs at g = 2: 1.1 trips of the capped grid); ties between window elements included."""
    n, h, w, cout = 20, 256, 256, 64
    rng = np.random.default_rng(40 + g)
    x = rng.uniform(-1, 1, (n, h, w, g)).astype(np.float32)
    x[:, ::7, ::2] = x[:, ::7, 1::2]                          # exact ties inside some windows
    bx = ctx.from_numpy(x)
    out = Out(ctx, n * (h // 2) * (w // 2), g, ld=128, off=cout, esize=2)
    ctx.call("bsl_maxpool2x2_f32_bf16", C.c_int(n), C.c_int(h), C.c_int(w), C.c_int(g), bx.p, out.p, C.c_int(128),
             ctx.stream)
    want = f32_to_bf16_bits(O.max_pool_2x2(x)).reshape(-1, g)
    got = out.raw()
    assert np.array_equal(got, want), f"{int((got != want).sum())} of {got.size} pooled guide values differ"
    _free(bx, out)


# ------------------------------------------------------------------ GUNet guide pyramid
@pytest.mark.parametrize("g", [1, 2])
def test_avgpool_guide_pyramid(ctx, g):
    """The four slim.avg_pool2d levels a GUNet cfg3 step runs (batch 32, 512 -> 256 -> 128 -> 64 -> 32), chained on the
    device as gunet_engine.forward does; each level bit for bit ((p00 + p01) + (p10 + p11)) * 0.25 in fp32. The first
    level has 2.1 M * g outputs, 3.5 * g trips of the 606 208 threads of the capped grid."""
    n, hw = 32, 512
    rng = np.random.default_rng(50 + g)
    x = rng.uniform(0.5, 1.0, (n, hw, hw, g)).astype(np.float32)
    src = ctx.from_numpy(x)
    bufs = [src]
    for level in range(4):
        ho = hw >> (level + 1)
        out = Out(ctx, n * ho * ho, g)
        ctx.call("bsl_avgpool2x2_f32", C.c_int(n), C.c_int(2 * ho), C.c_int(2 * ho), C.c_int(g), bufs[-1].p, out.p,
                 ctx.stream)
        r = x.reshape(n, ho, 2, ho, 2, g)
        x = ((r[:, :, 0, :, 0] + r[:, :, 0, :, 1]) + (r[:, :, 1, :, 0] + r[:, :, 1, :, 1])) * np.float32(0.25)
        assert x.dtype == np.float32
        got = out.raw()
        assert np.array_equal(got, x.reshape(-1, g).view(np.uint32)), \
            f"level {level + 1}: {int((got != x.reshape(-1, g).view(np.uint32)).sum())} values differ"
        bufs.append(out.buf)
    _free(*bufs)


# ------------------------------------------------------------------ backbone --dropout, in place
def _multipliers(start, stop, keep, seed, offset):
    """O.dropout_multipliers(stop, keep, seed, offset)[start:stop] for start % 4 == 0, with one Philox call per counter
    instead of one per element (the test checks the two agree)."""
    blk = np.arange(start // 4, (stop + 3) // 4, dtype=np.uint64)
    off = np.full(blk.size, offset, np.uint64)
    lo = np.uint64(0xFFFFFFFF)
    ctr = np.stack([blk & lo, blk >> np.uint64(32), off & lo, off >> np.uint64(32)], axis=-1).astype(np.uint32)
    words = O.philox4x32_10(ctr, np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32)).ravel()[:stop - start]
    u = ((words & np.uint32(0x7FFFFF)) | np.uint32(0x3F800000)).view(np.float32) - np.float32(1.0)
    k = np.float32(keep)
    return np.where(np.floor(k + u) >= 1.0, np.float32(1.0) / k, np.float32(0.0)).astype(np.float32)


# (pixels, c, level, --dropout) of GUNet cfg3 layers (batch 32 at 512 x 512). The 64-channel case runs 32 x 128 x 128
# pixels, not the 32 x 512 x 512 of level 0, whose 537 M elements would keep the host's Philox busy for a minute.
DROP_CASES = [
    pytest.param(32 * 128 * 128, 64, 0, 0.3, id="c64"),     # 4.2 M 8-lane items: 6.9 trips of the capped grid
    pytest.param(32 * 64 * 64, 512, 3, 0.5, id="c512"),     # level 3: 8.4 M items, 13.8 trips
    pytest.param(32 * 32 * 32, 1024, 4, 0.3, id="c1024"),   # the bridge: 4.2 M items
]


@pytest.mark.parametrize("pixels,c,level,rate", DROP_CASES)
def test_dropout_bf16_in_place(ctx, pixels, c, level, rate):
    """bsl_dropout_bf16 with x == out, as gunet_engine calls it forward and backward: bf16(x * multiplier(p * c + ch))
    bit for bit, the descriptor built by the engine's _drop_desc at a step whose counter offset is above 2^32."""
    eng = NS(cfg=GUNetConfig(batch=32, dropout=rate, dropout_seed=0x5EED0000ABC), step_count=(1 << 28) + 3)
    d = GUNetEngine._drop_desc(eng, NS(level=level))
    assert d.offset > 1 << 32 and d.seed > 1 << 32
    keep, seed, offset = d.keep_prob, d.seed, d.offset
    assert np.array_equal(_multipliers(0, 4096, keep, seed, offset), O.dropout_multipliers(4096, keep, seed, offset))
    assert np.array_equal(_multipliers(1024, 3000, keep, seed, offset),
                          O.dropout_multipliers(3000, keep, seed, offset)[1024:])
    rng = np.random.default_rng(c)
    x = f32_to_bf16_bits(rng.standard_normal((pixels, c), dtype=np.float32))
    buf = Out(ctx, pixels, c, esize=2, init=x)
    ctx.call("bsl_dropout_bf16", C.byref(d), C.c_longlong(pixels), C.c_int(c), buf.p, C.c_int(c), buf.p, C.c_int(c),
             ctx.stream)
    got = buf.raw()
    step = (1 << 22) // c                                   # pixels per host chunk
    bad = 0
    for p0 in range(0, pixels, step):
        p1 = min(pixels, p0 + step)
        m = _multipliers(p0 * c, p1 * c, keep, seed, offset).reshape(p1 - p0, c)
        want = f32_to_bf16_bits(bf16_bits_to_f32(x[p0:p1]).reshape(p1 - p0, c) * m).reshape(p1 - p0, c)
        bad += int((got[p0:p1] != want).sum())
    assert bad == 0, f"{bad} of {got.size} elements differ"
    _free(buf)


# ------------------------------------------------------------------ GUNet context MLP
STEP = 41     # the engine's step counter: dropout offsets 16 * 42 + layer


@pytest.mark.parametrize("n", [2, 32])
def test_context_mlp_at_gunet_dimensions(ctx, n):
    """slim_nets.mlp of GUNet.yml: 200 -> 256 -> 256 -> n_modulator_param (3840), ReLU + dropout (keep 0.5) on the
    hidden layers, with the descriptors of gunet_engine._fc_desc; forward in order, then backward in reverse with
    dx = NULL on the first layer, each call fed the device's own outputs of the previous one. Per element against fp64
    (O.fully_connected_grad) with the Philox masks of O.dropout_multipliers."""
    cfg = GUNetConfig(batch=n)
    assert cfg.n_modulator_param == 3840
    specs = GUNetEngine._fc_specs(NS(cfg=cfg))
    assert [s[1:] for s in specs] == [(200, 256, True), (256, 256, True), (256, 3840, False)]
    eng = NS(cfg=cfg, step_count=STEP)
    descs = [GUNetEngine._fc_desc(eng, cin, cout, hidden, k, True) for k, (_, cin, cout, hidden) in enumerate(specs)]
    rng = np.random.default_rng(60 + n)
    x = rng.random((n, 200), dtype=np.float32)                   # the context: histogram features in [0, 1)
    W, bufs, hosts, mults, ys = [], [], [x], [], []
    for k, (_, cin, cout, hidden) in enumerate(specs):
        lim = np.float32(np.sqrt(6.0 / (cin + cout)))
        w = rng.uniform(-lim, lim, (cin, cout)).astype(np.float32)
        b = rng.standard_normal(cout, dtype=np.float32) * np.float32(0.1)
        W.append((w, b))
        bufs.append((ctx.from_numpy(w), ctx.from_numpy(b)))
    checks = {}
    inp = ctx.from_numpy(x)
    ins = [inp]
    for k, ((_, cin, cout, hidden), d) in enumerate(zip(specs, descs)):
        assert bool(d.use_dropout) == hidden and bool(d.relu) == hidden
        y = Out(ctx, n, cout)
        ctx.call("bsl_fc_fwd", C.byref(d), ins[-1].p, bufs[k][0].p, bufs[k][1].p, y.p, ctx.stream)
        got = y.get()
        m = (O.dropout_multipliers(n * cout, d.dropout.keep_prob, d.dropout.seed, d.dropout.offset).reshape(n, cout)
             if d.use_dropout else np.ones((n, cout), np.float32)).astype(np.float64)
        x64, w64, b64 = hosts[-1].astype(np.float64), W[k][0].astype(np.float64), W[k][1].astype(np.float64)
        pre = x64 @ w64 + b64
        ref = (np.maximum(pre, 0.0) if d.relu else pre) * m
        wk = checks.setdefault(f"y{k}", Worst(f"y{k}"))
        wk.check(got, ref, (np.abs(x64) @ np.abs(w64) + np.abs(b64)) * m, m=cin + 1)
        mults.append(m)
        ys.append(y)
        hosts.append(got)
        ins.append(y.buf)
    dy = rng.standard_normal((n, 3840), dtype=np.float32)
    bdy, dy_host = ctx.from_numpy(dy), dy
    grads = [bdy]
    for k in reversed(range(len(specs))):
        _, cin, cout, hidden = specs[k]
        d = descs[k]
        ws_bytes = ctx.lib.bsl_fc_bwd_workspace(ctx.h, C.byref(d))
        assert ws_bytes >= n * cout * 4
        ws = ctx.alloc(ws_bytes)
        dx = Out(ctx, n, cin) if k > 0 else None
        dw, db = Out(ctx, cin, cout), Out(ctx, 1, cout)
        ctx.call("bsl_fc_bwd", C.byref(d), ins[k].p, bufs[k][0].p, ys[k].p, bdy.p, dx.p if dx else None, dw.p, db.p,
                 ws.p, C.c_size_t(ws_bytes), ctx.stream)
        # d(out)/d(pre) = multiplier where the stored output is > 0 (the forward check pinned those to kept, pre > 0)
        gate = mults[k] * (hosts[k + 1] > 0) if d.relu else mults[k]
        dpre = dy_host.astype(np.float64) * gate
        x64, w64 = hosts[k].astype(np.float64), W[k][0].astype(np.float64)
        g_dx, g_dw, g_db = O.fully_connected_grad(x64, w64, dpre)
        checks.setdefault(f"dw{k}", Worst(f"dw{k}")).check(dw.get(), g_dw, np.abs(x64).T @ np.abs(dpre), m=n + 1)
        checks.setdefault(f"db{k}", Worst(f"db{k}")).check(db.get()[0], g_db, np.abs(dpre).sum(axis=0), m=n + 1)
        if dx is not None:
            got_dx = dx.get()
            # lanes of a warp stride over cout, then a 5-level shuffle tree
            checks.setdefault(f"dx{k}", Worst(f"dx{k}")).check(got_dx, g_dx, np.abs(dpre) @ np.abs(w64).T,
                                                                m=cout // 32 + 6)
            bdy, dy_host = dx.buf, got_dx
            grads.append(bdy)
        _free(ws, dw, db)
    numbers = {}
    for wk in checks.values():
        numbers.update(wk.numbers())
    report(f"context mlp n={n}", **numbers)
    _free(inp, *[b for pair in bufs for b in pair], *ys, *grads)


# ------------------------------------------------------------------ logits head
HEAD_CASES = [
    # UNet / GUNet AdjustChannels: 64 -> 3 classes; 129 600 px: 2368 blocks x 32 px = 75 776 px per trip, 1.7 trips
    pytest.param(dict(n=3, h=200, w=216, cin=64, classes=3, x_ld=64), id="cin64-k3"),
    # UNet3D logits on the pixel-pair level: cpb(30, "conv_d0") = 32 lanes, 2 classes, 4 x 16 x 128 x 131 voxels =
    # 1 073 152 px. 4-lane shuffle groups, 64 px per block, 151 552 px per trip: the second U = 4 round is partial
    # (1.77 rounds). Filter gradient: 592 blocks of 1813 px
    pytest.param(dict(n=4 * 16, h=128, w=131, cin=32, classes=2, x_ld=32), id="cin32-k2-1M"),
    # 128 of the 192 lanes of a wider buffer, 4 classes, 16-lane shuffle groups
    pytest.param(dict(n=2, h=96, w=100, cin=128, classes=4, x_ld=192), id="cin128-k4-ld192"),
]


@pytest.mark.parametrize("cs", HEAD_CASES)
def test_logits_head_at_engine_shapes(ctx, cs):
    """logits = x @ w + b (fp32 [P, classes]), dx = bf16(dlogits @ w^T) written into lanes [0, cin) of x_ld-lane rows,
    dw = x^T @ dlogits and db = sum dlogits. Lanes of x beyond cin hold bf16 NaN (a read of them shows); lanes of dx
    beyond cin keep their canary. Gates: logits 2 ulp + 16 * 2^-24 * (sum|x w| + |b|) (8 products per lane, <= 5
    shuffle levels, the bias); dx 1 bf16 ulp + 4 * 2^-24 * sum|dl w| (the fp32 dot product before the rounding); dw
    and db 128 * 2^-24 * sum|x dl|, resp. sum|dl| (the longest fp32 chain is about 100 additions: a thread's pixels
    and the rows of its block, resp. a thread's rows, 5 shuffle levels and 8 warps; the blocks are added in fp64)."""
    n, h, w_, cin, K, x_ld = cs["n"], cs["h"], cs["w"], cs["cin"], cs["classes"], cs["x_ld"]
    P = n * h * w_
    rng = np.random.default_rng(P + cin + K)
    x = round_bf16(rng.standard_normal((P, cin), dtype=np.float32))
    w = rng.standard_normal((cin, K), dtype=np.float32) * np.float32(0.1)
    b = rng.standard_normal(K, dtype=np.float32)
    dl = rng.standard_normal((P, K), dtype=np.float32) * np.float32(0.3)
    bx, bw, bb, bdl = _bf16_strided(ctx, x, x_ld, np.nan), ctx.from_numpy(w), ctx.from_numpy(b), ctx.from_numpy(dl)
    d = _lib.Conv2dDesc(n, h, w_, cin, K, 1, 1, x_ld, K)
    logits, dx = Out(ctx, P, K), Out(ctx, P, cin, ld=x_ld, esize=2)
    dw, db = Out(ctx, cin, K), Out(ctx, 1, K)
    ctx.call("bsl_conv2d_head_fprop", C.byref(d), bx.p, bw.p, bb.p, logits.p, ctx.stream)
    ctx.call("bsl_conv2d_head_dgrad", C.byref(d), bdl.p, bw.p, dx.p, ctx.stream)
    ctx.call("bsl_conv2d_head_wgrad", C.byref(d), bx.p, bdl.p, dw.p, db.p, ctx.stream)
    got_l, got_dx = logits.get(), dx.get()
    w64, b64, aw = w.astype(np.float64), b.astype(np.float64), np.abs(w.astype(np.float64))
    wl, wd = Worst("logits"), Worst("dx")
    chunk = 1 << 18
    for p0 in range(0, P, chunk):
        x64, dl64 = x[p0:p0 + chunk].astype(np.float64), dl[p0:p0 + chunk].astype(np.float64)
        wl.check(got_l[p0:p0 + chunk], x64 @ w64 + b64, np.abs(x64) @ aw + np.abs(b64), m=16)
        wd.check(got_dx[p0:p0 + chunk], dl64 @ w64.T, np.abs(dl64) @ aw.T, m=4, k_ulp=1.0, ulp=_ulp_bf16)
    x64, dl64 = x.astype(np.float64), dl.astype(np.float64)
    ww, wb = Worst("dw"), Worst("db")
    ww.check(dw.get(), x64.T @ dl64, np.abs(x64).T @ np.abs(dl64), m=128, k_ulp=1.0)
    wb.check(db.get()[0], dl64.sum(axis=0), np.abs(dl64).sum(axis=0), m=128, k_ulp=1.0)
    report(f"logits head P={P} cin={cin} classes={K} x_ld={x_ld}", **wl.numbers(), **wd.numbers(), **ww.numbers(),
           **wb.numbers())
    _free(bx, bw, bb, bdl, logits, dx, dw, db)


# ------------------------------------------------------------------ cross-replica mean of the moving statistics
@pytest.mark.parametrize("world", [8, 3])
def test_scale_f32_in_place(ctx, world):
    """bsl_scale_f32(x, 1 / world) after the SUM all-reduce of the moving statistics (engine.py, unet3d_engine.py):
    x * fp32(1 / world) bit for bit over 1 000 003 values (3.3 trips of the 303 104-thread grid)."""
    rng = np.random.default_rng(world)
    x = rng.standard_normal(1000003, dtype=np.float32) * np.float32(world)
    buf = Out(ctx, 1, x.size, init=x)
    a = np.float32(1.0 / world)
    ctx.call("bsl_scale_f32", buf.p, C.c_size_t(x.size), C.c_float(a), ctx.stream)
    assert np.array_equal(buf.raw()[0], (x * a).view(np.uint32))
    _free(buf)


# ------------------------------------------------------------------ refusals
def test_aux_refusals(ctx):
    """Return codes of malformed calls; every refusal comes before any launch, so the buffers are never read."""
    lib, h, s = ctx.lib, ctx.h, ctx.stream
    buf = ctx.alloc(1 << 16)
    p = buf.p
    i = C.c_int
    for hh, ww in ((7, 8), (8, 7)):
        assert lib.bsl_avgpool2x2_f32(h, i(2), i(hh), i(ww), i(1), p, p, s) == BSL_EUNSUPPORTED, (hh, ww)
        assert lib.bsl_maxpool2x2_f32_bf16(h, i(2), i(hh), i(ww), i(1), p, p, i(128), s) == BSL_EUNSUPPORTED, (hh, ww)
    assert lib.bsl_maxpool2x2_f32_bf16(h, i(2), i(8), i(8), i(2), p, p, i(1), s) == BSL_EUNSUPPORTED
    assert lib.bsl_image_gradients_pack(h, i(2), i(8), i(8), i(3), p, p, i(8), s) == BSL_EINVAL
    assert lib.bsl_image_gradients_pack(h, i(2), i(8), i(8), i(1), p, p, i(2), s) == BSL_EINVAL
    ll = C.c_longlong
    assert lib.bsl_add_bf16(h, ll(16), i(60), p, i(64), p, i(128), p, i(64), s) == BSL_EUNSUPPORTED
    assert lib.bsl_add_bf16(h, ll(16), i(64), p, i(68), p, i(128), p, i(64), s) == BSL_EUNSUPPORTED
    assert lib.bsl_add_bf16(h, ll(16), i(64), p, i(64), p, i(132), p, i(64), s) == BSL_EUNSUPPORTED
    assert lib.bsl_add_bf16(h, ll(16), i(64), p, i(64), p, i(128), p, i(100), s) == BSL_EUNSUPPORTED
    assert lib.bsl_fold_pair_sums(h, p, i(0), i(32), p, s) == BSL_EINVAL
    assert lib.bsl_fold_pair_sums(h, p, i(1), i(0), p, s) == BSL_EINVAL
    d = _lib.DropoutDesc(0.5, 1, 2)
    assert lib.bsl_dropout_bf16(h, C.byref(d), ll(16), i(20), p, i(24), p, i(24), s) == BSL_EUNSUPPORTED
    for cin, classes, x_ld in ((48, 2, 48), (64, 5, 64), (64, 3, 56), (512, 2, 512)):
        dd = _lib.Conv2dDesc(1, 4, 4, cin, classes, 1, 1, x_ld, classes)
        assert lib.bsl_conv2d_head_fprop(h, C.byref(dd), p, p, p, p, s) == BSL_EUNSUPPORTED, (cin, classes, x_ld)
        assert lib.bsl_conv2d_head_dgrad(h, C.byref(dd), p, p, p, s) == BSL_EUNSUPPORTED, (cin, classes, x_ld)
        assert lib.bsl_conv2d_head_wgrad(h, C.byref(dd), p, p, p, p, s) == BSL_EUNSUPPORTED, (cin, classes, x_ld)
    ctx.check_device()
    buf.free()
