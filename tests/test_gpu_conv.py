"""Parity of the tcgen05 implicit-GEMM convolutions (through the C ABI) against the numpy oracle."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from oracle import tf_ops as O
from tests.gpu_util import TOL_BF16, TOL_F32, bf16_randn, padded, rel

pytestmark = pytest.mark.gpu

CONV_CASES = [
    # n, h, w, cin, cout, k, x_ld, y_ld
    (2, 16, 16, 64, 64, 3, None, None),      # column tile 64
    (1, 16, 16, 128, 128, 3, None, None),    # column tile 128, two k-blocks per tap
    (1, 8, 16, 64, 256, 3, None, None),      # column tile 256
    (1, 16, 16, 256, 64, 3, None, None),
    (2, 12, 20, 64, 128, 3, None, None),     # ragged spatial size: out-of-bounds rows masked
    (3, 4, 4, 128, 64, 3, None, None),       # box spans several images
    (2, 16, 16, 64, 64, 3, 128, 192),        # skip-concat views (channel stride > channels)
    (2, 16, 16, 128, 64, 1, None, None),     # 1x1
    (1, 2, 2, 1024, 1024, 3, None, None),    # bridge layer of a 32x32 input
    # halo-tile kernels (w % 8 == 0, h % 16 == 0): one TMA box + 9 shifted UMMA descriptors
    (2, 32, 32, 128, 64, 3, None, None),     # Decode1/conv1 shape class: 2 k-blocks, column tile 64, sub-tile pairs
    (3, 16, 24, 64, 192, 3, None, None),     # odd number of sub-tiles (single sub-tile units), 3 column tiles of 64
    (2, 32, 16, 64, 256, 3, None, None),     # column tile 128 x 2
    (1, 48, 40, 192, 128, 3, 256, 192),      # concat views, 3 k-blocks, wgrad tiles of 16 x 4
    (4, 16, 16, 512, 64, 3, None, None),     # long reduction (8 k-blocks): ring wrap-around of both pipelines
    (5, 16, 32, 64, 64, 1, None, None),      # 1x1 through the 1-tap path (stem after im2col)
    (2, 64, 64, 64, 64, 3, None, None),      # many tiles per CTA? no: 64 sub-tiles; wgrad split over pixel tiles
    # ragged extents on the halo-tile kernels (ceil(extent / tile) tiles, masked edge rows): the deep levels of the shipped
    # 960 x 320 / 512 x 160 / 480 x 160 scripts
    (1, 60, 20, 256, 256, 3, None, None),    # level 4 of 960 x 320: column tile 256, TMA-store epilogue clips the edge
    (2, 20, 12, 128, 128, 3, None, None),    # 20 x 12: both extents ragged, wide filter-gradient kernel
    (2, 30, 40, 64, 64, 3, None, None),      # level 3 of 480 x 160 / 2: resident filter, column tile 64
    (1, 24, 36, 128, 64, 3, 192, 128),       # ragged + concat views
    (3, 10, 8, 64, 128, 1, None, None),      # 1x1, ragged rows
    # CTA pairs (cta_group::2, 128-wide tiles): sub-tile count a multiple of 4, several column tiles, reductions long
    # enough to wrap both operand rings; filter gradient with 4 / 8 input blocks per class-b CTA pair
    (2, 32, 32, 256, 512, 3, None, None),    # fprop: 4 column tiles x 4 k-blocks; dgrad: 2 column tiles x 8 k-blocks
    (4, 16, 16, 128, 256, 3, 192, 320),      # pairs writing into / reading from concat views
]


GUARD = np.full(8192, 0xABCD, np.uint16)


def guarded(ctx, nbytes):
    """Zeroed device buffer of `nbytes` followed by a canary region (edge tiles must not store past the tensor)."""
    return ctx.alloc(nbytes + GUARD.nbytes).zero().upload(GUARD, byte_offset=nbytes)


def guard_intact(buf, nbytes):
    return np.array_equal(buf.download(np.uint16, GUARD.shape, byte_offset=nbytes), GUARD)


@pytest.mark.parametrize("n,h,w,cin,cout,k,x_ld,y_ld", CONV_CASES)
def test_conv2d_fprop_dgrad_wgrad(ctx, n, h, w, cin, cout, k, x_ld, y_ld):
    rng = np.random.default_rng(cin * 7 + cout + h)
    x_ld, y_ld = x_ld or cin, y_ld or cout
    x = bf16_randn(rng, (n, h, w, cin))
    wt = bf16_randn(rng, (k, k, cin, cout), 0.05)
    dy = bf16_randn(rng, (n, h, w, cout))
    dx_ = ctx.bf16_from_f32(padded(x, x_ld))
    dw_ = ctx.bf16_from_f32(wt)
    ddy = ctx.bf16_from_f32(padded(dy, y_ld))
    # a canary region behind every output: edge tiles of ragged extents (and of the last image) must not store past it
    guard = np.full(8192, 0xABCD, np.uint16)
    ny, nx = n * h * w * y_ld * 2, n * h * w * x_ld * 2
    yo = ctx.alloc(ny + guard.nbytes).zero().upload(guard, byte_offset=ny)
    dxo = ctx.alloc(nx + guard.nbytes).zero().upload(guard, byte_offset=nx)
    desc = _lib.Conv2dDesc(n, h, w, cin, cout, k, k, x_ld, y_ld)
    x64, w64, dy64 = x.astype(np.float64), wt.astype(np.float64), dy.astype(np.float64)

    def intact(buf, nbytes):
        return np.array_equal(buf.download(np.uint16, guard.shape, byte_offset=nbytes), guard)

    ctx.call("bsl_conv2d_fprop", C.byref(desc), dx_.p, dw_.p, yo.p, ctx.stream)
    ctx.check_device()
    assert intact(yo, ny), "fprop stored past the end of its output"
    got = ctx.bf16_to_f32(yo, (n, h, w, y_ld))
    assert rel(got[..., :cout], O.conv2d(x64, w64)) < TOL_BF16
    assert not got[..., cout:].any(), "fprop wrote outside its channel slice"

    ctx.call("bsl_conv2d_dgrad", C.byref(desc), ddy.p, dw_.p, dxo.p, ctx.stream)
    ctx.check_device()
    assert intact(dxo, nx), "dgrad stored past the end of its output"
    got = ctx.bf16_to_f32(dxo, (n, h, w, x_ld))
    assert rel(got[..., :cin], O.conv2d_backprop_input(x.shape, w64, dy64)) < TOL_BF16
    assert not got[..., cin:].any()

    ws_bytes = ctx.lib.bsl_conv2d_wgrad_workspace(ctx.h, C.byref(desc))
    ws = ctx.alloc(max(ws_bytes, 16))
    dwo = ctx.alloc(k * k * cin * cout * 4).zero()
    ctx.call("bsl_conv2d_wgrad", C.byref(desc), dx_.p, ddy.p, dwo.p, ws.p, C.c_size_t(ws_bytes), ctx.stream)
    ctx.check_device()
    got1 = dwo.download(np.float32, (k, k, cin, cout))
    assert rel(got1, O.conv2d_backprop_filter(x64, wt.shape, dy64)) < TOL_F32
    # split-K partials are reduced in a fixed order: a second run is bit-identical
    ctx.call("bsl_conv2d_wgrad", C.byref(desc), dx_.p, ddy.p, dwo.p, ws.p, C.c_size_t(ws_bytes), ctx.stream)
    assert np.array_equal(got1, dwo.download(np.float32, (k, k, cin, cout)))
    for b in (dx_, dw_, ddy, yo, dxo, ws, dwo):
        b.free()


@pytest.mark.parametrize("n,h,w,cout", [(2, 16, 32, 64), (3, 12, 20, 64), (1, 32, 32, 128)])
def test_conv2d_narrow_rows_equal_zero_padded(ctx, n, h, w, cout):
    """x_ld = 32 < cin = 64 (the stem's 32-column im2col matrix, bsl_stem_im2col_ld): the TMA box is wider than the
    tensor and its upper half is zero-filled, so fprop (+ statistics) and wgrad are bit-identical to the same call on
    a 64-column matrix whose columns 32..63 are zero. Halo-tile and general kernels."""
    rng = np.random.default_rng(h * 3 + cout)
    x = bf16_randn(rng, (n, h, w, 32))
    wt = bf16_randn(rng, (1, 1, 64, cout), 0.05)
    dy = bf16_randn(rng, (n, h, w, cout))
    xn, xw = ctx.bf16_from_f32(x), ctx.bf16_from_f32(padded(x, 64))
    dw_, ddy = ctx.bf16_from_f32(wt), ctx.bf16_from_f32(dy)
    outs = []
    for buf, ld in ((xw, 64), (xn, 32)):
        desc = _lib.Conv2dDesc(n, h, w, 64, cout, 1, 1, ld, cout)
        yo = ctx.alloc(n * h * w * cout * 2).zero()
        sums = ctx.alloc(2 * cout * 8).zero()
        ctx.call("bsl_conv2d_fprop_stats", C.byref(desc), buf.p, dw_.p, yo.p, sums.p, ctx.stream)
        ws_bytes = ctx.lib.bsl_conv2d_wgrad_workspace(ctx.h, C.byref(desc))
        ws = ctx.alloc(max(ws_bytes, 16))
        dwo = ctx.alloc(64 * cout * 4).zero()
        ctx.call("bsl_conv2d_wgrad", C.byref(desc), buf.p, ddy.p, dwo.p, ws.p, C.c_size_t(ws_bytes), ctx.stream)
        ctx.check_device()
        outs.append((yo.download(np.uint16, (n, h, w, cout)), sums.download(np.float64, (2, cout)),
                     dwo.download(np.float32, (64, cout))))
        for b in (yo, sums, ws, dwo):
            b.free()
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    assert rel(ctx_bf16(outs[1][0]), O.conv2d(x.astype(np.float64), wt[:, :, :32].astype(np.float64))) < TOL_BF16
    assert not outs[1][2][32:].any(), "filter-gradient rows of the zero-filled channels must be zero"
    # dgrad writes x_ld-pitched rows: a narrow pitch is rejected there
    desc = _lib.Conv2dDesc(n, h, w, 64, cout, 1, 1, 32, cout)
    with pytest.raises(Exception):
        ctx.call("bsl_conv2d_dgrad", C.byref(desc), ddy.p, dw_.p, xw.p, ctx.stream)
    for b in (xn, xw, dw_, ddy):
        b.free()


def ctx_bf16(bits):
    return (bits.astype(np.uint32) << 16).view(np.float32)


def test_conv2d_fprop_fused_statistics(ctx):
    """bsl_conv2d_fprop_stats == bsl_conv2d_fprop followed by bsl_norm_stats (batch mode), on both kernel paths."""
    for (n, h, w, cin, cout, y_ld) in [(2, 32, 32, 64, 64, 64), (3, 16, 24, 128, 192, 256), (2, 12, 20, 64, 128, 128),
                                       (6, 32, 32, 64, 256, 256), (3, 30, 20, 64, 64, 64), (2, 20, 36, 128, 128, 128)]:
        rng = np.random.default_rng(h + cout)
        x = bf16_randn(rng, (n, h, w, cin))
        wt = bf16_randn(rng, (3, 3, cin, cout), 0.05)
        dx_, dw_ = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt)
        y1 = ctx.alloc(n * h * w * y_ld * 2).zero()
        y2 = ctx.alloc(n * h * w * y_ld * 2).zero()
        s1, s2 = ctx.alloc(2 * cout * 8).zero(), ctx.alloc(2 * cout * 8).zero()
        desc = _lib.Conv2dDesc(n, h, w, cin, cout, 3, 3, cin, y_ld)
        ctx.call("bsl_conv2d_fprop_stats", C.byref(desc), dx_.p, dw_.p, y1.p, s1.p, ctx.stream)
        ctx.call("bsl_conv2d_fprop", C.byref(desc), dx_.p, dw_.p, y2.p, ctx.stream)
        nd = _lib.NormDesc(0, n, h * w, cout, y_ld, y_ld, 1e-3, 0.999, 1, 1, 1)
        ctx.call("bsl_norm_stats", C.byref(nd), y2.p, s2.p, ctx.stream)
        ctx.check_device()
        a = y1.download(np.uint16, (n, h, w, y_ld))
        assert np.array_equal(a, y2.download(np.uint16, (n, h, w, y_ld)))
        yv = ctx.bf16_to_f32(y1, (n, h, w, y_ld))[..., :cout].astype(np.float64)
        got = s1.download(np.float64, (2, cout))
        assert rel(got[0], yv.sum(axis=(0, 1, 2))) < 1e-5
        assert rel(got[1], (yv * yv).sum(axis=(0, 1, 2))) < 1e-5
        assert rel(got, s2.download(np.float64, (2, cout))) < 1e-5
        # static tile schedule + fixed-order reductions: bit-reproducible
        ctx.call("bsl_conv2d_fprop_stats", C.byref(desc), dx_.p, dw_.p, y1.p, s2.p, ctx.stream)
        assert np.array_equal(got, s2.download(np.float64, (2, cout)))
        for b in (dx_, dw_, y1, y2, s1, s2):
            b.free()


@pytest.mark.parametrize("n,h,w,cin,cout,y_ld,gi", [
    (4, 32, 32, 64, 64, 64, 1),      # column tile 64 (per-thread running sums), several units per image
    (6, 16, 8, 64, 64, 64, 1),       # one 8x16 sub-tile per image: a unit of two sub-tiles spans two groups
    (6, 16, 8, 64, 128, 128, 2),     # column tile 128, groups of two images
    (3, 16, 24, 128, 192, 256, 1),   # three column tiles of 64, odd sub-tile count, output inside a wider buffer
    (8, 32, 32, 64, 128, 128, 4),    # UNet3D-style: 4 depth slices per volume
    (2, 64, 64, 64, 64, 64, 1),      # more units than CTAs would take in one round
    (5, 32, 32, 64, 256, 256, 1),    # column tile 256: falls back to the separate statistics pass
    (2, 12, 20, 64, 128, 128, 1),    # ragged extents: edge rows of the tiles are not counted
    (4, 30, 20, 64, 64, 64, 2),      # ragged, column tile 64 (per-thread running sums), groups of two images
    (3, 20, 36, 128, 128, 128, 1),   # ragged, column tile 128
])
def test_conv2d_fprop_group_statistics(ctx, n, h, w, cin, cout, y_ld, gi):
    """bsl_conv2d_fprop_group_stats == bsl_conv2d_fprop followed by bsl_norm_stats in instance mode over groups of `gi`
    consecutive images: bit-identical bf16 outputs, sums equal to 1e-5 (different fixed summation order), and
    bit-reproducible across runs."""
    rng = np.random.default_rng(h + cout + gi)
    from boxsegliver_b200.device import round_bf16
    # distinct statistics per image
    x = round_bf16(bf16_randn(rng, (n, h, w, cin)) + np.arange(n, dtype=np.float32)[:, None, None, None] * 0.25)
    wt = bf16_randn(rng, (3, 3, cin, cout), 0.05)
    dx_, dw_ = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt)
    y1 = guarded(ctx, n * h * w * y_ld * 2)
    y2 = ctx.alloc(n * h * w * y_ld * 2).zero()
    groups = n // gi
    s1, s2 = ctx.alloc(groups * 2 * cout * 8).zero(), ctx.alloc(groups * 2 * cout * 8).zero()
    desc = _lib.Conv2dDesc(n, h, w, cin, cout, 3, 3, cin, y_ld)
    ctx.call("bsl_conv2d_fprop_group_stats", C.byref(desc), dx_.p, dw_.p, y1.p, C.c_int(gi), s1.p, ctx.stream)
    ctx.call("bsl_conv2d_fprop", C.byref(desc), dx_.p, dw_.p, y2.p, ctx.stream)
    nd = _lib.NormDesc(1, groups, gi * h * w, cout, y_ld, y_ld, 1e-6, 0.0, 1, 1, 1)
    ctx.call("bsl_norm_stats", C.byref(nd), y2.p, s2.p, ctx.stream)
    ctx.check_device()
    assert guard_intact(y1, n * h * w * y_ld * 2), "the statistics epilogue stored past the end of its output"
    assert np.array_equal(y1.download(np.uint16, (n, h, w, y_ld)), y2.download(np.uint16, (n, h, w, y_ld)))
    yv = ctx.bf16_to_f32(y1, (n, h, w, y_ld))[..., :cout].astype(np.float64).reshape(groups, -1, cout)
    got = s1.download(np.float64, (groups, 2, cout))
    assert rel(got[:, 0], yv.sum(axis=1)) < 1e-5
    assert rel(got[:, 1], (yv * yv).sum(axis=1)) < 1e-5
    for g in range(groups):     # per group, so that a small group cannot hide behind a large one
        assert rel(got[g], s2.download(np.float64, (groups, 2, cout))[g]) < 1e-5, g
    ctx.call("bsl_conv2d_fprop_group_stats", C.byref(desc), dx_.p, dw_.p, y1.p, C.c_int(gi), s2.p, ctx.stream)
    assert np.array_equal(got, s2.download(np.float64, (groups, 2, cout)))
    with pytest.raises(Exception):
        ctx.call("bsl_conv2d_fprop_group_stats", C.byref(desc), dx_.p, dw_.p, y1.p, C.c_int(n + 1), s1.p, ctx.stream)
    for b in (dx_, dw_, y1, y2, s1, s2):
        b.free()


@pytest.mark.parametrize("n,h,w,cin,cout,y_ld", [
    (2, 8, 8, 128, 64, None), (1, 16, 16, 64, 64, None), (2, 4, 8, 256, 128, None), (1, 6, 10, 128, 64, None),
    (2, 8, 8, 128, 64, 128), (1, 2, 2, 1024, 512, 1024),
    (2, 16, 16, 128, 64, 128), (3, 32, 8, 256, 128, None), (1, 16, 24, 64, 64, 192),    # 1-tap halo-kernel path
    (2, 30, 20, 128, 64, None), (1, 12, 20, 256, 128, 192),                             # ragged extents
    # cout = 32: the half-block form (UNet3D's pixel-pair packed level: both column parities in one 64-wide block)
    (8, 16, 16, 64, 32, 64), (2, 32, 16, 128, 32, None), (4, 16, 8, 64, 32, 64)])
def test_conv2d_transpose(ctx, n, h, w, cin, cout, y_ld):
    rng = np.random.default_rng(cin + cout + h)
    y_ld = y_ld or cout
    x = bf16_randn(rng, (n, h, w, cin))
    wt = bf16_randn(rng, (2, 2, cout, cin), 0.05)
    bias = (rng.standard_normal(cout) * 0.1).astype(np.float32)
    dy = bf16_randn(rng, (n, 2 * h, 2 * w, cout))
    dx_, dw_, db_ = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt), ctx.from_numpy(bias)
    yo = guarded(ctx, n * 4 * h * w * y_ld * 2)
    dxo = guarded(ctx, n * h * w * cin * 2)
    desc = _lib.ConvT2dDesc(n, h, w, cin, cout, cin, y_ld, 1)
    x64, w64, dy64 = x.astype(np.float64), wt.astype(np.float64), dy.astype(np.float64)
    ctx.call("bsl_convT2d_fwd", C.byref(desc), dx_.p, dw_.p, db_.p, yo.p, ctx.stream)
    ctx.check_device()
    assert guard_intact(yo, n * 4 * h * w * y_ld * 2), "the scatter epilogue stored past the end of its output"
    got = ctx.bf16_to_f32(yo, (n, 2 * h, 2 * w, y_ld))
    assert rel(got[..., :cout], O.relu(O.conv2d_transpose(x64, w64) + bias)) < TOL_BF16
    assert not got[..., cout:].any()
    rdx, rdw = O.conv2d_transpose_grad(x64, w64, dy64)
    if cout == 32:      # the half-block form reads a dense gradient (both column parities = 64 contiguous values)
        if y_ld != 32:
            ddy = ctx.bf16_from_f32(padded(dy, y_ld))
            with pytest.raises(Exception):
                ctx.call("bsl_convT2d_bwd_data", C.byref(desc), ddy.p, dw_.p, dxo.p, ctx.stream)
            ddy.free()
        y_ld = 32
        desc = _lib.ConvT2dDesc(n, h, w, cin, cout, cin, y_ld, 1)
    ddy = ctx.bf16_from_f32(padded(dy, y_ld))
    ctx.call("bsl_convT2d_bwd_data", C.byref(desc), ddy.p, dw_.p, dxo.p, ctx.stream)
    ctx.check_device()
    assert guard_intact(dxo, n * h * w * cin * 2)
    assert rel(ctx.bf16_to_f32(dxo, (n, h, w, cin)), rdx) < TOL_BF16
    ws_bytes = ctx.lib.bsl_convT2d_bwd_filter_workspace(ctx.h, C.byref(desc))
    ws = ctx.alloc(max(ws_bytes, 16))
    dwo, dbo = ctx.alloc(4 * cout * cin * 4).zero(), ctx.alloc(cout * 4).zero()
    ctx.call("bsl_convT2d_bwd_filter", C.byref(desc), dx_.p, ddy.p, dwo.p, dbo.p, ws.p, C.c_size_t(ws_bytes), ctx.stream)
    ctx.check_device()
    assert rel(dwo.download(np.float32, (2, 2, cout, cin)), rdw) < TOL_F32
    assert rel(dbo.download(np.float32, (cout,)), dy64.sum(axis=(0, 1, 2))) < TOL_F32
    for b in (dx_, dw_, db_, ddy, yo, dxo, ws, dwo, dbo):
        b.free()


@pytest.mark.parametrize("n,h,w,cin", [(8, 16, 16, 64), (2, 32, 8, 128)])
def test_conv2d_transpose_into_voxel_pairs(ctx, n, h, w, cin):
    """bsl_convT2d_fwd_pairs: 32 output channels written into the `up` half of UNet3D's pixel-pair packed concat buffer
    (128 lanes per voxel pair: [enc even | enc odd | up even | up odd]); the other half must stay untouched."""
    rng = np.random.default_rng(cin + h)
    x = bf16_randn(rng, (n, h, w, cin))
    wt = bf16_randn(rng, (2, 2, 32, cin), 0.05)
    dx_, dw_ = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt)
    yo = ctx.alloc(n * 2 * h * w * 128 * 2).zero()
    desc = _lib.ConvT2dDesc(n, h, w, cin, 32, cin, 128, 1)
    ctx.call("bsl_convT2d_fwd_pairs", C.byref(desc), dx_.p, dw_.p, C.c_void_p(yo.ptr + 64 * 2), ctx.stream)
    ctx.check_device()
    got = ctx.bf16_to_f32(yo, (n, 2 * h, w, 128))
    ref = O.relu(O.conv2d_transpose(x.astype(np.float64), wt.astype(np.float64)))      # [n, 2h, 2w, 32]
    assert rel(got[..., 64:].reshape(n, 2 * h, 2 * w, 32), ref) < TOL_BF16
    assert not got[..., :64].any()
    for b in (dx_, dw_, yo):
        b.free()


def test_full_size_adjoint_identity(ctx):
    """BASELINE-size layer (Decode1 conv1 of cfg2: 64 x 256 x 256, 128 -> 64): the oracle cannot run it in
    seconds, but <fprop(x), dy> == <x, dgrad(dy)> == <w, wgrad(x, dy)> must hold for any correct triple."""
    n, h, w, cin, cout = 32, 256, 256, 128, 64   # half of cfg2's batch: bounds host RAM/time; same tiles, same kernels
    rng = np.random.default_rng(0)
    npx = n * h * w
    # low-rank random fields keep host generation cheap: x[p, c] = a[p] * b[c] (exactly bf16 products are not
    # needed; the identity holds for whatever bits are uploaded)
    # All fields are non-negative so the three inner products accumulate coherently: with random signs the sums
    # are residuals of cancelling terms and the bf16 output rounding (2^-9 per element) alone moves them by ~1e-3.
    x = np.abs(bf16_randn(rng, (npx, 1))) * np.abs(bf16_randn(rng, (1, cin)))
    dy = np.abs(bf16_randn(rng, (npx, 1))) * np.abs(bf16_randn(rng, (1, cout)))
    from boxsegliver_b200.device import round_bf16
    x, dy = round_bf16(x), round_bf16(dy)
    wt = np.abs(bf16_randn(rng, (3, 3, cin, cout), 0.05))
    dx_, ddy, dw_ = ctx.bf16_from_f32(x), ctx.bf16_from_f32(dy), ctx.bf16_from_f32(wt)
    yo, dxo = ctx.alloc(npx * cout * 2), ctx.alloc(npx * cin * 2)
    desc = _lib.Conv2dDesc(n, h, w, cin, cout, 3, 3, cin, cout)
    ws_bytes = ctx.lib.bsl_conv2d_wgrad_workspace(ctx.h, C.byref(desc))
    ws, dwo = ctx.alloc(max(ws_bytes, 16)), ctx.alloc(9 * cin * cout * 4)
    ctx.call("bsl_conv2d_fprop", C.byref(desc), dx_.p, dw_.p, yo.p, ctx.stream)
    ctx.call("bsl_conv2d_dgrad", C.byref(desc), ddy.p, dw_.p, dxo.p, ctx.stream)
    ctx.call("bsl_conv2d_wgrad", C.byref(desc), dx_.p, ddy.p, dwo.p, ws.p, C.c_size_t(ws_bytes), ctx.stream)
    ctx.check_device()
    def dot64(u, v, chunk=1 << 18):
        return sum(float(np.dot(u[i:i + chunk].ravel().astype(np.float64), v[i:i + chunk].ravel().astype(np.float64)))
                   for i in range(0, u.shape[0], chunk))

    a = dot64(ctx.bf16_to_f32(yo, (npx, cout)), dy)
    b = dot64(ctx.bf16_to_f32(dxo, (npx, cin)), x)
    dwg = dwo.download(np.float32, (3, 3, cin, cout)).astype(np.float64)
    c = float((dwg * wt).sum())
    scale = max(abs(a), abs(b), abs(c), 1e-30)
    assert abs(a - c) / scale < 5e-4 and abs(b - c) / scale < 5e-4, (a, b, c)
    for buf in (dx_, ddy, dw_, yo, dxo, ws, dwo):
        buf.free()


def test_rejects_unsupported_shapes(ctx):
    from boxsegliver_b200._lib import BslError
    d = _lib.Conv2dDesc(1, 8, 8, 48, 64, 3, 3, 48, 64)  # cin not a multiple of 64 -> loud failure, no fallback
    buf = ctx.alloc(1 << 16)
    with pytest.raises(BslError):
        ctx.call("bsl_conv2d_fprop", C.byref(d), buf.p, buf.p, buf.p, ctx.stream)
    d = _lib.Conv2dDesc(1, 8, 8, 64, 64, 5, 5, 64, 64)
    with pytest.raises(BslError):
        ctx.call("bsl_conv2d_fprop", C.byref(d), buf.p, buf.p, buf.p, ctx.stream)
    d = _lib.Conv2dDesc(1, 8, 8, 64, 64, 3, 3, 64, 64)
    with pytest.raises(BslError):
        ctx.call("bsl_conv2d_fprop", C.byref(d), None, buf.p, buf.p, ctx.stream)
    buf.free()

