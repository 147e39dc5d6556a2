"""3-D / strided convolutions of the UNet3D path (csrc/conv3d.cu) against the numpy oracle, through the C ABI.
Every (kernel, stride) combination of /root/reference/NetworksV2/UNet3D.py:31-59 is covered, on inputs the oracle
finishes in seconds. Tolerance: bf16 outputs rel <= 1e-2 (north_star); fp32 filter gradients <= 1e-4."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from boxsegliver_b200.device import bf16_bits_to_f32, round_bf16
from oracle import tf_ops as O
from tests.gpu_util import TOL_BF16, TOL_F32, bf16_randn, rel

pytestmark = pytest.mark.gpu

CASES = [  # (n, d, h, w, cin, cout, kernel, stride)
    (2, 4, 16, 16, 64, 64, (1, 3, 3), (1, 2, 2)),      # conv_e1/conv1
    (1, 6, 16, 16, 64, 128, (3, 3, 3), (1, 2, 2)),     # conv_e2/conv1
    (2, 5, 8, 16, 128, 128, (3, 3, 3), (1, 1, 1)),     # conv_e2/conv2 (odd depth, non-square)
    (1, 8, 8, 8, 128, 64, (3, 3, 3), (2, 2, 2)),       # bridge/conv1
    (1, 4, 8, 8, 64, 64, (1, 3, 3), (1, 1, 1)),        # (1,3,3) through the 3-D entry point
    (1, 4, 8, 8, 64, 64, (1, 1, 1), (1, 1, 1)),
    # stride-1 layers whose slices tile into 8x16 / 16x4 boxes: halo-tile kernels with the depth loop
    (2, 3, 16, 16, 128, 128, (3, 3, 3), (1, 1, 1)),    # conv_e2/conv2: wide wgrad (cout % 128 == 0)
    (1, 4, 16, 32, 128, 64, (3, 3, 3), (1, 1, 1)),     # cout 64: first wgrad kernel, resident filter in dgrad
    (1, 2, 32, 16, 64, 320, (3, 3, 3), (1, 1, 1)),     # cout 320 (bridge width): not a multiple of 128
    (2, 2, 16, 16, 256, 128, (1, 3, 3), (1, 1, 1)),
    # the strided conv that leaves the pixel-pair packed level: super voxels along W (stride 1 there), stride 2 along H
    (2, 4, 32, 16, 128, 64, (1, 3, 3), (1, 2, 1)),
    (2, 4, 32, 16, 64, 64, (1, 3, 2), (1, 2, 1)),      # ... as the engine runs it: 2-tap rows (super voxels X, X + 1)
    # strided layers whose output grid tiles into 8x16 boxes: dgrad = one halo-tile launch per output phase (tap tables)
    (1, 3, 32, 32, 64, 128, (3, 3, 3), (1, 2, 2)),     # conv_e2/conv1: 4 phases, depth loop
    (2, 2, 64, 16, 64, 64, (1, 3, 2), (1, 2, 1)),      # conv_e1/conv1 on the pair-packed level: 2 phases
    (1, 2, 32, 16, 128, 64, (1, 3, 3), (1, 2, 2)),     # resident filter, two reduction blocks
    (1, 3, 32, 32, 128, 256, (3, 3, 3), (1, 2, 2)),    # conv_e3/conv1: cout 256
    # ragged extents (the deep levels of the shipped 10 x 512 x 160 volumes): halo-tile kernels with masked edge rows
    (1, 5, 32, 10, 128, 128, (3, 3, 3), (1, 1, 1)),    # level 4: 32 x 10
    (1, 4, 40, 24, 64, 128, (3, 3, 3), (1, 2, 2)),     # strided: phase grid 20 x 12
    (2, 2, 20, 12, 64, 64, (1, 3, 3), (1, 1, 1)),
]


@pytest.mark.parametrize("n,d,h,w,cin,cout,k,s", CASES)
def test_conv3d_fprop_dgrad_wgrad(ctx, n, d, h, w, cin, cout, k, s):
    rng = np.random.default_rng(cin + cout + d)
    x = bf16_randn(rng, (n, d, h, w, cin))
    wt = bf16_randn(rng, k + (cin, cout), scale=0.1)
    y_ref = O.conv3d(x.astype(np.float64), wt.astype(np.float64), s)
    od, oh, ow = y_ref.shape[1:4]
    dy = bf16_randn(rng, (n, od, oh, ow, cout))
    desc = _lib.Conv3dDesc(n, d, h, w, cin, cout, k[0], k[1], k[2], s[0], s[1], s[2], cin, cout)
    bx, bw, bdy = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt), ctx.bf16_from_f32(dy)
    guard = np.full(8192, 0xABCD, np.uint16)      # canaries: edge tiles of ragged extents must not store past the tensors
    by = ctx.alloc(y_ref.size * 2 + guard.nbytes).zero().upload(guard, byte_offset=y_ref.size * 2)
    bdx = ctx.alloc(x.size * 2 + guard.nbytes).zero().upload(guard, byte_offset=x.size * 2)
    bdw = ctx.alloc(wt.size * 4)
    ws_bytes = ctx.lib.bsl_conv3d_wgrad_workspace(ctx.h, C.byref(desc))
    ws = ctx.alloc(max(ws_bytes, 16))
    ctx.call("bsl_conv3d_fprop", C.byref(desc), bx.p, bw.p, by.p, ctx.stream)
    ctx.call("bsl_conv3d_dgrad", C.byref(desc), bdy.p, bw.p, bdx.p, ctx.stream)
    ctx.call("bsl_conv3d_wgrad", C.byref(desc), bx.p, bdy.p, bdw.p, ws.p, C.c_size_t(ws_bytes), ctx.stream)
    ctx.check_device()
    y = ctx.bf16_to_f32(by, y_ref.shape)
    dx = ctx.bf16_to_f32(bdx, x.shape)
    dw = bdw.download(np.float32, wt.shape)
    ok_y = np.array_equal(by.download(np.uint16, guard.shape, byte_offset=y_ref.size * 2), guard)
    ok_dx = np.array_equal(bdx.download(np.uint16, guard.shape, byte_offset=x.size * 2), guard)
    for b in (bx, bw, bdy, by, bdx, bdw, ws):
        b.free()
    assert ok_y and ok_dx, "a store past the end of an output tensor"
    assert rel(y, y_ref) < TOL_BF16
    assert rel(y, round_bf16(y_ref.astype(np.float32))) < 2e-3
    dx_ref = O.conv3d_backprop_input(x.shape, wt.astype(np.float64), dy.astype(np.float64), s)
    assert rel(dx, dx_ref) < TOL_BF16
    dw_ref = O.conv3d_backprop_filter(x.astype(np.float64), wt.shape, dy.astype(np.float64), s)
    assert rel(dw, dw_ref) < TOL_F32


@pytest.mark.parametrize("n,d,h,w,cin,cout,sd", [(1, 4, 8, 8, 128, 64, 2), (2, 3, 8, 8, 64, 64, 1), (1, 2, 4, 4, 320, 256, 2)])
def test_convT3d_fwd_bwd(ctx, n, d, h, w, cin, cout, sd):
    rng = np.random.default_rng(7 + cin)
    x = bf16_randn(rng, (n, d, h, w, cin))
    wt = bf16_randn(rng, (sd, 2, 2, cout, cin), scale=0.1)
    st = (sd, 2, 2)
    pre = O.conv3d_transpose(x.astype(np.float64), wt.astype(np.float64), st)
    y_ref = np.maximum(pre, 0)
    dyr = bf16_randn(rng, y_ref.shape) * (y_ref > 0)
    desc = _lib.ConvT3dDesc(n, d, h, w, cin, cout, sd, cin, cout, 1)
    bx, bw, bdy = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt), ctx.bf16_from_f32(dyr.astype(np.float32))
    by, bdx, bdw = ctx.alloc(y_ref.size * 2), ctx.alloc(x.size * 2), ctx.alloc(wt.size * 4)
    ws_bytes = ctx.lib.bsl_convT3d_bwd_filter_workspace(ctx.h, C.byref(desc))
    ws = ctx.alloc(max(ws_bytes, 16))
    ctx.call("bsl_convT3d_fwd", C.byref(desc), bx.p, bw.p, None, by.p, ctx.stream)
    ctx.call("bsl_convT3d_bwd_data", C.byref(desc), bdy.p, bw.p, bdx.p, ctx.stream)
    ctx.call("bsl_convT3d_bwd_filter", C.byref(desc), bx.p, bdy.p, bdw.p, None, ws.p, C.c_size_t(ws_bytes), ctx.stream)
    ctx.check_device()
    y = ctx.bf16_to_f32(by, y_ref.shape)
    dx = ctx.bf16_to_f32(bdx, x.shape)
    dw = bdw.download(np.float32, wt.shape)
    for b in (bx, bw, bdy, by, bdx, bdw, ws):
        b.free()
    assert rel(y, y_ref) < TOL_BF16
    dx_ref, dw_ref = O.conv3d_transpose_grad(x.astype(np.float64), wt.astype(np.float64), dyr.astype(np.float64), st)
    assert rel(dx, dx_ref) < TOL_BF16
    assert rel(dw, dw_ref) < TOL_F32


def _poison_scratch(ctx):
    """Fill the stream's reduction scratch arena with large partials: bsl_norm_stats over 18944 px x 1024 channels of
    2^50 runs 4 * 148 = 592 blocks and leaves 592 x 2 x 1024 fp32 partials (4.8 MB) at the arena's start, more than
    any conv statistics epilogue of these shapes writes there (slots x 2 x cout <= 296 x 2 x 320 floats, or that x 4
    x volumes for instance statistics). A partial the conv then fails to write shows up in its sums as ~2^50."""
    px, c = 18944, 1024
    big = ctx.from_numpy(np.full(px * c, 0x5880, np.uint16))      # bf16 2^50
    s = ctx.alloc(2 * c * 8)
    nd = _lib.NormDesc(0, 1, px, c, c, c, 1e-3, 0.999, 0, 1, 1)
    ctx.call("bsl_norm_stats", C.byref(nd), big.p, s.p, ctx.stream)
    assert s.download(np.float64, (2, c))[0, 0] == px * 2.0 ** 50
    big.free()
    s.free()


@pytest.mark.parametrize("n,d,h,w,cin,cout,k,s", CASES + [
    (2, 3, 16, 16, 64, 256, (3, 3, 3), (1, 1, 1)),    # cout 256, stride 1: bn = 256 -> the separate statistics pass
])
def test_conv3d_fprop_fused_statistics(ctx, n, d, h, w, cin, cout, k, s):
    """bsl_conv3d_fprop_stats (batch: [2][cout] over every output voxel) and bsl_conv3d_fprop_group_stats (instance:
    [n][2][cout], one group per volume) on every layer shape: bf16 outputs bit-identical to bsl_conv3d_fprop, sums
    within 1e-5 of fp64 sums of the stored outputs and of bsl_norm_stats on them, bit-reproducible, nothing stored past
    y. The scratch arena is poisoned before each call, so a partial left unwritten cannot hide."""
    rng = np.random.default_rng(cin + cout + d + 5)
    x = round_bf16(bf16_randn(rng, (n, d, h, w, cin)) + np.arange(n, dtype=np.float32)[:, None, None, None, None] * 0.5)
    wt = bf16_randn(rng, k + (cin, cout), scale=0.1)
    od, oh, ow = (-(-d // s[0]), -(-h // s[1]), -(-w // s[2]))
    vox = od * oh * ow
    desc = _lib.Conv3dDesc(n, d, h, w, cin, cout, k[0], k[1], k[2], s[0], s[1], s[2], cin, cout)
    bx, bw = ctx.bf16_from_f32(x), ctx.bf16_from_f32(wt)
    ny = n * vox * cout
    guard = np.full(8192, 0xABCD, np.uint16)
    y_ref = ctx.alloc(ny * 2)
    ctx.call("bsl_conv3d_fprop", C.byref(desc), bx.p, bw.p, y_ref.p, ctx.stream)
    ref_bits = y_ref.download(np.uint16, (ny,))
    yv = bf16_bits_to_f32(ref_bits).astype(np.float64).reshape(n, vox, cout)
    nd_b = _lib.NormDesc(0, n, vox, cout, cout, cout, 1e-3, 0.999, 0, 1, 1)
    nd_i = _lib.NormDesc(1, n, vox, cout, cout, cout, 1e-6, 0.999, 0, 1, 1)
    ns_b, ns_i = ctx.alloc(2 * cout * 8), ctx.alloc(n * 2 * cout * 8)
    ctx.call("bsl_norm_stats", C.byref(nd_b), y_ref.p, ns_b.p, ctx.stream)
    ctx.call("bsl_norm_stats", C.byref(nd_i), y_ref.p, ns_i.p, ctx.stream)
    norm_b, norm_i = ns_b.download(np.float64, (2, cout)), ns_i.download(np.float64, (n, 2, cout))
    f64_b = np.stack([yv.sum(axis=(0, 1)), (yv * yv).sum(axis=(0, 1))])
    f64_i = np.stack([yv.sum(axis=1), (yv * yv).sum(axis=1)], axis=1)
    for name, groups, f64, norm in (("bsl_conv3d_fprop_stats", 1, f64_b[None], norm_b[None]),
                                    ("bsl_conv3d_fprop_group_stats", n, f64_i, norm_i)):
        got = []
        for _ in range(2):
            by = ctx.alloc(ny * 2 + guard.nbytes).zero().upload(guard, byte_offset=ny * 2)
            sums = ctx.alloc(groups * 2 * cout * 8).zero()
            _poison_scratch(ctx)
            ctx.call(name, C.byref(desc), bx.p, bw.p, by.p, sums.p, ctx.stream)
            ctx.check_device()
            assert np.array_equal(by.download(np.uint16, guard.shape, byte_offset=ny * 2), guard), (name, "guard")
            assert np.array_equal(by.download(np.uint16, (ny,)), ref_bits), (name, "bf16 outputs differ from fprop")
            got.append(sums.download(np.float64, (groups, 2, cout)))
            by.free()
            sums.free()
        assert np.array_equal(got[0], got[1]), (name, "not bit-reproducible")
        for g in range(groups):       # per volume: one volume cannot hide behind the others
            for j in range(2):
                assert rel(got[0][g, j], f64[g, j]) < 1e-5, (name, g, j, rel(got[0][g, j], f64[g, j]))
                assert rel(got[0][g, j], norm[g, j]) < 1e-5, (name, g, j)
    for b in (bx, bw, y_ref, ns_b, ns_i):
        b.free()
