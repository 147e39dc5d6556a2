"""bsl_conv2d_fprop_bias_relu (slim.conv2d with normalizer_fn=None: y = bf16(relu(conv + bias))) and bsl_maxpool2x2_bf16,
op by op through the C ABI.

Every fprop schedule is covered: the halo-tile kernel with a streamed filter (64-, 128- and 256-wide tiles, the latter
with the TMA-store epilogue), the resident-filter kernels, the CTA-pair and resident-pair kernels, the first-generation
igemm_kernel (shapes the 8 x 16 halo tiles do not fit) and the stem's 1x1 GEMM over 32-column im2col rows, at the layer
shapes of cfg2 (UNet 256 x 256, batch reduced to 4: the same tile classes), the ragged deep levels of 96 x 96 and
480 x 160 inputs, and concat-slice inputs / outputs."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from boxsegliver_b200._lib import BslError
from boxsegliver_b200.device import bf16_bits_to_f32, f32_to_bf16_bits, round_bf16
from tests.gpu_util import TOL_BF16, bf16_randn, rel

pytestmark = pytest.mark.gpu

CASES = [
    # n, h, w, cin, cout, k, x_ld, y_ld                    schedule of the fprop at this shape
    # cfg2 layers (UNet 256 x 256, base 64, depth 4)
    (4, 256, 256, 64, 64, 1, 32, 64),          # stem: 1x1 over 32-column im2col rows (resident filter, TMA zero-fill)
    (4, 256, 256, 64, 64, 3, 64, 128),         # Encode1/2 into its concat slice: resident filter, one block
    (4, 128, 128, 64, 128, 3, 64, 128),        # Encode2/1: resident filter, 128-wide tile
    (4, 128, 128, 128, 128, 3, 128, 256),      # Encode2/2: resident CTA pair, concat slice
    (4, 64, 64, 128, 256, 3, 128, 256),        # Encode3/1: CTA pair (128-wide tiles over sub-tile pairs)
    (4, 64, 64, 256, 256, 3, 256, 512),        # Encode3/2: CTA pair, concat slice
    (4, 32, 32, 256, 512, 3, 256, 512),        # Encode4/1: CTA pair, 4 column tiles
    (4, 32, 32, 512, 512, 3, 512, 1024),       # Encode4/2: CTA pair, concat slice
    (4, 16, 16, 512, 1024, 3, 512, 1024),      # ED-Bridge_1
    (4, 16, 16, 1024, 1024, 3, 1024, 1024),    # ED-Bridge_2
    (4, 32, 32, 1024, 512, 3, 1024, 512),      # Decode4/1 reads the concat buffer
    (4, 64, 64, 512, 256, 3, 512, 256),        # Decode3/1
    (4, 128, 128, 256, 128, 3, 256, 128),      # Decode2/1: resident CTA pair
    (4, 256, 256, 128, 64, 3, 128, 64),        # Decode1/1: resident CTA pair, 64-wide
    # single-CTA schedules the cfg2 shapes do not reach
    (1, 16, 16, 64, 256, 3, 64, 256),          # 256-wide tile, TMA-store epilogue, sub-tile pairs (2 sub-tiles)
    (1, 8, 16, 64, 256, 3, 64, 256),           # 256-wide tile, TMA-store epilogue, single sub-tiles
    (4, 16, 16, 512, 64, 3, 512, 64),          # streamed filter, 64-wide tile (filter too big to stay resident)
    (3, 16, 24, 64, 192, 3, 64, 192),          # resident filter, odd sub-tile count, 3 column tiles
    (1, 48, 40, 192, 128, 3, 256, 192),        # concat views on both sides, 3 k-blocks
    # first-generation igemm_kernel (halo tiles do not fit)
    (3, 4, 4, 128, 64, 3, 128, 64),
    (1, 2, 2, 1024, 1024, 3, 1024, 2048),      # with a concat-slice output
    # ragged deep levels: 96 x 96 (levels 12 x 12 halo-ragged, 6 x 6 igemm) and 480 x 160 (60 x 20, 30 x 10)
    (2, 12, 12, 256, 512, 3, 256, 1024),
    (2, 6, 6, 512, 1024, 3, 512, 1024),
    (1, 60, 20, 256, 512, 3, 256, 1024),
    (1, 30, 10, 512, 1024, 3, 512, 1024),
    (2, 20, 12, 128, 128, 3, 128, 256),
]

GUARD = np.full(8192, 0xABCD, np.uint16)
FILL = 0x3F80                                  # bf16 1.0 in every lane the call must not write


def _canon(bits):
    """-0 and +0 are the same value (the ReLU of a negative zero sum may carry either sign)."""
    b = bits.copy()
    b[b == 0x8000] = 0
    return b


def _out_buffer(ctx, n, h, w, y_ld):
    nbytes = n * h * w * y_ld * 2
    buf = ctx.alloc(nbytes + GUARD.nbytes)
    buf.upload(np.full(n * h * w * y_ld, FILL, np.uint16))
    buf.upload(GUARD, byte_offset=nbytes)
    return buf, nbytes


def _check_untouched(ctx, buf, nbytes, shape, cout):
    assert np.array_equal(buf.download(np.uint16, GUARD.shape, byte_offset=nbytes), GUARD), "store past the output"
    bits = buf.download(np.uint16, shape)
    assert (bits[..., cout:] == FILL).all(), "store outside the channel slice"
    return bits[..., :cout]


def _reference(x, wt, bias, pix):
    """fp64 relu(conv(x, w) + bias) at the flat output pixels `pix` (SAME padding, stride 1)."""
    n, h, w, cin = x.shape
    k = wt.shape[0]
    r = k // 2
    xp = np.pad(x.astype(np.float64), ((0, 0), (r, r), (r, r), (0, 0)))
    b, i, j = np.unravel_index(pix, (n, h, w))
    patches = np.stack([xp[b, i + di, j + dj] for di in range(k) for dj in range(k)], axis=1)   # [p, taps, cin]
    y = patches.reshape(len(pix), -1) @ wt.astype(np.float64).reshape(-1, wt.shape[-1]) + bias.astype(np.float64)
    return np.maximum(y, 0.0)


@pytest.mark.parametrize("n,h,w,cin,cout,k,x_ld,y_ld", CASES)
def test_fprop_bias_relu(ctx, n, h, w, cin, cout, k, x_ld, y_ld):
    rng = np.random.default_rng(cin * 3 + cout + h * 7 + w)
    cx = min(cin, x_ld)                        # the stem's 32-column rows: channels >= x_ld read as zero
    x = np.zeros((n, h, w, cin), np.float32)
    x[..., :cx] = bf16_randn(rng, (n, h, w, cx))
    xbuf = np.zeros((n, h, w, x_ld), np.float32)
    xbuf[..., :cx] = x[..., :cx]
    if x_ld > cin:
        xbuf[..., cin:] = 7.0                  # lanes beyond cin belong to the other half of a concat buffer
    wt = bf16_randn(rng, (k, k, cin, cout), 1.0 / np.sqrt(k * k * cx))
    bias = (rng.standard_normal(cout) * 0.5).astype(np.float32)
    dx, dw = ctx.bf16_from_f32(xbuf), ctx.bf16_from_f32(wt)
    dz = ctx.bf16_from_f32(np.zeros_like(wt))
    db, db0 = ctx.from_numpy(bias), ctx.from_numpy(np.zeros(cout, np.float32))
    desc = _lib.Conv2dDesc(n, h, w, cin, cout, k, k, x_ld, y_ld)
    shape = (n, h, w, y_ld)

    # plain fprop and the zero-bias epilogue: relu of the same bf16 values, bit for bit
    y0, nb = _out_buffer(ctx, n, h, w, y_ld)
    ctx.call("bsl_conv2d_fprop", C.byref(desc), dx.p, dw.p, y0.p, ctx.stream)
    y1, _ = _out_buffer(ctx, n, h, w, y_ld)
    ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(desc), dx.p, dw.p, db0.p, y1.p, ctx.stream)
    ctx.check_device()
    plain = _check_untouched(ctx, y0, nb, shape, cout)
    zero_bias = _check_untouched(ctx, y1, nb, shape, cout)
    relu_plain = np.where(plain & 0x8000, 0, plain).astype(np.uint16)
    assert np.array_equal(_canon(zero_bias), _canon(relu_plain)), "zero bias != relu(bsl_conv2d_fprop)"

    # random bias against fp64 conv + bias + ReLU (every pixel of small layers, a sample of the large ones)
    y2, _ = _out_buffer(ctx, n, h, w, y_ld)
    ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(desc), dx.p, dw.p, db.p, y2.p, ctx.stream)
    ctx.check_device()
    got = _check_untouched(ctx, y2, nb, shape, cout).reshape(-1, cout)
    npx = n * h * w
    pix = np.arange(npx) if npx <= 4096 else np.sort(rng.choice(npx, 2048, replace=False))
    ref = _reference(x, wt, bias, pix)
    assert rel(bf16_bits_to_f32(got[pix]), ref) < TOL_BF16
    assert not (bf16_bits_to_f32(got) < 0).any()

    # zero weights: exactly bf16(relu(bias)) in every pixel
    y3, _ = _out_buffer(ctx, n, h, w, y_ld)
    ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(desc), dx.p, dz.p, db.p, y3.p, ctx.stream)
    ctx.check_device()
    got = _check_untouched(ctx, y3, nb, shape, cout)
    want = f32_to_bf16_bits(np.maximum(bias, 0.0))
    assert np.array_equal(_canon(got), np.broadcast_to(_canon(want), got.shape))
    for b in (dx, dw, dz, db, db0, y0, y1, y2, y3):
        b.free()


@pytest.mark.parametrize("n,h,w,c,x_ld,y_ld", [
    (2, 16, 16, 64, 128, 64),       # encoder block: the activation's half of the concat buffer -> dense pooled tensor
    (3, 12, 20, 128, 256, 136),     # strided output (UNetInter --mid_cat lane layout)
    (1, 256, 256, 64, 128, 64),     # cfg2 Encode1
    (2, 30, 10, 512, 1024, 512),    # 480 x 160 deep level
    (1, 2, 2, 8, 8, 8),
])
def test_maxpool2x2_bf16_is_exact(ctx, n, h, w, c, x_ld, y_ld):
    rng = np.random.default_rng(h * w + c)
    x = round_bf16(rng.standard_normal((n, h, w, x_ld)).astype(np.float32))
    x[0, 0, 0, :c] = 0.0                                    # ties: equal values in a window
    x[0, 0, 1, :c] = 0.0
    dx = ctx.bf16_from_f32(x)
    ho, wo = h // 2, w // 2
    yb, nb = _out_buffer(ctx, n, ho, wo, y_ld)
    ctx.call("bsl_maxpool2x2_bf16", C.c_int(n), C.c_int(h), C.c_int(w), C.c_int(c), dx.p, C.c_int(x_ld), yb.p,
             C.c_int(y_ld), ctx.stream)
    ctx.check_device()
    got = _check_untouched(ctx, yb, nb, (n, ho, wo, y_ld), c)
    want = f32_to_bf16_bits(x[..., :c].reshape(n, ho, 2, wo, 2, c).max(axis=(2, 4)))
    assert np.array_equal(got, want)
    dx.free()
    yb.free()


def test_refusals(ctx):
    buf = ctx.alloc(1 << 16)
    f = buf.p
    ok = _lib.Conv2dDesc(1, 16, 16, 64, 64, 3, 3, 64, 64)
    with pytest.raises(BslError, match="null buffer"):
        ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(ok), f, f, None, f, ctx.stream)
    with pytest.raises(BslError, match="null buffer"):
        ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(ok), None, f, f, f, ctx.stream)
    for d in (_lib.Conv2dDesc(1, 16, 16, 48, 64, 3, 3, 48, 64),     # cin not a multiple of 64
              _lib.Conv2dDesc(1, 16, 16, 64, 64, 5, 5, 64, 64),     # 5x5
              _lib.Conv2dDesc(1, 16, 16, 64, 64, 3, 3, 64, 60),     # y_ld < cout
              _lib.Conv2dDesc(0, 16, 16, 64, 64, 3, 3, 64, 64)):    # empty batch
        with pytest.raises(BslError):
            ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(d), f, f, f, f, ctx.stream)
    for args in ((1, 15, 16, 64, 64, 64),      # odd height
                 (1, 16, 16, 60, 64, 64),      # c not a multiple of 8
                 (1, 16, 16, 64, 32, 64),      # x_ld < c
                 (1, 16, 16, 64, 64, 60)):     # y_ld < c
        n, h, w, c, xl, yl = args
        with pytest.raises(BslError, match="maxpool2x2_bf16"):
            ctx.call("bsl_maxpool2x2_bf16", C.c_int(n), C.c_int(h), C.c_int(w), C.c_int(c), f, C.c_int(xl), f,
                     C.c_int(yl), ctx.stream)
    with pytest.raises(BslError, match="null buffer"):
        ctx.call("bsl_maxpool2x2_bf16", C.c_int(1), C.c_int(16), C.c_int(16), C.c_int(64), None, C.c_int(64), f,
                 C.c_int(64), ctx.stream)
    with pytest.raises(BslError, match="maxpool2x2_bf16"):   # misaligned activation
        ctx.call("bsl_maxpool2x2_bf16", C.c_int(1), C.c_int(16), C.c_int(16), C.c_int(64), C.c_void_p(buf.ptr + 2),
                 C.c_int(64), f, C.c_int(64), ctx.stream)
    ctx.check_device()
    buf.free()
