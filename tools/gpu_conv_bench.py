"""Per-layer timing of the tensor-core convolutions at BASELINE cfg2 shapes (batch 64, 256x256 U-Net).

  python tools/gpu_conv_bench.py [--layers enc1_2,dec1_1] [--ops fprop,dgrad,wgrad] [--reps 10] [--batch 64]

One line per (layer, op): ms and algorithmic TFLOP/s (2 * MACs, un-padded). Inputs are random bf16 bits
replicated on the device; every tensor at the 256^2 levels is larger than L2, and successive reps of
smaller layers are separated by a write of a 256 MB scratch buffer (L2 flush). The library picks the kernel of each
layer from its shape, as in a training step.
"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import _lib  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402

LAYERS = {  # name: (hw, cin, cout)
    "enc1_2": (256, 64, 64), "enc2_1": (128, 64, 128), "enc2_2": (128, 128, 128), "enc3_1": (64, 128, 256),
    "enc3_2": (64, 256, 256), "enc4_1": (32, 256, 512), "enc4_2": (32, 512, 512), "br_1": (16, 512, 1024),
    "br_2": (16, 1024, 1024), "dec4_1": (32, 1024, 512), "dec4_2": (32, 512, 512), "dec3_1": (64, 512, 256),
    "dec3_2": (64, 256, 256), "dec2_1": (128, 256, 128), "dec2_2": (128, 128, 128), "dec1_1": (256, 128, 64),
    "dec1_2": (256, 64, 64),
}

ap = argparse.ArgumentParser()
ap.add_argument("--layers", default=",".join(LAYERS))
ap.add_argument("--ops", default="fprop,dgrad,wgrad")
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--stats", action="store_true", help="time bsl_conv2d_fprop_stats instead of bsl_conv2d_fprop")
ap.add_argument("--waits", action="store_true", help="print where the UMMA issuer thread waits (bsl_debug_set key 3)")
a = ap.parse_args()

ctx = Context(0)
if a.waits:
    ctx.call("bsl_debug_set", C.c_int(3), C.c_int(1))
rng = np.random.default_rng(0)
seed_block = (rng.standard_normal(1 << 20).astype(np.float32) * 0.5)
from boxsegliver_b200.device import f32_to_bf16_bits  # noqa: E402
seed_bits = f32_to_bf16_bits(seed_block)


def filled(nbytes):
    buf = ctx.alloc(nbytes)
    n0 = min(nbytes, seed_bits.nbytes)
    ctx.call("bsl_memcpy_h2d", buf.p, seed_bits.ctypes.data_as(C.c_void_p), C.c_size_t(n0), ctx.stream)
    done = n0
    while done < nbytes:
        n = min(done, nbytes - done)
        ctx.call("bsl_memcpy_d2d", buf.at(done), buf.p, C.c_size_t(n), ctx.stream)
        done += n
    ctx.sync()
    return buf


flush = ctx.alloc(256 << 20)
e0, e1 = ctx.new_event(), ctx.new_event()
tot = {}
for name in a.layers.split(","):
    hw, cin, cout = LAYERS[name]
    n = a.batch
    npx = n * hw * hw
    x, dy = filled(npx * cin * 2), filled(npx * cout * 2)
    w = filled(9 * cin * cout * 2)
    y, dx = ctx.alloc(npx * cout * 2), ctx.alloc(npx * cin * 2)
    dw = ctx.alloc(9 * cin * cout * 4)
    sums = ctx.alloc(2 * cout * 8)
    d = _lib.Conv2dDesc(n, hw, hw, cin, cout, 3, 3, cin, cout)
    ws_bytes = ctx.lib.bsl_conv2d_wgrad_workspace(ctx.h, C.byref(d))
    ws = ctx.alloc(max(ws_bytes, 16))
    flops = 2.0 * npx * 9 * cin * cout
    calls = {
        "fprop": (lambda: ctx.call("bsl_conv2d_fprop_stats", C.byref(d), x.p, w.p, y.p, sums.p, ctx.stream)) if a.stats
        else (lambda: ctx.call("bsl_conv2d_fprop", C.byref(d), x.p, w.p, y.p, ctx.stream)),
        "dgrad": lambda: ctx.call("bsl_conv2d_dgrad", C.byref(d), dy.p, w.p, dx.p, ctx.stream),
        "wgrad": lambda: ctx.call("bsl_conv2d_wgrad", C.byref(d), x.p, dy.p, dw.p, ws.p, C.c_size_t(ws_bytes), ctx.stream),
    }
    for op in a.ops.split(","):
        fn = calls[op]
        fn()
        ctx.sync()
        ms = 0.0
        for _ in range(a.reps):
            ctx.call("bsl_memset", flush.p, C.c_int(0), C.c_size_t(flush.nbytes), ctx.stream)
            ctx.record(e0)
            fn()
            ctx.record(e1)
            ms += ctx.elapsed_ms(e0, e1)
        ms /= a.reps
        ctx.check_device()
        tot[op] = tot.get(op, 0.0) + ms
        print(f"{name:8s} {op:6s} hw={hw:3d} cin={cin:4d} cout={cout:4d}  {ms:7.3f} ms  {flops / ms / 1e9:7.1f} TF/s", flush=True)
        if a.waits and op == "wgrad" and cout % 128 == 0:
            wt = np.zeros((1024, 4), np.int64)
            ctx.call("bsl_debug_read_waits", wt.ctypes.data_as(C.c_void_p), C.c_int(1024))
            ctx.call("bsl_debug_set", C.c_int(3), C.c_int(0))   # fresh (zeroed) buffer for the next layer
            ctx.call("bsl_debug_set", C.c_int(3), C.c_int(1))
            ok = wt[:, 0] > 0
            cls, tiles = wt[:, 2] >> 32, wt[:, 2] & 0xffffffff
            t_start = wt[ok, 3].min()
            for c in (0, 1):
                m = ok & (cls == c)
                if not m.any():
                    continue
                cyc, wf = wt[m, 0].astype(np.float64), wt[m, 1].astype(np.float64)
                print(f"         class {'ab'[c]}: {m.sum():4d} CTAs x {tiles[m].mean():6.1f} tiles  issuer {cyc.mean():9.0f} cycles "
                      f"(max {cyc.max():9.0f}) = {(cyc / np.maximum(tiles[m], 1)).mean():6.0f} / tile, waiting for a stage "
                      f"{100 * (wf / cyc).mean():5.1f} %, start +{(wt[m, 3] - t_start).mean() / 1e3:6.1f} us "
                      f"(last +{(wt[m, 3] - t_start).max() / 1e3:6.1f})", flush=True)
        if a.waits and op != "wgrad":
            wt = np.zeros((148, 4), np.int64)
            ctx.call("bsl_debug_read_waits", wt.ctypes.data_as(C.c_void_p), C.c_int(148))
            cyc = wt[:, 0].astype(np.float64)
            ok = cyc > 0
            f = lambda k: 100.0 * (wt[ok, k] / cyc[ok]).mean()   # noqa: E731
            print(f"         issuer: {cyc[ok].mean():.0f} cycles (min {cyc[ok].min():.0f}, max {cyc[ok].max():.0f}, {ok.sum()} CTAs); waiting acc_empty {f(1):.1f}%  a_full {f(2):.1f}%  "
                  f"b_full {f(3):.1f}%  issuing {100 - f(1) - f(2) - f(3):.1f}%", flush=True)
    for b in (x, dy, w, y, dx, dw, sums, ws):
        b.free()
print("totals (ms):", {k: round(v, 3) for k, v in tot.items()})
