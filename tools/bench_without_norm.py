"""UNet training-step time with batch norm against --without_norm (conv + bias + ReLU out of the conv epilogue), at the
cfg2 shape (256 x 256, batch 64) and the cfg5 shape (512 x 512, batch 32), and the cost of the bias + ReLU epilogue
itself: bsl_conv2d_fprop against bsl_conv2d_fprop_bias_relu at every 3x3 layer shape of cfg2.

Same method as tools/bench_models.py: CUDA events over `--steps` steps after 3 warm-ups, inputs resident in HBM. The
two variants alternate, `--rounds` times, so that a drift of the box shows as a spread between rounds. The per-layer
comparison alternates the two entry points over `--reps` launches each (after warm-up), per layer shape. One JSON line
per measurement; the first line names the card and its power limit.

  python tools/bench_without_norm.py [--steps 10] [--rounds 2] [--reps 20]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import _lib, synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402
from boxsegliver_b200.engine import EngineConfig, UNetEngine  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--reps", type=int, default=20)
a = ap.parse_args()

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except (OSError, IndexError, subprocess.SubprocessError):
    card = "unknown"
print(json.dumps({"card": card}), flush=True)

ctx = Context(0)


def timed(fn, steps, warm=3):
    for _ in range(warm):
        fn()
    ctx.sync()
    e0, e1 = ctx.new_event(), ctx.new_event()
    ctx.record(e0)
    for _ in range(steps):
        fn()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1) / steps
    ctx.check_device()
    return ms


# ---- whole training steps
SHAPES = {"cfg2": (64, 256), "cfg5": (32, 512)}
VARIANTS = {"batch_norm": dict(normalizer="batch_norm"), "without_norm": dict(without_norm=True)}
for cname, (n, hw) in SHAPES.items():
    im, lb = synthetic.make_batch(4, hw, hw, 3)
    im, lb = np.tile(im, (n // 4, 1, 1, 1)), np.tile(lb, (n // 4, 1, 1))
    engines = {}
    for vname, kw in VARIANTS.items():
        eng = UNetEngine(ctx, EngineConfig(batch=n, height=hw, width=hw, weight_decay_rate=1e-5,
                                           loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4), **kw))
        eng.init_weights(0)
        eng.set_inputs(im, lb)
        engines[vname] = eng
    for r in range(a.rounds):
        for vname, eng in engines.items():
            ms = timed(lambda: eng.train_step(1e-3), a.steps)
            print(json.dumps({"shape": cname, "variant": vname, "round": r, "batch": n, "hw": hw, "ms_per_step": ms,
                              "slices_per_s": n / ms * 1e3, "loss": sum(eng.read_loss())}), flush=True)
    for eng in engines.values():
        eng.close()

# ---- the epilogue alone, at the 3x3 layer shapes of cfg2 (x_ld / y_ld as the engine runs them)
layers = UNetEngine._layer_specs(types.SimpleNamespace(cfg=EngineConfig(batch=64)))
seen = set()
rng = np.random.default_rng(0)
for L in layers:
    if L.kind not in ("stem", "conv"):
        continue
    n = 64
    if L.kind == "stem":
        shape = (n, L.h, L.w, 64, L.cout, 1, 32, L.cout)
    else:
        x_ld = L.cin                                       # (dec1 reads the whole concat buffer: its ld is cin)
        y_ld = 2 * L.cout if L.role == "enc2" else L.cout
        shape = (n, L.h, L.w, L.cin, L.cout, 3, x_ld, y_ld)
    if shape in seen:
        continue
    seen.add(shape)
    n, h, w, cin, cout, k, x_ld, y_ld = shape
    x = ctx.alloc(n * h * w * x_ld * 2)
    chunk = rng.standard_normal(1 << 22).astype(np.float32)           # random bf16 activations, 8 MB at a time
    bits = (chunk.view(np.uint32) >> 16).astype(np.uint16)
    for off in range(0, x.nbytes, bits.nbytes):
        x.upload(bits[:(min(bits.nbytes, x.nbytes - off)) // 2], byte_offset=off)
    wt = ctx.bf16_from_f32((rng.standard_normal((k, k, cin, cout)) * 0.05).astype(np.float32))
    b = ctx.from_numpy((rng.standard_normal(cout) * 0.1).astype(np.float32))
    y = ctx.alloc(n * h * w * y_ld * 2)
    d = _lib.Conv2dDesc(n, h, w, cin, cout, k, k, x_ld, y_ld)
    plain = lambda: ctx.call("bsl_conv2d_fprop", C.byref(d), x.p, wt.p, y.p, ctx.stream)  # noqa: E731
    fused = lambda: ctx.call("bsl_conv2d_fprop_bias_relu", C.byref(d), x.p, wt.p, b.p, y.p, ctx.stream)  # noqa: E731
    res = {"plain": [], "bias_relu": []}
    for r in range(a.rounds):
        res["plain"].append(timed(plain, a.reps))
        res["bias_relu"].append(timed(fused, a.reps))
    fl = 2.0 * n * h * w * k * k * cin * cout
    mp, mf = min(res["plain"]), min(res["bias_relu"])
    print(json.dumps({"layer": L.scope, "n": n, "h": h, "w": w, "cin": cin, "cout": cout, "k": k, "x_ld": x_ld,
                      "y_ld": y_ld, "fprop_ms": res["plain"], "fprop_bias_relu_ms": res["bias_relu"],
                      "delta_pct": 100.0 * (mf - mp) / mp, "fprop_bias_relu_tflops": fl / mf / 1e9}), flush=True)
    for buf in (x, wt, b, y):
        buf.free()
ctx.close()
