"""Throughput of the other BASELINE.json configurations (parity-test cases in bench.py's contract, measured here
so that every model family has a number): cfg3 GUNet 512x512 batch 32, cfg4 UNet3D 64x128x128 batch 4, and
UNet 2-D inference. One JSON line per configuration; CUDA events over `--steps` steps after 3 warm-ups, inputs
resident in HBM.

  python tools/bench_models.py [--which gunet,unet3d,unet_infer] [--steps 5] [--normalizer instance_norm|batch_norm]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--which", default="gunet,unet3d,unet_infer")
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--breakdown", action="store_true")
ap.add_argument("--normalizer", default="instance_norm", choices=["instance_norm", "batch_norm"],
                help="normaliser of the unet3d configuration (cfg4 is instance norm)")
a = ap.parse_args()
ctx = Context(0)
peak = 1371.6
try:
    peak = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))[
        "bf16_tflops_sustained"]
except Exception:  # noqa: BLE001
    pass


def timed(fn, steps):
    for _ in range(3):
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


def breakdown(fn, steps=2):
    import collections
    ctx.profile_begin()
    for _ in range(steps):
        fn()
    rec = ctx.profile_end()
    by = collections.OrderedDict()
    for f, tag, ms in rec:
        by.setdefault(f, [0, 0.0])
        by[f][0] += 1
        by[f][1] += ms
    tot = sum(v[1] for v in by.values()) / steps
    print(f"  sum of bracketed calls {tot:.3f} ms/step", file=sys.stderr)
    for f, (c, ms) in sorted(by.items(), key=lambda kv: -kv[1][1])[:14]:
        print(f"  {ms / steps:8.3f} ms {c // steps:4d}x {f}", file=sys.stderr)
    lay = collections.OrderedDict()
    for f, tag, ms in rec:
        if "conv" in f and "head" not in f:
            lay.setdefault((tag, f), [0, 0.0])
            lay[(tag, f)][0] += 1
            lay[(tag, f)][1] += ms
    for (tag, f), (c, ms) in lay.items():
        print(f"    {ms / c:7.3f} ms  {f:26s} {tag}", file=sys.stderr)
    return rec


for which in a.which.split(","):
    if which == "gunet":
        from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine
        n, hw = 32, 512
        cfg = GUNetConfig(batch=n, height=hw, width=hw, loss_type="xentropy+dice", loss_weight_type="numerical",
                          loss_numeric_w=(0.2, 0.4, 4.4), weight_decay_rate=1e-5, guide_channel=1)
        eng = GUNetEngine(ctx, cfg)
        eng.init_weights(0)
        im, lb = synthetic.make_batch(4, hw, hw, 3)
        im, lb = np.tile(im, (n // 4, 1, 1, 1)), np.tile(lb, (n // 4, 1, 1))
        cx, sg = synthetic.make_guides(im, lb, 200, 1)
        eng.set_inputs(im, lb)
        eng.set_guides(cx, sg)
        ms = timed(lambda: eng.train_step(1e-3), a.steps)
        fl = eng.step_flops()["total"]
        line = {"config": "cfg3 GUNet 2D 512x512 batch 32, context (200-bin) + spatial guide, instance_norm, xentropy+dice, Adam",
                "metric": "gunet_512_train_slices_per_s", "value": n / ms * 1e3, "unit": "slices/s", "ms_per_step": ms,
                "step_tflop_algorithmic": fl / 1e12, "model_tflops_per_s": fl / ms / 1e9,
                "frac_of_sustained_bf16_peak": fl / ms / 1e9 / peak, "loss": sum(eng.read_loss())}
        print(json.dumps(line), flush=True)
        if a.breakdown:
            breakdown(lambda: eng.train_step(1e-3))
        eng.close()
    elif which == "unet3d":
        from boxsegliver_b200.unet3d_engine import UNet3DConfig, UNet3DEngine
        n, d, h, w = 4, 64, 128, 128
        cfg = UNet3DConfig(batch=n, depth=d, height=h, width=w, loss_numeric_w=(1.0, 1.0), normalizer=a.normalizer)
        eng = UNet3DEngine(ctx, cfg)
        eng.init_weights(0)
        im, lb = synthetic.make_volume_batch(n, d, h, w)
        eng.set_inputs(im, lb)
        ms = timed(lambda: eng.train_step(3e-4), a.steps)
        fl = eng.step_flops()["total"]
        line = {"config": f"cfg4 UNet3D 64x128x128 patch, batch 4, {a.normalizer}, weighted xent 1/1, Adam",
                "metric": "unet3d_train_voxels_per_s", "value": n * d * h * w / ms * 1e3, "unit": "voxels/s",
                "patches_per_s": n / ms * 1e3, "ms_per_step": ms, "step_tflop_algorithmic": fl / 1e12,
                "model_tflops_per_s": fl / ms / 1e9, "frac_of_sustained_bf16_peak": fl / ms / 1e9 / peak,
                "loss": sum(eng.read_loss())}
        print(json.dumps(line), flush=True)
        if a.breakdown:
            breakdown(lambda: eng.train_step(3e-4))
        eng.close()
    elif which == "unet_infer":
        from boxsegliver_b200.engine import EngineConfig, UNetEngine
        n, hw = 64, 256
        cfg = EngineConfig(batch=n, height=hw, width=hw, training=False)
        eng = UNetEngine(ctx, cfg)
        eng.init_weights(0)
        im, lb = synthetic.make_batch(n, hw, hw, 3)
        eng.set_inputs(im, lb)

        def infer():
            eng.forward(False)
            eng.predict_outputs(True)
        ms = timed(infer, a.steps)
        fl = eng.step_flops()["fwd"]
        line = {"config": "UNet 2D 256x256x3 inference (eval-mode BN, softmax, masks, argmax, Dice counts), batch 64",
                "metric": "unet2d_256_infer_slices_per_s", "value": n / ms * 1e3, "unit": "slices/s", "ms_per_step": ms,
                "model_tflops_per_s": fl / ms / 1e9, "frac_of_sustained_bf16_peak": fl / ms / 1e9 / peak}
        print(json.dumps(line), flush=True)
        eng.close()
