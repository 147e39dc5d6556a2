"""Step time of cfg3-shaped GUNet (512x512, batch 32, context + spatial guide, xentropy+dice, Adam) across the
normaliser matrix: batch norm, batch norm + after_affine, batch norm + --dropout 0.5, and instance norm as the
reference point. Same method as tools/bench_models.py: CUDA events over `--steps` steps after 3 warm-ups, inputs
resident in HBM. The variants run in turn, `--rounds` times, so that a drift of the box shows as a spread between
rounds. One JSON line per variant and round; the first line names the card and its power limit.

  python tools/bench_gunet_normalisers.py [--steps 10] [--rounds 2] [--variants bn,bn_aa,bn_drop,in]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402
from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine  # noqa: E402

VARIANTS = {
    "bn": dict(normalizer="batch_norm"),
    "bn_aa": dict(normalizer="batch_norm", after_affine=True),
    "bn_drop": dict(normalizer="batch_norm", dropout=0.5),
    "in": dict(normalizer="instance_norm"),
}

ap = argparse.ArgumentParser()
ap.add_argument("--variants", default="bn,bn_aa,bn_drop,in")
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--rounds", type=int, default=2)
a = ap.parse_args()

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except (OSError, IndexError, subprocess.SubprocessError):
    card = "unknown"
print(json.dumps({"card": card}), flush=True)

ctx = Context(0)
n, hw = 32, 512
im, lb = synthetic.make_batch(4, hw, hw, 3)
im, lb = np.tile(im, (n // 4, 1, 1, 1)), np.tile(lb, (n // 4, 1, 1))
cx, sg = synthetic.make_guides(im, lb, 200, 1)


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


for r in range(a.rounds):
    for name in a.variants.split(","):
        cfg = GUNetConfig(batch=n, height=hw, width=hw, loss_type="xentropy+dice", loss_weight_type="numerical",
                          loss_numeric_w=(0.2, 0.4, 4.4), weight_decay_rate=1e-5, guide_channel=1, **VARIANTS[name])
        eng = GUNetEngine(ctx, cfg)
        eng.init_weights(0)
        eng.set_inputs(im, lb)
        eng.set_guides(cx, sg)
        ms = timed(lambda: eng.train_step(1e-3), a.steps)
        print(json.dumps({"variant": name, "round": r, "config": {k: v for k, v in VARIANTS[name].items()},
                          "ms_per_step": ms, "slices_per_s": n / ms * 1e3, "loss": sum(eng.read_loss())}), flush=True)
        eng.close()
