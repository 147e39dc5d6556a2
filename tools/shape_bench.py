"""Training-step / inference time of the 2-D UNet engine at an arbitrary slice shape (the shipped scripts train at 256 x 256,
512 x 160, 480 x 160 and evaluate at 960 x 320). CUDA events over --steps steps after 3 warm-ups.

  python tools/shape_bench.py --h 512 --w 160 --batch 32 [--infer] [--normalizer instance_norm]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402
from boxsegliver_b200.engine import EngineConfig, UNetEngine  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--h", type=int, default=512)
ap.add_argument("--w", type=int, default=160)
ap.add_argument("--batch", type=int, default=32)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--normalizer", default="batch_norm")
ap.add_argument("--infer", action="store_true")
a = ap.parse_args()
ctx = Context(0)
eng = UNetEngine(ctx, EngineConfig(batch=a.batch, height=a.h, width=a.w, normalizer=a.normalizer, training=not a.infer,
                                   loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4)))
eng.init_weights(0)
eng.set_inputs(*synthetic.make_batch(a.batch, a.h, a.w, 3))


def step():
    if a.infer:
        eng.forward(False)
        eng.predict_outputs(True)
    else:
        eng.train_step(1e-3)


for _ in range(3):
    step()
ctx.sync()
e0, e1 = ctx.new_event(), ctx.new_event()
ctx.record(e0)
for _ in range(a.steps):
    step()
ctx.record(e1)
ms = ctx.elapsed_ms(e0, e1) / a.steps
ctx.check_device()
fl = eng.step_flops()["fwd" if a.infer else "total"]
print(json.dumps({"shape": f"{a.batch} x {a.h} x {a.w}", "mode": "inference" if a.infer else "training", "normalizer": a.normalizer,
                  "ms_per_step": ms, "slices_per_s": a.batch / ms * 1e3,
                  "model_tflops_per_s": fl / ms / 1e9}))
