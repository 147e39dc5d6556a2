"""Which gradients differ between engine schedules (tuning aid for the bit-identity test)?

  [BSL_LIB=...] python tools/schedule_diff.py

Runs two training steps of the small U-Net under each schedule (default twice, to separate run-to-run differences
from schedule differences) and prints, per schedule, the gradient tensors that are not bit-identical to the first run.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402
from boxsegliver_b200.engine import EngineConfig, UNetEngine  # noqa: E402

ctx = Context(0)
n, hw = 8, 64
images, labels = synthetic.make_batch(n, hw, hw, 3, seed=1401)
names = ["default", "default again", "no overlap", "no head fusion", "no head bwd"]
flags = [dict(), dict(), dict(_overlap_wgrad=False), dict(_fuse_head=False), dict(_fuse_head_bwd=False)]
ref = None
for name, fl in zip(names, flags):
    eng = UNetEngine(ctx, EngineConfig(batch=n, height=hw, width=hw, weight_decay_rate=1e-5,
                                       loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4)))
    for k, v in fl.items():
        setattr(eng, k, v)
    eng.init_weights(seed=5)
    eng.set_inputs(images, labels)
    per_step = []
    for _ in range(2):
        eng.train_step(1e-3)
        ctx.check_device()
        per_step.append(eng.get_grads())
    eng.close()
    if ref is None:
        ref = per_step
        continue
    for st in range(2):
        bad = [(k, float(np.abs(g - per_step[st][k]).max()), float(np.abs(g).max())) for k, g in ref[st].items()
               if not np.array_equal(g, per_step[st][k])]
        print(f"{name:16s} step {st}: {len(bad)} tensors differ", [(k.replace('UNet/', ''), f'{d:.2e}/{m:.2e}') for k, d, m in bad[:6]])
