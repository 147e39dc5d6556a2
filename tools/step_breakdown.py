"""Per-call device-time breakdown of one U-Net training step (CUDA events around every C-ABI enqueue).

  python tools/step_breakdown.py [--batch 64] [--hw 256] [--steps 3] [--json gpurun_out/breakdown.json]

Prints (a) time per C-ABI function, (b) per layer and pass for the tensor-core convs with algorithmic
TFLOP/s, so the kernel work can be aimed at the worst shapes. Events serialise nothing (same stream),
but they do add a little launch overhead: use bench.py for the headline number.
"""
import argparse
import collections
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402
from boxsegliver_b200.engine import EngineConfig, UNetEngine  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--hw", type=int, default=256)
ap.add_argument("--steps", type=int, default=3)
ap.add_argument("--normalizer", default="batch_norm")
ap.add_argument("--json", default="")
a = ap.parse_args()

ctx = Context(0)
eng = UNetEngine(ctx, EngineConfig(batch=a.batch, height=a.hw, width=a.hw, normalizer=a.normalizer,
                                   weight_decay_rate=1e-6, loss_weight_type="numerical",
                                   loss_numeric_w=(0.2, 0.4, 4.4)))
eng.init_weights(0)
im, lb = synthetic.make_batch(a.batch, a.hw, a.hw, 3)
eng.set_inputs(im, lb)
for _ in range(3):
    eng.train_step(1e-3)
ctx.sync()
ctx.profile_begin()
for _ in range(a.steps):
    eng.train_step(1e-3)
rec = ctx.profile_end()
ctx.check_device()

flops = {L.scope: eng._flops(L) for L in eng.layers}
by_fn = collections.OrderedDict()
by_layer = collections.OrderedDict()
for fn, tag, ms in rec:
    by_fn.setdefault(fn, [0, 0.0])
    by_fn[fn][0] += 1
    by_fn[fn][1] += ms
    by_layer.setdefault((tag, fn), [0, 0.0])
    by_layer[(tag, fn)][0] += 1
    by_layer[(tag, fn)][1] += ms
tot = sum(v[1] for v in by_fn.values()) / a.steps
print(f"sum of bracketed calls: {tot:.3f} ms/step")
for fn, (cnt, ms) in sorted(by_fn.items(), key=lambda kv: -kv[1][1]):
    print(f"  {ms / a.steps:8.3f} ms  {cnt // a.steps:4d}x  {100 * ms / a.steps / tot:5.1f}%  {fn}")
print("tensor-core convs per layer:")
TC = ("bsl_conv2d_fprop", "bsl_conv2d_fprop_stats", "bsl_conv2d_dgrad", "bsl_conv2d_wgrad", "bsl_convT2d_fwd", "bsl_convT2d_bwd_data",
      "bsl_convT2d_bwd_filter")
rows = []
for (tag, fn), (cnt, ms) in by_layer.items():
    if fn in TC:
        t = ms / cnt
        tf = flops[tag] / (t * 1e-3) / 1e12
        rows.append({"layer": tag, "fn": fn, "ms": t, "tflops": tf})
        print(f"  {t:7.3f} ms {tf:7.1f} TF/s  {fn:24s} {tag}")
# HBM-bound passes: algorithmic bytes (DESIGN.md section 3.2) / time, against the measured copy bandwidth
L_by_scope = {L.scope: L for L in eng.layers}
n = a.batch


def alg_bytes(fn, L):
    px_out = n * L.h * L.w * (4 if L.kind == "convT" else 1)
    c = L.cout
    full = px_out * c * 2
    return {"bsl_norm_apply_mod": 2 * full, "bsl_norm_apply": 2 * full, "bsl_norm_apply_pool_mod": 2.25 * full,
            "bsl_norm_apply_pool": 2.25 * full, "bsl_norm_stats": full, "bsl_norm_bwd_reduce": 2 * full,
            "bsl_norm_bwd_apply": 3 * full, "bsl_maxpool2x2_bwd_add": 3.25 * full, "bsl_relu_bwd": 3 * full,
            "bsl_stem_im2col": n * L.h * L.w * (L.cin * 4 + 128),
            "bsl_stem_im2col_ld": n * L.h * L.w * (L.cin * 4 + 2 * (32 if 9 * L.cin <= 32 else 64)),
            "bsl_conv2d_head_fprop": n * L.h * L.w * (L.cin * 2 + 4 * L.cout),
            "bsl_conv2d_head_dgrad": n * L.h * L.w * (L.cin * 2 + 4 * L.cout),
            "bsl_norm_bwd_reduce_head": full + px_out * 12, "bsl_norm_bwd_apply_head": 2 * full + px_out * 12,
            "bsl_norm_bwd_apply_mod": 3 * full, "bsl_relu_bwd_bias": 3 * full,
            "bsl_norm_apply_head": 2 * full + px_out * 12,
            "bsl_conv2d_head_wgrad": n * L.h * L.w * (L.cin * 2 + 4 * L.cout)}.get(fn)


print("HBM-bound passes per layer (algorithmic GB/s; measured copy peak 6541.8 GB/s):")
mem_rows = []
agg = collections.OrderedDict()
for (tag, fn), (cnt, ms) in by_layer.items():
    L = L_by_scope.get(tag)
    b = alg_bytes(fn, L) if L is not None else None
    if b is None:
        continue
    t = ms / cnt
    gbs = b / (t * 1e-3) / 1e9
    mem_rows.append({"layer": tag, "fn": fn, "ms": t, "gbs": gbs})
    g = agg.setdefault(fn, [0.0, 0.0])
    g[0] += b
    g[1] += t
    print(f"  {t:7.3f} ms {gbs:7.0f} GB/s  {fn:26s} {tag}")
print("HBM-bound passes, whole step:")
for fn, (b, t) in agg.items():
    print(f"  {t:7.3f} ms {b / (t * 1e-3) / 1e9:7.0f} GB/s ({100 * b / (t * 1e-3) / 1e9 / 6541.8:4.1f}% of peak)  {fn}")
if a.json:
    with open(a.json, "w") as f:
        json.dump({"ms_per_step_bracketed": tot, "by_fn": {k: [v[0] // a.steps, v[1] / a.steps] for k, v in by_fn.items()},
                   "tc_layers": rows, "mem_layers": mem_rows}, f, indent=1)
