#!/usr/bin/env python
"""Headline benchmark of the U-Net training hot path (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W [--config cfg2|cfg3|cfg4|cfg5]   # this repo (sm_100a kernels)
  python bench.py --impl reference --steps K --warmup W                          # the reference path's CPU stand-in

Workloads (BASELINE.json `configs`, SURVEY.md section 8d); a step = fwd + loss + bwd + gradient all-reduce + optimizer:
  cfg2 (default)  UNet 2-D 256x256x3 bf16, batch 64 per GPU, batch norm, weighted xent 0.2/0.4/4.4 + L2, Adam
  cfg3            GUNet 2-D 512x512, batch 32 per GPU, 200-bin context + spatial guide, instance norm, xent + dice
  cfg4            UNet3D 64x128x128 patches, batch 4 per GPU, instance norm (voxels/s)
  cfg5            UNet 2-D 512x512 data parallel: weak scaling at 32 per GPU, and the strong-scaling points of global
                  batch 256 that fit one GPU's memory (128 / 64 / 32 per GPU at N = 2 / 4 / 8)
                  (/root/reference/run_scripts/template/001_dist.sh:36, utils/distribution_utils.py:107-134)
The default line is cfg2 and carries an `other_configs` block with short runs (5 steps after 3 warm-ups) of cfg3, cfg4
and cfg5 at the same N, so that one driver invocation per N times every BASELINE configuration.

 * `value`   = units/s over all N GPUs, inputs resident in HBM, K steps timed with CUDA events on the compute stream,
               bracketed by barrier + stream sync, MAX over ranks.
 * `e2e`     = the same step through the host-fed call (pinned host batch -> H2D -> step -> D2H loss), wall clock.
 * `roofline`= whole step: algorithmic conv FLOPs of one step / step time, against the measured sustained bf16 peak of
               MEASURED_PEAKS.json. `kernels_frac` is the conv-launches-only figure (every tcgen05 launch of K extra
               steps bracketed by CUDA events, filter-gradient overlap off so that each kernel is timed alone).
 * `dp_check`= (N > 1) after the timed steps: CRC-32C of every rank's fp32 weight arena (must be identical), and
               max |NCCL-reduced gradient - sum over ranks of the local gradients| from one extra untimed backward.
 * `cpu_baseline` / `--impl reference`: the reference's own implementation is TensorFlow 1.13, which cannot be
               installed in this image (Python 3.12, no network; SURVEY.md section 0). The stand-in is the torch-CPU
               (oneDNN/MKL) restatement of the same training step (oracle/unet_torch.py) on cfg1 = batch 8 of 256x256x3
               fp32, all host cores, thread count printed; the numpy/BLAS port is kept as a second key.
 * `--dump-outputs DIR` (rank 0): after the K timed steps, what the last of them left for its caller, as .npy files
               (see dump_outputs). Inputs and initial weights are seeded, so two builds of the project run with the
               same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_SLICE_256 = 288.828e9  # BASELINE.md section 3, UNet 2-D 256x256x3, 3 classes, fwd+bwd

WORKLOADS = {
    "cfg2": dict(model="unet", hw=256, per_gpu_batch=64, unit="slices/s", metric="unet2d_256_train_slices_per_s",
                 baseline_config="configs[1]",
                 workload="UNet 2D 256x256x3 bf16 training (fwd+loss+bwd+allreduce+Adam), batch 64 per GPU "
                          "(BASELINE.json configs[1])"),
    "cfg3": dict(model="gunet", hw=512, per_gpu_batch=32, unit="slices/s", metric="gunet_512_train_slices_per_s",
                 baseline_config="configs[2]",
                 workload="GUNet 2D 512x512 bf16 training, batch 32 per GPU, 200-bin context + spatial guide, "
                          "instance norm, xentropy+dice (BASELINE.json configs[2])"),
    "cfg4": dict(model="unet3d", dhw=(64, 128, 128), per_gpu_batch=4, unit="voxels/s",
                 metric="unet3d_train_voxels_per_s", baseline_config="configs[3]",
                 workload="UNet3D 64x128x128 bf16 training, batch 4 per GPU, instance norm, weighted xent "
                          "(BASELINE.json configs[3])"),
    "cfg5": dict(model="unet", hw=512, per_gpu_batch=32, unit="slices/s", metric="unet2d_512_train_slices_per_s",
                 baseline_config="configs[4]", strong_global_batch=256,
                 workload="UNet 2D 512x512 bf16 data-parallel training, 32 per GPU weak scaling + global batch 256 "
                          "strong-scaling points (BASELINE.json configs[4])"),
}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_torch_throughput(steps: int, warmup: int, batch: int = 8, budget_s: float = 240.0):
    """oracle.unet_torch.train_step (torch-CPU, oneDNN/MKL, fp32) on cfg1: `batch` slices of 256x256x3, BN, weighted
    xent 0.2/0.4/4.4, L2, Adam. All host cores. Stops early (and says so) if `budget_s` would be exceeded."""
    import torch
    from boxsegliver_b200 import synthetic
    from oracle import unet_ref as R
    from oracle import unet_torch as T

    cores = host_cores()
    torch.set_num_threads(cores)
    cfg = R.UNetCfg(height=256, width=256, channel=3, loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4),
                    weight_decay_rate=1e-6)
    p = T.to_torch_params(R.init_params(cfg, seed=0))
    images, labels = synthetic.make_batch(batch, 256, 256, 3)
    x = torch.tensor(images).permute(0, 3, 1, 2).contiguous()
    y = torch.tensor(labels, dtype=torch.int64)
    slots, times, t_all = {}, [], time.perf_counter()
    done_w = 0
    for i in range(warmup):
        T.train_step(p, slots, i + 1, x, y, cfg, 1e-3)
        done_w += 1
        if time.perf_counter() - t_all > budget_s / 4:
            break
    for i in range(steps):
        t0 = time.perf_counter()
        T.train_step(p, slots, done_w + i + 1, x, y, cfg, 1e-3)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    sec = sum(times) / len(times)
    return {"slices_per_s": batch / sec, "sec_per_step": sec, "steps": len(times), "warmup": done_w, "batch": batch,
            "threads": torch.get_num_threads(), "cores": cores, "gflops": batch * FLOP_PER_SLICE_256 / sec / 1e9}


def cpu_port_throughput(steps: int = 1, batch: int = 1):
    """oracle.unet_ref.train_step (fp32, numpy + BLAS) on `batch` slices of 256x256x3: the second CPU figure."""
    from boxsegliver_b200 import synthetic
    from oracle import unet_ref as R

    cfg = R.UNetCfg(height=256, width=256, channel=3, loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4),
                    weight_decay_rate=1e-6)
    params = R.init_params(cfg, seed=0)
    slots = {}
    images, labels = synthetic.make_batch(batch, 256, 256, 3)
    times = []
    for i in range(steps):
        t0 = time.perf_counter()
        R.train_step(params, slots, i + 1, images, labels, cfg, 1e-3)
        times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return {"slices_per_s": batch / sec, "sec_per_step": sec, "steps": len(times), "batch": batch}


def cpu_baseline_block(r):
    return {"value": r["slices_per_s"], "unit": "slices/s", "cores": r["cores"], "threads": r["threads"], "kind": "port",
            "gflops": r["gflops"], "sec_per_step": r["sec_per_step"],
            "sample": f"{r['steps']} training step(s) after {r['warmup']} warm-up(s) of cfg1 = batch {r['batch']} at "
                      f"256x256x3 fp32 (BN, weighted xent, L2, Adam) with the torch-CPU/oneDNN restatement "
                      f"(oracle/unet_torch.py), {r['threads']} threads on {r['cores']} cores; the reference's "
                      f"TensorFlow 1.13 cannot be installed here"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    r = cpu_torch_throughput(steps=max(1, args.steps), warmup=max(0, args.warmup))
    w = WORKLOADS["cfg2"]
    line = {
        "impl": "reference", "metric": w["metric"], "value": r["slices_per_s"], "unit": "slices/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["sec_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["workload"],
                   "sample": "bounded sample of that workload: cfg1 = batch 8 per step, fp32 (BASELINE.json configs[0], "
                             "the reference's own CPU-runnable case)",
                   "per_gpu_batch": w["per_gpu_batch"], "classes": 3, "normalizer": "batch_norm"},
        "cpu_baseline": cpu_baseline_block(r),
        "e2e": {"value": r["slices_per_s"], "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_numpy_port:
        q = cpu_port_throughput(steps=1, batch=1)
        line["cpu_baseline"]["numpy_port"] = {"value": q["slices_per_s"], "unit": "slices/s",
                                              "sample": "1 step of batch 1 with the numpy/BLAS oracle (oracle/unet_ref.py)"}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.path = tempfile.mktemp(prefix="bsl_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        try:
            with open(self.path) as f:
                for ln in f:
                    parts = [p.strip() for p in ln.split(",")]
                    if len(parts) < 9:
                        continue
                    try:
                        a, b, c = float(parts[1]), float(parts[2]), float(parts[3])
                    except ValueError:
                        continue
                    sm.append(a)
                    mx.append(b)
                    pw.append(c)
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                       parts[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:  # noqa: BLE001
            pass
        if sm:
            # "under load" = samples drawing at least 60 % of the highest power seen in the window
            lim = 0.6 * max(pw)
            load = [a for a, c in zip(sm, pw) if c >= lim] or sm
            out.update(sm_mhz=statistics.median(load), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       samples_under_load=len(load), power_w_max=max(pw))
        return out


# ------------------------------------------------------------------------------------------------ engines
def _tile(a, n):
    import numpy as np
    reps = (n + a.shape[0] - 1) // a.shape[0]
    return np.ascontiguousarray(np.tile(a, (reps,) + (1,) * (a.ndim - 1))[:n])


def build_engine(ctx, name: str, batch: int, world: int, rank: int):
    """Engine + device-resident synthetic inputs of workload `name`; returns (engine, units per step per GPU, lr)."""
    from boxsegliver_b200 import synthetic
    w = WORKLOADS[name]
    if w["model"] == "unet":
        from boxsegliver_b200.engine import EngineConfig, UNetEngine
        hw = w["hw"]
        cfg = EngineConfig(batch=batch, height=hw, width=hw, channel=3, classes=("Background", "Liver", "Tumor"),
                           normalizer="batch_norm", weight_decay_rate=1e-6, loss_type="xentropy",
                           loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4), optimizer="adam", world=world)
        eng = UNetEngine(ctx, cfg)
        eng.init_weights(seed=0)      # identical on every rank (mirrored variables)
        # distinct slices per rank; large batches repeat a 64-slice set (the kernels do not depend on the data)
        images, labels = synthetic.make_batch(min(batch, 64), hw, hw, 3, seed=1357 + rank)
        eng.set_inputs(_tile(images, batch), _tile(labels, batch))
        return eng, batch, 1e-3
    if w["model"] == "gunet":
        from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine
        hw = w["hw"]
        cfg = GUNetConfig(batch=batch, height=hw, width=hw, loss_type="xentropy+dice", loss_weight_type="numerical",
                          loss_numeric_w=(0.2, 0.4, 4.4), weight_decay_rate=1e-5, guide_channel=1, world=world)
        eng = GUNetEngine(ctx, cfg)
        eng.init_weights(0)
        im, lb = synthetic.make_batch(8, hw, hw, 3, seed=1357 + rank)
        im, lb = _tile(im, batch), _tile(lb, batch)
        cx, sg = synthetic.make_guides(im, lb, 200, 1)
        eng.set_inputs(im, lb)
        eng.set_guides(cx, sg)
        return eng, batch, 1e-3
    from boxsegliver_b200.unet3d_engine import UNet3DConfig, UNet3DEngine
    d, h, wd = w["dhw"]
    cfg = UNet3DConfig(batch=batch, depth=d, height=h, width=wd, loss_numeric_w=(1.0, 1.0), world=world)
    eng = UNet3DEngine(ctx, cfg)
    eng.init_weights(0)
    im, lb = synthetic.make_volume_batch(batch, d, h, wd, seed=1357 + rank)
    eng.set_inputs(im, lb)
    return eng, batch * d * h * wd, 3e-4


class Harness:
    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist  # control plane only: id broadcast, barriers, max over ranks
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group(backend="gloo", rank=self.rank, world_size=self.world)
            self.dist = dist
        from boxsegliver_b200.device import Context
        self.ctx = Context(self.local)
        self.uid = None
        if self.world > 1:
            import ctypes as C
            uid = (C.c_char * 128)()
            if self.rank == 0:
                self.ctx.call("bsl_comm_unique_id", uid)
            box = [bytes(uid)]
            self.dist.broadcast_object_list(box, src=0)
            self.uid = box[0]

    def barrier(self):
        self.ctx.sync()
        if self.dist is not None:
            self.dist.barrier()

    def max_over_ranks(self, vals):
        if self.dist is None:
            return list(vals)
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def launches(self):
        import ctypes as C
        n = C.c_ulonglong()
        self.ctx.call("bsl_launch_count", C.byref(n))
        return n.value

    def engine(self, name, batch):
        eng, units, lr = build_engine(self.ctx, name, batch, self.world, self.rank)
        if self.world > 1:
            eng.attach_comm(self.rank, self.world, self.uid)
        return eng, units, lr

    def time_steps(self, eng, lr, steps, warmup):
        """(ms per step max over ranks, kernel launches in the timed region) for device-resident inputs."""
        ctx = self.ctx
        for _ in range(warmup):
            eng.train_step(lr)
        self.barrier()
        l0 = self.launches()
        e0, e1 = ctx.new_event(), ctx.new_event()
        ctx.record(e0)
        for _ in range(steps):
            eng.train_step(lr)
        ctx.record(e1)
        ms_total = ctx.elapsed_ms(e0, e1)
        self.barrier()
        n_launch = self.launches() - l0
        ctx.check_device()
        return self.max_over_ranks([ms_total])[0] / steps, n_launch

    def short_run(self, name, batch, steps=5, warmup=3, label=None):
        """One entry of `other_configs`: build, warm up, time, free."""
        w = WORKLOADS[name]
        eng, units, lr = self.engine(name, batch)
        ms, _ = self.time_steps(eng, lr, steps, warmup)
        fl = eng.step_flops()["total"]
        loss = sum(eng.read_loss())
        eng.close()
        peaks, _ = measured_peaks()
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        return {"workload": label or w["workload"], "baseline_config": w["baseline_config"], "metric": w["metric"],
                "unit": w["unit"], "value": self.world * units / (ms / 1e3), "ms_per_step": ms, "steps": steps,
                "warmup": warmup, "per_gpu_batch": batch, "global_batch": batch * self.world, "n_gpus": self.world,
                "step_tflop_algorithmic_per_gpu": fl / 1e12, "frac_of_sustained_bf16_peak": fl / (ms / 1e3) / 1e12 / peak,
                "last_loss": loss}

    def fits(self, name, batch) -> bool:
        """Does a `batch`-per-GPU engine of workload `name` fit the free memory of this GPU? (activations + gradients
        scale with batch x pixels: 13.3 GB measured at 64 x 256^2 on the 2-D U-Net; 25 % head-room)"""
        w = WORKLOADS[name]
        if w["model"] != "unet":
            return True
        need = 13.3e9 * batch * w["hw"] ** 2 / (64 * 256 ** 2) * 1.25 + 2e9
        free, _ = self.ctx.mem_info()
        ok = [1.0 if need < free else 0.0]
        if self.dist is not None:
            import torch
            t = torch.tensor(ok, dtype=torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
            ok = [float(t[0])]
        return ok[0] > 0.5


DUMP_SAMPLE = 1 << 21   # values kept of a larger output: five files of at most 8 MB each stay under 64 MB


def dump_outputs(eng, out_dir: str):
    """Writes what the training step just run computed, as a caller reads it back: loss.npy (float64 [data loss, L2
    loss]), logits.npy, grads.npy (flat trainable-gradient arena), weights.npy (flat fp32 weight arena after the
    optimizer update) and, for batch norm, moving_stats.npy, all float32. An output of more than DUMP_SAMPLE values is
    reduced to DUMP_SAMPLE of them at sorted positions drawn with a fixed seed from its length alone, so the same
    positions are kept on every run (and grads / weights keep the same parameters)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    data, reg = eng.read_loss()
    outputs = {"loss": np.array([data, reg], np.float64),
               "logits": eng.logits.download(np.float32, (eng.logits.nbytes // 4,)),
               "grads": eng.G.download(np.float32, (eng.n_train,)),
               "weights": eng.W.download(np.float32, (eng.n_train,))}
    if getattr(eng, "n_stats", 0) > 0:
        outputs["moving_stats"] = eng.S.download(np.float32, (eng.n_stats,))
    for name, a in outputs.items():
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def dp_check(h: Harness, eng, lr):
    """Correctness of the data-parallel step, carried in the bench line (N > 1).
    (1) every rank's fp32 weight arena has the same CRC-32C after the timed steps;
    (2) one extra backward WITHOUT the exchange gives the local gradients; their sum over ranks (gloo, fp64 on the
        host) is compared with the NCCL-reduced gradients of the same backward run again with the exchange."""
    import numpy as np
    import torch
    from boxsegliver_b200 import checkpoint
    ctx = h.ctx
    ctx.sync()
    wbytes = eng.W.download(np.uint8, (eng.n_train * 4,))
    crc = checkpoint.crc32c(wbytes)
    crcs = [None] * h.world
    h.dist.all_gather_object(crcs, int(crc))
    eng._skip_exchange = True
    eng.forward(True)
    eng.loss_backward()
    ctx.sync()
    local = eng.G.download(np.float32, (eng.n_train,))
    eng._skip_exchange = False
    eng.forward(True)
    if eng.cfg.normalizer == "batch_norm":
        eng._allreduce_moving_stats()
    eng.loss_backward()
    eng._allreduce_grads()
    ctx.sync()
    reduced = eng.G.download(np.float32, (eng.n_train,))
    t = torch.from_numpy(local.astype(np.float64))
    h.dist.all_reduce(t)
    want = t.numpy()
    err = float(np.abs(reduced.astype(np.float64) - want).max())
    scale = float(np.abs(want).max())
    errs = h.max_over_ranks([err])
    return {"dp_weights_identical": len(set(crcs)) == 1, "weight_crc32c": [f"{c:08x}" for c in crcs],
            "grad_sum_max_abs_err": errs[0], "grad_max_abs": scale, "grad_sum_rel_err": errs[0] / max(scale, 1e-30),
            "note": "reduced = ncclAllReduce(sum) of loss-pre-scaled (1/N) local gradients; compared with the fp64 "
                    "host sum of the ranks' local gradients from the same backward run without the exchange"}


def run_b200(args):
    import numpy as np

    h = Harness(args)
    ctx, rank, world = h.ctx, h.rank, h.world
    name = args.config
    w = WORKLOADS[name]
    batch = args.batch or w["per_gpu_batch"]
    warmup = max(args.warmup, 3)

    sampler = ClockSampler(h.local) if rank == 0 else None   # started before warm-up: nvidia-smi takes ~1 s to spin up
    eng, units, lr = h.engine(name, batch)
    ms, n_launch = h.time_steps(eng, lr, args.steps, warmup)
    if args.dump_outputs and rank == 0:     # before the untimed steps below move the weights on
        dump_outputs(eng, args.dump_outputs)

    # ---- roofline side measurement (2-D engines): the same K steps again with every tensor-core launch bracketed by
    # CUDA events on its stream and the filter-gradient side stream folded back into the compute stream, so that each
    # kernel is timed ALONE (with the overlap on, a bracket also contains time shared with the normalisation backward).
    conv = None
    if hasattr(eng, "enable_conv_timing"):
        eng.enable_conv_timing(True)
        overlap_was, eng._overlap_wgrad = eng._overlap_wgrad, False
        for _ in range(args.steps):
            eng.train_step(lr)
        conv = eng.conv_timing_report()
        eng.enable_conv_timing(False)
        eng._overlap_wgrad = overlap_was
    clocks = sampler.stop() if sampler else None
    ctx.check_device()

    # ---- end-to-end arm: host batches in (pinned memory -> H2D every step), loss out (D2H every step). The copy of
    # batch i + 1 is submitted before step i is launched, on a copy stream, and overlaps its compute.
    e2e = None
    if hasattr(eng, "staging_slot"):
        images = eng.images.download(np.float32, (batch, eng.cfg.height, eng.cfg.width, eng.cfg.channel))
        labels = eng.labels.download(np.int32, (batch, eng.cfg.height, eng.cfg.width))
        for j in (0, 1):
            si, sl = eng.staging_slot(j)
            si[...] = images
            sl[...] = labels
        eng.submit_staged(0)
        for i in range(2):
            eng.submit_staged((i + 1) % 2)
            eng.train_step_prefetched(lr)
        h.barrier()
        e0, e1 = ctx.new_event(), ctx.new_event()
        t0 = time.perf_counter()
        ctx.record(e0)
        loss = 0.0
        for i in range(args.steps):
            eng.submit_staged((i + 1) % 2)          # next batch's H2D (K copies for K timed steps)
            loss = eng.train_step_prefetched(lr)    # waits for its own batch's copy, runs the step, reads the loss back
        ctx.record(e1)
        e2e_ms_total = ctx.elapsed_ms(e0, e1)
        e2e_wall = (time.perf_counter() - t0) * 1e3
        e2e_ms_total = max(e2e_ms_total, e2e_wall)  # the host waits on the loss every step: wall clock is the honest one
        ctx.sync(eng.copy_stream)
        h.barrier()
        ctx.check_device()
        e2e_ms_total = h.max_over_ranks([e2e_ms_total])[0]
        e2e = {"value": world * units * args.steps / (e2e_ms_total / 1e3), "unit": w["unit"],
               "h2d_bytes_per_step": eng.h2d_bytes_per_step(), "d2h_bytes_per_step": 12, "last_loss": loss}

    dp = dp_check(h, eng, lr) if (world > 1 and hasattr(eng, "_skip_exchange")) else None
    fl = eng.step_flops()
    cfg_norm = eng.cfg.normalizer
    wgrad_overlap = bool(getattr(eng, "_overlap_wgrad", False))
    eng.close()

    # ---- the other BASELINE configurations, short runs at the same N
    others = {}
    if name == "cfg2" and not args.no_other_configs:
        for other in ("cfg3", "cfg4", "cfg5"):
            others[other] = h.short_run(other, WORKLOADS[other]["per_gpu_batch"])
    if (name == "cfg5" or (name == "cfg2" and not args.no_other_configs)) and world > 1:
        g = WORKLOADS["cfg5"]["strong_global_batch"]
        if g % world == 0 and g // world != WORKLOADS["cfg5"]["per_gpu_batch"]:
            if h.fits("cfg5", g // world):
                others["cfg5_strong"] = h.short_run(
                    "cfg5", g // world, label=f"UNet 2D 512x512 data parallel, global batch {g} = {g // world} per GPU "
                                              f"(strong-scaling point of BASELINE.json configs[4])")
            else:
                others["cfg5_strong"] = {"skipped": f"{g // world} slices of 512x512 per GPU exceed the free HBM"}
        elif g % world == 0:
            others["cfg5_strong"] = {"same_as": "cfg5", "note": f"global batch {g} on {world} GPUs IS the weak point "
                                                                f"({g // world} per GPU)"}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        value = world * units / (ms / 1e3)
        peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        burst = float(peaks.get("bf16_tflops", peak))
        step_tflops = fl["total"] / (ms / 1e3) / 1e12          # per GPU: every rank runs the same step
        roof = {"bound": "tensor", "achieved": step_tflops, "peak": peak, "unit": "TFLOP/s",
                "frac": step_tflops / peak, "frac_of_burst_peak": step_tflops / burst, "traffic": None,
                "traffic_note": "DRAM bytes are not measurable inside this run; the ncu --set full captures of the "
                                "conv kernels are summarised under profiles/ (r01_traffic.json, r02_*)",
                "scope": "whole training step: algorithmic conv FLOPs of one step (2*MACs, un-padded) / step time",
                "peak_source": f"{peak_src} MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"}
        if conv is not None and conv["ms"] > 0:
            kt = conv["flops"] / (conv["ms"] / 1e3) / 1e12
            roof.update(
                kernels_achieved=kt, kernels_frac=kt / peak, kernels_launches_timed=conv["launches"],
                kernels_ms_per_step=conv["ms"] / args.steps,
                kernels="bsl::conv_halo_kernel (single CTAs and cta_group::2 CTA pairs) + bsl::wgrad_halo3_kernel / wgrad_halo_kernel + bsl::igemm_kernel (every tcgen05 conv / convT "
                        "fprop, dgrad, wgrad launch of K extra steps, CUDA events on the launching stream, overlap off)",
                per_kind={k: {"launches_per_step": v[0] // args.steps, "ms_per_step": v[1] / args.steps,
                              "tflops": v[2] / (v[1] / 1e3) / 1e12 if v[1] > 0 else 0.0}
                          for k, v in conv["per_kind"].items()})
        line = {
            "metric": w["metric"], "value": value, "unit": w["unit"], "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": w["workload"], "baseline_config": w["baseline_config"], "per_gpu_batch": batch,
                       "global_batch": batch * world, "classes": 3 if w["model"] != "unet3d" else 2,
                       "normalizer": cfg_norm, "optimizer": "adam", "parallelism": f"dp{world}",
                       "wgrad_overlap": wgrad_overlap,
                       "l2_cache": "inputs larger than L2: every step touches > 10 GB of activations/gradients"},
            "model_tflops_per_s": step_tflops * world,
            "step_tflop_algorithmic": fl["total"] / 1e12,
            "roofline": roof,
            "e2e": e2e,
            "gpu_launches": int(n_launch),
            "clocks": clocks,
        }
        if dp is not None:
            line["dp_check"] = dp
        if others:
            line["other_configs"] = others
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_torch_throughput(steps=2, warmup=1, budget_s=60.0)
            line["cpu_baseline"] = cpu_baseline_block(r)
        print(json.dumps(line), flush=True)
    if h.dist is not None:
        h.dist.barrier()
        h.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-other-configs", dest="no_other_configs", action="store_true")
    ap.add_argument("--no-numpy-port", dest="no_numpy_port", action="store_true")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
