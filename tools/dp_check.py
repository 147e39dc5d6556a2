"""Data-parallel correctness on real GPUs (run under torchrun, one rank per GPU):

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/dp_check.py [unet3d]

Checks, for the 2-D U-Net engine with the bucketed all-reduce overlapped with backward (or, with `unet3d`, for the
3-D U-Net engine with --normalizer batch_norm and its whole-arena gradient all-reduce):
  1. the all-reduced gradient arena equals the SUM over ranks of the local gradients (computed first without the
     communicator and exchanged through gloo), to fp32 rounding of a different summation order;
  2. batch-norm moving statistics are the cross-replica MEAN of the per-replica updates;
  3. after 3 training steps every rank holds bit-identical weights (mirrored variables stay mirrored).
MirroredStrategy semantics: /root/reference/core/estimator.py:570-613, utils/distribution_utils.py:85-98.
"""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boxsegliver_b200 import synthetic  # noqa: E402
from boxsegliver_b200.device import Context  # noqa: E402
from boxsegliver_b200.engine import EngineConfig, UNetEngine  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dist.init_process_group("gloo", rank=rank, world_size=world)
ctx = Context(local)
unet3d = sys.argv[1:] == ["unet3d"]
if unet3d:
    from boxsegliver_b200.unet3d_engine import UNet3DConfig, UNet3DEngine  # noqa: E402
    n, d, hw = 2, 8, 64
    eng = UNet3DEngine(ctx, UNet3DConfig(batch=n, depth=d, height=hw, width=hw, normalizer="batch_norm",
                                         weight_decay_rate=3e-5, world=world))
    im, lb = synthetic.make_volume_batch(n, d, hw, hw, seed=1357 + rank)

    def allreduce_grads():
        ctx.call("bsl_allreduce_sum_f32", eng.G.p, C.c_size_t(eng.n_train), eng.stream)
else:
    n, hw = 4, 128
    cfg = EngineConfig(batch=n, height=hw, width=hw, loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4),
                       weight_decay_rate=1e-5, world=world)
    eng = UNetEngine(ctx, cfg)
    im, lb = synthetic.make_batch(n, hw, hw, 3, seed=1357 + rank)
    allreduce_grads = eng._allreduce_grads
w0 = eng.init_weights(seed=0)
eng.set_inputs(im, lb)

# local gradients (no communicator attached yet: _after_grad is inert, no all-reduce is issued)
eng.forward(True)
eng.loss_backward()
ctx.check_device()
g_local = torch.from_numpy(eng.G.download(np.float32, (eng.n_train,)).astype(np.float64))
s_local = torch.from_numpy(eng.S.download(np.float32, (eng.n_stats,)).astype(np.float64))
dist.all_reduce(g_local)
dist.all_reduce(s_local)

uid = (C.c_char * 128)()
if rank == 0:
    ctx.call("bsl_comm_unique_id", uid)
box = [bytes(uid)]
dist.broadcast_object_list(box, src=0)
eng.attach_comm(rank, world, box[0])
eng.set_weights(w0)
eng.forward(True)
eng._allreduce_moving_stats()
eng.loss_backward()
allreduce_grads()
ctx.check_device()
g_dev = eng.G.download(np.float32, (eng.n_train,)).astype(np.float64)
s_dev = eng.S.download(np.float32, (eng.n_stats,)).astype(np.float64)
e_g = float(np.linalg.norm(g_dev - g_local.numpy()) / np.linalg.norm(g_local.numpy()))
e_s = float(np.linalg.norm(s_dev - s_local.numpy() / world) / np.linalg.norm(s_local.numpy() / world))
assert e_g < 1e-6, e_g
assert e_s < 1e-6, e_s

eng.set_weights(w0)
for _ in range(3):
    eng.train_step(1e-3)
ctx.check_device()
wflat = torch.from_numpy(eng.W.download(np.float32, (eng.n_train,)).view(np.int32).astype(np.int64))
lo, hi = wflat.clone(), wflat.clone()
dist.all_reduce(lo, op=dist.ReduceOp.MIN)
dist.all_reduce(hi, op=dist.ReduceOp.MAX)
assert bool((lo == hi).all()), "mirrored weights diverged across ranks"
if rank == 0:
    what = "unet3d batch_norm" if unet3d else f"unet buckets={len(eng._bucket_at)}"
    print(f"dp_check OK: world={world} {what} grad rel err {e_g:.2e} moving-stat rel err {e_s:.2e} "
          f"weights bit-identical on all ranks after 3 steps")
dist.barrier()
dist.destroy_process_group()
