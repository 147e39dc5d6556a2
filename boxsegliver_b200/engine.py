"""U-Net 2-D training / inference engine on the sm_100a kernels (host side, Python + ctypes only).

What TF's executor does for the reference's graph (/root/reference/NetworksV2/UNet.py:58-155 built by
BaseNet.__call__, differentiated and updated by Solver, /root/reference/core/solver.py:221-243) this
module does explicitly: it plans every buffer once, then a step is a fixed sequence of C-ABI enqueues
on one compute stream (plus a side stream for the gradient all-reduce), replayable as a CUDA graph.

Memory plan (all NHWC, bf16 unless noted):
  * per conv layer: `y` (pre-norm conv output, kept for backward) and `a` (post norm+ReLU); --without_norm keeps only
    `a` = relu(conv + bias), out of the conv epilogue;
  * skip-concat is zero-copy: encoder level i writes `a` into channels [0,C) of cat_i, the
    transposed conv writes into [C,2C) (UNet.py:93 order: skip first, up second);
  * parameters live in flat fp32 arenas W / G / M / V with a bf16 shadow of W for the tensor-core
    convs; region A (L2-regularised: weights, biases) precedes region B (gamma, beta);
  * two ping-pong gradient buffers + one dcat_i per level carry activation gradients.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from .device import Context, DeviceBuffer
from .engine_base import BF16, F32, EngineBase, Param, TrainConfig, _align


@dataclass
class EngineConfig(TrainConfig):
    height: int = 256
    width: int = 256
    channel: int = 3
    init_channels: int = 64
    num_down_samples: int = 4
    without_norm: bool = False         # --without_norm: slim.conv2d(normalizer_fn=None) -> weights + biases, bias + ReLU


class View:
    """A strided NHWC window into a device buffer: channels [c0, c0+c) of a tensor with stride ld."""

    def __init__(self, buf: DeviceBuffer, n, h, w, c, ld=None, c0=0, esize=BF16):
        self.buf, self.n, self.h, self.w, self.c = buf, n, h, w, c
        self.ld = ld or c
        self.c0 = c0
        self.esize = esize

    @property
    def p(self) -> C.c_void_p:
        return C.c_void_p(self.buf.ptr + self.c0 * self.esize)

    @property
    def pixels(self):
        return self.n * self.h * self.w

    def slice(self, c0, c):
        return View(self.buf, self.n, self.h, self.w, c, self.ld, self.c0 + c0, self.esize)


@dataclass
class ConvL:
    kind: str                # "stem" | "conv" | "convT" | "logits"
    scope: str
    cin: int
    cout: int
    h: int
    w: int                   # INPUT spatial size
    level: int
    role: str = ""           # enc1 | enc2 (pooled afterwards) | bridge1 | bridge2 | dec1 (reads the concat) | dec2
    center: bool = True      # normaliser has beta / gamma (GUNet's modulated blocks take them from the YAML)
    scale: bool = True
    mod_off: int = None      # GUNet: first column of this layer's slice of the context-MLP output
    sp_off: int = None       # GUNet: first column of this layer's slice of the level's 1x1 guide conv
    affine: str = None       # GUNet after_affine: scope of the ChannelWiseAffine variables of this encoder layer
    bn_decay: float = None   # batch-norm moving-average decay of this layer (None: cfg.bn_decay; GUNet encoder: 0.99)
    x: View = None
    y: View = None           # pre-norm conv output (conv/stem; None under --without_norm), or output (convT)
    a: View = None           # post-activation
    pooled: View = None
    params: dict = field(default_factory=dict)
    norm: dict = field(default_factory=dict)


class UNetEngine(EngineBase):
    def __init__(self, ctx: Context, cfg: EngineConfig):
        self.ctx, self.cfg = ctx, cfg
        self.pixels_per_sample = cfg.height * cfg.width
        if 9 * cfg.channel > 64:
            raise ValueError("im_channel must be <= 7 (the stem's im2col row holds 9 * channels <= 64 columns)")
        if cfg.init_channels % 64:
            raise ValueError("init_channels must be a multiple of 64 for the tcgen05 conv path")
        ds = 2 ** cfg.num_down_samples
        if cfg.height % ds or cfg.width % ds:
            raise ValueError(f"height/width must be multiples of {ds}")
        self._check_train_config()
        self._init_plumbing()
        self._skip_exchange = False   # bench.py's data-parallel check runs one backward without the gradient exchange
        self._plan_params()
        self._plan_activations()
        self.comm_stream = None
        self._graph = None
        self._grad_stream = self.stream
        self._overlap_wgrad = cfg.training
        self._dy_busy = [None, None]
        # logits out of the last normalised layer's apply pass (bsl_norm_apply_head) instead of a 1x1 conv over the stored
        # activation; bit-identical (tests/test_gpu_unet.py compares both ways)
        self._fuse_head = True
        # backward of the last normalised layer with the logits-layer dgrad recomputed per pixel from dlogits
        # (bsl_norm_bwd_reduce_head / _apply_head) instead of a 128-byte-per-pixel gradient tensor; bit-identical
        self._fuse_head_bwd = True
        self._head_grad = None

    # ------------------------------------------------------------------ per-kernel timing (bench roofline)
    def enable_conv_timing(self, on: bool = True):
        """Bracket every tcgen05 conv launch with CUDA events on the compute stream (bench.py roofline)."""
        self._timing = on
        self._timed = []          # (name, flops, ev0, ev1) in launch order for the current step(s)
        self._ev_pool = getattr(self, "_ev_pool", [])
        self._ev_next = 0

    def _ev(self):
        if self._ev_next == len(self._ev_pool):
            self._ev_pool.append(self.ctx.new_event())
        e = self._ev_pool[self._ev_next]
        self._ev_next += 1
        return e

    def _tc(self, name: str, flops: float, fn_name: str, *args, stream=None):
        """Enqueue a tensor-core conv call, optionally bracketed by events on the stream it is launched on."""
        if getattr(self, "_timing", False):
            e0, e1 = self._ev(), self._ev()
            st = stream if stream is not None else self.stream
            self.ctx.record(e0, st)
            self.ctx.call(fn_name, *args)
            self.ctx.record(e1, st)
            self._timed.append((name, flops, e0, e1))
        else:
            self.ctx.call(fn_name, *args)

    def conv_timing_report(self):
        """Sum of device time and algorithmic FLOPs over the bracketed conv launches since enable_conv_timing."""
        self.ctx.sync(self.stream)
        tot_ms, tot_fl, per = 0.0, 0.0, {}
        for name, fl, e0, e1 in self._timed:
            ms = self.ctx.elapsed_ms(e0, e1)
            tot_ms += ms
            tot_fl += fl
            a = per.setdefault(name, [0, 0.0, 0.0])
            a[0] += 1
            a[1] += ms
            a[2] += fl
        return {"launches": len(self._timed), "ms": tot_ms, "flops": tot_fl, "per_kind": per}

    # ------------------------------------------------------------------ data parallel
    def attach_comm(self, rank: int, world: int, unique_id: bytes):
        """Join the NCCL communicator (one process per GPU). cfg.world must equal `world`."""
        assert world == self.cfg.world, (world, self.cfg.world)
        self.ctx.attach_comm(rank, world, unique_id)
        self.rank = rank
        self._plan_buckets()

    # Gradient exchange overlapped with backward (replaces AllReduceCrossDeviceOps("nccl", num_packs=2),
    # /root/reference/utils/distribution_utils.py:91-98): the regularised region of the gradient arena is laid out in
    # forward layer order and backward fills it from the end, so a bucket is a suffix range that is complete as soon
    # as its first layer's wgrad has been enqueued. Each bucket is all-reduced on a side stream behind an event.
    BUCKET_ELEMS = 6 << 20

    def _plan_buckets(self):
        self.comm_stream = self.ctx.new_stream()
        self._ev_ready = [self.ctx.new_event() for _ in range(16)]
        self._ev_done = self.ctx.new_event()
        self._bucket_at = {}          # scope of the layer that closes a bucket -> (offset, count)
        # parameters outside the conv trunk (GUNet guide convs) sit after the last layer in region A and get their
        # gradients late in backward: they travel with the tail
        lastp = [p for p in self.params.values() if p.region == "A" and p.name.startswith(self.layers[-1].scope + "/")]
        self._trunk_end = max(p.offset + _align(max(p.size, p.alloc)) for p in lastp)
        end, acc, last = self._trunk_end, 0, None
        # the final bucket closes at the stem's filter gradient, the last kernel of backward, and overlaps nothing: a
        # boundary at the first conv of the second level keeps it down to the first level's ~40 K values
        early = next((L.scope for L in self.layers if L.kind == "conv" and L.level == 1), None)
        for L in reversed(self.layers):
            p = self.params[f"{L.scope}/weights"]
            acc = end - p.offset
            last = L
            full = acc >= self.BUCKET_ELEMS or (L.scope == early and acc > 0)
            if full and len(self._bucket_at) < len(self._ev_ready) - 1:
                self._bucket_at[L.scope] = (p.offset, acc)
                end, acc = p.offset, 0
        if end > 0:
            self._bucket_at[last.scope] = (0, end)
        self._bucket_i = 0

    def _after_grad(self, L: ConvL):
        """Called when layer L's parameter gradients have been enqueued (backward order)."""
        if self.cfg.world <= 1 or self._skip_exchange or L.scope not in getattr(self, "_bucket_at", {}):
            return
        off, cnt = self._bucket_at[L.scope]
        ev = self._ev_ready[self._bucket_i]
        self._bucket_i += 1
        self.ctx.record(ev, self._grad_stream)
        self.ctx.call("bsl_stream_wait_event", self.comm_stream, ev)
        self.ctx.call("bsl_allreduce_sum_f32", C.c_void_p(self.G.ptr + off * F32), C.c_size_t(cnt), self.comm_stream)

    def _allreduce_grads(self):
        """Tail of the exchange: the un-regularised region (gamma / beta / FC, tiny) follows the buckets on the side
        stream -- every gradient has been enqueued once loss_backward returns -- then the compute stream joins it, so
        the only collective work the optimizer waits for is the last bucket and this tail."""
        if self.cfg.world <= 1 or self._skip_exchange:
            return
        if self.comm_stream is None:       # attach_comm not called: single all-reduce on the compute stream
            self.ctx.call("bsl_allreduce_sum_f32", self.G.p, C.c_size_t(self.n_train), self.stream)
            return
        nb = self.n_train - self._trunk_end
        if nb > 0:
            ev = self._ev_ready[-1]
            self.ctx.record(ev, self.stream)
            self.ctx.call("bsl_stream_wait_event", self.comm_stream, ev)
            self.ctx.call("bsl_allreduce_sum_f32", C.c_void_p(self.G.ptr + self._trunk_end * F32), C.c_size_t(nb),
                          self.comm_stream)
        self.ctx.record(self._ev_done, self.comm_stream)
        self.ctx.call("bsl_stream_wait_event", self.stream, self._ev_done)
        self._bucket_i = 0

    def _allreduce_moving_stats(self):
        # Nothing reads the moving statistics before the next step's forward, so the exchange rides the side stream
        # (ahead of the gradient buckets) and is ordered before the optimizer by the same join as the gradients.
        if not self._skip_exchange:
            super()._allreduce_moving_stats(self.comm_stream)

    # ------------------------------------------------------------------ planning
    def _layer_specs(self):
        cfg = self.cfg
        specs = []
        c, cin = cfg.init_channels, cfg.channel
        h, w = cfg.height, cfg.width
        for i in range(cfg.num_down_samples):
            for j in (1, 2):
                kind = "stem" if (i == 0 and j == 1) else "conv"
                specs.append(ConvL(kind, f"UNet/Encode{i + 1}/Repeat/convolution2d_{j}", cin, c, h, w, i, role=f"enc{j}"))
                cin = c
            c *= 2
            h //= 2
            w //= 2
        for j in (1, 2):
            specs.append(ConvL("conv", f"UNet/ED-Bridge/ED-Bridge_{j}", cin, c, h, w, cfg.num_down_samples,
                               role=f"bridge{j}"))
            cin = c
        for i in reversed(range(cfg.num_down_samples)):
            c //= 2
            specs.append(ConvL("convT", f"UNet/Decode{i + 1}/Conv2d_transpose", cin, cin // 2, h, w, i))
            h *= 2
            w *= 2
            for j in (1, 2):
                specs.append(ConvL("conv", f"UNet/Decode{i + 1}/Repeat/convolution2d_{j}",
                                   c + cin // 2 if j == 1 else c, c, h, w, i, role=f"dec{j}"))
            cin = c
        specs.append(ConvL("logits", "UNet/AdjustChannels", cin, cfg.num_classes, h, w, 0))
        return specs

    def _plan_params(self):
        cfg = self.cfg
        self.layers = self._layer_specs()
        ns = "BatchNorm" if cfg.normalizer == "batch_norm" else "InstanceNorm"
        self.norm_scope = ns
        plist = []
        for L in self.layers:
            if L.kind in ("stem", "conv"):
                # the convs reduce over whole 64-channel blocks: a conv's input channels beyond cin (UNetInter --mid_cat
                # 66 -> 128, GUNet --img_grad 9 -> 64) are stored as zero rows; the im2col stem reserves 64 rows instead
                cin = L.cin if L.kind == "stem" else _align(L.cin, 64)
                plist.append(Param(f"{L.scope}/weights", (3, 3, L.cin, L.cout), (3, 3, cin, L.cout),
                                   (slice(None), slice(None), slice(L.cin)), alloc=64 * L.cout if L.kind == "stem" else 0))
                if cfg.without_norm:     # no normalizer_fn: slim keeps the conv's biases
                    plist.append(Param(f"{L.scope}/biases", (L.cout,), region="B" if cfg.bias_decay else "A"))
                    continue
                if L.scale:
                    plist.append(Param(f"{L.scope}/{ns}/gamma", (L.cout,), region="B"))
                if L.center:
                    plist.append(Param(f"{L.scope}/{ns}/beta", (L.cout,), region="B"))
                if cfg.normalizer == "batch_norm":
                    plist.append(Param(f"{L.scope}/{ns}/moving_mean", (L.cout,), region="S"))
                    plist.append(Param(f"{L.scope}/{ns}/moving_variance", (L.cout,), region="S"))
            elif L.kind == "convT":
                plist.append(Param(f"{L.scope}/weights", (2, 2, L.cout, L.cin)))
                plist.append(Param(f"{L.scope}/biases", (L.cout,), region="B" if cfg.bias_decay else "A"))
            else:
                plist.append(Param(f"{L.scope}/weights", (1, 1, L.cin, L.cout)))
                plist.append(Param(f"{L.scope}/biases", (L.cout,), region="B" if cfg.bias_decay else "A"))
        self._layout(plist + self._extra_params())

    def _extra_params(self):
        """Parameters outside the conv trunk (GUNet: context MLP, guide convs)."""
        return []

    def _pp(self, arena: DeviceBuffer, name: str, esize=F32, off: int = 0) -> C.c_void_p:
        if name not in self.params:
            return None
        return C.c_void_p(arena.ptr + (self.params[name].offset + off) * esize)

    def _guide_channels(self, L: ConvL) -> int:
        return 0

    def _first_input(self, L: ConvL) -> View:
        raise NotImplementedError("the first layer of this engine is the im2col stem")

    def _pooled_lanes(self, L: ConvL) -> int:
        """Channel stride of the pooled tensor behind an encoder block."""
        return L.cout

    def _after_pool(self, L: ConvL, stream):
        """Hook behind the fused norm + ReLU + pool pass of an encoder block (UNetInter --mid_cat adds the guide lanes)."""

    def _norm_groups(self, L: ConvL, default: int) -> int:
        """Entries per channel of the layer's normalisation scalars (1 batch norm, n instance norm / modulated)."""
        return default

    def _apply_desc(self, L: ConvL, nd):
        """Descriptor of the apply / backward passes (GUNet: the per-sample view of a modulated batch-norm layer)."""
        return nd

    def _plan_activations(self):
        cfg = self.cfg
        n = cfg.batch
        cat = {}
        max_act = 0
        prev_a = None
        groups_max = n if cfg.normalizer == "instance_norm" else 1
        small = 0  # floats for per-layer normalisation scalars
        for L in self.layers:
            if L.kind in ("stem", "conv"):
                if not cfg.without_norm:
                    L.y = View(self._alloc(n * L.h * L.w * L.cout * BF16), n, L.h, L.w, L.cout)
                is_enc2 = L.role == "enc2"
                if is_enc2:
                    cbuf = View(self._alloc(n * L.h * L.w * 2 * L.cout * BF16), n, L.h, L.w, 2 * L.cout)
                    cat[L.level] = cbuf
                    L.a = cbuf.slice(0, L.cout)
                    pl = self._pooled_lanes(L)      # > cout: extra lanes behind the activation's (UNetInter --mid_cat)
                    pbuf = self._alloc(n * (L.h // 2) * (L.w // 2) * pl * BF16)
                    if pl != L.cout:
                        pbuf.zero()
                    L.pooled = View(pbuf, n, L.h // 2, L.w // 2, L.cout, pl)
                else:
                    L.a = View(self._alloc(n * L.h * L.w * L.cout * BF16), n, L.h, L.w, L.cout)
                if L.kind == "conv":
                    L.x = cat[L.level] if L.role == "dec1" else prev_a
                    if L.x is None:      # a first layer that is not the im2col stem (GUNet --img_grad: 9 input channels)
                        L.x = self._first_input(L)
                prev_a = L.pooled if is_enc2 else L.a
                if is_enc2 and L.pooled.ld != L.cout:
                    prev_a = View(L.pooled.buf, n, L.h // 2, L.w // 2, L.pooled.ld)
                max_act = max(max_act, L.h * L.w * L.cout)
                if cfg.without_norm:
                    continue
                g = self._norm_groups(L, groups_max)
                k = 2 + self._guide_channels(L)
                L.norm = dict(groups=g, off=small, k=k)
                small += self._norm_scalar_floats(g * L.cout, k)
            elif L.kind == "convT":
                L.x = prev_a
                L.a = cat[L.level].slice(L.cout, L.cout)   # upper channel half of the concat buffer
                L.y = L.a
                prev_a = cat[L.level]
            else:
                L.x = prev_a
        self.cat = cat
        self.images = self._alloc(n * cfg.height * cfg.width * cfg.channel * F32)
        # im2col rows of the stem: 9 * channels live columns in a pitch of 32 (3 input channels) or 64 columns; the conv
        # kernels read a 32-column matrix as cin = 64 with the upper half zero-filled by TMA (bsl_stem_im2col_ld)
        sc = 32 if 9 * cfg.channel <= 32 else 64
        self.stem_cols = sc
        self.stem_col = View(self._alloc(n * cfg.height * cfg.width * sc * BF16), n, cfg.height, cfg.width, sc)
        self.labels = self._alloc(n * cfg.height * cfg.width * 4)
        npx = n * cfg.height * cfg.width
        self.logits = self._alloc(npx * cfg.num_classes * F32)
        self.prob = self._alloc(npx * cfg.num_classes * F32)
        self.masks = self._alloc(npx * (cfg.num_classes - 1))
        self.argmax = self._alloc(npx)
        self.ilr = self._alloc(n * (cfg.num_classes - 1) * 3 * 4)
        self.counts = self._alloc(n * cfg.num_classes * 4)
        self.loss_dev = self._alloc(16)
        self.small = self._alloc(max(small, 16) * F32)
        ld = self._loss_desc()
        self.loss_ws_bytes = self.ctx.lib.bsl_loss_workspace(self.ctx.h, C.byref(ld))
        self.loss_ws = self._alloc(self.loss_ws_bytes)
        if cfg.training:
            self.dlogits = self._alloc(npx * cfg.num_classes * F32)
            self.g1 = self._alloc(n * max_act * BF16)
            self.g2 = self._alloc(n * max_act * BF16)
            self.dyb = [self._alloc(n * max_act * BF16), self._alloc(n * max_act * BF16)]
            self.dcat = {i: View(self._alloc(v.pixels * v.c * BF16), n, v.h, v.w, v.c) for i, v in cat.items()}
            ws = 0
            for L in self.layers:
                if L.kind == "stem":
                    d = _lib.Conv2dDesc(n, L.h, L.w, 64, L.cout, 1, 1, self.stem_cols, L.cout)
                    ws = max(ws, self.ctx.lib.bsl_conv2d_wgrad_workspace(self.ctx.h, C.byref(d)))
                elif L.kind == "conv":
                    d = self._conv_desc(L)
                    ws = max(ws, self.ctx.lib.bsl_conv2d_wgrad_workspace(self.ctx.h, C.byref(d)))
                elif L.kind == "convT":
                    d = self._convT_desc(L)
                    ws = max(ws, self.ctx.lib.bsl_convT2d_bwd_filter_workspace(self.ctx.h, C.byref(d)))
            self.wgrad_ws_bytes = int(ws)
            self.wgrad_ws = self._alloc(max(ws, 16))

    def _flops(self, L: ConvL) -> float:
        """Algorithmic FLOPs of ONE pass (fprop, dgrad or wgrad) of layer L: 2 * MACs, un-padded (BASELINE.md section 3)."""
        n = self.cfg.batch
        if L.kind == "convT":
            return 2.0 * n * (2 * L.h) * (2 * L.w) * L.cin * L.cout   # one tap per output pixel
        k = 1 if L.kind == "logits" else 9
        return 2.0 * n * L.h * L.w * k * L.cin * L.cout

    def _loss_terms(self):
        """UNet accepts exactly "xentropy" or "dice" (UNet.py:123-132); GUNet overrides with substring matching."""
        return [self.cfg.loss_type] if self.cfg.loss_type in ("xentropy", "dice") else []

    def step_flops(self) -> dict:
        """Algorithmic fwd / bwd FLOPs of one training step (bwd = dgrad + wgrad, no dgrad for the stem)."""
        fwd = sum(self._flops(L) for L in self.layers)
        bwd = sum(self._flops(L) * (1 if L.kind == "stem" else 2) for L in self.layers)
        tc = sum(self._flops(L) * (2 if L.kind == "stem" else 3) for L in self.layers if L.kind != "logits")
        return {"fwd": fwd, "bwd": bwd, "total": fwd + bwd, "tensor_core": tc}

    # ------------------------------------------------------------------ descriptors
    def _conv_desc(self, L: ConvL):
        k = 1 if L.kind == "logits" else 3
        x_ld = L.x.ld if L.x is not None else L.cin
        y_ld = L.y.ld if L.y is not None else (L.a.ld if L.a is not None else L.cout)   # --without_norm: y is a
        cin = self.params[f"{L.scope}/weights"].stored[2]       # zero-padded input channels
        return _lib.Conv2dDesc(self.cfg.batch, L.h, L.w, cin, L.cout, k, k, x_ld, y_ld)

    def _convT_desc(self, L: ConvL):
        return _lib.ConvT2dDesc(self.cfg.batch, L.h, L.w, L.cin, L.cout, L.x.ld, L.a.ld, 1)

    def _norm_desc(self, L: ConvL):
        cfg = self.cfg
        bn = cfg.normalizer == "batch_norm"
        return _lib.NormDesc(0 if bn else 1, cfg.batch, L.h * L.w, L.cout, L.y.ld, L.a.ld,
                             cfg.bn_eps if bn else cfg.in_eps, L.bn_decay if L.bn_decay is not None else cfg.bn_decay, 1,
                             int(L.center), int(L.scale))

    def _norm_ptrs(self, L: ConvL):
        return self._norm_scalars(self.small.ptr + L.norm["off"] * F32, L.norm["groups"] * L.cout, L.norm["k"])

    # ------------------------------------------------------------------ stored activations
    def get_stored_forward(self) -> dict:
        """{scope: {"y": pre-norm conv output, "a": activation}} as fp32 numpy (what backward will read)."""
        out = {}
        for L in self.layers:
            if L.kind == "logits":
                continue
            d = {}
            for key, v in (("y", L.y), ("a", L.a)):
                if v is None:
                    continue
                full = self.ctx.bf16_to_f32(v.buf, (v.n, v.h, v.w, v.ld))
                d[key] = full[..., v.c0:v.c0 + v.c].copy()
            out[L.scope] = d
        return out

    # ------------------------------------------------------------------ inputs
    def set_inputs(self, images: np.ndarray, labels: np.ndarray | None = None, stream=None):
        cfg = self.cfg
        assert images.shape == (cfg.batch, cfg.height, cfg.width, cfg.channel), images.shape
        self.images.upload(np.ascontiguousarray(images, np.float32), stream)
        if labels is not None:
            assert labels.shape == (cfg.batch, cfg.height, cfg.width), labels.shape
            self.labels.upload(np.ascontiguousarray(labels, np.int32), stream)

    # ------------------------------------------------------------------ forward
    def forward(self, is_training: bool):
        ctx, s = self.ctx, self.stream
        call = ctx.call
        self._head_done = False
        for idx, L in enumerate(self.layers):
            ctx.tag = L.scope
            if L.kind in ("stem", "conv") and self.cfg.without_norm:
                self._forward_bias_relu(L)
            elif L.kind in ("stem", "conv"):
                d = self._conv_desc(L)
                nd = self._norm_desc(L)
                q = self._norm_ptrs(L)
                ns = self.norm_scope
                bn = self.cfg.normalizer == "batch_norm"
                # batch-norm training: the per-channel sums come out of the conv epilogue (no pass over y); instance norm
                # (training and inference): per-(sample, channel) sums from the same epilogue (bsl_conv2d_fprop_group_stats);
                # batch-norm inference normalises with the moving statistics and needs no sums
                fn, extra = "bsl_conv2d_fprop", ()
                if bn and is_training:
                    fn, extra = "bsl_conv2d_fprop_stats", (q["sums"],)
                elif not bn:
                    fn, extra = "bsl_conv2d_fprop_group_stats", (C.c_int(1), q["sums"])
                wbf = self._pp(self.Wbf, f"{L.scope}/weights", BF16)
                if L.kind == "stem":
                    # im2col (27 -> 64 columns, bf16) + 1x1 conv on the tensor cores
                    call("bsl_stem_im2col_ld", C.byref(d), self.images.p, self.stem_col.p, C.c_int(self.stem_cols), s)
                    d1 = _lib.Conv2dDesc(self.cfg.batch, L.h, L.w, 64, L.cout, 1, 1, self.stem_cols, L.y.ld)
                    self._tc("fprop", self._flops(L), fn, C.byref(d1), self.stem_col.p, wbf, L.y.p, *extra, s)
                else:
                    self._tc("fprop", self._flops(L), fn, C.byref(d), L.x.p, wbf, L.y.p, *extra, s)
                mm = C.c_void_p(self.S.ptr + self.params[f"{L.scope}/{ns}/moving_mean"].offset * F32) if bn else None
                mv = C.c_void_p(self.S.ptr + self.params[f"{L.scope}/{ns}/moving_variance"].offset * F32) if bn else None
                call("bsl_norm_finalize", C.byref(nd), C.c_int(1 if is_training else 0), q["sums"],
                     self._pp(self.W, f"{L.scope}/{ns}/gamma"), self._pp(self.W, f"{L.scope}/{ns}/beta"), mm, mv,
                     q["mean"], q["rstd"], q["scale"], q["shift"], s)
                src = self._dropout_stage(L, nd, q, is_training)   # GUNet --dropout: a dropped copy of the normalised tensor
                guide = self._modulate(L, nd, q)   # GUNet: folds gamma_mod / guide bias into scale, shift
                nd = self._apply_desc(L, nd)
                gp = C.byref(guide) if guide is not None else None
                nxt = self.layers[idx + 1] if idx + 1 < len(self.layers) else None
                cg = L.cout // 8
                if (self._fuse_head and nxt is not None and nxt.kind == "logits" and gp is None and L.pooled is None
                        and cg <= 32 and cg & (cg - 1) == 0 and 2 <= self.cfg.num_classes <= 4):
                    # last normalised layer: the logits come out of the same pass (no second read of the activation)
                    call("bsl_norm_apply_head", C.byref(nd), src, q["scale"], q["shift"], L.a.p,
                         self._pp(self.W, f"{nxt.scope}/weights"), self._pp(self.W, f"{nxt.scope}/biases"),
                         C.c_int(self.cfg.num_classes), self.logits.p, s)
                    self._head_done = True
                elif L.pooled is not None:
                    call("bsl_norm_apply_pool_mod", C.byref(nd), C.c_int(L.h), C.c_int(L.w), src, q["scale"],
                         q["shift"], gp, L.a.p, L.pooled.p, C.c_int(L.pooled.ld), s)
                    self._after_pool(L, s)
                else:
                    call("bsl_norm_apply_mod", C.byref(nd), src, q["scale"], q["shift"], gp, L.a.p, s)
            elif L.kind == "convT":
                d = self._convT_desc(L)
                self._tc("convT_fwd", self._flops(L), "bsl_convT2d_fwd", C.byref(d), L.x.p,
                         self._pp(self.Wbf, f"{L.scope}/weights", BF16), self._pp(self.W, f"{L.scope}/biases"), L.a.p, s)
            elif not self._head_done:
                d = self._conv_desc(L)
                call("bsl_conv2d_head_fprop", C.byref(d), L.x.p, self._pp(self.W, f"{L.scope}/weights"),
                     self._pp(self.W, f"{L.scope}/biases"), self.logits.p, s)

    def _forward_bias_relu(self, L: ConvL):
        """--without_norm: a = relu(conv + bias) out of the conv epilogue, then the 2x2 max-pool of an encoder block."""
        ctx, s = self.ctx, self.stream
        wbf = self._pp(self.Wbf, f"{L.scope}/weights", BF16)
        b = self._pp(self.W, f"{L.scope}/biases")
        if L.kind == "stem":
            ctx.call("bsl_stem_im2col_ld", C.byref(self._conv_desc(L)), self.images.p, self.stem_col.p,
                     C.c_int(self.stem_cols), s)
            d1 = _lib.Conv2dDesc(self.cfg.batch, L.h, L.w, 64, L.cout, 1, 1, self.stem_cols, L.a.ld)
            self._tc("fprop", self._flops(L), "bsl_conv2d_fprop_bias_relu", C.byref(d1), self.stem_col.p, wbf, b, L.a.p, s)
        else:
            self._tc("fprop", self._flops(L), "bsl_conv2d_fprop_bias_relu", C.byref(self._conv_desc(L)), L.x.p, wbf, b,
                     L.a.p, s)
        if L.pooled is not None:
            ctx.call("bsl_maxpool2x2_bf16", C.c_int(self.cfg.batch), C.c_int(L.h), C.c_int(L.w), C.c_int(L.cout), L.a.p,
                     C.c_int(L.a.ld), L.pooled.p, C.c_int(L.pooled.ld), s)
            self._after_pool(L, s)

    def _modulate(self, L: ConvL, nd, q):
        """Hook between norm_finalize and norm_apply; returns the bsl_guide of the layer (or None)."""
        return None

    def _dropout_stage(self, L: ConvL, nd, q, is_training: bool):
        """Hook behind norm_finalize: the tensor the apply pass reads (GUNet's backbone --dropout substitutes a dropped
        copy of the normalised conv output and turns (scale, shift) into the identity)."""
        return L.y.p

    def _is_modulated(self, L: ConvL) -> bool:
        return False

    def _norm_backward_reduce(self, L: ConvL, nd, q, cur):
        """First half of the gradient through ReLU + normalisation of layer L: the per-channel sums over `cur` (the
        gradient w.r.t. the activation) and the gradients of the normaliser's own parameters (into G)."""
        call, s, ns = self.ctx.call, self.stream, self.norm_scope
        if self._head_grad is not None:
            dl, wh, classes = self._head_grad
            call("bsl_norm_bwd_reduce_head", C.byref(nd), L.y.p, dl, wh, C.c_int(classes), q["mean"], q["rstd"],
                 q["scale"], q["shift"], q["sums"], s)
        else:
            call("bsl_norm_bwd_reduce", C.byref(nd), L.y.p, cur.p, C.c_int(L.cout), q["mean"], q["rstd"],
                 q["scale"], q["shift"], q["sums"], s)
        call("bsl_norm_bwd_finalize", C.byref(nd), q["sums"], q["c1"], q["c2"],
             self._pp(self.G, f"{L.scope}/{ns}/gamma"), self._pp(self.G, f"{L.scope}/{ns}/beta"), s)

    def _norm_backward_apply(self, L: ConvL, nd, q, cur, oth, stream):
        """Second half: `cur` -> `oth` (gradient w.r.t. the conv output)."""
        if self._head_grad is not None:
            dl, wh, classes = self._head_grad
            self._head_grad = None
            self.ctx.call("bsl_norm_bwd_apply_head", C.byref(nd), L.y.p, dl, wh, C.c_int(classes), q["mean"], q["rstd"],
                          q["scale"], q["shift"], q["c1"], q["c2"], oth.p, C.c_int(L.cout), stream)
            return
        self.ctx.call("bsl_norm_bwd_apply_mod", C.byref(nd), L.y.p, cur.p, C.c_int(L.cout), q["mean"], q["rstd"],
                      q["scale"], q["shift"], q["c1"], q["c2"], None, oth.p, C.c_int(L.cout), stream)

    def _norm_backward(self, L: ConvL, nd, q, cur, oth):
        self._norm_backward_reduce(L, nd, q, cur)
        self._norm_backward_apply(L, nd, q, cur, oth, self.stream)

    # ------------------------------------------------------------------ loss + backward
    def loss_backward(self):
        ctx, s, cfg = self.ctx, self.stream, self.cfg
        call = ctx.call
        ld = self._loss_desc()
        terms = self._loss_terms()
        if "xentropy" in terms:
            call("bsl_label_counts", C.byref(ld), self.labels.p, self.counts.p, s)
            call("bsl_wxent_fwd_bwd", C.byref(ld), self.logits.p, self.labels.p, self.counts.p, self.loss_dev.p,
                 self.dlogits.p, self.loss_ws.p, C.c_size_t(self.loss_ws_bytes), s)
        if "dice" in terms:   # second scalar slot; dlogits accumulate when both terms are present (GUNet.py:399-408)
            call("bsl_dice_fwd_bwd", C.byref(ld), self.logits.p, self.labels.p,
                 self.loss_dev.at(4 * terms.index("dice")), self.dlogits.p, C.c_int(1 if len(terms) > 1 else 0),
                 self.loss_ws.p, C.c_size_t(self.loss_ws_bytes), s)
        n = cfg.batch
        # `cur` holds the gradient w.r.t. the current activation; dY (w.r.t. the conv output) alternates between two
        # buffers so that the filter gradient of layer L can run on the side stream while the main stream goes on
        # with dgrad(L) and the HBM-bound normalisation backward of layer L-1 (tensor-bound and memory-bound work
        # overlap); a dY buffer is reused two conv layers later, behind an event.
        cur, alt = self.g1, self.g2
        overlap = self._overlap_wgrad and ctx._prof is None
        ws = self.wg_stream if overlap else s
        self._grad_stream = ws
        k = 0
        wsb = C.c_size_t(self.wgrad_ws_bytes)

        def fork():
            """side stream waits for everything enqueued on the main stream so far"""
            if overlap:
                self._stream_wait(ws, s)

        for idx in range(len(self.layers) - 1, -1, -1):
            L = self.layers[idx]
            ctx.tag = L.scope
            if L.kind == "logits":
                d = self._conv_desc(L)
                fork()
                call("bsl_conv2d_head_wgrad", C.byref(d), L.x.p, self.dlogits.p, self._pp(self.G, f"{L.scope}/weights"),
                     self._pp(self.G, f"{L.scope}/biases"), ws)
                prev = self.layers[idx - 1]
                if (self._fuse_head_bwd and not cfg.without_norm and prev.kind == "conv" and prev.pooled is None
                        and not self._is_modulated(prev) and prev.a is L.x
                        and ctx.lib.bsl_norm_bwd_head_ok(ctx.h, C.byref(self._norm_desc(prev)), C.c_int(L.cout))):
                    # no Conv2DBackpropInput launch: the two normalisation-backward passes of `prev` recompute it
                    self._head_grad = (self.dlogits.p, self._pp(self.W, f"{L.scope}/weights"), L.cout)
                else:
                    call("bsl_conv2d_head_dgrad", C.byref(d), self.dlogits.p, self._pp(self.W, f"{L.scope}/weights"),
                         cur.p, s)
                self._after_grad(L)
                continue
            if L.kind in ("stem", "conv"):
                if L.pooled is not None:
                    # `cur` is the gradient w.r.t. the POOLED tensor; merge MaxPoolGrad with the skip gradient
                    dc = self.dcat[L.level]
                    call("bsl_maxpool2x2_bwd_add", C.c_int(n), C.c_int(L.h), C.c_int(L.w), C.c_int(L.cout), L.a.p,
                         C.c_int(L.a.ld), cur.p, C.c_int(L.pooled.ld), dc.p, C.c_int(dc.ld), alt.p, C.c_int(L.cout), s)
                    cur, alt = alt, cur
                dyb = self.dyb[k]
                if cfg.without_norm:
                    if overlap and self._dy_busy[k] is not None:
                        call("bsl_stream_wait_event", s, self._dy_busy[k])
                    # ReluGrad into dY and BiasAddGrad from the same pass
                    call("bsl_relu_bwd_bias", C.c_longlong(L.a.pixels), C.c_int(L.cout), L.a.p, C.c_int(L.a.ld), cur.p,
                         C.c_int(L.cout), dyb.p, C.c_int(L.cout), self._pp(self.G, f"{L.scope}/biases"), s)
                else:
                    nd = self._norm_desc(L)
                    q = self._norm_ptrs(L)
                    self._norm_backward_reduce(L, nd, q, cur)
                    if overlap and self._dy_busy[k] is not None:   # the wgrad that read this buffer two layers ago
                        call("bsl_stream_wait_event", s, self._dy_busy[k])
                    self._norm_backward_apply(L, nd, q, cur, dyb, s)
                # dyb = dY (gradient w.r.t. the conv output), dense with ld = cout
                d = self._conv_desc(L)
                d.y_ld = L.cout
                gw = self._pp(self.G, f"{L.scope}/weights")
                # the side stream forks before dgrad, so that the filter gradient of this layer runs beside dgrad and the
                # HBM-bound normalisation backward of the next one
                fork()
                if L.kind != "stem" and idx > 0:     # no gradient w.r.t. the network input
                    wbf = self._pp(self.Wbf, f"{L.scope}/weights", BF16)
                    dd = self._conv_desc(L)
                    dd.y_ld = L.cout
                    if L.role == "dec1":
                        dc = self.dcat[L.level]
                        dd.x_ld = dc.ld
                        self._tc("dgrad", self._flops(L), "bsl_conv2d_dgrad", C.byref(dd), dyb.p, wbf, dc.p, s)
                    else:
                        dd.x_ld = dd.cin
                        self._tc("dgrad", self._flops(L), "bsl_conv2d_dgrad", C.byref(dd), dyb.p, wbf, cur.p, s)
                if L.kind == "stem":
                    d1 = _lib.Conv2dDesc(n, L.h, L.w, 64, L.cout, 1, 1, self.stem_cols, L.cout)
                    self._tc("wgrad", self._flops(L), "bsl_conv2d_wgrad", C.byref(d1), self.stem_col.p, dyb.p, gw,
                             self.wgrad_ws.p, wsb, ws, stream=ws)
                else:
                    self._tc("wgrad", self._flops(L), "bsl_conv2d_wgrad", C.byref(d), L.x.p, dyb.p, gw,
                             self.wgrad_ws.p, wsb, ws, stream=ws)
                if overlap:
                    self._dy_busy[k] = self._dy_events[k]
                    ctx.record(self._dy_busy[k], ws)
                k ^= 1
                self._after_grad(L)
            elif L.kind == "convT":
                dc = self.dcat[L.level]
                dup = dc.slice(L.cout, L.cout)
                # ReluGrad in place on the upper half of dcat, and the bias gradient (sum over pixels of the masked
                # gradient) from the same pass
                call("bsl_relu_bwd_bias", C.c_longlong(L.a.pixels), C.c_int(L.cout), L.a.p, C.c_int(L.a.ld), dup.p,
                     C.c_int(dup.ld), dup.p, C.c_int(dup.ld), self._pp(self.G, f"{L.scope}/biases"), s)
                d = self._convT_desc(L)
                d.y_ld = dup.ld
                d.x_ld = L.cin
                self._tc("convT_dgrad", self._flops(L), "bsl_convT2d_bwd_data", C.byref(d), dup.p,
                         self._pp(self.Wbf, f"{L.scope}/weights", BF16), cur.p, s)
                fork()
                d.x_ld = L.x.ld
                self._tc("convT_wgrad", self._flops(L), "bsl_convT2d_bwd_filter", C.byref(d), L.x.p, dup.p,
                         self._pp(self.G, f"{L.scope}/weights"), None,
                         self.wgrad_ws.p, wsb, ws, stream=ws)
                self._after_grad(L)
        if overlap:     # join: everything downstream (optimizer, host reads of G) is ordered after the filter gradients
            self._stream_wait(s, ws)
            self._dy_busy = [None, None]

    def train_step(self, lr: float, with_metrics: bool = False):
        """One `sess.run(train_op)` on device-resident inputs (/root/reference/core/estimator.py:756-757)."""
        self.forward(True)
        if self.cfg.normalizer == "batch_norm" and not self.cfg.without_norm:
            self._allreduce_moving_stats()
        if with_metrics:
            self.predict_outputs(True)
        self.loss_backward()
        self._allreduce_grads()
        self.optimizer_step(lr)

    # ------------------------------------------------------------------ host-fed step (end-to-end path)
    def pinned_inputs(self):
        """numpy views of page-locked staging buffers (images fp32 [N,H,W,C], labels int32 [N,H,W])."""
        if not hasattr(self, "_pin"):
            cfg = self.cfg
            shp_i = (cfg.batch, cfg.height, cfg.width, cfg.channel)
            shp_l = (cfg.batch, cfg.height, cfg.width)
            pi, pl, po = C.c_void_p(), C.c_void_p(), C.c_void_p()
            self.ctx.call("bsl_host_alloc", C.c_size_t(int(np.prod(shp_i)) * 4), C.byref(pi))
            self.ctx.call("bsl_host_alloc", C.c_size_t(int(np.prod(shp_l)) * 4), C.byref(pl))
            self.ctx.call("bsl_host_alloc", C.c_size_t(64), C.byref(po))
            img = np.ctypeslib.as_array(C.cast(pi, C.POINTER(C.c_float)), shape=shp_i)
            lab = np.ctypeslib.as_array(C.cast(pl, C.POINTER(C.c_int32)), shape=shp_l)
            out = np.ctypeslib.as_array(C.cast(po, C.POINTER(C.c_double)), shape=(8,))
            self._pin = (img, lab, out, pi, pl, po)
        return self._pin[0], self._pin[1]

    def train_step_host(self, lr: float, with_metrics: bool = False):
        """H2D copy of the staged batch, one training step, D2H read of (loss, sum w^2). Returns total loss.

        This is the call a user of the reference makes per step (feed a batch, fetch the loss)."""
        img, lab, out, pi, pl, po = self._pin
        s = self.stream
        self.ctx.call("bsl_memcpy_h2d", self.images.p, pi, C.c_size_t(img.nbytes), s)
        self.ctx.call("bsl_memcpy_h2d", self.labels.p, pl, C.c_size_t(lab.nbytes), s)
        self.train_step(lr, with_metrics)
        nt = len(self._loss_terms())
        self.ctx.call("bsl_memcpy_d2h", po, self.loss_dev.p, C.c_size_t(4 * nt), s)
        self.ctx.call("bsl_memcpy_d2h", C.c_void_p(po.value + 8), self.sumsq.p, C.c_size_t(8), s)
        self.ctx.sync(s)
        data = float(np.frombuffer(out[:1].tobytes(), np.float32)[:nt].sum())
        reg = float(self.cfg.weight_decay_rate * 0.5 * out[1]) if self.cfg.weight_decay_rate > 0 else 0.0
        return data + reg

    # ---- prefetching variant: a 2-deep ring of pinned staging slots + device input buffers. The H2D copy of batch
    # i + 1 runs on a copy stream while step i computes (what tf.data prefetch / StagingArea does for the reference's
    # feed path); every step still pays one H2D of its own inputs and one D2H of its loss.
    def staging_slot(self, j: int):
        """numpy views (images, labels) of pinned slot j in {0, 1}. Do not refill a slot between submit_staged(j) and
        the train_step_prefetched() that consumes it."""
        if not hasattr(self, "_ring"):
            cfg = self.cfg
            shp_i = (cfg.batch, cfg.height, cfg.width, cfg.channel)
            shp_l = (cfg.batch, cfg.height, cfg.width)
            self._ring = []
            for k in range(2):
                pi, pl = C.c_void_p(), C.c_void_p()
                self.ctx.call("bsl_host_alloc", C.c_size_t(int(np.prod(shp_i)) * 4), C.byref(pi))
                self.ctx.call("bsl_host_alloc", C.c_size_t(int(np.prod(shp_l)) * 4), C.byref(pl))
                img = np.ctypeslib.as_array(C.cast(pi, C.POINTER(C.c_float)), shape=shp_i)
                lab = np.ctypeslib.as_array(C.cast(pl, C.POINTER(C.c_int32)), shape=shp_l)
                dimg = self.images if k == 0 else self._alloc(img.nbytes)
                dlab = self.labels if k == 0 else self._alloc(lab.nbytes)
                self._ring.append(dict(img=img, lab=lab, pi=pi, pl=pl, dimg=dimg, dlab=dlab, ev=self.ctx.new_event()))
            self.copy_stream = self.ctx.new_stream()
            self._submitted = []
            self.pinned_inputs()   # the D2H slot for the loss
        return self._ring[j]["img"], self._ring[j]["lab"]

    def submit_staged(self, j: int):
        """Enqueue the H2D copy of pinned slot j into device input buffer j on the copy stream."""
        r = self._ring[j]
        cs = self.copy_stream
        self.ctx.call("bsl_memcpy_h2d", r["dimg"].p, r["pi"], C.c_size_t(r["img"].nbytes), cs)
        self.ctx.call("bsl_memcpy_h2d", r["dlab"].p, r["pl"], C.c_size_t(r["lab"].nbytes), cs)
        self.ctx.record(r["ev"], cs)
        self._submitted.append(j)

    def train_step_prefetched(self, lr: float, with_metrics: bool = False):
        """One training step on the oldest submitted slot; returns the total loss (D2H read, host sync)."""
        j = self._submitted.pop(0)
        r = self._ring[j]
        s = self.stream
        self.ctx.call("bsl_stream_wait_event", s, r["ev"])
        self.images, self.labels = r["dimg"], r["dlab"]
        self.train_step(lr, with_metrics)
        out, po = self._pin[2], self._pin[5]
        nt = len(self._loss_terms())
        self.ctx.call("bsl_memcpy_d2h", po, self.loss_dev.p, C.c_size_t(4 * nt), s)
        self.ctx.call("bsl_memcpy_d2h", C.c_void_p(po.value + 8), self.sumsq.p, C.c_size_t(8), s)
        self.ctx.sync(s)
        data = float(np.frombuffer(out[:1].tobytes(), np.float32)[:nt].sum())
        reg = float(self.cfg.weight_decay_rate * 0.5 * out[1]) if self.cfg.weight_decay_rate > 0 else 0.0
        return data + reg

    def h2d_bytes_per_step(self):
        cfg = self.cfg
        return cfg.batch * cfg.height * cfg.width * (cfg.channel * 4 + 4)
