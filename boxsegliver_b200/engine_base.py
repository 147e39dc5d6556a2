"""Host-side plumbing shared by the 2-D (engine.UNetEngine and its subclasses) and 3-D (unet3d_engine.UNet3DEngine)
training engines: the training hyper-parameters, the parameter arenas and their layout, weight / gradient / optimizer-slot
I/O in TF variable shapes, the loss descriptor and the reads of its results, the fused optimizer, the layout of the
per-layer normalisation scalars, the filter-gradient side stream and the mean all-reduce of the moving statistics.

Parameter arenas (flat, element offsets aligned to 64): W (fp32 master), Wbf (bf16 shadow for the tensor-core convs), G,
M, V (gradient and optimizer slots) hold region A (L2-regularised) followed by region B (not regularised); S holds
region S, the moving statistics, which are not trained. A variable is stored in a `stored` shape that may be larger than
its TF shape (channel axes zero-padded to the blocks the kernels reduce over); the pad elements are zero in every arena.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from .device import DeviceBuffer, f32_to_bf16_bits

F32 = 4
BF16 = 2
OPTIMIZERS = ("adam", "momentum", "adamw")


def _align(n, a=64):
    return (n + a - 1) // a * a


def truncated_normal(rng, shape, stddev: float, mean: float = 0.0) -> np.ndarray:
    """tf.truncated_normal semantics: N(mean, stddev) samples, values beyond 2 stddev are dropped and re-drawn."""
    out = rng.standard_normal(shape)
    bad = np.abs(out) > 2.0
    while bad.any():
        out[bad] = rng.standard_normal(int(bad.sum()))
        bad = np.abs(out) > 2.0
    return (mean + stddev * out).astype(np.float32)


@dataclass
class TrainConfig:
    batch: int
    classes: tuple = ("Background", "Liver", "Tumor")
    normalizer: str = "batch_norm"
    weight_decay_rate: float = 1e-5
    bias_decay: bool = False
    loss_type: str = "xentropy"
    loss_weight_type: str = "none"
    loss_numeric_w: tuple = ()
    loss_proportion_decay: float = 1000.0
    optimizer: str = "adam"            # adam | momentum | adamw (core/solver.py:204-219)
    adam_beta1: float = 0.9            # reference defaults {"beta1": 0.9, "beta2": 0.99} (solver.py:206)
    adam_beta2: float = 0.99
    adam_eps: float = 1e-8
    momentum: float = 0.9              # solver.py:209
    use_nesterov: bool = False
    adamw_weight_decay: float = None   # AdamW decoupled decay; None -> weight_decay_rate (solver.py:212)
    weight_init: str = "xavier"        # xavier | trunc_norm (base.py:137-151)
    bn_decay: float = 0.999            # slim.batch_norm defaults (BaseNet._get_normalization)
    bn_eps: float = 1e-3
    in_eps: float = 1e-6
    training: bool = True              # allocate backward / optimizer state
    world: int = 1                     # data-parallel replicas (gradient mean over `world`)

    @property
    def num_classes(self):
        return len(self.classes)


@dataclass(eq=False)
class Param:
    name: str
    shape: tuple             # TF variable shape
    stored: tuple = None     # shape in the arena (None: `shape`)
    sel: tuple = ()          # index of the TF variable inside the stored shape; every other stored element is zero
    region: str = "A"        # "A" regularised, "B" not, "S" moving statistics (not trained)
    alloc: int = 0           # elements reserved in the arena when more than size (the 2-D stem filter: 64 rows)
    offset: int = 0          # element offset in the arena
    size: int = 0            # stored elements

    def __post_init__(self):
        if self.stored is None:
            self.stored = tuple(self.shape)

    def to_dev(self, a: np.ndarray) -> np.ndarray:
        """TF-shaped variable -> flat stored layout."""
        out = np.zeros(self.stored, np.float32)
        out[self.sel] = a.reshape(out[self.sel].shape)
        return out.ravel()

    def from_dev(self, flat: np.ndarray) -> np.ndarray:
        """The variable out of a whole host copy of its arena."""
        return flat[self.offset:self.offset + self.size].reshape(self.stored)[self.sel].reshape(self.shape).copy()


class EngineBase:
    """Arenas, weight I/O, loss and optimizer plumbing of an engine. A subclass sets ctx, cfg and pixels_per_sample
    (per-sample pixels or voxels of the loss), calls _init_plumbing, then _layout with its parameter list, and defines
    _loss_terms."""

    def _init_plumbing(self):
        self.step_count = 0
        self._bufs = []
        self.stream = self.ctx.stream
        self._ev_ring, self._ev_ring_i = [self.ctx.new_event() for _ in range(160)], 0
        if self.cfg.training:
            self.wg_stream = self.ctx.new_stream()
            self._dy_events = [self.ctx.new_event(), self.ctx.new_event()]

    def _check_train_config(self):
        cfg = self.cfg
        if not self._loss_terms():
            raise ValueError("Not supported loss_type: {}".format(cfg.loss_type))
        if cfg.loss_weight_type not in ("none", "numerical", "proportion"):
            raise ValueError("Not supported weight type: " + cfg.loss_weight_type)
        if cfg.loss_weight_type == "numerical" and len(cfg.loss_numeric_w) != cfg.num_classes:
            raise KeyError("w_type `numerical` need keyword argument `numeric_w` (one value per class)")
        if cfg.optimizer not in OPTIMIZERS:
            raise ValueError("Not supported optimizer: " + cfg.optimizer)       # solver.py:217
        if cfg.weight_init not in ("xavier", "trunc_norm"):
            raise ValueError("Not supported weight initializer: " + cfg.weight_init)   # base.py:147

    def _alloc(self, nbytes) -> DeviceBuffer:
        b = self.ctx.alloc(max(int(nbytes), 16))
        self._bufs.append(b)
        return b

    def close(self):
        for b in self._bufs:
            b.free()
        self._bufs = []

    # ------------------------------------------------------------------ parameter arenas
    def _layout(self, plist):
        """Offsets of region A, then B, in the trained arenas and of S in its own; allocates the arenas."""
        ends = {}
        for region in ("A", "B", "S"):
            off = 0 if region != "B" else ends["A"]
            for p in plist:
                if p.region == region:
                    p.size = int(np.prod(p.stored))
                    p.offset = off
                    off += _align(max(p.size, p.alloc))
            ends[region] = off
        self.n_reg, self.n_train, self.n_stats = ends["A"], ends["B"], ends["S"]
        self.params = {p.name: p for p in plist}
        self.W = self._alloc(self.n_train * F32)
        self.Wbf = self._alloc(self.n_train * BF16)
        self.S = self._alloc(max(self.n_stats, 1) * F32)
        if self.cfg.training:
            self.G = self._alloc(self.n_train * F32).zero()
            self.M = self._alloc(self.n_train * F32).zero()
            self.V = self._alloc(self.n_train * F32).zero() if self.cfg.optimizer in ("adam", "adamw") else None
        self.sumsq = self._alloc(16)

    def set_weights(self, weights: dict):
        """Load a {tf variable name: numpy array} map (TF layouts) into W, its bf16 shadow and S."""
        hostW = np.zeros(self.n_train, np.float32)
        hostS = np.zeros(max(self.n_stats, 1), np.float32)
        for name, p in self.params.items():
            if name not in weights:
                raise KeyError(f"missing variable {name}")
            a = np.asarray(weights[name], np.float32)
            if tuple(a.shape) != tuple(p.shape):
                raise ValueError(f"{name}: shape {a.shape} != {p.shape}")
            (hostS if p.region == "S" else hostW)[p.offset:p.offset + p.size] = p.to_dev(a)
        self.W.upload(hostW)
        self.Wbf.upload(f32_to_bf16_bits(hostW))
        self.S.upload(hostS)

    def get_weights(self) -> dict:
        hostW = self.W.download(np.float32, (self.n_train,))
        hostS = self.S.download(np.float32, (max(self.n_stats, 1),))
        return {name: p.from_dev(hostS if p.region == "S" else hostW) for name, p in self.params.items()}

    def get_grads(self) -> dict:
        hostG = self.G.download(np.float32, (self.n_train,))
        return {name: p.from_dev(hostG) for name, p in self.params.items() if p.region != "S"}

    def get_slots(self) -> dict:
        """Optimizer slots in TF variable shapes: {variable name: (m, v)} for Adam / AdamW, {name: (acc,)} for Momentum."""
        arenas = [self.M.download(np.float32, (self.n_train,))]
        if self.V is not None:
            arenas.append(self.V.download(np.float32, (self.n_train,)))
        return {name: tuple(p.from_dev(a) for a in arenas) for name, p in self.params.items() if p.region != "S"}

    def set_slots(self, slots: dict):
        """Inverse of get_slots (every trainable variable must be present)."""
        arenas = [np.zeros(self.n_train, np.float32) for _ in range(2 if self.V is not None else 1)]
        for name, p in self.params.items():
            if p.region == "S":
                continue
            if name not in slots:
                raise KeyError(f"missing optimizer slots of {name}")
            for dst, a in zip(arenas, slots[name]):
                a = np.asarray(a, np.float32)
                if tuple(a.shape) != tuple(p.shape):
                    raise ValueError(f"{name}: slot shape {a.shape} != {p.shape}")
                dst[p.offset:p.offset + p.size] = p.to_dev(a)
        self.M.upload(arenas[0])
        if self.V is not None:
            self.V.upload(arenas[1])

    def _draw_weight(self, rng, shp, fan_in, fan_out):
        """--weight_init (/root/reference/NetworksV2/base.py:137-151): slim.xavier_initializer() (uniform) or
        tf.truncated_normal_initializer(stddev=0.01) -- normal samples re-drawn while |x| > 2 sigma."""
        if self.cfg.weight_init == "trunc_norm":
            return truncated_normal(rng, shp, 0.01)
        lim = np.sqrt(6.0 / (fan_in + fan_out))
        return rng.uniform(-lim, lim, size=shp).astype(np.float32)

    def init_weights(self, seed: int = 0):
        """--weight_init filters (seeded numpy stream), zero biases, gamma 1, beta 0, moving 0 / 1."""
        rng = np.random.default_rng(seed)
        w = {}
        for name, p in self.params.items():
            shp = p.shape
            if name.endswith("/weights"):
                rf = int(np.prod(shp[:-2]))
                w[name] = self._draw_weight(rng, shp, rf * shp[-2], rf * shp[-1])
            elif name.endswith(("gamma", "moving_variance")):
                w[name] = np.ones(shp, np.float32)
            else:
                w[name] = np.zeros(shp, np.float32)
        self.set_weights(w)
        return w

    # ------------------------------------------------------------------ normalisation scalars
    @staticmethod
    def _norm_scalar_floats(entries: int, k: int = 2) -> int:
        """Floats of one layer's scalar set: k fp64 sums, then mean, rstd, scale, shift, c1, c2, per entry (group x channel)."""
        return (2 * k + 6) * _align(entries, 16)

    @staticmethod
    def _norm_scalars(base: int, entries: int, k: int = 2) -> dict:
        """Pointers into a scalar set laid out as _norm_scalar_floats counts it, starting at address `base`."""
        n = _align(entries, 16)
        out = {"sums": C.c_void_p(base)}
        for i, nm in enumerate(("mean", "rstd", "scale", "shift", "c1", "c2")):
            out[nm] = C.c_void_p(base + (2 * k + i) * n * F32)
        return out

    # ------------------------------------------------------------------ streams
    def _stream_wait(self, waiter, stream):
        """`waiter` waits for everything enqueued on `stream` so far (an event of a ring far longer than a step uses)."""
        ev = self._ev_ring[self._ev_ring_i]
        self._ev_ring_i = (self._ev_ring_i + 1) % len(self._ev_ring)
        self.ctx.record(ev, stream)
        self.ctx.call("bsl_stream_wait_event", waiter, ev)

    def _allreduce_moving_stats(self, stream=None):
        # MirroredStrategy aggregates the moving-average updates with MEAN across replicas
        # (/root/reference/core/estimator.py:570-613); batch statistics themselves stay per replica (no sync-BN).
        # On a stream other than the compute stream the exchange runs behind everything enqueued there so far.
        if self.cfg.world > 1 and self.n_stats > 0:
            st = self.stream if stream is None else stream
            if st is not self.stream:
                self._stream_wait(st, self.stream)
            self.ctx.call("bsl_allreduce_sum_f32", self.S.p, C.c_size_t(self.n_stats), st)
            self.ctx.call("bsl_scale_f32", self.S.p, C.c_size_t(self.n_stats), C.c_float(1.0 / self.cfg.world), st)

    # ------------------------------------------------------------------ loss, outputs, optimizer
    def _loss_desc(self):
        cfg = self.cfg
        wt = {"none": 0, "numerical": 1, "proportion": 2}[cfg.loss_weight_type]
        nw = (C.c_float * 8)(*([float(x) for x in cfg.loss_numeric_w] + [0.0] * (8 - len(cfg.loss_numeric_w))))
        return _lib.LossDesc(cfg.batch, self.pixels_per_sample, cfg.num_classes, wt, nw,
                             float(cfg.loss_proportion_decay), 1.0 / cfg.world)

    def predict_outputs(self, with_counts: bool):
        """softmax, `<Cls>Pred` masks, argmax and (optionally) the integer Dice sums, one pass over the logits."""
        ld = self._loss_desc()
        self.ctx.call("bsl_softmax_threshold", C.byref(ld), self.logits.p, self.labels.p if with_counts else None,
                      self.prob.p, self.masks.p, self.argmax.p, self.ilr.p if with_counts else None, self.stream)

    def read_loss(self):
        """(data loss, L2 regularisation loss) of the step just run; the only D2H read of a train step."""
        data = float(self.loss_dev.download(np.float32, (len(self._loss_terms()),)).sum())
        sq = self.sumsq.download(np.float64, (1,))[0]
        return data, float(self.cfg.weight_decay_rate * 0.5 * sq) if self.cfg.weight_decay_rate > 0 else 0.0

    def read_counts(self):
        return self.ilr.download(np.uint32, (self.cfg.batch, self.cfg.num_classes - 1, 3))

    def optimizer_step(self, lr: float):
        """One fused update over region A ([0, n_reg), L2-regularised) and region B of the trained arenas.
        Hyper-parameters come from the config (core/solver.py:86-97,204-219)."""
        self.step_count += 1
        ctx, s, cfg = self.ctx, self.stream, self.cfg
        l2 = cfg.weight_decay_rate if cfg.weight_decay_rate > 0 else 0.0
        regions = [(0, self.n_reg, l2, self.sumsq.p), (self.n_reg, self.n_train - self.n_reg, 0.0, None)]
        if cfg.optimizer not in OPTIMIZERS:
            raise ValueError("Not supported optimizer: " + cfg.optimizer)
        decay = 0.0
        if cfg.optimizer == "adamw":       # DecoupledWeightDecayExtension decays EVERY variable (decay_var_list=None)
            decay = cfg.weight_decay_rate if cfg.adamw_weight_decay is None else cfg.adamw_weight_decay
        for off, n, rate, sq in regions:
            if n <= 0:
                continue
            w = C.c_void_p(self.W.ptr + off * F32)
            g = C.c_void_p(self.G.ptr + off * F32)
            m = C.c_void_p(self.M.ptr + off * F32)
            wb = C.c_void_p(self.Wbf.ptr + off * BF16)
            if cfg.optimizer in ("adam", "adamw"):
                v = C.c_void_p(self.V.ptr + off * F32)
                d = _lib.AdamDesc(lr, cfg.adam_beta1, cfg.adam_beta2, cfg.adam_eps, rate, 1.0, self.step_count, decay)
                ctx.call("bsl_adam_step", C.byref(d), w, g, m, v, wb, C.c_size_t(n), sq, s)
            else:
                ctx.call("bsl_momentum_step", C.c_float(lr), C.c_float(cfg.momentum), C.c_int(int(cfg.use_nesterov)),
                         C.c_float(rate), C.c_float(1.0), w, g, m, wb, C.c_size_t(n), sq, s)
