"""`UNet` with the reference's constructor / call contract (/root/reference/NetworksV2/UNet.py:29-155),
running on the sm_100a engine. `model(inputs, mode, **yaml)` plans the network for the bound input
shapes; the returned loss handle is what `Solver(args)(loss)` turns into a train op.
"""
from __future__ import annotations

import numpy as np

from .. import distribution_utils
from ..engine import EngineConfig, UNetEngine
from ..loss_metrics import metrics_from_counts
from ..solver import engine_optimizer_kwargs
from .base import BaseNet, ModeKeys


class LossHandle:
    """Stands for the `total_loss` tensor (UNet.py:134): data loss + slim L2 regularisation losses."""

    def __init__(self, model):
        self.model = model
        self.value = None

    def __float__(self):
        return float(self.value)


class UNet(BaseNet):
    def __init__(self, args, name=None):
        super().__init__(args)
        self._name = name or "UNet"
        self.classes.extend(self.args.classes)
        self.bs = distribution_utils.per_device_batch_size(args.batch_size, getattr(args, "num_gpus", 1))
        self.height = args.im_height
        self.width = args.im_width
        self.channel = args.im_channel
        self.ctx = None

    def bind_context(self, ctx, world: int = 1):
        self.ctx = ctx
        self.world = world
        return self

    def _build_network(self, *args, **kwargs):
        if getattr(self.args, "img_grad", False):
            raise NotImplementedError("--img_grad (tf.image.image_gradients inputs) is outside the accelerated path")
        if self.ctx is None:
            from ..device import Context
            self.ctx = Context(0)
            self.world = 1
        w_rate, b_rate = self._get_regularizer()
        cfg = EngineConfig(
            batch=self.bs, height=int(self.height), width=int(self.width), channel=self.channel,
            classes=tuple(self.classes), init_channels=kwargs.get("init_channels", 64),
            num_down_samples=kwargs.get("num_down_samples", 4), normalizer=self._get_normalization(),
            weight_decay_rate=w_rate or 0.0, bias_decay=(w_rate is not None and b_rate is None),
            loss_type=getattr(self.args, "loss_type", "xentropy"),
            loss_weight_type=getattr(self.args, "loss_weight_type", "none"),
            loss_numeric_w=tuple(getattr(self.args, "loss_numeric_w", None) or ()),
            loss_proportion_decay=getattr(self.args, "loss_proportion_decay", 1000.0),
            **engine_optimizer_kwargs(self.args), weight_init=self._get_initializer(),
            training=self.mode == ModeKeys.TRAIN, world=getattr(self, "world", 1),
            without_norm=bool(getattr(self.args, "without_norm", False)))
        if self.engine is None or self.engine.cfg != cfg:
            if self.engine is not None:
                self.engine.close()
            self.engine = UNetEngine(self.ctx, cfg)
            self.engine.init_weights(seed=getattr(self.args, "seed", 0))
        self.ret_prob = kwargs.get("ret_prob", False)
        self.ret_pred = kwargs.get("ret_pred", False)
        self._layers["logits"] = self.engine.logits

    def _build_loss(self):
        if self.args.loss_type not in ("xentropy", "dice"):
            raise ValueError("Not supported loss_type: {}".format(self.args.loss_type))   # UNet.py:132
        self._loss = LossHandle(self)
        return self._loss

    def _build_metrics(self):
        if not self.ret_pred:
            return
        self._want_metrics = True

    # -- execution (what sess.run does for the reference) ------------------------------------------
    def feed(self, images: np.ndarray, labels: np.ndarray | None = None):
        self.engine.set_inputs(images, labels)

    def run_forward(self):
        """Forward in the current mode; fills `probability`, `predictions["<Cls>Pred"]`, `metrics_dict`."""
        eng = self.engine
        eng.forward(self.is_training)
        want_counts = getattr(self, "_want_metrics", False) and "labels" in self._inputs
        eng.predict_outputs(want_counts)
        n, h, w, k = eng.cfg.batch, eng.cfg.height, eng.cfg.width, eng.cfg.num_classes
        self.probability = eng.prob.download(np.float32, (n, h, w, k))
        masks = eng.masks.download(np.uint8, (k - 1, n, h, w))
        for i in range(1, k):
            self.predictions[self.classes[i] + "Pred"] = masks[i - 1][..., None]
        if want_counts:
            self.metrics_dict = metrics_from_counts(eng.read_counts(), self.classes,
                                                    getattr(self.args, "metrics_train", ["Dice"]))
        return self.probability

    def collect_metrics(self):
        self.metrics_dict = metrics_from_counts(self.engine.read_counts(), self.classes,
                                                getattr(self.args, "metrics_train", ["Dice"]))
        return self.metrics_dict
