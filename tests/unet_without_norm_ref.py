"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY: the 2-D UNet (oracle/unet_ref.py) with --without_norm.

slim.conv2d with normalizer_fn=None (tensorflow/contrib/layers convolution2d, the arg scope of
/root/reference/NetworksV2/UNet.py:41-56 without a normaliser) keeps its `biases` variable (zeros initializer), adds it
and applies ReLU: a = relu(conv2d(x, w) + b), stored with one rounding; backward d = da * (a > 0), db = sum of d.
Variables UNet/<scope>/{weights, biases} for every 3x3 conv. Everything that does not depend on the normaliser (layer
table, transposed convs, pools, logits, loss, L2 term, weight initialisation order) is oracle/unet_ref.py's own.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle import tf_ops as O
from oracle import unet_ref as U
from oracle.unet_ref import (Tape, loss_and_dlogits, regularization_loss, regularized_names,  # noqa: F401
                             total_grads, trainable_names)


@dataclass
class UNetCfg(U.UNetCfg):
    without_norm: bool = True


def init_params(cfg: UNetCfg, seed: int = 0, dtype=np.float32) -> dict:
    """Seeded slim.xavier_initializer() weights (U.init_params' random stream: biases draw nothing), zero biases."""
    rng = np.random.default_rng(seed)
    p = {}
    for kind, scope, cin, cout, _ in U.conv_specs(cfg):
        if kind == "conv":
            p[f"{scope}/weights"] = O.xavier_uniform(rng, (3, 3, cin, cout), 9 * cin, 9 * cout, dtype)
        elif kind == "convT":
            p[f"{scope}/weights"] = O.xavier_uniform(rng, (2, 2, cout, cin), 4 * cout, 4 * cin, dtype)
        else:
            p[f"{scope}/weights"] = O.xavier_uniform(rng, (1, 1, cin, cout), cin, cout, dtype)
        p[f"{scope}/biases"] = np.zeros(cout, dtype)
    return p


def _identity(a):
    return a


def _walk(cfg: UNetCfg, x, conv, up):
    """UNet._build_network's trunk: conv(x, scope, first) for the 3x3 layers, up(x, scope) for the transposed convs.
    Returns (tape layers without the logits entry, last activation)."""
    layers, skips = [], []
    first = True
    for i in range(cfg.num_down_samples):
        for j in (1, 2):
            x = conv(x, f"UNet/Encode{i + 1}/Repeat/convolution2d_{j}", first, layers)
            first = False
        skips.append(x)
        layers.append(dict(kind="pool", x=x))
        x = O.max_pool_2x2(x)
    for j in (1, 2):
        x = conv(x, f"UNet/ED-Bridge/ED-Bridge_{j}", False, layers)
    for i in reversed(range(cfg.num_down_samples)):
        scope = f"UNet/Decode{i + 1}/Conv2d_transpose"
        u = up(x, scope, layers)
        x = np.concatenate((skips[i], u), axis=-1)
        layers.append(dict(kind="concat", split=skips[i].shape[-1], level=i))
        for j in (1, 2):
            x = conv(x, f"UNet/Decode{i + 1}/Repeat/convolution2d_{j}", False, layers)
    return layers, x


def forward(params: dict, images: np.ndarray, cfg: UNetCfg, is_training: bool = True, rnd=_identity, wrnd=None,
            stem_fp32: bool = True) -> Tape:
    """Same in training and evaluation (no normaliser state). `rnd` / `wrnd` / `stem_fp32` as in U.forward."""
    wrnd = wrnd or rnd
    dt = images.dtype

    def W(scope, master=False):
        w = params[f"{scope}/weights"].astype(dt)
        return w if master else wrnd(w).astype(dt)

    def conv(x, scope, first, layers):
        w = W(scope, master=first and stem_fp32)
        a = rnd(O.relu(O.conv2d(x, w) + params[f"{scope}/biases"].astype(dt))).astype(dt)
        layers.append(dict(kind="conv", scope=scope, x=x, w=w, a=a, first=first))
        return a

    def up(x, scope, layers):
        w = W(scope)
        a = rnd(O.relu(O.conv2d_transpose(x, w) + params[f"{scope}/biases"].astype(dt))).astype(dt)
        layers.append(dict(kind="convT", scope=scope, x=x, w=w, a=a))
        return a

    tape = Tape()
    tape.layers, x = _walk(cfg, images, conv, up)
    scope = "UNet/AdjustChannels"
    w = W(scope, master=True)
    tape.layers.append(dict(kind="logits", scope=scope, x=x, w=w))
    tape.logits = O.conv2d(x, w) + params[f"{scope}/biases"].astype(dt)
    tape.prob = O.softmax(tape.logits)
    return tape


def tape_from_stored(params: dict, images: np.ndarray, stored: dict, logits: np.ndarray, cfg: UNetCfg,
                     wrnd=_identity) -> Tape:
    """Backward tape from activations STORED by another implementation (`stored[scope]["a"]`), as U.tape_from_stored."""
    dt = images.dtype

    def conv(x, scope, first, layers):
        w = params[f"{scope}/weights"].astype(dt)
        w = w if first else wrnd(w).astype(dt)
        a = stored[scope]["a"].astype(dt)
        layers.append(dict(kind="conv", scope=scope, x=x, w=w, a=a, first=first))
        return a

    def up(x, scope, layers):
        a = stored[scope]["a"].astype(dt)
        layers.append(dict(kind="convT", scope=scope, x=x, w=wrnd(params[f"{scope}/weights"].astype(dt)).astype(dt), a=a))
        return a

    tape = Tape()
    tape.layers, x = _walk(cfg, images, conv, up)
    scope = "UNet/AdjustChannels"
    tape.layers.append(dict(kind="logits", scope=scope, x=x, w=params[f"{scope}/weights"].astype(dt)))
    tape.logits = logits.astype(dt)
    tape.prob = O.softmax(tape.logits)
    return tape


def layerwise_forward_errors(params: dict, images: np.ndarray, stored: dict, logits: np.ndarray, cfg: UNetCfg,
                             is_training: bool = True, wrnd=_identity) -> dict:
    """Op-by-op forward parity on identical inputs, as U.layerwise_forward_errors: {"<scope>:a" | "logits": rel L2}."""
    dt = np.float64
    errs = {}

    def rel(a, b):
        a, b = np.asarray(a, dt), np.asarray(b, dt)
        return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))

    def conv(x, scope, first, layers):
        w = params[f"{scope}/weights"].astype(dt)
        w = w if first else wrnd(w).astype(dt)
        a = stored[scope]["a"].astype(dt)
        errs[f"{scope}:a"] = rel(a, O.relu(O.conv2d(x, w) + params[f"{scope}/biases"].astype(dt)))
        return a

    def up(x, scope, layers):
        w = wrnd(params[f"{scope}/weights"].astype(dt)).astype(dt)
        a = stored[scope]["a"].astype(dt)
        errs[f"{scope}:a"] = rel(a, O.relu(O.conv2d_transpose(x, w) + params[f"{scope}/biases"].astype(dt)))
        return a

    _, x = _walk(cfg, images.astype(dt), conv, up)
    scope = "UNet/AdjustChannels"
    errs["logits"] = rel(logits, O.conv2d(x, params[f"{scope}/weights"].astype(dt)) + params[f"{scope}/biases"].astype(dt))
    return errs


def backward(tape: Tape, dlogits: np.ndarray, cfg: UNetCfg, rnd=_identity) -> dict:
    """tf.gradients of the data loss w.r.t. every trainable variable (no L2 term: see total_grads)."""
    grads = {}
    dt = dlogits.dtype
    d = dlogits
    skip_grads = {}
    for L in reversed(tape.layers):
        k = L["kind"]
        if k == "logits":
            grads[f"{L['scope']}/weights"] = O.conv2d_backprop_filter(L["x"], L["w"].shape, d)
            grads[f"{L['scope']}/biases"] = d.sum(axis=(0, 1, 2))
            d = rnd(O.conv2d_backprop_input(L["x"].shape, L["w"], d)).astype(dt)
        elif k == "conv":
            dy = rnd(O.relu_grad(d, L["a"])).astype(dt)
            grads[f"{L['scope']}/biases"] = dy.sum(axis=(0, 1, 2))
            grads[f"{L['scope']}/weights"] = O.conv2d_backprop_filter(L["x"], L["w"].shape, dy)
            d = None if L["first"] else rnd(O.conv2d_backprop_input(L["x"].shape, L["w"], dy)).astype(dt)
        elif k == "concat":
            skip_grads[L["level"]] = d[..., :L["split"]]
            d = d[..., L["split"]:]
        elif k == "convT":
            dyr = rnd(O.relu_grad(d, L["a"])).astype(dt)
            dx, dw = O.conv2d_transpose_grad(L["x"], L["w"], dyr)
            grads[f"{L['scope']}/weights"] = dw
            grads[f"{L['scope']}/biases"] = dyr.sum(axis=(0, 1, 2))
            d = rnd(dx).astype(dt)
        elif k == "pool":
            level = max(skip_grads)  # deepest pending skip belongs to this pool's input
            d = rnd(O.max_pool_2x2_grad(L["x"], d) + skip_grads.pop(level)).astype(dt)
    return grads

