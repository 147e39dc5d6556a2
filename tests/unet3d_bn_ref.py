"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY: UNet3D (oracle/unet3d_ref.py) with --normalizer batch_norm.

slim.batch_norm after every conv3d (/root/reference/NetworksV2/UNet3D.py:151-158 through BaseNet._get_normalization,
NetworksV2/base.py:154-162): per-channel batch statistics over all n*d*h*w voxels in training (biased variance for the
normalisation, the Bessel-corrected one fed to the moving variance), the moving statistics in eval mode. Variables
UNet3D/<block>/<layer>/BatchNorm/{gamma, beta, moving_mean, moving_variance}. Everything that does not depend on the
normaliser (layer table, loss, L2 term, weight initialisation order) is oracle/unet3d_ref.py's own.
"""
from __future__ import annotations

from dataclasses import dataclass, replace

import numpy as np

from oracle import tf_ops as O
from oracle import unet3d_ref as U
from oracle.unet3d_ref import Tape, loss_and_dlogits, regularization_loss, total_grads  # noqa: F401


@dataclass
class UNet3DBNCfg(U.UNet3DCfg):
    normalizer: str = "batch_norm"
    bn_eps: float = 1e-3
    bn_decay: float = 0.999


def layer_specs(cfg: UNet3DBNCfg):
    return U.layer_specs(replace(cfg, normalizer="instance_norm"))


def init_params(cfg: UNet3DBNCfg, seed: int = 0, dtype=np.float32) -> dict:
    """U.init_params (same random stream), normaliser variables renamed, moving mean 0 / variance 1 added."""
    p = {}
    for k, v in U.init_params(replace(cfg, normalizer="instance_norm"), seed, dtype).items():
        k = k.replace("/InstanceNorm/", "/BatchNorm/")
        p[k] = v
        if k.endswith("/BatchNorm/beta"):
            ns = k[:-len("beta")]
            p[ns + "moving_mean"] = np.zeros_like(v)
            p[ns + "moving_variance"] = np.ones_like(v)
    return p


def moving_names(params: dict):
    return [k for k in params if k.endswith(("moving_mean", "moving_variance"))]


def forward(params: dict, inputs: dict, cfg: UNet3DBNCfg, is_training: bool, rnd=U._identity, wrnd=None,
            stored=None) -> Tape:
    """U.forward with batch norm. Training: tape.moving holds the updated moving statistics. `stored` as in U.forward."""
    wrnd = wrnd or rnd
    tape = Tape()
    tape.moving = {}
    x = inputs["images"]
    if cfg.use_spatial:
        x = np.concatenate((inputs["images"], inputs["sp_guide"]), axis=-1)
    dt = x.dtype

    def rel(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))

    skips = {}
    first = True
    for s in layer_specs(cfg):
        sc = s["scope"]
        if s["kind"] == "conv":
            w = params[f"{sc}/weights"].astype(dt)
            w = w if first else wrnd(w).astype(dt)
            y = rnd(O.conv3d(x, w, s["s"])).astype(dt)
            if stored is not None:
                tape.errs[f"{sc}:y"] = rel(stored[sc]["y"], y)
                y = stored[sc]["y"].astype(dt)
            ns = f"{sc}/BatchNorm"
            g, b = params[f"{ns}/gamma"].astype(dt), params[f"{ns}/beta"].astype(dt)
            mm, mv = params[f"{ns}/moving_mean"].astype(dt), params[f"{ns}/moving_variance"].astype(dt)
            if is_training:
                z, cache, nmm, nmv = O.batch_norm_train(y, g, b, mm, mv, cfg.bn_eps, cfg.bn_decay)
                tape.moving[f"{ns}/moving_mean"], tape.moving[f"{ns}/moving_variance"] = nmm, nmv
            else:
                z, cache = O.batch_norm_infer(y, g, b, mm, mv, cfg.bn_eps), None
            a = rnd(O.relu(z)).astype(dt)
            if stored is not None:
                tape.errs[f"{sc}:a"] = rel(stored[sc]["a"], a)
                a = stored[sc]["a"].astype(dt)
            tape.layers.append(dict(kind="conv", spec=s, x=x, w=w, z=z, a=a, cache=cache, first=first))
            first = False
            x = a
            if s["layer"] == "conv2" and s["block"].startswith("conv_e"):
                skips[s["block"]] = a
                tape.layers.append(dict(kind="fork", block=s["block"]))
        elif s["kind"] == "convT":
            w = wrnd(params[f"{sc}/weights"].astype(dt)).astype(dt)
            up = rnd(O.relu(O.conv3d_transpose(x, w, s["s"]))).astype(dt)
            if stored is not None:
                tape.errs[f"{sc}:a"] = rel(stored[sc]["a"], up)
                up = stored[sc]["a"].astype(dt)
            tape.layers.append(dict(kind="convT", spec=s, x=x, w=w, a=up))
            skip = skips[s["block"].replace("d", "e")]
            x = np.concatenate((skip, up), axis=-1)
            tape.layers.append(dict(kind="concat", split=skip.shape[-1], block=s["block"].replace("d", "e")))
        else:
            w = params[f"{sc}/weights"].astype(dt)
            logits = O.conv3d(x, w) + params[f"{sc}/biases"].astype(dt)
            if stored is not None:
                tape.errs["logits"] = rel(stored["logits"], logits)
                logits = stored["logits"].astype(dt)
            tape.layers.append(dict(kind="logits", spec=s, x=x, w=w))
            tape.logits = logits
            tape.prob = O.softmax(logits)
    return tape


def backward(tape: Tape, dlogits: np.ndarray, cfg: UNet3DBNCfg, rnd=U._identity) -> dict:
    """U.backward with FusedBatchNormGrad; gradients of the trainable variables only."""
    grads = {}
    dt = dlogits.dtype
    d = dlogits
    skip_grads = {}
    for L in reversed(tape.layers):
        k = L["kind"]
        if k == "logits":
            sc = L["spec"]["scope"]
            grads[f"{sc}/weights"] = O.conv3d_backprop_filter(L["x"], L["w"].shape, d)
            grads[f"{sc}/biases"] = d.sum(axis=(0, 1, 2, 3))
            d = rnd(O.conv3d_backprop_input(L["x"].shape, L["w"], d)).astype(dt)
        elif k == "conv":
            s = L["spec"]
            sc = s["scope"]
            dz = O.relu_grad(d, L["a"])
            dy, dg, db = O.batch_norm_grad(dz, L["cache"])
            dy = rnd(dy).astype(dt)
            grads[f"{sc}/BatchNorm/gamma"] = dg
            grads[f"{sc}/BatchNorm/beta"] = db
            grads[f"{sc}/weights"] = O.conv3d_backprop_filter(L["x"], L["w"].shape, dy, s["s"])
            d = None if L["first"] else rnd(O.conv3d_backprop_input(L["x"].shape, L["w"], dy, s["s"])).astype(dt)
        elif k == "concat":
            skip_grads[L["block"]] = d[..., :L["split"]]
            d = d[..., L["split"]:]
        elif k == "convT":
            s = L["spec"]
            dyr = rnd(O.relu_grad(d, L["a"])).astype(dt)
            dx, dw = O.conv3d_transpose_grad(L["x"], L["w"], dyr, s["s"])
            grads[f"{s['scope']}/weights"] = dw
            d = rnd(dx).astype(dt)
        elif k == "fork":
            d = rnd(d + skip_grads.pop(L["block"])).astype(dt)
    return grads
