"""fp64 reference of one normalised layer as the normalisation passes of csrc/norm.cu compute it (numpy only).

Forward, for y [n, h, w, c] (the bf16 conv output, given as float values):

    xhat = (y - mean) * rstd                 instance (per sample and channel) or batch (per channel) moments
    t    = xhat * gamma + beta               each optional (slim's scale / center)
    v    = t * gamma_mod[n, c]               optional: GUNet conditional normalisation (GUNet.py:119-133)
    u    = v + guide @ w_guide + b_guide     optional: GUNet's 1x1 spatial-guide conv, G = 1 or 2 channels
    z    = ga * u + ba                       optional: after_affine (channel_wise_affine, GUNet.py:213-214)
    a    = relu(z)                           optional
    then a 2x2 max-pool of a, or the 1x1 logits conv a @ w_head + b_head (optional)

which is modulated_conv_block as oracle/gunet_ref.py states it inline. The batch-norm forward also returns the moving
statistics after one update, fed the Bessel-corrected variance (oracle.tf_ops.batch_norm_train).

The backward is written out by hand. `mask` replaces (z > 0) as the ReLU's gradient gate: a device test passes the
device's stored activation > 0, so that an fp32 z within rounding of zero cannot flip a gate bit between the kernel and
this reference."""
from __future__ import annotations

import numpy as np

from oracle import tf_ops as O


def _f8(a):
    return None if a is None else np.asarray(a, np.float64)


def forward(y, mode: str, eps: float, gamma=None, beta=None, gamma_mod=None, guide=None, w_guide=None, b_guide=None,
            ga=None, ba=None, relu: bool = True, pool: bool = False, w_head=None, b_head=None, moving=None,
            decay: float = 0.999) -> dict:
    """mode "instance" or "batch". guide [n, h, w, G], w_guide [G, c], gamma_mod [n, c], w_head [c, classes].
    moving = (moving_mean, moving_var) before the update (batch mode). Returns the intermediates the backward needs and
    mean / rstd with shape [n, c] (instance) or [c] (batch)."""
    assert mode in ("instance", "batch")
    y = np.asarray(y, np.float64)
    n, h, w, c = y.shape
    axes = (1, 2) if mode == "instance" else (0, 1, 2)
    mean = y.mean(axis=axes, keepdims=True)
    var = y.var(axis=axes, keepdims=True)
    rstd = 1.0 / np.sqrt(var + eps)
    xhat = (y - mean) * rstd
    gamma, beta, gamma_mod, guide = _f8(gamma), _f8(beta), _f8(gamma_mod), _f8(guide)
    t = xhat * gamma if gamma is not None else xhat.copy()
    if beta is not None:
        t += beta
    v = t * gamma_mod[:, None, None, :] if gamma_mod is not None else t
    u = v
    if guide is not None:
        u = v + guide @ _f8(w_guide)
        if b_guide is not None:
            u += _f8(b_guide)
    elif b_guide is not None:
        u = v + _f8(b_guide)
    z = u * _f8(ga) + _f8(ba) if ga is not None else u
    a = np.maximum(z, 0.0) if relu else z
    out = dict(mode=mode, y=y, mean_k=mean, rstd_k=rstd, xhat=xhat, t=t, v=v, u=u, z=z, a=a, relu=relu, gamma=gamma,
               beta=beta, gamma_mod=gamma_mod, guide=guide, w_guide=_f8(w_guide), ga=_f8(ga), w_head=_f8(w_head),
               mean=mean.reshape(n, c) if mode == "instance" else mean.reshape(c),
               rstd=rstd.reshape(n, c) if mode == "instance" else rstd.reshape(c), var=var)
    if pool:
        out["pooled"] = O.max_pool_2x2(a)
    if w_head is not None:
        out["logits"] = a @ out["w_head"] + (_f8(b_head) if b_head is not None else 0.0)
    if mode == "batch" and moving is not None:
        m = n * h * w
        mm, mv = _f8(moving[0]), _f8(moving[1])
        out["moving_mean"] = mm * decay + mean.reshape(c) * (1.0 - decay)
        out["moving_var"] = mv * decay + var.reshape(c) * (m / max(m - 1, 1)) * (1.0 - decay)
    return out


def backward(f: dict, da=None, dpooled=None, dlogits=None, mask=None) -> dict:
    """Gradients of the forward `f` given the gradient w.r.t. the activation `da`, w.r.t. the pooled tensor `dpooled`
    (MaxPoolGrad: the first maximum of a window takes it) and / or w.r.t. the logits `dlogits`; they add up.
    Returns dy, dgamma, dbeta, dgamma_mod [n, c], dw_guide [G, c], dbias_guide, dga, dba, dw_head, db_head (the ones
    the forward had parameters for; dgamma / dbeta always, as the gradients of a gamma of one / a beta of zero)."""
    a = f["a"]
    g = np.zeros_like(a) if da is None else np.asarray(da, np.float64).copy()
    out = {}
    if dpooled is not None:
        g += O.max_pool_2x2_grad(a, np.asarray(dpooled, np.float64))
    if dlogits is not None:
        dl = np.asarray(dlogits, np.float64)
        out["dw_head"] = np.einsum("nhwc,nhwk->ck", a, dl)
        out["db_head"] = dl.sum(axis=(0, 1, 2))
        g += dl @ f["w_head"].T
    if f["relu"]:
        g *= (f["z"] > 0) if mask is None else np.asarray(mask, bool)
    red = (0, 1, 2)
    if f["ga"] is not None:
        out["dga"] = (g * f["u"]).sum(axis=red)
        out["dba"] = g.sum(axis=red)
        g *= f["ga"]
    if f["guide"] is not None:
        out["dw_guide"] = np.einsum("nhwg,nhwc->gc", f["guide"], g)
    out["dbias_guide"] = g.sum(axis=red)
    if f["gamma_mod"] is not None:
        out["dgamma_mod"] = (g * f["t"]).sum(axis=(1, 2))
        g *= f["gamma_mod"][:, None, None, :]
    xhat = f["xhat"]
    out["dgamma"] = (g * xhat).sum(axis=red)
    out["dbeta"] = g.sum(axis=red)
    if f["gamma"] is not None:
        g *= f["gamma"]
    axes = (1, 2) if f["mode"] == "instance" else red
    m1 = g.mean(axis=axes, keepdims=True)
    m2 = (g * xhat).mean(axis=axes, keepdims=True)
    g -= m1
    g -= xhat * m2
    g *= f["rstd_k"]
    out["dy"] = g
    return out
