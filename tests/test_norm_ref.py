"""Pins the fp64 normalised-layer reference (tests/norm_ref.py): without modulation it is oracle.tf_ops' instance_norm /
batch_norm_train and their gradients; with every option it matches torch float64 autograd of the same forward."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import tf_ops as O
from tests import norm_ref as R


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _inputs(rng, n, h, w, c, G, classes):
    return dict(
        y=rng.standard_normal((n, h, w, c)) * 1.3 + rng.standard_normal((n, 1, 1, c)),
        gamma=rng.uniform(0.5, 1.5, c), beta=rng.normal(0, 0.3, c), gamma_mod=rng.uniform(0.5, 1.5, (n, c)),
        guide=rng.uniform(0, 1, (n, h, w, max(G, 1)))[..., :G], w_guide=rng.normal(0, 0.5, (max(G, 1), c))[:G],
        b_guide=rng.normal(0, 0.3, c), ga=rng.uniform(0.5, 1.5, c), ba=rng.normal(0, 0.3, c),
        w_head=rng.normal(0, 0.3, (c, classes)), b_head=rng.normal(0, 0.3, classes),
        mm=rng.normal(0, 0.2, c), mv=rng.uniform(0.5, 1.5, c),
        da=rng.standard_normal((n, h, w, c)), dpooled=rng.standard_normal((n, h // 2, w // 2, c)),
        dlogits=rng.standard_normal((n, h, w, classes)))


@pytest.mark.parametrize("mode", ["instance", "batch"])
def test_reference_without_modulation_is_the_tf_oracle(mode):
    rng = np.random.default_rng(3)
    n, h, w, c = 3, 6, 10, 16
    x = _inputs(rng, n, h, w, c, 0, 2)
    eps = 1e-6 if mode == "instance" else 1e-3
    f = R.forward(x["y"], mode, eps, x["gamma"], x["beta"], relu=False, moving=(x["mm"], x["mv"]), decay=0.99)
    b = R.backward(f, da=x["da"])
    if mode == "instance":
        z, cache = O.instance_norm(x["y"], x["gamma"], x["beta"], eps)
        dx, dg, db = O.instance_norm_grad(x["da"], cache)
    else:
        z, cache, nmm, nmv = O.batch_norm_train(x["y"], x["gamma"], x["beta"], x["mm"], x["mv"], eps, 0.99)
        dx, dg, db = O.batch_norm_grad(x["da"], cache)
        assert _rel(f["moving_mean"], nmm) < 1e-12 and _rel(f["moving_var"], nmv) < 1e-12
    assert _rel(f["a"], z) < 1e-12
    for got, ref in ((b["dy"], dx), (b["dgamma"], dg), (b["dbeta"], db)):
        assert _rel(got, ref) < 1e-12


def _torch_layer(x, mode, eps, o):
    """The same layer with torch ops (NCHW), autograd through every parameter; returns outputs and gradients."""
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, requires_grad=True)  # noqa: E731
    P = {k: t(x[k]) for k in ("y", "gamma", "beta", "gamma_mod", "w_guide", "b_guide", "ga", "ba", "w_head", "b_head")}
    y = P["y"].permute(0, 3, 1, 2)
    c = y.shape[1]
    if mode == "instance":
        zn = F.instance_norm(y, eps=eps)
        mm = mv = None
    else:
        mm, mv = torch.tensor(x["mm"], dtype=torch.float64), torch.tensor(x["mv"], dtype=torch.float64)
        zn = F.batch_norm(y, mm, mv, training=True, momentum=1.0 - o["decay"], eps=eps)
    col = lambda v: v.view(1, c, 1, 1)  # noqa: E731
    if o["scale"]:
        zn = zn * col(P["gamma"])
    if o["center"]:
        zn = zn + col(P["beta"])
    if o["gm"]:
        zn = zn * P["gamma_mod"].view(-1, c, 1, 1)
    if o["G"]:
        gd = torch.tensor(x["guide"], dtype=torch.float64).permute(0, 3, 1, 2)
        zn = zn + F.conv2d(gd, P["w_guide"].t().reshape(c, o["G"], 1, 1), P["b_guide"])
    if o["affine"]:
        zn = zn * col(P["ga"]) + col(P["ba"])
    a = torch.relu(zn) if o["relu"] else zn
    loss = (a * torch.tensor(x["da"], dtype=torch.float64).permute(0, 3, 1, 2)).sum()
    res = dict(a=a.detach().permute(0, 2, 3, 1).numpy())
    if o["tail"] == "pool":
        p = F.max_pool2d(a, 2)
        res["pooled"] = p.detach().permute(0, 2, 3, 1).numpy()
        loss = loss + (p * torch.tensor(x["dpooled"], dtype=torch.float64).permute(0, 3, 1, 2)).sum()
    if o["tail"] == "head":
        k = P["w_head"].shape[1]
        lg = F.conv2d(a, P["w_head"].t().reshape(k, c, 1, 1), P["b_head"])
        res["logits"] = lg.detach().permute(0, 2, 3, 1).numpy()
        loss = loss + (lg * torch.tensor(x["dlogits"], dtype=torch.float64).permute(0, 3, 1, 2)).sum()
    loss.backward()
    res["grads"] = {k: (v.grad.numpy() if v.grad is not None else None) for k, v in P.items()}
    if mm is not None:
        res["moving_mean"], res["moving_var"] = mm.numpy(), mv.numpy()
    return res


OPTS = [  # mode, G, gm, affine, relu, scale, center, tail
    ("instance", 0, False, False, True, True, True, None),
    ("instance", 1, True, False, True, True, True, "pool"),
    ("instance", 2, False, False, True, True, False, None),
    ("instance", 2, True, False, False, False, False, None),
    ("instance", 0, True, False, False, True, True, None),
    ("instance", 1, True, True, True, False, False, None),
    ("instance", 2, False, True, True, True, True, "pool"),
    ("instance", 0, True, True, True, False, True, None),
    ("instance", 0, False, False, True, True, True, "head"),
    ("instance", 0, False, False, False, True, True, "head"),
    ("batch", 0, False, False, True, True, True, None),
    ("batch", 1, True, False, True, True, True, None),
    ("batch", 2, True, False, True, True, True, "pool"),
    ("batch", 0, True, False, False, True, False, None),
    ("batch", 2, False, True, True, True, True, None),
    ("batch", 0, False, False, True, True, True, "head"),
]


@pytest.mark.parametrize("mode,G,gm,affine,relu,scale,center,tail", OPTS)
def test_reference_matches_torch_autograd(mode, G, gm, affine, relu, scale, center, tail):
    rng = np.random.default_rng(G + 2 * gm + 4 * affine + 8 * relu + 16 * scale + 32 * center)
    n, h, w, c, classes = 3, 6, 8, 16, 3
    x = _inputs(rng, n, h, w, c, G, classes)
    eps, decay = (1e-6, 0.999) if mode == "instance" else (1e-3, 0.99)
    o = dict(G=G, gm=gm, affine=affine, relu=relu, scale=scale, center=center, tail=tail, decay=decay)
    f = R.forward(x["y"], mode, eps, x["gamma"] if scale else None, x["beta"] if center else None,
                  x["gamma_mod"] if gm else None, x["guide"] if G else None, x["w_guide"] if G else None,
                  x["b_guide"] if G else None, x["ga"] if affine else None, x["ba"] if affine else None, relu,
                  pool=tail == "pool", w_head=x["w_head"] if tail == "head" else None,
                  b_head=x["b_head"] if tail == "head" else None, moving=(x["mm"], x["mv"]), decay=decay)
    b = R.backward(f, da=x["da"], dpooled=x["dpooled"] if tail == "pool" else None,
                   dlogits=x["dlogits"] if tail == "head" else None)
    ref = _torch_layer(x, mode, eps, o)
    g = ref["grads"]
    pairs = [(f["a"], ref["a"]), (b["dy"], g["y"])]
    if tail == "pool":
        pairs.append((f["pooled"], ref["pooled"]))
    if tail == "head":
        pairs += [(f["logits"], ref["logits"]), (b["dw_head"], g["w_head"]), (b["db_head"], g["b_head"])]
    if scale:
        pairs.append((b["dgamma"], g["gamma"]))
    if center:
        pairs.append((b["dbeta"], g["beta"]))
    if gm:
        pairs.append((b["dgamma_mod"], g["gamma_mod"]))
    if G:
        pairs += [(b["dw_guide"], g["w_guide"]), (b["dbias_guide"], g["b_guide"])]
    if affine:
        pairs += [(b["dga"], g["ga"]), (b["dba"], g["ba"])]
    if mode == "batch":
        pairs += [(f["moving_mean"], ref["moving_mean"]), (f["moving_var"], ref["moving_var"])]
    for i, (got, want) in enumerate(pairs):
        assert _rel(got, want) < 1e-10, (i, _rel(got, want))


def test_reference_gamma_and_beta_gradients_without_parameters():
    """With scale / center off, dgamma / dbeta are the gradients of a gamma of one and a beta of zero: what the
    finalisers emit when they are handed the pointers anyway."""
    rng = np.random.default_rng(11)
    x = _inputs(rng, 2, 4, 6, 8, 1, 2)
    f0 = R.forward(x["y"], "instance", 1e-6, None, None, x["gamma_mod"], x["guide"], x["w_guide"], x["b_guide"])
    f1 = R.forward(x["y"], "instance", 1e-6, np.ones(8), np.zeros(8), x["gamma_mod"], x["guide"], x["w_guide"],
                   x["b_guide"])
    b0, b1 = R.backward(f0, da=x["da"]), R.backward(f1, da=x["da"])
    for k in ("dy", "dgamma", "dbeta", "dgamma_mod", "dw_guide", "dbias_guide"):
        assert _rel(b0[k], b1[k]) < 1e-14, k
