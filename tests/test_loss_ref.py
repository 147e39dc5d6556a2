"""Pins the oracle loss functions that tests/test_gpu_loss_ops.py compares the device with (oracle/tf_ops.py:
weighted_sparse_softmax_cross_entropy with its three weightings, sparse_dice_loss and softmax_grad) to an independent
torch float64 restatement: log_softmax, per-pixel weights built from the labels, SUM_BY_NONZERO_WEIGHTS, and autograd
for every gradient. Gate: 1e-12 relative."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import tf_ops as O

TOL = 1e-12


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _inputs(classes, every_class, seed):
    """5 images of 6 x 10 px; logits with per-image, per-class offsets. Unless every class must be present: image 0
    is all background, image 1 lacks one class, image 4 is background with foreground probabilities near 1e-13."""
    rng = np.random.default_rng(seed)
    n, h, w = 5, 6, 10
    logits = rng.standard_normal((n, h, w, classes)) * 2 + rng.normal(0, 1.5, (n, 1, 1, classes))
    labels = rng.integers(0, classes, (n, h, w))
    if every_class:
        labels[:, 0, :classes] = np.arange(classes)
    else:
        labels[0] = 0
        missing = classes - 1 if classes > 2 else 0
        labels[1][labels[1] == missing] = (missing + 1) % classes
        labels[4] = 0
        logits[4, ..., 1:] -= 30.0
    return logits.astype(np.float32).astype(np.float64), labels.astype(np.int32)


def _torch_weights(lab, classes, wtype, numeric_w, decay):
    """Per-pixel weights of loss_metrics._compute_weights, written per pixel from the labels."""
    n, h, w = lab.shape
    if wtype == "none":
        return torch.ones((n, h, w), dtype=torch.float64)
    oh = F.one_hot(lab, classes).to(torch.float64)
    if wtype == "numerical":
        wpx = torch.tensor(numeric_w, dtype=torch.float64)[lab]
    else:
        num = oh.sum(dim=(1, 2))
        if decay > 0:
            num = num + decay
        prop = 1.0 / num
        wc = prop / prop.sum(dim=1, keepdim=True)
        wpx = torch.gather(wc, 1, lab.reshape(n, -1)).reshape(n, h, w)
    return wpx / wpx.sum(dim=(1, 2), keepdim=True) * (h * w)


XENT = [pytest.param(wtype, classes, numeric, decay, id=f"{wtype}{'' if decay is None else decay}-c{classes}")
        for classes in (2, 3, 4)
        for wtype, numeric, decay in (("none", None, None), ("numerical", (0.2, 0.4, 4.4, 1.3)[:classes], None),
                                      ("proportion", None, 0.0), ("proportion", None, 1000.0))]
# a class with numerical weight 0: its pixels leave the SUM_BY_NONZERO_WEIGHTS denominator
XENT.append(pytest.param("numerical", 3, (1.0, 0.0, 3.0), None, id="numerical-zero-weight-c3"))


@pytest.mark.parametrize("wtype,classes,numeric,decay", XENT)
def test_weighted_xent_matches_torch(wtype, classes, numeric, decay):
    # proportion without decay divides by the class count: every class must be in every image
    logits, labels = _inputs(classes, every_class=(decay == 0.0), seed=classes * 10 + len(wtype))
    kw = {}
    if wtype == "numerical":
        kw["numeric_w"] = numeric
    if wtype == "proportion":
        kw["proportion_decay"] = decay
    loss, dl = O.weighted_sparse_softmax_cross_entropy(logits, labels, wtype, **kw)

    x = torch.tensor(logits, requires_grad=True)
    lab = torch.tensor(labels, dtype=torch.int64)
    wt = _torch_weights(lab, classes, wtype, numeric, decay or 0.0)
    ce = -torch.gather(F.log_softmax(x, dim=-1), -1, lab[..., None])[..., 0]
    t_loss = (wt * ce).sum() / (wt != 0).sum()
    t_loss.backward()
    assert np.isfinite(float(loss))
    assert abs(float(loss) - t_loss.item()) <= TOL * abs(t_loss.item())
    assert _rel(dl, x.grad.numpy()) <= TOL


@pytest.mark.parametrize("classes", [2, 3, 4])
def test_dice_loss_and_softmax_grad_match_torch(classes):
    logits, labels = _inputs(classes, every_class=False, seed=classes)
    prob = O.softmax(logits)
    loss, dprob = O.sparse_dice_loss(prob, labels)
    dl = O.softmax_grad(dprob, prob)

    x = torch.tensor(logits, requires_grad=True)
    p = torch.softmax(x, dim=-1)
    p.retain_grad()
    oh = F.one_hot(torch.tensor(labels, dtype=torch.int64), classes).to(torch.float64)[..., 1:]
    inter = (oh * p[..., 1:]).sum(dim=(1, 2, 3))
    union = (oh + p[..., 1:]).sum(dim=(1, 2, 3))
    t_loss = 1.0 - (2.0 * inter / (union + 1e-8)).mean()
    t_loss.backward()
    assert _rel(prob, p.detach().numpy()) <= TOL
    assert abs(float(loss) - t_loss.item()) <= TOL * abs(t_loss.item())
    assert _rel(dprob, p.grad.numpy()) <= TOL
    assert _rel(dl, x.grad.numpy()) <= TOL
    # softmax_grad on its own, with an incoming gradient on every class (the Dice one is zero on class 0)
    g = np.random.default_rng(classes).standard_normal(prob.shape)
    x.grad = None
    torch.softmax(x, dim=-1).backward(torch.tensor(g))
    assert _rel(O.softmax_grad(g, prob), x.grad.numpy()) <= TOL
