"""Pins the UNet3D batch-norm oracle (tests/unet3d_bn_ref.py) against an independent torch-CPU fp64 autograd restatement
(F.batch_norm in training mode, momentum = 1 - decay): logits, loss, every gradient and both moving statistics."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import tf_ops as O
from tests import unet3d_bn_ref as B


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _torch_unet3d_bn(params, inputs, labels, cfg):
    train = {k: v for k, v in params.items() if not k.endswith(("moving_mean", "moving_variance"))}
    P = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in train.items()}
    moving = {k: torch.tensor(v, dtype=torch.float64) for k, v in params.items() if k not in train}
    t = lambda a: torch.tensor(a, dtype=torch.float64)  # noqa: E731
    x = t(inputs["images"])
    if cfg.use_spatial:
        x = torch.cat((x, t(inputs["sp_guide"])), dim=-1)
    x = x.permute(0, 4, 1, 2, 3)
    skips = {}
    for s in B.layer_specs(cfg):
        sc = s["scope"]
        if s["kind"] == "conv":
            pads = [O.same_pads(x.shape[2 + i], s["k"][i], s["s"][i]) for i in range(3)]
            xp = F.pad(x, (pads[2][1], pads[2][2], pads[1][1], pads[1][2], pads[0][1], pads[0][2]))
            y = F.conv3d(xp, P[f"{sc}/weights"].permute(4, 3, 0, 1, 2), stride=s["s"])
            ns = f"{sc}/BatchNorm"
            y = F.batch_norm(y, moving[f"{ns}/moving_mean"], moving[f"{ns}/moving_variance"], weight=P[f"{ns}/gamma"],
                             bias=P[f"{ns}/beta"], training=True, momentum=1.0 - cfg.bn_decay, eps=cfg.bn_eps)
            x = torch.relu(y)
            if s["layer"] == "conv2" and s["block"].startswith("conv_e"):
                skips[s["block"]] = x
        elif s["kind"] == "convT":
            up = torch.relu(F.conv_transpose3d(x, P[f"{sc}/weights"].permute(4, 3, 0, 1, 2), stride=s["s"]))
            x = torch.cat((skips[s["block"].replace("d", "e")], up), dim=1)
        else:
            logits = F.conv3d(x, P[f"{sc}/weights"].permute(4, 3, 0, 1, 2), P[f"{sc}/biases"])
    lab = torch.tensor(labels, dtype=torch.long)
    oh = F.one_hot(lab, cfg.num_classes).double()
    w = (oh * t(np.array(cfg.loss_numeric_w))).sum(-1)
    w = w / w.sum(dim=(1, 2, 3), keepdim=True) * float(np.prod(labels.shape[1:]))
    ce = F.cross_entropy(logits, lab, reduction="none")
    loss = (w * ce).sum() / (w != 0).sum()
    loss.backward()
    return (logits.detach().permute(0, 2, 3, 4, 1).numpy(), float(loss.detach()), {k: v.grad.numpy() for k, v in P.items()},
            {k: v.numpy() for k, v in moving.items()})


@pytest.mark.parametrize("pools,use_spatial,depth", [(4, False, 4), (4, True, 2), (5, False, 2), (5, True, 2)])
def test_batch_norm_oracle_matches_torch_autograd(pools, use_spatial, depth):
    hw = 16 * 2 ** (pools - 4) * 2
    cfg = B.UNet3DBNCfg(depth=depth, height=hw, width=hw, channel=1, init_channels=3, max_channels=20,
                        num_pool_layers=pools, use_spatial=use_spatial, loss_numeric_w=(1.0, 10.0), weight_decay_rate=0.0)
    rng = np.random.default_rng(pools + depth)
    n = 2
    inputs = dict(images=rng.standard_normal((n, depth, hw, hw, 1)))
    if use_spatial:
        inputs["sp_guide"] = rng.uniform(0, 1, (n, depth, hw, hw, 2))
    labels = rng.integers(0, 2, (n, depth, hw, hw)).astype(np.int32)
    params = B.init_params(cfg, seed=2, dtype=np.float64)
    for k, v in params.items():
        if k.endswith(("beta", "gamma", "biases", "moving_mean")):
            params[k] = v + 0.1 * rng.standard_normal(v.shape)
        elif k.endswith("moving_variance"):
            params[k] = v + 0.1 * rng.uniform(0, 1, v.shape)
    tape = B.forward(params, inputs, cfg, is_training=True)
    loss, dl = B.loss_and_dlogits(tape, labels, cfg)
    grads = B.backward(tape, dl, cfg)
    t_logits, t_loss, t_grads, t_moving = _torch_unet3d_bn(params, inputs, labels, cfg)
    assert _rel(tape.logits, t_logits) <= 1e-10
    assert abs(loss - t_loss) <= 1e-10 * abs(t_loss)
    assert set(grads) == set(t_grads) and set(tape.moving) == set(t_moving) == set(B.moving_names(params))
    for k, g in grads.items():
        assert _rel(g, t_grads[k]) <= 1e-10, k
    for k, m in tape.moving.items():
        assert _rel(m, t_moving[k]) <= 1e-10, k


def test_batch_norm_variables_and_eval_mode():
    cfg = B.UNet3DBNCfg(depth=2, height=32, width=32, init_channels=3, max_channels=20)
    params = B.init_params(cfg, seed=0)
    norm = [k for k in params if "/BatchNorm/" in k]
    assert len(norm) == 18 * 4 and not any("InstanceNorm" in k for k in params)
    assert all(np.all(params[k] == 0) for k in norm if k.endswith("moving_mean"))
    assert all(np.all(params[k] == 1) for k in norm if k.endswith("moving_variance"))
    # same random stream as the instance-norm oracle: the filters are identical
    from oracle import unet3d_ref as U
    p_in = U.init_params(U.UNet3DCfg(depth=2, height=32, width=32, init_channels=3, max_channels=20), seed=0)
    assert all(np.array_equal(params[k], v) for k, v in p_in.items() if k.endswith("/weights"))
    # eval mode normalises with the moving statistics and reports no update
    rng = np.random.default_rng(0)
    inputs = dict(images=rng.standard_normal((1, 2, 32, 32, 1)))
    tape = B.forward(params, inputs, cfg, is_training=False)
    assert tape.moving == {} and np.isfinite(tape.logits).all()
    first = tape.layers[0]
    y = O.conv3d(inputs["images"], params["UNet3D/conv_e0/conv1/weights"])
    assert np.allclose(first["z"], y / np.sqrt(1.0 + cfg.bn_eps))
