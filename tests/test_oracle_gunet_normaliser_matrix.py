"""Pins oracle/gunet_ref.py (CPU only) on the cells of GUNet's normaliser matrix that combine batch norm, after_affine
and the backbone --dropout (/root/reference/NetworksV2/GUNet.py:162-217, modulated_conv_block): an independent torch-CPU
autograd implementation must give the same logits, loss, gradients and moving statistics in fp64."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import gunet_ref as G
from oracle import tf_ops as O


def _inputs(cfg, n, rng):
    images = rng.uniform(0, 1, (n, cfg.height, cfg.width, cfg.channel))
    context = np.abs(rng.normal(0, 1, (n, cfg.context_dim)))
    context[0, cfg.context_dim // 2:] = 0.0           # tumour-free slice: second histogram all zero
    guide = 0.5 + 0.5 * rng.uniform(0, 1, (n, cfg.height, cfg.width, cfg.guide_channel))
    labels = rng.integers(0, cfg.num_classes, (n, cfg.height, cfg.width)).astype(np.int32)
    return dict(images=images, context=context, sp_guide=guide), labels


def _torch_gunet(params, inputs, labels, cfg, mults):
    """Independent implementation: NCHW torch functional ops + autograd."""
    P = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params.items() if "/moving_" not in k}
    t = lambda a: torch.tensor(a, dtype=torch.float64)
    x = t(inputs["images"]).permute(0, 3, 1, 2)
    if getattr(cfg, "img_grad", False) and cfg.prefix == "GUNet":     # tf.image.image_gradients: forward differences
        dy = F.pad(x[:, :, 1:] - x[:, :, :-1], (0, 0, 0, 1))
        dx = F.pad(x[:, :, :, 1:] - x[:, :, :, :-1], (0, 1))
        x = torch.cat((x, dy, dx), dim=1)
    ctxp = None
    if cfg.use_context:
        h = t(inputs["context"])
        fcs = G.fc_specs(cfg)
        for k, (sc, _, _, hidden) in enumerate(fcs):
            h = h @ P[f"{sc}/weights"] + P[f"{sc}/biases"]
            if hidden:
                h = torch.relu(h)
                if mults is not None:
                    h = h * t(mults[k])
        ctxp = h
    guides = []
    if cfg.use_spatial:
        g = t(inputs["sp_guide"]).permute(0, 3, 1, 2)
        for i in range(cfg.num_down_samples + 1):
            guides.append(g)
            g = F.avg_pool2d(g, 2)

    def conv(x, s):
        sc, co = s["scope"], s["cout"]
        y = F.conv2d(x, P[f"{sc}/weights"].permute(3, 2, 0, 1), padding=1)
        if cfg.normalizer == "batch_norm":
            y = F.batch_norm(y, None, None, weight=P[f"{sc}/BatchNorm/gamma"] if s["scale"] else None,
                             bias=P[f"{sc}/BatchNorm/beta"] if s["center"] else None, training=True, eps=cfg.bn_eps)
        else:
            y = F.instance_norm(y, weight=P[f"{sc}/InstanceNorm/gamma"] if s["scale"] else None,
                                bias=P[f"{sc}/InstanceNorm/beta"] if s["center"] else None, eps=cfg.in_eps)
        if getattr(cfg, "_drop_mults", None) and s.get("drop") and s["scope"] in cfg._drop_mults:
            y = y * t(cfg._drop_mults[s["scope"]]).permute(0, 3, 1, 2)
        if s["mod_off"] is not None:
            y = y * ctxp[:, s["mod_off"]:s["mod_off"] + co][:, :, None, None]
        if s["sp_off"] is not None:
            ssc = f"GUNet/spatial/conv{s['level'] + 1}"
            full = F.conv2d(guides[s["level"]], P[f"{ssc}/weights"].permute(3, 2, 0, 1), P[f"{ssc}/biases"])
            y = y + full[:, s["sp_off"]:s["sp_off"] + co]
        if s.get("affine"):
            y = y * P[f"{s['affine']}/gamma"][None, :, None, None] + P[f"{s['affine']}/beta"][None, :, None, None]
        return torch.relu(y)

    it = iter(G.layer_specs(cfg))
    skips = []
    for i in range(cfg.num_down_samples + 1):
        x = conv(conv(x, next(it)), next(it))
        if i < cfg.num_down_samples:
            skips.append(x)
            if getattr(cfg, "mid_cat", False) and i == 0:
                x = torch.cat((x, t(inputs["sp_guide"]).permute(0, 3, 1, 2)), dim=1)
            x = F.max_pool2d(x, 2)
    for i in reversed(range(cfg.num_down_samples)):
        s = next(it)
        up = torch.relu(F.conv_transpose2d(x, P[f"{s['scope']}/weights"].permute(3, 2, 0, 1), P[f"{s['scope']}/biases"],
                                           stride=2))
        x = torch.cat((skips[i], up), dim=1)
        x = conv(conv(x, next(it)), next(it))
    s = next(it)
    logits = F.conv2d(x, P[f"{s['scope']}/weights"].permute(3, 2, 0, 1), P[f"{s['scope']}/biases"])
    lab = torch.tensor(labels, dtype=torch.long)
    loss = 0.0
    if "xentropy" in cfg.loss_type:
        assert cfg.loss_weight_type == "numerical"
        oh = F.one_hot(lab, cfg.num_classes).double()
        w = (oh * t(np.array(cfg.loss_numeric_w))).sum(-1)
        w = w / w.sum(dim=(1, 2), keepdim=True) * (cfg.height * cfg.width)
        ce = F.cross_entropy(logits, lab, reduction="none")
        loss = loss + (w * ce).sum() / (w != 0).sum()
    if "dice" in cfg.loss_type:
        prob = torch.softmax(logits, dim=1)[:, 1:]
        oh = F.one_hot(lab, cfg.num_classes).double().permute(0, 3, 1, 2)[:, 1:]
        inter = (oh * prob).sum(dim=(1, 2, 3))
        union = (oh + prob).sum(dim=(1, 2, 3))
        loss = loss + 1.0 - (2.0 * inter / (union + 1e-8)).mean()
    loss.backward()
    return logits.detach().permute(0, 2, 3, 1).numpy(), float(loss), {k: v.grad.numpy() for k, v in P.items()}


_SMALL = dict(height=16, width=16, init_channels=4, num_down_samples=2, context_fc_channels=(12, 10), context_dim=20,
              loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4), weight_decay_rate=0.0, dropout_seed=5)


@pytest.mark.parametrize("kw", [
    # batch norm + after_affine (ext_config/GUNet_BOTH_AA.yml with the default normaliser)
    dict(normalizer="batch_norm", after_affine=True, use_context=True, use_spatial=True, guide_channel=1,
         norm_with_center=True, norm_with_scale=True, loss_type="xentropy+dice"),
    # context only; blocks 1 and 2 un-modulated with their own centre / scale and the affine
    dict(normalizer="batch_norm", after_affine=True, use_context=True, use_spatial=False, side_dropout=0.0,
         mod_layers=(0, 1), loss_type="xentropy"),
    # batch norm + --dropout
    dict(normalizer="batch_norm", dropout=0.5, use_context=True, use_spatial=True, guide_channel=1,
         loss_type="xentropy+dice"),
    # batch norm + --dropout + after_affine, two guide channels
    dict(normalizer="batch_norm", dropout=0.25, after_affine=True, use_context=True, use_spatial=True, guide_channel=2,
         norm_with_scale=True, loss_type="xentropy"),
    # instance norm + --dropout + after_affine
    dict(normalizer="instance_norm", dropout=0.5, after_affine=True, use_context=True, use_spatial=True, guide_channel=1,
         loss_type="xentropy+dice"),
])
def test_normaliser_matrix_oracle_matches_torch_autograd(kw):
    cfg = G.GUNetCfg(mod_layers=kw.pop("mod_layers", (1, 2)), **_SMALL, **kw)
    rng = np.random.default_rng(12)
    n = 3
    inputs, labels = _inputs(cfg, n, rng)
    params = {k: v.astype(np.float64) + (0.1 * rng.standard_normal(v.shape) if k.endswith(("beta", "gamma", "biases")) else 0)
              for k, v in G.init_params(cfg, seed=1, dtype=np.float64).items()}
    tape = G.forward(params, inputs, cfg, True, step=2)
    loss, dl = G.loss_and_dlogits(tape, labels, cfg)
    grads = G.backward(tape, dl, cfg)
    drops = {L["spec"]["scope"]: L["mult"] for L in tape.layers if L.get("mult") is not None}
    if cfg.dropout:       # the first conv of every encoder block, the bridge included
        assert sorted(drops) == [f"GUNet/Encode/down_conv{i + 1}/mod_conv1/Conv" for i in range(cfg.num_down_samples + 1)]
        for m in drops.values():
            assert set(np.unique(m)) == {0.0, np.float64(np.float32(1 / (1 - cfg.dropout)))}
        cfg._drop_mults = drops
    else:
        assert not drops
    mults = [f["mult"] if f["mult"] is not None else np.ones_like(f["pre"]) for f in tape.fc] if cfg.use_context else None
    t_logits, t_loss, t_grads = _torch_gunet(params, inputs, labels, cfg, mults)
    assert np.allclose(tape.logits, t_logits, rtol=1e-9, atol=1e-10)
    assert abs(loss - t_loss) < 1e-10
    assert set(grads) == {k for k in params if "/moving_" not in k}
    for k, g in grads.items():
        assert np.allclose(g, t_grads[k], rtol=1e-7, atol=1e-10), k
    if cfg.after_affine:
        assert any("ChannelWiseAffine" in k for k in grads)
    if cfg.normalizer == "batch_norm":
        assert set(tape.new_moving) == {k for k in params if "/moving_" in k}
        # moving statistics from the normaliser's batch moments (ahead of the dropout and the affine): decay 0.99 on the
        # modulated blocks, 0.999 on the un-modulated ones
        for L in tape.layers:
            if L["kind"] != "conv":
                continue
            s = L["spec"]
            y = O.conv2d(L["x"], L["w"])
            decay = 0.99 if s["mod"] else 0.999
            assert np.allclose(tape.new_moving[f"{s['scope']}/BatchNorm/moving_mean"],
                               params[f"{s['scope']}/BatchNorm/moving_mean"] * decay + y.mean(axis=(0, 1, 2)) * (1 - decay),
                               rtol=1e-9, atol=1e-12), s["scope"]
    # inference: moving statistics, no mask
    inf = G.forward(params, inputs, cfg, False)
    assert all(L.get("mult") is None for L in inf.layers) and not inf.new_moving


def test_batch_norm_after_affine_parameter_inventory():
    """after_affine under batch norm: ChannelWiseAffine/{gamma,beta} next to BatchNorm/{gamma,beta,moving_mean,
    moving_variance} of every encoder conv; the modulated blocks' normaliser loses centre and scale (GUNet.py:318-319);
    the affine variables are not regularised."""
    cfg = G.GUNetCfg(height=32, width=32, normalizer="batch_norm", after_affine=True, norm_with_scale=True, dropout=0.5)
    p = G.init_params(cfg)
    for i in range(cfg.num_down_samples + 1):
        for j in (1, 2):
            base = f"GUNet/Encode/down_conv{i + 1}/mod_conv{j}"
            assert f"{base}/ChannelWiseAffine/gamma" in p and f"{base}/ChannelWiseAffine/beta" in p
            assert f"{base}/Conv/BatchNorm/moving_mean" in p and f"{base}/Conv/BatchNorm/moving_variance" in p
            mod = i in cfg.mod_layers
            assert (f"{base}/Conv/BatchNorm/gamma" in p) == (not mod)
            assert (f"{base}/Conv/BatchNorm/beta" in p) == (not mod)
    assert not any("InstanceNorm" in k for k in p)
    assert not any("Decode" in k and "ChannelWiseAffine" in k for k in p)
    reg = G.regularized_names(cfg, p)
    assert not any("ChannelWiseAffine" in k or "BatchNorm" in k for k in reg)
    assert "GUNet/Encode/down_conv1/mod_conv1/Conv/weights" in reg
