"""UNet --without_norm on the CPU: the numpy oracle's forward, loss and hand-derived backward against torch autograd and
against central finite differences (fp64), slim's variable inventory of a normaliser-free graph, and the lowering of
such a graph by bsl_slim to the engine config and the C-ABI call sequence of engine.UNetEngine (traced without a GPU).

Without a normaliser, slim.conv2d keeps its `biases` variable (zeros initializer), adds it and applies ReLU
(tf.contrib.layers.convolution2d with normalizer_fn=None)."""
import numpy as np
import pytest
import torch

from boxsegliver_b200 import bsl_slim as slim
from boxsegliver_b200 import synthetic
from tests import unet_without_norm_ref as R
from tests.fake_ctx import FakeContext
from tests import unet_without_norm_torch as T

tf = slim.tf


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def _random_biases(p, seed):
    """Non-zero biases: a zero bias puts ReLU on its kink wherever a padded input patch is all zero."""
    rng = np.random.default_rng(seed)
    for k in p:
        if k.endswith("/biases"):
            p[k] = rng.normal(0, 0.1, p[k].shape)
    return p


@pytest.mark.parametrize("hw,base,depth,bias_decay,kw", [
    (32, 8, 3, False, dict(loss_type="xentropy", loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4))),
    (32, 8, 3, True, dict(loss_type="xentropy", loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4))),
    (48, 4, 2, False, dict(loss_type="dice", loss_weight_type="none")),
    (48, 4, 2, True, dict(loss_type="xentropy", loss_weight_type="proportion")),
])
def test_forward_loss_and_gradients_match_torch(hw, base, depth, bias_decay, kw):
    cfg = R.UNetCfg(height=hw, width=hw, channel=3, init_channels=base, num_down_samples=depth, weight_decay_rate=1e-3,
                    bias_decay=bias_decay, without_norm=True, **kw)
    params = _random_biases(R.init_params(cfg, seed=3, dtype=np.float64), 4)
    images, labels = synthetic.make_batch(2, hw, hw, 3, seed=11)
    images = images.astype(np.float64)
    tape = R.forward(params, images, cfg, True)
    loss, dl = R.loss_and_dlogits(tape, labels, cfg)
    grads = R.total_grads(params, R.backward(tape, dl, cfg), cfg)
    total = float(loss) + R.regularization_loss(params, cfg)
    assert not tape.new_moving

    tp = T.to_torch_params(params, torch.float64)
    tl, tlogits = T.total_loss(tp, torch.tensor(images).permute(0, 3, 1, 2), torch.tensor(labels, dtype=torch.long), cfg)
    tl.backward()
    assert rel(tape.logits, tlogits.permute(0, 2, 3, 1).detach().numpy()) < 1e-10
    assert abs(total - float(tl.detach())) < 1e-10 * max(1.0, abs(total))
    assert set(grads) == {k for k, t in tp.items() if t.requires_grad}
    for k, g in grads.items():
        assert rel(g, tp[k].grad.numpy()) < 1e-10, k


def test_finite_differences():
    cfg = R.UNetCfg(height=32, width=32, channel=3, init_channels=8, num_down_samples=2, without_norm=True,
                    loss_type="xentropy", loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4),
                    weight_decay_rate=1e-3)
    p = _random_biases(R.init_params(cfg, 0, np.float64), 1)
    rng = np.random.default_rng(2)
    x = rng.uniform(0, 1, (2, 32, 32, 3))
    lab = rng.integers(0, 3, (2, 32, 32)).astype(np.int32)

    def total(q):
        t = R.forward(q, x, cfg, True)
        l, _ = R.loss_and_dlogits(t, lab, cfg)
        return float(l) + R.regularization_loss(q, cfg)

    t = R.forward(p, x, cfg, True)
    _, dl = R.loss_and_dlogits(t, lab, cfg)
    g = R.total_grads(p, R.backward(t, dl, cfg), cfg)
    for k in R.trainable_names(cfg, p):
        for _ in range(2):
            idx = tuple(rng.integers(0, s) for s in p[k].shape)
            # without a normaliser a bias moves every pre-activation of its channel; with 1e-6 one of them (4e-7 from
            # zero at these seeds) crosses the ReLU kink, so the step stays below that
            e = 1e-7
            q = {a: b.copy() for a, b in p.items()}
            q[k][idx] += e
            lp = total(q)
            q[k][idx] -= 2 * e
            lm = total(q)
            fd, an = (lp - lm) / (2 * e), g[k][idx]
            assert abs(fd - an) <= 1e-4 * (abs(fd) + abs(an)) + 1e-9, (k, idx, fd, an)


def test_training_and_eval_forwards_are_identical():
    cfg = R.UNetCfg(height=16, width=16, channel=3, init_channels=8, num_down_samples=2, without_norm=True)
    p = _random_biases(R.init_params(cfg, 5, np.float64), 6)
    x, _ = synthetic.make_batch(2, 16, 16, 3, seed=3)
    a = R.forward(p, x.astype(np.float64), cfg, True).logits
    b = R.forward(p, x.astype(np.float64), cfg, False).logits
    assert np.array_equal(a, b)


# ------------------------------------------------------------------ slim's variable inventory (scoping rules alone)
def without_norm_variable_names(num_down_samples=4):
    """slim names of UNet --without_norm: every conv2d (normalizer_fn=None) has weights and biases."""
    names = []
    for i in range(1, num_down_samples + 1):
        for j in (1, 2):
            names += [f"UNet/Encode{i}/Repeat/convolution2d_{j}/{v}" for v in ("weights", "biases")]
    for j in (1, 2):
        names += [f"UNet/ED-Bridge/ED-Bridge_{j}/{v}" for v in ("weights", "biases")]
    for i in range(num_down_samples, 0, -1):
        names += [f"UNet/Decode{i}/Conv2d_transpose/{v}" for v in ("weights", "biases")]
        for j in (1, 2):
            names += [f"UNet/Decode{i}/Repeat/convolution2d_{j}/{v}" for v in ("weights", "biases")]
    names += ["UNet/AdjustChannels/weights", "UNet/AdjustChannels/biases"]
    return names


@pytest.mark.parametrize("bias_decay", [False, True])
def test_variable_inventory_follows_slim(bias_decay):
    depth = 3
    cfg = R.UNetCfg(height=32, width=32, init_channels=8, num_down_samples=depth, without_norm=True, bias_decay=bias_decay)
    p = R.init_params(cfg, 0)
    assert list(p) == without_norm_variable_names(depth)
    assert not any("BatchNorm" in k or "InstanceNorm" in k for k in p)
    assert all(not p[k].any() for k in p if k.endswith("/biases"))
    regs = set(R.regularized_names(cfg, p))
    assert regs == {k for k in p if k.endswith("/weights") or (k.endswith("/biases") and not bias_decay)}
    # the engine's plan: the same variables, biases in the L2-regularised region unless --bias_decay
    from boxsegliver_b200.engine import EngineConfig, UNetEngine
    ecfg = EngineConfig(batch=1, height=32, width=32, init_channels=64, num_down_samples=depth, without_norm=True,
                        bias_decay=bias_decay, training=False)
    eng = _engine(UNetEngine, ecfg)
    names = without_norm_variable_names(depth)
    assert set(eng.params) == set(names)
    for k, prm in eng.params.items():
        assert prm.region == ("A" if k.endswith("/weights") or not bias_decay else "B"), k
    assert eng.n_stats == 0


# ------------------------------------------------------------------ bsl_slim lowering, traced without a device
def _engine(cls, cfg):
    return cls(FakeContext(), cfg)


def build_unet(images, num_classes, norm_fn=None, norm_params=None, plain_scope=None, weight_decay_rate=1e-5,
               bias_decay=False, num_down_samples=3, name="UNet"):
    """UNet._net_arg_scope + UNet._build_network (UNet.py:41-100) with `slim` / `tf` bound to bsl_slim; norm_fn=None
    is --without_norm. `plain_scope`: that one block's convolutions get no normaliser (a mixed graph)."""
    w_reg = slim.l2_regularizer(weight_decay_rate) if weight_decay_rate > 0 else None
    b_reg = None if bias_decay else w_reg
    layers = {}
    with slim.arg_scope([slim.conv2d, slim.conv2d_transpose], weights_regularizer=w_reg,
                        weights_initializer=slim.xavier_initializer(), biases_regularizer=b_reg):
        with slim.arg_scope([slim.conv2d], normalizer_fn=norm_fn, normalizer_params=norm_params):
            out_channels = 64
            x = images
            with tf.variable_scope(name, "UNet"):
                for i in range(num_down_samples):
                    with tf.variable_scope("Encode{:d}".format(i + 1)):
                        if plain_scope == f"Encode{i + 1}":
                            with slim.arg_scope([slim.conv2d], normalizer_fn=None, normalizer_params=None):
                                x = slim.repeat(x, 2, slim.conv2d, out_channels, 3)
                        else:
                            x = slim.repeat(x, 2, slim.conv2d, out_channels, 3)
                        layers[i + 1] = x
                        x = slim.max_pool2d(x, [2, 2])
                    out_channels *= 2
                x = slim.repeat(x, 2, slim.conv2d, out_channels, 3, scope="ED-Bridge")
                for i in reversed(range(num_down_samples)):
                    out_channels //= 2
                    with tf.variable_scope("Decode{:d}".format(i + 1)):
                        x = slim.conv2d_transpose(x, x.get_shape()[-1] // 2, 2, 2)
                        x = tf.concat((layers[i + 1], x), axis=-1)
                        x = slim.repeat(x, 2, slim.conv2d, out_channels, 3)
                with slim.arg_scope([slim.conv2d], activation_fn=None, normalizer_fn=None, normalizer_params=None):
                    return slim.conv2d(x, num_classes, 1, scope="AdjustChannels")


def _step_trace(eng):
    eng.ctx.trace = []
    eng.train_step(1e-3, with_metrics=True)
    return eng.ctx.trace


@pytest.mark.parametrize("bias_decay", [False, True])
def test_lowered_graph_gives_the_engine_config_and_call_sequence(bias_decay):
    from boxsegliver_b200.engine import EngineConfig, UNetEngine
    n, hw, depth = 2, 64, 3
    classes = ("Background", "Liver", "Tumor")
    with slim.graph_as_default() as g:
        logits = build_unet(slim.placeholder((n, hw, hw, 3)), 3, bias_decay=bias_decay, num_down_samples=depth)
        table, info = slim.lower_to_layer_table(g, logits)
        geng = slim.lower(g, logits, FakeContext(), classes)
    assert info["normalizer"] is None and info["num_down_samples"] == depth
    names = set()
    for L in table:
        names |= {L["scope"] + "/weights", L["scope"] + "/biases"}
    assert names == set(without_norm_variable_names(depth))
    cfg = EngineConfig(batch=n, height=hw, width=hw, num_down_samples=depth, weight_decay_rate=1e-5,
                       bias_decay=bias_decay, without_norm=True)
    assert geng.cfg == cfg
    ref = _engine(UNetEngine, cfg)
    assert set(geng.params) == set(ref.params) and geng.n_reg == ref.n_reg and geng.n_train == ref.n_train
    trace = _step_trace(ref)
    assert _step_trace(geng) == trace

    # forward: conv epilogue + pool per encoder block, no normalisation pass, plain logits layer
    fwd = trace[:trace.index("bsl_softmax_threshold")]
    expect = []
    for L in ref.layers:
        if L.kind == "stem":
            expect += ["bsl_stem_im2col_ld", "bsl_conv2d_fprop_bias_relu"]
        elif L.kind == "conv":
            expect += ["bsl_conv2d_fprop_bias_relu"] + (["bsl_maxpool2x2_bf16"] if L.role == "enc2" else [])
        elif L.kind == "convT":
            expect += ["bsl_convT2d_fwd"]
        else:
            expect += ["bsl_conv2d_head_fprop"]
    assert fwd == expect
    assert not [c for c in trace if "norm" in c]
    n_conv = 4 * depth + 2
    assert trace.count("bsl_relu_bwd_bias") == n_conv + depth      # every 3x3 conv and every transposed conv
    assert trace.count("bsl_maxpool2x2_bwd_add") == depth
    assert trace.count("bsl_conv2d_head_dgrad") == 1
    assert trace.count("bsl_conv2d_wgrad") == n_conv and trace.count("bsl_conv2d_dgrad") == n_conv - 1


def test_normalised_engine_plan_is_unchanged_by_the_flag_default():
    from boxsegliver_b200.engine import EngineConfig, UNetEngine
    cfg = EngineConfig(batch=2, height=64, width=64, num_down_samples=3)
    eng = _engine(UNetEngine, cfg)
    assert not cfg.without_norm
    assert all(L.y is not None for L in eng.layers if L.kind in ("stem", "conv"))
    assert not any(k.endswith("/biases") for k in eng.params if "convolution2d" in k or "ED-Bridge" in k)


def test_mixed_graph_is_rejected():
    with slim.graph_as_default() as g:
        logits = build_unet(slim.placeholder((1, 64, 64, 3)), 3, norm_fn=slim.batch_norm,
                            norm_params={"scale": True, "is_training": True}, plain_scope="Encode2")
        with pytest.raises(NotImplementedError, match="mixed normalisers"):
            slim.lower_to_layer_table(g, logits)


def test_plain_conv_without_bias_is_rejected():
    with slim.graph_as_default() as g:
        x = slim.placeholder((1, 32, 32, 3))
        y = slim.conv2d(x, 64, 3, biases_initializer=None)
        with pytest.raises(NotImplementedError, match="conv \\+ bias \\+ ReLU"):
            slim.lower_to_layer_table(g, y)


def test_gunet_and_unetinter_engines_still_raise():
    from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine, UNetInterConfig, UNetInterEngine
    with pytest.raises(NotImplementedError, match="without_norm"):
        GUNetEngine(FakeContext(), GUNetConfig(batch=1, height=64, width=64, without_norm=True))
    with pytest.raises(NotImplementedError, match="without_norm"):
        UNetInterEngine(FakeContext(), UNetInterConfig(batch=1, height=64, width=64, without_norm=True))
