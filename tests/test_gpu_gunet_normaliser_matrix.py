"""GUNet's normaliser matrix on the device: batch norm with after_affine, batch norm with the backbone --dropout, both
together, and instance norm with --dropout and after_affine (/root/reference/NetworksV2/GUNet.py:162-217,
modulated_conv_block), one training step against oracle/gunet_ref.py through the C ABI, the eval forward behind
inference.Predictor, ten training steps, and a checkpoint round trip.

Gates are those of test_gpu_gunet.py's train-step parity: every layer on the device's stored input <= 1e-2,
tests/gpu_util.gate_gradients on the oracle backward over the stored tape, moving statistics <= 1e-4, loss 1e-4 relative,
dlogits <= 1e-5, context-MLP gradients op by op <= 1e-4."""
import numpy as np
import pytest

from boxsegliver_b200 import checkpoint as K
from boxsegliver_b200 import synthetic
from boxsegliver_b200.device import round_bf16
from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine
from boxsegliver_b200.inference import Predictor
from oracle import gunet_ref as G
from tests.gpu_util import gate_gradients, rel, report

pytestmark = pytest.mark.gpu


def _make(n, hw, **kw):
    base = dict(height=hw, width=hw, channel=3, init_channels=64, num_down_samples=4, weight_decay_rate=1e-5,
                loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4), dropout_seed=21)
    base.update(kw)
    ecfg = GUNetConfig(batch=n, **base)
    rcfg = G.GUNetCfg(**base)
    images, labels = synthetic.make_batch(n, hw, hw, 3, seed=1360 + n)
    context, guide = synthetic.make_guides(images, labels, rcfg.context_dim, rcfg.guide_channel, seed=5)
    return ecfg, rcfg, dict(images=images, context=context, sp_guide=guide), labels


def _params(rcfg, seed=4):
    params = G.init_params(rcfg, seed=seed)
    rng = np.random.default_rng(2)
    for k in params:                      # non-trivial affine / bias / moving values so every term is exercised
        if k.endswith(("beta", "biases", "moving_mean")):
            params[k] = (0.1 * rng.standard_normal(params[k].shape)).astype(np.float32)
        if k.endswith(("gamma", "moving_variance")):
            params[k] = (1 + 0.1 * rng.standard_normal(params[k].shape)).astype(np.float32)
    return params


def _engine(ctx, ecfg, params, inputs, labels):
    eng = GUNetEngine(ctx, ecfg)
    assert set(eng.params) == set(params)
    eng.set_weights(params)
    eng.set_inputs(inputs["images"], labels)
    eng.set_guides(inputs.get("context"), inputs.get("sp_guide"))
    return eng


def _f64(d):
    return {k: v.astype(np.float64) for k, v in d.items()}


CASES = [
    # batch norm + after_affine: ext_config/GUNet_BOTH_AA.yml with the default normaliser
    (2, 64, dict(normalizer="batch_norm", after_affine=True, use_context=True, use_spatial=True, guide_channel=1,
                 norm_with_center=True, norm_with_scale=True, context_fc_channels=(200, 200), loss_type="xentropy+dice")),
    # context only; blocks 2..4 un-modulated: per-channel batch-norm scalars with the folded affine
    (2, 64, dict(normalizer="batch_norm", after_affine=True, use_context=True, use_spatial=False, mod_layers=(0, 1),
                 loss_type="xentropy")),
    # 96 x 96: ragged 6 x 6 / 12 x 12 deep levels
    (3, 96, dict(normalizer="batch_norm", after_affine=True, use_context=True, use_spatial=True, guide_channel=2,
                 loss_type="xentropy")),
    # batch norm + --dropout
    (2, 64, dict(normalizer="batch_norm", dropout=0.5, use_context=True, use_spatial=True, guide_channel=1,
                 loss_type="xentropy+dice")),
    # batch norm + --dropout + after_affine, two guide channels
    (2, 64, dict(normalizer="batch_norm", dropout=0.5, after_affine=True, use_context=True, use_spatial=True,
                 guide_channel=2, norm_with_scale=True, loss_type="xentropy")),
    # instance norm + --dropout + after_affine
    (2, 64, dict(normalizer="instance_norm", dropout=0.5, after_affine=True, use_context=True, use_spatial=True,
                 guide_channel=1, loss_type="xentropy+dice")),
]


@pytest.mark.parametrize("n,hw,kw", CASES)
def test_gunet_normaliser_matrix_train_step_parity(ctx, n, hw, kw):
    ecfg, rcfg, inputs, labels = _make(n, hw, **kw)
    params = _params(rcfg)
    eng = _engine(ctx, ecfg, params, inputs, labels)
    eng.forward(True)
    eng.predict_outputs(True)
    eng.loss_backward()
    ctx.check_device()
    k = rcfg.num_classes
    logits = eng.logits.download(np.float32, (n, hw, hw, k))
    dlogits = eng.dlogits.download(np.float32, (n, hw, hw, k))
    grads = eng.get_grads()
    stored = eng.get_stored_forward()
    stored["logits"] = logits
    ctxp = eng.get_context_params()
    dctx = eng.get_context_grad()
    eng.optimizer_step(1e-3)
    ctx.check_device()
    data_loss, reg_loss = eng.read_loss()
    new_w = eng.get_weights()
    eng.close()

    rin = dict(inputs, images=round_bf16(inputs["images"]))
    tft = G.forward(_f64(params), _f64(rin), rcfg, True, wrnd=round_bf16, stored=stored, step=1)
    assert max(tft.errs.values()) < 1e-2, max(tft.errs.items(), key=lambda t: t[1])
    assert rel(ctxp, tft.ctx_params) < 1e-5
    if rcfg.dropout:        # the oracle's multipliers mask the first conv of every encoder block, the bridge included
        dropped = [L for L in tft.layers if L.get("mult") is not None]
        assert [L["spec"]["scope"] for L in dropped] == \
            [f"GUNet/Encode/down_conv{i + 1}/mod_conv1/Conv" for i in range(rcfg.num_down_samples + 1)]
        assert all((L["mult"] == 0).any() for L in dropped)
    loss_o, dl = G.loss_and_dlogits(tft, labels, rcfg)
    assert abs(data_loss - loss_o) < 1e-4 * abs(loss_o)
    assert abs(reg_loss - G.regularization_loss(params, rcfg)) < 1e-6
    assert rel(dlogits, dl) < 1e-5
    assert set(tft.new_moving) == {k_ for k_ in params if "/moving_" in k_}
    for name, v in tft.new_moving.items():     # decay 0.99 on the modulated blocks, 0.999 elsewhere
        assert rel(new_w[name], v) < 1e-4, name
    g_ref = G.backward(tft, dl, rcfg, rnd=round_bf16)
    assert set(g_ref) == set(grads)
    if rcfg.after_affine:
        assert any("ChannelWiseAffine" in name for name in g_ref)
    errs = {name: rel(grads[name], g) for name, g in g_ref.items() if "/context/" not in name}
    e_fc_end_to_end = max(rel(grads[name], g) for name, g in g_ref.items() if "/context/" in name)
    for s_ in G.layer_specs(rcfg):
        if s_.get("mod_off") is not None:
            sl = slice(s_["mod_off"], s_["mod_off"] + s_["cout"])
            errs[f"{s_['scope']}/d_gamma_mod"] = rel(dctx[:, sl], tft.dctx[:, sl])
    for name, g in G.fc_backward(tft, dctx.astype(np.float64)).items():
        assert rel(grads[name], g) < 1e-4, name
    worst = max(errs.items(), key=lambda t: t[1])
    report("gunet normaliser matrix step", layer_worst=max(tft.errs.values()),
           grad_median=float(np.median(list(errs.values()))), grad_worst=worst[1], grad_worst_name=worst[0],
           fc_grads_end_to_end=e_fc_end_to_end)
    gate_gradients(errs)
    assert e_fc_end_to_end < 3e-2


@pytest.mark.parametrize("kw", [
    dict(after_affine=True),
    dict(after_affine=True, dropout=0.5, guide_channel=2),
])
def test_gunet_batch_norm_eval_forward_after_training(ctx, kw):
    """forward(False) after a training step: moving statistics, no mask, the affine folded; the argmax of
    inference.Predictor equals np.argmax of the oracle's probabilities."""
    n, hw = 2, 64
    ecfg, rcfg, inputs, labels = _make(n, hw, normalizer="batch_norm", use_context=True, use_spatial=True,
                                       loss_type="xentropy", **kw)
    eng = _engine(ctx, ecfg, _params(rcfg), inputs, labels)
    eng.train_step(1e-3)
    ctx.check_device()
    trained = eng.get_weights()
    s0 = eng.S.download(np.uint32, (eng.n_stats,))
    eng.forward(False)
    eng.predict_outputs(False)
    ctx.check_device()
    assert np.array_equal(eng.S.download(np.uint32, (eng.n_stats,)), s0), "an eval forward moved the moving statistics"
    stored = eng.get_stored_forward()
    stored["logits"] = eng.logits.download(np.float32, (n, hw, hw, rcfg.num_classes))
    pr = Predictor(eng)
    pred = pr.predict(inputs["images"], inputs["context"], inputs["sp_guide"])
    ctx.check_device()
    pr.close()
    eng.close()
    rin = _f64(dict(inputs, images=round_bf16(inputs["images"])))
    tape = G.forward(_f64(trained), rin, rcfg, False, wrnd=round_bf16, stored=stored)
    assert max(tape.errs.values()) < 1e-2, max(tape.errs.items(), key=lambda t: t[1])
    assert all(L.get("mult") is None for L in tape.layers)
    free = G.forward(_f64(trained), rin, rcfg, False, rnd=round_bf16, wrnd=round_bf16)
    e_free = rel(stored["logits"], free.logits)
    report("gunet batch-norm eval", layer_worst=max(tape.errs.values()), logits_free_running=e_free)
    assert e_free < 3e-2
    assert np.array_equal(pred, np.argmax(tape.prob, axis=-1).astype(np.uint8))


def test_gunet_batch_norm_affine_dropout_trains_ten_steps(ctx):
    ecfg, rcfg, inputs, labels = _make(2, 64, normalizer="batch_norm", after_affine=True, dropout=0.5, use_context=True,
                                       use_spatial=True, loss_type="xentropy")
    eng = GUNetEngine(ctx, ecfg)
    eng.init_weights(seed=3)
    eng.set_inputs(inputs["images"], labels)
    eng.set_guides(inputs["context"], inputs["sp_guide"])
    losses = []
    for _ in range(10):
        eng.train_step(1e-3)
        losses.append(sum(eng.read_loss()))
    ctx.check_device()
    eng.close()
    report("gunet batch_norm + after_affine + dropout, 10 steps", first=losses[0], last=losses[-1])
    assert np.isfinite(losses).all()
    assert np.mean(losses[-3:]) < losses[0], losses


def test_gunet_batch_norm_affine_dropout_checkpoint_continues_bit_identically(ctx, tmp_path):
    ecfg, rcfg, inputs, labels = _make(2, 64, normalizer="batch_norm", after_affine=True, dropout=0.5, use_context=True,
                                       use_spatial=True, guide_channel=2, loss_type="xentropy", weight_decay_rate=3e-5)

    def fresh(seed):
        e = GUNetEngine(ctx, ecfg)
        e.init_weights(seed=seed)
        e.set_inputs(inputs["images"], labels)
        e.set_guides(inputs["context"], inputs["sp_guide"])
        return e

    a = fresh(2)
    for _ in range(2):
        a.train_step(1e-3)
    path = K.save_engine(a, tmp_path / "model.ckpt")
    shapes = K.load_checkpoint(path).get_variable_to_shape_map()
    assert shapes["GUNet/Encode/down_conv2/mod_conv1/ChannelWiseAffine/gamma"] == [128]
    assert shapes["GUNet/Encode/down_conv2/mod_conv1/Conv/BatchNorm/moving_variance"] == [128]
    assert "Optimizer/GUNet/Encode/down_conv1/mod_conv2/ChannelWiseAffine/beta/Adam" in shapes
    saved = a.get_weights()
    a.train_step(1e-3)
    loss_a, w_a = a.read_loss(), a.get_weights()
    a.close()

    b = fresh(77)
    assert K.restore_engine(b, tmp_path, with_slots=True) == 2 and b.step_count == 2
    back = b.get_weights()
    assert all(np.array_equal(back[k], saved[k]) for k in saved)
    b.train_step(1e-3)                   # the same dropout masks: the stream is keyed by (seed, step, 8 + level)
    loss_b, w_b = b.read_loss(), b.get_weights()
    b.close()
    assert loss_a == loss_b
    for k in w_a:
        assert np.array_equal(w_a[k], w_b[k]), k
