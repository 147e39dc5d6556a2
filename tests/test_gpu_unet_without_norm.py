"""UNet --without_norm (every 3x3 conv is conv + bias + ReLU out of the tensor-core epilogue) on the B200, model level:
one training step against the fp64 oracle (op by op on identical inputs, every gradient over the device's stored tape),
the cfg2 shape with sampled forward outputs, ten steps of falling loss, TTA prediction, checkpoint round trip, and
the reference's model_fn through networks/unet.py. GUNet and UNetInter still refuse the flag."""
import argparse

import numpy as np
import pytest

from boxsegliver_b200 import checkpoint as K
from boxsegliver_b200 import models, solver, synthetic
from boxsegliver_b200.device import f32_to_bf16_bits, round_bf16
from boxsegliver_b200.engine import EngineConfig, UNetEngine
from boxsegliver_b200.inference import Predictor
from boxsegliver_b200.networks.base import ModeKeys
from oracle import tf_ops as O
from tests import unet_without_norm_ref as R
from tests import sampling as S
from tests.gpu_util import FREE_RUNNING_SANITY, gate_gradients, rel, report

pytestmark = pytest.mark.gpu


def _cfgs(n, h, w, training=True, **kw):
    kw = {**dict(height=h, width=w, channel=3, init_channels=64, num_down_samples=4, without_norm=True,
                 weight_decay_rate=1e-5, loss_type="xentropy", loss_weight_type="numerical",
                 loss_numeric_w=(0.2, 0.4, 4.4)), **kw}
    return EngineConfig(batch=n, training=training, **kw), R.UNetCfg(**kw)


def _params(rcfg, seed):
    p = R.init_params(rcfg, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for k in p:
        if k.endswith("/biases"):
            p[k] = (0.05 * rng.standard_normal(p[k].shape)).astype(np.float32)
    return p


@pytest.mark.parametrize("n,h,w,kw", [
    (2, 64, 64, {}),
    (2, 64, 64, dict(bias_decay=True, loss_type="dice", loss_weight_type="none", loss_numeric_w=())),
    (1, 96, 80, {}),             # ragged: the levels below full resolution run on the first-generation kernel
])
def test_train_step_against_oracle(ctx, n, h, w, kw):
    ecfg, rcfg = _cfgs(n, h, w, **kw)
    images, labels = synthetic.make_batch(n, h, w, 3, seed=1500 + n)
    params = _params(rcfg, 7)
    eng = UNetEngine(ctx, ecfg)
    assert all(L.y is None for L in eng.layers if L.kind in ("stem", "conv"))
    eng.set_weights(params)
    eng.set_inputs(images, labels)
    eng.forward(True)
    eng.loss_backward()
    ctx.check_device()
    k = rcfg.num_classes
    logits = eng.logits.download(np.float32, (n, h, w, k))
    dlogits = eng.dlogits.download(np.float32, (n, h, w, k))
    grads = eng.get_grads()
    stored = eng.get_stored_forward()
    eng.optimizer_step(1e-3)
    ctx.check_device()
    data_loss, reg_loss = eng.read_loss()
    eng.close()

    tape = R.forward(params, round_bf16(images), rcfg, True, rnd=round_bf16, stem_fp32=False)
    loss_o, _ = R.loss_and_dlogits(tape, labels, rcfg)
    e_free = rel(logits, tape.logits)
    assert e_free < FREE_RUNNING_SANITY
    assert abs(data_loss - float(loss_o)) < 1e-2 * abs(float(loss_o))
    assert abs(reg_loss - R.regularization_loss(params, rcfg)) < 1e-6 * max(1.0, reg_loss)
    lw = R.layerwise_forward_errors(params, round_bf16(images), stored, logits, rcfg, True, wrnd=round_bf16)
    assert max(lw.values()) < 1e-2, max(lw.items(), key=lambda t: t[1])
    tft = R.tape_from_stored(params, round_bf16(images), stored, logits, rcfg, wrnd=round_bf16)
    _, dl = R.loss_and_dlogits(tft, labels, rcfg)
    assert rel(dlogits, dl) < 1e-5
    g_ref = R.backward(tft, dl, rcfg, rnd=round_bf16)
    assert set(g_ref) == set(grads)
    errs = {name: rel(grads[name], g) for name, g in g_ref.items()}
    worst = gate_gradients(errs)
    report(f"unet --without_norm {n}x{h}x{w} {kw}", op_by_op_worst=max(lw.values()), grad_worst=worst[1],
           grad_worst_name=worst[0], free_running_logits=e_free)


def _bits(view):
    return view.buf.download(np.uint16, (view.n, 1, view.h, view.w, view.ld))


def test_cfg2_shape_sampled(ctx):
    """cfg2 (batch 64, 256 x 256 x 3): every forward op at sampled outputs against fp64 conv + bias + ReLU on the
    device's stored inputs, the pools exact, loss and dlogits over all pixels, and the bias gradient of the last 3x3
    layer (every pixel) against its fp64 sum."""
    n, hw = 64, 256
    ecfg, rcfg = _cfgs(n, hw, hw)
    params = _params(rcfg, 11)
    images, labels = synthetic.make_batch(n, hw, hw, 3, seed=1359)
    eng = UNetEngine(ctx, ecfg)
    eng.set_weights(params)
    eng.set_inputs(images, labels)
    eng.forward(True)
    eng.loss_backward()
    ctx.check_device()
    rng = np.random.default_rng(5)
    worst = {}
    for L in eng.layers:
        if L.kind == "logits":
            continue
        wt = round_bf16(params[f"{L.scope}/weights"]).astype(np.float64)
        b = params[f"{L.scope}/biases"].astype(np.float64)
        if L.kind in ("stem", "conv"):
            pos = S.sample_positions(rng, (n, 1, L.h, L.w), 256)
            if L.kind == "stem":
                xb, c0 = f32_to_bf16_bits(images).reshape(n, 1, L.h, L.w, 3), 0
            else:
                xb, c0 = _bits(L.x), L.x.c0
            want = np.maximum(S.conv_at(xb, c0, L.cin, wt[None], pos) + b, 0.0)
            del xb
            abits = _bits(L.a)
            worst[L.scope] = S.rel(S.gather(abits, L.a.c0, L.cout, pos), want)
            if L.pooled is not None:
                pp = S.sample_positions(rng, (n, 1, L.h // 2, L.w // 2), 256)
                mx = None
                for dy in (0, 1):
                    for dx in (0, 1):
                        v = S.gather(abits, L.a.c0, L.cout, (pp[0], pp[1], 2 * pp[2] + dy, 2 * pp[3] + dx))
                        mx = v if mx is None else np.maximum(mx, v)
                assert np.array_equal(S.gather(_bits(L.pooled), L.pooled.c0, L.cout, pp), mx), L.scope
            del abits
        else:
            pos = S.sample_positions(rng, (n, 1, 2 * L.h, 2 * L.w), 256)
            want = S.conv_transpose_at(_bits(L.x), L.x.c0, L.cin, wt[None], b, pos, (1, 2, 2))
            worst[L.scope] = S.rel(S.gather(_bits(L.a), L.a.c0, L.cout, pos), want)
    print(f"\ncfg2 --without_norm: {len(worst)} sampled forward ops, worst {max(worst.values()):.2e}")
    assert max(worst.values()) < 1e-2, max(worst.items(), key=lambda t: t[1])

    k = rcfg.num_classes
    logits = eng.logits.download(np.float32, (n, hw, hw, k))
    loss, dl = O.weighted_sparse_softmax_cross_entropy(logits, labels, "numerical", numeric_w=(0.2, 0.4, 4.4))
    assert abs(eng.read_loss()[0] - float(loss)) < 1e-4 * abs(float(loss))
    assert rel(eng.dlogits.download(np.float32, (n, hw, hw, k)), dl) < 1e-5
    # last 3x3 layer: dA = bf16(dlogits @ W_logits^T), db = sum over pixels of dA * (a > 0)
    last, head = eng.layers[-2], eng.layers[-1]
    a = last.a.buf.download(np.uint16, (n * hw * hw, last.a.ld))[:, :last.cout]
    wl = params[f"{head.scope}/weights"].reshape(head.cin, k).astype(np.float32)
    db = np.zeros(last.cout)
    dlf = dl.reshape(-1, k).astype(np.float32)
    for i in range(0, a.shape[0], 1 << 18):
        da = round_bf16(dlf[i:i + (1 << 18)] @ wl.T).astype(np.float64)
        db += (da * (S.bf16_bits_to_f64(a[i:i + (1 << 18)]) > 0)).sum(axis=0)
    g = eng.get_grads()[f"{last.scope}/biases"]
    assert rel(g, db) < 1e-2
    eng.close()


def test_ten_steps_loss_falls(ctx):
    ecfg, rcfg = _cfgs(4, 64, 64)
    eng = UNetEngine(ctx, ecfg)
    eng.init_weights(seed=3)
    images, labels = synthetic.make_batch(4, 64, 64, 3, seed=1401)
    eng.set_inputs(images, labels)
    losses = []
    for _ in range(10):
        eng.train_step(1e-3)
        losses.append(sum(eng.read_loss()))
    ctx.check_device()
    # without a normaliser Adam's early steps are not smooth: at this seed the loss spikes once at step 8 and recovers,
    # and the fp32 oracle (tests/unet_without_norm_ref.py with Adam, from the same initial weights) takes the same path,
    # spike included
    assert all(np.isfinite(losses)) and losses[-1] < losses[0] and min(losses[-3:]) < min(losses[:3]), losses


def test_training_and_eval_forwards_are_identical(ctx):
    ecfg, rcfg = _cfgs(2, 64, 64)
    eng = UNetEngine(ctx, ecfg)
    eng.set_weights(_params(rcfg, 4))
    images, _ = synthetic.make_batch(2, 64, 64, 3, seed=9)
    eng.set_inputs(images)
    eng.forward(True)
    a = eng.logits.download(np.float32, (2, 64, 64, 3))
    eng.forward(False)
    assert np.array_equal(a, eng.logits.download(np.float32, (2, 64, 64, 3)))
    eng.close()


def test_tta_prediction(ctx):
    from tests.test_gpu_inference import AX2, _host_tta
    n, hw = 3, 64
    ecfg, rcfg = _cfgs(n, hw, hw, training=False)
    eng = UNetEngine(ctx, ecfg)
    eng.set_weights(_params(rcfg, 6))
    images, labels = synthetic.make_batch(n, hw, hw, 3, seed=78)
    eng.set_inputs(images, labels)
    pr = Predictor(eng, 3, True)
    pred = pr.predict(images, keep_variant_probs=True)
    ctx.check_device()
    assert np.array_equal(pred, _host_tta(pr.variant_probs, pr.variants, AX2, True))
    pr.close()
    eng.close()


def test_checkpoint_round_trip(ctx, tmp_path):
    images, labels = synthetic.make_batch(2, 64, 64, 3, seed=1402)
    ecfg, _ = _cfgs(2, 64, 64)
    a = UNetEngine(ctx, ecfg)
    a.init_weights(seed=2)
    a.set_inputs(images, labels)
    for _ in range(2):
        a.train_step(1e-3)
    path = K.save_engine(a, tmp_path / "model.ckpt")
    names = K.load_checkpoint(path).get_variable_to_shape_map()
    assert names["UNet/Encode1/Repeat/convolution2d_1/biases"] == [64]
    assert not any("BatchNorm" in k for k in names)
    a.train_step(1e-3)
    loss_a, w_a = a.read_loss(), a.get_weights()
    a.close()
    b = UNetEngine(ctx, ecfg)
    b.init_weights(seed=77)
    assert K.restore_engine(b, tmp_path, with_slots=True) == 2
    b.set_inputs(images, labels)
    b.train_step(1e-3)
    loss_b, w_b = b.read_loss(), b.get_weights()
    b.close()
    assert loss_a == loss_b
    for k in w_a:
        assert np.array_equal(w_a[k], w_b[k]), k


def _args(model, **kw):
    p = argparse.ArgumentParser()
    models.add_arguments(p)
    solver.add_arguments(p)
    a = p.parse_args(["--model", model, "--classes", "Liver", "Tumor", "--batch_size", "2", "--without_norm",
                      "--learning_rate", "1e-3"])
    base = dict(im_height=64, im_width=64, im_channel=3, num_gpus=1, seed=3, weight_decay_rate=1e-5, bias_decay=False,
                loss_type="xentropy", loss_weight_type="numerical", loss_numeric_w=[0.2, 0.4, 4.4],
                loss_proportion_decay=1000.0, metrics_train=["Dice"], use_spatial=False, use_context=False)
    base.update(kw)
    for k, v in base.items():
        setattr(a, k, v)
    return a


def test_model_fn_train_and_eval(ctx):
    args = _args("UNet")
    params = models.get_model_params(args, build_metrics=True)
    params.update(args=args, solver=solver.Solver, ctx=ctx, world=1)
    images, labels = synthetic.make_batch(2, 64, 64, 3, seed=1400)
    spec = models.model_fn(dict(images=images), labels, ModeKeys.TRAIN, params)
    model = spec.model
    assert model.engine.cfg.without_norm
    model.feed(images, labels)
    losses = []
    for _ in range(4):
        spec.train_op.run(with_metrics=True)
        losses.append(spec.train_op.fetch_loss())
    ctx.check_device()
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    assert set(model.collect_metrics()) == {"Liver/Dice", "Tumor/Dice"}
    model.mode = ModeKeys.EVAL
    prob = model.run_forward()
    assert prob.shape == (2, 64, 64, 3) and np.allclose(prob.sum(-1), 1.0, atol=1e-5)
    eng = model.engine
    model.engine = None
    eng.close()
    # the first loss is the engine's own step with the same seed
    ecfg = EngineConfig(batch=2, height=64, width=64, channel=3, classes=("Background", "Liver", "Tumor"),
                        weight_decay_rate=1e-5, loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4),
                        without_norm=True)
    eng = UNetEngine(ctx, ecfg)
    eng.init_weights(seed=3)
    eng.set_inputs(images, labels)
    eng.train_step(1e-3)
    assert losses[0] == pytest.approx(sum(eng.read_loss()), rel=1e-6)
    eng.close()


@pytest.mark.parametrize("model", ["GUNet", "UNetInter"])
def test_gunet_and_unetinter_refuse_the_flag(ctx, model):
    args = _args(model, normalizer="instance_norm")
    params = models.get_model_params(args, build_metrics=True)
    params.update(args=args, solver=solver.Solver, ctx=ctx, world=1)
    with pytest.raises(NotImplementedError, match="without_norm"):
        models.model_fn(dict(images=None), None, ModeKeys.TRAIN, params)
