"""UNet3D with --normalizer batch_norm (the reference's default normaliser) on the device: slim variable names, parity of
one training step against the batch-norm oracle (tests/unet3d_bn_ref.py) with the method of test_gpu_unet3d.py, the
moving-statistics update, eval-mode forwards on the moving statistics (layers, TTA), the cfg4 shape, model_fn with
default flags, and checkpoint round trips of the moving statistics."""
import argparse
import dataclasses

import numpy as np
import pytest

from boxsegliver_b200 import checkpoint as K
from boxsegliver_b200 import models, solver, synthetic
from boxsegliver_b200.device import round_bf16
from boxsegliver_b200.inference import Predictor
from boxsegliver_b200.networks.base import ModeKeys
from boxsegliver_b200.unet3d_engine import UNet3DConfig, UNet3DEngine
from oracle import unet3d_ref as U
from tests import sampling as S
from tests import unet3d_bn_ref as B
from tests.gpu_util import rel, report
from tests.test_gpu_baseline_shapes import _bits
from tests.test_gpu_inference import AX3, _host_tta

pytestmark = pytest.mark.gpu

SHAPES = [
    (2, 4, 32, dict()),                                                     # UNet3D.yml channels, 4 pools
    (1, 2, 64, dict(num_pool_layers=5, use_spatial=True, guide_channel=2, loss_numeric_w=(1.0, 10.0))),
    (2, 6, 32, dict(init_channels=16, max_channels=128, loss_weight_type="proportion", loss_numeric_w=())),
    (2, 4, 32, dict(_pair="0")),                                            # 64-lane storage of the full-resolution level
    (1, 2, 32, dict(init_channels=48, max_channels=96, _pair=None)),         # 48 > 32 channels: never packed
]


def _is_moving(name):
    return name.endswith(("moving_mean", "moving_variance"))


def _params(rcfg, seed=6):
    """Oracle initial values with non-trivial gamma / beta / biases and moving statistics."""
    params = B.init_params(rcfg, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for k, v in params.items():
        if k.endswith(("beta", "biases", "moving_mean")):
            params[k] = (0.1 * rng.standard_normal(v.shape)).astype(np.float32)
        elif k.endswith("gamma"):
            params[k] = (1 + 0.1 * rng.standard_normal(v.shape)).astype(np.float32)
        elif k.endswith("moving_variance"):
            params[k] = rng.uniform(0.5, 1.5, v.shape).astype(np.float32)
    return params


def _inputs(rcfg, n, seed=9):
    d, hw = rcfg.depth, rcfg.height
    if rcfg.use_spatial:
        images, labels, guide = synthetic.make_volume_batch(n, d, hw, hw, seed=seed, guide_channel=rcfg.guide_channel)
    else:
        (images, labels), guide = synthetic.make_volume_batch(n, d, hw, hw, seed=seed), None
    inputs = dict(images=round_bf16(images).astype(np.float64))
    if guide is not None:
        inputs["sp_guide"] = round_bf16(guide).astype(np.float64)
    return images, labels, guide, inputs


def _expected_moving(stored, params, rcfg):
    """decay * before + (1 - decay) * (fp64 mean, unbiased variance of the device's own stored pre-norm tensor)."""
    out = {}
    for sp in B.layer_specs(rcfg):
        if sp["kind"] != "conv":
            continue
        ns = f"{sp['scope']}/BatchNorm"
        y = stored[sp["scope"]]["y"].astype(np.float64).reshape(-1, sp["cout"])
        dec = np.float64(np.float32(rcfg.bn_decay))
        out[f"{ns}/moving_mean"] = dec * params[f"{ns}/moving_mean"] + (1 - dec) * y.mean(0)
        out[f"{ns}/moving_variance"] = dec * params[f"{ns}/moving_variance"] + (1 - dec) * y.var(0, ddof=1)
    return out


def test_batch_norm_variable_names_and_round_trip(ctx):
    rcfg = B.UNet3DBNCfg(depth=2, height=32, width=32)
    eng = UNet3DEngine(ctx, UNet3DConfig(batch=1, depth=2, height=32, width=32, normalizer="batch_norm"))
    params = _params(rcfg)
    assert set(eng.params) == set(params)
    assert len([k for k in eng.params if "/BatchNorm/" in k]) == 18 * 4
    assert not any("InstanceNorm" in k for k in eng.params)
    eng.set_weights(params)
    back = eng.get_weights()
    for k in params:
        assert np.array_equal(back[k], params[k]), k
    assert set(eng.get_slots()) == set(eng.get_grads()) == {k for k in params if not _is_moving(k)}
    w0 = eng.init_weights(seed=0)
    for k in w0:
        if k.endswith("moving_mean"):
            assert not w0[k].any()
        elif k.endswith("moving_variance"):
            assert (w0[k] == 1).all()
    eng.close()
    with pytest.raises(ValueError, match="Not supported normalization function"):
        UNet3DEngine(ctx, UNet3DConfig(batch=1, depth=2, height=32, width=32, normalizer="group_norm"))


@pytest.mark.parametrize("n,d,hw,kw", SHAPES)
def test_unet3d_batch_norm_train_step_parity(ctx, n, d, hw, kw, monkeypatch):
    base = dict(depth=d, height=hw, width=hw, channel=1, weight_decay_rate=3e-5)
    kw = dict(kw)
    pair = kw.pop("_pair", "1")
    if pair is not None:
        monkeypatch.setenv("BSL_UNET3D_PAIR", pair)
    base.update(kw)
    ecfg, rcfg = UNet3DConfig(batch=n, normalizer="batch_norm", **base), B.UNet3DBNCfg(**base)
    images, labels, guide, inputs = _inputs(rcfg, n)
    params = _params(rcfg)
    eng = UNet3DEngine(ctx, ecfg)
    assert eng._pair == (pair == "1")
    eng.set_weights(params)
    eng.set_inputs(images, labels, guide)
    eng.forward(True)
    eng.predict_outputs(True)
    eng.loss_backward()
    ctx.check_device()
    kcls = rcfg.num_classes
    logits = eng.logits.download(np.float32, (n, d, hw, hw, kcls))
    dlogits = eng.dlogits.download(np.float32, (n, d, hw, hw, kcls))
    grads = eng.get_grads()
    moving = {k: v for k, v in eng.get_weights().items() if _is_moving(k)}
    stored = eng.get_stored_forward()         # also asserts the pad lanes are exactly zero
    stored["logits"] = logits
    eng.optimizer_step(1e-3)
    ctx.check_device()
    data_loss, reg_loss = eng.read_loss()
    new_w = eng.get_weights()
    eng.close()

    # moving statistics: one update from the device's own batch statistics; the optimizer leaves them alone
    want = _expected_moving(stored, params, rcfg)
    assert set(want) == set(moving)
    m_errs = {k: rel(moving[k], want[k]) for k in want}
    assert max(m_errs.values()) <= 1e-6, max(m_errs.items(), key=lambda t: t[1])
    assert all(np.array_equal(new_w[k], moving[k]) for k in moving)

    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    tft = B.forward(p64, inputs, rcfg, True, wrnd=round_bf16, stored=stored)
    assert max(tft.errs.values()) < 1e-2, max(tft.errs.items(), key=lambda t: t[1])
    loss_o, dl = B.loss_and_dlogits(tft, labels, rcfg)
    assert abs(data_loss - loss_o) < 1e-4 * abs(loss_o)
    assert abs(reg_loss - B.regularization_loss(params, rcfg)) < 1e-6
    assert rel(dlogits, dl) < 1e-5
    g_ref = B.backward(tft, dl, rcfg, rnd=round_bf16)
    assert set(g_ref) == set(grads)
    errs = {name: rel(grads[name], g) for name, g in g_ref.items()}
    assert np.median(list(errs.values())) < 1e-2, errs
    # batch statistics reduce over n * voxels values; below 256 the tolerance of test_gpu_unet3d.py's tiny layers applies
    vox = {}
    for sp in B.layer_specs(rcfg):
        o = [-(-sp["dhw"][i] // sp["s"][i]) for i in range(3)] if sp["kind"] == "conv" else [sp["dhw"][i] * sp["s"][i] for i in range(3)]
        vox[sp["scope"]] = n * int(np.prod(o))
    scope = lambda name: name.rsplit("/BatchNorm", 1)[0].rsplit("/weights", 1)[0].rsplit("/biases", 1)[0]  # noqa: E731
    for name, e in errs.items():
        assert e < (1e-2 if vox[scope(name)] >= 256 else 5e-2), (name, e, vox[scope(name)])
    big = [e for nm, e in errs.items() if vox[scope(nm)] >= 256]
    report(f"unet3d batch_norm {n}x{d}x{hw}x{hw}", layer_worst=max(tft.errs.values()),
           grad_median=float(np.median(list(errs.values()))), grad_worst_ge256_values=max(big),
           grad_worst_tiny_statistics=max(errs.values()), moving_worst=max(m_errs.values()))
    tg = U.total_grads(params, grads, rcfg)
    for name in tg:
        w, _, _ = U.O.adam_step(params[name].astype(np.float64), tg[name].astype(np.float64), 0.0, 0.0, 1, 1e-3)
        assert rel(new_w[name].astype(np.float64) - params[name], w - params[name]) < 1e-3, name


@pytest.mark.parametrize("pair", ["1", "0"])
def test_unet3d_batch_norm_eval_forward_uses_moving_statistics(ctx, pair, monkeypatch):
    monkeypatch.setenv("BSL_UNET3D_PAIR", pair)
    n, d, hw = 2, 4, 32
    rcfg = B.UNet3DBNCfg(depth=d, height=hw, width=hw)
    images, labels, _, inputs = _inputs(rcfg, n, seed=11)
    params = _params(rcfg, seed=3)
    eng = UNet3DEngine(ctx, UNet3DConfig(batch=n, depth=d, height=hw, width=hw, normalizer="batch_norm"))
    eng.set_weights(params)
    eng.set_inputs(images, labels)
    s0 = eng.S.download(np.uint32, (eng.n_stats,))
    eng.forward(False)
    eng.predict_outputs(False)
    ctx.check_device()
    assert np.array_equal(eng.S.download(np.uint32, (eng.n_stats,)), s0), "an eval forward moved the moving statistics"
    stored = eng.get_stored_forward()
    stored["logits"] = eng.logits.download(np.float32, (n, d, hw, hw, 2))
    eng.close()
    tape = B.forward({k: v.astype(np.float64) for k, v in params.items()}, inputs, rcfg, False, wrnd=round_bf16,
                     stored=stored)
    assert max(tape.errs.values()) < 1e-2, max(tape.errs.items(), key=lambda t: t[1])


def test_unet3d_batch_norm_tta_all_mirrors(ctx):
    n, d, hw = 1, 4, 32
    rcfg = B.UNet3DBNCfg(depth=d, height=hw, width=hw)
    eng = UNet3DEngine(ctx, UNet3DConfig(batch=n, depth=d, height=hw, width=hw, normalizer="batch_norm", training=False))
    eng.set_weights(_params(rcfg, seed=1))
    images, labels = synthetic.make_volume_batch(n, d, hw, hw, seed=4)
    eng.set_inputs(images, labels)
    s0 = eng.S.download(np.uint32, (eng.n_stats,))
    pr = Predictor(eng, random_flip=7, eval_mirror=True)
    pred = pr.predict(images, keep_variant_probs=True)
    ctx.check_device()
    assert np.array_equal(pred, _host_tta(pr.variant_probs, pr.variants, AX3, False))
    assert np.array_equal(eng.S.download(np.uint32, (eng.n_stats,)), s0)
    pr.close()
    eng.close()


def test_cfg4_unet3d_batch_norm_full_size_sampled_parity(ctx):
    """cfg4 shape (4 x 64 x 128 x 128, UNet3D.yml channels) with batch norm: every conv / transposed conv at sampled
    output voxels, batch norm + ReLU at the same voxels, the moving-statistics update of every layer (mean error relative
    to the channels' RMS), loss + dlogits."""
    n, d, h, w = 4, 64, 128, 128
    cfg = UNet3DConfig(batch=n, depth=d, height=h, width=w, loss_numeric_w=(1.0, 1.0), normalizer="batch_norm")
    eng = UNet3DEngine(ctx, cfg)
    params = eng.init_weights(5)
    rng = np.random.default_rng(6)
    for k_ in params:
        if k_.endswith("beta"):
            params[k_] = (0.1 * rng.standard_normal(params[k_].shape)).astype(np.float32)
        if k_.endswith("gamma"):
            params[k_] = (1 + 0.1 * rng.standard_normal(params[k_].shape)).astype(np.float32)
    eng.set_weights(params)
    im, lb = synthetic.make_volume_batch(n, d, h, w, seed=1357 + 4)
    eng.set_inputs(im, lb)
    eng.forward(True)
    eng.loss_backward()
    ctx.check_device()
    moving = eng.get_weights()
    from boxsegliver_b200.device import f32_to_bf16_bits
    worst, m_worst = {}, {}
    dec = np.float64(np.float32(cfg.bn_decay))
    for L in eng.layers:
        if L.kind == "logits":
            continue
        wt = round_bf16(params[f"{L.scope}/weights"]).astype(np.float64)
        od, oh, ow = L.odhw
        pos = S.sample_positions(rng, (n, od, oh, ow), 256)
        if L.kind == "convT":
            ab = _bits(L.a, (n,) + L.odhw)
            want = S.conv_transpose_at(_bits(L.x, (n,) + L.dhw), L.x.c0, L.cin, wt, None, pos, L.s)
            worst[f"{L.scope} convT"] = S.rel(S.gather(ab, L.a.c0, L.cout, pos), want)
            continue
        if L.kind == "stem":
            xb, c0, cmap = f32_to_bf16_bits(im).reshape(n, d, h, w, cfg.in_channels), 0, None
        else:
            xb, c0, cmap = _bits(L.x, (n,) + L.dhw, getattr(L, "catpair", False)), L.x.c0, L.cin_map
        want = S.conv_at(xb, c0, L.cin, wt, pos, stride=L.s, cin_map=cmap)
        yb = _bits(L.y, (n,) + L.odhw)
        got = S.gather(yb, L.y.c0, L.cout, pos)
        worst[f"{L.scope} conv{L.k}/{L.s}"] = S.rel(got, want)
        mean, var = S.channel_moments(yb, L.y.c0, L.cout, per_sample=False, chunk=1)
        mean, var = mean[0], var[0]
        ns = f"{L.scope}/BatchNorm"
        g, b = params[f"{ns}/gamma"].astype(np.float64), params[f"{ns}/beta"].astype(np.float64)
        a_ref = np.maximum((got - mean) / np.sqrt(var + cfg.bn_eps) * g + b, 0.0)
        worst[f"{L.scope} norm+relu"] = S.rel(S.gather(_bits(L.a, (n,) + L.odhw), L.a.c0, L.cout, pos), a_ref)
        m = n * int(np.prod(L.odhw))
        # the mean's error is taken relative to the channels' RMS: the sums are accumulated from fp32 per-CTA partials,
        # and at this size a channel mean can be ~1e-3 of its RMS (the stem), where a plain relative error measures the
        # cancellation, not the reduction
        rms = np.sqrt(var + mean * mean)
        m_worst[f"{ns}/moving_mean"] = float(np.linalg.norm(moving[f"{ns}/moving_mean"] - (1 - dec) * mean)
                                             / ((1 - dec) * np.linalg.norm(rms)))
        m_worst[f"{ns}/moving_variance"] = rel(moving[f"{ns}/moving_variance"], dec + (1 - dec) * var * m / (m - 1))
    bad = {k: v for k, v in worst.items() if not v < 1e-2}
    print(f"\ncfg4 batch_norm: {len(worst)} sampled forward ops, worst {max(worst.values()):.2e} "
          f"({max(worst, key=worst.get)}); moving statistics worst {max(m_worst.values()):.2e}")
    assert not bad, bad
    assert max(m_worst.values()) <= 1e-6, max(m_worst.items(), key=lambda t: t[1])
    logits = eng.logits.download(np.float32, (n, d, h, w, 2))
    loss, dl = U.O.weighted_sparse_softmax_cross_entropy(logits.reshape(n, d * h, w, 2), lb.reshape(n, d * h, w),
                                                         "numerical", numeric_w=(1.0, 1.0))
    assert abs(eng.read_loss()[0] - float(loss)) < 1e-4 * abs(float(loss))
    assert rel(eng.dlogits.download(np.float32, (n, d * h, w, 2)), dl) < 1e-5
    eng.close()


def _unet3d_args():
    p = argparse.ArgumentParser()
    models.add_arguments(p)
    solver.add_arguments(p)
    a = p.parse_args(["--model", "UNet3D", "--classes", "NF", "--batch_size", "2", "--learning_rate", "1e-3"])
    for k, v in dict(im_depth=4, im_height=32, im_width=32, im_channel=1, num_gpus=1, seed=3, weight_decay_rate=3e-5,
                     bias_decay=False, loss_type="xentropy", loss_weight_type="numerical", loss_numeric_w=[1.0, 1.0],
                     loss_proportion_decay=1000.0, metrics_train=["Dice"], use_spatial=False).items():
        setattr(a, k, v)
    return a


def test_unet3d_default_normalizer_through_model_fn(ctx):
    args = _unet3d_args()
    assert args.normalizer == "batch_norm"                     # the reference's default
    params = models.get_model_params(args, build_metrics=True)
    params.update(args=args, solver=solver.Solver, ctx=ctx, world=1)
    images, labels = synthetic.make_volume_batch(2, 4, 32, 32, seed=1401)
    spec = models.model_fn(dict(images=images), labels, ModeKeys.TRAIN, params)
    model = spec.model
    assert model.engine.cfg.normalizer == "batch_norm"
    model.feed(images, labels)
    losses = []
    for _ in range(4):
        spec.train_op.run()
        losses.append(spec.train_op.fetch_loss())
    ctx.check_device()
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    model.mode = ModeKeys.EVAL
    s0 = model.engine.S.download(np.uint32, (model.engine.n_stats,))
    prob = model.run_forward()
    assert np.array_equal(model.engine.S.download(np.uint32, (model.engine.n_stats,)), s0)
    assert prob.shape == (2, 4, 32, 32, 2) and np.allclose(prob.sum(-1), 1.0, atol=1e-5)
    m = model.predictions["NFPred"]
    assert m.dtype == np.uint8 and np.array_equal(m[..., 0], (prob[..., 1] > 0.5).astype(np.uint8))
    cfg = dataclasses.replace(model.engine.cfg)
    model.engine.close()
    model.engine = None

    eng = UNet3DEngine(ctx, cfg)
    eng.init_weights(seed=3)
    eng.set_inputs(images, labels)
    eng.train_step(1e-3)
    direct = sum(eng.read_loss())
    eng.close()
    assert losses[0] == pytest.approx(direct, rel=1e-6)


def test_unet3d_batch_norm_checkpoint_continues_bit_identically(ctx, tmp_path):
    cfg = UNet3DConfig(batch=2, depth=4, height=32, width=32, weight_decay_rate=3e-5, normalizer="batch_norm")
    images, labels = synthetic.make_volume_batch(2, 4, 32, 32, seed=1403)
    a = UNet3DEngine(ctx, cfg)
    a.init_weights(seed=2)
    a.set_inputs(images, labels)
    for _ in range(2):
        a.train_step(1e-3)
    path = K.save_engine(a, tmp_path / "model.ckpt")
    r = K.load_checkpoint(path)
    shapes = r.get_variable_to_shape_map()
    assert shapes["UNet3D/conv_e0/conv1/BatchNorm/moving_variance"] == [30]
    assert "Optimizer/UNet3D/conv_e0/conv1/BatchNorm/gamma/Adam" in shapes
    assert not any(k.startswith("Optimizer/") and "moving_" in k for k in shapes)
    saved = a.get_weights()
    assert np.array_equal(r.get_tensor("UNet3D/bridge/conv2/BatchNorm/moving_mean"), saved["UNet3D/bridge/conv2/BatchNorm/moving_mean"])
    a.train_step(1e-3)
    w_a = a.get_weights()
    a.close()

    b = UNet3DEngine(ctx, cfg)
    b.init_weights(seed=77)
    assert K.restore_engine(b, tmp_path, with_slots=True) == 2
    back = b.get_weights()
    assert all(np.array_equal(back[k], saved[k]) for k in saved)
    b.set_inputs(images, labels)
    b.train_step(1e-3)
    w_b = b.get_weights()
    b.close()
    for k in w_a:
        assert np.array_equal(w_a[k], w_b[k]), k
