"""End-to-end parity of the U-Net engine (forward, loss, backward, optimizer, masks, counts) against the
numpy oracle, plus full-size properties at BASELINE cfg2 (batch 64, 256x256x3).

Gates (relative L2 norm per tensor, bf16 path, north_star tolerance 1e-2):
  * every forward op on identical inputs (fp64 oracle op vs the stored device output) ............ <= 1e-2
  * gradients: oracle backward over the DEVICE's stored forward tensors, so that ReLU masks and max-pool
    arg-maxes are the same bits on both sides: tests/gpu_util.gate_gradients -- every tensor <= 1e-2 at the
    BASELINE shapes (tests/test_gpu_baseline_shapes.py); at these tiny code-path shapes median and 90th
    percentile <= 1e-2, worst <= 1.25e-2
  * `p > 0.5` masks, argmax and Dice I/L/R counts ................................ bit-exact given the logits
Reported, bounded only by a sanity limit (tests/gpu_util.FREE_RUNNING_SANITY): the free-running logits vs the oracle
with bf16-storage emulation (tiny-batch BN statistics amplify last-ulp differences).
"""
import numpy as np
import pytest

from boxsegliver_b200 import synthetic
from boxsegliver_b200.device import round_bf16
from boxsegliver_b200.engine import EngineConfig, UNetEngine
from oracle import unet_ref as R
from tests.gpu_util import FREE_RUNNING_SANITY, gate_gradients, rel, report

pytestmark = pytest.mark.gpu


def _hw(hw):
    return hw if isinstance(hw, tuple) else (hw, hw)


def _cfgs(n, hw, normalizer, loss_type, wtype):
    kw = dict(height=_hw(hw)[0], width=_hw(hw)[1], channel=3, init_channels=64, num_down_samples=4, normalizer=normalizer,
              weight_decay_rate=1e-5, loss_type=loss_type, loss_weight_type=wtype,
              loss_numeric_w=(0.2, 0.4, 4.4) if wtype == "numerical" else ())
    return EngineConfig(batch=n, **kw), R.UNetCfg(**kw)


@pytest.mark.parametrize("n,hw,normalizer,loss_type,wtype", [
    (2, 128, "batch_norm", "xentropy", "numerical"),
    (3, 64, "instance_norm", "xentropy", "numerical"),
    (2, 64, "batch_norm", "dice", "none"),
    (2, 64, "batch_norm", "xentropy", "proportion"),
    # ragged: 96 x 80 (the shipped scripts also train at 256 x 80 / 960 x 320): levels 48x40 .. 6x5 are not multiples
    # of the 8 x 16 halo tile, so every conv below full resolution runs on the general implicit-GEMM kernel; batch 1
    (1, (96, 80), "batch_norm", "xentropy", "numerical"),
    (2, (32, 48), "instance_norm", "dice", "none"),
])
def test_train_step_parity(ctx, n, hw, normalizer, loss_type, wtype):
    ecfg, rcfg = _cfgs(n, hw, normalizer, loss_type, wtype)
    hh, ww = _hw(hw)
    images, labels = synthetic.make_batch(n, hh, ww, 3, seed=1357 + n)
    params = R.init_params(rcfg, seed=7)
    eng = UNetEngine(ctx, ecfg)
    eng.set_weights(params)
    eng.set_inputs(images, labels)
    lr = 1e-3
    eng.forward(True)
    eng.predict_outputs(True)
    eng.loss_backward()
    ctx.check_device()
    k = rcfg.num_classes
    logits = eng.logits.download(np.float32, (n, hh, ww, k))
    dlogits = eng.dlogits.download(np.float32, (n, hh, ww, k))
    grads = eng.get_grads()
    stored = eng.get_stored_forward()
    masks = eng.masks.download(np.uint8, (k - 1, n, hh, ww))
    argmax = eng.argmax.download(np.uint8, (n, hh, ww))
    counts = eng.read_counts()
    eng.optimizer_step(lr)
    ctx.check_device()
    data_loss, reg_loss = eng.read_loss()
    new_w = eng.get_weights()
    eng.close()

    # forward: free-running oracle with bf16 storage emulation
    tape = R.forward(params, round_bf16(images), rcfg, True, rnd=round_bf16, stem_fp32=False)
    loss_o, _ = R.loss_and_dlogits(tape, labels, rcfg)
    e_free = rel(logits, tape.logits)
    assert e_free < FREE_RUNNING_SANITY
    assert abs(data_loss - float(loss_o)) < 1e-3 * abs(float(loss_o))
    assert abs(reg_loss - R.regularization_loss(params, rcfg)) < 1e-6
    if normalizer == "batch_norm":
        for name, v in tape.new_moving.items():
            assert rel(new_w[name], v) < 1e-2, name

    # forward, op by op on identical inputs (fp64 oracle op vs the stored device output): the 1e-2 bf16 gate
    lw = R.layerwise_forward_errors(params, round_bf16(images), stored, logits, rcfg, True, wrnd=round_bf16)
    assert max(lw.values()) < 1e-2, max(lw.items(), key=lambda t: t[1])

    # backward: oracle over the device's stored forward tape
    tft = R.tape_from_stored(params, round_bf16(images), stored, logits, rcfg, wrnd=round_bf16)
    _, dl = R.loss_and_dlogits(tft, labels, rcfg)
    assert rel(dlogits, dl) < 1e-5
    g_ref = R.backward(tft, dl, rcfg, rnd=round_bf16)
    errs = {name: rel(grads[name], g) for name, g in g_ref.items()}
    worst = max(errs.items(), key=lambda t: t[1])
    report(f"unet {n}x{hh}x{ww} {normalizer} {loss_type}/{wtype}", op_by_op_worst=max(lw.values()),
           grad_median=float(np.median(list(errs.values()))), grad_worst=worst[1], grad_worst_name=worst[0],
           free_running_logits=e_free)
    gate_gradients(errs)

    # masks / argmax / counts: bit-exact functions of the device's own logits
    prob = R.O.softmax(logits)
    decided = np.abs(prob[..., 1:] - 0.5).transpose(3, 0, 1, 2) > 1e-6
    m_ref = np.stack([(prob[..., c] > 0.5).astype(np.uint8) for c in range(1, k)])
    assert not ((masks != m_ref) & decided).any()
    srt = np.sort(prob, axis=-1)
    clear = (srt[..., -1] - srt[..., -2]) > 1e-6
    assert np.array_equal(argmax[clear], np.argmax(prob, axis=-1).astype(np.uint8)[clear])
    for c in range(1, k):
        i_, l_, r_ = R.O.seg_counts(masks[c - 1][..., None], labels, c)
        assert np.array_equal(counts[:, c - 1, 0], i_)
        assert np.array_equal(counts[:, c - 1, 1], l_)
        assert np.array_equal(counts[:, c - 1, 2], r_)

    # optimizer: oracle Adam applied to the device gradients reproduces the device update
    tg = R.total_grads(params, grads, rcfg)
    for name in R.trainable_names(rcfg, params):
        w, _, _ = R.O.adam_step(params[name].astype(np.float64), tg[name].astype(np.float64), 0.0, 0.0, 1, lr)
        assert rel(new_w[name].astype(np.float64) - params[name], w - params[name]) < 1e-3, name


def test_eval_mode_uses_moving_statistics(ctx):
    n, hw = 2, 64
    ecfg, rcfg = _cfgs(n, hw, "batch_norm", "xentropy", "none")
    ecfg.training = False
    params = R.init_params(rcfg, seed=3)
    rng = np.random.default_rng(0)
    for name in params:
        if name.endswith("moving_mean"):
            params[name] = rng.normal(0, 0.05, params[name].shape).astype(np.float32)
        if name.endswith("moving_variance"):
            params[name] = rng.uniform(0.5, 1.5, params[name].shape).astype(np.float32)
    images, labels = synthetic.make_batch(n, hw, hw, 3, seed=5)
    eng = UNetEngine(ctx, ecfg)
    eng.set_weights(params)
    eng.set_inputs(images, labels)
    eng.forward(False)
    eng.predict_outputs(False)
    ctx.check_device()
    logits = eng.logits.download(np.float32, (n, hw, hw, 3))
    after = eng.get_weights()
    stored = eng.get_stored_forward()
    eng.close()
    tape = R.forward(params, round_bf16(images), rcfg, False, rnd=round_bf16, stem_fp32=False)
    assert rel(logits, tape.logits) < FREE_RUNNING_SANITY
    lw = R.layerwise_forward_errors(params, round_bf16(images), stored, logits, rcfg, False, wrnd=round_bf16)
    assert max(lw.values()) < 1e-2, max(lw.items(), key=lambda t: t[1])
    for name in params:
        assert np.array_equal(after[name], params[name]), f"{name} changed in eval mode"


def test_full_size_training_properties(ctx):
    """BASELINE cfg2 shapes (batch 64, 256x256x3): properties the oracle is not needed for."""
    n, hw = 64, 256
    ecfg, _ = _cfgs(n, hw, "batch_norm", "xentropy", "numerical")
    images, labels = synthetic.make_batch(n, hw, hw, 3)
    eng = UNetEngine(ctx, ecfg)
    eng.init_weights(seed=0)
    eng.set_inputs(images, labels)
    w0 = eng.get_weights()
    # (1) determinism: two forward+backward passes from the same state give bit-identical gradients
    eng.forward(True); eng.predict_outputs(True); eng.loss_backward(); ctx.check_device()
    g1 = eng.G.download(np.float32, (eng.n_train,))
    c1 = eng.read_counts()
    eng.set_weights(w0)     # forward(True) advanced the moving statistics: restore
    eng.forward(True); eng.predict_outputs(True); eng.loss_backward(); ctx.check_device()
    g2 = eng.G.download(np.float32, (eng.n_train,))
    assert np.array_equal(g1, g2), "gradients are not bit-reproducible"
    assert np.all(np.isfinite(g1))
    # (2) integer identities of the Dice counts: R equals the label histogram, I <= min(L, R)
    for c in (1, 2):
        r = (labels.reshape(n, -1) == c).sum(axis=1)
        assert np.array_equal(c1[:, c - 1, 2], r)
        assert np.all(c1[:, c - 1, 0] <= np.minimum(c1[:, c - 1, 1], c1[:, c - 1, 2]))
    # (3) sum over classes of dlogits is zero per pixel (softmax - onehot, any weight)
    dl = eng.dlogits.download(np.float32, (n * hw * hw, 3))
    assert np.abs(dl.sum(axis=1)).max() < 1e-9
    # (4) training on a fixed batch reduces the loss
    losses = []
    eng.set_weights(w0)
    for _ in range(6):
        eng.train_step(1e-3)
        losses.append(sum(eng.read_loss()))
    ctx.check_device()
    assert np.all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    eng.close()


def test_host_fed_steps_match_device_resident_steps(ctx):
    """The e2e entry points (pinned batch -> H2D -> step -> D2H loss; with and without prefetch) run the same
    arithmetic as the device-resident step: identical loss sequences and bit-identical weights."""
    n, hw = 2, 64
    ecfg, _ = _cfgs(n, hw, "batch_norm", "xentropy", "numerical")
    batches = [synthetic.make_batch(n, hw, hw, 3, seed=40 + i) for i in range(3)]

    def run(mode):
        eng = UNetEngine(ctx, ecfg)
        eng.init_weights(seed=2)
        losses = []
        if mode == "resident":
            for im, lb in batches:
                eng.set_inputs(im, lb)
                eng.train_step(1e-3)
                losses.append(sum(eng.read_loss()))
        elif mode == "host":
            pi, pl = eng.pinned_inputs()
            for im, lb in batches:
                pi[...] = im
                pl[...] = lb
                losses.append(eng.train_step_host(1e-3))
        else:
            for j in (0, 1):
                eng.staging_slot(j)
            si, sl = eng.staging_slot(0)
            si[...], sl[...] = batches[0]
            eng.submit_staged(0)
            for i in range(len(batches)):
                if i + 1 < len(batches):
                    si, sl = eng.staging_slot((i + 1) % 2)
                    si[...], sl[...] = batches[i + 1]
                    eng.submit_staged((i + 1) % 2)
                losses.append(eng.train_step_prefetched(1e-3))
        ctx.check_device()
        w = eng.W.download(np.float32, (eng.n_train,))
        eng.close()
        return np.array(losses), w

    l0, w0 = run("resident")
    for mode in ("host", "prefetch"):
        l, w = run(mode)
        assert np.allclose(l, l0, rtol=1e-6), (mode, l, l0)
        assert np.array_equal(w, w0), mode


def test_head_fusion_is_bit_identical(ctx):
    """The logits conv fused into the last normalisation pass (bsl_norm_apply_head) and the logits-layer dgrad recomputed
    inside the last layer's normalisation backward (bsl_norm_bwd_*_head), each on or off: logits, loss and every
    gradient are bit-identical to the unfused passes."""
    from boxsegliver_b200.engine import EngineConfig, UNetEngine
    n, hw = 8, 64
    images, labels = synthetic.make_batch(n, hw, hw, 3, seed=1401)
    out = []
    for head, head_bwd in ((False, False), (True, False), (True, True), (False, True)):
        eng = UNetEngine(ctx, EngineConfig(batch=n, height=hw, width=hw, weight_decay_rate=1e-5,
                                           loss_weight_type="numerical", loss_numeric_w=(0.2, 0.4, 4.4)))
        eng._fuse_head, eng._fuse_head_bwd = head, head_bwd
        eng.init_weights(seed=5)
        eng.set_inputs(images, labels)
        for _ in range(2):
            eng.train_step(1e-3)
        ctx.check_device()
        out.append((eng.logits.download(np.float32, (n, hw, hw, 3)), eng.read_loss(), eng.get_grads()))
        eng.close()
    for other in out[1:]:
        assert np.array_equal(out[0][0], other[0])
        assert out[0][1] == other[1]          # (data loss, L2 term)
        for k, g in out[0][2].items():
            assert np.array_equal(g, other[2][k]), k
