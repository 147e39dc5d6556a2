"""The parameter arenas and weight I/O that engine_base.EngineBase gives the 2-D and 3-D engines, checked on the CPU
against the in-memory fake context: TF-shaped variables round-trip bit-exactly through W, G and the optimizer slots,
every stored element outside the variables (pad lanes, the stem's reserved rows, UNetInter's 66 -> 128 lanes) is zero,
the regions are laid out A, B, then S apart, both engines reject a bad training config with the same error, and a
whole training step enqueues."""
import dataclasses

import numpy as np
import pytest

from boxsegliver_b200.engine import EngineConfig, UNetEngine
from boxsegliver_b200.gunet_engine import GUNetConfig, GUNetEngine, UNetInterConfig, UNetInterEngine
from boxsegliver_b200.unet3d_engine import UNet3DConfig, UNet3DEngine
from tests.fake_ctx import FakeContext

TWO_D = dict(batch=2, height=32, width=32, num_down_samples=2)
THREE_D = dict(batch=1, depth=4, height=32, width=32, max_channels=128)

CONFIGS = {
    "unet_bn": (UNetEngine, EngineConfig(**TWO_D, normalizer="batch_norm")),
    "unet_in": (UNetEngine, EngineConfig(**TWO_D, normalizer="instance_norm")),
    "unet_without_norm": (UNetEngine, EngineConfig(**TWO_D, without_norm=True)),
    "gunet_in": (GUNetEngine, GUNetConfig(**TWO_D, mod_layers=(1, 2))),
    "gunet_bn_affine_dropout": (GUNetEngine, GUNetConfig(**TWO_D, mod_layers=(1, 2), normalizer="batch_norm",
                                                         after_affine=True, dropout=0.3)),
    "unetinter_mid_cat": (UNetInterEngine, UNetInterConfig(**TWO_D, mid_cat=True)),
    "unet3d_in_pair": (UNet3DEngine, UNet3DConfig(**THREE_D, normalizer="instance_norm")),
    "unet3d_in_nopair": (UNet3DEngine, UNet3DConfig(**THREE_D, normalizer="instance_norm")),
    "unet3d_bn_pair": (UNet3DEngine, UNet3DConfig(**THREE_D, normalizer="batch_norm")),
    "unet3d_bn_nopair": (UNet3DEngine, UNet3DConfig(**THREE_D, normalizer="batch_norm")),
}


def _engine(name, monkeypatch, **overrides):
    cls, cfg = CONFIGS[name]
    if name.startswith("unet3d"):
        monkeypatch.setenv("BSL_UNET3D_PAIR", "0" if name.endswith("nopair") else "1")
    eng = cls(FakeContext(), dataclasses.replace(cfg, **overrides))
    if name.startswith("unet3d"):
        assert eng._pair == name.endswith("_pair")
    return eng


def _random(eng, seed):
    """Values that are never zero, so a zero in an arena can only be a pad element."""
    rng = np.random.default_rng(seed)
    return {k: rng.uniform(0.5, 1.5, p.shape).astype(np.float32) * rng.choice([-1, 1], p.shape)
            for k, p in eng.params.items()}


def _assert_same(got, want):
    assert got.keys() == want.keys()
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k


@pytest.mark.parametrize("name", list(CONFIGS))
def test_weights_and_grads_round_trip(name, monkeypatch):
    eng = _engine(name, monkeypatch)
    w = _random(eng, 1)
    eng.set_weights(w)
    _assert_same(eng.get_weights(), w)
    eng.G.upload(eng.W.download(np.float32, (eng.n_train,)))
    _assert_same(eng.get_grads(), {k: v for k, v in w.items() if eng.params[k].region != "S"})


@pytest.mark.parametrize("optimizer", ["adam", "momentum"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_slots_round_trip(name, optimizer, monkeypatch):
    eng = _engine(name, monkeypatch, optimizer=optimizer)
    trained = [k for k, p in eng.params.items() if p.region != "S"]
    parts = 2 if optimizer == "adam" else 1
    draws = [_random(eng, 2 + i) for i in range(parts)]
    slots = {k: tuple(d[k] for d in draws) for k in trained}
    eng.set_slots(slots)
    got = eng.get_slots()
    assert got.keys() == slots.keys()
    for k in trained:
        assert len(got[k]) == parts
        for a, b in zip(got[k], slots[k]):
            assert np.array_equal(a, b), k


@pytest.mark.parametrize("name", list(CONFIGS))
def test_arena_elements_outside_the_variables_are_zero(name, monkeypatch):
    eng = _engine(name, monkeypatch)
    eng.set_weights(_random(eng, 3))
    arenas = {"W": eng.W.download(np.float32, (eng.n_train,)), "S": eng.S.download(np.float32, (max(eng.n_stats, 1),))}
    live = {k: np.zeros(a.size, bool) for k, a in arenas.items()}
    for p in eng.params.values():
        idx = np.arange(p.size).reshape(p.stored)[p.sel].ravel() + p.offset
        assert idx.size == int(np.prod(p.shape)), p.name
        live["S" if p.region == "S" else "W"][idx] = True
    for k, a in arenas.items():
        assert not a[~live[k]].any(), k
        assert a[live[k]].all(), k
    if name == "unetinter_mid_cat":
        p = eng.params["UNetInter/Encode/down_conv2/mod_conv1/Conv/weights"]
        assert p.shape[2] == 66 and p.stored[2] == 128


@pytest.mark.parametrize("name", list(CONFIGS))
def test_regions_are_laid_out_a_then_b_and_s_apart(name, monkeypatch):
    eng = _engine(name, monkeypatch)
    assert 0 <= eng.n_reg <= eng.n_train
    bounds = {"A": (0, eng.n_reg), "B": (eng.n_reg, eng.n_train), "S": (0, eng.n_stats)}
    for p in eng.params.values():
        lo, hi = bounds[p.region]
        assert lo <= p.offset and p.offset + max(p.size, p.alloc) <= hi, p.name
        if p.name.endswith("/weights") and "/context/" not in p.name:     # slim l2_regularizer on every conv filter
            assert p.region == "A", p.name
        if p.name.endswith(("/gamma", "/beta")):
            assert p.region == "B", p.name
        if p.name.endswith(("/moving_mean", "/moving_variance")):
            assert p.region == "S", p.name
    for region in "ABS":
        ps = sorted((p for p in eng.params.values() if p.region == region), key=lambda p: p.offset)
        for a, b in zip(ps, ps[1:]):
            assert a.offset + max(a.size, a.alloc) <= b.offset, (a.name, b.name)


@pytest.mark.parametrize("name", list(CONFIGS))
def test_train_step_enqueues(name, monkeypatch):
    eng = _engine(name, monkeypatch)
    eng.init_weights(0)
    eng.ctx.trace.clear()
    eng.train_step(1e-3, with_metrics=True)
    trace = eng.ctx.trace
    assert "bsl_softmax_threshold" in trace and "bsl_wxent_fwd_bwd" in trace
    assert trace[-1] in ("bsl_adam_step", "bsl_momentum_step") and eng.step_count == 1


@pytest.mark.parametrize("bad", [dict(optimizer="sgd"), dict(weight_init="he_normal"), dict(loss_weight_type="log"),
                                 dict(loss_weight_type="numerical", loss_numeric_w=(1.0,))])
def test_both_engines_reject_a_bad_training_config_alike(bad):
    errors = []
    for cls, cfg in (CONFIGS["unet_in"], CONFIGS["unet3d_in_nopair"]):
        with pytest.raises((ValueError, KeyError)) as e:
            cls(FakeContext(), dataclasses.replace(cfg, **bad))
        errors.append((e.type, str(e.value)))
    assert errors[0] == errors[1]
