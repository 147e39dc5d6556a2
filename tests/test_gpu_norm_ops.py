"""Op-level parity of the normalisation passes of csrc/norm.cu that the plain op tests (test_gpu_ops.py) do not reach:
GUNet's guide modulation (instance norm and batch norm), the folded after_affine, the last layer fused with the logits
conv, and the shape-selected kernel variants (1 / 2 guide channels, channel counts that do not divide the 256-thread
block, more samples than a block has lanes, grids capped below the work). Each case calls the C ABI in the order the
engines do (gunet_engine.py _modulate / _norm_backward_reduce / _norm_backward_apply, engine.py's head fusion) and
compares with the fp64 reference tests/norm_ref.py.

Gates (relative L2 unless stated; "per row" = per sample, per guide channel): activations and dx <= 5e-3; mean / rstd /
scale / shift / moving statistics <= 1e-5 per row; dgamma, dbeta, dga, dba, dbias_guide <= 1e-4; dgamma_mod and
dw_guide <= 1e-4 per row. The ReLU gate of the reference is the device's stored activation > 0. Every output is
surrounded by canaries (unused lanes of strided views, a guard region after the end), and every case runs twice with
bit-identical results.

Grid arithmetic in the comments is for 148 SMs: elementwise passes cap at 16 * 148 / groups blocks, the 8-channel
reductions at 4 * 148 / groups, the 4-channel backward reduce at 8 * 148 / groups."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from boxsegliver_b200.device import bf16_bits_to_f32, round_bf16
from oracle import tf_ops as O
from tests import norm_ref as R
from tests.gpu_util import rel

pytestmark = pytest.mark.gpu

BSL_EUNSUPPORTED = -2
GUARD = 256                     # canary elements after every output
_BITS = {2: np.uint16, 4: np.uint32, 8: np.uint64}
_CANARY = {2: 0xABCD, 4: 0x7FBADBAD, 8: 0x7FF0DEADBEEF0BAD}   # bf16 -1.5e-12, fp32 / fp64 NaN payloads
GM_OFF = 8                      # the layer's slice of the context-MLP output starts at this column


class Out:
    """Output operand of `rows` x `width` elements inside a buffer of `rows` x `ld` elements (lanes [off, off + width)
    of each row) followed by GUARD elements; the whole buffer starts as a canary, or the operand as `init` (values of
    its element size, for kernels that work in place)."""

    def __init__(self, ctx, rows, width, ld=None, off=0, esize=4, init=None):
        self.rows, self.width, self.ld, self.off, self.esize = rows, width, ld or width, off, esize
        self.bits = _BITS[esize]
        self.total = rows * self.ld + GUARD
        host = np.full(self.total, _CANARY[esize], self.bits)
        if init is not None:
            host[:rows * self.ld].reshape(rows, self.ld)[:, off:off + width] = \
                np.asarray(init).view(self.bits).reshape(rows, width)
        self.buf = ctx.from_numpy(host)

    @property
    def p(self):
        return C.c_void_p(self.buf.ptr + self.off * self.esize)

    def raw(self):
        """Bit patterns of the operand [rows, width]; every other lane and the guard must still hold the canary."""
        r = self.buf.download(self.bits, (self.total,))
        body = r[:self.rows * self.ld].reshape(self.rows, self.ld)
        can = self.bits(_CANARY[self.esize])
        assert (r[self.rows * self.ld:] == can).all(), "a store past the end of an output"
        assert (body[:, :self.off] == can).all() and (body[:, self.off + self.width:] == can).all(), \
            "a store into a lane outside the operand"
        return body[:, self.off:self.off + self.width].copy()

    def get(self):
        r = self.raw()
        if self.esize == 2:
            return bf16_bits_to_f32(r).reshape(r.shape)
        return r.view({4: np.float32, 8: np.float64}[self.esize])


def _bf16_strided(ctx, a, ld, fill):
    """[pixels, c] values in a bf16 buffer of row pitch ld; lanes >= c hold `fill` (a kernel reading them would show)."""
    buf = np.full((a.shape[0], ld), fill, np.float32)
    buf[:, :a.shape[1]] = a
    return ctx.bf16_from_f32(buf)


def _rows_rel(got, ref):
    got, ref = np.atleast_2d(got), np.atleast_2d(ref)
    return max(rel(g, r) for g, r in zip(got, ref))


# ------------------------------------------------------------------ modulated / affine / batch-modulated / plain layers
# kind: "mod" = instance norm + modulation (bsl_norm_modulate, finalize_mod), "affine" = the same with after_affine
# (affine_fold, finalize_affine), "bnmod" = batch norm with per-sample modulation (modulate_bn, finalize_bnmod,
# apply_bnmod on the mode-1 view), "plain" = no modulation (bsl_norm_apply[_pool], bwd_reduce / finalize / apply).
def _case(cid, kind, n, h, w, c, G=0, gm=False, mode="instance", pool=False, relu=True, center=True, scale=True,
          strided=False, dropped=False):
    return pytest.param(dict(kind=kind, mode="batch" if kind == "bnmod" else mode, n=n, h=h, w=w, c=c, G=G, gm=gm,
                             pool=pool, relu=relu, center=center, scale=scale, strided=strided, dropped=dropped), id=cid)


CASES = [
    # apply_pool<1>: 3 samples x 96 pooled px, rows 32 -> 3 blocks of 256; BwdFG<1>; bwd apply4g<4,1> (256 % 16 == 0)
    _case("M1", "mod", 3, 16, 24, 64, G=1, gm=True, pool=True),
    # apply<2>, bwd apply4g<2,2>; no centre (beta absent); dy / dx with row pitch 2c
    _case("M2", "mod", 2, 12, 20, 128, G=2, center=False, strided=True),
    # c = 320: 256 % 80 != 0 -> generic 8-channel norm_bwd_apply_kernel<2>, BwdFG<2> with 240-thread blocks
    _case("M3", "mod", 3, 8, 8, 320, G=2, gm=True),
    # c = 1024: 128 8-channel groups -> 2 pixel rows per apply block, 256 4-channel groups -> 1 row per apply4g block
    _case("M4", "mod", 2, 6, 6, 1024, G=1, gm=True),
    # n = 40 > FM_S = 32 sample lanes of finalize_mod. Caps (groups = 40): apply want 9216 / (32 * 4) = 72 > 2368 / 40
    # -> 60 blocks; pool want 2304 / 32 = 72 > 60; bwd apply4g want 9216 / 64 = 144 > 60; BwdFG want 18 > 592 / 40 -> 15
    _case("M5", "mod", 40, 96, 96, 64, G=1, gm=True),
    # gamma_mod without a guide: modulate scales only, the passes take the un-guided kernels; no ReLU
    _case("M6", "mod", 3, 16, 16, 64, gm=True, relu=False),
    # the dropped-layer call: finalize_mod with gamma = beta = NULL under a descriptor with centre = scale = 1
    _case("M7", "mod", 2, 16, 16, 64, G=1, gm=True, dropped=True),
    # affine_fold + finalize_affine with a guide (after_affine layers have neither centre nor scale)
    _case("A1", "affine", 3, 16, 16, 64, G=1, gm=True, center=False, scale=False),
    # w_eff of two guide channels; the norm's own gamma / beta present
    _case("A2", "affine", 2, 16, 16, 128, G=2),
    # 34 samples through finalize_affine's serial sample loop; scale without centre
    _case("A3", "affine", 34, 32, 32, 64, gm=True, center=False),
    # modulate_bn, finalize_bnmod, premul norm_bwd_apply_kernel<1>; moving statistics with decay 0.99
    _case("B1", "bnmod", 3, 16, 16, 64, G=1, gm=True),
    # premul on the generic c = 320 kernel with two guide channels
    _case("B2", "bnmod", 4, 8, 8, 320, G=2, gm=True),
    # 40 samples: modulate_bn's and finalize_bnmod's sample loops; stats want 92160 * 128 / 32768 = 360 blocks (< 592)
    _case("B3", "bnmod", 40, 48, 48, 128, gm=True),
    # 40 groups: norm_bwd_finalize takes glanes = 32 and loops g += 32. Caps: stats want 18 > 15, apply 72 > 60,
    # bwd apply4 want 9216 / 64 = 144 > 60
    _case("P1", "plain", 40, 96, 96, 64),
    # batch, 131072 px: reduce4 want 131072 * 64 / 32768 = 256 blocks (cap 1184) -> the final reduce's 4-way loop
    # (more than 96 partial blocks); stats also 256 blocks (cap 592)
    _case("P2", "plain", 8, 128, 128, 64, mode="batch"),
    # c = 24: 3 channel groups -> 255-thread blocks; 256 % 6 != 0 -> BwdFG<0> and norm_bwd_apply_kernel<0>
    _case("P3-inst-24", "plain", 3, 10, 10, 24, strided=True),
    _case("P3-batch-24", "plain", 3, 10, 10, 24, mode="batch", pool=True),
    # c = 320: 40 groups -> 240-thread blocks; generic kernels
    _case("P3-inst-320", "plain", 3, 10, 10, 320, pool=True),
    _case("P3-batch-320", "plain", 3, 10, 10, 320, mode="batch", strided=True),
]


def _host(cs, seed):
    rng = np.random.default_rng(seed)
    n, h, w, c, G = cs["n"], cs["h"], cs["w"], cs["c"], cs["G"]
    gm_ld = c + 2 * GM_OFF
    y = rng.standard_normal((n, h, w, c), dtype=np.float32) * np.float32(1.3)
    y += (rng.standard_normal((n, 1, 1, c)) * 0.8).astype(np.float32)           # distinct moments per sample
    # the incoming gradient has a mean and a component along y per (sample, channel): the c1 / c2 terms of the backward
    # then weigh as much at 92160 values per channel as at 768 (with white noise they fade as 1 / sqrt(values))
    da = rng.standard_normal((n, h, w, c), dtype=np.float32) + rng.normal(0, 0.5, (n, 1, 1, c)).astype(np.float32)
    da += np.float32(0.3) * y
    return dict(
        y=round_bf16(y),
        gamma=rng.uniform(0.5, 1.5, c).astype(np.float32), beta=rng.normal(0, 0.3, c).astype(np.float32),
        mm=rng.normal(0, 0.2, c).astype(np.float32), mv=rng.uniform(0.5, 1.5, c).astype(np.float32),
        gm_buf=rng.uniform(0.5, 1.5, (n, gm_ld)).astype(np.float32),
        guide=rng.uniform(0, 1, (n, h, w, max(G, 1))).astype(np.float32)[..., :G],
        w_buf=rng.normal(0, 0.5, (max(G, 1), 2 * c)).astype(np.float32),     # the layer's columns: [c, 2c)
        b_guide=rng.normal(0, 0.3, c).astype(np.float32),
        ga=rng.uniform(0.5, 1.5, c).astype(np.float32), ba=rng.normal(0, 0.3, c).astype(np.float32),
        da=round_bf16(da.reshape(n * h * w, c)))


def _run_layer(ctx, cs, hs):
    """One forward and backward of the layer on the device; returns every output (and the in-place parameter arrays
    after each stage) as numpy arrays."""
    kind, n, h, w, c, G = cs["kind"], cs["n"], cs["h"], cs["w"], cs["c"], cs["G"]
    hw, P = h * w, n * h * w
    inst = cs["mode"] == "instance"
    ld = 2 * c if cs["strided"] else c
    gm_ld = hs["gm_buf"].shape[1]
    eps, decay = (1e-6, 0.999) if inst else (1e-3, 0.99)
    center, scale = (1, 1) if cs["dropped"] else (int(cs["center"]), int(cs["scale"]))
    d = _lib.NormDesc(1 if inst else 0, n, hw, c, c, ld, eps, decay, int(cs["relu"]), center, scale)
    dv = _lib.NormDesc(1, n, hw, c, c, ld, eps, decay, int(cs["relu"]), center, scale)   # per-sample view (bnmod)
    da_ = dv if kind == "bnmod" else d
    res, bufs = {}, []

    def up(a):
        b = ctx.from_numpy(np.ascontiguousarray(a))
        bufs.append(b)
        return b

    def out(*a, **k):
        o = Out(ctx, *a, **k)
        bufs.append(o.buf)
        return o

    y = ctx.bf16_from_f32(hs["y"].reshape(P, c))
    bufs.append(y)
    gamma = up(np.ones(c, np.float32) if cs["dropped"] else hs["gamma"]) if scale else None
    beta = up(np.zeros(c, np.float32) if cs["dropped"] else hs["beta"]) if center else None
    gmb = up(hs["gm_buf"]) if cs["gm"] else None
    gm = C.c_void_p(gmb.ptr + GM_OFF * 4) if gmb else None
    gmap = up(hs["guide"]) if G else None
    wb = up(hs["w_buf"]) if G else None
    wsp = C.c_void_p(wb.ptr + c * 4) if G else None          # w[g * 2c + c + ch]: w_ld = 2c, as in the filter arena
    bsp = up(hs["b_guide"]) if G else None
    ga, ba = (up(hs["ga"]), up(hs["ba"])) if kind == "affine" else (None, None)
    mm, mv = (up(hs["mm"]), up(hs["mv"])) if not inst else (None, None)
    groups = n if inst else 1
    pbuf = lambda b: b.p if b is not None else None  # noqa: E731

    sums = out(groups, 2 * c, esize=8)
    ctx.call("bsl_norm_stats", C.byref(d), y.p, sums.p, ctx.stream)
    res["sums_fwd"] = sums.get()
    q = {k: out(n, c) for k in ("mean", "rstd", "scale", "shift", "c1", "c2")}
    ctx.call("bsl_norm_finalize", C.byref(d), C.c_int(1), sums.p, pbuf(gamma), pbuf(beta), pbuf(mm), pbuf(mv),
             q["mean"].p, q["rstd"].p, q["scale"].p, q["shift"].p, ctx.stream)
    for k in ("mean", "rstd", "scale", "shift"):
        res[f"fin_{k}"] = q[k].get()[:groups]      # batch mode writes the first c entries only
    if mm is not None:
        res["moving_mean"], res["moving_var"] = mm.download(np.float32, (c,)), mv.download(np.float32, (c,))
    if kind != "plain" and (cs["gm"] or G):
        if kind == "bnmod":
            ctx.call("bsl_norm_modulate_bn", C.byref(dv), gm, C.c_int(gm_ld), pbuf(bsp), q["mean"].p, q["rstd"].p,
                     q["scale"].p, q["shift"].p, ctx.stream)
        else:
            ctx.call("bsl_norm_modulate", C.byref(d), gm, C.c_int(gm_ld), pbuf(bsp), q["scale"].p, q["shift"].p,
                     ctx.stream)
        for k in ("mean", "rstd", "scale", "shift"):
            res[f"mod_{k}"] = q[k].get()
    guide = _lib.Guide(gmap.ptr, G, wsp.value, 2 * c) if G else None
    if kind == "affine":
        sp, hp = out(n, c), out(n, c)
        weff = out(G, c) if G else None
        ctx.call("bsl_norm_affine_fold", C.byref(d), ga.p, ba.p, q["scale"].p, q["shift"].p, sp.p, hp.p, wsp,
                 C.c_int(2 * c), C.c_int(G), weff.p if G else None, ctx.stream)
        res["fold_scale"], res["fold_shift"] = q["scale"].get(), q["shift"].get()
        res["scale_pre"], res["shift_pre"] = sp.get(), hp.get()
        if G:
            res["w_eff"] = weff.get()
            guide = _lib.Guide(gmap.ptr, G, weff.p.value, c)     # the passes read the gamma_a-scaled filter
    gp = C.byref(guide) if guide is not None else None

    a = out(P, c, ld=ld, esize=2)
    if cs["pool"]:
        pooled = out(P // 4, c, ld=2 * c, esize=2)              # the lower half of a concat buffer
        ctx.call("bsl_norm_apply_pool_mod", C.byref(da_), C.c_int(h), C.c_int(w), y.p, q["scale"].p, q["shift"].p, gp,
                 a.p, pooled.p, C.c_int(2 * c), ctx.stream)
        res["pooled"] = pooled.get()
    else:
        ctx.call("bsl_norm_apply_mod", C.byref(da_), y.p, q["scale"].p, q["shift"].p, gp, a.p, ctx.stream)
    res["a"] = a.get()

    dy = _bf16_strided(ctx, hs["da"], ld, 1e4)
    bufs.append(dy)
    K = 2 + G
    sb = out(n if da_.mode else 1, K * c, esize=8)
    ctx.call("bsl_norm_bwd_reduce_mod", C.byref(da_), y.p, dy.p, C.c_int(ld), q["mean"].p, q["rstd"].p, q["scale"].p,
             q["shift"].p, gp, sb.p, ctx.stream)
    g = dict(dgamma=out(1, c) if scale and not cs["dropped"] else None,
             dbeta=out(1, c) if center and not cs["dropped"] else None,
             dgamma_mod=out(n, c, ld=gm_ld, off=GM_OFF) if cs["gm"] else None,
             dw_guide=out(G, c, ld=2 * c, off=c) if G else None, dbias_guide=out(1, c) if G else None)
    gpt = {k: (v.p if v is not None else None) for k, v in g.items()}
    if kind == "plain":
        ctx.call("bsl_norm_bwd_finalize", C.byref(d), sb.p, q["c1"].p, q["c2"].p, gpt["dgamma"], gpt["dbeta"],
                 ctx.stream)
    elif cs["dropped"]:
        ctx.call("bsl_norm_bwd_finalize_mod", C.byref(d), sb.p, C.c_int(G), gm, C.c_int(gm_ld), None, None, q["c1"].p,
                 q["c2"].p, None, None, gpt["dgamma_mod"], gpt["dw_guide"], C.c_int(2 * c), gpt["dbias_guide"],
                 ctx.stream)
    elif kind == "affine":
        g["dga"], g["dba"] = out(1, c), out(1, c)
        ctx.call("bsl_norm_bwd_finalize_affine", C.byref(d), sb.p, C.c_int(G), gm, C.c_int(gm_ld), pbuf(gamma),
                 pbuf(beta), ga.p, q["mean"].p, q["rstd"].p, sp.p, hp.p, wsp, C.c_int(2 * c), q["c1"].p, q["c2"].p,
                 gpt["dgamma"], gpt["dbeta"], gpt["dgamma_mod"], gpt["dw_guide"], C.c_int(2 * c), gpt["dbias_guide"],
                 g["dga"].p, g["dba"].p, ctx.stream)
    elif kind == "bnmod":
        ctx.call("bsl_norm_bwd_finalize_bnmod", C.byref(dv), sb.p, C.c_int(G), gm, C.c_int(gm_ld), pbuf(gamma),
                 pbuf(beta), q["rstd"].p, q["c1"].p, q["c2"].p, gpt["dgamma"], gpt["dbeta"], gpt["dgamma_mod"],
                 gpt["dw_guide"], C.c_int(2 * c), gpt["dbias_guide"], ctx.stream)
    else:
        ctx.call("bsl_norm_bwd_finalize_mod", C.byref(d), sb.p, C.c_int(G), gm, C.c_int(gm_ld), pbuf(gamma),
                 pbuf(beta), q["c1"].p, q["c2"].p, gpt["dgamma"], gpt["dbeta"], gpt["dgamma_mod"], gpt["dw_guide"],
                 C.c_int(2 * c), gpt["dbias_guide"], ctx.stream)
    dx = out(P, c, ld=ld, esize=2)
    ctx.call("bsl_norm_bwd_apply_bnmod" if kind == "bnmod" else "bsl_norm_bwd_apply_mod", C.byref(da_), y.p, dy.p,
             C.c_int(ld), q["mean"].p, q["rstd"].p, q["scale"].p, q["shift"].p, q["c1"].p, q["c2"].p, gp, dx.p,
             C.c_int(ld), ctx.stream)
    ctx.check_device()
    res["sums_bwd"], res["c1"], res["c2"], res["dx"] = sb.get(), q["c1"].get(), q["c2"].get(), dx.get()
    for k, v in g.items():
        if v is not None:
            res[k] = v.get()
    for b in bufs:
        b.free()
    return res


def _check_layer(cs, hs, res):
    n, h, w, c, G = cs["n"], cs["h"], cs["w"], cs["c"], cs["G"]
    inst = cs["mode"] == "instance"
    eps, decay = (1e-6, 0.999) if inst else (1e-3, 0.99)
    f8 = lambda a: np.asarray(a, np.float64)  # noqa: E731
    gm = f8(hs["gm_buf"][:, GM_OFF:GM_OFF + c]) if cs["gm"] else None
    w_guide = f8(hs["w_buf"][:G, c:])
    gamma = f8(hs["gamma"]) if cs["scale"] and not cs["dropped"] else None
    beta = f8(hs["beta"]) if cs["center"] and not cs["dropped"] else None
    affine = cs["kind"] == "affine"
    f = R.forward(hs["y"], cs["mode"], eps, gamma, beta, gm, hs["guide"] if G else None, w_guide if G else None,
                  hs["b_guide"] if G else None, hs["ga"] if affine else None, hs["ba"] if affine else None, cs["relu"],
                  moving=None if inst else (hs["mm"], hs["mv"]), decay=decay)
    errs = {}
    # per-(sample, channel) affine after each stage, from the fp64 moments
    mean, rstd = np.atleast_2d(f["mean"]), np.atleast_2d(f["rstd"])
    sc = (gamma if gamma is not None else 1.0) * rstd
    sh = (beta if beta is not None else 0.0) - mean * sc
    stages = [("fin", mean, rstd, sc, sh)]
    if "mod_scale" in res:
        rows = lambda a: np.broadcast_to(a, (n, c))  # noqa: E731
        sc = rows(sc) * (gm if gm is not None else 1.0)
        sh = rows(sh) * (gm if gm is not None else 1.0) + (f8(hs["b_guide"]) if G else 0.0)
        stages.append(("mod", rows(mean), rows(rstd), sc, sh))
    for tag, m_, r_, sc_, sh_ in stages:
        for k, ref in (("mean", m_), ("rstd", r_), ("scale", sc_), ("shift", sh_)):
            if f"{tag}_{k}" in res and (tag == "fin" or k in ("scale", "shift") or cs["kind"] == "bnmod"):
                errs[f"{tag}_{k}"] = (_rows_rel(res[f"{tag}_{k}"], ref), 1e-5)
    if affine:
        errs["scale_pre"], errs["shift_pre"] = (_rows_rel(res["scale_pre"], sc), 1e-5), (_rows_rel(res["shift_pre"], sh), 1e-5)
        errs["fold_scale"] = (_rows_rel(res["fold_scale"], sc * f8(hs["ga"])), 1e-5)
        errs["fold_shift"] = (_rows_rel(res["fold_shift"], sh * f8(hs["ga"]) + f8(hs["ba"])), 1e-5)
        if G:
            errs["w_eff"] = (_rows_rel(res["w_eff"], w_guide * f8(hs["ga"])), 1e-5)
    if not inst:
        errs["moving_mean"] = (rel(res["moving_mean"], f["moving_mean"]), 1e-5)
        errs["moving_var"] = (rel(res["moving_var"], f["moving_var"]), 1e-5)
    a = res["a"].reshape(n, h, w, c)
    errs["a"] = (rel(a, f["a"]), 5e-3)
    if cs["pool"]:
        assert np.array_equal(res["pooled"].reshape(n, h // 2, w // 2, c), O.max_pool_2x2(a)), \
            "pooled tensor must be the exact max of the stored activation"
    b = R.backward(f, da=hs["da"].reshape(n, h, w, c), mask=a > 0 if cs["relu"] else None)
    errs["dx"] = (rel(res["dx"].reshape(n, h, w, c), b["dy"]), 5e-3)
    for k in ("dgamma", "dbeta", "dbias_guide", "dga", "dba"):
        if k in res:
            errs[k] = (rel(res[k][0], b[k]), 1e-4)
    for k in ("dgamma_mod", "dw_guide"):
        if k in res:
            errs[k] = (_rows_rel(res[k], b[k]), 1e-4)
    bad = {k: v for k, v in errs.items() if not v[0] <= v[1]}
    assert not bad, f"over the gate: {bad}"


@pytest.mark.parametrize("cs", CASES)
def test_norm_layer_op_parity(ctx, cs):
    hs = _host(cs, seed=cs["n"] * 7 + cs["c"] + cs["G"])
    r1 = _run_layer(ctx, cs, hs)
    _check_layer(cs, hs, r1)
    r2 = _run_layer(ctx, cs, hs)
    assert r1.keys() == r2.keys()
    for k in r1:      # fixed-order reductions, no atomics: every output and every fp64 sum bit-identical
        assert np.array_equal(r1[k].view(_BITS[r1[k].dtype.itemsize]), r2[k].view(_BITS[r2[k].dtype.itemsize])), k


# ------------------------------------------------------------------ last normalised layer fused with the logits conv
HEAD = [pytest.param(m, n, h, w, c, k, relu, id=f"{m}-{n}x{h}x{w}-c{c}-k{k}-relu{relu}")
        for m in ("instance", "batch") for (n, h, w) in ((3, 7, 13),) for c in (8, 64, 256) for k in (2, 3, 4)
        for relu in (1, 0)]
# 2 x 256 x 256: grid-stride loops. apply_head (c = 64: rows 32, want 65536 / 128 = 512 blocks per group, stride
# 16384 px, 2 px per thread per trip -> 2 trips per group; c = 256: want 2048 > 1184 / 2 = 592 blocks, 6.9 trips with a
# masked tail); reduce4 (instance: want 128 blocks per group, cap 592); apply4 (want 1024 per group > 592)
HEAD += [pytest.param(m, 2, 256, 256, c, k, relu, id=f"{m}-2x256x256-c{c}-k{k}-relu{relu}")
         for m, c, k, relu in (("instance", 64, 2, 1), ("instance", 64, 3, 0), ("instance", 64, 4, 1),
                               ("batch", 64, 2, 0), ("batch", 64, 3, 1), ("batch", 64, 4, 1),
                               ("instance", 256, 3, 1), ("batch", 8, 4, 0))]


def _run_head(ctx, mode, n, h, w, c, classes, relu, hs):
    """The fused passes and the unfused ones they replace, on the same inputs."""
    P = n * h * w
    inst = mode == "instance"
    d = _lib.NormDesc(1 if inst else 0, n, h * w, c, c, c, 1e-6 if inst else 1e-3, 0.999, relu, 1, 1)
    cd = _lib.Conv2dDesc(n, h, w, c, classes, 1, 1, c, classes)
    groups = n if inst else 1
    res, bufs = {}, []

    def up(a):
        bufs.append(ctx.from_numpy(np.ascontiguousarray(a)))
        return bufs[-1]

    def out(*a, **k):
        o = Out(ctx, *a, **k)
        bufs.append(o.buf)
        return o

    y = ctx.bf16_from_f32(hs["y"].reshape(P, c))
    bufs.append(y)
    gamma, beta, wh, bh, dl = up(hs["gamma"]), up(hs["beta"]), up(hs["wh"]), up(hs["bh"]), up(hs["dl"])
    mm, mv = up(hs["mm"]), up(hs["mv"])
    sums = out(groups, 2 * c, esize=8)
    q = {k: out(groups, c) for k in ("mean", "rstd", "scale", "shift", "c1", "c2", "c1u", "c2u")}
    ctx.call("bsl_norm_stats", C.byref(d), y.p, sums.p, ctx.stream)
    ctx.call("bsl_norm_finalize", C.byref(d), C.c_int(1), sums.p, gamma.p, beta.p, None if inst else mm.p,
             None if inst else mv.p, q["mean"].p, q["rstd"].p, q["scale"].p, q["shift"].p, ctx.stream)
    a1, a2 = out(P, c, esize=2), out(P, c, esize=2)
    l1, l2 = out(P, classes), out(P, classes)
    ctx.call("bsl_norm_apply_head", C.byref(d), y.p, q["scale"].p, q["shift"].p, a1.p, wh.p, bh.p, C.c_int(classes),
             l1.p, ctx.stream)
    ctx.call("bsl_norm_apply", C.byref(d), y.p, q["scale"].p, q["shift"].p, a2.p, ctx.stream)
    ctx.call("bsl_conv2d_head_fprop", C.byref(cd), a2.p, wh.p, bh.p, l2.p, ctx.stream)
    s1, s2 = out(groups, 2 * c, esize=8), out(groups, 2 * c, esize=8)
    dx1, dx2 = out(P, c, esize=2), out(P, c, esize=2)
    dg1, db1, dg2, db2 = (out(1, c) for _ in range(4))
    ctx.call("bsl_norm_bwd_reduce_head", C.byref(d), y.p, dl.p, wh.p, C.c_int(classes), q["mean"].p, q["rstd"].p,
             q["scale"].p, q["shift"].p, s1.p, ctx.stream)
    ctx.call("bsl_norm_bwd_finalize", C.byref(d), s1.p, q["c1"].p, q["c2"].p, dg1.p, db1.p, ctx.stream)
    ctx.call("bsl_norm_bwd_apply_head", C.byref(d), y.p, dl.p, wh.p, C.c_int(classes), q["mean"].p, q["rstd"].p,
             q["scale"].p, q["shift"].p, q["c1"].p, q["c2"].p, dx1.p, C.c_int(c), ctx.stream)
    da = out(P, c, esize=2)
    ctx.call("bsl_conv2d_head_dgrad", C.byref(cd), dl.p, wh.p, da.p, ctx.stream)
    ctx.call("bsl_norm_bwd_reduce", C.byref(d), y.p, da.p, C.c_int(c), q["mean"].p, q["rstd"].p, q["scale"].p,
             q["shift"].p, s2.p, ctx.stream)
    ctx.call("bsl_norm_bwd_finalize", C.byref(d), s2.p, q["c1u"].p, q["c2u"].p, dg2.p, db2.p, ctx.stream)
    ctx.call("bsl_norm_bwd_apply", C.byref(d), y.p, da.p, C.c_int(c), q["mean"].p, q["rstd"].p, q["scale"].p,
             q["shift"].p, q["c1u"].p, q["c2u"].p, dx2.p, C.c_int(c), ctx.stream)
    ctx.check_device()
    for k, o in dict(a=a1, a_unfused=a2, logits=l1, logits_unfused=l2, da=da, sums=s1, sums_unfused=s2, dx=dx1,
                     dx_unfused=dx2, dgamma=dg1, dbeta=db1, dgamma_unfused=dg2, dbeta_unfused=db2).items():
        res[k] = o.raw()
    for b in bufs:
        b.free()
    return res


@pytest.mark.parametrize("mode,n,h,w,c,classes,relu", HEAD)
def test_norm_head_fusion_op_parity(ctx, mode, n, h, w, c, classes, relu):
    rng = np.random.default_rng(c + 10 * classes + relu + h)
    P = n * h * w
    y = rng.standard_normal((n, h, w, c), dtype=np.float32) + (rng.standard_normal((n, 1, 1, c)) * 0.5).astype(np.float32)
    hs = dict(y=round_bf16(y), gamma=rng.uniform(0.5, 1.5, c).astype(np.float32),
              beta=rng.normal(0, 0.3, c).astype(np.float32), mm=np.zeros(c, np.float32), mv=np.ones(c, np.float32),
              wh=(rng.standard_normal((c, classes)) / np.sqrt(c)).astype(np.float32),
              bh=rng.normal(0, 0.3, classes).astype(np.float32),
              dl=rng.standard_normal((P, classes), dtype=np.float32))
    r = _run_head(ctx, mode, n, h, w, c, classes, relu, hs)
    # the header's promise: bit-identical to the unfused passes
    for k in ("a", "logits", "sums", "dx", "dgamma", "dbeta"):
        assert np.array_equal(r[k], r[f"{k}_unfused"]), k
    f = R.forward(hs["y"], mode, 1e-6 if mode == "instance" else 1e-3, hs["gamma"], hs["beta"], relu=bool(relu),
                  w_head=hs["wh"], b_head=hs["bh"])
    a = bf16_bits_to_f32(r["a"]).reshape(n, h, w, c)
    assert rel(a, f["a"]) < 5e-3
    logits = r["logits"].view(np.float32).reshape(n, h, w, classes)
    assert rel(logits, a.astype(np.float64) @ hs["wh"].astype(np.float64) + hs["bh"]) < 1e-5
    # the activation gradient is bf16(dlogits @ w_head^T), as bsl_conv2d_head_dgrad stores it: the reference backward
    # starts from the device's rounding of it (an fp64 one differs by 2^-9 per element, 1e-3 on the sums)
    da = bf16_bits_to_f32(r["da"]).reshape(n, h, w, c)
    assert rel(da, hs["dl"].reshape(n, h, w, classes).astype(np.float64) @ hs["wh"].T.astype(np.float64)) < 5e-3
    b = R.backward(f, da=da, mask=a > 0 if relu else None)
    assert rel(bf16_bits_to_f32(r["dx"]).reshape(n, h, w, c), b["dy"]) < 5e-3
    assert rel(r["dgamma"].view(np.float32), b["dgamma"]) < 1e-4
    assert rel(r["dbeta"].view(np.float32), b["dbeta"]) < 1e-4
    r2 = _run_head(ctx, mode, n, h, w, c, classes, relu, hs)
    for k in r:
        assert np.array_equal(r[k], r2[k]), k


def test_norm_head_domain(ctx):
    """bsl_norm_bwd_head_ok is 1 exactly on c in {8, .., 256} with 256 % (c / 4) == 0 and classes 2..4;
    bsl_norm_apply_head refuses channel counts and class counts outside its kernels (return codes only: the refusals
    come before any launch)."""
    for c in range(8, 1025, 8):
        d = _lib.NormDesc(1, 2, 16, c, c, c, 1e-6, 0.999, 1, 1, 1)
        for classes in range(0, 7):
            want = int(c <= 256 and 256 % (c // 4) == 0 and 2 <= classes <= 4)
            assert ctx.lib.bsl_norm_bwd_head_ok(ctx.h, C.byref(d), C.c_int(classes)) == want, (c, classes)
    for c in (24, 320, 512):
        d = _lib.NormDesc(1, 2, 16, c, c, c, 1e-6, 0.999, 1, 1, 1)
        assert ctx.lib.bsl_norm_bwd_head_ok(ctx.h, C.byref(d), C.c_int(3)) == 0
    buf = ctx.alloc(1 << 16)
    p = buf.p
    for c, classes in ((24, 3), (512, 3), (64, 5), (64, 1)):
        d = _lib.NormDesc(1, 2, 16, c, c, c, 1e-6, 0.999, 1, 1, 1)
        rc = ctx.lib.bsl_norm_apply_head(ctx.h, C.byref(d), p, p, p, p, p, p, C.c_int(classes), p, ctx.stream)
        assert rc == BSL_EUNSUPPORTED, (c, classes, rc)
    ctx.check_device()
    buf.free()
