"""Op-level parity of the after_affine fold and finaliser under every normaliser GUNet runs them with (csrc/norm.cu,
bsl_norm_affine_fold and bsl_norm_bwd_finalize_affine_jac), against the fp64 reference tests/norm_ref.py:

  "bn-mod"   batch norm with per-sample modulation: finalize (mode 0) -> modulate_bn -> fold on the per-sample view ->
             apply -> bwd_reduce_mod -> finalize_affine_jac(BSL_NORM_JAC_BATCH) -> bwd_apply_bnmod
  "bn-plain" an un-modulated batch-norm block: fold of the per-channel scale / shift (mode 0) -> apply ->
             bwd_reduce -> finalize_affine_jac(BSL_NORM_JAC_GROUP) -> bwd_apply
  "ident"    the modulation stage of a --dropout block: identity normaliser (mean 0, rstd 1) -> modulate -> fold ->
             apply -> bwd_reduce_mod -> finalize_affine_jac(BSL_NORM_JAC_NONE, c1 = c2 = 0) -> bwd_apply_mod

Each case calls the C ABI in the order gunet_engine.py does. Gates as tests/test_gpu_norm_ops.py: activations and dx
<= 5e-3; scalars <= 1e-5 per row; dgamma, dbeta, dga, dba, dbias_guide <= 1e-4; dgamma_mod, dw_guide <= 1e-4 per row.
Every output sits between canaries, and every case runs twice with bit-identical results."""
import ctypes as C

import numpy as np
import pytest

from boxsegliver_b200 import _lib
from tests import norm_ref as R
from tests.gpu_util import rel
from tests.test_gpu_norm_ops import _BITS, GM_OFF, Out, _bf16_strided, _host, _rows_rel

pytestmark = pytest.mark.gpu

BSL_EINVAL = -1
JAC_GROUP, JAC_BATCH, JAC_NONE = 0, 1, 2


def _case(cid, kind, n, h, w, c, G=0, gm=False, center=True, scale=True, strided=False):
    return pytest.param(dict(kind=kind, n=n, h=h, w=w, c=c, G=G, gm=gm, center=center, scale=scale, strided=strided),
                        id=cid)


CASES = [
    # modulated batch-norm blocks have neither centre nor scale under after_affine; premul generic kernel (c = 320)
    _case("BM1", "bn-mod", 4, 8, 8, 320, G=2, gm=True, center=False, scale=False),
    # 34 samples through the finaliser's two sample loops; one guide channel; normaliser's own gamma / beta present
    _case("BM2", "bn-mod", 34, 16, 16, 64, G=1, gm=True),
    # gamma_mod without a guide, 40 samples, strided activations
    _case("BM3", "bn-mod", 40, 12, 12, 128, gm=True, center=False, scale=False, strided=True),
    # un-modulated block (centre and scale on): per-channel scalars, c = 320 generic kernels
    _case("BP1", "bn-plain", 3, 10, 10, 320),
    # 40 samples, the 4-channel backward kernels
    _case("BP2", "bn-plain", 40, 24, 24, 64, strided=True),
    _case("ID1", "ident", 3, 8, 8, 320, G=2, gm=True),
    _case("ID2", "ident", 34, 16, 16, 64, G=1, gm=True),
    _case("ID3", "ident", 40, 12, 12, 128),
]


def _run(ctx, cs, hs):
    kind, n, h, w, c, G = cs["kind"], cs["n"], cs["h"], cs["w"], cs["c"], cs["G"]
    hw, P = h * w, n * h * w
    ld = 2 * c if cs["strided"] else c
    gm_ld = hs["gm_buf"].shape[1]
    ident = kind == "ident"
    center, scale = (0, 0) if ident else (int(cs["center"]), int(cs["scale"]))
    d0 = _lib.NormDesc(0, n, hw, c, c, ld, 1e-3, 0.99, 1, center, scale)
    dv = _lib.NormDesc(1, n, hw, c, c, ld, 1e-3 if not ident else 1e-6, 0.99, 1, center, scale)
    dl = d0 if kind == "bn-plain" else dv            # the view of the fold and of the passes
    groups = 1 if kind == "bn-plain" else n
    res, bufs = {}, []

    def up(a):
        bufs.append(ctx.from_numpy(np.ascontiguousarray(a)))
        return bufs[-1]

    def out(*a, **k):
        o = Out(ctx, *a, **k)
        bufs.append(o.buf)
        return o

    pbuf = lambda b: b.p if b is not None else None  # noqa: E731
    x = ctx.bf16_from_f32(hs["y"].reshape(P, c))
    bufs.append(x)
    gamma = up(hs["gamma"]) if scale else None
    beta = up(hs["beta"]) if center else None
    gmb = up(hs["gm_buf"]) if cs["gm"] else None
    gm = C.c_void_p(gmb.ptr + GM_OFF * 4) if gmb else None
    gmap = up(hs["guide"]) if G else None
    wb = up(hs["w_buf"]) if G else None
    wsp = C.c_void_p(wb.ptr + c * 4) if G else None
    bsp = up(hs["b_guide"]) if G else None
    ga, ba = up(hs["ga"]), up(hs["ba"])
    q = {k: out(n, c) for k in ("mean", "rstd", "scale", "shift", "c1", "c2")}
    if ident:
        for k, v in (("mean", 0.0), ("rstd", 1.0), ("scale", 1.0), ("shift", 0.0)):
            arr = q[k].buf.download(np.float32, (q[k].total,))     # the guard keeps its canary
            arr[:n * c] = v
            q[k].buf.upload(arr)
        if cs["gm"] or G:
            ctx.call("bsl_norm_modulate", C.byref(dv), gm, C.c_int(gm_ld), pbuf(bsp), q["scale"].p, q["shift"].p,
                     ctx.stream)
    else:
        mm, mv = up(hs["mm"]), up(hs["mv"])
        sums = out(1, 2 * c, esize=8)
        ctx.call("bsl_norm_stats", C.byref(d0), x.p, sums.p, ctx.stream)
        ctx.call("bsl_norm_finalize", C.byref(d0), C.c_int(1), sums.p, pbuf(gamma), pbuf(beta), mm.p, mv.p,
                 q["mean"].p, q["rstd"].p, q["scale"].p, q["shift"].p, ctx.stream)
        if kind == "bn-mod":
            ctx.call("bsl_norm_modulate_bn", C.byref(dv), gm, C.c_int(gm_ld), pbuf(bsp), q["mean"].p, q["rstd"].p,
                     q["scale"].p, q["shift"].p, ctx.stream)
    res["mean"], res["rstd"] = q["mean"].get()[:groups], q["rstd"].get()[:groups]
    sp, hp = out(groups, c), out(groups, c)
    weff = out(G, c) if G else None
    ctx.call("bsl_norm_affine_fold", C.byref(dl), ga.p, ba.p, q["scale"].p, q["shift"].p, sp.p, hp.p, wsp,
             C.c_int(2 * c), C.c_int(G), weff.p if G else None, ctx.stream)
    res["scale_pre"], res["shift_pre"] = sp.get(), hp.get()
    res["fold_scale"], res["fold_shift"] = q["scale"].get()[:groups], q["shift"].get()[:groups]
    guide = None
    if G:
        res["w_eff"] = weff.get()
        guide = _lib.Guide(gmap.ptr, G, weff.p.value, c)
    gp = C.byref(guide) if guide is not None else None
    a = out(P, c, ld=ld, esize=2)
    ctx.call("bsl_norm_apply_mod", C.byref(dl), x.p, q["scale"].p, q["shift"].p, gp, a.p, ctx.stream)
    res["a"] = a.get()
    dy = _bf16_strided(ctx, hs["da"], ld, 1e4)
    bufs.append(dy)
    sb = out(groups, (2 + G) * c, esize=8)
    ctx.call("bsl_norm_bwd_reduce_mod", C.byref(dl), x.p, dy.p, C.c_int(ld), q["mean"].p, q["rstd"].p, q["scale"].p,
             q["shift"].p, gp, sb.p, ctx.stream)
    g = dict(dgamma=out(1, c) if scale else None, dbeta=out(1, c) if center else None,
             dgamma_mod=out(n, c, ld=gm_ld, off=GM_OFF) if cs["gm"] else None,
             dw_guide=out(G, c, ld=2 * c, off=c) if G else None, dbias_guide=out(1, c) if G else None,
             dga=out(1, c), dba=out(1, c))
    gpt = {k: (v.p if v is not None else None) for k, v in g.items()}
    jac = {"bn-mod": JAC_BATCH, "bn-plain": JAC_GROUP, "ident": JAC_NONE}[kind]
    ctx.call("bsl_norm_bwd_finalize_affine_jac", C.byref(dl), C.c_int(jac), sb.p, C.c_int(G), gm, C.c_int(gm_ld),
             pbuf(gamma), pbuf(beta), ga.p, q["mean"].p, q["rstd"].p, sp.p, hp.p, wsp, C.c_int(2 * c), q["c1"].p,
             q["c2"].p, gpt["dgamma"], gpt["dbeta"], gpt["dgamma_mod"], gpt["dw_guide"], C.c_int(2 * c),
             gpt["dbias_guide"], gpt["dga"], gpt["dba"], ctx.stream)
    dx = out(P, c, ld=ld, esize=2)
    ctx.call("bsl_norm_bwd_apply_bnmod" if kind == "bn-mod" else "bsl_norm_bwd_apply_mod", C.byref(dl), x.p, dy.p,
             C.c_int(ld), q["mean"].p, q["rstd"].p, q["scale"].p, q["shift"].p, q["c1"].p, q["c2"].p, gp, dx.p,
             C.c_int(ld), ctx.stream)
    ctx.check_device()
    res["c1"], res["c2"], res["dx"] = q["c1"].get()[:groups], q["c2"].get()[:groups], dx.get()
    for k, v in g.items():
        if v is not None:
            res[k] = v.get()
    for b in bufs:
        b.free()
    return res


def _ident_ref(hs, cs):
    """The modulation stage over a dropped tensor T (= y here): u = T*gm + guide.w + b, z = ga*u + ba, a = relu(z)."""
    n, h, w, c, G = cs["n"], cs["h"], cs["w"], cs["c"], cs["G"]
    T = np.asarray(hs["y"], np.float64)
    gm = np.asarray(hs["gm_buf"][:, GM_OFF:GM_OFF + c], np.float64) if cs["gm"] else np.ones((n, c))
    u = T * gm[:, None, None, :]
    wg = np.asarray(hs["w_buf"][:G, c:], np.float64)
    if G:
        u = u + np.asarray(hs["guide"], np.float64) @ wg + np.asarray(hs["b_guide"], np.float64)
    ga, ba = np.asarray(hs["ga"], np.float64), np.asarray(hs["ba"], np.float64)
    z = u * ga + ba
    return T, gm, u, z, wg, ga, ba


def _check(cs, hs, res):
    n, h, w, c, G = cs["n"], cs["h"], cs["w"], cs["c"], cs["G"]
    f8 = lambda v: np.asarray(v, np.float64)  # noqa: E731
    ga, ba = f8(hs["ga"]), f8(hs["ba"])
    errs = {}
    mask = res["a"].reshape(n, h, w, c) > 0
    da = f8(hs["da"]).reshape(n, h, w, c)
    if cs["kind"] == "ident":
        T, gm, u, z, wg, _, _ = _ident_ref(hs, cs)
        sc, sh = gm, np.broadcast_to(f8(hs["b_guide"]) if G else 0.0, (n, c))
        errs["a"] = (rel(res["a"].reshape(n, h, w, c), np.maximum(z, 0)), 5e-3)
        gz = da * mask
        b = dict(dga=(gz * u).sum(axis=(0, 1, 2)), dba=gz.sum(axis=(0, 1, 2)))
        gu = gz * ga
        if G:
            b["dw_guide"] = np.einsum("nhwg,nhwc->gc", f8(hs["guide"]), gu)
            b["dbias_guide"] = gu.sum(axis=(0, 1, 2))
        if cs["gm"]:
            b["dgamma_mod"] = (gu * T).sum(axis=(1, 2))
        b["dy"] = gu * gm[:, None, None, :]
        assert not res["c1"].any() and not res["c2"].any(), "the identity normaliser has no Jacobian terms"
        if G:
            errs["w_eff"] = (_rows_rel(res["w_eff"], wg * ga), 1e-5)
    else:
        gamma = f8(hs["gamma"]) if cs["scale"] else None
        beta = f8(hs["beta"]) if cs["center"] else None
        mod = cs["kind"] == "bn-mod"
        gm = f8(hs["gm_buf"][:, GM_OFF:GM_OFF + c]) if cs["gm"] else None
        wg = f8(hs["w_buf"][:G, c:])
        f = R.forward(hs["y"], "batch", 1e-3, gamma, beta, gm, hs["guide"] if G else None, wg if G else None,
                      hs["b_guide"] if G else None, ga, ba, True)
        errs["a"] = (rel(res["a"].reshape(n, h, w, c), f["a"]), 5e-3)
        errs["mean"] = (_rows_rel(res["mean"], np.broadcast_to(f["mean"], res["mean"].shape)), 1e-5)
        errs["rstd"] = (_rows_rel(res["rstd"], np.broadcast_to(f["rstd"], res["rstd"].shape)), 1e-5)
        sc = (gamma if gamma is not None else 1.0) * f["rstd"]
        sh = (beta if beta is not None else 0.0) - f["mean"] * sc
        if mod:
            sc = sc * (gm if gm is not None else 1.0)
            sh = sh * (gm if gm is not None else 1.0) + (f8(hs["b_guide"]) if G else 0.0)
        sc, sh = np.broadcast_to(sc, res["scale_pre"].shape), np.broadcast_to(sh, res["scale_pre"].shape)
        b = R.backward(f, da=da, mask=mask)
        if G:
            errs["w_eff"] = (_rows_rel(res["w_eff"], wg * ga), 1e-5)
        if not mod:     # c1 / c2 of the plain backward apply: means over the batch of the gradient after the affine
            gz = da * mask
            errs["c1"] = (rel(res["c1"][0], gz.mean(axis=(0, 1, 2))), 1e-5)
            errs["c2"] = (rel(res["c2"][0], (gz * f["xhat"]).mean(axis=(0, 1, 2))), 1e-5)
        else:           # one value for every sample
            assert (res["c1"] == res["c1"][0]).all() and (res["c2"] == res["c2"][0]).all()
    errs["scale_pre"] = (_rows_rel(res["scale_pre"], sc), 1e-5)
    errs["shift_pre"] = (_rows_rel(res["shift_pre"], sh), 1e-5)
    errs["fold_scale"] = (_rows_rel(res["fold_scale"], sc * ga), 1e-5)
    errs["fold_shift"] = (_rows_rel(res["fold_shift"], sh * ga + ba), 1e-5)
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
def test_affine_fold_and_finaliser_op_parity(ctx, cs):
    hs = _host(dict(cs), seed=cs["n"] * 5 + cs["c"] + cs["G"])
    r1 = _run(ctx, cs, hs)
    _check(cs, hs, r1)
    r2 = _run(ctx, cs, hs)
    assert r1.keys() == r2.keys()
    for k in r1:
        assert np.array_equal(r1[k].view(_BITS[r1[k].dtype.itemsize]), r2[k].view(_BITS[r2[k].dtype.itemsize])), k


def test_affine_finaliser_refusals(ctx):
    """Return codes only (the refusals come before any launch): an unknown jacobian, the pooled batch Jacobian on a
    mode-0 descriptor, and gamma_mod on the single group of a mode-0 descriptor."""
    buf = ctx.alloc(1 << 16)
    p = buf.p
    d0 = _lib.NormDesc(0, 2, 16, 64, 64, 64, 1e-3, 0.99, 1, 0, 0)
    d1 = _lib.NormDesc(1, 2, 16, 64, 64, 64, 1e-3, 0.99, 1, 0, 0)

    def fin(d, jac, gm=None):
        return ctx.lib.bsl_norm_bwd_finalize_affine_jac(ctx.h, C.byref(d), C.c_int(jac), p, C.c_int(0), gm, C.c_int(64),
                                                        None, None, p, p, p, p, p, None, C.c_int(0), p, p, None, None, p,
                                                        None, C.c_int(0), None, p, p, ctx.stream)
    assert fin(d1, 3) == BSL_EINVAL
    assert fin(d0, JAC_BATCH) == BSL_EINVAL
    assert fin(d0, JAC_GROUP, gm=p) == BSL_EINVAL
    ctx.check_device()
    buf.free()
