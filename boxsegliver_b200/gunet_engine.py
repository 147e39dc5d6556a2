"""Guided U-Net (GUNet) training / inference engine on the sm_100a kernels.

Mirrors /root/reference/NetworksV2/GUNet.py:259-413 the way engine.UNetEngine mirrors UNet.py: the trunk is the
same conv / norm / pool / transposed-conv sequence (same tcgen05 kernels, same zero-copy concat), and the blocks
listed in `mod_layers` are modulated (modulated_conv_block, GUNet.py:162-217):

    conv -> instance_norm(center, scale per YAML) -> * gamma_mod[n, c] -> + (sp_guide . w_sp[:, c] + b_sp[c]) -> ReLU

gamma_mod is a slice of the context MLP output (GUNet.py:31-59: fc(200 -> 256 -> 256 -> 3840), dropout after the
hidden layers); the additive map is the level's 1x1 guide convolution (GUNet.py:136-159) evaluated on the fly inside
the normalisation kernels, so modulation adds no pass over the activations. `after_affine` (5 of the 13 shipped
ext_config/*.yml; slim_nets.channel_wise_affine before every encoder ReLU, GUNet.py:213-214) folds into the same
per-(sample, channel) scale / shift and a gamma-scaled copy of the guide filter (bsl_norm_affine_fold): no extra pass.
`--normalizer batch_norm` (GUNet.py:301,321-325): batch statistics; modulated and dropped blocks run on the per-sample view
(bsl_norm_modulate_bn), un-modulated blocks keep per-channel scalars, and the affine folds into whichever the block has.
Backbone `--dropout` (GUNet.py:189-190: slim.dropout behind the normaliser of the first conv of every encoder block, in
front of the modulation; no shipped script enables it) runs un-fused: normalise without ReLU into a bf16 copy, multiply it
by the Philox mask in place (bsl_dropout_bf16), then the ordinary modulated apply pass over that copy with an identity
normaliser (folding the affine under after_affine); backward mirrors the three stages. Every combination of normaliser,
after_affine and --dropout trains and evaluates.
`--img_grad` (GUNet.py:333-337, scripts/103_grad.sh): the input becomes concat(images, dy, dx) of
tf.image.image_gradients, packed as bf16 [n, h, w, 64] (9 live lanes) by bsl_image_gradients_pack; the first layer then
runs as an ordinary 64-lane conv instead of the im2col stem.
Scope: context_model "fc"; --use_se, --fix, --without_norm and ct_conv raise NotImplementedError.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass

import numpy as np

from . import _lib
from .engine import BF16, F32, ConvL, EngineConfig, Param, UNetEngine, View, _align

JAC_GROUP, JAC_BATCH, JAC_NONE = 0, 1, 2      # BSL_NORM_JAC_* of include/bsl_b200.h


@dataclass
class GUNetConfig(EngineConfig):
    height: int = 512
    width: int = 512
    normalizer: str = "instance_norm"
    mod_layers: tuple = (1, 2, 3, 4)               # NetworksV2/GUNet.yml
    context_fc_channels: tuple = (256, 256)
    norm_with_center: bool = True
    norm_with_scale: bool = False
    after_affine: bool = False
    context_model: str = "fc"
    use_context: bool = True                       # --use_context
    use_spatial: bool = True                       # --use_spatial
    guide_channel: int = 1                         # --guide_channel
    context_dim: int = 200
    side_dropout: float = 0.5                      # --side_dropout
    dropout_seed: int = 0
    use_se: bool = False
    fix: bool = False
    dropout: float = None
    img_grad: bool = False                         # --img_grad: concat(images, dy, dx) of tf.image.image_gradients as input

    @property
    def n_modulator_param(self):
        return self.init_channels * sum(2 ** i for i in range(self.num_down_samples + 1) if i in self.mod_layers) * 2


class GUNetEngine(UNetEngine):
    prefix = "GUNet"      # variable-scope root (UNetInterEngine reuses the graph under "UNetInter")

    def __init__(self, ctx, cfg: GUNetConfig):
        for flag in ("use_se", "fix", "without_norm"):
            if getattr(cfg, flag):
                raise NotImplementedError(f"GUNet engine: --{flag} is not supported")
        if cfg.dropout:
            if not 0.0 < cfg.dropout < 1.0:
                raise ValueError("--dropout must lie in (0, 1)")
        if cfg.context_model != "fc":
            raise ValueError("Not supported context model")          # GUNet.py:79
        if cfg.use_spatial and cfg.guide_channel not in (1, 2):
            raise ValueError("guide_channel must be 1 or 2")
        super().__init__(ctx, cfg)
        self._plan_guides()
        self._plan_dropout()

    # ------------------------------------------------------------------ graph
    def _loss_terms(self):
        return [t for t in ("xentropy", "dice") if t in self.cfg.loss_type]   # GUNet.py:399-408

    def _layer_specs(self):
        cfg = self.cfg
        specs = []
        c, cin = cfg.init_channels, cfg.channel
        h, w = cfg.height, cfg.width
        nd = cfg.num_down_samples
        off = 0
        grad_in = bool(getattr(cfg, "img_grad", False)) and self.prefix == "GUNet"
        if grad_in:
            cin = 3 * cfg.channel     # GUNet.py:333-337; too many im2col columns for the stem: an ordinary conv, 9 -> 64 lanes
        for i in range(nd + 1):
            mod = i in cfg.mod_layers and (cfg.use_context or cfg.use_spatial)
            for j in (1, 2):
                kind = "stem" if (i == 0 and j == 1 and not grad_in) else "conv"
                role = f"enc{j}" if i < nd else f"bridge{j}"
                aa = bool(getattr(cfg, "after_affine", False))
                # encoder_arg_scope (GUNet.py:313-330): after_affine turns centre / scale of the MODULATED blocks' normaliser
                # off; un-modulated blocks pass normalizer_params={} (slim defaults, both on) and still get the affine
                L = ConvL(kind, f"{self.prefix}/Encode/down_conv{i + 1}/mod_conv{j}/Conv", cin, c, h, w, i, role=role,
                          center=(cfg.norm_with_center and not aa) if mod else True,
                          scale=(cfg.norm_with_scale and not aa) if mod else True)
                if aa:
                    L.affine = f"{self.prefix}/Encode/down_conv{i + 1}/mod_conv{j}/ChannelWiseAffine"
                # batch norm: the encoder arg scope's decay 0.99 reaches GUNet's modulated blocks (the un-modulated ones
                # override the params, GUNet.py:171-178) and every encoder conv of UNetInter (UNetInter.py:100-117)
                if mod or self.prefix == "UNetInter":
                    L.bn_decay = 0.99
                if mod and cfg.use_context:
                    L.mod_off = off
                    off += c
                if mod and cfg.use_spatial:
                    L.sp_off = (j - 1) * c
                specs.append(L)
                cin = c
            if i == 0 and getattr(cfg, "mid_cat", False):
                cin = c + cfg.guide_channel          # UNetInter.py:124-125: concat(block output, sp_guide) is what gets pooled
            if i < nd:
                c *= 2
                h //= 2
                w //= 2
        for i in reversed(range(nd)):
            c //= 2
            specs.append(ConvL("convT", f"{self.prefix}/Decode/up{i + 1}", cin, cin // 2, h, w, i))
            h *= 2
            w *= 2
            for j in (1, 2):
                specs.append(ConvL("conv", f"{self.prefix}/Decode/up_conv{i + 1}/up_conv{i + 1}_{j}",
                                   c + cin // 2 if j == 1 else c, c, h, w, i, role=f"dec{j}"))
            cin = c
        specs.append(ConvL("logits", f"{self.prefix}/AdjustChannels", cin, cfg.num_classes, h, w, 0))
        return specs

    def _fc_specs(self):
        cfg = self.cfg
        chans = list(cfg.context_fc_channels) + [cfg.n_modulator_param]
        out, cin = [], cfg.context_dim
        for k, co in enumerate(chans):
            out.append((f"GUNet/context/fc{k + 1}", cin, co, k < len(chans) - 1))
            cin = co
        return out

    def _extra_params(self):
        cfg = self.cfg
        plist = []
        for L in self.layers:
            if L.affine:           # variables.model_variable without a regulariser (slim_nets.py:186-201)
                plist.append(Param(f"{L.affine}/gamma", (L.cout,), region="B"))
                plist.append(Param(f"{L.affine}/beta", (L.cout,), region="B"))
        if cfg.use_context:
            for sc, cin, cout, _ in self._fc_specs():      # slim.fully_connected: no regulariser in GUNet's arg scope
                plist.append(Param(f"{sc}/weights", (cin, cout), region="B"))
                plist.append(Param(f"{sc}/biases", (cout,), region="B"))
        if cfg.use_spatial:
            for i in range(cfg.num_down_samples + 1):
                if i in cfg.mod_layers:
                    co = cfg.init_channels * 2 ** (i + 1)
                    sc = f"GUNet/spatial/conv{i + 1}"
                    plist.append(Param(f"{sc}/weights", (1, 1, cfg.guide_channel, co)))
                    plist.append(Param(f"{sc}/biases", (co,), region="B" if cfg.bias_decay else "A"))
        return plist

    def _guide_channels(self, L: ConvL) -> int:
        return self.cfg.guide_channel if L.sp_off is not None else 0

    def _first_input(self, L: ConvL):
        """--img_grad: the bf16 tensor [n, h, w, 64] that bsl_image_gradients_pack fills with (images, dy, dx)."""
        cfg = self.cfg
        lanes = self.params[f"{L.scope}/weights"].stored[2]
        self.input_packed = View(self._alloc(cfg.batch * L.h * L.w * lanes * BF16).zero(), cfg.batch, L.h, L.w, lanes)
        return self.input_packed

    def _bn_mod(self, L: ConvL) -> bool:
        """A modulated or --dropout block under batch norm: batch statistics, per-sample scale / shift (the mode-1 view).
        An un-modulated block with only the affine keeps per-channel scalars and folds the affine into them."""
        return self.cfg.normalizer == "batch_norm" and (L.mod_off is not None or L.sp_off is not None or self._drops(L))

    def _norm_groups(self, L: ConvL, default: int) -> int:
        return self.cfg.batch if self._bn_mod(L) else default

    def _apply_desc(self, L: ConvL, nd):
        if not self._bn_mod(L):
            return nd
        return _lib.NormDesc(1, nd.n, nd.hw, nd.c, nd.x_ld, nd.y_ld, nd.eps, nd.decay, nd.relu, nd.center, nd.scale)

    def _plan_guides(self):
        cfg, n = self.cfg, self.cfg.batch
        self.guides = []
        # after_affine: un-folded scale / shift of every encoder layer (backward finaliser) + the gamma-scaled guide filter
        self.aff_bufs = {L.scope: self._alloc((2 * _align(n * L.cout, 16) + 2 * L.cout) * F32)
                         for L in self.layers if L.affine}
        if cfg.use_spatial:
            h, w = cfg.height, cfg.width
            for _ in range(cfg.num_down_samples + 1):
                self.guides.append((self._alloc(n * h * w * cfg.guide_channel * F32), h, w))
                h //= 2
                w //= 2
        self.fc_bufs = []
        if cfg.use_context:
            self.context = self._alloc(n * cfg.context_dim * F32)
            ws = 0
            for sc, cin, cout, hidden in self._fc_specs():
                y = self._alloc(n * cout * F32)
                dy = self._alloc(n * cout * F32) if cfg.training else None
                self.fc_bufs.append((y, dy))
                d = self._fc_desc(cin, cout, hidden, 0, True)
                ws = max(ws, self.ctx.lib.bsl_fc_bwd_workspace(self.ctx.h, C.byref(d)))
            self.fc_ws_bytes = int(ws)
            self.fc_ws = self._alloc(max(ws, 16))

    # ------------------------------------------------------------------ backbone --dropout
    def _drops(self, L: ConvL) -> bool:
        return bool(self.cfg.dropout) and self.prefix == "GUNet" and L.role in ("enc1", "bridge1")

    def _plan_dropout(self):
        """Per dropped layer: the normalised-and-dropped bf16 tensor (kept for backward) and the normaliser's own
        scalars (the layer's main scalar set then describes the identity normaliser of the modulation stage)."""
        cfg, n = self.cfg, self.cfg.batch
        self.drop = {}
        layers = [L for L in self.layers if L.kind in ("stem", "conv") and self._drops(L)]
        if not layers:
            return
        cmax = max(L.cout for L in layers)
        ones = np.ones(_align(n * cmax, 16), np.float32)
        self._ones = self._alloc(ones.nbytes)
        self._ones.upload(ones)
        self._zeros = self._alloc(ones.nbytes).zero()
        for L in layers:
            self.drop[L.scope] = dict(T=self._alloc(n * L.h * L.w * L.cout * BF16),
                                      small=self._alloc(self._norm_scalar_floats(n * L.cout) * F32))
        if cfg.training:
            self.drop_grad = self._alloc(n * max(L.h * L.w * L.cout for L in layers) * BF16)

    def _drop_ptrs(self, L: ConvL):
        return self._norm_scalars(self.drop[L.scope]["small"].ptr, self.cfg.batch * L.cout)

    def _drop_desc(self, L: ConvL):
        return _lib.DropoutDesc(1.0 - self.cfg.dropout, self.cfg.dropout_seed, (self.step_count + 1) * 16 + 8 + L.level)

    def _dropout_stage(self, L: ConvL, nd, q, is_training: bool):
        if not (is_training and L.scope in getattr(self, "drop", {})):
            self._dropped = getattr(self, "_dropped", set()) - {L.scope}
            return L.y.p
        cfg, call, s = self.cfg, self.ctx.call, self.stream
        T, qn = self.drop[L.scope]["T"], self._drop_ptrs(L)
        # the normaliser's scalars are [n][cout] under instance norm, [cout] under batch norm (mode 0); the identity of
        # the modulation stage fills the layer's whole scalar arrays ([n][cout]: the per-sample view)
        nbytes = C.c_size_t((cfg.batch if nd.mode else 1) * L.cout * F32)
        nbytes_id = C.c_size_t(L.norm["groups"] * L.cout * F32)
        for k in ("mean", "rstd", "scale", "shift"):       # the normaliser's own scalars move aside ...
            call("bsl_memcpy_d2d", qn[k], q[k], nbytes, s)
        ndn = _lib.NormDesc(nd.mode, nd.n, nd.hw, nd.c, nd.x_ld, L.cout, nd.eps, nd.decay, 0, nd.center, nd.scale)
        call("bsl_norm_apply", C.byref(ndn), L.y.p, qn["scale"], qn["shift"], T.p, s)
        dd = self._drop_desc(L)
        call("bsl_dropout_bf16", C.byref(dd), C.c_longlong(cfg.batch * L.h * L.w), C.c_int(L.cout), T.p, C.c_int(L.cout),
             T.p, C.c_int(L.cout), s)
        for k, src in (("mean", self._zeros), ("rstd", self._ones), ("scale", self._ones), ("shift", self._zeros)):
            call("bsl_memcpy_d2d", q[k], src.p, nbytes_id, s)  # ... and the modulation stage sees an identity normaliser
        self._dropped = getattr(self, "_dropped", set()) | {L.scope}
        return T.p

    def _fc_desc(self, cin, cout, hidden, layer, is_training):
        cfg = self.cfg
        drop = bool(hidden and is_training and cfg.side_dropout)
        dd = _lib.DropoutDesc(1.0 - cfg.side_dropout if drop else 1.0, cfg.dropout_seed,
                              (self.step_count + 1) * 16 + layer)
        return _lib.FcDesc(cfg.batch, cin, cout, int(hidden), int(drop), dd)

    # ------------------------------------------------------------------ weights / inputs
    def init_weights(self, seed: int = 0):
        """xavier for convs and hidden FC layers, he_normal for the final FC (GUNet.py:56), zeros / ones elsewhere."""
        rng = np.random.default_rng(seed)
        w = {}
        for name, p in self.params.items():
            shp = p.shape
            if name.endswith("/weights") and len(shp) == 4:
                rf = shp[0] * shp[1]
                w[name] = self._draw_weight(rng, shp, rf * shp[2], rf * shp[3])
            elif name.endswith("/weights"):
                last = name.startswith(f"GUNet/context/fc{len(self._fc_specs())}/")
                if last:
                    w[name] = np.clip(rng.standard_normal(shp), -2, 2).astype(np.float32) * np.float32(
                        np.sqrt(2.0 / shp[0]) / 0.87962566103423978)
                else:
                    lim = np.sqrt(6.0 / (shp[0] + shp[1]))
                    w[name] = rng.uniform(-lim, lim, size=shp).astype(np.float32)
            elif name.endswith("gamma"):
                w[name] = np.ones(shp, np.float32)
            else:
                w[name] = np.zeros(shp, np.float32)
        self.set_weights(w)
        return w

    def set_guides(self, context: np.ndarray | None = None, sp_guide: np.ndarray | None = None):
        cfg = self.cfg
        if cfg.use_context:
            assert context is not None and context.shape == (cfg.batch, cfg.context_dim), "context [N, context_dim]"
            self.context.upload(np.ascontiguousarray(context, np.float32))
        if cfg.use_spatial:
            shp = (cfg.batch, cfg.height, cfg.width, cfg.guide_channel)
            assert sp_guide is not None and sp_guide.shape == shp, f"sp_guide {shp}"
            self.guides[0][0].upload(np.ascontiguousarray(sp_guide, np.float32))

    # ------------------------------------------------------------------ forward
    def forward(self, is_training: bool):
        cfg, call, s = self.cfg, self.ctx.call, self.stream
        self.ctx.tag = "GUNet/context"
        if cfg.use_context:
            x = self.context
            for k, (sc, cin, cout, hidden) in enumerate(self._fc_specs()):
                d = self._fc_desc(cin, cout, hidden, k, is_training)
                call("bsl_fc_fwd", C.byref(d), x.p, self._pp(self.W, f"{sc}/weights"), self._pp(self.W, f"{sc}/biases"),
                     self.fc_bufs[k][0].p, s)
                x = self.fc_bufs[k][0]
            self.ctx_params = x
        self.ctx.tag = "GUNet/spatial"
        if cfg.use_spatial:
            for i in range(cfg.num_down_samples):
                (src, h, w), (dst, _, _) = self.guides[i], self.guides[i + 1]
                call("bsl_avgpool2x2_f32", C.c_int(cfg.batch), C.c_int(h), C.c_int(w), C.c_int(cfg.guide_channel), src.p,
                     dst.p, s)
        self._fwd_training = is_training
        if getattr(self, "input_packed", None) is not None:
            self.ctx.tag = "GUNet/image_gradients"
            call("bsl_image_gradients_pack", C.c_int(cfg.batch), C.c_int(cfg.height), C.c_int(cfg.width), C.c_int(cfg.channel),
                 self.images.p, self.input_packed.p, C.c_int(self.input_packed.ld), s)
        super().forward(is_training)

    def _aff_ptrs(self, L: ConvL):
        """(scale_pre, shift_pre, w_eff) of an after_affine layer."""
        base, n = self.aff_bufs[L.scope].ptr, _align(self.cfg.batch * L.cout, 16)
        return C.c_void_p(base), C.c_void_p(base + n * F32), C.c_void_p(base + 2 * n * F32)

    def _guide_struct(self, L: ConvL):
        if L.sp_off is None:
            return None
        sc = f"GUNet/spatial/conv{L.level + 1}"
        if L.affine:     # the passes read the filter scaled by the affine's gamma (bsl_norm_affine_fold wrote it)
            return _lib.Guide(self.guides[L.level][0].ptr, self.cfg.guide_channel, self._aff_ptrs(L)[2].value, L.cout)
        return _lib.Guide(self.guides[L.level][0].ptr, self.cfg.guide_channel,
                          self._pp(self.W, f"{sc}/weights", off=L.sp_off).value, 2 * L.cout)

    def _modulate(self, L: ConvL, nd, q):
        gm = C.c_void_p(self.ctx_params.ptr + L.mod_off * F32) if L.mod_off is not None else None
        bsp = self._pp(self.W, f"GUNet/spatial/conv{L.level + 1}/biases", off=L.sp_off) if L.sp_off is not None else None
        if self._bn_mod(L):      # (an un-modulated --dropout block: expansion to the per-sample view only)
            self.ctx.call("bsl_norm_modulate_bn", C.byref(self._apply_desc(L, nd)), gm,
                          C.c_int(self.cfg.n_modulator_param), bsp, q["mean"], q["rstd"], q["scale"], q["shift"],
                          self.stream)
        elif L.mod_off is not None or L.sp_off is not None:
            self.ctx.call("bsl_norm_modulate", C.byref(nd), gm, C.c_int(self.cfg.n_modulator_param), bsp, q["scale"],
                          q["shift"], self.stream)
        if L.affine:
            sp, hp, weff = self._aff_ptrs(L)
            g = self._guide_channels(L)
            wsp = self._pp(self.W, f"GUNet/spatial/conv{L.level + 1}/weights", off=L.sp_off) if g else None
            self.ctx.call("bsl_norm_affine_fold", C.byref(self._apply_desc(L, nd)),
                          self._pp(self.W, f"{L.affine}/gamma"), self._pp(self.W, f"{L.affine}/beta"), q["scale"], q["shift"], sp, hp, wsp,
                          C.c_int(2 * L.cout), C.c_int(g), weff if g else None, self.stream)
        return self._guide_struct(L)

    # ------------------------------------------------------------------ backward
    def _is_modulated(self, L: ConvL) -> bool:
        return L.mod_off is not None or L.sp_off is not None or bool(L.affine) or self._was_dropped(L)

    def _was_dropped(self, L: ConvL) -> bool:
        return L.scope in getattr(self, "_dropped", ())

    def _norm_backward_reduce(self, L: ConvL, nd, q, cur):
        if not self._is_modulated(L):
            return super()._norm_backward_reduce(L, nd, q, cur)
        call, s, ns = self.ctx.call, self.stream, self.norm_scope
        nd = self._apply_desc(L, nd)
        guide = self._guide_struct(L)
        gp = C.byref(guide) if guide is not None else None
        nmod = self.cfg.n_modulator_param
        gm = C.c_void_p(self.ctx_params.ptr + L.mod_off * F32) if L.mod_off is not None else None
        dgm = C.c_void_p(self.fc_bufs[-1][1].ptr + L.mod_off * F32) if L.mod_off is not None else None
        ssc = f"GUNet/spatial/conv{L.level + 1}"
        dwg = self._pp(self.G, f"{ssc}/weights", off=L.sp_off) if L.sp_off is not None else None
        dbg = self._pp(self.G, f"{ssc}/biases", off=L.sp_off) if L.sp_off is not None else None
        dropped = self._was_dropped(L)
        xin = self.drop[L.scope]["T"].p if dropped else L.y.p
        call("bsl_norm_bwd_reduce_mod", C.byref(nd), xin, cur.p, C.c_int(L.cout), q["mean"], q["rstd"], q["scale"],
             q["shift"], gp, q["sums"], s)
        if dropped and L.affine:
            # modulation stage over the dropped tensor with the folded affine: identity normaliser, no Jacobian
            sp, hp, _ = self._aff_ptrs(L)
            wsp = self._pp(self.W, f"{ssc}/weights", off=L.sp_off) if L.sp_off is not None else None
            call("bsl_norm_bwd_finalize_affine_jac", C.byref(nd), C.c_int(JAC_NONE), q["sums"],
                 C.c_int(self._guide_channels(L)), gm, C.c_int(nmod), None, None, self._pp(self.W, f"{L.affine}/gamma"),
                 q["mean"], q["rstd"], sp, hp, wsp, C.c_int(2 * L.cout), q["c1"], q["c2"], None, None, dgm, dwg,
                 C.c_int(2 * L.cout), dbg, self._pp(self.G, f"{L.affine}/gamma"), self._pp(self.G, f"{L.affine}/beta"), s)
            return
        if dropped:
            # modulation stage over the dropped tensor: identity normaliser (no gamma / beta, no Jacobian: c1 = c2 = 0);
            # sum(dz * T) is the gradient of gamma_mod, the guide rows those of the 1x1 guide conv
            call("bsl_norm_bwd_finalize_mod", C.byref(nd), q["sums"], C.c_int(self._guide_channels(L)), gm, C.c_int(nmod),
                 None, None, q["c1"], q["c2"], None, None, dgm, dwg, C.c_int(2 * L.cout), dbg, s)
            nbytes = C.c_size_t(self.cfg.batch * L.cout * F32)
            call("bsl_memset", q["c1"], C.c_int(0), nbytes, s)
            call("bsl_memset", q["c2"], C.c_int(0), nbytes, s)
            return
        if L.affine:
            # batch norm: modulated blocks on the per-sample view (pooled Jacobian), the others on their single group
            sp, hp, _ = self._aff_ptrs(L)
            wsp = self._pp(self.W, f"{ssc}/weights", off=L.sp_off) if L.sp_off is not None else None
            call("bsl_norm_bwd_finalize_affine_jac", C.byref(nd), C.c_int(JAC_BATCH if self._bn_mod(L) else JAC_GROUP),
                 q["sums"], C.c_int(self._guide_channels(L)), gm, C.c_int(nmod),
                 self._pp(self.W, f"{L.scope}/{ns}/gamma"), self._pp(self.W, f"{L.scope}/{ns}/beta"),
                 self._pp(self.W, f"{L.affine}/gamma"), q["mean"], q["rstd"], sp, hp, wsp, C.c_int(2 * L.cout),
                 q["c1"], q["c2"], self._pp(self.G, f"{L.scope}/{ns}/gamma"), self._pp(self.G, f"{L.scope}/{ns}/beta"),
                 dgm, dwg, C.c_int(2 * L.cout), dbg, self._pp(self.G, f"{L.affine}/gamma"),
                 self._pp(self.G, f"{L.affine}/beta"), s)
            return
        if self._bn_mod(L):
            call("bsl_norm_bwd_finalize_bnmod", C.byref(nd), q["sums"], C.c_int(self._guide_channels(L)), gm, C.c_int(nmod),
                 self._pp(self.W, f"{L.scope}/{ns}/gamma"), self._pp(self.W, f"{L.scope}/{ns}/beta"), q["rstd"], q["c1"],
                 q["c2"], self._pp(self.G, f"{L.scope}/{ns}/gamma"), self._pp(self.G, f"{L.scope}/{ns}/beta"), dgm, dwg,
                 C.c_int(2 * L.cout), dbg, s)
            return
        call("bsl_norm_bwd_finalize_mod", C.byref(nd), q["sums"], C.c_int(self._guide_channels(L)), gm, C.c_int(nmod),
             self._pp(self.W, f"{L.scope}/{ns}/gamma"), self._pp(self.W, f"{L.scope}/{ns}/beta"), q["c1"], q["c2"],
             self._pp(self.G, f"{L.scope}/{ns}/gamma"), self._pp(self.G, f"{L.scope}/{ns}/beta"), dgm, dwg,
             C.c_int(2 * L.cout), dbg, s)

    def _norm_backward_apply(self, L: ConvL, nd, q, cur, oth, stream):
        if self._head_grad is not None:
            return super()._norm_backward_apply(L, nd, q, cur, oth, stream)
        guide = self._guide_struct(L)
        if self._was_dropped(L):
            call, ns = self.ctx.call, self.norm_scope
            T, dT, qn = self.drop[L.scope]["T"], self.drop_grad, self._drop_ptrs(L)
            c = C.c_int(L.cout)
            call("bsl_norm_bwd_apply_mod", C.byref(self._apply_desc(L, nd)), T.p, cur.p, c, q["mean"], q["rstd"],
                 q["scale"], q["shift"], q["c1"], q["c2"], C.byref(guide) if guide is not None else None, dT.p, c, stream)
            dd = self._drop_desc(L)
            call("bsl_dropout_bf16", C.byref(dd), C.c_longlong(self.cfg.batch * L.h * L.w), c, dT.p, c, dT.p, c, stream)
            ndn = _lib.NormDesc(nd.mode, nd.n, nd.hw, nd.c, nd.x_ld, nd.y_ld, nd.eps, nd.decay, 0, nd.center, nd.scale)
            call("bsl_norm_bwd_reduce", C.byref(ndn), L.y.p, dT.p, c, qn["mean"], qn["rstd"], qn["scale"], qn["shift"],
                 qn["sums"], stream)
            call("bsl_norm_bwd_finalize", C.byref(ndn), qn["sums"], qn["c1"], qn["c2"],
                 self._pp(self.G, f"{L.scope}/{ns}/gamma"), self._pp(self.G, f"{L.scope}/{ns}/beta"), stream)
            call("bsl_norm_bwd_apply", C.byref(ndn), L.y.p, dT.p, c, qn["mean"], qn["rstd"], qn["scale"], qn["shift"],
                 qn["c1"], qn["c2"], oth.p, c, stream)
            return
        if self._bn_mod(L):
            self.ctx.call("bsl_norm_bwd_apply_bnmod", C.byref(self._apply_desc(L, nd)), L.y.p, cur.p, C.c_int(L.cout),
                          q["mean"], q["rstd"], q["scale"], q["shift"], q["c1"], q["c2"],
                          C.byref(guide) if guide is not None else None, oth.p, C.c_int(L.cout), stream)
            return
        self.ctx.call("bsl_norm_bwd_apply_mod", C.byref(nd), L.y.p, cur.p, C.c_int(L.cout), q["mean"], q["rstd"],
                      q["scale"], q["shift"], q["c1"], q["c2"], C.byref(guide) if guide is not None else None, oth.p,
                      C.c_int(L.cout), stream)

    def loss_backward(self):
        super().loss_backward()
        cfg, call, s = self.cfg, self.ctx.call, self.stream
        if not cfg.use_context:
            return
        self.ctx.tag = "GUNet/context"
        specs = self._fc_specs()
        for k in range(len(specs) - 1, -1, -1):
            sc, cin, cout, hidden = specs[k]
            d = self._fc_desc(cin, cout, hidden, k, True)
            x = self.context if k == 0 else self.fc_bufs[k - 1][0]
            dx = self.fc_bufs[k - 1][1].p if k > 0 else None
            call("bsl_fc_bwd", C.byref(d), x.p, self._pp(self.W, f"{sc}/weights"), self.fc_bufs[k][0].p,
                 self.fc_bufs[k][1].p, dx, self._pp(self.G, f"{sc}/weights"), self._pp(self.G, f"{sc}/biases"),
                 self.fc_ws.p, C.c_size_t(self.fc_ws_bytes), s)

    def get_context_grad(self):
        """Gradient w.r.t. the context MLP output after loss_backward ([n, n_modulator_param], fp32)."""
        return self.fc_bufs[-1][1].download(np.float32, (self.cfg.batch, self.cfg.n_modulator_param))

    def get_context_params(self):
        return self.ctx_params.download(np.float32, (self.cfg.batch, self.cfg.n_modulator_param))


@dataclass
class UNetInterConfig(GUNetConfig):
    """UNetInter (/root/reference/NetworksV2/UNetInter.py:44-160): the interactive-segmentation U-Net. `channel` is the
    image channel count; the `guide_channel`-channel click guide is concatenated to the images at the input."""
    height: int = 256
    width: int = 256
    use_context: bool = False
    use_spatial: bool = False
    mod_layers: tuple = ()
    guide_channel: int = 2
    mid_cat: bool = False


class UNetInterEngine(GUNetEngine):
    """UNetInter = GUNet's variable layout (Encode/down_conv*/mod_conv*/Conv, Decode/up*, up_conv*) without modulation:
    every conv is conv -> norm(center, scale) -> ReLU, and the network input is concat(images, sp_guide)
    (UNetInter.py:89-92). With --mid_cat (UNetInter.py:87-92,124-125) the images alone enter the first block and the guide
    is concatenated to its output in front of the first max-pool: the pooled tensor is stored with 128 lanes (64
    activation lanes from the fused norm + ReLU + pool pass, guide_channel lanes from bsl_maxpool2x2_f32_bf16, zeros), and
    the second block's first conv runs with its 64 + guide_channel input channels zero-padded to 128."""
    prefix = "UNetInter"

    def __init__(self, ctx, cfg: UNetInterConfig):
        if cfg.use_context or cfg.use_spatial or cfg.mod_layers:
            raise ValueError("UNetInter has no guide modulation: the guide is an input channel")
        if cfg.mid_cat and cfg.init_channels % 64:
            raise ValueError("--mid_cat: init_channels must be a multiple of 64 (the guide lanes follow a whole channel block)")
        self.image_channels = cfg.channel
        self.user_cfg = cfg
        super().__init__(ctx, cfg if cfg.mid_cat else dataclasses.replace(cfg, channel=cfg.channel + cfg.guide_channel))
        if cfg.mid_cat:
            self.guide_in = self._alloc(cfg.batch * cfg.height * cfg.width * cfg.guide_channel * F32)

    def _pooled_lanes(self, L: ConvL) -> int:
        if self.cfg.mid_cat and L.level == 0:
            return _align(L.cout + self.cfg.guide_channel, 64)
        return L.cout

    def _after_pool(self, L: ConvL, stream):
        cfg = self.cfg
        if cfg.mid_cat and L.level == 0:
            self.ctx.call("bsl_maxpool2x2_f32_bf16", C.c_int(cfg.batch), C.c_int(L.h), C.c_int(L.w),
                          C.c_int(cfg.guide_channel), self.guide_in.p, C.c_void_p(L.pooled.p.value + L.cout * BF16),
                          C.c_int(L.pooled.ld), stream)

    def set_inputs(self, images: np.ndarray, labels: np.ndarray | None = None, sp_guide: np.ndarray | None = None,
                   stream=None):
        cfg = self.cfg
        if cfg.mid_cat:
            assert sp_guide is not None and sp_guide.shape == images.shape[:3] + (cfg.guide_channel,), "sp_guide"
            self.guide_in.upload(np.ascontiguousarray(sp_guide, np.float32), stream)
        elif images.shape[-1] == self.image_channels:
            assert sp_guide is not None and sp_guide.shape == images.shape[:3] + (cfg.guide_channel,), "sp_guide"
            images = np.concatenate((images, sp_guide), axis=-1)          # UNetInter.py:90
        super().set_inputs(images, labels, stream)
