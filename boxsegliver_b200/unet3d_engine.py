"""3-D U-Net (UNet3D) training / inference engine on the sm_100a kernels.

Mirrors /root/reference/NetworksV2/UNet3D.py:31-202: conv3d + instance-norm + ReLU blocks with kernels (1,3,3) /
(3,3,3), strided-conv down-sampling ((1,2,2), bridge (2,2,2)), bias-free conv3d_transpose + ReLU up-sampling, skip
concat [encoder, up], 1x1x1 logits, weighted cross-entropy. What differs from the 2-D engine:

  * --normalizer batch_norm (slim.batch_norm, eps 1e-3, decay 0.999) or instance_norm; batch statistics are per
    channel over all n*d*h*w voxels of the replica's batch, the moving statistics live in their own arena (region S)
    padded like gamma / beta, and eval-mode forwards normalise with them;
  * activations are NDHWC bf16; (1,3,3)/stride-1 layers run as 2-D convolutions over n*d images on the halo-tile
    kernels, everything else goes through bsl_conv3d_* / bsl_convT3d_* (csrc/conv3d.cu);
  * UNet3D's channel counts (30, 60, 120, 240, 320) are stored zero-padded to multiples of 64 (64, 64, 128, 256, 320)
    because the tcgen05 kernels reduce over 64-channel blocks. Pad lanes are exactly zero everywhere and stay zero
    through instance-norm (y = 0 -> z = beta_pad = 0), ReLU, the backward pass (dz = 0 where z = 0) and Adam
    (g = 0 -> no update), so numerics are those of the un-padded network; FLOP accounting uses the un-padded counts;
  * parameter arenas hold the PADDED layouts; set_weights / get_weights / get_grads pack and unpack TF-shaped
    variables ([kd,kh,kw,Cin,Cout], concat inputs split as [encoder | up]);
  * there is no pooling: an encoder block's output feeds the skip and the next strided conv, so its gradient is an
    explicit add (bsl_add_bf16) of the two branches;
  * PIXEL-PAIR PACKING of the full-resolution level (init_channels <= 32, W % 16 == 0, H % 32 == 0; BSL_UNET3D_PAIR=0
    turns it off): its tensors are stored with 32 channel lanes, not 64, and its (1,3,3) convolutions run on the SAME
    64-channel tcgen05 kernels over PAIRS of horizontally adjacent voxels -- the NDHWC tensor [n,d,h,w,32] reinterpreted
    as [n,d,h,w/2,64] ("super" voxels). A 3-tap row of the real filter becomes a 3-tap row of a 2*cin x 64 super filter
    (tap S of the super filter, input half hi, output half ho holds the real tap 2S + hi - ho + 1), a fixed
    re-arrangement built from the slim variable by an index table (bsl_gather_f32_bf16) and undone for the filter
    gradient (bsl_gather_add2_f32). Half the MMAs and half the HBM bytes of the 64-lane storage on the layers that
    hold most of the voxels; the normalisation / ReLU / add passes see the real 32-lane view. The level's concat buffer
    holds 128 lanes per voxel PAIR, [encoder even | encoder odd | up even | up odd]: the encoder half alone is again a
    64-lane super tensor (stride 128), so the strided conv that leaves the level reads only it -- super voxels X and
    X + 1 (a 2-tap row, horizontal stride 1 = pixel stride 2) -- and the transposed conv that enters the level writes
    the `up` half with bsl_convT2d_fwd_pairs; its backward kernels read the ReluGrad output as a dense 32-lane tensor
    (both column parities = 64 contiguous values).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from .device import Context, DeviceBuffer
from .engine_base import BF16, F32, EngineBase, Param, TrainConfig, _align

CPAD = 64


@dataclass
class UNet3DConfig(TrainConfig):
    depth: int = 64
    height: int = 128
    width: int = 128
    channel: int = 1
    classes: tuple = ("Background", "NF")
    init_channels: int = 30           # NetworksV2/UNet3D.yml
    max_channels: int = 320
    num_pool_layers: int = 4
    use_spatial: bool = False
    guide_channel: int = 2
    normalizer: str = "instance_norm"
    weight_decay_rate: float = 3e-5
    loss_weight_type: str = "numerical"
    loss_numeric_w: tuple = (1.0, 1.0)

    @property
    def in_channels(self):
        return self.channel + (self.guide_channel if self.use_spatial else 0)


class View3:
    """Channels [c0, c0 + c) of an NDHWC bf16 tensor with channel stride ld."""

    def __init__(self, buf: DeviceBuffer, n, dhw, c, ld=None, c0=0):
        self.buf, self.n, self.dhw, self.c = buf, n, tuple(dhw), c
        self.ld = ld or c
        self.c0 = c0

    @property
    def p(self):
        return C.c_void_p(self.buf.ptr + self.c0 * BF16)

    @property
    def voxels(self):
        return self.n * self.dhw[0] * self.dhw[1] * self.dhw[2]

    def slice(self, c0, c):
        return View3(self.buf, self.n, self.dhw, c, self.ld, self.c0 + c0)


class PairView(View3):
    """One half (part 0 = encoder, 1 = up) of the pixel-pair packed level's concat buffer: voxel pairs of 64 lanes
    ((voxel parity, 32 lanes)) with stride 128. `ld` and `c` are those of the voxel-PAIR view."""

    def __init__(self, buf: DeviceBuffer, n, dhw, part):
        super().__init__(buf, n, dhw, 64, 128, 64 * part)
        self.part = part

    @property
    def pairs(self):
        return self.voxels // 2


@dataclass
class Layer3:
    kind: str                 # stem | conv | convT | logits
    scope: str
    block: str
    layer: str
    cin: int                  # real channels
    cout: int
    k: tuple
    s: tuple
    dhw: tuple                # input spatial size
    odhw: tuple = None
    cinp: int = 0             # stored (padded) channels of the input view
    coutp: int = 0
    cin_map: np.ndarray = None   # real input channel -> stored input channel
    fork: bool = False        # encoder conv2: output also feeds the skip connection
    pair: str = ""            # pixel-pair packing: "conv" (stride-1 super conv), "strided" (level 0 -> 1), "stem", or ""
    catpair: bool = False     # pair == "conv" reading the level's concat buffer ([enc even | enc odd | up even | up odd])
    x: View3 = None
    y: View3 = None
    a: View3 = None
    norm_off: int = 0
    params: dict = field(default_factory=dict)


def _cp(c):
    return _align(c, CPAD)


def _model_config(pools: int):
    """UNet3D._ModelConfig.config[pools] (UNet3D.py:31-91) as (block, layer, kernel, stride)."""
    if pools not in (4, 5):
        raise KeyError(f"num_pool_layers {pools}: the reference defines configs for 4 and 5")
    out = []
    for i in range(pools):
        k = (1, 3, 3) if i < 2 else (3, 3, 3)
        out.append((f"conv_e{i}", "conv1", k, (1, 1, 1) if i == 0 else (1, 2, 2)))
        out.append((f"conv_e{i}", "conv2", k, (1, 1, 1)))
    out += [("bridge", "conv1", (3, 3, 3), (2, 2, 2)), ("bridge", "conv2", (3, 3, 3), (1, 1, 1))]
    for i in reversed(range(pools)):
        up = (2, 2, 2) if i == pools - 1 else (1, 2, 2)
        k = (1, 3, 3) if i < 2 else (3, 3, 3)
        out += [(f"conv_d{i}", "up", up, up), (f"conv_d{i}", "conv1", k, (1, 1, 1)), (f"conv_d{i}", "conv2", k, (1, 1, 1))]
    return out


class UNet3DEngine(EngineBase):
    def __init__(self, ctx: Context, cfg: UNet3DConfig):
        self.ctx, self.cfg = ctx, cfg
        self.pixels_per_sample = cfg.depth * cfg.height * cfg.width
        if cfg.normalizer not in ("batch_norm", "instance_norm"):
            raise ValueError("Not supported normalization function: " + cfg.normalizer)
        self.bn = cfg.normalizer == "batch_norm"
        self.norm_scope = "BatchNorm" if self.bn else "InstanceNorm"
        self._check_train_config()
        if 9 * cfg.in_channels > 64:
            raise ValueError("input channels must be <= 7 (the stem's im2col row holds 9 * channels <= 64 columns)")
        ds = 2 ** cfg.num_pool_layers
        if cfg.height % ds or cfg.width % ds or cfg.depth % 2:
            raise ValueError(f"height/width must be multiples of {ds} and depth even")
        self._init_plumbing()
        self._pair = (cfg.init_channels <= 32 and cfg.width % 16 == 0 and cfg.height % 32 == 0
                      and 9 * cfg.in_channels <= 32 and os.environ.get("BSL_UNET3D_PAIR", "1") != "0")
        # filter gradients on a side stream, as in engine.UNetEngine.loss_backward
        self._overlap_wgrad = cfg.training
        self._plan_layers()
        self._plan_params()
        self._plan_activations()

    # ------------------------------------------------------------------ planning
    def _plan_layers(self):
        cfg = self.cfg
        layers = []
        c, cin = cfg.init_channels, cfg.in_channels
        dhw = (cfg.depth, cfg.height, cfg.width)
        enc = {}
        first = True
        pair = self._pair

        def cpb(ch, block):
            """stored channel lanes of a tensor produced in `block` (32 on the pixel-pair packed level, else 64-padded)"""
            return _align(ch, 32) if pair and block in ("conv_e0", "conv_d0") else _cp(ch)

        prev_block = None
        for block, layer, k, s in _model_config(cfg.num_pool_layers):
            scope = f"UNet3D/{block}/{layer}"
            if layer == "up":
                e = enc[block.replace("d", "e")]
                c = e["c"]
                L = Layer3("convT", scope, block, layer, cin, c, k, s, dhw, cinp=_cp(cin), coutp=cpb(c, block))
                L.odhw = tuple(dhw[i] * s[i] for i in range(3))
                assert L.odhw == e["dhw"]
                dhw = L.odhw
                layers.append(L)
                cin = 2 * c
                continue
            L = Layer3("stem" if first else "conv", scope, block, layer, cin, c, k, s, dhw, coutp=cpb(c, block))
            L.odhw = tuple(-(-dhw[i] // s[i]) for i in range(3))
            lvl0 = pair and block in ("conv_e0", "conv_d0")
            if first:
                L.cinp = 32 if lvl0 else 64          # im2col pitch
                L.pair = "stem" if lvl0 else ""
            elif block.startswith("conv_d") and layer == "conv1":
                cp_ = cpb(c, block)
                L.cinp = 2 * cp_
                L.cin_map = np.r_[0:c, cp_:cp_ + c]
                L.pair = "conv" if lvl0 else ""
                L.catpair = bool(lvl0)
            elif pair and block == "conv_e1" and layer == "conv1":
                # reads the encoder half of the level-0 concat buffer: 64-lane voxel pairs with stride 128
                L.cinp = cpb(cin, "conv_e0")
                L.pair = "strided"
            else:
                L.cinp = cpb(cin, prev_block)
                L.pair = "conv" if lvl0 else ""
            if L.cin_map is None:
                L.cin_map = np.arange(cin)
            first = False
            prev_block = block
            dhw = L.odhw
            layers.append(L)
            cin = c
            if layer == "conv2" and (block.startswith("conv_e") or block == "bridge"):
                if block != "bridge":
                    L.fork = True
                    enc[block] = dict(c=c, dhw=dhw)
                c = min(c * 2, cfg.max_channels)
        L = Layer3("logits", "UNet3D/logits", "logits", "logits", cin, cfg.num_classes, (1, 1, 1), (1, 1, 1), dhw,
                   cinp=cpb(cin, "conv_d0"), coutp=cfg.num_classes)
        L.odhw = dhw
        L.cin_map = np.arange(cin)
        layers.append(L)
        self.layers = layers

    def _plan_params(self):
        """TF-shaped variables inside their padded stored layouts (concat inputs split as [encoder | up] by cin_map)."""
        cfg = self.cfg
        plist = []
        every = (slice(None),) * 3
        for L in self.layers:
            if L.kind in ("stem", "conv"):
                name, shape = f"{L.scope}/weights", L.k + (L.cin, L.cout)
                if L.kind == "stem":     # im2col rows (kh, kw, cin) of the 1x1 conv over the stem's im2col matrix
                    plist.append(Param(name, shape, (L.cinp, L.coutp), (slice(int(np.prod(shape[:4]))), slice(L.cout))))
                else:
                    plist.append(Param(name, shape, L.k + (L.cinp, L.coutp), every + (L.cin_map, slice(L.cout))))
                ns = f"{L.scope}/{self.norm_scope}"
                for v, region in (("gamma", "B"), ("beta", "B")) + ((("moving_mean", "S"), ("moving_variance", "S"))
                                                                     if self.bn else ()):
                    plist.append(Param(f"{ns}/{v}", (L.cout,), (L.coutp,), (slice(L.cout),), region=region))
            elif L.kind == "convT":
                plist.append(Param(f"{L.scope}/weights", L.k + (L.cout, L.cin), L.k + (L.coutp, L.cinp),
                                   every + (slice(L.cout), slice(L.cin))))
            else:
                plist.append(Param(f"{L.scope}/weights", (1, 1, 1, L.cin, L.cout), (L.cinp, L.cout),
                                   (L.cin_map, slice(None))))
                plist.append(Param(f"{L.scope}/biases", (L.cout,), region="B" if cfg.bias_decay else "A"))
        self._layout(plist)
        self._plan_super_filters()

    # ------------------------------------------------------------------ pixel-pair packing: super filters
    @staticmethod
    def _super_index(L: Layer3):
        """idx[i] = flat index into the layer's stored (master) filter that super-filter element i copies, or -1.
        Shapes: master (3, 3, cinp, coutp) [depth extent 1 dropped] / (cinp, coutp) for the stem;
        super (3, 3, 2*cinp, 64) / (3, 2, 2*cinp, coutp) for the strided layer / (64, 64)."""
        cinp, coutp = L.cinp, L.coutp
        if L.pair == "stem":
            idx = np.full((2, cinp, 2, coutp), -1, np.int64)
            m = np.arange(cinp * coutp).reshape(cinp, coutp)
            idx[0, :, 0, :] = m
            idx[1, :, 1, :] = m
            return idx.reshape(2 * cinp, 2 * coutp)
        m = np.arange(3 * 3 * cinp * coutp).reshape(3, 3, cinp, coutp)
        if L.pair == "strided":     # output voxel X reads input voxels 2X + s: super voxel X + (s >> 1), half s & 1
            idx = np.full((3, 2, 2, cinp, coutp), -1, np.int64)
            for s_ in range(3):
                idx[:, s_ >> 1, s_ & 1] = m[:, s_]
            return idx.reshape(3, 2, 2 * cinp, coutp)
        idx = np.full((3, 3, 2, cinp, 2, coutp), -1, np.int64)
        for sx in (-1, 0, 1):
            for hi in (0, 1):
                for ho in (0, 1):
                    s_ = 2 * sx + hi - ho + 1      # input voxel 2(X + sx) + hi, output voxel 2X + ho
                    if 0 <= s_ <= 2:
                        idx[:, sx + 1, hi, :, ho, :] = m[:, s_]
        if getattr(L, "catpair", False):
            # the input is the level's concat buffer: lanes [encoder even | encoder odd | up even | up odd] per voxel
            # pair, while the stored filter's input axis is [encoder | up] -> reduction order (part, half, lane)
            half = cinp // 2
            idx = idx.reshape(3, 3, 2, 2, half, 2, coutp).transpose(0, 1, 3, 2, 4, 5, 6)
        return idx.reshape(3, 3, 2 * cinp, 2 * coutp)

    @staticmethod
    def _fold_table(idx: np.ndarray, msize: int) -> np.ndarray:
        """Adjoint of the gather: fold[j] = the (at most two) super elements that copy stored element j, -1 = none."""
        idx = np.asarray(idx).ravel()
        order = np.argsort(idx, kind="stable")
        srt = idx[order]
        first = np.searchsorted(srt, np.arange(msize), side="left")
        last = np.searchsorted(srt, np.arange(msize), side="right")
        cnt = last - first
        assert cnt.max() <= 2, "a filter element is copied at most twice"
        fold = np.full((msize, 2), -1, np.int32)
        has1, has2 = cnt >= 1, cnt >= 2
        fold[has1, 0] = order[first[has1]]
        fold[has2, 1] = order[first[has2] + 1]
        return fold

    def _plan_super_filters(self):
        self.sup = {}
        pairs = [L for L in self.layers if L.pair]
        if not pairs:
            return
        off, gmax = 0, 0
        for L in pairs:
            idx = self._super_index(L).ravel()
            msize = self.params[f"{L.scope}/weights"].size
            fold = self._fold_table(idx, msize)
            self.sup[L.scope] = dict(off=off, size=idx.size, msize=msize,
                                     idx=self._upload_i32(idx.astype(np.int32)), fold=self._upload_i32(fold))
            off += _align(idx.size)
            gmax = max(gmax, idx.size)
        self.Wsup = self._alloc(off * BF16)
        self.Gsup = self._alloc(gmax * F32) if self.cfg.training else None

    def _upload_i32(self, a: np.ndarray) -> DeviceBuffer:
        b = self._alloc(a.nbytes)
        b.upload(np.ascontiguousarray(a, np.int32))
        return b

    def _wsup(self, L: Layer3):
        return C.c_void_p(self.Wsup.ptr + self.sup[L.scope]["off"] * BF16)

    def _pack_super_filters(self):
        """master fp32 filters -> bf16 super filters (start of every forward: the optimizer has just moved the masters)"""
        for L in self.layers:
            if L.pair:
                t = self.sup[L.scope]
                self.ctx.call("bsl_gather_f32_bf16", self._pp(self.W, f"{L.scope}/weights"), t["idx"].p,
                              C.c_size_t(t["size"]), self._wsup(L), self.stream)

    def _fold_super_grad(self, L: Layer3, stream):
        t = self.sup[L.scope]
        self.ctx.call("bsl_gather_add2_f32", self.Gsup.p, t["fold"].p, C.c_size_t(t["msize"]),
                      self._pp(self.G, f"{L.scope}/weights"), stream)

    def _pp(self, arena, name, esize=F32):
        return C.c_void_p(arena.ptr + self.params[name].offset * esize)

    def _plan_activations(self):
        cfg, n = self.cfg, self.cfg.batch
        cat, max_act, max_grad, small = {}, 0, 0, 0
        prev = None
        for L in self.layers:
            vox = int(np.prod(L.odhw))
            if L.kind in ("stem", "conv"):
                L.y = View3(self._alloc(n * vox * L.coutp * BF16), n, L.odhw, L.coutp)
                if L.fork:
                    cb = View3(self._alloc(n * vox * 2 * L.coutp * BF16).zero(), n, L.odhw, 2 * L.coutp)
                    cat[L.block] = cb
                    L.a = PairView(cb.buf, n, L.odhw, 0) if L.pair else cb.slice(0, L.coutp)
                else:
                    L.a = View3(self._alloc(n * vox * L.coutp * BF16), n, L.odhw, L.coutp)
                is_dec1 = L.block.startswith("conv_d") and L.layer == "conv1"
                L.x = cat[L.block.replace("d", "e")] if is_dec1 else prev
                prev = L.a
                L.norm_off = small
                small += self._norm_scalar_floats(n * L.coutp)
                max_act = max(max_act, vox * L.coutp)
                if L.kind == "conv" and not is_dec1:      # its dgrad writes in-voxels x cinp lanes into a ping-pong buffer
                    max_grad = max(max_grad, int(np.prod(L.dhw)) * L.cinp)
            elif L.kind == "convT":
                max_grad = max(max_grad, int(np.prod(L.dhw)) * L.cinp)
                L.x = prev
                cb = cat[L.block.replace("d", "e")]
                L.a = PairView(cb.buf, n, L.odhw, 1) if L.coutp == 32 else cb.slice(L.coutp, L.coutp)
                L.y = L.a
                prev = cb
            else:
                L.x = prev
        self.cat = cat
        d, h, w = cfg.depth, cfg.height, cfg.width
        nvox = n * d * h * w
        self.images = self._alloc(nvox * cfg.in_channels * F32)
        self.stem_col = self._alloc(nvox * self.layers[0].cinp * BF16)
        self.labels = self._alloc(nvox * 4)
        k = cfg.num_classes
        self.logits = self._alloc(nvox * k * F32)
        self.prob = self._alloc(nvox * k * F32)
        self.masks = self._alloc(nvox * (k - 1))
        self.argmax = self._alloc(nvox)
        self.ilr = self._alloc(n * (k - 1) * 3 * 4)
        self.counts = self._alloc(n * k * 4)
        self.loss_dev = self._alloc(16)
        self.small = self._alloc(max(small, 16) * F32)
        self.sums_sup = self._alloc(n * 2 * 64 * 8)       # fp64 [n][2][64]: statistics over super channels
        ld = self._loss_desc()
        self.loss_ws_bytes = self.ctx.lib.bsl_loss_workspace(self.ctx.h, C.byref(ld))
        self.loss_ws = self._alloc(self.loss_ws_bytes)
        if cfg.training:
            self.dlogits = self._alloc(nvox * k * F32)
            max_grad = max(max_grad, max_act, int(np.prod(self.layers[-1].dhw)) * self.layers[-1].cinp)
            self.g1 = self._alloc(n * max_grad * BF16)
            self.g2 = self._alloc(n * max_grad * BF16)
            self.dyb = [self._alloc(n * max_act * BF16), self._alloc(n * max_act * BF16)]
            self.dcat = {b: View3(self._alloc(v.voxels * v.c * BF16), n, v.dhw, v.c) for b, v in cat.items()}
            # pixel-pair packed level: the transposed conv's backward kernels read its 32-lane gradient DENSE (the two
            # column parities of an input voxel are then 64 contiguous values), so ReluGrad writes it here
            self.dup_dense = self._alloc(nvox * 32 * BF16) if self._pair else None
            ws = 0
            for L in self.layers:
                if L.kind == "stem":
                    dd = self._desc_stem(L)
                    ws = max(ws, self.ctx.lib.bsl_conv2d_wgrad_workspace(self.ctx.h, C.byref(dd)))
                elif L.kind == "conv":
                    if L.pair == "strided":
                        ws = max(ws, self.ctx.lib.bsl_conv3d_wgrad_workspace(self.ctx.h, C.byref(self._desc3s(L))))
                    elif self._is2d(L):
                        ws = max(ws, self.ctx.lib.bsl_conv2d_wgrad_workspace(self.ctx.h, C.byref(self._desc2(L))))
                    else:
                        ws = max(ws, self.ctx.lib.bsl_conv3d_wgrad_workspace(self.ctx.h, C.byref(self._desc3(L))))
                elif L.kind == "convT":
                    if L.s[0] == 1:
                        ws = max(ws, self.ctx.lib.bsl_convT2d_bwd_filter_workspace(self.ctx.h, C.byref(self._descT2(L))))
                    else:
                        ws = max(ws, self.ctx.lib.bsl_convT3d_bwd_filter_workspace(self.ctx.h, C.byref(self._descT3(L))))
            self.wgrad_ws_bytes = int(ws)
            self.wgrad_ws = self._alloc(max(ws, 16))

    # ------------------------------------------------------------------ descriptors
    @staticmethod
    def _is2d(L: Layer3):
        return L.k[0] == 1 and L.s == (1, 1, 1)

    def _desc2(self, L: Layer3):
        n = self.cfg.batch
        if L.pair == "conv":   # super voxels: [.., w, ld] seen as [.., w/2, 2*ld]; 2*coutp = 64 output lanes
            return _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2] // 2, 2 * L.cinp, 2 * L.coutp, L.k[1], L.k[2],
                                   2 * L.x.ld, 2 * L.y.ld)
        return _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.coutp, L.k[1], L.k[2], L.x.ld, L.y.ld)

    def _desc_stem(self, L: Layer3):
        """The stem as a 1x1 convolution over its im2col matrix (pitch cinp; pixel pairs when packed)."""
        n = self.cfg.batch
        if L.pair == "stem":
            return _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2] // 2, 2 * L.cinp, 2 * L.coutp, 1, 1, 2 * L.cinp,
                                   2 * L.y.ld)
        return _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], 64, L.coutp, 1, 1, 64, L.y.ld)

    def _desc3s(self, L: Layer3):
        """The strided conv that leaves the pixel-pair packed level: super voxels along W (stride 1 there, a 2-tap row:
        super voxels X and X + 1), the real strides along D and H. Its input is the encoder half of the concat buffer."""
        return _lib.Conv3dDesc(self.cfg.batch, L.dhw[0], L.dhw[1], L.dhw[2] // 2, 2 * L.cinp, L.coutp, L.k[0], L.k[1], 2,
                               L.s[0], L.s[1], 1, L.x.ld, L.y.ld)

    def _desc3(self, L: Layer3):
        return _lib.Conv3dDesc(self.cfg.batch, L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.coutp, L.k[0], L.k[1], L.k[2],
                               L.s[0], L.s[1], L.s[2], L.x.ld, L.y.ld)

    def _descT2(self, L: Layer3):
        return _lib.ConvT2dDesc(self.cfg.batch * L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.coutp, L.x.ld, L.a.ld, 1)

    def _descT3(self, L: Layer3):
        return _lib.ConvT3dDesc(self.cfg.batch, L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.coutp, L.s[0], L.x.ld, L.a.ld, 1)

    def _norm_desc(self, L: Layer3):
        cfg = self.cfg
        a_ld = L.coutp if isinstance(L.a, PairView) else L.a.ld     # (the pair view is written by two half calls)
        return _lib.NormDesc(0 if self.bn else 1, cfg.batch, int(np.prod(L.odhw)), L.coutp, L.y.ld, a_ld,
                             cfg.bn_eps if self.bn else cfg.in_eps, cfg.bn_decay if self.bn else 0.0, 1, 1, 1)

    def _norm_ptrs(self, L: Layer3):
        return self._norm_scalars(self.small.ptr + L.norm_off * F32, self.cfg.batch * L.coutp)

    def _loss_terms(self):
        return ["xentropy"] if "xentropy" in self.cfg.loss_type else []     # UNet3D.py:198-199

    def _flops(self, L: Layer3) -> float:
        n = self.cfg.batch
        taps = 1 if L.kind == "convT" else int(np.prod(L.k))
        return 2.0 * n * float(np.prod(L.odhw)) * taps * L.cin * L.cout

    def step_flops(self) -> dict:
        fwd = sum(self._flops(L) for L in self.layers)
        bwd = sum(self._flops(L) * (1 if L.kind == "stem" else 2) for L in self.layers)
        return {"fwd": fwd, "bwd": bwd, "total": fwd + bwd}

    # ------------------------------------------------------------------ inputs
    def set_inputs(self, images: np.ndarray, labels: np.ndarray | None = None, sp_guide: np.ndarray | None = None):
        cfg = self.cfg
        shp = (cfg.batch, cfg.depth, cfg.height, cfg.width)
        assert images.shape == shp + (cfg.channel,), images.shape
        if cfg.use_spatial:
            assert sp_guide is not None and sp_guide.shape == shp + (cfg.guide_channel,)
            images = np.concatenate((images, sp_guide), axis=-1)      # UNet3D.py:142-144
        self.images.upload(np.ascontiguousarray(images, np.float32))
        if labels is not None:
            assert labels.shape == shp, labels.shape
            self.labels.upload(np.ascontiguousarray(labels, np.int32))

    def get_stored_forward(self) -> dict:
        out = {}
        for L in self.layers:
            if L.kind == "logits":
                continue
            dct = {}
            for key, v in (("y", L.y), ("a", L.a)):
                if isinstance(v, PairView):     # [.., w/2, 128] -> this half's 64 lanes -> [.., w, 32]
                    full = self.ctx.bf16_to_f32(v.buf, (v.n,) + v.dhw[:2] + (v.dhw[2] // 2, 128))
                    full = full[..., v.c0:v.c0 + 64].reshape((v.n,) + v.dhw + (32,))
                    dct[key] = full[..., :L.cout].copy()
                    pad = full[..., L.cout:]
                else:
                    full = self.ctx.bf16_to_f32(v.buf, (v.n,) + v.dhw + (v.ld,))
                    dct[key] = full[..., v.c0:v.c0 + L.cout].copy()
                    pad = full[..., v.c0 + L.cout:v.c0 + v.c]
                assert not pad.any(), f"{L.scope}: pad lanes of {key} are not zero"
            out[L.scope] = dct
        return out

    # ------------------------------------------------------------------ forward
    def forward(self, is_training: bool = True):
        ctx, s, cfg = self.ctx, self.stream, self.cfg
        call = ctx.call
        n = cfg.batch
        self._pack_super_filters()
        # statistics come from the conv epilogue: per (volume, channel) for instance norm -- for layers that run as 2-D
        # convolutions over n*d images a statistics group is the `depth` consecutive images of one volume -- and per
        # channel over the whole batch for batch norm in training; batch-norm inference normalises with the moving
        # statistics and needs no sums. Pixel-pair packed layers sum over super channels (voxel parity, lane), folded to
        # the real channels afterwards.
        if self.bn and not is_training:
            conv2, conv3 = "bsl_conv2d_fprop", "bsl_conv3d_fprop"
        elif self.bn:
            conv2, conv3 = "bsl_conv2d_fprop_stats", "bsl_conv3d_fprop_stats"
        else:
            conv2, conv3 = "bsl_conv2d_fprop_group_stats", "bsl_conv3d_fprop_group_stats"
        with_sums = is_training or not self.bn
        for L in self.layers:
            ctx.tag = L.scope
            if L.kind in ("stem", "conv"):
                wbf = self._wsup(L) if L.pair else self._pp(self.Wbf, f"{L.scope}/weights", BF16)
                nd, q = self._norm_desc(L), self._norm_ptrs(L)
                sums = self.sums_sup.p if L.pair in ("conv", "stem") else q["sums"]
                extra3 = (sums,) if with_sums else ()
                extra2 = ((sums,) if self.bn else (C.c_int(L.dhw[0]), sums)) if with_sums else ()
                if L.kind == "stem":
                    d0 = _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], L.cin, 64, 3, 3, L.cin, 64)
                    call("bsl_stem_im2col_ld", C.byref(d0), self.images.p, self.stem_col.p, C.c_int(L.cinp), s)
                    call(conv2, C.byref(self._desc_stem(L)), self.stem_col.p, wbf, L.y.p, *extra2, s)
                elif self._is2d(L) and L.pair != "strided":
                    call(conv2, C.byref(self._desc2(L)), L.x.p, wbf, L.y.p, *extra2, s)
                else:
                    d3 = self._desc3s(L) if L.pair == "strided" else self._desc3(L)
                    call(conv3, C.byref(d3), L.x.p, wbf, L.y.p, *extra3, s)
                if with_sums and L.pair in ("conv", "stem"):
                    call("bsl_fold_pair_sums", sums, C.c_int(1 if self.bn else n), C.c_int(L.coutp), q["sums"], s)
                ns = f"{L.scope}/{self.norm_scope}"
                mm = self._pp(self.S, f"{ns}/moving_mean") if self.bn else None
                mv = self._pp(self.S, f"{ns}/moving_variance") if self.bn else None
                call("bsl_norm_finalize", C.byref(nd), C.c_int(1 if is_training else 0), q["sums"],
                     self._pp(self.W, f"{ns}/gamma"), self._pp(self.W, f"{ns}/beta"), mm, mv, q["mean"], q["rstd"],
                     q["scale"], q["shift"], s)
                if isinstance(L.a, PairView):
                    # even / odd voxels of the dense 32-lane tensor -> the two 32-lane quarters of the encoder half
                    ndh = _lib.NormDesc(nd.mode, n, nd.hw // 2, 32, 64, L.a.ld, nd.eps, nd.decay, 1, 1, 1)
                    for b in (0, 1):
                        call("bsl_norm_apply", C.byref(ndh), C.c_void_p(L.y.p.value + b * 32 * BF16), q["scale"], q["shift"],
                             C.c_void_p(L.a.p.value + b * 32 * BF16), s)
                else:
                    call("bsl_norm_apply", C.byref(nd), L.y.p, q["scale"], q["shift"], L.a.p, s)
            elif L.kind == "convT":
                wbf = self._pp(self.Wbf, f"{L.scope}/weights", BF16)
                if isinstance(L.a, PairView):
                    dT = _lib.ConvT2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.coutp, L.x.ld, L.a.ld, 1)
                    call("bsl_convT2d_fwd_pairs", C.byref(dT), L.x.p, wbf, L.a.p, s)
                elif L.s[0] == 1:
                    call("bsl_convT2d_fwd", C.byref(self._descT2(L)), L.x.p, wbf, None, L.a.p, s)
                else:
                    call("bsl_convT3d_fwd", C.byref(self._descT3(L)), L.x.p, wbf, None, L.a.p, s)
            else:
                dh = _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.cout, 1, 1, L.x.ld, L.cout)
                call("bsl_conv2d_head_fprop", C.byref(dh), L.x.p, self._pp(self.W, f"{L.scope}/weights"),
                     self._pp(self.W, f"{L.scope}/biases"), self.logits.p, s)

    # ------------------------------------------------------------------ loss + backward
    def loss_backward(self):
        ctx, s, cfg = self.ctx, self.stream, self.cfg
        call = ctx.call
        n = cfg.batch
        ld = self._loss_desc()
        call("bsl_label_counts", C.byref(ld), self.labels.p, self.counts.p, s)
        call("bsl_wxent_fwd_bwd", C.byref(ld), self.logits.p, self.labels.p, self.counts.p, self.loss_dev.p,
             self.dlogits.p, self.loss_ws.p, C.c_size_t(self.loss_ws_bytes), s)
        cur, alt = self.g1, self.g2
        cur_ld = 0          # channel stride of the gradient currently in `cur`
        wsb = C.c_size_t(self.wgrad_ws_bytes)
        overlap = self._overlap_wgrad and ctx._prof is None
        ws = self.wg_stream if overlap else s
        busy = [None, None]
        k = 0

        def fork():
            if overlap:
                self._stream_wait(ws, s)

        for L in reversed(self.layers):
            ctx.tag = L.scope
            if L.kind == "logits":
                dh = _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.cout, 1, 1, L.x.ld, L.cout)
                fork()
                call("bsl_conv2d_head_wgrad", C.byref(dh), L.x.p, self.dlogits.p, self._pp(self.G, f"{L.scope}/weights"),
                     self._pp(self.G, f"{L.scope}/biases"), ws)
                dh2 = _lib.Conv2dDesc(n * L.dhw[0], L.dhw[1], L.dhw[2], L.cinp, L.cout, 1, 1, L.cinp, L.cout)
                call("bsl_conv2d_head_dgrad", C.byref(dh2), self.dlogits.p, self._pp(self.W, f"{L.scope}/weights"), cur.p, s)
                cur_ld = L.cinp
            elif L.kind in ("stem", "conv"):
                vox = n * int(np.prod(L.odhw))
                if L.fork:   # AddN: gradient through the next block's strided conv + gradient through the skip
                    dc = self.dcat[L.block]
                    if isinstance(L.a, PairView):    # voxel pairs: 64 dense lanes + the encoder half of the concat gradient
                        assert cur_ld == 32
                        call("bsl_add_bf16", C.c_longlong(vox // 2), C.c_int(64), cur.p, C.c_int(64), dc.p,
                             C.c_int(L.a.ld), alt.p, C.c_int(64), s)
                    else:
                        call("bsl_add_bf16", C.c_longlong(vox), C.c_int(L.coutp), cur.p, C.c_int(cur_ld), dc.p,
                             C.c_int(dc.ld), alt.p, C.c_int(L.coutp), s)
                    cur, alt = alt, cur
                    cur_ld = L.coutp
                assert cur_ld == L.coutp, (L.scope, cur_ld, L.coutp)
                dyb = self.dyb[k]
                if overlap and busy[k] is not None:
                    call("bsl_stream_wait_event", s, busy[k])
                nd, q = self._norm_desc(L), self._norm_ptrs(L)
                call("bsl_norm_bwd_reduce", C.byref(nd), L.y.p, cur.p, C.c_int(L.coutp), q["mean"], q["rstd"], q["scale"],
                     q["shift"], q["sums"], s)
                call("bsl_norm_bwd_finalize", C.byref(nd), q["sums"], q["c1"], q["c2"],
                     self._pp(self.G, f"{L.scope}/{self.norm_scope}/gamma"),
                     self._pp(self.G, f"{L.scope}/{self.norm_scope}/beta"), s)
                call("bsl_norm_bwd_apply", C.byref(nd), L.y.p, cur.p, C.c_int(L.coutp), q["mean"], q["rstd"], q["scale"],
                     q["shift"], q["c1"], q["c2"], dyb.p, C.c_int(L.coutp), s)
                # pixel-pair packed layers: the filter gradient of the SUPER filter goes to scratch and is folded back onto
                # the stored filter (each stored element is the sum of the <= 2 super elements that copy it)
                gw = self.Gsup.p if L.pair else self._pp(self.G, f"{L.scope}/weights")
                wbf = self._wsup(L) if L.pair else self._pp(self.Wbf, f"{L.scope}/weights", BF16)
                sup = 2 if L.pair in ("conv", "stem") else 1        # output lanes per super voxel / coutp
                fork()
                if L.kind == "stem":
                    d1 = self._desc_stem(L)
                    d1.y_ld = sup * L.coutp
                    call("bsl_conv2d_wgrad", C.byref(d1), self.stem_col.p, dyb.p, gw, self.wgrad_ws.p, wsb, ws)
                else:
                    is_dec1 = L.block.startswith("conv_d") and L.layer == "conv1"
                    dx = self.dcat[L.block.replace("d", "e")] if is_dec1 else None
                    two_d = self._is2d(L) and L.pair != "strided"
                    mk = (lambda: self._desc3s(L)) if L.pair == "strided" else ((lambda: self._desc2(L)) if two_d else
                                                                                 (lambda: self._desc3(L)))
                    d = mk()
                    d.y_ld = sup * L.coutp
                    call("bsl_conv2d_wgrad" if two_d else "bsl_conv3d_wgrad", C.byref(d), L.x.p, dyb.p, gw,
                         self.wgrad_ws.p, wsb, ws)
                    dd = mk()
                    dd.y_ld = sup * L.coutp
                    xin = 2 if L.pair else 1                        # input lanes per super voxel / stored lanes
                    dd.x_ld = xin * (dx.ld if dx is not None else L.cinp)
                    call("bsl_conv2d_dgrad" if two_d else "bsl_conv3d_dgrad", C.byref(dd), dyb.p, wbf,
                         dx.p if dx is not None else cur.p, s)
                    cur_ld = L.cinp
                if L.pair:
                    self._fold_super_grad(L, ws)
                if overlap:
                    busy[k] = self._dy_events[k]
                    ctx.record(busy[k], ws)
                k ^= 1
            else:  # convT
                dc = self.dcat[L.block.replace("d", "e")]
                dup = dc.slice(L.coutp, L.coutp)
                vox = n * int(np.prod(L.odhw))
                if isinstance(L.a, PairView):   # voxel pairs of the `up` half -> dense 32-lane gradient
                    dpv = PairView(dc.buf, n, L.odhw, 1)
                    dup = View3(self.dup_dense, n, L.odhw, 32)
                    call("bsl_relu_bwd", C.c_longlong(vox // 2), C.c_int(64), L.a.p, C.c_int(L.a.ld), dpv.p,
                         C.c_int(dpv.ld), dup.p, C.c_int(64), s)
                else:
                    call("bsl_relu_bwd", C.c_longlong(vox), C.c_int(L.coutp), L.a.p, C.c_int(L.a.ld), dup.p,
                         C.c_int(dup.ld), dup.p, C.c_int(dup.ld), s)
                gw = self._pp(self.G, f"{L.scope}/weights")
                wbf = self._pp(self.Wbf, f"{L.scope}/weights", BF16)
                two_d = L.s[0] == 1
                d = self._descT2(L) if two_d else self._descT3(L)
                d.y_ld = dup.ld
                fork()
                call("bsl_convT2d_bwd_filter" if two_d else "bsl_convT3d_bwd_filter", C.byref(d), L.x.p, dup.p, gw, None,
                     self.wgrad_ws.p, wsb, ws)
                dd = self._descT2(L) if two_d else self._descT3(L)
                dd.y_ld = dup.ld
                dd.x_ld = L.cinp
                call("bsl_convT2d_bwd_data" if two_d else "bsl_convT3d_bwd_data", C.byref(dd), dup.p, wbf, cur.p, s)
                cur_ld = L.cinp
        if overlap:
            self._stream_wait(s, ws)

    # ------------------------------------------------------------------ optimizer / step
    def attach_comm(self, rank: int, world: int, unique_id: bytes):
        assert world == self.cfg.world
        self.ctx.attach_comm(rank, world, unique_id)

    def train_step(self, lr: float, with_metrics: bool = False):
        self.forward(True)
        self._allreduce_moving_stats()
        if with_metrics:
            self.predict_outputs(True)
        self.loss_backward()
        if self.cfg.world > 1:
            self.ctx.call("bsl_allreduce_sum_f32", self.G.p, C.c_size_t(self.n_train), self.stream)
        self.optimizer_step(lr)
