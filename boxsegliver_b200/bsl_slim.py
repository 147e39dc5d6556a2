"""`bsl_slim`: the slim layer-function seam of the reference (SURVEY.md section 8b) as a graph-capturing front end.

The reference's model classes build their networks out of `tf.contrib.slim` calls
(/root/reference/NetworksV2/UNet.py:45-117): `slim.arg_scope`, `slim.repeat`, `slim.conv2d`, `slim.max_pool2d`,
`slim.conv2d_transpose`, `tf.concat`, `tf.variable_scope`. This module offers the same functions with the same
signatures, defaults and VARIABLE-NAMING rules, so that the body of `UNet._build_network` runs textually unchanged
with `import boxsegliver_b200.bsl_slim as slim` (and `tf = slim.tf`). Like TF-1.x graph mode, calling a layer function
computes nothing: it appends a node to the default `Graph` and returns a symbolic `Tensor`. `lower(graph, ctx, ...)`
then recognises the U-Net family the accelerated path covers --

    [conv3x3 + norm + ReLU] x 2 -> max_pool 2x2 (x depth) -> bridge -> [conv_transpose 2x2/2 + bias + ReLU ->
    concat(skip, up) -> [conv3x3 + norm + ReLU] x 2] (x depth) -> conv1x1 + bias

with every 3x3 convolution either normalised (one normaliser throughout) or, with normalizer_fn=None, conv + bias + ReLU
(engine --without_norm)

-- and turns it into the layer table of `engine.UNetEngine`, i.e. into exactly the C-ABI launch sequence the engine
issues (fused statistics epilogues, norm+pool in one pass, zero-copy concat, ...). Anything else raises
NotImplementedError naming the node: a drop-in must never silently run something different.

Naming rules restated from tensorflow/contrib/layers (TF 1.13):
  * `variable_scope(name_or_scope, default_name)`: an explicit name is used as is (re-entering it is allowed);
    `None` takes `default_name`, uniquified within the parent scope as `name`, `name_1`, `name_2`, ...;
  * `slim.conv2d` is `convolution2d` (default scope "Conv"), `slim.conv2d_transpose` defaults to "Conv2d_transpose",
    `slim.batch_norm` to "BatchNorm", `slim.instance_norm` to "InstanceNorm", `slim.max_pool2d` to "MaxPool2D";
  * `slim.repeat(x, n, layer, *args, scope=S)` opens `variable_scope(S, "Repeat")` and calls
    `layer(..., scope=(S or layer.__name__) + "_" + str(i + 1))`;
  * a `normalizer_fn` drops the conv bias; variables are "weights" / "biases" / "beta" / "gamma" / "moving_*".
"""
from __future__ import annotations

import contextlib
import functools
from dataclasses import dataclass, field

import numpy as np


# ------------------------------------------------------------------------------------------------ graph objects
@dataclass
class Node:
    kind: str                      # input | conv | conv_transpose | max_pool | concat | softmax
    name: str                      # full variable scope of the layer ("UNet/Encode1/Repeat/convolution2d_1")
    inputs: list
    attrs: dict = field(default_factory=dict)


class Tensor:
    """Symbolic NHWC tensor: static shape + the node that produces it."""

    def __init__(self, shape, node: Node):
        self.shape = tuple(shape)
        self.node = node

    def get_shape(self):
        return list(self.shape)

    def set_shape(self, shape):
        shape = tuple(shape)
        assert len(shape) == len(self.shape) and all(a is None or b is None or a == b for a, b in zip(shape, self.shape))
        self.shape = tuple(b if a is None else a for a, b in zip(shape, self.shape))


class Graph:
    def __init__(self):
        self.nodes: list[Node] = []
        self.scope_stack: list[str] = []
        self.used: dict[str, dict[str, int]] = {}       # parent scope -> default name -> count
        self.arg_stack: list[dict] = [{}]

    def add(self, node: Node) -> Node:
        self.nodes.append(node)
        return node


_default = [Graph()]


def get_default_graph() -> Graph:
    return _default[-1]


@contextlib.contextmanager
def graph_as_default(g: Graph | None = None):
    g = g or Graph()
    _default.append(g)
    try:
        yield g
    finally:
        _default.pop()


def placeholder(shape, name="images") -> Tensor:
    g = get_default_graph()
    return Tensor(shape, g.add(Node("input", name, [])))


# ------------------------------------------------------------------------------------------------ scopes
@contextlib.contextmanager
def variable_scope(name_or_scope=None, default_name=None, values=None, reuse=None):
    g = get_default_graph()
    parent = "/".join(g.scope_stack)
    if name_or_scope is None:
        if default_name is None:
            raise ValueError("If default_name is None then name_or_scope is required")
        counts = g.used.setdefault(parent, {})
        k = counts.get(default_name, 0)
        counts[default_name] = k + 1
        name = default_name if k == 0 else f"{default_name}_{k}"
    else:
        name = str(name_or_scope)
        g.used.setdefault(parent, {}).setdefault(name, 1)
    g.scope_stack.append(name)
    try:
        yield "/".join(g.scope_stack)
    finally:
        g.scope_stack.pop()


_ARG_SCOPED = {}


def add_arg_scope(fn):
    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        defaults = get_default_graph().arg_stack[-1].get(fn.__name__, {})
        merged = dict(defaults)
        merged.update(kwargs)
        return fn(*args, **merged)
    wrapper._arg_scope_key = fn.__name__
    _ARG_SCOPED[fn.__name__] = wrapper
    return wrapper


@contextlib.contextmanager
def arg_scope(list_ops_or_scope, **kwargs):
    """slim.arg_scope: either a list of arg-scoped functions + defaults, or a scope captured earlier (re-entered)."""
    g = get_default_graph()
    if isinstance(list_ops_or_scope, dict):
        if kwargs:
            raise ValueError("When attempting to re-use a scope by suppling a dictionary, kwargs must be empty.")
        new = {k: dict(v) for k, v in list_ops_or_scope.items()}
    else:
        new = {k: dict(v) for k, v in g.arg_stack[-1].items()}
        for op in list_ops_or_scope:
            key = getattr(op, "_arg_scope_key", None)
            if key is None:
                raise ValueError("%s is not decorated with @add_arg_scope" % getattr(op, "__name__", op))
            new.setdefault(key, {}).update(kwargs)
    g.arg_stack.append(new)
    try:
        yield new
    finally:
        g.arg_stack.pop()


def current_arg_scope():
    return get_default_graph().arg_stack[-1]


# ------------------------------------------------------------------------------------------------ initialisers etc.
def xavier_initializer(uniform=True, seed=None):
    return ("xavier", dict(uniform=uniform, seed=seed))


def l2_regularizer(scale, scope=None):
    return ("l2", float(scale))


def relu(x):        # tf.nn.relu as an activation_fn marker
    return x


relu.__name__ = "relu"


@add_arg_scope
def batch_norm(inputs, decay=0.999, center=True, scale=False, epsilon=0.001, is_training=True, scope=None, **kw):
    raise TypeError("bsl_slim.batch_norm is used as a normalizer_fn marker of conv2d, not called directly")


@add_arg_scope
def instance_norm(inputs, center=True, scale=True, epsilon=1e-6, scope=None, **kw):
    raise TypeError("bsl_slim.instance_norm is used as a normalizer_fn marker of conv2d, not called directly")


def _pair(v):
    return (int(v), int(v)) if np.isscalar(v) else tuple(int(a) for a in v)


# ------------------------------------------------------------------------------------------------ layers
@add_arg_scope
def convolution2d(inputs, num_outputs, kernel_size, stride=1, padding="SAME", data_format=None, rate=1,
                  activation_fn=relu, normalizer_fn=None, normalizer_params=None, weights_initializer=None,
                  weights_regularizer=None, biases_initializer="zeros", biases_regularizer=None, reuse=None,
                  variables_collections=None, outputs_collections=None, trainable=True, scope=None):
    g = get_default_graph()
    with variable_scope(scope, "Conv") as sc:
        n, h, w, cin = inputs.shape
        k, s = _pair(kernel_size), _pair(stride)
        if padding != "SAME":
            raise NotImplementedError(f"{sc}: padding {padding!r} (the accelerated path covers SAME)")
        oh, ow = -(-h // s[0]), -(-w // s[1])
        attrs = dict(cin=cin, cout=int(num_outputs), kernel=k, stride=s, rate=_pair(rate), activation=activation_fn,
                     normalizer=None, norm_params={}, has_bias=normalizer_fn is None and biases_initializer is not None,
                     weights_regularizer=weights_regularizer, biases_regularizer=biases_regularizer,
                     weights_initializer=weights_initializer, in_hw=(h, w))
        if normalizer_fn is not None:
            key = getattr(normalizer_fn, "_arg_scope_key", None)
            if key not in ("batch_norm", "instance_norm"):
                raise NotImplementedError(f"{sc}: normalizer_fn {normalizer_fn!r}")
            params = dict(g.arg_stack[-1].get(key, {}))
            params.update(normalizer_params or {})
            attrs["normalizer"] = key
            attrs["norm_params"] = params
        node = g.add(Node("conv", sc, [inputs], attrs))
        return Tensor((n, oh, ow, int(num_outputs)), node)


conv2d = convolution2d


@add_arg_scope
def convolution2d_transpose(inputs, num_outputs, kernel_size, stride=1, padding="SAME", data_format=None,
                            activation_fn=relu, normalizer_fn=None, normalizer_params=None, weights_initializer=None,
                            weights_regularizer=None, biases_initializer="zeros", biases_regularizer=None, reuse=None,
                            variables_collections=None, outputs_collections=None, trainable=True, scope=None):
    g = get_default_graph()
    with variable_scope(scope, "Conv2d_transpose") as sc:
        n, h, w, cin = inputs.shape
        k, s = _pair(kernel_size), _pair(stride)
        attrs = dict(cin=cin, cout=int(num_outputs), kernel=k, stride=s, activation=activation_fn,
                     normalizer=getattr(normalizer_fn, "_arg_scope_key", None) if normalizer_fn else None,
                     has_bias=normalizer_fn is None and biases_initializer is not None,
                     weights_regularizer=weights_regularizer, biases_regularizer=biases_regularizer, in_hw=(h, w))
        node = g.add(Node("conv_transpose", sc, [inputs], attrs))
        return Tensor((n, h * s[0], w * s[1], int(num_outputs)), node)


conv2d_transpose = convolution2d_transpose


@add_arg_scope
def max_pool2d(inputs, kernel_size, stride=2, padding="VALID", data_format=None, outputs_collections=None, scope=None):
    g = get_default_graph()
    with variable_scope(scope, "MaxPool2D") as sc:
        n, h, w, c = inputs.shape
        k, s = _pair(kernel_size), _pair(stride)
        node = g.add(Node("max_pool", sc, [inputs], dict(kernel=k, stride=s, padding=padding)))
        if padding == "VALID":
            oh, ow = (h - k[0]) // s[0] + 1, (w - k[1]) // s[1] + 1
        else:
            oh, ow = -(-h // s[0]), -(-w // s[1])
        return Tensor((n, oh, ow, c), node)


def repeat(inputs, repetitions, layer, *args, **kwargs):
    scope = kwargs.pop("scope", None)
    with variable_scope(scope, "Repeat"):
        scope = scope or getattr(layer, "__name__", "repeat")
        outputs = inputs
        for i in range(repetitions):
            kwargs["scope"] = scope + "_" + str(i + 1)
            outputs = layer(outputs, *args, **kwargs)
        return outputs


def softmax(logits, scope=None):
    g = get_default_graph()
    with variable_scope(scope, "softmax") as sc:
        return Tensor(logits.shape, g.add(Node("softmax", sc, [logits])))


def concat(values, axis=-1, name="concat"):
    g = get_default_graph()
    shapes = [v.shape for v in values]
    if axis not in (-1, 3) or any(s[:3] != shapes[0][:3] for s in shapes):
        raise NotImplementedError("concat: channel-axis concatenation of equally sized NHWC tensors only")
    node = g.add(Node("concat", "/".join(g.scope_stack + [name]), list(values)))
    return Tensor(shapes[0][:3] + (sum(s[3] for s in shapes),), node)


class _TfNamespace:
    """The handful of `tf.*` symbols UNet._build_network touches, so the method body needs no edit beyond imports."""
    variable_scope = staticmethod(variable_scope)
    concat = staticmethod(concat)

    class nn:
        relu = staticmethod(relu)


tf = _TfNamespace()


# ------------------------------------------------------------------------------------------------ lowering
def _fail(node: Node, why: str):
    raise NotImplementedError(f"bsl_slim.lower: node {node.name!r} ({node.kind}) is outside the accelerated U-Net "
                              f"family: {why}")


def lower_to_layer_table(graph: Graph, logits: Tensor):
    """Pattern-match the captured graph; returns (list of layer dicts in forward order, summary dict).
    Layer dict keys mirror engine.ConvL: kind, scope, cin, cout, h, w (input size), level, role."""
    # walk back from the logits along the trunk
    order = []
    seen = set()

    def visit(t: Tensor):
        if id(t.node) in seen:
            return
        seen.add(id(t.node))
        for i in t.node.inputs:
            visit(i)
        order.append(t)

    visit(logits)
    nodes = [t.node for t in order]
    if nodes[0].kind != "input":
        _fail(nodes[0], "the trunk must start at the images placeholder")
    batch, height, width, channel = order[0].shape
    layers, level, skips = [], 0, {}
    phase = "enc"
    convs_at_level = 0
    normalizer = None
    norm_params = None
    norms_seen = set()     # normalizer attribute of every 3x3 conv (None: conv + bias + ReLU)
    regs = set()
    it = list(zip(order[1:], nodes[1:]))
    pos = 0
    depth = sum(1 for _, nd in it if nd.kind == "max_pool")
    pending_up = None
    for t, nd in it:
        a = nd.attrs
        if nd.kind == "conv":
            h, w = a["in_hw"]
            if a["kernel"] == (3, 3):
                if a["stride"] != (1, 1) or a["rate"] != (1, 1):
                    _fail(nd, f"stride {a['stride']} / rate {a['rate']} (3x3 stride 1 rate 1 is covered)")
                if a["activation"] is not relu or (a["normalizer"] is None and not a["has_bias"]):
                    _fail(nd, "3x3 convolutions are conv + batch/instance norm + ReLU, or conv + bias + ReLU")
                norms_seen.add(a["normalizer"])
                if len(norms_seen) > 1:
                    _fail(nd, "mixed normalisers (normalised and plain 3x3 convolutions count as mixed)")
                normalizer, norm_params = a["normalizer"], a["norm_params"]
                convs_at_level += 1
                if convs_at_level > 2:
                    _fail(nd, "more than two convolutions in a block")
                if phase == "enc":
                    role = f"enc{convs_at_level}" if level < depth else f"bridge{convs_at_level}"
                else:
                    role = f"dec{convs_at_level}"
                    if convs_at_level == 1 and nd.inputs[0].node.kind != "concat":
                        _fail(nd, "the first decoder convolution reads concat(skip, up)")
                kind = "stem" if not layers else "conv"
                layers.append(dict(kind=kind, scope=nd.name, cin=a["cin"], cout=a["cout"], h=h, w=w, level=level, role=role))
                regs.add((a["weights_regularizer"], a["biases_regularizer"]))
            elif a["kernel"] == (1, 1):
                if a["normalizer"] is not None or a["activation"] is not None or not a["has_bias"]:
                    _fail(nd, "the 1x1 convolution is the logits layer: bias, no normaliser, no activation")
                if t is not logits:
                    _fail(nd, "1x1 convolution that is not the final logits layer")
                layers.append(dict(kind="logits", scope=nd.name, cin=a["cin"], cout=a["cout"], h=h, w=w, level=0, role=""))
            else:
                _fail(nd, f"kernel {a['kernel']}")
        elif nd.kind == "max_pool":
            if a["kernel"] != (2, 2) or a["stride"] != (2, 2) or phase != "enc" or convs_at_level != 2:
                _fail(nd, "2x2 stride-2 pooling after the second convolution of an encoder block")
            skips[level] = nd.inputs[0]
            level += 1
            convs_at_level = 0
        elif nd.kind == "conv_transpose":
            if a["kernel"] != (2, 2) or a["stride"] != (2, 2) or a["normalizer"] or a["activation"] is not relu or not a["has_bias"]:
                _fail(nd, "conv2d_transpose 2x2 stride 2 with bias + ReLU")
            if convs_at_level != 2:
                _fail(nd, "up-sampling follows a block of two convolutions")
            phase = "dec"
            level -= 1
            convs_at_level = 0
            h, w = a["in_hw"]
            layers.append(dict(kind="convT", scope=nd.name, cin=a["cin"], cout=a["cout"], h=h, w=w, level=level, role=""))
            pending_up = t
        elif nd.kind == "concat":
            if len(nd.inputs) != 2 or nd.inputs[0] is not skips.get(level) or nd.inputs[1] is not pending_up:
                _fail(nd, "concat((encoder output of the same level, up-sampled tensor)) in that order")
        else:
            _fail(nd, "unsupported op on the trunk")
        pos += 1
    if not layers or layers[-1]["kind"] != "logits" or level != 0:
        raise NotImplementedError("bsl_slim.lower: the graph does not end in the logits layer at full resolution")
    summary = dict(batch=batch, height=height, width=width, channel=channel, num_down_samples=depth,
                   init_channels=layers[0]["cout"], normalizer=normalizer, norm_params=norm_params,
                   num_classes=layers[-1]["cout"], regularizers=regs)
    return layers, summary


def lower(graph: Graph, logits: Tensor, ctx, classes, **engine_kw):
    """Captured graph -> a planned engine (engine.UNetEngine subclass whose layer table comes from the graph)."""
    from .engine import ConvL, EngineConfig, UNetEngine

    table, info = lower_to_layer_table(graph, logits)
    if len(classes) != info["num_classes"]:
        raise ValueError(f"{len(classes)} classes but the logits layer has {info['num_classes']} outputs")
    np_ = info["norm_params"] or {}
    if info["normalizer"] is None:
        engine_kw["without_norm"] = True
    elif info["normalizer"] == "batch_norm":
        if not np_.get("scale", False):
            raise NotImplementedError("bsl_slim.lower: batch_norm without scale (the reference passes scale=True)")
        engine_kw.setdefault("bn_decay", np_.get("decay", 0.999))
        engine_kw.setdefault("bn_eps", np_.get("epsilon", 0.001))
    wd = [r for pair in info["regularizers"] for r in pair[:1] if r]
    rate = wd[0][1] if wd else 0.0
    bias_reg = any(pair[1] for pair in info["regularizers"])
    cfg = EngineConfig(batch=info["batch"], height=info["height"], width=info["width"], channel=info["channel"],
                       classes=tuple(classes), init_channels=info["init_channels"],
                       num_down_samples=info["num_down_samples"], normalizer=info["normalizer"] or "batch_norm",
                       weight_decay_rate=rate, bias_decay=bool(wd) and not bias_reg, **engine_kw)

    class GraphEngine(UNetEngine):
        """UNetEngine planned from a captured bsl_slim graph instead of its built-in layer table."""

        def _layer_specs(self):
            return [ConvL(L["kind"], L["scope"], L["cin"], L["cout"], L["h"], L["w"], L["level"], role=L["role"])
                    for L in table]

    return GraphEngine(ctx, cfg)
