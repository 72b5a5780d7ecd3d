"""Run an exported model on its integer codes.

``build_integer_model(model, blob)`` returns an eval-mode copy of ``model`` (sharing the parameters
of the layers it keeps) in which every quantized
``Sequential(activations_quantizer=NoisyAct, "0"=NoisyConv2d | NoisyLinear)`` of ``blob`` (from
``export_quantized``) is an ``IntegerConv2d`` / ``IntegerLinear``: the layer quantizes its fp32 input
to uint8 activation codes and runs an int8 tensor-core GEMM against the exported weight codes
(include/mhaq_fq.h "Integer layers", DESIGN §3).  Everything between those layers (BN, ReLU,
pooling, residual adds, unquantized layers) stays as it is.

The convolution geometry (stride, padding, and with ``allow_groups_and_dilation=True`` groups and
dilation) comes from the model's modules; every number comes
from the blob: the weight codes are unpacked from the packed format with integer operations, never
re-derived from dequantized floats.
"""
import collections
import copy
import dataclasses
import operator
from typing import Optional

import torch
import torch.nn.functional as F
from torch import fx, nn

from ... import ops
from ...aux.types import is_per_channel
from .export import FORMAT, VERSION, _layer_kind
from .layers.gdnsq_conv2d import NoisyConv2d
from .layers.gdnsq_linear import NoisyLinear


def unpack_weight_codes(e) -> torch.Tensor:
    """int64 codes ``[O, ...]`` (the layer's weight shape, row-major logical order) of an export
    entry, from its packed rows (one row per output channel, or one row for a per-tensor weight)."""
    bits, data, shape = e["bits"], e["codes"], tuple(e["shape"])
    numel = 1
    for s in shape:
        numel *= s
    rows = data.shape[0]
    per = 8 // bits
    shifts = torch.arange(per, dtype=torch.int64, device=data.device) * bits
    codes = (data.to(torch.int64)[:, :, None] >> shifts) & ((1 << bits) - 1)
    return codes.reshape(rows, -1)[:, :numel // rows].reshape(shape)


class _IntegerLayer(nn.Module):
    def __init__(self, act, operands: ops.IntLayerOperands):
        super().__init__()
        dev = operands.weight.device
        self.act_scale, self.act_zero_point, self.act_max_val = (
            act[k].to(device=dev, dtype=torch.float32).reshape(1).contiguous()
            for k in ("scale", "zero_point", "max_val"))
        self.operands = operands


class IntegerConv2d(_IntegerLayer):
    """``NoisyAct`` + ``NoisyConv2d`` (eval) on integer codes; returns channels_last fp32.

    An input whose code falls outside [0, 255] (only NaN can: the codes are clamped) is saturated,
    NaN to code 0, and the forward neither counts nor reports it, so it stays free of host
    synchronisation; the fake-quant layer would propagate the NaN instead.  ``ops.act_codes``
    with ``check=True`` finds such inputs."""

    def __init__(self, act, operands, stride, padding):
        super().__init__(act, operands)
        self.stride, self.padding = tuple(stride), tuple(padding)
        self.dilation, self.groups = tuple(operands.dilation), operands.groups

    def forward(self, x):
        codes, _ = ops.act_codes(x, self.act_scale, self.act_zero_point, self.act_max_val)
        return ops.int_conv2d(codes, self.operands, self.stride, self.padding)


class IntegerLinear(_IntegerLayer):
    """``NoisyAct`` + ``NoisyLinear`` (eval) on integer codes.  NaN inputs are saturated to code 0
    without a report, as in ``IntegerConv2d``."""

    def forward(self, x):
        lead = x.shape[:-1]
        codes, _ = ops.act_codes(x.reshape(-1, x.shape[-1]), self.act_scale, self.act_zero_point,
                                 self.act_max_val)
        return ops.int_linear(codes, self.operands).reshape(*lead, self.operands.n_out)


def _qscheme(m):
    return "PER_CHANNEL" if is_per_channel(m.qscheme) else "PER_TENSOR"


def _check_pair(name, act_e, w, we, allow_groups_and_dilation=False):
    """ValueError naming the layer for everything the integer kernels cannot run exactly (grouped
    and dilated convolutions unless ``allow_groups_and_dilation``)."""
    if act_e["disabled"]:
        raise ValueError(f"build_integer_model: {name}: the activation quantizer is disabled (act_bit = -1); "
                         "an integer layer needs activation codes")
    if act_e["n_levels"] > 256:
        raise ValueError(f"build_integer_model: {name}: {act_e['n_levels']} activation levels do not fit uint8 codes")
    if we["bits"] > 8:
        raise ValueError(f"build_integer_model: {name}: {we['bits']}-bit weight codes are not supported (at most 8)")
    if list(w.weight.shape) != list(we["shape"]) or we["qscheme"] != _qscheme(w):
        raise ValueError(f"build_integer_model: {name}: the model's layer differs from the export's "
                         "(shape or qscheme)")
    dense = not isinstance(w, NoisyConv2d) or (w.groups == 1 and tuple(w.dilation) == (1, 1))
    if isinstance(w, NoisyConv2d):
        if not dense and not allow_groups_and_dilation:
            raise ValueError(f"build_integer_model: {name}: grouped or dilated convolutions are not supported")
        if w.padding_mode != "zeros" or isinstance(w.padding, str):
            raise ValueError(f"build_integer_model: {name}: only explicit zero padding is supported "
                             f"(padding_mode={w.padding_mode!r}, padding={w.padding!r})")
    kk = w.weight[0, 0].numel() if w.weight.dim() == 4 else 1
    # a grouped / dilated channel sums kh * kw * (C / groups) products, without padding channels
    k_bytes = kk * (ops.code_channels(w.weight.shape[1]) if dense else w.weight.shape[1])
    if not ops.int32_bound_ok(k_bytes, max(1, act_e["n_levels"] - 1), (1 << we["bits"]) - 1):
        raise ValueError(f"build_integer_model: {name}: K * (n_levels - 1) * (2^bits - 1) >= 2^31 would "
                         "overflow the int32 accumulator")


def _integer_layer(name, act_e, w, we, allow_groups_and_dilation=False):
    _check_pair(name, act_e, w, we, allow_groups_and_dilation)
    dev = w.weight.device
    cw = unpack_weight_codes(we).to(dev)
    if cw.dim() == 2:
        cw = cw[:, :, None, None]
    geo = dict(groups=w.groups, dilation=tuple(w.dilation)) if isinstance(w, NoisyConv2d) else {}
    ops_ = ops.int_layer_operands(cw, we["scale"], we["zero_point"], act_e["scale"], act_e["zero_point"],
                                  we["bias"], a_top=max(1, act_e["n_levels"] - 1), w_top=(1 << we["bits"]) - 1,
                                  **geo)
    if isinstance(w, NoisyConv2d):
        return IntegerConv2d(act_e, ops_, w.stride, w.padding)
    return IntegerLinear(act_e, ops_)


def _tree_copy(m: nn.Module) -> nn.Module:
    """A copy of the module tree that shares its parameters and buffers: replacing a submodule,
    registering a hook or switching to eval mode in the copy leaves `m` as it was.  (``copy.deepcopy`` cannot copy the
    quantizers: they hold non-leaf tensors.)"""
    c = copy.copy(m)
    for k, v in m.__dict__.items():        # parameters, buffers, every hook registry
        if isinstance(v, (dict, set)):
            c.__dict__[k] = copy.copy(v)
    c._modules = {k: None if v is None else _tree_copy(v) for k, v in m._modules.items()}
    return c


@torch.no_grad()
def build_integer_model(model, blob, *, allow_groups_and_dilation=False) -> nn.Module:
    """An eval-mode copy of ``model`` whose quantized layers run on the integer codes of ``blob``
    (from ``export_quantized``); the other layers share their parameters with ``model``.  ``model`` must have the exporter's architecture; every mismatch
    and every layer the integer kernels cannot run raises ValueError naming the layer.

    Grouped and dilated convolutions are refused unless ``allow_groups_and_dilation=True``; with it
    they become integer layers too (``ops.int_conv2d``: depthwise layers on the CUDA cores, the
    other grouped and dilated layers on the tensor cores)."""
    if blob.get("format") != FORMAT or blob.get("version") != VERSION:
        raise ValueError(f"build_integer_model: not a {FORMAT} v{VERSION} export")
    mods = {n: m for n, m in model.named_modules() if _layer_kind(m) is not None}
    layers = blob["layers"]
    if set(mods) != set(layers):
        raise ValueError("build_integer_model: the model's quantized layers differ from the export's: "
                         f"{sorted(set(mods) ^ set(layers))}")
    for n, e in layers.items():
        if _layer_kind(mods[n]) != e["kind"]:
            raise ValueError(f"build_integer_model: {n} is a {_layer_kind(mods[n])} layer, the export has {e['kind']}")
    pairs = []
    for n, m in model.named_modules():
        if isinstance(m, nn.Sequential) and hasattr(m, "activations_quantizer") and hasattr(m, "0") \
                and isinstance(getattr(m, "0"), (NoisyConv2d, NoisyLinear)):
            pre = f"{n}." if n else ""
            pairs.append((n, layers[pre + "activations_quantizer"], getattr(m, "0"), layers[pre + "0"]))
    built = {n: _integer_layer(n, ae, w, we, allow_groups_and_dilation) for n, ae, w, we in pairs}     # validates all before copying
    out = _tree_copy(model).eval()
    for n, layer in built.items():
        parent, _, leaf = n.rpartition(".")
        setattr(out.get_submodule(parent) if parent else out, leaf, layer)
    return out


# ---------------------------------------------------------------------------------------------
# fused epilogues (DESIGN §3 "Fused epilogue", §5)
# ---------------------------------------------------------------------------------------------
class FusedIntegerConv2d(nn.Module):
    """An ``IntegerConv2d`` with the chain ``[BatchNorm2d] -> [+ residual] -> [ReLU | LeakyReLU]``
    that followed it in its epilogue (``ops.int_conv2d_fused``), one launch.  Its input is fp32
    (quantized with its own ``act_codes``) or, with ``codes_in``, the codes the previous fused layer
    already made.  ``forward(x[, residual])`` returns ``(y, codes)``: y the fp32 result or None,
    codes the next integer convolution's input codes or None.  The pattern tables are built on
    first use of each input size, so a warmed-up model can be captured in a CUDA graph."""

    def __init__(self, conv: IntegerConv2d, operands, codes_in: bool, residual: bool, activation,
                 negative_slope, out_fp32: bool, next_conv: Optional[IntegerConv2d]):
        super().__init__()
        self.act_scale, self.act_zero_point, self.act_max_val = conv.act_scale, conv.act_zero_point, conv.act_max_val
        self.operands = operands
        self.stride, self.padding = conv.stride, conv.padding
        self.codes_in, self.residual = codes_in, residual
        self.activation, self.negative_slope = activation, negative_slope
        self.out_fp32 = out_fp32
        self.code_params = None if next_conv is None else (
            next_conv.act_scale, next_conv.act_zero_point, next_conv.act_max_val)

    def forward(self, x, residual=None):
        codes = x if self.codes_in else ops.act_codes(x, self.act_scale, self.act_zero_point, self.act_max_val)[0]
        if residual is not None:
            residual = _as_add_operand(residual, codes, self.operands, self.stride, self.padding)
        return ops.int_conv2d_fused(codes, self.operands, self.stride, self.padding, residual=residual,
                                    activation=self.activation, negative_slope=self.negative_slope,
                                    out_fp32=self.out_fp32, code_params=self.code_params)


def _as_add_operand(r, codes, L, stride, padding):
    """The fused add's operand for ``y + r`` as torch computes it: ``r`` broadcast to the output's
    shape and converted to fp32 when torch's type promotion with fp32 keeps fp32 (the conversion
    is exact for every such dtype, and torch converts the same way before it adds).  Anything
    else is left to ``int_conv2d_fused`` to refuse."""
    b, h, w, _ = codes.shape
    out = (b, L.n_out, *L.out_size(h, w, stride, padding))
    if (not isinstance(r, torch.Tensor) or torch.promote_types(r.dtype, torch.float32) != torch.float32
            or (r.dtype == torch.float32 and tuple(r.shape) == out)):
        return r
    try:
        if torch.broadcast_shapes(tuple(r.shape), out) != out:
            return r
    except RuntimeError:
        return r
    return r.to(torch.float32).expand(out)


class _Tracer(fx.Tracer):
    """Integer layers and the library's quantizer modules are leaves (their forwards call the C ABI)."""

    def is_leaf_module(self, m, qualname):
        if isinstance(m, (_IntegerLayer, FusedIntegerConv2d)) or type(m).__module__.startswith(
                "mhaq_b200.quantization."):
            return True
        return super().is_leaf_module(m, qualname)


_ADDS = (operator.add, operator.iadd, torch.add)
_RELUS = (F.relu, torch.relu, torch.relu_, F.relu_)


def _module(gm_mods, n, cls):
    return n.op == "call_module" and isinstance(gm_mods.get(n.target), cls)


def _only_user(n):
    return next(iter(n.users)) if len(n.users) == 1 else None


def _match_bn(mods, n, cur, n_out):
    if not (_module(mods, n, nn.BatchNorm2d) and n.args == (cur,) and not n.kwargs):
        return None
    bn = mods[n.target]
    return bn if ops.batchnorm_foldable(bn) and bn.num_features == n_out else None


def _match_add(n, cur):
    """The other operand of ``cur + other`` (no alpha), or None.  For ``+=`` the chain's value must
    be the left operand: ``other += cur`` updates ``other`` in place, which the fused layer would
    not do."""
    if n.op != "call_function" or n.target not in _ADDS or n.kwargs or len(n.args) != 2:
        return None
    a, b = n.args
    other = b if a is cur else (a if b is cur and n.target is not operator.iadd else None)
    if not isinstance(other, fx.Node) or other is cur or other.op == "get_attr":
        return None
    return other


def _match_act(mods, n, cur):
    """("relu" | "leaky_relu", slope) of an activation applied to ``cur`` alone, or None."""
    if _module(mods, n, nn.ReLU) and n.args == (cur,):
        return "relu", None
    if _module(mods, n, nn.LeakyReLU) and n.args == (cur,):
        return "leaky_relu", float(mods[n.target].negative_slope)
    if not n.args or n.args[0] is not cur:
        return None
    kw = {k: v for k, v in n.kwargs.items() if k != "inplace"}
    if n.op == "call_function" and n.target in _RELUS and len(n.args) == 1 and not kw:
        return "relu", None
    if n.op == "call_method" and n.target in ("relu", "relu_") and len(n.args) == 1 and not kw:
        return "relu", None
    if n.op == "call_function" and n.target is F.leaky_relu and len(n.args) <= 3 and set(kw) <= {"negative_slope"}:
        slope = n.args[1] if len(n.args) > 1 else kw.get("negative_slope", 0.01)
        if isinstance(slope, (int, float)):
            return "leaky_relu", float(slope)
    return None


@torch.no_grad()
def fuse_integer_model(int_model: nn.Module) -> fx.GraphModule:
    """A ``torch.fx.GraphModule`` with ``int_model``'s forward signature (``int_model`` from
    ``build_integer_model``) in which every chain

        IntegerConv2d -> [BatchNorm2d (eval, running stats)] -> [+ residual] -> [ReLU | LeakyReLU]

    whose intermediate nodes have one user each runs as one ``FusedIntegerConv2d`` launch (the
    BatchNorm folded into the operands, ``ops.fold_batchnorm``).  Among the chain's users, the
    first ``IntegerConv2d`` in graph order that takes the chain's value as its only input (other
    users may come before it) becomes its consumer: the fused layer writes that consumer's codes
    and the consumer reads them instead of running ``act_codes``; fp32 is written as well only for
    the chain's other users.  An ``IntegerConv2d`` called at more than one site is left unfused.
    Unmatched nodes and modules stay as they are, the fused layers share their weight operands with
    ``int_model`` and ``int_model`` itself is not modified.  A model torch.fx cannot trace raises
    ValueError."""
    tracer = _Tracer()
    try:
        graph = tracer.trace(int_model)
    except Exception as exc:
        raise ValueError(f"fuse_integer_model: torch.fx cannot trace the model: {exc}") from exc
    gm = fx.GraphModule(tracer.root, graph, type(int_model).__name__ + "Fused")
    mods = dict(gm.named_modules())
    pos = {n: i for i, n in enumerate(gm.graph.nodes)}
    # a layer called at more than one site (shared weights) stays unfused: its module is replaced
    # by target, so one site's chain would change what the other site runs
    sites = collections.Counter(n.target for n in gm.graph.nodes if n.op == "call_module")

    def int_conv(node):
        return _module(mods, node, IntegerConv2d) and sites[node.target] == 1

    takes_codes = set()                  # consumer nodes whose input is now a producer's codes
    for n in list(gm.graph.nodes):
        if not int_conv(n):
            continue
        conv = mods[n.target]
        chain, cur, bn, res, act = [n], n, None, None, (None, None)
        nxt = _only_user(cur)
        if nxt is not None and (bn := _match_bn(mods, nxt, cur, conv.operands.n_out)) is not None:
            chain.append(nxt)
            cur, nxt = nxt, _only_user(nxt)
        if nxt is not None and (res := _match_add(nxt, cur)) is not None:
            chain.append(nxt)
            cur, nxt = nxt, _only_user(nxt)
        if nxt is not None and (m := _match_act(mods, nxt, cur)) is not None:
            act = m
            chain.append(nxt)
            cur = nxt
        users = sorted(cur.users, key=pos.__getitem__)
        consumer = next((u for u in users if int_conv(u) and u.args == (cur,) and not u.kwargs
                         and mods[u.target].operands.cin == conv.operands.n_out), None)
        codes_in = n in takes_codes
        if len(chain) == 1 and consumer is None and not codes_in:
            continue
        out_fp32 = consumer is None or len(users) > 1
        operands = (ops.fold_batchnorm(conv.operands, bn) if bn is not None
                    else dataclasses.replace(conv.operands, tables={}))
        fused = FusedIntegerConv2d(conv, operands, codes_in, res is not None, act[0], act[1], out_fp32,
                                   None if consumer is None else mods[consumer.target])
        gm.add_submodule(n.target, fused)
        with gm.graph.inserting_before(cur):
            fn = gm.graph.call_module(n.target, (n.args[0],) if res is None else (n.args[0], res))
            fn.meta["fused_chain"] = tuple(c.name for c in chain)     # the traced nodes it replaces
            y = gm.graph.call_function(operator.getitem, (fn, 0)) if out_fp32 else None
            codes = gm.graph.call_function(operator.getitem, (fn, 1)) if consumer is not None else None
        if consumer is not None:
            consumer.args = (codes,)
            takes_codes.add(consumer)
        if y is not None:
            cur.replace_all_uses_with(y)
        for c in reversed(chain):
            gm.graph.erase_node(c)
    gm.graph.lint()
    gm.delete_all_unused_submodules()
    gm.recompile()
    return gm
