"""Run an exported model on its integer codes.

``build_integer_model(model, blob)`` returns an eval-mode copy of ``model`` (sharing the parameters
of the layers it keeps) in which every quantized
``Sequential(activations_quantizer=NoisyAct, "0"=NoisyConv2d | NoisyLinear)`` of ``blob`` (from
``export_quantized``) is an ``IntegerConv2d`` / ``IntegerLinear``: the layer quantizes its fp32 input
to uint8 activation codes and runs an int8 tensor-core GEMM against the exported weight codes
(include/mhaq_fq.h "Integer layers", DESIGN §3).  Everything between those layers (BN, ReLU,
pooling, residual adds, unquantized layers) stays as it is.

The convolution geometry (stride, padding) comes from the model's modules; every number comes
from the blob: the weight codes are unpacked from the packed format with integer operations, never
re-derived from dequantized floats.
"""
import copy

import torch
from torch import nn

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


def _check_pair(name, act_e, w, we):
    """ValueError naming the layer for everything the integer kernels cannot run exactly."""
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
    if isinstance(w, NoisyConv2d):
        if w.groups != 1 or tuple(w.dilation) != (1, 1):
            raise ValueError(f"build_integer_model: {name}: grouped or dilated convolutions are not supported")
        if w.padding_mode != "zeros" or isinstance(w.padding, str):
            raise ValueError(f"build_integer_model: {name}: only explicit zero padding is supported "
                             f"(padding_mode={w.padding_mode!r}, padding={w.padding!r})")
    kk = w.weight[0, 0].numel() if w.weight.dim() == 4 else 1
    k_bytes = kk * ops.code_channels(w.weight.shape[1])
    if not ops.int32_bound_ok(k_bytes, max(1, act_e["n_levels"] - 1), (1 << we["bits"]) - 1):
        raise ValueError(f"build_integer_model: {name}: K * (n_levels - 1) * (2^bits - 1) >= 2^31 would "
                         "overflow the int32 accumulator")


def _integer_layer(name, act_e, w, we):
    _check_pair(name, act_e, w, we)
    dev = w.weight.device
    cw = unpack_weight_codes(we).to(dev)
    if cw.dim() == 2:
        cw = cw[:, :, None, None]
    ops_ = ops.int_layer_operands(cw, we["scale"], we["zero_point"], act_e["scale"], act_e["zero_point"],
                                  we["bias"], a_top=max(1, act_e["n_levels"] - 1), w_top=(1 << we["bits"]) - 1)
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
def build_integer_model(model, blob) -> nn.Module:
    """An eval-mode copy of ``model`` whose quantized layers run on the integer codes of ``blob``
    (from ``export_quantized``); the other layers share their parameters with ``model``.  ``model`` must have the exporter's architecture; every mismatch
    and every layer the integer kernels cannot run raises ValueError naming the layer."""
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
    built = {n: _integer_layer(n, ae, w, we) for n, ae, w, we in pairs}     # validates all before copying
    out = _tree_copy(model).eval()
    for n, layer in built.items():
        parent, _, leaf = n.rpartition(".")
        setattr(out.get_submodule(parent) if parent else out, leaf, layer)
    return out
