"""Export a QAT-trained model as packed low-bit integer codes, and load such an export back.

``export_quantized(model)`` walks the model's quantizers and returns a nested dict of CPU tensors
and plain values (``torch.save`` / ``torch.load(weights_only=True)`` both handle it):

    {"format": "mhaq-packed", "version": 1, "layers": {module name: entry}}

A ``NoisyConv2d`` / ``NoisyLinear`` entry holds the weight's codes in the packed format of
include/mhaq_fq.h (rows in row-major logical order, whatever the parameter's memory format) at
the smallest width that holds them, with the scale and zero point that turn them back into the
layer's fake-quantized weight, the true width per row and the bias the layer's forward uses.  A
``NoisyAct`` entry holds the quantizer's scale, zero point, upper bound and number of levels.

``load_quantized(model, blob)`` writes the dequantized weights into a model whose quantizer
parameters are the exporter's (load the ordinary state dict first) and checks that the layers
quantize them back to exactly what was written.
"""
import torch

from ... import ops
from ...aux.types import is_per_channel
from .layers.gdnsq_act import NoisyAct
from .layers.gdnsq_conv2d import NoisyConv2d
from .layers.gdnsq_linear import NoisyLinear
from .utils.model_stats import _code_span_bits

FORMAT, VERSION = "mhaq-packed", 1
_WEIGHT_LAYERS = {NoisyConv2d: "conv2d", NoisyLinear: "linear"}


def _layer_kind(m):
    if isinstance(m, NoisyAct):
        return "act"
    for cls, kind in _WEIGHT_LAYERS.items():
        if isinstance(m, cls):
            return kind
    return None


def _smallest_bits(top: int):
    for b in ops.PACK_BITS:
        if top <= (1 << b) - 1:
            return b
    return None


def _weight_operands(m):
    """(scale, zero point) per row of the logical [O, rest] weight view, as the layer forms them."""
    w = m.weight.detach()
    if is_per_channel(m.qscheme):
        return torch.exp2(m.log_wght_s.detach()).reshape(-1), w.reshape(w.shape[0], -1).amin(1)
    return torch.exp2(m.log_wght_s.detach()).reshape(1), w.amin().reshape(1)


def _layer_bias(m):
    if m.bias is None:
        return None
    if isinstance(m, NoisyConv2d) and m.quant_bias:
        return m.quantized_weight()[1]
    return m.bias


def _export_weight(m, kind):
    if not m.Q.positive_scale:
        raise ValueError("export_quantized: a weight quantizer without a positive scale has no integer codes")
    w = m.weight.detach().contiguous()          # row-major logical order, whatever the training layout
    scale, zp = _weight_operands(m)
    if is_per_channel(m.qscheme):
        # the layers' fused weight path: s = 2^log_wght_s in the kernel, zero point = row minimum
        p = ops.pack_weight_codes(w, m.log_wght_s.detach().reshape(-1), zp)
    else:
        p = ops.pack_codes(w, scale, zp)
    bias = _layer_bias(m)
    return {
        "kind": kind,
        "shape": list(w.shape),
        "qscheme": "PER_CHANNEL" if is_per_channel(m.qscheme) else "PER_TENSOR",
        "bits": p.bits,
        "codes": p.data.cpu(),
        "scale": scale.cpu(),
        "zero_point": zp.cpu(),
        "true_bits": _code_span_bits(m).float().reshape(-1).cpu(),
        "quant_bias": bool(getattr(m, "quant_bias", False)),
        "bias": None if bias is None else bias.detach().cpu().clone(),
    }


def _act_operands(m):
    """(scale, zero point = min_val, max_val) in the reference's op order (gdnsq_act.py:42-48)."""
    s = torch.exp2(m.log_act_s.detach())
    q = torch.exp2(m.log_act_q.detach())
    b = m.act_b.detach()
    return s, b, b + q - s


def _export_act(m):
    if m.disable:
        return {"kind": "act", "disabled": True}
    s, b, hi = _act_operands(m)
    top = int(torch.round((hi - b) / s).item())      # the code of max_val: the highest level
    return {"kind": "act", "disabled": False, "scale": s.cpu(), "zero_point": b.cpu().clone(),
            "max_val": hi.cpu(), "n_levels": top + 1, "bits": _smallest_bits(top)}


@torch.no_grad()
def export_quantized(model) -> dict:
    """Packed integer weights and quantizer constants of every quantized layer of `model`."""
    layers = {}
    for name, m in model.named_modules():
        kind = _layer_kind(m)
        if kind == "act":
            layers[name] = _export_act(m)
        elif kind is not None:
            layers[name] = _export_weight(m, kind)
    return {"format": FORMAT, "version": VERSION, "layers": layers}


def _same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    a, b = a.detach().float().cpu().reshape(-1), b.detach().float().cpu().reshape(-1)
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def _load_weight(name, m, e):
    scale, _ = _weight_operands(m)
    if e["qscheme"] != ("PER_CHANNEL" if is_per_channel(m.qscheme) else "PER_TENSOR") or \
            list(m.weight.shape) != list(e["shape"]) or not _same_bits(scale, e["scale"]):
        raise ValueError(f"load_quantized: {name}: the model's weight quantizer differs from the exporter's "
                         "(load the exporter's state dict first)")
    dev = m.weight.device
    shape = tuple(e["shape"])
    n_rows = shape[0] if e["qscheme"] == "PER_CHANNEL" else 1
    n_inner = m.weight.numel() // n_rows
    p = ops.PackedCodes(data=e["codes"].to(dev), bits=e["bits"], shape=shape,
                        stride=torch.empty(shape, device="meta").stride(), n_rows=n_rows, n_inner=n_inner,
                        n_ch=n_rows, scale=e["scale"].to(dev).contiguous(),
                        zero_point=e["zero_point"].to(dev).contiguous(),
                        n_out_of_range=torch.zeros(1, dtype=torch.int64, device=dev))
    w = ops.unpack_codes(p)
    m.weight.copy_(w)                         # in place: same Parameter, same memory format
    if e["bias"] is not None:
        m.bias.copy_(e["bias"].to(dev))
    out = m.quantized_weight()
    wq, bq = (out[0], out[1]) if isinstance(out, tuple) else (out, m.bias)
    if not _same_bits(wq, m.weight) or (e["bias"] is not None and not _same_bits(bq, e["bias"])):
        raise ValueError(f"load_quantized: {name}: re-quantizing the unpacked weight does not reproduce it "
                         "(|zero point| / scale too large for fp32)")


def _load_act(name, m, e):
    if bool(m.disable) != bool(e["disabled"]):
        raise ValueError(f"load_quantized: {name}: the activation quantizer is "
                         f"{'disabled' if m.disable else 'enabled'} here but not in the export")
    if m.disable:
        return
    s, b, hi = _act_operands(m)
    if not (_same_bits(s, e["scale"]) and _same_bits(b, e["zero_point"]) and _same_bits(hi, e["max_val"])):
        raise ValueError(f"load_quantized: {name}: the model's activation quantizer differs from the "
                         "exporter's (load the exporter's state dict first)")


@torch.no_grad()
def load_quantized(model, blob) -> None:
    """Overwrite every quantized weight (and quantized bias) of `model` with the dequantized codes
    of `blob` (from ``export_quantized``).  `model` must carry the exporter's quantizer parameters;
    every mismatch, and every layer that would not quantize the written weight back to itself,
    raises ValueError."""
    if blob.get("format") != FORMAT or blob.get("version") != VERSION:
        raise ValueError(f"load_quantized: not a {FORMAT} v{VERSION} export")
    mods = {n: m for n, m in model.named_modules() if _layer_kind(m) is not None}
    layers = blob["layers"]
    if set(mods) != set(layers):
        raise ValueError("load_quantized: the model's quantized layers differ from the export's: "
                         f"{sorted(set(mods) ^ set(layers))}")
    for name, e in layers.items():
        m = mods[name]
        if _layer_kind(m) != e["kind"]:
            raise ValueError(f"load_quantized: {name} is a {_layer_kind(m)} layer, the export has {e['kind']}")
        if e["kind"] == "act":
            _load_act(name, m, e)
        else:
            _load_weight(name, m, e)


from .inference import build_integer_model  # noqa: E402,F401  (runs an export on its integer codes)
from .inference import fuse_integer_model  # noqa: E402,F401  (fuses BN / add / activation / codes into it)
