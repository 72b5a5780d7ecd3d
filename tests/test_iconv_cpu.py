"""CPU: the integer layers' host side (mhaq_b200.ops integer-layer helpers, quantization/gdnsq/
inference.py) and the argument checks of their C ABI, without a GPU.

- The expansion y = alpha*S + beta*SA + ctab[p] (DESIGN §3, "Integer layers"), with the library's
  pattern classes and constant table, equals fp64 F.conv2d on the dequantized values.
- The weight operand equals a numpy restatement built from tests/pack_ref.py's unpacker.
- build_integer_model refuses what the integer kernels cannot run, naming the layer."""
import ctypes
from collections import OrderedDict

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from mhaq_b200 import ops
from mhaq_b200.aux.types import QScheme
from mhaq_b200.quantization.gdnsq.export import build_integer_model
from mhaq_b200.quantization.gdnsq.inference import IntegerConv2d, IntegerLinear, unpack_weight_codes
from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
from mhaq_b200.quantization.gdnsq.layers.gdnsq_linear import NoisyLinear
from tests import pack_ref as R


# ---------------------------------------------------------------------------------------------
# the expansion of DESIGN §3 against fp64 convolution
# ---------------------------------------------------------------------------------------------
CASES = [  # (C, N, (kh, kw), (sh, sw), (ph, pw), H, W)
    (3, 8, (3, 3), (1, 1), (1, 1), 9, 7),
    (5, 4, (3, 3), (2, 2), (1, 1), 10, 11),
    (16, 6, (1, 1), (1, 1), (0, 0), 5, 5),
    (4, 3, (7, 7), (2, 2), (3, 3), 12, 9),
    (12, 5, (3, 3), (2, 2), (0, 0), 9, 9),
    (2, 3, (7, 7), (1, 1), (3, 3), 5, 6),       # kernel wider than the image: every pixel is a border pixel
    (6, 4, (1, 1), (2, 2), (0, 0), 7, 8),
    (7, 2, (3, 3), (1, 1), (0, 0), 4, 4),
    # per-axis geometry
    (4, 5, (1, 3), (1, 2), (0, 1), 9, 12),
    (3, 4, (3, 1), (1, 1), (1, 0), 10, 7),
    (5, 3, (5, 3), (1, 3), (0, 0), 13, 14),
    (6, 4, (7, 3), (2, 1), (3, 0), 15, 9),
    (3, 5, (2, 4), (2, 1), (1, 2), 9, 10),
    (4, 3, (2, 3), (3, 4), (1, 0), 12, 13),     # stride larger than the kernel
    (3, 4, (3, 3), (1, 1), (3, 3), 2, 2),       # pad >= k: outputs with no valid tap
    (5, 2, (3, 3), (1, 1), (4, 1), 1, 1),
    (4, 3, (1, 1), (3, 2), (0, 0), 11, 10),
]

@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("zpa_nonzero", [False, True])
@pytest.mark.parametrize("per_channel", [False, True])
@pytest.mark.parametrize("with_bias", [False, True])
def test_expansion_equals_fp64_conv(case, zpa_nonzero, per_channel, with_bias):
    c, n, (kh, kw), stride, pad, h, w = case
    g = torch.Generator().manual_seed(hash((case, zpa_nonzero, per_channel, with_bias)) & 0xFFFF)
    a_top, w_top = 15, 7
    ca = torch.randint(0, a_top + 1, (2, c, h, w), generator=g)
    cw = torch.randint(0, w_top + 1, (n, c, kh, kw), generator=g)
    sa = 2.0 ** -5
    zpa = -1.375 if zpa_nonzero else 0.0
    rows = n if per_channel else 1
    sw = torch.exp2(torch.randint(-9, -5, (rows,), generator=g).float())
    zpw = -torch.rand(rows, generator=g) * 0.1
    bias = torch.randn(n, generator=g) if with_bias else None
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, bias, a_top, w_top)

    a = ca.double() * sa + zpa
    wt = cw.double() * sw.double().reshape(-1, 1, 1, 1) + zpw.double().reshape(-1, 1, 1, 1)
    ref = F.conv2d(a, wt, None if bias is None else bias.double(), stride=stride, padding=pad)

    s = F.conv2d(ca.double(), cw.double(), stride=stride, padding=pad)
    sa_m = F.conv2d(ca.double(), torch.ones(1, c, kh, kw, dtype=torch.float64), stride=stride, padding=pad)
    hc, hv = ops.tap_classes(h, kh, stride[0], pad[0])
    wc, wv = ops.tap_classes(w, kw, stride[1], pad[1])
    ctab = L.constant_table(hv, wv)                               # fp64 [classes, N]
    # the cached tables of the layer are the same classes
    phc, pwc, nwc, pctab = L.pattern_tables(h, w, stride, pad)
    assert torch.equal(phc, hc) and torch.equal(pwc, wc) and nwc == wv.shape[0]
    assert torch.equal(pctab, ctab.float())
    p = hc.long()[:, None] * wv.shape[0] + wc.long()[None, :]     # [Ho, Wo]
    cterm = ctab[p].permute(2, 0, 1)[None]                        # [1, N, Ho, Wo]
    swn, zpwn = L.sw.reshape(1, -1, 1, 1), L.zpw.reshape(1, -1, 1, 1)
    y = sa * swn * s + sa * zpwn * sa_m + cterm
    scale = (sa * swn * s).abs() + (sa * zpwn * sa_m).abs() + cterm.abs()
    assert y.shape == ref.shape
    assert torch.all((y - ref).abs() <= 1e-12 * scale + 1e-300)
    # alpha / beta are the fp64 products rounded once to fp32
    assert torch.equal(L.alpha, (sa * L.sw).float()) and torch.equal(L.beta, (sa * L.zpw).float())


def test_tap_classes():
    cls, valid = ops.tap_classes(8, 3, 1, 1)
    assert cls.tolist() == [cls[0].item()] + [cls[1].item()] * 6 + [cls[7].item()]
    assert valid[cls[0]].tolist() == [False, True, True] and valid[cls[7]].tolist() == [True, True, False]
    cls, valid = ops.tap_classes(1, 1, 1, 0)                      # a linear layer: one pattern
    assert cls.tolist() == [0] and valid.tolist() == [[True]]


@pytest.mark.parametrize("size,k,stride,pad", [
    (2, 3, 1, 3), (1, 3, 1, 4), (5, 1, 1, 1), (1, 1, 1, 2), (4, 2, 3, 2),          # pad >= k
    (12, 2, 3, 1), (11, 1, 3, 0), (13, 3, 4, 0), (9, 1, 2, 0),                     # stride > k
])
def test_tap_classes_against_direct_enumeration(size, k, stride, pad):
    """Each output position's class holds exactly its taps inside [0, size); with pad >= k some
    position has no valid tap at all, with stride > k some input positions are never read."""
    cls, valid = ops.tap_classes(size, k, stride, pad)
    out = (size + 2 * pad - k) // stride + 1
    assert cls.shape == (out,) and valid.shape[1] == k
    assert len({tuple(v) for v in valid.tolist()}) == valid.shape[0]              # classes are distinct
    for o in range(out):
        want = [0 <= o * stride - pad + t < size for t in range(k)]
        assert valid[cls[o]].tolist() == want, (o, want)
    empty = [o for o in range(out) if not valid[cls[o]].any()]
    if pad >= k:
        assert empty == [o for o in range(out) if o * stride - pad + k <= 0 or o * stride - pad >= size] != []
    else:
        assert not empty
    if stride > k:
        read = {o * stride - pad + t for o in range(out) for t in range(k)}
        assert set(range(size)) - read


# ---------------------------------------------------------------------------------------------
# the weight operand
# ---------------------------------------------------------------------------------------------
def _numpy_operand(cw: np.ndarray) -> np.ndarray:
    n, c, kh, kw = cw.shape
    cp = (c + 15) // 16 * 16
    k = kh * kw * cp
    nbytes, nt, tn, to, ks = ops.iconv_layout(n, k)
    rows = np.zeros((n, kh, kw, cp), np.uint8)
    rows[..., :c] = cw.transpose(0, 2, 3, 1)
    rows = rows.reshape(n, k)
    out = np.zeros(nbytes, np.uint8)
    for t in range(nt):
        for r in range(tn):
            ch = t * to + r
            for kk in range(ks * 128):
                if r < to and ch < n and kk < k:
                    v = rows[ch, kk]
                else:
                    v = 1 if r == to else 0
                st, q = divmod(kk, 128)
                c16, j = divmod(q, 16)
                out[((t * ks + st) * tn * 128) + (r // 8) * 1024 + c16 * 128 + (r % 8) * 16 + j] = v
    return out


@pytest.mark.parametrize("shape,bits,per_channel", [
    ((10, 3, 3, 3), 4, True),
    ((16, 16, 1, 1), 2, False),
    ((40, 12, 3, 3), 8, True),
    ((300, 5, 1, 1), 1, True),          # two N tiles
    ((7, 33, 1, 1), 4, False),
])
def test_weight_operand_matches_numpy_restatement(shape, bits, per_channel):
    rng = np.random.default_rng(sum(shape) * 7 + bits)
    cw = rng.integers(0, 1 << bits, size=shape, dtype=np.int64)
    rows = shape[0] if per_channel else 1
    packed = R.pack(cw.reshape(rows, -1), bits)
    e = {"bits": bits, "codes": torch.from_numpy(packed), "shape": list(shape)}
    got = unpack_weight_codes(e)
    assert np.array_equal(got.numpy(), R.unpack(packed, bits, cw.size // rows).reshape(shape))
    assert np.array_equal(ops.iconv_weight_operand(got).numpy(), _numpy_operand(cw.astype(np.uint8)))


# ---------------------------------------------------------------------------------------------
# build_integer_model refusals
# ---------------------------------------------------------------------------------------------
def _pair(layer):
    return nn.Sequential(OrderedDict([("activations_quantizer", NoisyAct(signed=True)), ("0", layer)]))


class _Net(nn.Module):
    def __init__(self, conv=None):
        super().__init__()
        self.c = _pair(conv if conv is not None else
                       NoisyConv2d(3, 8, 3, padding=1, bias=False, qscheme=QScheme.PER_CHANNEL))
        self.fc = _pair(NoisyLinear(8, 4, qscheme=QScheme.PER_TENSOR))


def _blob(net, a_levels=16, w_bits=4):
    layers = {}
    g = torch.Generator().manual_seed(0)
    for name, m in net.named_modules():
        if isinstance(m, NoisyAct):
            layers[name] = {"kind": "act", "disabled": False, "scale": torch.tensor([2.0 ** -4]),
                            "zero_point": torch.tensor([-0.5]), "max_val": torch.tensor([-0.5 + (a_levels - 1) / 16]),
                            "n_levels": a_levels, "bits": 8}
        elif isinstance(m, (NoisyConv2d, NoisyLinear)):
            rows = m.weight.shape[0] if isinstance(m, NoisyConv2d) and m.qscheme == QScheme.PER_CHANNEL else 1
            cw = torch.randint(0, 1 << min(w_bits, 8), (rows, m.weight.numel() // rows), generator=g)
            layers[name] = {"kind": "conv2d" if isinstance(m, NoisyConv2d) else "linear",
                            "shape": list(m.weight.shape), "bits": w_bits,
                            "qscheme": "PER_CHANNEL" if rows > 1 else "PER_TENSOR",
                            "codes": torch.from_numpy(R.pack(cw.numpy(), w_bits)),
                            "scale": torch.full((rows,), 2.0 ** -6), "zero_point": torch.full((rows,), -0.1),
                            "bias": None if m.bias is None else torch.zeros(m.weight.shape[0])}
    return {"format": "mhaq-packed", "version": 1, "layers": layers}


def test_builds_integer_layers_on_cpu_operands():
    net = _Net()
    q = build_integer_model(net, _blob(net))
    assert isinstance(q.c, IntegerConv2d) and isinstance(q.fc, IntegerLinear)
    assert not q.training and isinstance(net.c, nn.Sequential)     # the original is untouched
    assert q.c.stride == (1, 1) and q.c.padding == (1, 1)
    # hooks registered on the copy stay on the copy (and the other way round)
    q.register_forward_hook(lambda *a: None)
    net.fc.register_forward_pre_hook(lambda *a: None)
    assert not net._forward_hooks and len(q._forward_hooks) == 1
    assert len(net.fc._forward_pre_hooks) == 1 and not q.fc._forward_pre_hooks


def test_weight_tiles_fit_the_mma():
    """Every width gets tiles of at most 256 rows (real channels + the ones row, rounded to 16),
    none of them empty, that together cover every output channel."""
    for n_out in list(range(1, 4097)) + [65535, 65536, 70000, 100003]:
        nbytes, nt, tn, to, ks = ops.iconv_layout(n_out, 144)
        assert tn % 16 == 0 and to + 1 <= tn <= 256, n_out
        assert (nt - 1) * to < n_out <= nt * to, n_out
        assert nbytes == nt * ks * tn * 128, n_out


@pytest.mark.parametrize("what", ["disabled", "levels", "bits16", "groups", "dilation", "padding_mode",
                                  "int32", "shape", "kinds"])
def test_refusals(what):
    conv = None
    if what == "groups":
        conv = NoisyConv2d(4, 8, 3, padding=1, groups=2, qscheme=QScheme.PER_CHANNEL)
    elif what == "dilation":
        conv = NoisyConv2d(3, 8, 3, padding=2, dilation=2, qscheme=QScheme.PER_CHANNEL)
    elif what == "padding_mode":
        conv = NoisyConv2d(3, 8, 3, padding=1, padding_mode="reflect", qscheme=QScheme.PER_CHANNEL)
    elif what == "int32":
        conv = NoisyConv2d(4096, 2, 3, padding=1, qscheme=QScheme.PER_CHANNEL)
    net = _Net(conv)
    blob = _blob(net, a_levels=256 if what == "int32" else 16, w_bits=16 if what == "bits16" else
                 (8 if what == "int32" else 4))
    lay = blob["layers"]
    match = "c"
    if what == "disabled":
        lay["fc.activations_quantizer"] = {"kind": "act", "disabled": True}
        match = "fc: the activation quantizer is disabled"
    elif what == "levels":
        lay["c.activations_quantizer"]["n_levels"] = 257
        match = "c: 257 activation levels"
    elif what == "bits16":
        match = "c: 16-bit weight codes"
    elif what in ("groups", "dilation"):
        match = "c: grouped or dilated"
    elif what == "padding_mode":
        match = "c: only explicit zero padding"
    elif what == "int32":
        match = "c: K .* overflow"
    elif what == "shape":
        lay["fc.0"]["shape"] = [4, 9]
        match = "fc: the model's layer differs"
    elif what == "kinds":
        lay["fc.0"]["kind"] = "conv2d"
        match = "fc.0 is a linear layer"
    with pytest.raises(ValueError, match=match):
        build_integer_model(net, blob)


def test_refuses_a_foreign_export():
    net = _Net()
    blob = _blob(net)
    del blob["layers"]["fc.0"]
    with pytest.raises(ValueError, match="differ from the export"):
        build_integer_model(net, blob)
    with pytest.raises(ValueError, match="not a mhaq-packed"):
        build_integer_model(net, {"format": "other"})


# ---------------------------------------------------------------------------------------------
# C ABI argument errors (no kernel is launched)
# ---------------------------------------------------------------------------------------------
def test_abi_argument_errors_without_gpu():
    from mhaq_b200 import _lib
    L = _lib.lib
    d = ctypes.c_void_p(16)          # 16-byte aligned dummy pointer, never dereferenced
    # act codes: null pointers, Cp % 16, Cp < C, misaligned codes
    assert L.mhaq_fq_act_codes_f32(None, d, d, d, d, 4, 3, 16, None, None) == -2
    assert L.mhaq_fq_act_codes_f32(d, d, d, d, None, 4, 3, 16, None, None) == -2
    assert L.mhaq_fq_act_codes_f32(d, d, d, d, d, 4, 3, 8, None, None) == -1
    assert L.mhaq_fq_act_codes_f32(d, d, d, d, d, 4, 20, 16, None, None) == -1
    assert L.mhaq_fq_act_codes_f32(d, ctypes.c_void_p(17), d, d, d, 4, 3, 16, None, None) == -1
    assert L.mhaq_fq_act_codes_f32(d, d, d, d, d, 0, 3, 16, None, None) == 0     # nothing to do

    def iconv(**kw):
        a = dict(codes=d, weights=d, alpha=d, beta=d, ctab=d, hc=d, wc=d, nwc=1, y=d, b=2, h=8, w=8, cp=16,
                 n=10, kh=3, kw=3, sh=1, sw=1, ph=1, pw=1, at=15, wt=15)
        a.update(kw)
        return L.mhaq_fq_iconv_u8(a["codes"], a["weights"], a["alpha"], a["beta"], a["ctab"], a["hc"], a["wc"],
                                  a["nwc"], a["y"], a["b"], a["h"], a["w"], a["cp"], a["n"], a["kh"], a["kw"],
                                  a["sh"], a["sw"], a["ph"], a["pw"], a["at"], a["wt"], None)
    assert iconv(weights=None) == -2
    assert iconv(ctab=None) == -2
    assert iconv(cp=24) == -1                      # Cp % 16 != 0
    assert iconv(b=0) == -1
    assert iconv(n=0) == -1
    assert iconv(sh=0) == -1
    assert iconv(ph=-1) == -1
    assert iconv(h=1, ph=0) == -1                  # kernel larger than the padded image
    assert iconv(at=0) == -1 and iconv(wt=256) == -1
    assert iconv(codes=ctypes.c_void_p(24)) == -1  # not 16-byte aligned
    # int32 bound: K * 255 * 255 >= 2^31 at K = 3*3*4096, and the first refused K of each kernel size
    # (K = 33024 and 3 * 3 * 3664 are accepted: tests/test_gpu_iconv_limits.py runs them)
    assert iconv(cp=4096, at=255, wt=255) == -1
    assert iconv(kh=1, kw=1, ph=0, pw=0, cp=33040, at=255, wt=255) == -1
    assert iconv(cp=3680, at=255, wt=255) == -1
    # layout helper
    assert L.mhaq_fq_iconv_weight_bytes(0, 16, None, None, None, None) == -1
    assert L.mhaq_fq_iconv_weight_bytes(10, 24, None, None, None, None) == -1
    assert L.mhaq_fq_iconv_weight_bytes(10, 144, None, None, None, None) == 2 * 16 * 128
    assert ops.iconv_layout(512, 4608) == (3 * 36 * 176 * 128, 3, 176, 171, 36)
    assert ops.iconv_layout(255, 16)[1:4] == (1, 256, 255)
