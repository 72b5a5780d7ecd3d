"""CPU: the host side of grouped, depthwise and dilated integer layers, without a GPU.

- The block-diagonal tile plan of mhaq_fq_iconv_grouped_weight_bytes over a broad range of
  (groups, cin / groups, cout / groups), and the weight operands against a numpy restatement.
- The expansion y = alpha*S + beta*SA[g(n)] + ctab[p] (DESIGN §3, "Grouped and dilated layers")
  against fp64 grouped / dilated F.conv2d of the dequantized values.
- tap_classes with dilation against direct enumeration.
- build_integer_model's default refusal and its opt-in; the fused structure of the torchvision
  models with grouped, depthwise and dilated layers; the argument checks of the new C ABI."""
import collections
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from mhaq_b200 import _lib, harness, ops
from mhaq_b200.aux.types import QScheme
from mhaq_b200.quantization.gdnsq.export import build_integer_model, fuse_integer_model
from mhaq_b200.quantization.gdnsq.inference import FusedIntegerConv2d, IntegerConv2d
from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
from mhaq_b200.quantization.quantizer import Quantizer
from tests.test_iconv_cpu import _blob, _Net
from tests.test_ifuse_cpu import fused_structure


# ---------------------------------------------------------------------------------------------
# the tile plan
# ---------------------------------------------------------------------------------------------
def _tiles(n_in, n_out, kh, kw, groups):
    nbytes, nt, tn, to, gpt, parts, ks = ops.iconv_grouped_layout(n_in, n_out, kh, kw, groups)
    cin_g, cout_g = n_in // groups, n_out // groups
    return (nbytes, nt, tn, to, gpt, parts, ks,
            [ops.grouped_tile(t, groups, cin_g, cout_g, to, gpt, parts) for t in range(nt)])


@pytest.mark.parametrize("groups", [1, 2, 3, 5, 8, 32, 64, 129])
def test_tile_plan(groups):
    """At most 256 rows per tile, no empty tile, every output channel in exactly one tile and
    within its own group, a group split only when it is wider than a tile, and each tile's K
    window exactly its groups' channels rounded out to 16."""
    for cin_g in (1, 2, 3, 4, 8, 16, 17, 32, 48):
        for cout_g in (1, 2, 3, 4, 7, 8, 16, 33, 64, 85, 127, 128, 254, 255, 256, 300, 511, 600):
            n_in, n_out = groups * cin_g, groups * cout_g
            if groups == n_in == n_out:
                continue                                   # depthwise: no tiles
            for kh, kw in ((3, 3), (1, 5)):
                nbytes, nt, tn, to, gpt, parts, ks, tiles = _tiles(n_in, n_out, kh, kw, groups)
                key = (groups, cin_g, cout_g)
                assert tn % 16 == 0 and to + gpt <= tn <= 256, key
                assert (parts > 1) == (cout_g + 1 > 256) and (parts == 1 or gpt == 1), key
                assert nbytes == nt * ks * tn * 128, key
                owner = np.zeros(n_out, np.int64)
                kc_max = 0
                for n_base, n_here, g_lo, n_grp, c_lo, kc in tiles:
                    assert n_here > 0 and n_grp > 0 and n_here <= to, key
                    owner[n_base:n_base + n_here] += 1
                    # the tile's channels belong to its groups, and the groups are whole unless split
                    assert n_base // cout_g == g_lo and (n_base + n_here - 1) // cout_g == g_lo + n_grp - 1, key
                    if parts == 1:
                        assert n_base == g_lo * cout_g and n_here == n_grp * cout_g, key
                    assert c_lo * 16 <= g_lo * cin_g and (g_lo * cin_g) - c_lo * 16 < 16, key
                    assert (c_lo + kc) * 16 >= (g_lo + n_grp) * cin_g > (c_lo + kc - 1) * 16, key
                    kc_max = max(kc_max, kc)
                assert (owner == 1).all(), key
                assert ks == (kh * kw * kc_max + 7) // 8, key


def test_depthwise_layout():
    for c in (1, 17, 32, 960):
        for kh, kw in ((3, 3), (5, 7)):
            nbytes, nt, tn, to, gpt, parts, ks = ops.iconv_grouped_layout(c, c, kh, kw, c)
            assert nbytes == kh * kw * ops.code_channels(c) and (nt, tn, to, gpt, parts, ks) == (0,) * 6


# ---------------------------------------------------------------------------------------------
# the weight operands
# ---------------------------------------------------------------------------------------------
def _numpy_operand(cw: np.ndarray, groups: int) -> np.ndarray:
    """Restatement of include/mhaq_fq.h's grouped weight operand, one byte at a time."""
    n, cin_g, kh, kw = cw.shape
    cin, cout_g, taps = cin_g * groups, n // groups, kh * kw
    cp = (cin + 15) // 16 * 16
    nbytes, nt, tn, to, gpt, parts, ks = ops.iconv_grouped_layout(cin, n, kh, kw, groups)
    if nt == 0:
        out = np.zeros((taps, cp), np.uint8)
        for ch in range(n):
            out[:, ch] = cw[ch, 0].reshape(-1)
        return out.reshape(-1)
    out = np.zeros(nbytes, np.uint8)
    for t in range(nt):
        if parts == 1:
            groups_t = list(range(t * gpt, min(groups, (t + 1) * gpt)))
            chans = list(range(groups_t[0] * cout_g, (groups_t[-1] + 1) * cout_g))
        else:
            groups_t = [t // parts]
            lo = groups_t[0] * cout_g + (t % parts) * to
            chans = list(range(lo, min(lo + to, (groups_t[0] + 1) * cout_g)))
        c_lo = groups_t[0] * cin_g // 16
        kc = ((groups_t[-1] + 1) * cin_g + 15) // 16 - c_lo
        for r in range(tn):
            for kk in range(ks * 128):
                v = 0
                tap, q = divmod(kk, kc * 16)
                if tap < taps:
                    ch_in = c_lo * 16 + q
                    if r < len(chans):
                        nn_ = chans[r]
                        g = nn_ // cout_g
                        if g * cin_g <= ch_in < (g + 1) * cin_g:
                            v = cw[nn_, ch_in - g * cin_g].reshape(-1)[tap]
                    elif to <= r < to + len(groups_t):
                        g = groups_t[r - to]
                        v = 1 if g * cin_g <= ch_in < (g + 1) * cin_g else 0
                st, qq = divmod(kk, 128)
                c16, j = divmod(qq, 16)
                out[((t * ks + st) * tn * 128) + (r // 8) * 1024 + c16 * 128 + (r % 8) * 16 + j] = v
    return out


@pytest.mark.parametrize("n,cin,groups,k", [
    (8, 8, 8, (3, 3)),          # depthwise
    (17, 17, 17, (5, 3)),       # depthwise, a partial chunk
    (16, 8, 8, (3, 3)),         # channel multiplier 2
    (12, 6, 3, (3, 3)),         # 2 channels per group
    (64, 32, 8, (1, 3)),        # 4 per group
    (30, 51, 3, (3, 3)),        # 17 per group: groups straddle chunks
    (6, 4, 1, (3, 3)),          # one group (a dilated dense layer)
    (520, 6, 2, (1, 1)),        # groups wider than a tile: split in two
    (200, 96, 2, (3, 3)),       # 48 per group
])
def test_weight_operand_matches_numpy_restatement(n, cin, groups, k):
    rng = np.random.default_rng(n * 131 + cin * 7 + groups)
    cw = rng.integers(0, 256, size=(n, cin // groups, *k), dtype=np.int64)
    got = ops.iconv_grouped_weight_operand(torch.from_numpy(cw), groups).numpy()
    assert np.array_equal(got, _numpy_operand(cw.astype(np.uint8), groups))


# ---------------------------------------------------------------------------------------------
# the expansion against fp64 grouped / dilated convolution
# ---------------------------------------------------------------------------------------------
GCASES = [  # (C, N, groups, (kh, kw), (sh, sw), (ph, pw), (dh, dw), H, W)
    (6, 6, 6, (3, 3), (1, 1), (1, 1), (1, 1), 9, 7),        # depthwise
    (5, 5, 5, (5, 3), (2, 1), (2, 0), (1, 2), 13, 11),      # depthwise, per-axis geometry and dilation
    (4, 8, 4, (3, 3), (2, 2), (1, 1), (1, 1), 8, 9),        # channel multiplier 2
    (8, 6, 2, (3, 3), (1, 1), (2, 2), (2, 2), 10, 9),       # grouped and dilated
    (12, 9, 3, (3, 1), (1, 2), (1, 0), (3, 1), 12, 10),
    (3, 4, 1, (3, 3), (1, 1), (4, 4), (4, 4), 9, 12),       # dilated, groups = 1
    (4, 4, 1, (2, 3), (2, 3), (0, 3), (2, 3), 7, 14),
    (6, 6, 6, (3, 3), (1, 1), (5, 1), (3, 1), 2, 4),        # outputs with no valid tap
]


@pytest.mark.parametrize("case", GCASES)
@pytest.mark.parametrize("zpa_nonzero", [False, True])
@pytest.mark.parametrize("with_bias", [False, True])
def test_expansion_equals_fp64_conv(case, zpa_nonzero, with_bias):
    c, n, groups, (kh, kw), stride, pad, dil, h, w = case
    g = torch.Generator().manual_seed(hash((case, zpa_nonzero, with_bias)) & 0xFFFF)
    a_top, w_top = 15, 7
    ca = torch.randint(0, a_top + 1, (2, c, h, w), generator=g)
    cw = torch.randint(0, w_top + 1, (n, c // groups, kh, kw), generator=g)
    sa, zpa = 2.0 ** -5, (-1.375 if zpa_nonzero else 0.0)
    sw = torch.exp2(torch.randint(-9, -5, (n,), generator=g).float())
    zpw = -torch.rand(n, generator=g) * 0.1
    bias = torch.randn(n, generator=g) if with_bias else None
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, bias, a_top, w_top, groups=groups, dilation=dil)
    assert L.groups == groups and L.dilation == dil and L.cin == c

    conv = dict(stride=stride, padding=pad, dilation=dil, groups=groups)
    a = ca.double() * sa + zpa
    wt = cw.double() * sw.double().reshape(-1, 1, 1, 1) + zpw.double().reshape(-1, 1, 1, 1)
    ref = F.conv2d(a, wt, None if bias is None else bias.double(), **conv)

    s = F.conv2d(ca.double(), cw.double(), **conv)
    sa_m = F.conv2d(ca.double(), torch.ones(n, c // groups, kh, kw, dtype=torch.float64), **conv)  # SA[m][g(n)]
    hc, hv = ops.tap_classes(h, kh, stride[0], pad[0], dil[0])
    wc, wv = ops.tap_classes(w, kw, stride[1], pad[1], dil[1])
    ctab = L.constant_table(hv, wv)
    phc, pwc, nwc, pctab = L.pattern_tables(h, w, stride, pad)
    assert torch.equal(phc, hc) and torch.equal(pwc, wc) and nwc == wv.shape[0]
    assert torch.equal(pctab, ctab.float())
    assert L.out_size(h, w, stride, pad) == tuple(ref.shape[2:])
    p = hc.long()[:, None] * wv.shape[0] + wc.long()[None, :]
    cterm = ctab[p].permute(2, 0, 1)[None]
    swn, zpwn = L.sw.reshape(1, -1, 1, 1), L.zpw.reshape(1, -1, 1, 1)
    y = sa * swn * s + sa * zpwn * sa_m + cterm
    scale = (sa * swn * s).abs() + (sa * zpwn * sa_m).abs() + cterm.abs()
    assert y.shape == ref.shape
    assert torch.all((y - ref).abs() <= 1e-12 * scale + 1e-300)


@pytest.mark.parametrize("size,k,stride,pad,dil", [
    (9, 3, 1, 2, 2), (9, 3, 2, 4, 4), (14, 3, 1, 4, 4), (5, 3, 1, 4, 3), (7, 5, 2, 2, 2),
    (3, 2, 1, 3, 5), (12, 3, 3, 0, 2), (1, 3, 1, 2, 2),
])
def test_tap_classes_with_dilation_against_direct_enumeration(size, k, stride, pad, dil):
    cls, valid = ops.tap_classes(size, k, stride, pad, dil)
    out = (size + 2 * pad - dil * (k - 1) - 1) // stride + 1
    assert cls.shape == (out,) and valid.shape[1] == k
    assert len({tuple(v) for v in valid.tolist()}) == valid.shape[0]
    for o in range(out):
        assert valid[cls[o]].tolist() == [0 <= o * stride - pad + t * dil < size for t in range(k)], o


# ---------------------------------------------------------------------------------------------
# build_integer_model: the refusal by default, the layers on request
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("what", ["groups", "dilation", "depthwise"])
def test_refused_by_default_built_on_request(what):
    conv = {"groups": NoisyConv2d(4, 8, 3, padding=1, groups=2, qscheme=QScheme.PER_CHANNEL),
            "dilation": NoisyConv2d(3, 8, 3, padding=2, dilation=2, qscheme=QScheme.PER_CHANNEL),
            "depthwise": NoisyConv2d(8, 8, 3, padding=1, groups=8, qscheme=QScheme.PER_CHANNEL)}[what]
    net = _Net(conv)
    blob = _blob(net)
    with pytest.raises(ValueError, match="c: grouped or dilated convolutions are not supported"):
        build_integer_model(net, blob)
    q = build_integer_model(net, blob, allow_groups_and_dilation=True)
    assert isinstance(q.c, IntegerConv2d)
    assert q.c.groups == conv.groups and q.c.dilation == tuple(conv.dilation)
    L = q.c.operands
    assert not L.dense and L.groups == conv.groups and L.dilation == tuple(conv.dilation)
    cw = torch.zeros(conv.weight.shape, dtype=torch.int64)
    assert L.weight.numel() == ops.iconv_grouped_weight_operand(cw, conv.groups).numel()


def test_int32_bound_counts_the_channels_of_one_group():
    # 3x3 x 4096 input channels at 8 x 8 bits overflows densely, not in 16 groups of 256
    for groups, refused in ((1, True), (16, False)):
        net = _Net(NoisyConv2d(4096, 32, 3, padding=1, dilation=2, groups=groups, qscheme=QScheme.PER_CHANNEL))
        blob = _blob(net, a_levels=256, w_bits=8)
        if refused:
            with pytest.raises(ValueError, match="c: K .* overflow"):
                build_integer_model(net, blob, allow_groups_and_dilation=True)
        else:
            build_integer_model(net, blob, allow_groups_and_dilation=True)


def test_operand_geometry_must_match():
    L = ops.int_layer_operands(torch.zeros(4, 2, 3, 3, dtype=torch.int64), 1.0, 0.0, 1.0, 0.0, None, 15, 15,
                               groups=2, dilation=2)
    codes = torch.zeros(1, 5, 5, 16, dtype=torch.uint8)
    with pytest.raises(ValueError, match="groups=1 differs"):
        ops.int_conv2d(codes, L, 1, 2, groups=1)
    with pytest.raises(ValueError, match="dilation"):
        ops.int_conv2d_fused(codes, L, 1, 2, dilation=1)


# ---------------------------------------------------------------------------------------------
# the torchvision models: which layers become integer layers and how the pass fuses them
# ---------------------------------------------------------------------------------------------
def _integer_stand_in(name):
    torch.manual_seed(0)
    model = harness.build_model(name)
    lm = harness.LModule(model, nn.MSELoss())
    cfg = harness.make_config(act_bit=4, weight_bit=4, qscheme=1, qnmethod="STE",
                              excluded_layers=harness.EXCLUDED[name], quantize_bias=False)
    qm = Quantizer(cfg)().quantize(lm, in_place=True)
    blob = _blob(qm)
    with pytest.raises(ValueError, match="grouped or dilated"):
        build_integer_model(qm, blob)
    return build_integer_model(qm, blob, allow_groups_and_dilation=True)


# model -> (Counter of (groups, dilation) over the integer convolutions,
#           fused structure: ({codes only, fp32 only, both}, act_codes inputs, unfused))
TV = {
    # 17 depthwise 3x3 layers, each fused with its BatchNorm; ReLU6 stays in torch, so fp32 out
    "mobilenet_v2": ({"dw": 17}, ({"fp32": 17}, 17, 0)),
    # 16 grouped 3x3 conv2 layers (32 groups) -> bn2 -> relu -> conv3 (an fp32 1x1)
    "resnext50_32x4d": ({(32, (1, 1)): 16}, ({"fp32": 16}, 16, 0)),
    # the 3x3 conv2 of every bottleneck.  torchvision gives each dilated stage's first block the
    # previous stage's dilation: layer1, layer2 and layer3.0 at 1, layer3.1-5 and layer4.0 at 2,
    # layer4.1-2 at 4
    "resnet50_dilated": ({(1, (1, 1)): 8, (1, (2, 2)): 6, (1, (4, 4)): 2}, ({"fp32": 16}, 16, 0)),
}


@pytest.mark.parametrize("name", list(TV))
def test_torchvision_models_fused_structure(name):
    want_geo, want_fused = TV[name]
    qi = _integer_stand_in(name)
    convs = [m for m in qi.modules() if isinstance(m, IntegerConv2d)]
    geo = collections.Counter(
        "dw" if m.groups == m.operands.cin == m.operands.n_out else (m.groups, m.dilation) for m in convs)
    assert dict(geo) == want_geo
    gm = fuse_integer_model(qi)
    kinds, act_in, unfused = fused_structure(gm)
    assert (dict(kinds), act_in, unfused) == want_fused
    fused = [m for m in gm.modules() if isinstance(m, FusedIntegerConv2d)]
    assert all(m.operands.groups == c.groups and m.operands.dilation == c.dilation for m, c in zip(fused, convs))
    # every quantized layer's BatchNorm is folded: the ones left belong to fp32 layers
    n_bn = sum(isinstance(m, nn.BatchNorm2d) for m in gm.modules())
    assert n_bn == sum(isinstance(m, nn.BatchNorm2d) for m in qi.modules()) - len(fused)


# ---------------------------------------------------------------------------------------------
# the C ABI's argument checks
# ---------------------------------------------------------------------------------------------
def test_grouped_abi_argument_errors_without_gpu():
    L = _lib.lib
    d = ctypes.c_void_p(16)

    def geo(**kw):
        g = dict(kernel_h=3, kernel_w=3, stride_h=1, stride_w=1, pad_h=1, pad_w=1, dilation_h=1, dilation_w=1,
                 groups=4)
        g.update(kw)
        return _lib.IConvGeometry(**g)

    def epi(**kw):
        e = dict(residual=None, activation=_lib.ACT_NONE, negative_slope=0.0, y=16, codes=None,
                 code_scale=None, code_zero_point=None, code_max_val=None)
        e.update(kw)
        return _lib.IConvEpilogue(**e)

    def run(g=None, e=None, **kw):
        a = dict(codes=d, weights=d, alpha=d, beta=d, ctab=d, hc=d, wc=d, nwc=1, b=2, h=8, w=8, cin=16, n=8,
                 at=15, wt=15)
        a.update(kw)
        g = geo() if g is None else g
        e = epi() if e is None else e
        return L.mhaq_fq_iconv_grouped_u8(a["codes"], a["weights"], a["alpha"], a["beta"], a["ctab"], a["hc"],
                                          a["wc"], a["nwc"], a["b"], a["h"], a["w"], a["cin"], a["n"],
                                          ctypes.byref(g), a["at"], a["wt"], ctypes.byref(e), None)

    # groups that do not divide the channels, no groups, dilation < 1
    assert run(geo(groups=3)) == -1 and run(n=6, g=geo(groups=4)) == -1 and run(geo(groups=0)) == -1
    assert run(geo(dilation_h=0)) == -1 and run(geo(dilation_w=-1)) == -1
    # the dilated kernel wider than the padded image
    assert run(geo(dilation_h=5, pad_h=0)) == -1 and run(geo(dilation_w=4, pad_w=0, kernel_w=3), w=8) == -1
    # the int32 bound counts one channel's products: kh * kw * cin_g * a_top * w_top < 2^31
    big = 2 ** 31 // (9 * 255 * 255)                 # cin_g just under the bound
    assert run(cin=4 * (big + 1), n=4, at=255, wt=255) == -1
    assert L.mhaq_fq_iconv_grouped_weight_bytes(4 * big, 4, ctypes.byref(geo()), None, None, None, None, None,
                                                None) > 0
    # the other geometry, size and code-bound checks
    assert run(geo(kernel_h=0)) == -1 and run(geo(stride_w=0)) == -1 and run(geo(pad_h=-1)) == -1
    assert run(b=0) == -1 and run(h=0) == -1 and run(nwc=0) == -1 and run(at=0) == -1 and run(wt=256) == -1
    assert run(codes=ctypes.c_void_p(24)) == -1 and run(weights=ctypes.c_void_p(8)) == -1
    # null operands, geometry and epilogue
    assert run(weights=None) == -2 and run(ctab=None) == -2 and run(hc=None) == -2
    assert L.mhaq_fq_iconv_grouped_u8(d, d, d, d, d, d, d, 1, 2, 8, 8, 16, 8, None, 15, 15,
                                      ctypes.byref(epi()), None) == -2
    assert L.mhaq_fq_iconv_grouped_u8(d, d, d, d, d, d, d, 1, 2, 8, 8, 16, 8, ctypes.byref(geo()), 15, 15,
                                      None, None) == -2
    # the epilogue's checks, as in mhaq_fq_iconv_fused_u8
    assert run(e=epi(y=None)) == -1
    assert run(e=epi(codes=16, code_scale=16, code_zero_point=16)) == -2
    assert run(e=epi(activation=3)) == -1
    assert run(e=epi(y=None, codes=24, code_scale=16, code_zero_point=16, code_max_val=16)) == -1
    # the layout query refuses the same geometries
    for g in (geo(groups=3), geo(dilation_h=0), geo(groups=0)):
        assert L.mhaq_fq_iconv_grouped_weight_bytes(16, 8, ctypes.byref(g), None, None, None, None, None, None) == -1
    assert L.mhaq_fq_iconv_grouped_weight_bytes(16, 8, None, None, None, None, None, None, None) == -1


def test_integration_stubs_match_the_header():
    """The ctypes stubs of INTEGRATION.md section C for the new entry points, run against the built
    library, have the header's arities."""
    from tests.test_abi import ROOT, _header_param_counts
    counts = _header_param_counts()
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = re.search(r"```python\n(import ctypes, torch\n.*?)\ndef fake_quant_fwd", md, flags=re.S).group(1)
    ns = {}
    exec(block.replace('ctypes.CDLL("libmhaq_fq.so")', f"ctypes.CDLL({_lib.LIB_PATH!r})"), ns)
    for fn in ("mhaq_fq_iconv_grouped_u8", "mhaq_fq_iconv_grouped_weight_bytes"):
        assert len(getattr(ns["L"], fn).argtypes) == counts[fn], fn
    assert [f[0] for f in ns["Geometry"]._fields_] == [f[0] for f in _lib.IConvGeometry._fields_]
