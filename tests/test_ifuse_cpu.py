"""CPU: the fused integer epilogue's host side, without a GPU.

- The BatchNorm fold (ops.fold_batchnorm, DESIGN §3 "Fused epilogue"): alpha'*S + beta'*SA + C'[p] with
  the fp64 terms of the folded operands equals the fp64 BatchNorm of the fp64 convolution of the
  dequantized values, and alpha' / beta' / C' are those fp64 terms rounded once.
- The graph pass (fuse_integer_model) on integer stand-ins of the harness models: how many fused
  layers of each kind it makes, how many layers still quantize fp32 with act_codes, and what it
  must leave alone.
- The argument checks of mhaq_fq_iconv_fused_u8."""
import collections
import ctypes
import operator
from collections import OrderedDict

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from mhaq_b200 import harness, ops
from mhaq_b200.aux.types import QScheme
from mhaq_b200.quantization.gdnsq.export import build_integer_model, fuse_integer_model
from mhaq_b200.quantization.gdnsq.inference import FusedIntegerConv2d, IntegerConv2d, IntegerLinear
from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
from mhaq_b200.quantization.quantizer import Quantizer
from tests.test_gpu_pack import _AsymNet, _BiasNet
from tests.test_iconv_cpu import CASES, _blob


# ---------------------------------------------------------------------------------------------
# the BatchNorm fold against fp64 BatchNorm(conv)
# ---------------------------------------------------------------------------------------------
def _bn(n, g, affine=True, tiny_var=False, negative=False):
    bn = nn.BatchNorm2d(n, eps=1e-5, affine=affine).eval()
    with torch.no_grad():
        bn.running_mean.copy_(torch.randn(n, generator=g))
        bn.running_var.copy_(torch.rand(n, generator=g) * (1e-9 if tiny_var else 2.0) + (0 if tiny_var else 0.1))
        if affine:
            bn.weight.copy_(torch.randn(n, generator=g) * 2)
            if negative:
                bn.weight[::2] = -bn.weight[::2].abs()
            bn.bias.copy_(torch.randn(n, generator=g))
    return bn


@pytest.mark.parametrize("case", CASES[:5])
@pytest.mark.parametrize("bn_kind", ["plain", "negative_gamma", "tiny_var", "no_affine"])
@pytest.mark.parametrize("per_channel,with_bias", [(True, True), (False, False), (True, False)])
def test_batchnorm_fold_equals_fp64_batchnorm_of_fp64_conv(case, bn_kind, per_channel, with_bias):
    c, n, (kh, kw), stride, pad, h, w = case
    g = torch.Generator().manual_seed(hash((case, bn_kind, per_channel, with_bias)) & 0xFFFF)
    a_top, w_top = 15, 7
    ca = torch.randint(0, a_top + 1, (2, c, h, w), generator=g)
    cw = torch.randint(0, w_top + 1, (n, c, kh, kw), generator=g)
    sa, zpa = 2.0 ** -5, -1.375
    rows = n if per_channel else 1
    sw = torch.exp2(torch.randint(-9, -5, (rows,), generator=g).float())
    zpw = -torch.rand(rows, generator=g) * 0.1
    bias = torch.randn(n, generator=g) if with_bias else None
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, bias, a_top, w_top)
    bn = _bn(n, g, affine=bn_kind != "no_affine", tiny_var=bn_kind == "tiny_var",
             negative=bn_kind == "negative_gamma")
    Lf = ops.fold_batchnorm(L, bn)

    a = ca.double() * sa + zpa
    wt = cw.double() * sw.double().reshape(-1, 1, 1, 1) + zpw.double().reshape(-1, 1, 1, 1)
    conv = F.conv2d(a, wt, None if bias is None else bias.double(), stride=stride, padding=pad)
    mean, var = bn.running_mean.double(), bn.running_var.double()
    gamma = bn.weight.double() if bn.affine else torch.ones(n, dtype=torch.float64)
    beta = bn.bias.double() if bn.affine else torch.zeros(n, dtype=torch.float64)
    ref = ((conv - mean.reshape(1, -1, 1, 1)) / torch.sqrt(var + bn.eps).reshape(1, -1, 1, 1)
           * gamma.reshape(1, -1, 1, 1) + beta.reshape(1, -1, 1, 1))

    s = F.conv2d(ca.double(), cw.double(), stride=stride, padding=pad)
    sa_m = F.conv2d(ca.double(), torch.ones(1, c, kh, kw, dtype=torch.float64), stride=stride, padding=pad)
    hc, hv = ops.tap_classes(h, kh, stride[0], pad[0])
    wc, wv = ops.tap_classes(w, kw, stride[1], pad[1])
    ctab = Lf.constant_table(hv, wv)
    p = hc.long()[:, None] * wv.shape[0] + wc.long()[None, :]
    cterm = ctab[p].permute(2, 0, 1)[None]
    al, be = sa * Lf.sw.reshape(1, -1, 1, 1), sa * Lf.zpw.reshape(1, -1, 1, 1)
    y = al * s + be * sa_m + cterm
    scale = (al * s).abs() + (be * sa_m).abs() + cterm.abs()
    assert torch.all((y - ref).abs() <= 1e-12 * scale + 1e-300)

    # alpha' / beta' / C' are the fp64 terms rounded once, the k * ... products formed in fp64
    kk = gamma / torch.sqrt(var + bn.eps)
    assert torch.equal(Lf.sw, kk * L.sw) and torch.equal(Lf.zpw, kk * L.zpw)
    assert torch.equal(Lf.alpha, (sa * Lf.sw).float()) and torch.equal(Lf.beta, (sa * Lf.zpw).float())
    assert torch.equal(Lf.pattern_tables(h, w, stride, pad)[3], ctab.float())
    # the weight operand is shared, the unfolded operands are untouched
    assert Lf.weight is L.weight and torch.equal(L.alpha, (sa * L.sw).float())


def test_fold_refuses_batch_statistics():
    L = ops.int_layer_operands(torch.zeros(4, 3, 3, 3, dtype=torch.int64), 0.1, 0.0, 0.5, 0.0, None, 15, 15)
    with pytest.raises(ValueError, match="running statistics"):
        ops.fold_batchnorm(L, nn.BatchNorm2d(4, track_running_stats=False).eval())
    with pytest.raises(ValueError, match="running statistics"):
        ops.fold_batchnorm(L, nn.BatchNorm2d(4).train())
    with pytest.raises(ValueError, match="features"):
        ops.fold_batchnorm(L, nn.BatchNorm2d(5).eval())


# ---------------------------------------------------------------------------------------------
# the graph pass on the harness models
# ---------------------------------------------------------------------------------------------
def _integer_stand_in(name):
    """build_integer_model of the quantized harness model (or the biased test net) with a
    synthetic export: the structure is what the pass sees, the numbers do not matter here."""
    torch.manual_seed(0)
    if name in ("bias_net", "asym_net"):   # per tensor: the synthetic export has per-tensor Linear weights
        model, excl, qb, qscheme = (_BiasNet() if name == "bias_net" else _AsymNet()), (), False, 0
    else:
        model, excl, qb, qscheme = harness.build_model(name), harness.EXCLUDED[name], False, 1
    lm = (harness.SRModule if name == "rfdn" else harness.LModule)(model, nn.MSELoss())
    cfg = harness.make_config(act_bit=4, weight_bit=4, qscheme=qscheme, qnmethod="STE", excluded_layers=excl,
                              quantize_bias=qb)
    qm = Quantizer(cfg)().quantize(lm, in_place=True)
    return build_integer_model(qm, _blob(qm))


def fused_structure(gm):
    """(Counter of fused layers by output kind, layers that still quantize fp32 with act_codes,
    IntegerConv2d layers left unfused)."""
    kinds = collections.Counter()
    act_in, unfused = 0, 0
    for m in gm.modules():
        if isinstance(m, FusedIntegerConv2d):
            kinds["both" if (m.code_params is not None and m.out_fp32)
                  else ("codes" if m.code_params is not None else "fp32")] += 1
            act_in += not m.codes_in
        elif isinstance(m, (IntegerConv2d, IntegerLinear)):
            act_in += 1
            unfused += isinstance(m, IntegerConv2d)
    return kinds, act_in, unfused


# model -> ({codes only, fp32 only, both}, act_codes inputs, IntegerConv2d left unfused)
STRUCTURE = {
    "resnet20": ({"codes": 9, "fp32": 1, "both": 8}, 1, 0),
    "resnet18": ({"codes": 8, "fp32": 1, "both": 7}, 1, 0),
    # per RFDB: c1_r, c2_r -> add -> LeakyReLU feed c2_r / c3_r and fp32 users (both); c3_r -> c4,
    # ESA conv_max -> conv3 -> conv3_ (codes); c4 -> LeakyReLU -> cat, conv3_ -> interpolate
    # (fp32); ESA conv2 -> max_pool stays an IntegerConv2d.  Plus LR_conv -> add (fp32).  The
    # c1_r, conv_max, conv2 of each block and LR_conv quantize fp32: 13 act_codes inputs.
    "rfdn": ({"codes": 12, "fp32": 9, "both": 8}, 13, 4),
    # c1 -> relu -> c2 (codes), c2 -> relu -> pool (fp32, codes in); the Linear head keeps act_codes
    "bias_net": ({"codes": 1, "fp32": 1}, 2, 0),
    # c1 (1x3) -> relu -> c2 (codes); c2 (3x1) -> bn -> relu feeds b1 and the fp32 downsample
    # (both); b1 -> bn -> relu -> b2 (codes); b2 -> bn -> + downsample -> relu -> pool and
    # c3 -> relu -> pool (fp32).  c1, c3 and the Linear head quantize fp32: 3 act_codes inputs
    "asym_net": ({"codes": 2, "both": 1, "fp32": 2}, 3, 0),
}


@pytest.mark.parametrize("name", list(STRUCTURE))
def test_pass_structure(name):
    qi = _integer_stand_in(name)
    before = {n: m for n, m in qi.named_modules()}
    gm = fuse_integer_model(qi)
    kinds, act_in, unfused = fused_structure(gm)
    want_kinds, want_act, want_unfused = STRUCTURE[name]
    assert dict(kinds) == want_kinds and act_in == want_act and unfused == want_unfused
    # no block BatchNorm remains (the stem's and the unquantized 1x1 shortcuts' do)
    left = [n for n, m in gm.named_modules() if isinstance(m, nn.BatchNorm2d)]
    assert all(n == "model.bn1" or ".downsample." in n for n in left), left
    # the argument is unmodified and shares its weight operands with the fused model
    assert {n: m for n, m in qi.named_modules()} == before
    ints = {n: m for n, m in qi.named_modules() if isinstance(m, IntegerConv2d)}
    for n, m in gm.named_modules():
        if isinstance(m, FusedIntegerConv2d):
            assert m.operands.weight is ints[n].operands.weight and m.act_scale is ints[n].act_scale
    # consumers read their producer's codes: every codes output has exactly one integer consumer
    for node in gm.graph.nodes:
        if node.op == "call_function" and node.target is operator.getitem and node.args[1] == 1:
            (user,) = node.users
            assert isinstance(gm.get_submodule(user.target), FusedIntegerConv2d)
            assert gm.get_submodule(user.target).codes_in


# ---------------------------------------------------------------------------------------------
# what the pass leaves alone
# ---------------------------------------------------------------------------------------------
def _pair(cin, cout):
    conv = NoisyConv2d(cin, cout, 3, padding=1, bias=False, qscheme=QScheme.PER_CHANNEL)
    return nn.Sequential(OrderedDict([("activations_quantizer", NoisyAct(signed=True)), ("0", conv)]))


class _Small(nn.Module):
    def __init__(self, variant):
        super().__init__()
        self.variant = variant
        self.a, self.b = _pair(8, 8), _pair(8, 8)
        self.bn = nn.BatchNorm2d(8, track_running_stats=variant != "bn_without_stats")
        self.plain = nn.Conv2d(8, 8, 1)

    def forward(self, x):
        y = self.bn(self.a(x))
        if self.variant == "second_user":
            return self.b(F.relu(y)) + y
        if self.variant == "add_alpha":
            return self.b(torch.add(y, x, alpha=2))
        if self.variant == "non_integer_consumer":
            return self.plain(F.relu(y))
        if self.variant == "data_dependent":
            return self.b(y) if bool(y.sum() > 0) else y
        return self.b(F.relu(y + x))


def _small(variant):
    net = _Small(variant)
    return build_integer_model(net, _blob(net))


def _nodes(gm, pred):
    return [n for n in gm.graph.nodes if pred(n)]


def test_pass_fuses_the_whole_chain():
    gm = fuse_integer_model(_small("full"))
    assert isinstance(gm.a, FusedIntegerConv2d) and isinstance(gm.b, FusedIntegerConv2d)
    a, b = gm.a, gm.b
    assert (a.residual, a.activation, a.out_fp32, a.codes_in) == (True, "relu", False, False)
    assert a.code_params[0] is b.act_scale and b.codes_in and b.out_fp32 and b.code_params is None
    assert not hasattr(gm, "bn") and not _nodes(gm, lambda n: n.target in (F.relu, operator.add))


def test_pass_leaves_a_batchnorm_without_running_stats():
    gm = fuse_integer_model(_small("bn_without_stats"))
    assert isinstance(gm.a, IntegerConv2d) and isinstance(gm.bn, nn.BatchNorm2d)
    assert _nodes(gm, lambda n: n.target == "bn")


def test_pass_stops_at_an_intermediate_with_a_second_user():
    gm = fuse_integer_model(_small("second_user"))
    a = gm.a
    assert isinstance(a, FusedIntegerConv2d) and a.activation is None and not a.residual
    assert a.code_params is None and a.out_fp32          # the BatchNorm folded, nothing else
    assert _nodes(gm, lambda n: n.target is F.relu)
    assert isinstance(gm.b, FusedIntegerConv2d) and gm.b.residual and not gm.b.codes_in   # b(...) + y


def test_pass_leaves_an_add_with_alpha():
    gm = fuse_integer_model(_small("add_alpha"))
    assert isinstance(gm.a, FusedIntegerConv2d) and not gm.a.residual and gm.a.code_params is None
    assert _nodes(gm, lambda n: n.target is torch.add and n.kwargs.get("alpha") == 2)


def test_pass_writes_no_codes_for_a_non_integer_consumer():
    gm = fuse_integer_model(_small("non_integer_consumer"))
    a = gm.a
    assert isinstance(a, FusedIntegerConv2d) and a.activation == "relu" and a.code_params is None and a.out_fp32
    assert isinstance(gm.plain, nn.Conv2d)


def test_untraceable_model_raises():
    with pytest.raises(ValueError, match="torch.fx cannot trace"):
        fuse_integer_model(_small("data_dependent"))


def test_leaky_relu_slopes_are_taken_from_call_and_module():
    class M(nn.Module):
        def __init__(self, mod):
            super().__init__()
            self.a, self.b, self.c = _pair(8, 8), _pair(8, 8), _pair(8, 8)
            self.act = nn.LeakyReLU(0.2) if mod else None

        def forward(self, x):
            y = self.act(self.a(x)) if self.act is not None else F.leaky_relu(self.a(x), negative_slope=0.3)
            return self.c(F.leaky_relu(self.b(y)))
    for mod, slope in ((True, 0.2), (False, 0.3)):
        net = M(mod)
        gm = fuse_integer_model(build_integer_model(net, _blob(net)))
        assert (gm.a.activation, gm.a.negative_slope) == ("leaky_relu", slope)
        assert (gm.b.activation, gm.b.negative_slope) == ("leaky_relu", 0.01)


# ---------------------------------------------------------------------------------------------
# C ABI argument errors (no kernel is launched)
# ---------------------------------------------------------------------------------------------
def test_fused_abi_argument_errors_without_gpu():
    from mhaq_b200 import _lib
    L = _lib.lib
    d = ctypes.c_void_p(16)

    def fused(epi=None, **kw):
        a = dict(codes=d, weights=d, alpha=d, beta=d, ctab=d, hc=d, wc=d, nwc=1, b=2, h=8, w=8, cp=16,
                 n=10, kh=3, kw=3, sh=1, sw=1, ph=1, pw=1, at=15, wt=15)
        a.update(kw)
        return L.mhaq_fq_iconv_fused_u8(a["codes"], a["weights"], a["alpha"], a["beta"], a["ctab"], a["hc"],
                                        a["wc"], a["nwc"], a["b"], a["h"], a["w"], a["cp"], a["n"], a["kh"],
                                        a["kw"], a["sh"], a["sw"], a["ph"], a["pw"], a["at"], a["wt"],
                                        None if epi is None else ctypes.byref(epi), None)

    def epi(**kw):
        e = dict(residual=None, activation=_lib.ACT_RELU, negative_slope=0.0, y=16, codes=None,
                 code_scale=None, code_zero_point=None, code_max_val=None)
        e.update(kw)
        return _lib.IConvEpilogue(**e)
    assert fused(None) == -2                                           # no epilogue
    assert fused(epi(y=None)) == -1                                    # no output
    assert fused(epi(codes=16, code_scale=16, code_zero_point=16)) == -2   # codes without max_val
    assert fused(epi(codes=16, code_scale=None, code_zero_point=16, code_max_val=16)) == -2
    assert fused(epi(activation=3)) == -1 and fused(epi(activation=-1)) == -1
    assert fused(epi(y=None, codes=24, code_scale=16, code_zero_point=16, code_max_val=16)) == -1  # misaligned
    # and everything mhaq_fq_iconv_u8 checks
    e = epi()
    assert fused(e, weights=None) == -2 and fused(e, ctab=None) == -2
    assert fused(e, cp=24) == -1 and fused(e, b=0) == -1 and fused(e, n=0) == -1
    assert fused(e, sh=0) == -1 and fused(e, ph=-1) == -1 and fused(e, h=1, ph=0) == -1
    assert fused(e, at=0) == -1 and fused(e, wt=256) == -1
    assert fused(e, codes=ctypes.c_void_p(24)) == -1
    assert fused(e, cp=4096, at=255, wt=255) == -1


class _Shared(nn.Module):
    """One quantized layer called at two sites (shared weights)."""

    def __init__(self):
        super().__init__()
        self.a, self.b = _pair(8, 8), _pair(8, 8)
        self.bn1, self.bn2 = nn.BatchNorm2d(8), nn.BatchNorm2d(8)

    def forward(self, x):
        return self.b(F.relu(self.bn2(self.a(F.relu(self.bn1(self.a(x)))))))


def test_pass_leaves_a_layer_called_at_two_sites():
    net = _Shared().eval()
    gm = fuse_integer_model(build_integer_model(net, _blob(net)))
    assert isinstance(gm.a, IntegerConv2d)                       # neither site fused, no codes into it
    assert len(_nodes(gm, lambda n: n.target == "a")) == 2
    assert _nodes(gm, lambda n: n.target == "bn1") and _nodes(gm, lambda n: n.target == "bn2")
    assert isinstance(gm.b, IntegerConv2d)                       # its producer is the shared layer's BN


def test_inplace_add_into_the_other_operand_is_not_matched():
    """``other += cur`` (an ``operator.iadd`` node with the chain's value on the right) updates
    ``other`` in place, which a fused layer would not do; ``cur += other`` may be fused."""
    from torch import fx
    from mhaq_b200.quantization.gdnsq.inference import _match_add
    g = fx.Graph()
    other, cur = g.placeholder("other"), g.placeholder("cur")
    into_other = g.call_function(operator.iadd, (other, cur))
    into_cur = g.call_function(operator.iadd, (cur, other))
    plain = g.call_function(operator.add, (other, cur))
    alpha = g.call_function(torch.add, (cur, other), {"alpha": 2})
    assert _match_add(into_other, cur) is None
    assert _match_add(into_cur, cur) is other and _match_add(plain, cur) is other
    assert _match_add(alpha, cur) is None


def test_broadcast_residual_becomes_the_full_fp32_operand():
    from mhaq_b200.quantization.gdnsq.inference import _as_add_operand
    L = ops.int_layer_operands(torch.zeros(4, 3, 3, 3, dtype=torch.int64), 0.1, 0.0, 0.5, 0.0, None, 15, 15)
    codes = torch.zeros(2, 6, 5, 16, dtype=torch.uint8)
    out = (2, 4, 6, 5)
    r = torch.arange(4, dtype=torch.float16).reshape(1, 4, 1, 1)
    got = _as_add_operand(r, codes, L, (1, 1), (1, 1))
    assert got.dtype == torch.float32 and tuple(got.shape) == out
    assert torch.equal(got, torch.zeros(out) + r)                # what torch's add would see
    full = torch.randn(out)
    assert _as_add_operand(full, codes, L, (1, 1), (1, 1)) is full
    for bad in (torch.zeros(out, dtype=torch.float64), torch.zeros(2, 4, 6, 6)):   # left for the op to refuse
        assert _as_add_operand(bad, codes, L, (1, 1), (1, 1)) is bad
