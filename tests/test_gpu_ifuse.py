"""GPU: the fused epilogue of the integer convolution (mhaq_fq_iconv_fused_u8, ops.int_conv2d_fused)
and the fused integer models of fuse_integer_model.

- The epilogue equals the composition int_conv2d -> + residual -> torch activation -> act_codes
  bit for bit, fp32 compared as int32 and codes exactly (padding channels included).
- A folded BatchNorm stays within the operator bar of tests/test_gpu_iconv.py.
- Exported models: every fused layer, fed the inputs its unfused counterpart received, lies within
  its bar of the fp64 chain; whole networks agree with the fake-quant and the unfused models;
  a fused ResNet-20 replays bit-identically in a CUDA graph and runs one act_codes launch."""
import copy
import operator

import pytest
import torch
import torch.nn.functional as F
from torch import fx

from mhaq_b200 import harness, ops
from mhaq_b200.quantization.gdnsq.export import build_integer_model, export_quantized, fuse_integer_model
from mhaq_b200.quantization.gdnsq.inference import FusedIntegerConv2d, IntegerConv2d, _Tracer, unpack_weight_codes
from tests.test_gpu_iconv import OP_CASES, _act_operands, _check_bar, _random_layer, _trained
from tests.test_gpu_pack import _batches
from tests.test_ifuse_cpu import STRUCTURE, fused_structure

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
U = 2.0 ** -24


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _random_bn(n, seed):
    g = torch.Generator().manual_seed(seed)
    bn = torch.nn.BatchNorm2d(n).eval()
    with torch.no_grad():
        bn.running_mean.copy_(torch.randn(n, generator=g))
        bn.running_var.copy_(torch.rand(n, generator=g) * 2 + 1e-3)
        bn.weight.copy_(torch.randn(n, generator=g))
        bn.bias.copy_(torch.randn(n, generator=g))
    return bn.to(DEV)


def _i32(t):
    return t.contiguous(memory_format=torch.channels_last).view(torch.int32)


NEXT = [(2, False), (16, True), (256, True), (256, False)]      # next quantizer: levels, signed


@pytest.mark.parametrize("ci", range(len(OP_CASES)))
@pytest.mark.parametrize("residual", [False, True])
@pytest.mark.parametrize("activation", [None, "relu", "leaky_relu"])
@pytest.mark.parametrize("outputs", ["fp32", "codes", "both"])
def test_epilogue_equals_composition(ci, residual, activation, outputs):
    bsz, h, w, c, n, k, stride, pad, w_bits, levels = OP_CASES[ci]
    seed = 1000 + ci
    L, *_ = _random_layer(n, c, k, w_bits, levels, True, True, True, seed)
    L = ops.fold_batchnorm(L, _random_bn(n, seed))
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    ca = torch.randint(0, levels, (bsz, c, h, w), generator=g, device=DEV)
    codes = torch.zeros(bsz, h, w, L.cp, dtype=torch.uint8, device=DEV)
    codes[..., :c] = ca.permute(0, 2, 3, 1).to(torch.uint8)
    # channel 0 gives t = -0 exactly: alpha = beta = -0 and C = -0 (fma(-0, x, -0) = -0)
    hc, wc, nwc, ctab = L.pattern_tables(h, w, stride, pad)
    L.alpha[0], L.beta[0] = -0.0, -0.0
    ctab[:, 0] = -0.0
    plain = ops.int_conv2d(codes, L, stride, pad)
    levels_n, signed = NEXT[ci % len(NEXT)]
    s, b, hi = _act_operands(levels_n, signed, seed=ci)
    r = None
    if residual:
        r = torch.randn(plain.shape, generator=g, device=DEV) * levels_n * float(s) / 4
        flat = r.view(-1)
        pv = plain.contiguous().view(-1)
        flat[0::7] = -pv[0::7]                                    # t = +0
        tie = b + (torch.randint(0, levels_n, pv.shape, generator=g, device=DEV) + 0.5) * s
        flat[3::7] = (tie - pv)[3::7]                             # t on (or next to) a rounding tie
        flat[5::97] = float("nan")
        r[:, 0] = -0.0                                            # -0 + -0 = -0 in channel 0
        r = r.contiguous()                                         # NCHW: int_conv2d_fused copies it
    slope = 0.125 if activation == "leaky_relu" else None
    want_y, want_c = outputs in ("fp32", "both"), outputs in ("codes", "both")
    torch.full((bsz * plain.shape[2] * plain.shape[3] * ops.code_channels(n) + 4096,), 255, dtype=torch.uint8,
               device=DEV)                                        # leave 0xff in the allocator's free blocks
    y, cod = ops.int_conv2d_fused(codes, L, stride, pad, residual=r, activation=activation, negative_slope=slope,
                                  out_fp32=want_y, code_params=(s, b, hi) if want_c else None)
    ref = plain if r is None else plain + r
    if activation == "relu":
        ref = torch.relu(ref)
    elif activation == "leaky_relu":
        ref = F.leaky_relu(ref, slope)
    assert (y is not None) == want_y and (cod is not None) == want_c
    if want_y:
        assert y.is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(_i32(y), _i32(ref))
    if want_c:
        assert torch.equal(cod, ops.act_codes(ref, s, b, hi)[0])
    if activation is None and not residual:
        assert bool((_i32(ref)[:, 0] == -2 ** 31).all())     # channel 0 is -0: exercised


@pytest.mark.parametrize("case", OP_CASES)
def test_batchnorm_fold_bar(case):
    """|y - ref64| <= 4u (|alpha' S| + |beta' SA| + |C'|), ref64 the fp64 BatchNorm of the fp64
    convolution of the exact dequantized values (its fold is exact in fp64 to ~1e-15 relative)."""
    bsz, h, w, c, n, k, stride, pad, w_bits, levels = case
    seed = hash(case) & 0xFFFF
    L, cw, sw, zpw, sa, zpa, bias = _random_layer(n, c, k, w_bits, levels, True, True, True, seed)
    Lf = ops.fold_batchnorm(L, _random_bn(n, seed))
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    ca = torch.randint(0, levels, (bsz, c, h, w), generator=g, device=DEV)
    codes = torch.zeros(bsz, h, w, L.cp, dtype=torch.uint8, device=DEV)
    codes[..., :c] = ca.permute(0, 2, 3, 1).to(torch.uint8)
    y, _ = ops.int_conv2d_fused(codes, Lf, stride, pad)
    _check_bar(y, ca, Lf, cw, Lf.sw, Lf.zpw, sa, zpa, Lf.bias, stride, pad)


# ---------------------------------------------------------------------------------------------
# exported models
# ---------------------------------------------------------------------------------------------
def _resnet18():
    torch.manual_seed(0)
    x = torch.randn(8, 3, 64, 64, device=DEV)
    qm = harness.build_qat("resnet18", qnmethod="STE", distillation=False, num_classes=10, calib_batch=x,
                          calib_bits=4)
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for m in qm.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
    return qm.eval(), torch.randn(16, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))


def _rfdn():
    torch.manual_seed(0)
    x = torch.rand(2, 3, 32, 32, device=DEV)
    qm = harness.build_qat("rfdn", qnmethod="LSQ", distillation=False, calib_batch=x, calib_bits=4)
    return qm.eval(), torch.rand(2, 3, 32, 32, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))


MODELS = [("resnet20", "STE", False), ("resnet20", "LSQ", False), ("resnet20", "STE", True),
          ("bias_net", "STE", False), ("asym_net", "STE", False), ("resnet18", "STE", False),
          ("rfdn", "LSQ", False)]


def _model(kind, method, channels_last):
    if kind == "resnet18":
        return _resnet18()
    if kind == "rfdn":
        return _rfdn()
    return _trained(kind, method, channels_last), torch.cat([b[0] for b in _batches(8, 11, channels_last)])


def _node_values(gm, x):
    """Every node's value (by name) in one run of the traced graph."""
    vals = {}

    class Rec(fx.Interpreter):
        def run_node(self, n):
            out = super().run_node(n)
            vals[n.name] = out
            return out
    Rec(gm).run(x)
    return vals


def _ref64(codes_nchw, L, cw, stride, pad):
    """fp64 convolution of the exact dequantized values with the (folded) fp64 operands, and the
    bar terms |alpha S| + |beta SA| + |C| of the fp32 operands."""
    ca = codes_nchw.double()
    c, kh, kw = cw.shape[1:]
    a = ca * L.sa + L.zpa
    wt = cw.double() * L.sw.reshape(-1, 1, 1, 1) + L.zpw.reshape(-1, 1, 1, 1)
    ref = F.conv2d(a, wt, L.bias, stride=stride, padding=pad)
    s = F.conv2d(ca, cw.double(), stride=stride, padding=pad)
    sam = F.conv2d(ca, torch.ones(1, c, kh, kw, dtype=torch.float64, device=DEV), stride=stride, padding=pad)
    hc, wc, nwc, ctab = L.pattern_tables(ca.shape[2], ca.shape[3], stride, pad)
    cterm = ctab.double()[hc.long()[:, None] * nwc + wc.long()[None, :]].permute(2, 0, 1)[None]
    terms = ((L.alpha.double().reshape(1, -1, 1, 1) * s).abs() + (L.beta.double().reshape(1, -1, 1, 1) * sam).abs()
             + cterm.abs())
    return ref, terms


@pytest.mark.parametrize("kind,method,channels_last", MODELS)
def test_fused_layers_within_their_bar(kind, method, channels_last):
    """Each fused layer, fed the input (its codes, or the fp32 input it quantizes) and the residual
    its unfused counterpart received in the unfused integer model, returns fp32 y with
        |y - ref64| <= 4u (|alpha' S| + |beta' SA| + |C'|) + (n_add + n_leaky) * u * |y|,
    ref64 the fp64 chain: the fp64 convolution of the exact dequantized values with the folded fp64
    operands (= the fp64 BatchNorm of it), + the residual, then the activation, in fp64.  The first
    term is the fold bar (tests/test_gpu_iconv.py), each residual add and LeakyReLU multiply adds at
    most one rounding of |y| (a slope <= 1 does not enlarge the earlier error; ReLU is exact).  Its
    codes equal act_codes of its own fp32 output."""
    qm, x = _model(kind, method, channels_last)
    blob = export_quantized(qm)
    qi = build_integer_model(qm, blob)
    gm = fuse_integer_model(qi)
    if kind in STRUCTURE:
        kinds, act_in, unfused = fused_structure(gm)
        assert (dict(kinds), act_in, unfused) == STRUCTURE[kind]
    with torch.no_grad():
        ref_gm = fx.GraphModule(qi, _Tracer().trace(qi))
        vals = _node_values(ref_gm, x[:4])
        ints = {n: m for n, m in qi.named_modules() if isinstance(m, IntegerConv2d)}
        conv_nodes = {n.target: n for n in ref_gm.graph.nodes if n.op == "call_module" and n.target in ints}
        n_checked = 0
        for node in gm.graph.nodes:
            if node.op != "call_module" or not isinstance(gm.get_submodule(node.target), FusedIntegerConv2d):
                continue
            m = gm.get_submodule(node.target)
            unf = ints[node.target]
            xin = vals[conv_nodes[node.target].args[0].name]
            codes, _ = ops.act_codes(xin, unf.act_scale, unf.act_zero_point, unf.act_max_val)
            res = None
            if m.residual:      # an original node, or the fp32 output of a fused chain: its last node
                rn = node.args[1]
                src = rn.args[0] if rn.op == "call_function" and rn.target is operator.getitem else None
                res = vals[src.meta["fused_chain"][-1] if src is not None else rn.name]
            probe = copy.copy(m)
            probe.out_fp32 = True
            y, cod = probe(codes if m.codes_in else xin, *(() if res is None else (res,)))
            cw = unpack_weight_codes(blob["layers"][f"{node.target}.0"]).to(DEV)
            c = cw.shape[1]
            ref, terms = _ref64(codes[..., :c].permute(0, 3, 1, 2), m.operands, cw, m.stride, m.padding)
            n_round = 0
            if res is not None:
                ref = ref + res.double()
                n_round += 1
            if m.activation == "relu":
                ref = ref.clamp_min(0)
            elif m.activation == "leaky_relu":
                ref = torch.where(ref > 0, ref, ref * m.negative_slope)
                n_round += 1
            err = (y.double() - ref).abs()
            bound = 4 * U * terms + n_round * U * y.double().abs()
            assert bool((err <= bound).all()), \
                f"{kind} {node.target}: max err / bound {float((err / bound.clamp_min(1e-300)).max()):.3g}"
            if cod is not None:
                assert torch.equal(cod, ops.act_codes(y, *m.code_params)[0]), node.target
            n_checked += 1
        assert n_checked > 0


@pytest.mark.parametrize("kind,method,channels_last", MODELS)
def test_fused_network_agrees(kind, method, channels_last):
    """Classifiers: the fused model picks the fake-quant model's and the unfused integer model's
    class for >= 90 % of a fixed batch (as test_network_logits_agree; a last-bit difference can flip
    a later code, so no per-sample bound).  RFDN: a finite output; the largest differences are
    printed."""
    qm, x = _model(kind, method, channels_last)
    qi = build_integer_model(qm, export_quantized(qm))
    gm = fuse_integer_model(qi)
    with torch.no_grad():
        ref, unf, got = qm(x).float(), qi(x).float(), gm(x).float()
    d_fq, d_int = float((got - ref).abs().max()), float((got - unf).abs().max())
    print(f"{kind}/{method}/cl={channels_last}: max |d| vs fake-quant {d_fq:.3e}, vs integer {d_int:.3e}")
    assert got.shape == ref.shape and bool(torch.isfinite(got).all())
    if kind != "rfdn":
        assert float((got.argmax(1) == ref.argmax(1)).float().mean()) >= 0.9
        assert float((got.argmax(1) == unf.argmax(1)).float().mean()) >= 0.9


def _fused_resnet20():
    qm = _trained("resnet20", "STE", False)
    return fuse_integer_model(build_integer_model(qm, export_quantized(qm)))


def test_graph_capture_of_the_fused_resnet20():
    gm = _fused_resnet20()
    x = _batches(1, 3)[0][0]
    with torch.no_grad():
        eager = gm(x)                      # builds the per-size pattern tables
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            gm(x)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = gm(x)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), eager.view(torch.int32))


def test_launches_of_the_fused_resnet20():
    """One act_codes launch (layer1.0.conv1's input), 18 integer convolutions, and no BatchNorm
    kernel after the stem's."""
    gm = _fused_resnet20()
    x = _batches(1, 3)[0][0]
    with torch.no_grad():
        gm(x)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            gm(x)
            torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [n for n in names if "memcpy" not in n.lower() and "memset" not in n.lower()]
    assert sum("fq_act_codes_kernel" in n for n in kernels) == 1, kernels
    assert sum("fq_iconv_kernel" in n for n in kernels) == 18, kernels
    first_int = next(i for i, n in enumerate(kernels) if "fq_act_codes_kernel" in n)
    bn_after = [n for n in kernels[first_int:] if "bn_" in n.lower() or "batch_norm" in n.lower()]
    assert not bn_after, bn_after


def test_broadcast_residual_matches_the_unfused_model_bit_for_bit():
    """conv -> + x.mean(keepdim) ([B, C, 1, 1], broadcast) -> ReLU -> conv, no BatchNorm: the fused
    layer adds the broadcast operand as torch does, so fused and unfused models agree bitwise."""
    from collections import OrderedDict
    from torch import nn
    from mhaq_b200.aux.types import QScheme
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
    from tests.test_iconv_cpu import _blob

    def pair():
        conv = NoisyConv2d(8, 8, 3, padding=1, bias=False, qscheme=QScheme.PER_CHANNEL)
        return nn.Sequential(OrderedDict([("activations_quantizer", NoisyAct(signed=True)), ("0", conv)]))

    class M(nn.Module):
        def __init__(self):
            super().__init__()
            self.a, self.b = pair(), pair()

        def forward(self, x):
            return self.b(F.relu(self.a(x) + x.mean((2, 3), keepdim=True)))
    net = M().to(DEV)
    qi = build_integer_model(net, _blob(net))          # operands on the model's device
    gm = fuse_integer_model(qi)
    assert isinstance(gm.a, FusedIntegerConv2d) and gm.a.residual and gm.b.codes_in
    x = torch.randn(3, 8, 9, 7, device=DEV)
    with torch.no_grad():
        assert torch.equal(gm(x).view(torch.int32), qi(x).view(torch.int32))
