"""GPU: integer layers (include/mhaq_fq.h "Integer layers"): activation codes, the int8 tensor-core
convolution / linear operator, and exported models run on their codes (build_integer_model).

Operator bar.  The kernel forms y = RN32(alpha*S + beta*SA + C) in fp64 from the exact int32 sums
S, SA and the fp32 operands alpha = RN32(sa*sw), beta = RN32(sa*zpw), C = RN32(C64).  Against ref64,
the fp64 convolution of the exact dequantized values, each of alpha, beta and C contributes at most
one fp32 rounding of its own term (2^-24 relative), the fp64 products and sums at most a few 2^-53,
and the final rounding 2^-24 of |y| <= |alpha*S| + |beta*SA| + |C|.  So
    |y - ref64| <= (2 * 2^-24 + 2^-50) * (|alpha*S| + |beta*SA| + |C|) < 4 * 2^-24 * (...).
That is far below the fake-quant model's own fp32 convolution error, gamma_K * sum |a||w| with
gamma_K = K*u / (1 - K*u), K >= 16."""
import pytest
import torch
import torch.nn.functional as F

from mhaq_b200 import harness, ops
from mhaq_b200.quantization.gdnsq.export import build_integer_model, export_quantized
from mhaq_b200.quantization.gdnsq.inference import IntegerConv2d, IntegerLinear, unpack_weight_codes
from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
from tests.test_gpu_pack import _batches, _build

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
U = 2.0 ** -24


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _act_operands(levels, signed, seed=0):
    g = torch.Generator().manual_seed(seed)
    s = torch.tensor([2.0 ** float(torch.randint(-7, -2, (1,), generator=g))])
    b = torch.tensor([-(levels // 2) * float(s)]) if signed else torch.zeros(1)
    return s.to(DEV), b.to(DEV), (b + (levels - 1) * s).to(DEV)


def _u8_codes(fp32_codes: torch.Tensor) -> torch.Tensor:
    return torch.nan_to_num(fp32_codes, nan=0.0).clamp(0, 255).to(torch.uint8)


# ---------------------------------------------------------------------------------------------
# activation codes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [3, 12, 16, 50, 64])
@pytest.mark.parametrize("levels,signed", [(2, False), (16, True), (256, True), (256, False)])
def test_act_codes_equal_the_forward_codes(c, levels, signed):
    s, b, hi = _act_operands(levels, signed, seed=c + levels)
    x = torch.randn(3, c, 7, 9, device=DEV) * levels * float(s) / 2
    x.view(-1)[::97] = float("nan")
    x.view(-1)[5::101] = 1e30
    x = x.to(memory_format=torch.channels_last)
    codes, n_bad = ops.act_codes(x, s, b, hi)
    ref = ops.quantize_codes(x, s, b, b, hi).permute(0, 2, 3, 1)         # NHWC fp32 codes
    cp = ops.code_channels(c)
    assert codes.shape == (3, 7, 9, cp) and codes.dtype == torch.uint8
    assert torch.equal(codes[..., :c], _u8_codes(ref))
    assert not codes[..., c:].any()
    bad = int((~((ref >= 0) & (ref <= 255))).sum())
    assert bad > 0 and int(n_bad) == bad
    with pytest.raises(ValueError, match="outside"):
        ops.act_codes(x, s, b, hi, check=True)
    # a [B, in] matrix
    x2 = x.permute(0, 2, 3, 1).reshape(-1, c).contiguous()
    codes2, _ = ops.act_codes(x2, s, b, hi)
    assert torch.equal(codes2, codes.reshape(-1, cp))


@pytest.mark.parametrize("c", [16, 64])
def test_act_codes_equal_packed_8bit_codes(c):
    act = NoisyAct(signed=True).to(DEV).eval()
    with torch.no_grad():
        act.log_act_s.fill_(-5.0)
        act.log_act_q.fill_(3.0)
        act.act_b.fill_(-4.0)
    s, b, _, hi = (t.detach() for t in act._operands())
    x = torch.randn(4, c, 6, 5, device=DEV).to(memory_format=torch.channels_last) * 3
    codes, _ = ops.act_codes(x, s, b, hi)
    p = ops.pack_act_codes(x, act.log_act_s, act.log_act_q, act.act_b, bits=8, check=False)
    assert torch.equal(codes.reshape(-1), p.data.reshape(-1)[:x.numel()])


# ---------------------------------------------------------------------------------------------
# operator bar against the fp64 convolution of the exact dequantized values
# ---------------------------------------------------------------------------------------------
def _random_layer(n, c, k, w_bits, levels, per_channel, bias, signed, seed):
    """Random operands of an n x c layer with kernel ``k`` = (kh, kw) (or one int for k x k)."""
    kh, kw = (k, k) if isinstance(k, int) else k
    g = torch.Generator(device=DEV).manual_seed(seed)
    cw = torch.randint(0, 1 << w_bits, (n, c, kh, kw), generator=g, device=DEV)
    rows = n if per_channel else 1
    sw = torch.exp2(torch.randint(-10, -4, (rows,), generator=g, device=DEV).float()
                    + torch.rand(rows, generator=g, device=DEV))
    zpw = -torch.rand(rows, generator=g, device=DEV) * 0.2
    sa = float(torch.exp2(torch.tensor(-5.0) + torch.rand(1)).item())
    zpa = -(levels // 2) * sa if signed else 0.0
    b = torch.randn(n, generator=g, device=DEV) if bias else None
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, b, a_top=levels - 1, w_top=(1 << w_bits) - 1)
    return L, cw, sw, zpw, sa, zpa, b


def _check_bar(y, codes_nchw, L, cw, sw, zpw, sa, zpa, b, stride, pad):
    """|y - ref64| <= 4u (|alpha S| + |beta SA| + |C|), the terms exact (integer sums in int64).
    ``stride`` and ``pad`` are (h, w) pairs."""
    n, c, kh, kw = cw.shape
    ca = codes_nchw.double()
    a = ca * sa + zpa
    wt = cw.double() * sw.double().reshape(-1, 1, 1, 1) + zpw.double().reshape(-1, 1, 1, 1)
    ref = F.conv2d(a, wt, None if b is None else b.double(), stride=stride, padding=pad)
    s = F.conv2d(ca, cw.double(), stride=stride, padding=pad).round().long()
    sa_m = F.conv2d(ca, torch.ones(1, c, kh, kw, dtype=torch.float64, device=DEV), stride=stride,
                    padding=pad).round().long()
    h, w = codes_nchw.shape[2:]
    hc, wc, nwc, ctab = L.pattern_tables(h, w, stride, pad)
    p = hc.long()[:, None] * nwc + wc.long()[None, :]
    cterm = ctab.double()[p].permute(2, 0, 1)[None]
    terms = ((L.alpha.double().reshape(1, -1, 1, 1) * s.double()).abs()
             + (L.beta.double().reshape(1, -1, 1, 1) * sa_m.double()).abs() + cterm.abs())
    y = y.double()
    assert y.shape == ref.shape
    err = (y - ref).abs()
    ok = err <= 4 * U * terms
    assert bool(ok.all()), f"max err / bar {float((err / (4 * U * terms)).max()):.3g}"


OP_CASES = [  # (B, H, W, C, N, (kh, kw), (sh, sw), (ph, pw), w_bits, levels)
    (2, 9, 7, 3, 10, (3, 3), (1, 1), (1, 1), 4, 16),
    (3, 11, 11, 8, 16, (3, 3), (2, 2), (1, 1), 2, 4),
    (2, 16, 16, 12, 48, (3, 3), (2, 2), (0, 0), 8, 256),
    (4, 8, 8, 16, 64, (3, 3), (1, 1), (1, 1), 1, 2),
    (2, 13, 10, 50, 64, (3, 3), (1, 1), (1, 1), 4, 16),
    (1, 9, 9, 64, 512, (3, 3), (2, 2), (1, 1), 4, 3),
    (2, 5, 6, 512, 48, (3, 3), (1, 1), (1, 1), 8, 256),
    (3, 10, 10, 12, 16, (1, 1), (1, 1), (0, 0), 2, 200),
    (2, 7, 7, 16, 10, (7, 7), (2, 2), (3, 3), 4, 16),
    (2, 6, 6, 16, 511, (3, 3), (1, 1), (1, 1), 4, 16),          # 511 = 2 * 255 + 1: three weight tiles
    # per-axis geometry: every axis pair differs, so a swapped kh / kw, sh / sw or ph / pw fails
    (2, 9, 12, 16, 24, (1, 3), (1, 2), (0, 1), 4, 16),
    (2, 10, 7, 8, 20, (3, 1), (1, 1), (1, 0), 2, 4),
    (2, 13, 14, 5, 33, (5, 3), (1, 3), (0, 0), 4, 16),
    (2, 15, 9, 12, 40, (7, 3), (2, 1), (3, 0), 8, 256),
    (3, 8, 8, 16, 16, (2, 2), (1, 1), (0, 0), 4, 16),          # even kernels
    (2, 9, 10, 24, 18, (2, 4), (2, 1), (1, 2), 4, 16),
    (2, 12, 13, 16, 16, (2, 3), (3, 4), (1, 0), 4, 16),        # stride larger than the kernel
    # degenerate windows: pad >= k gives rows / columns with no valid tap (C alone)
    (2, 2, 2, 16, 12, (3, 3), (1, 1), (3, 3), 4, 16),          # image smaller than the kernel
    (2, 5, 6, 16, 20, (1, 1), (1, 1), (1, 1), 4, 16),
    (3, 1, 1, 16, 24, (3, 3), (1, 1), (4, 1), 4, 16),          # 1 x 1 image, 7 x 1 output
    (2, 11, 10, 16, 32, (1, 1), (3, 2), (0, 0), 4, 16),
    (4, 14, 14, 64, 128, (1, 1), (2, 2), (0, 0), 4, 16),       # ResNet downsample
    (3, 5, 7, 16, 40, (5, 7), (1, 1), (0, 0), 4, 16),          # kernel = image: 1 x 1 output
    (5, 1, 1, 32, 48, (1, 1), (1, 1), (0, 0), 4, 16),          # H = W = 1
]


@pytest.mark.parametrize("case", OP_CASES)
@pytest.mark.parametrize("per_channel,bias,signed", [(True, True, True), (False, False, False)])
def test_int_conv2d_operator_bar(case, per_channel, bias, signed):
    bsz, h, w, c, n, k, stride, pad, w_bits, levels = case
    seed = hash((case, per_channel)) & 0xFFFF
    L, cw, sw, zpw, sa, zpa, b = _random_layer(n, c, k, w_bits, levels, per_channel, bias, signed, seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    ca = torch.randint(0, levels, (bsz, c, h, w), generator=g, device=DEV)
    codes = torch.zeros(bsz, h, w, L.cp, dtype=torch.uint8, device=DEV)
    codes[..., :c] = ca.permute(0, 2, 3, 1).to(torch.uint8)
    y = ops.int_conv2d(codes, L, stride, pad)
    assert y.is_contiguous(memory_format=torch.channels_last)
    _check_bar(y, ca, L, cw, sw, zpw, sa, zpa, b, stride, pad)


@pytest.mark.parametrize("bsz,c,n,w_bits,levels", [(37, 16, 10, 4, 16), (300, 50, 512, 8, 256),
                                                    (129, 64, 16, 1, 2), (5, 3, 64, 2, 7),
                                                    (70, 32, 767, 4, 16), (33, 16, 255, 4, 16)])
def test_int_linear_operator_bar(bsz, c, n, w_bits, levels):
    L, cw, sw, zpw, sa, zpa, b = _random_layer(n, c, 1, w_bits, levels, True, True, True, bsz)
    ca = torch.randint(0, levels, (bsz, c), device=DEV)
    codes = torch.zeros(bsz, L.cp, dtype=torch.uint8, device=DEV)
    codes[:, :c] = ca.to(torch.uint8)
    y = ops.int_linear(codes, L)
    assert y.shape == (bsz, n)
    _check_bar(y[:, :, None, None], ca[:, :, None, None], L, cw, sw, zpw, sa, zpa, b, (1, 1), (0, 0))


def test_more_than_2p31_outputs():
    """64-bit offsets: a linear layer with M * N > 2^31 output elements, checked on sampled rows."""
    n, c = 20, 16
    m = (1 << 31) // n + 4097
    L, cw, sw, zpw, sa, zpa, b = _random_layer(n, c, 1, 4, 16, True, True, True, 5)
    codes = torch.randint(0, 16, (m, L.cp), dtype=torch.uint8, device=DEV)
    y = ops.int_linear(codes, L)
    assert y.numel() > 1 << 31
    rows = torch.cat([torch.arange(0, 3000, device=DEV), torch.arange(m - 3000, m, device=DEV),
                      torch.randint(0, m, (3000,), device=DEV)])
    ca = codes[rows, :c].long()
    _check_bar(y[rows][:, :, None, None], ca[:, :, None, None], L, cw, sw, zpw, sa, zpa, b, (1, 1), (0, 0))
    del y, codes
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# exported models
# ---------------------------------------------------------------------------------------------
MODELS = [("resnet20", "STE", False), ("resnet20", "LSQ", False), ("resnet20", "STE", True),
          ("resnet20_per_tensor", "LSQ", False), ("bias_net", "STE", False), ("asym_net", "STE", False)]


def _trained(kind, method, channels_last):
    qm = _build(kind, method)
    if channels_last:
        qm.model.to(memory_format=torch.channels_last)
    harness.fit_steps(qm, _batches(3, 1, channels_last))
    qm.eval()
    return qm


@pytest.mark.parametrize("kind,method,channels_last", MODELS)
def test_layers_match_the_fake_quant_pairs(kind, method, channels_last):
    """Each integer layer, fed the exact input its fake-quant pair received, matches the pair's eval
    output within the fp32 convolution bound gamma_K * sum|a||w| plus the integer layer's own bar."""
    qm = _trained(kind, method, channels_last)
    blob = export_quantized(qm)
    qi = build_integer_model(qm, blob)
    pairs = {n: m for n, m in qm.named_modules() if isinstance(m, torch.nn.Sequential)
             and hasattr(m, "activations_quantizer")}
    ints = dict(qi.named_modules())
    seen = {}
    hooks = [m.register_forward_hook(lambda mod, inp, out, n=n: seen.__setitem__(n, (inp[0], out)))
             for n, m in pairs.items()]
    x = _batches(1, 7, channels_last)[0][0]
    with torch.no_grad():
        qm(x)
    for h in hooks:
        h.remove()
    assert set(seen) == set(pairs) and len(pairs) > 0
    for n, (xin, yref) in seen.items():
        layer = ints[n]
        assert isinstance(layer, (IntegerConv2d, IntegerLinear))
        with torch.no_grad():
            y = layer(xin)
            act, wl = pairs[n].activations_quantizer, getattr(pairs[n], "0")
            a = act(xin).double()
            out = wl.quantized_weight() if hasattr(wl, "quantized_weight") else None
            wq = (out[0] if isinstance(out, tuple) else out).double()
            bq = blob["layers"][f"{n}.0"]["bias"]
            if isinstance(layer, IntegerConv2d):
                absum = F.conv2d(a.abs(), wq.abs(), None, layer.stride, layer.padding)
                k = wq[0].numel()
            else:
                absum = a.abs() @ wq.abs().t()
                k = wq.shape[1]
            if bq is not None:
                absum = absum + bq.to(DEV).double().abs().reshape(1, -1, *([1] * (absum.dim() - 2)))
                k += 1
            gamma = k * U / (1 - k * U)
            # the integer layer's own bar, from its codes and operands
            codes, _ = ops.act_codes(xin, layer.act_scale, layer.act_zero_point, layer.act_max_val)
            L = layer.operands
            cw = unpack_weight_codes(blob["layers"][f"{n}.0"]).to(DEV).double()
            if cw.dim() == 2:
                cw = cw[:, :, None, None]
            c = cw.shape[1]
            ca = (codes[..., :c].permute(0, 3, 1, 2) if codes.dim() == 4 else codes[:, :c, None, None]).double()
            st, pd = (layer.stride, layer.padding) if isinstance(layer, IntegerConv2d) else ((1, 1), (0, 0))
            s = F.conv2d(ca, cw, stride=st, padding=pd)
            sam = F.conv2d(ca, torch.ones_like(cw[:1]), stride=st, padding=pd)
            hc, wc, nwc, ctab = L.pattern_tables(ca.shape[2], ca.shape[3], st, pd)
            cterm = ctab.double()[hc.long()[:, None] * nwc + wc.long()[None, :]].permute(2, 0, 1)[None]
            terms = ((L.alpha.double().reshape(1, -1, 1, 1) * s).abs()
                     + (L.beta.double().reshape(1, -1, 1, 1) * sam).abs() + cterm.abs())
            if y.dim() == 2:
                terms = terms[:, :, 0, 0]
            err = (y.double() - yref.double()).abs()
            bound = gamma * absum + 4 * U * terms
            assert bool((err <= bound).all()), f"{kind} {n}: max err / bound {float((err / bound).max()):.3g}"


@pytest.mark.parametrize("kind,method,channels_last", MODELS)
def test_network_logits_agree(kind, method, channels_last):
    """Whole network: the integer model picks the fake-quant model's class for at least 90 % of a
    fixed batch of 128 samples (the largest logit difference is printed).  The two models
    may differ by more than rounding: a layer's output that differs in the last bits can move the
    next quantizer's input across a rounding boundary and flip one of its codes, so no per-sample
    bound is asserted here.  Each layer on its own is held to its bound by
    test_layers_match_the_fake_quant_pairs."""
    qm = _trained(kind, method, channels_last)
    qi = build_integer_model(qm, export_quantized(qm))
    x = torch.cat([b[0] for b in _batches(8, 11, channels_last)])
    with torch.no_grad():
        ref, got = qm(x).float(), qi(x).float()
    d = float((got - ref).abs().max())
    spread = float(ref.max(1).values.sub(ref.min(1).values).mean())
    agree = float((got.argmax(1) == ref.argmax(1)).float().mean())
    print(f"{kind}/{method}/cl={channels_last}: max |dlogit| = {d:.3e}, mean logit spread = {spread:.3e}, "
          f"argmax agreement = {agree:.3f}")
    assert agree >= 0.9


def test_graph_capture_of_the_integer_resnet20():
    qm = _trained("resnet20", "STE", False)
    qi = build_integer_model(qm, export_quantized(qm))
    x = _batches(1, 3)[0][0]
    with torch.no_grad():
        eager = qi(x)                      # builds the per-size pattern tables
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            qi(x)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = qi(x)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), eager.view(torch.int32))
    assert any(isinstance(m, IntegerConv2d) for m in qi.modules())
