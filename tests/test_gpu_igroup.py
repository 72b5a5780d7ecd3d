"""GPU: grouped, depthwise and dilated integer convolutions (mhaq_fq_iconv_grouped_u8).

Operator bar, as for the dense layer (tests/test_gpu_iconv.py): the kernels form
y = RN32(alpha*S + beta*SA[g(n)] + C) in fp64 from exact int32 sums, so against ref64, the fp64
grouped / dilated convolution of the exact dequantized values,
    |y - ref64| <= 4 * 2^-24 * (|alpha*S| + |beta*SA| + |C|).
The fused epilogue equals int_conv2d -> + r -> torch activation -> act_codes bit for bit, on both
kernels (depthwise on the CUDA cores, the rest on the tensor cores).  The torchvision models with
such layers run through build_integer_model(..., allow_groups_and_dilation=True)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from mhaq_b200 import _lib, harness, ops
from mhaq_b200.quantization.gdnsq.export import build_integer_model, export_quantized, fuse_integer_model
from mhaq_b200.quantization.gdnsq.inference import FusedIntegerConv2d, IntegerConv2d, unpack_weight_codes
from tests.test_gpu_iconv_limits import SENTINEL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
U = 2.0 ** -24


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _pair2(v):
    return (v, v) if isinstance(v, int) else tuple(v)


def _layer(n, c, groups, k, dil, w_bits, levels, seed, bias=True):
    kh, kw = _pair2(k)
    g = torch.Generator(device=DEV).manual_seed(seed)
    cw = torch.randint(0, 1 << w_bits, (n, c // groups, kh, kw), generator=g, device=DEV)
    sw = torch.exp2(torch.randint(-10, -4, (n,), generator=g, device=DEV).float() + torch.rand(n, generator=g, device=DEV))
    zpw = -torch.rand(n, generator=g, device=DEV) * 0.2
    sa = float(torch.exp2(torch.tensor(-5.0) + torch.rand(1)).item())
    zpa = -(levels // 2) * sa
    b = torch.randn(n, generator=g, device=DEV) if bias else None
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, b, a_top=levels - 1, w_top=(1 << w_bits) - 1,
                               groups=groups, dilation=dil)
    return L, cw


def _codes(bsz, h, w, c, levels, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    ca = torch.randint(0, levels, (bsz, c, h, w), generator=g, device=DEV)
    codes = torch.zeros(bsz, h, w, ops.code_channels(c), dtype=torch.uint8, device=DEV)
    codes[..., :c] = ca.permute(0, 2, 3, 1).to(torch.uint8)
    return ca, codes


def _terms(L, ca, cw, stride, pad):
    """(S, SA per output channel, C term) in fp64, exact."""
    conv = dict(stride=stride, padding=pad, dilation=L.dilation, groups=L.groups)
    s = F.conv2d(ca.double(), cw.double(), **conv)
    sam = F.conv2d(ca.double(), torch.ones_like(cw, dtype=torch.float64), **conv)
    hc, wc, nwc, ctab = L.pattern_tables(ca.shape[2], ca.shape[3], stride, pad)
    cterm = ctab.double()[hc.long()[:, None] * nwc + wc.long()[None, :]].permute(2, 0, 1)[None]
    return s, sam, cterm


def _check_bar(y, ca, L, cw, stride, pad):
    stride, pad = _pair2(stride), _pair2(pad)
    a = ca.double() * L.sa + L.zpa
    wt = cw.double() * L.sw.reshape(-1, 1, 1, 1) + L.zpw.reshape(-1, 1, 1, 1)
    ref = F.conv2d(a, wt, L.bias, stride=stride, padding=pad, dilation=L.dilation, groups=L.groups)
    s, sam, cterm = _terms(L, ca, cw, stride, pad)
    terms = ((L.alpha.double().reshape(1, -1, 1, 1) * s).abs()
             + (L.beta.double().reshape(1, -1, 1, 1) * sam).abs() + cterm.abs())
    assert y.shape == ref.shape
    err = (y.double() - ref).abs()
    assert bool((err <= 4 * U * terms).all()), f"max err / bar {float((err / (4 * U * terms)).max()):.3g}"


# ---------------------------------------------------------------------------------------------
# depthwise (CUDA cores)
# ---------------------------------------------------------------------------------------------
DW_CASES = [  # (B, H, W, C, (kh, kw), (sh, sw), (ph, pw), (dh, dw), w_bits, levels)
    pytest.param(2, *((11, 13) if c >= 144 else (19, 17)), c, (k, k), (s, s), (d * (k - 1) // 2,) * 2, (d, d), 8, 256,
                 id=f"{d}-{s}-{k}-{c}")
    for d in (1, 2, 4) for s in (1, 2) for k in (3, 5, 7) for c in (1, 17, 32, 96, 144, 960)
] + [
    # per-axis geometry: every axis pair differs, so a swapped kh / kw, sh / sw, ph / pw or dh / dw fails
    (2, 9, 11, 16, (1, 3), (1, 1), (0, 1), (1, 1), 4, 16),
    (2, 11, 8, 17, (3, 1), (2, 1), (1, 0), (1, 1), 2, 4),
    (2, 13, 12, 33, (5, 3), (1, 3), (2, 1), (1, 2), 8, 256),
    (2, 15, 19, 15, (3, 7), (1, 1), (1, 3), (3, 1), 4, 16),
    (2, 14, 9, 17, (3, 3), (2, 1), (3, 1), (1, 2), 2, 4),
    # pad >= the dilated extent on one axis: rows / columns with no valid tap (the constant term alone)
    (2, 7, 8, 16, (3, 3), (1, 1), (5, 1), (2, 1), 4, 16),
    (1, 6, 5, 33, (2, 3), (1, 2), (0, 4), (1, 1), 2, 4),
    (2, 12, 13, 17, (2, 3), (3, 4), (1, 0), (1, 1), 8, 256),     # stride larger than the kernel
    (3, 8, 8, 16, (2, 2), (1, 1), (0, 0), (1, 1), 4, 16),        # even kernels
    (2, 9, 10, 15, (4, 2), (2, 1), (1, 2), (1, 2), 2, 4),
    (2, 5, 6, 33, (1, 1), (2, 1), (1, 0), (1, 1), 8, 256),       # 1 x 1 kernel, padded rows
    (3, 1, 1, 16, (3, 3), (1, 1), (2, 2), (2, 1), 4, 16),        # 1 x 1 image, 1 x 3 output
    (2, 5, 7, 17, (3, 4), (1, 1), (0, 0), (2, 2), 4, 16),        # dilated extent = image: one output pixel
    (2, 10, 9, 1, (3, 3), (1, 2), (2, 1), (2, 1), 8, 256),       # C = N = groups = 1, dilated
    (1, 7, 6, 1, (2, 3), (2, 1), (0, 2), (1, 3), 2, 4),
]


@pytest.mark.parametrize("bsz,h,w,c,k,stride,pad,dil,w_bits,levels", DW_CASES)
def test_depthwise_operator_bar(bsz, h, w, c, k, stride, pad, dil, w_bits, levels):
    seed = hash((h, w, c, k, stride, pad, dil, w_bits)) & 0xFFFF
    L, cw = _layer(c, c, c, k, dil, w_bits, levels, seed)
    assert ops.iconv_grouped_layout(c, c, *k, c)[1] == 0            # the CUDA-core kernel
    ca, codes = _codes(bsz, h, w, c, levels, seed + 1)
    y = ops.int_conv2d(codes, L, stride, pad)
    _check_bar(y, ca, L, cw, stride, pad)


# ---------------------------------------------------------------------------------------------
# grouped and dilated (tensor cores)
# ---------------------------------------------------------------------------------------------
GCASES = [  # (B, H, W, C, N, groups, k, stride, pad, dilation, w_bits, levels)
    (2, 12, 12, 32, 64, 32, 3, 1, 1, 1, 4, 16),          # cin/g = 1: channel multiplier 2
    (2, 12, 11, 64, 64, 32, 3, 2, 1, 1, 8, 256),         # 2
    (2, 14, 14, 128, 128, 32, 3, 1, 1, 1, 4, 16),        # 4 (ResNeXt-50 layer1)
    (2, 10, 10, 256, 256, 32, 3, 1, 2, 2, 8, 256),       # 8, dilated
    (2, 9, 9, 512, 512, 32, 3, 2, 1, 1, 4, 16),          # 16
    (1, 7, 7, 1024, 1024, 32, 3, 1, 1, 1, 8, 256),       # 32 (ResNeXt-50 layer4)
    (2, 8, 8, 96, 96, 2, (3, 1), 1, (1, 0), 1, 8, 256),  # 48
    (2, 8, 8, 16, 600, 2, 3, 1, 1, 1, 4, 16),            # a group wider than a tile (300 channels)
    (2, 6, 7, 24, 680, 8, 3, 1, 1, 2, 4, 16),            # 3 per group: groups straddle 16-channel chunks
    (2, 16, 16, 8, 24, 1, 3, 1, 4, 4, 8, 256),           # dilated, groups = 1
    (3, 13, 17, 48, 48, 3, (5, 3), (2, 1), (2, 1), (2, 3), 4, 16),    # per-axis geometry
    (1, 1, 1, 64, 64, 4, 3, 1, 2, 2, 4, 16),             # M = 1, no tap but the centre valid
    (1, 3, 43, 64, 32, 2, 3, 1, 1, 1, 4, 16),            # M = 129: a second, one-row M tile
    (1, 6, 6, 512, 64, 2, 3, 1, 1, 1, 2, 4),             # 18 pipeline stages
    (2, 5, 5, 40, 80, 5, (1, 1), 1, 0, 1, 8, 256),       # K = 1 chunk: a zero-filled stage
]


@pytest.mark.parametrize("case", GCASES)
def test_grouped_operator_bar(case):
    bsz, h, w, c, n, groups, k, stride, pad, dil, w_bits, levels = case
    seed = hash(case) & 0xFFFF
    L, cw = _layer(n, c, groups, k, dil, w_bits, levels, seed)
    ca, codes = _codes(bsz, h, w, c, levels, seed + 1)
    y = ops.int_conv2d(codes, L, stride, pad)
    _check_bar(y, ca, L, cw, stride, pad)


# ---------------------------------------------------------------------------------------------
# the fused epilogue, bit for bit against the composition
# ---------------------------------------------------------------------------------------------
FCASES = [  # (B, H, W, C, N, groups, k, stride, pad, dilation)
    (2, 9, 10, 40, 40, 40, 3, 1, 2, 2),                  # depthwise, C % 16 != 0
    (2, 8, 8, 144, 144, 144, 5, 2, 2, 1),                # depthwise
    (2, 9, 9, 64, 64, 16, 3, 1, 1, 1),                   # grouped
    (2, 11, 9, 24, 52, 4, 3, 2, 2, 2),                   # grouped, dilated, N % 16 != 0
    (2, 9, 11, 33, 33, 33, (1, 3), (2, 1), (1, 0), (2, 1)),           # depthwise, per-axis geometry
    (2, 10, 8, 16, 16, 16, (3, 2), (1, 2), (2, 1), (1, 3)),
    (1, 7, 9, 20, 20, 20, (5, 3), (1, 1), (3, 1), (1, 2)),            # pad >= the dilated extent on H
]
NEXT = [(2, False), (16, True), (256, True), (256, False)]


def _act_operands(levels, signed, seed):
    g = torch.Generator().manual_seed(seed)
    s = torch.tensor([2.0 ** float(torch.randint(-7, -2, (1,), generator=g))])
    b = torch.tensor([-(levels // 2) * float(s)]) if signed else torch.zeros(1)
    return s.to(DEV), b.to(DEV), (b + (levels - 1) * s).to(DEV)


def _i32(t):
    return t.contiguous(memory_format=torch.channels_last).view(torch.int32)


@pytest.mark.parametrize("ci", range(len(FCASES)))
@pytest.mark.parametrize("residual", [False, True])
@pytest.mark.parametrize("activation", [None, "relu", "leaky_relu"])
@pytest.mark.parametrize("outputs", ["fp32", "codes", "both"])
def test_epilogue_equals_composition(ci, residual, activation, outputs):
    bsz, h, w, c, n, groups, k, stride, pad, dil = FCASES[ci]
    seed = 2000 + ci
    L, _ = _layer(n, c, groups, k, dil, 4, 16, seed)
    g = torch.Generator(device=DEV).manual_seed(seed)
    bn = torch.nn.BatchNorm2d(n).to(DEV).eval()
    with torch.no_grad():
        bn.weight.copy_(torch.randn(n, generator=g, device=DEV))
        bn.running_var.copy_(torch.rand(n, generator=g, device=DEV) + 0.5)
        bn.running_mean.copy_(torch.randn(n, generator=g, device=DEV))
    L = ops.fold_batchnorm(L, bn)
    _, codes = _codes(bsz, h, w, c, 16, seed + 1)
    _check_epilogue(L, codes, stride, pad, residual, activation, outputs, NEXT[ci % len(NEXT)], ci)


def _check_epilogue(L, codes, stride, pad, residual, activation, outputs, next_act, seed):
    """The fused launch equals int_conv2d -> + r -> torch activation -> act_codes bit for bit; the
    residual has exact zeros, rounding ties of the next quantizer and NaNs planted in it."""
    bsz = codes.shape[0]
    n = L.n_out
    g = torch.Generator(device=DEV).manual_seed(seed)
    plain = ops.int_conv2d(codes, L, stride, pad)
    levels_n, signed = next_act
    s, b, hi = _act_operands(levels_n, signed, seed)
    r = None
    if residual:
        r = torch.randn(plain.shape, generator=g, device=DEV) * levels_n * float(s) / 4
        flat, pv = r.view(-1), plain.contiguous().view(-1)
        flat[0::7] = -pv[0::7]
        tie = b + (torch.randint(0, levels_n, pv.shape, generator=g, device=DEV) + 0.5) * s
        flat[3::7] = (tie - pv)[3::7]
        flat[5::97] = float("nan")
        r = r.contiguous()
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
        assert torch.equal(_i32(y), _i32(ref))
    if want_c:
        assert torch.equal(cod, ops.act_codes(ref, s, b, hi)[0])


# ---------------------------------------------------------------------------------------------
# nothing written outside the outputs; 64-bit offsets
# ---------------------------------------------------------------------------------------------
def _grouped_launch(codes, L, weight, stride, pad, y, out_codes, residual=None, activation=None, code_params=None):
    """mhaq_fq_iconv_grouped_u8 on L's alpha, beta and pattern tables with the weight operand
    ``weight``, writing through the raw pointers of ``y`` / ``out_codes`` (either may be None)."""
    bsz, h, w, _ = codes.shape
    stride, pad = _pair2(stride), _pair2(pad)
    hc, wc, nwc, ctab = L.pattern_tables(h, w, stride, pad)
    prm = [p.contiguous() for p in code_params] if code_params is not None else [None] * 3
    ptr = lambda t: None if t is None else t.data_ptr()       # noqa: E731
    geo = _lib.IConvGeometry(L.kh, L.kw, *stride, *pad, *L.dilation, L.groups)
    epi = _lib.IConvEpilogue(ptr(residual), ops.ACTIVATIONS[activation], 0.125, ptr(y), ptr(out_codes),
                             *(ptr(p) for p in prm))
    rc = _lib.lib.mhaq_fq_iconv_grouped_u8(codes.data_ptr(), weight.data_ptr(), L.alpha.data_ptr(),
                                           L.beta.data_ptr(), ctab.data_ptr(), hc.data_ptr(), wc.data_ptr(), nwc,
                                           bsz, h, w, L.cin, L.n_out, ctypes.byref(geo), L.a_top, L.w_top,
                                           ctypes.byref(epi), torch.cuda.current_stream().cuda_stream)
    assert rc == 0


# the 3-part row of tests/test_gpu_igroup_limits.py: tiles at n_base 0, 171, 342 (not multiples of 4 or 16)
THREE_PARTS = (2, 6, 5, 2, 1022, 2, 3, 1, 1, 1)


@pytest.mark.parametrize("y_offset", [4, 1, 3])
@pytest.mark.parametrize("case", [FCASES[0], FCASES[3], THREE_PARTS])
def test_stores_stay_inside_the_outputs(case, y_offset):
    """y at ``y_offset`` floats into a buffer of SENTINEL words (offset 4 is 16-byte aligned: the
    float4 stores where N % 4 == 0; 1 and 3 the scalar ones), the residual one float off a 16-byte
    boundary (the scalar loads), the codes in a 16-byte-aligned view of a 0xAB buffer.  Every word
    outside the outputs keeps its fill; y and the codes equal the fresh-tensor result bit for bit."""
    bsz, h, w, c, n, groups, k, stride, pad, dil = case
    L, _ = _layer(n, c, groups, k, dil, 4, 16, 7)
    _, codes = _codes(bsz, h, w, c, 16, 8)
    prm = _act_operands(16, True, 1)
    ho, wo = L.out_size(h, w, _pair2(stride), _pair2(pad))
    m, cp_out = bsz * ho * wo, ops.code_channels(n)
    rb = torch.randn(m * n + 1, generator=torch.Generator(device=DEV).manual_seed(9), device=DEV)
    r = rb[1:].view(bsz, ho, wo, n).permute(0, 3, 1, 2)
    assert r.data_ptr() % 16 == 4
    ref, ref_codes = ops.int_conv2d_fused(codes, L, stride, pad, residual=r.contiguous(), activation="relu",
                                          code_params=prm)
    yb = torch.full((m * n + 2 * 64,), SENTINEL, dtype=torch.int32, device=DEV)
    cb = torch.full((m * cp_out + 2 * 64,), 0xAB, dtype=torch.uint8, device=DEV)
    lo = y_offset
    _grouped_launch(codes, L, L.weight, stride, pad, yb.view(torch.float32)[lo:], cb[64:], r, "relu", prm)
    torch.cuda.synchronize()
    assert bool((yb[:lo] == SENTINEL).all()) and bool((yb[lo + m * n:] == SENTINEL).all())
    assert bool((cb[:64] == 0xAB).all()) and bool((cb[64 + m * cp_out:] == 0xAB).all())
    assert torch.equal(yb[lo:lo + m * n], _i32(ref).permute(0, 2, 3, 1).reshape(-1))
    assert torch.equal(cb[64:64 + m * cp_out], ref_codes.reshape(-1))


@pytest.mark.parametrize("c,n,groups", [(16, 16, 16), (32, 32, 16)])
def test_more_than_2p31_outputs(c, n, groups):
    """One image repeated over a batch with M * N > 2^31 output elements: every image's output
    equals the single image's, checked on the first, last and sampled images."""
    h = w = 256
    bsz = (1 << 31) // (h * w * n) + 2
    L, cw = _layer(n, c, groups, 3, 1, 4, 16, 11)
    ca, one = _codes(1, h, w, c, 16, 12)
    want = ops.int_conv2d(one, L, 1, 1)
    _check_bar(want, ca, L, cw, 1, 1)
    codes = one.expand(bsz, -1, -1, -1).contiguous()
    y = ops.int_conv2d(codes, L, 1, 1)
    assert y.numel() > 1 << 31
    del codes
    for i in [0, 1, bsz // 2, bsz - 2, bsz - 1] + torch.randint(0, bsz, (4,)).tolist():
        assert torch.equal(_i32(y[i:i + 1]), _i32(want)), i
    del y
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# torchvision models
# ---------------------------------------------------------------------------------------------
TV = ["mobilenet_v2", "resnext50_32x4d", "resnet50_dilated"]
# whole-network agreement needs a reference that depends on the input; the MobileNetV2 test model's
# signal dies by features.12 (every input of that layer is 0, so recalibration cannot help), so
# its logits are constant and only its per-layer and operator tests apply
TV_NET = ["resnext50_32x4d", "resnet50_dilated"]
RES = 64


def _batches(n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [(torch.randn(16, 3, RES, RES, generator=g, device=DEV).to(memory_format=torch.channels_last),
             torch.randint(0, 10, (16,), generator=g, device=DEV)) for _ in range(n)]


@pytest.fixture(scope="module")
def tv_models():
    """Each model calibrated at 4 bits and trained for three steps, in eval mode, channels_last."""
    out = {}
    # trained in fp32 as the tests run (a module fixture is set up before _no_tf32), so that the
    # models, and whether their references depend on the input, do not change with TF32 rounding
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    for name in TV:
        torch.manual_seed(0)
        qm = harness.build_qat(name, qnmethod="STE", distillation=False, num_classes=10,
                               calib_batch=_batches(1, 1)[0][0], calib_bits=4)
        qm.model.to(memory_format=torch.channels_last)
        if name == "resnext50_32x4d":
            # BatchNorm statistics averaged over the training batches (after three steps at the
            # default momentum they are still mostly (0, 1)); otherwise the model picks one class
            # for every input
            for bn in qm.model.modules():
                if isinstance(bn, torch.nn.BatchNorm2d):
                    bn.momentum = None
        harness.fit_steps(qm, _batches(3, 2))
        if name == "resnext50_32x4d":
            # and activation ranges of the trained network, not of the untrained one
            harness.calibrate(qm, _batches(1, 1)[0][0], act_bits=4, weight_bits=0)
        qm.eval()
        blob = export_quantized(qm)
        out[name] = (qm, blob, build_integer_model(qm, blob, allow_groups_and_dilation=True))
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    return out


@pytest.mark.parametrize("name", TV)
def test_layers_match_the_fake_quant_pairs(tv_models, name):
    """Each integer layer, fed its fake-quant pair's input, is within the fp32 convolution bound
    gamma_K * sum|a||w| (K = kh * kw * cin / groups + bias) plus its own operator bar."""
    qm, blob, qi = tv_models[name]
    pairs = {n: m for n, m in qm.named_modules() if isinstance(m, torch.nn.Sequential)
             and hasattr(m, "activations_quantizer")}
    ints = dict(qi.named_modules())
    seen = {}
    hooks = [m.register_forward_hook(lambda mod, inp, out, n=n: seen.__setitem__(n, (inp[0], out)))
             for n, m in pairs.items()]
    with torch.no_grad():
        qm(_batches(1, 7)[0][0])
    for hk in hooks:
        hk.remove()
    assert set(seen) == set(pairs) and len(pairs) >= 16
    worst = 0.0
    for n, (xin, yref) in seen.items():
        layer = ints[n]
        assert isinstance(layer, IntegerConv2d)
        L = layer.operands
        conv = dict(stride=layer.stride, padding=layer.padding, dilation=L.dilation, groups=L.groups)
        with torch.no_grad():
            y = layer(xin)
            act, wl = pairs[n].activations_quantizer, getattr(pairs[n], "0")
            a = act(xin).double()
            out = wl.quantized_weight()
            wq = (out[0] if isinstance(out, tuple) else out).double()
            absum = F.conv2d(a.abs(), wq.abs(), None, **conv)
            kk = wq[0].numel()
            bq = blob["layers"][f"{n}.0"]["bias"]
            if bq is not None:
                absum = absum + bq.to(DEV).double().abs().reshape(1, -1, 1, 1)
                kk += 1
            gamma = kk * U / (1 - kk * U)
            codes, _ = ops.act_codes(xin, layer.act_scale, layer.act_zero_point, layer.act_max_val)
            cw = unpack_weight_codes(blob["layers"][f"{n}.0"]).to(DEV)
            ca = codes[..., :L.cin].permute(0, 3, 1, 2)
            s, sam, cterm = _terms(L, ca, cw, layer.stride, layer.padding)
            terms = ((L.alpha.double().reshape(1, -1, 1, 1) * s).abs()
                     + (L.beta.double().reshape(1, -1, 1, 1) * sam).abs() + cterm.abs())
            err = (y.double() - yref.double()).abs()
            bound = gamma * absum + 4 * U * terms
            worst = max(worst, float((err / bound).max()))
            assert bool((err <= bound).all()), f"{name} {n}: max err / bound {float((err / bound).max()):.3g}"
    print(f"{name}: {len(seen)} layers, worst err / bound {worst:.3g}")


@pytest.mark.parametrize("name", TV_NET)
def test_network_agrees(tv_models, name):
    """Whole network, plain and fused: the integer model picks the fake-quant model's class for at
    least 90 % of 128 samples (the threshold of the dense models' tests)."""
    qm, _, qi = tv_models[name]
    gm = fuse_integer_model(qi)
    assert any(isinstance(m, FusedIntegerConv2d) for m in gm.modules())
    x = torch.cat([b[0] for b in _batches(8, 11)])
    with torch.no_grad():
        ref, got, fused = qm(x).float(), qi(x).float(), gm(x).float()
    # a reference whose logits ignore the input would make the agreement below meaningless
    assert len(set(ref.argmax(1).tolist())) >= 2, f"{name}: the fake-quant model predicts one class"
    assert bool((ref[1:] != ref[:1]).any(1).all()), f"{name}: the fake-quant logits do not depend on the input"
    for what, t in (("integer", got), ("fused", fused)):
        agree = float((t.argmax(1) == ref.argmax(1)).float().mean())
        print(f"{name} {what}: max |dlogit| = {float((t - ref).abs().max()):.3e}, argmax agreement = {agree:.3f}")
        assert agree >= 0.9, (name, what)


def test_graph_capture_of_the_fused_resnext50(tv_models):
    """Replay with a new input equals the eager forward of that input (and differs from the old)."""
    _, _, qi = tv_models["resnext50_32x4d"]
    gm = fuse_integer_model(qi)
    x = _batches(1, 3)[0][0]
    with torch.no_grad():
        eager = gm(x)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            gm(x)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = gm(x)
        x.copy_(_batches(1, 4)[0][0])
        g.replay()
        torch.cuda.synchronize()
        want = gm(x)
    assert torch.equal(out.view(torch.int32), want.view(torch.int32))
    assert not torch.equal(out.view(torch.int32), eager.view(torch.int32))


def test_graph_capture_of_depthwise_then_grouped():
    """A depthwise int_conv2d_fused (CUDA cores) feeding its codes to a grouped one (tensor cores),
    codes out, captured in a CUDA graph: replay with new input codes equals the eager run of those
    codes bit for bit and differs from the old output."""
    dw, _ = _layer(48, 48, 48, (3, 5), (2, 1), 4, 16, 31)
    gr, _ = _layer(80, 48, 16, 3, 1, 4, 16, 32)
    prm = _act_operands(16, True, 3)

    def run(codes):
        _, mid = ops.int_conv2d_fused(codes, dw, 1, (2, 2), activation="relu", out_fp32=False, code_params=prm)
        return ops.int_conv2d_fused(mid, gr, (2, 1), 1, activation="leaky_relu", negative_slope=0.125,
                                    code_params=prm)

    _, codes = _codes(2, 12, 10, 48, 16, 33)
    _, new_codes = _codes(2, 12, 10, 48, 16, 34)
    eager = run(codes)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(codes)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = run(codes)
    codes.copy_(new_codes)
    g.replay()
    torch.cuda.synchronize()
    want = run(new_codes)
    assert torch.equal(_i32(out[0]), _i32(want[0])) and torch.equal(out[1], want[1])
    assert not torch.equal(out[1], eager[1])
