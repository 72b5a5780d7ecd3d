"""GPU: packed integer codes (include/mhaq_fq.h "Packed codes", ops.pack_codes / unpack_codes) and
the model export built on them (quantization/gdnsq/export.py).

Every packed byte is compared with a reference packer applied to the forward's own fp32 codes,
every unpacked value with the forward's output (value and bit pattern), and every saturation
count with the count torch derives from those codes."""
import io
import zlib

import numpy as np
import pytest
import torch
from torch import nn

from mhaq_b200 import harness, ops
from mhaq_b200.ops import _Launch, _dense, _forward_impl, _pack
from mhaq_b200.quantization.gdnsq.export import export_quantized, load_quantized
from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
from mhaq_b200.quantization.gdnsq.layers.gdnsq_linear import NoisyLinear
from mhaq_b200.quantization.gdnsq.utils import model_stats
from mhaq_b200.quantization.quantizer import Quantizer
from tests import pack_ref as R

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


# ---------------------------------------------------------------------------------------------
# reference packer (the format of tests/pack_ref.py, vectorised with torch for large tensors)
# ---------------------------------------------------------------------------------------------
def torch_pack(codes: torch.Tensor, bits: int) -> torch.Tensor:
    """uint codes [n_rows, n_inner] (int64, each < 2^bits) -> uint8 [n_rows, row_bytes]."""
    n_rows, n = codes.shape
    out = torch.zeros(n_rows, R.row_bytes(n, bits), dtype=torch.uint8, device=codes.device)
    if bits == 16:
        out[:, :2 * n] = torch.stack([codes & 0xFF, codes >> 8], -1).reshape(n_rows, 2 * n).to(torch.uint8)
        return out
    per = 8 // bits
    nb = (n * bits + 7) // 8
    cp = torch.zeros(n_rows, nb * per, dtype=torch.int64, device=codes.device)
    cp[:, :n] = codes
    shifts = torch.arange(per, device=codes.device) * bits
    out[:, :nb] = (cp.view(n_rows, nb, per) << shifts).sum(-1).to(torch.uint8)
    return out


def storage_rows(t: torch.Tensor, n_rows: int) -> torch.Tensor:
    """[n_rows, n_inner] view of a dense tensor in storage order."""
    return torch.as_strided(t, (t.numel(),), (1,)).view(n_rows, -1)


def expected(codes: torch.Tensor, bits: int, n_rows: int):
    """(packed bytes, in-range mask in storage order, #out of range) from the forward's fp32 codes."""
    c = storage_rows(codes, n_rows)
    top = (1 << bits) - 1
    ok = (c >= 0) & (c <= top)
    sat = torch.nan_to_num(c, nan=0.0).clamp(0, top).to(torch.int64)
    return torch_pack(sat, bits), ok, int((~ok).sum())


def bits_of(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("n_inner", [1, 3, 5, 8, 33, 4095, 4097])
@pytest.mark.parametrize("bits", R.WIDTHS)
def test_torch_packer_matches_numpy_packer(bits, n_inner):
    rng = np.random.default_rng(n_inner * 31 + bits)
    codes = rng.integers(0, 1 << bits, size=(3, n_inner), dtype=np.int64)
    got = torch_pack(torch.from_numpy(codes).to(DEV), bits).cpu().numpy()
    assert np.array_equal(got, R.pack(codes, bits))


# ---------------------------------------------------------------------------------------------
# round trip: every width, every parameter mode, clamped and unclamped, many layouts
# ---------------------------------------------------------------------------------------------
def _shape_cases():
    return {
        "tiny": None,                                   # 1-D tensors of 1..5 elements (looped)
        "ragged4097": lambda g: torch.randn(4097, generator=g, device=DEV) * 3,
        "rows4096x256": lambda g: torch.randn(4096, 256, generator=g, device=DEV) * 3,
        "rows512x2p19": lambda g: torch.randn(512, 1 << 19, generator=g, device=DEV) * 3,
        "channels_last": lambda g: (torch.randn(32, 16, 6, 6, generator=g, device=DEV) * 3).to(
            memory_format=torch.channels_last),
        "misaligned": lambda g: (torch.randn(10001, generator=g, device=DEV) * 3)[1:],   # 4-byte offset
        "per_tensor2p26": lambda g: torch.randn(1 << 26, generator=g, device=DEV) * 3,
    }


MODES = ("linear", "linear_clamp", "act_log", "weight_log", "unit")


def _launch(mode, x, bits, g):
    """(launch description, public packing call or None, fake_quant call or None) for `mode`."""
    top = (1 << bits) - 1
    per_channel = x.dim() >= 2
    if mode in ("linear", "linear_clamp"):
        if per_channel:
            pshape = (x.shape[0],) + (1,) * (x.dim() - 1)
            s = (6.0 / top) * (1 + 0.1 * torch.rand(pshape, generator=g, device=DEV))
        else:
            s = torch.full((1,), 6.0 / top, device=DEV)
        zp = torch.full_like(s, -3.0)
        lo, hi = (zp, zp + top * s) if mode == "linear_clamp" else (None, None)
        return (_Launch(x, s, zp, lo, hi), lambda b, c: ops.pack_codes(x, s, zp, lo, hi, bits=b, check=c),
                lambda: ops.fake_quant(x, s, zp, lo, hi))
    if mode == "act_log":
        las = torch.tensor([-3.3], device=DEV)
        laq = las + bits
        ab = torch.tensor([-2.7], device=DEV)
        return (_Launch.act_log(x, las, laq, ab),
                lambda b, c: ops.pack_act_codes(x, las, laq, ab, bits=b, check=c), None)
    if mode == "weight_log":
        rows = x.shape[0]
        ls = -2.0 - bits * 0.5 - torch.rand(rows, generator=g, device=DEV)
        mn = x.reshape(rows, -1).amin(1)
        return (_Launch.weight_log(x, ls, mn), lambda b, c: ops.pack_weight_codes(x, ls, mn, bits=b, check=c),
                None)
    scale = torch.ones((x.shape[0],) + (1,) * (x.dim() - 1) if per_channel else (1,), device=DEV)
    return _Launch.unit(x, scale), None, None


def _check_round_trip(x, mode, bits, g):
    L, public, fake_quant = _launch(mode, x, bits, g)
    xd = _dense(x, L.geo.axis)
    y, codes, _ = _forward_impl(xd, L, True, True, False)
    want, ok, n_bad = expected(codes, bits, L.geo.n_rows)
    p = _pack(xd, L, bits, False)
    assert p.data.shape == want.shape
    assert torch.equal(p.data, want), f"{mode} b={bits}: packed bytes differ"
    assert int(p.n_out_of_range.item()) == n_bad
    if public is not None:
        assert torch.equal(public(bits, False).data, want)
        if n_bad:
            with pytest.raises(ValueError, match="outside"):
                public(bits, True)
        else:
            public(bits, True)
    u = ops.unpack_codes(p)
    assert u.shape == x.shape and u.stride() == xd.stride()
    uy, yy = storage_rows(u, L.geo.n_rows), storage_rows(y, L.geo.n_rows)
    assert torch.equal(bits_of(uy[ok]), bits_of(yy[ok])), f"{mode} b={bits}: unpacked values differ"
    if fake_quant is not None:          # the public operator's forward, in the packed tensor's layout
        fq = _dense(fake_quant(), L.geo.axis)
        assert torch.equal(bits_of(storage_rows(fq, L.geo.n_rows)[ok]), bits_of(uy[ok]))


@pytest.mark.parametrize("bits", R.WIDTHS)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", list(_shape_cases()))
def test_round_trip(shape, mode, bits):
    g = torch.Generator(device=DEV).manual_seed(zlib.crc32(f"{shape}/{mode}/{bits}".encode()))
    make = _shape_cases()[shape]
    if make is None:
        xs = [torch.randn(n, generator=g, device=DEV) * 3 for n in range(1, 6)]
    else:
        x = make(g)
        if x.numel() > 100:               # NaN inputs give NaN codes: stored as 0 and counted
            flat = torch.as_strided(x, (x.numel(),), (1,))
            flat[torch.randint(0, x.numel(), (7,), generator=g, device=DEV)] = float("nan")
        xs = [x]
    for x in xs:
        _check_round_trip(x, mode, bits, g)


def test_zero_code_with_negative_zero_point():
    """v in (-0.5, 0] gives the code +0 in the forward (v + (rint(v) - v) rounds to +0), so with a
    zero point of -0.0 the forward's output and the unpacked value are both +0."""
    s = torch.tensor([0.25], device=DEV)
    zp = torch.tensor([-0.0], device=DEV)
    x = torch.tensor([-0.1, -0.03, -0.0, 0.0, -1e-30, 0.05] * 700, device=DEV)
    for xx in (x, x[1:]):                   # fast and general paths
        y = ops.fake_quant(xx, s, zp)
        u = ops.unpack_codes(ops.pack_codes(xx, s, zp, bits=4))
        assert torch.equal(bits_of(u), bits_of(y))
        assert not torch.signbit(u).any()


# ---------------------------------------------------------------------------------------------
# automatic width, int64 addressing, graph capture
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("top", [0, 1, 2, 3, 4, 15, 16, 200, 255, 256, 65535])
def test_auto_width_is_the_smallest(top):
    x = torch.linspace(0, float(top), 5000, device=DEV)
    p = ops.pack_codes(x, torch.ones(1, device=DEV), torch.zeros(1, device=DEV))
    want = next(b for b in R.WIDTHS if top <= (1 << b) - 1)
    assert p.bits == want
    assert torch.equal(ops.unpack_codes(p), torch.round(x))


def test_auto_width_raises_when_nothing_fits():
    one, zero = torch.ones(1, device=DEV), torch.zeros(1, device=DEV)
    with pytest.raises(ValueError, match="no unsigned width"):
        ops.pack_codes(torch.tensor([-2.0, 3.0], device=DEV), one, zero)
    with pytest.raises(ValueError, match="16 bits"):
        ops.pack_codes(torch.tensor([0.0, 70000.0], device=DEV), one, zero)
    with pytest.raises(ValueError, match="no unsigned width"):
        ops.pack_codes(torch.tensor([0.0, float("nan")], device=DEV), one, zero)


def test_beyond_2p31_elements_one_bit():
    n = (1 << 31) + 3 * 4096 + 4         # vector path, with a ragged last sub-tile
    g = torch.Generator(device=DEV).manual_seed(3)
    xb = torch.randint(0, 2, (n,), dtype=torch.uint8, generator=g, device=DEV)
    x = xb.float()
    one, zero = torch.ones(1, device=DEV), torch.zeros(1, device=DEV)
    p = ops.pack_codes(x, one, zero, zero, one, bits=1)
    assert p.data.shape == (1, R.row_bytes(n, 1)) and int(p.n_out_of_range.item()) == 0
    chunk = 1 << 28                                   # codes per reference chunk (multiple of 8)
    for c0 in range(0, n, chunk):
        c = xb[c0:c0 + chunk].to(torch.int64).view(1, -1)
        want = torch_pack(c, 1)[0, :(c.numel() + 7) // 8]
        assert torch.equal(p.data[0, c0 // 8:c0 // 8 + want.numel()], want), f"chunk at {c0}"
    assert not p.data[0, (n + 7) // 8:].any()
    del want, c
    u = ops.unpack_codes(p)
    assert torch.equal(u, x)


def test_graph_capture_pack_and_unpack():
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn(64, 4096 + 12, generator=g, device=DEV)
    s = torch.full((64, 1), 0.5, device=DEV)
    zp = torch.full((64, 1), -4.0, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up outside the capture
        ops.unpack_codes(ops.pack_codes(x, s, zp, zp, zp + 15 * s, bits=4, check=False))
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        p = ops.pack_codes(x, s, zp, zp, zp + 15 * s, bits=4, check=False)
        u = ops.unpack_codes(p)
    for seed in (11, 12):
        x.copy_(torch.randn(x.shape, generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV))
        graph.replay()
        torch.cuda.synchronize()
        eager = ops.pack_codes(x, s, zp, zp, zp + 15 * s, bits=4)
        assert torch.equal(p.data, eager.data)
        assert torch.equal(u, ops.unpack_codes(eager))
        first = p.data.clone()
        graph.replay()
        assert torch.equal(p.data, first)


# ---------------------------------------------------------------------------------------------
# model export / load
# ---------------------------------------------------------------------------------------------
def _batches(n, seed, channels_last=False):
    g = torch.Generator(device=DEV).manual_seed(seed)
    out = []
    for _ in range(n):
        x = torch.randn(16, 3, 32, 32, generator=g, device=DEV)
        if channels_last:
            x = x.to(memory_format=torch.channels_last)
        out.append((x, torch.randint(0, 10, (16,), generator=g, device=DEV)))
    return out


class _BiasNet(nn.Module):
    """Small classifier whose convolutions carry a bias, with a quantized Linear head."""

    def __init__(self):
        super().__init__()
        self.c1 = nn.Conv2d(3, 8, 3, padding=1)
        self.c2 = nn.Conv2d(8, 16, 3, stride=2, padding=1)
        self.fc = nn.Linear(16, 10)

    def forward(self, x):
        x = torch.relu(self.c2(torch.relu(self.c1(x))))
        return self.fc(torch.nn.functional.adaptive_avg_pool2d(x, 1).flatten(1))


class _AsymNet(nn.Module):
    """Classifier with per-axis convolution geometry: a (1, 3) stride-(1, 2) conv, a (3, 1) conv ->
    BN -> ReLU, a residual block whose shortcut is a 1x1 stride-2 conv (which the quantizer leaves in
    fp32, as ResNet-18's downsample), a 3x3 pad-2 conv on a 4 x 4 map (border outputs with a single
    valid tap row) and a 1000-way Linear head.  Every quantized convolution carries a bias: with
    quantize_bias the bias quantizer needs one (as in the reference's NoisyConv2d), and the BatchNorm
    fold takes it into C."""

    def __init__(self):
        super().__init__()
        self.c1 = nn.Conv2d(3, 16, (1, 3), stride=(1, 2), padding=(0, 1))
        self.c2 = nn.Conv2d(16, 16, (3, 1), padding=(1, 0))
        self.bn2 = nn.BatchNorm2d(16)
        self.b1 = nn.Conv2d(16, 32, 3, stride=2, padding=1)
        self.bn_b1 = nn.BatchNorm2d(32)
        self.b2 = nn.Conv2d(32, 32, 3, padding=1)
        self.bn_b2 = nn.BatchNorm2d(32)
        self.downsample = nn.Sequential(nn.Conv2d(16, 32, 1, stride=2, bias=False), nn.BatchNorm2d(32))
        self.c3 = nn.Conv2d(32, 32, 3, padding=2)
        self.fc = nn.Linear(32, 1000)

    def forward(self, x):
        x = torch.relu(self.c1(x))                                   # 32 x 16
        x = torch.relu(self.bn2(self.c2(x)))
        y = torch.relu(self.bn_b1(self.b1(x)))                       # 16 x 8
        x = torch.relu(self.bn_b2(self.b2(y)) + self.downsample(x))
        x = torch.nn.functional.avg_pool2d(x, (4, 2))                # 4 x 4
        x = torch.relu(self.c3(x))                                   # 6 x 6
        return self.fc(torch.nn.functional.adaptive_avg_pool2d(x, 1).flatten(1))


def _build(kind, method, channels_last=False, calib=True):
    torch.manual_seed(0)
    if kind == "resnet20":
        return harness.build_qat("resnet20", qnmethod=method, act_bit=4, weight_bit=4, distillation=False,
                                 calib_batch=_batches(1, 99)[0][0] if calib else None, calib_bits=4)
    if kind == "resnet20_per_tensor":
        model, excl, qb = harness.build_model("resnet20"), harness.EXCLUDED["resnet20"], False
        qscheme = 0
    else:
        model, excl, qb, qscheme = (_AsymNet() if kind == "asym_net" else _BiasNet()), (), True, 1
    lm = harness.LModule(model.to(DEV), nn.CrossEntropyLoss())
    cfg = harness.make_config(act_bit=4, weight_bit=4, qscheme=qscheme, qnmethod=method,
                              excluded_layers=excl, quantize_bias=qb)
    qm = Quantizer(cfg)().quantize(lm, in_place=True).to(DEV)
    if calib:
        # per-tensor weight scales by hand: the calibration's quantile rule is written per channel
        harness.calibrate(qm, _batches(1, 99)[0][0], act_bits=4, weight_bits=4 if qscheme else 0)
        if not qscheme:
            with torch.no_grad():
                for m in _weight_layers(qm).values():
                    w = m.weight.detach()
                    m.log_wght_s.fill_(float(torch.log2((w.amax() - w.amin()) / 15)))
    return qm


def _weight_layers(qm):
    return {n: m for n, m in qm.named_modules() if isinstance(m, (NoisyConv2d, NoisyLinear))}


@pytest.mark.parametrize("kind,method,channels_last", [
    ("resnet20", "STE", False),
    ("resnet20", "LSQ", False),
    ("resnet20", "STE", True),
    ("resnet20_per_tensor", "LSQ", False),
    ("bias_net", "STE", False),
])
def test_model_export_round_trip(kind, method, channels_last):
    qm = _build(kind, method)
    if channels_last:
        qm.model.to(memory_format=torch.channels_last)
    harness.fit_steps(qm, _batches(3, 1, channels_last))
    xfix = _batches(1, 7, channels_last)[0][0]
    qm.eval()
    with torch.no_grad():
        out_ref = qm(xfix)
    blob = export_quantized(qm)
    buf = io.BytesIO()
    torch.save(blob, buf)
    buf.seek(0)
    blob = torch.load(buf, weights_only=True)
    assert blob["format"] == "mhaq-packed" and blob["version"] == 1

    layers = _weight_layers(qm)
    assert set(layers) <= set(blob["layers"])
    packed = ideal = 0
    for name, m in layers.items():
        e = blob["layers"][name]
        assert float(e["true_bits"].max()) == float(model_stats.get_true_layer_bit_width(m))
        assert e["bits"] == next(b for b in R.WIDTHS if float(e["true_bits"].max()) <= b)
        rows = m.weight.shape[0] if e["qscheme"] == "PER_CHANNEL" else 1
        assert e["codes"].shape == (rows, R.row_bytes(m.weight.numel() // rows, e["bits"]))
        packed += e["codes"].numel()
        ideal += m.weight.numel() * e["bits"] / 8
        if kind == "bias_net" and isinstance(m, NoisyConv2d):
            assert e["quant_bias"] and e["bias"] is not None
    if kind.startswith("resnet20"):
        # b/32 of the fp32 bytes; rows of 144 codes pad to 16 bytes (at most 1/9 more)
        assert ideal <= packed <= ideal * 10 / 9
    acts = [n for n, m in qm.named_modules() if isinstance(m, NoisyAct)]
    for n in acts:
        e = blob["layers"][n]
        assert not e["disabled"] and e["bits"] is not None and e["n_levels"] <= 1 << e["bits"]

    fresh = _build(kind, method, calib=False)
    if channels_last:
        fresh.model.to(memory_format=torch.channels_last)
    fresh.load_state_dict(qm.state_dict())
    with torch.no_grad():
        for m in _weight_layers(fresh).values():
            m.weight.normal_()
            if m.bias is not None:
                m.bias.normal_()
    params = {n: m.weight for n, m in _weight_layers(fresh).items()}
    load_quantized(fresh, blob)
    for n, m in _weight_layers(fresh).items():
        assert m.weight is params[n]
        if channels_last and m.weight.dim() == 4 and m.weight.shape[-1] > 1:
            assert m.weight.is_contiguous(memory_format=torch.channels_last)
    fresh.eval()
    with torch.no_grad():
        out = fresh(xfix)
    assert torch.equal(bits_of(out), bits_of(out_ref))


def test_load_refuses_other_quantizer_parameters():
    qm = _build("resnet20", "STE")
    blob = export_quantized(qm)
    other = _build("resnet20", "STE")
    other.load_state_dict(qm.state_dict())
    name, m = next(iter(_weight_layers(other).items()))
    with torch.no_grad():
        m.log_wght_s.add_(0.25)
    with pytest.raises(ValueError, match="differs from the exporter"):
        load_quantized(other, blob)
