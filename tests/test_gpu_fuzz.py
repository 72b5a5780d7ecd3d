"""Seeded differential fuzz: the CUDA path (through mhaq_b200.fake_quant -> the C ABI) against the
LIVE reference (oracle/_ref) on the same GPU, over randomly drawn shapes, layouts, parameter
shapes, estimators, bit widths, scale magnitudes, clamp ranges and awkward values.

The parity tests elsewhere pin named configurations; this one walks the space between them:
ragged / tiny / misaligned sizes, per-tensor and per-channel (dim 0) parameters, clamp ranges that
are finite, one-sided or absent, channels_last and sliced (non-contiguous) inputs, inputs sitting
exactly on rounding ties and on the clamp bounds, zeros, signed zeros and huge magnitudes.
Where the reference is not staged, oracle/ref_port.py (its API on the golden-pinned oracle) stands in.

Bars: y and the STE / LSQ input gradient bit-exact; parameter gradients by
oracle/checks.py:assert_param_grad (1e-5 of the reference's fp32 value, or as close as the
reference itself to the fp64 sum of its own fp32 terms).
"""
import math
import os
import random
import types

import pytest
import torch

from oracle import checks as C
from oracle import fq_oracle as O
from oracle import ref_loader, ref_port

pytestmark = pytest.mark.gpu

REL = 1e-5
N_CASES = int(os.environ.get("MHAQ_FUZZ_CASES", "96"))
N_LAYER_CASES = int(os.environ.get("MHAQ_FUZZ_LAYER_CASES", "24"))     # more seeds: MHAQ_FUZZ_CASES=1000 pytest ...


@pytest.fixture(scope="module")
def ref():
    # the live reference where oracle/_ref/ is staged, else its restatement on the oracle
    return ref_loader.load_ops() if ref_loader.available() else ref_port.load()


@pytest.fixture(scope="module")
def fq():
    import mhaq_b200
    return mhaq_b200


def _draw_shape(rng):
    kind = rng.choice(["vec", "mat", "conv_w", "act", "tiny", "ragged"])
    if kind == "vec":
        return (rng.choice([1, 3, 4, 511, 2044, 2048, 4099, 70001, 1 << 18]),)
    if kind == "mat":
        return (rng.choice([1, 2, 7, 64, 300]), rng.choice([1, 5, 64, 577, 4096, 9001]))
    if kind == "conv_w":
        return (rng.choice([1, 8, 48, 130]), rng.choice([1, 3, 16, 50]), rng.choice([1, 3]), rng.choice([1, 3]))
    if kind == "act":
        return (rng.choice([1, 2, 5]), rng.choice([3, 16, 33]), rng.choice([7, 14, 17]), rng.choice([7, 14, 17]))
    if kind == "tiny":
        return tuple(rng.choice([1, 2, 3]) for _ in range(rng.choice([1, 2, 3, 4])))
    return (rng.choice([2, 3, 5]), rng.choice([4096 + 1000, 8192 + 3, 12289]))


def _layout(rng, x):
    """Return a tensor with the same values in a randomly chosen memory layout."""
    how = rng.choice(["contig", "contig", "channels_last", "sliced", "transposed"])
    if how == "channels_last" and x.dim() == 4:
        return x.contiguous(memory_format=torch.channels_last)
    if how == "sliced" and x.dim() >= 1:
        pad = torch.zeros(x.shape[:-1] + (x.shape[-1] + 3,), device=x.device)
        pad[..., 1:1 + x.shape[-1]] = x
        return pad[..., 1:1 + x.shape[-1]]
    if how == "transposed" and x.dim() == 2:
        return x.t().contiguous().t()
    return x.contiguous()


def _case(seed):
    rng = random.Random(seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    shape = _draw_shape(rng)
    method = rng.choice(["STE", "STE", "LSQ"])
    bits = rng.choice([1, 2, 3, 4, 5, 8])
    per_channel = len(shape) >= 2 and rng.random() < 0.5
    pshape = ((shape[0],) + (1,) * (len(shape) - 1)) if per_channel else (1,)
    mag = 2.0 ** rng.choice([-9, -3, 0, 0, 2, 6])
    x = torch.randn(shape, device="cuda", generator=g) * mag
    go = torch.randn(shape, device="cuda", generator=g) * 2.0 ** rng.choice([-20, -6, 0, 0, 5])
    lo = (-2.0 * mag * (0.5 + torch.rand(pshape, device="cuda", generator=g)))
    width = 4.0 * mag * (0.5 + torch.rand(pshape, device="cuda", generator=g))
    scale = width / (2 ** bits - 1 if bits > 1 else 1)
    if rng.random() < 0.3:                       # a power-of-two scale: many exact ties
        scale = torch.exp2(torch.round(torch.log2(scale)))
    hi = lo + scale * (2 ** bits - 1)
    zp = lo.clone()
    clamp = rng.choice(["both", "both", "none", "lo_only", "hi_only"])
    awkward = rng.random() < 0.6
    if awkward and x.numel() >= 8:
        flat = x.reshape(-1)
        k = max(1, flat.numel() // 16)
        idx = torch.randperm(flat.numel(), device="cuda", generator=g)
        s0 = scale.reshape(-1)[0]
        z0 = zp.reshape(-1)[0]
        ties = z0 + s0 * (torch.randint(0, 2 ** bits, (k,), device="cuda", generator=g).float() + 0.5)
        flat[idx[:k]] = ties                                         # exact rounding ties (channel 0's grid)
        flat[idx[k:2 * k]] = 0.0
        flat[idx[2 * k:2 * k + 1]] = -0.0
        flat[idx[2 * k + 1:2 * k + 2]] = float(lo.reshape(-1)[0])    # exactly on the bounds
        flat[idx[2 * k + 2:2 * k + 3]] = float(hi.reshape(-1)[0])
        # far outside: beyond 2^80 (the kernels' exact-division range guard) when the clamp catches it
        flat[idx[2 * k + 3:2 * k + 4]] = 3.0e30 if clamp == "both" else 1.0e4 * mag
        go.reshape(-1)[idx[:1]] = 0.0
    x = _layout(rng, x)
    go = _layout(rng, go)
    return dict(shape=shape, method=method, bits=bits, per_channel=per_channel, clamp=clamp,
                x=x, go=go, scale=scale, zp=zp, lo=lo, hi=hi, seed=seed)


def _kernel_noise(fq, x, scale, seed, offset):
    """The noise the kernels draw for `x`, as a tensor indexed like x.  The stream is a function of
    the STORAGE position inside the [rows][inner] view (DESIGN.md §3): a dense channels_last
    tensor is walked as it lies in memory (NHWC), anything else in row-major order."""
    if x.dim() == 4 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last):
        nhwc = x.permute(0, 2, 3, 1)                               # contiguous view of the storage
        sc = scale.reshape(-1, 1, 1, 1) if scale.numel() > 1 else None
        return fq.philox_noise(nhwc, sc, seed=seed, offset=offset).permute(0, 3, 1, 2)
    return fq.philox_noise(x.contiguous(), scale if scale.numel() > 1 else None, seed=seed, offset=offset)


@pytest.mark.parametrize("seed", range(N_CASES))
def test_fuzz_against_the_live_reference(fq, ref, seed):
    c = _case(1000 + seed)
    x, go, scale, zp = c["x"], c["go"], c["scale"], c["zp"]
    use_lo = c["clamp"] in ("both", "lo_only")
    use_hi = c["clamp"] in ("both", "hi_only")
    method = c["method"]
    r = None if method == "LSQ" else _kernel_noise(fq, x, scale, 11, seed)
    orig_randint_like = torch.randint_like

    def leaves():
        mk = lambda t: t.detach().clone().requires_grad_(True)
        return mk(scale), mk(zp), (mk(c["lo"]) if use_lo else None), (mk(c["hi"]) if use_hi else None)

    # ---- live reference
    xr = x.detach().clone().requires_grad_(True)
    s_r, z_r, l_r, h_r = leaves()
    # (torch.clamp takes two tensors or two numbers: a one-sided range is a tensor of +-inf there)
    inf = torch.full_like(c["lo"], math.inf)
    none = not (use_lo or use_hi)
    Q = ref.Quantizer(types.SimpleNamespace(training=True), s_r, z_r,
                      l_r if use_lo else (-math.inf if none else -inf),
                      h_r if use_hi else (math.inf if none else inf), qnmethod=ref.QNMethod[method])
    if r is not None:
        torch.randint_like = lambda t, high, **kw: (r.to(t.dtype) + 0.5)
    try:
        y_r = Q.dequantize(Q.quantize(xr))
        y_r.backward(go)
    finally:
        torch.randint_like = orig_randint_like
    # ---- CUDA path
    xo = x.detach().clone().requires_grad_(True)
    s_o, z_o, l_o, h_o = leaves()
    y_o = fq.fake_quant(xo, s_o, z_o, l_o if use_lo else -math.inf, h_o if use_hi else math.inf,
                        method=method, philox=(11, seed))
    y_o.backward(go)
    tag = f"seed {seed}: {c['shape']} {method} {c['bits']}b {'per-channel' if c['per_channel'] else 'per-tensor'} clamp={c['clamp']}"
    C.assert_bit_exact(y_o, y_r, "y " + tag)
    C.assert_bit_exact(xo.grad, xr.grad, "gx " + tag)
    # ---- parameter gradients
    n_per = x.numel() // scale.numel()
    ex = C.exact_param_grads(O.fake_quant, x.detach().contiguous(), go.contiguous(), scale, zp,
                             c["lo"] if use_lo else (None if none else -inf),
                             c["hi"] if use_hi else (None if none else inf), method,
                             None if r is None else r.contiguous())
    # fp32 rounding of the per-element terms: go*code and g*(v/s) are formed at the magnitude
    # |go| * |v|, the estimator's term (3^-1/2 * g * r, or g * e for LSQ) at up to 0.5 * |go| * s
    xc = x.detach()
    if use_lo:
        xc = torch.maximum(xc, c["lo"])
    if use_hi:
        xc = torch.minimum(xc, c["hi"])
    vmax = float(((xc - zp) / scale).abs().max())
    gmax = float(go.abs().max()) + 1e-30
    floor = 2e-7 * math.sqrt(n_per) * gmax * (vmax + 4 + 0.5 * float(scale.abs().max()))
    C.assert_param_grad(s_o.grad, s_r.grad, ex[0], REL, "g_scale " + tag, floor)
    C.assert_param_grad(z_o.grad, z_r.grad, ex[1], REL, "g_zp " + tag, floor)
    if use_lo:
        C.assert_param_grad(l_o.grad, l_r.grad, ex[2], REL, "g_lo " + tag, floor)
    if use_hi:
        C.assert_param_grad(h_o.grad, h_r.grad, ex[3], REL, "g_hi " + tag, floor)


@pytest.mark.parametrize("seed", range(32))
def test_fuzz_per_channel_weights_all_estimators(fq, ref, seed):
    """Weight-style tensors (per-channel, no clamp, calibration-formula scale) at random [C, inner]
    shapes and bit widths, every estimator the reference can run — AEWGS included, whose input
    gradient depends on per-channel fp32 means (1e-5 relative instead of bit-exact)."""
    from tests.test_gpu_live_reference import _check_per_channel, _per_channel_case
    rng = random.Random(7000 + seed)
    C_ = rng.choice([1, 2, 3, 16, 48, 64, 130, 512])
    inner = rng.choice([1, 2, 9, 27, 144, 576, 1152, 4095, 4096, 4608, 8192 + 5, 20000])
    if C_ * inner < 2:
        inner = 9
    bits = rng.choice([1, 2, 3, 4, 8])
    method = rng.choice(["STE", "LSQ", "AEWGS", "AEWGS"])
    x, go, scale, zp = _per_channel_case(C_, inner, bits, seed=seed)
    if inner == 1:                                   # max == min: the calibration formula gives scale 0
        scale = torch.full_like(scale, 0.125)
    _check_per_channel(fq, ref, x, go, scale, zp, method, bits, philox=(17, seed))


# ---------------------------------------------------------------------------
# layer level: NoisyAct / NoisyConv2d of this repo against the live reference's layers
# ---------------------------------------------------------------------------
class _SameNoise:
    """Make both sides use the same noise: the tensor of `noises` whose SHAPE matches the quantized
    tensor (the reference draws in backward, in autograd's order; this repo's ops take it in
    forward) — the reference through torch.randint_like, this repo through the explicit `noise`
    argument of every op a layer may route to."""

    _OPS = ("act_fake_quant", "weight_fake_quant_rows", "weight_fake_quant_log", "weight_fake_quant", "fake_quant")

    def __init__(self, *noises):
        self.by_shape = {tuple(n.shape): n for n in noises}

    def __enter__(self):
        from mhaq_b200 import ops
        self.ops = ops
        self._rl = torch.randint_like
        self._real = {name: getattr(ops, name) for name in self._OPS}
        pick = lambda t: self.by_shape[tuple(t.shape)]
        torch.randint_like = lambda t, high, **kw: (pick(t).to(t.dtype) + 0.5)

        def wrap(real):
            def f(x, *a, **kw):
                kw.pop("philox", None)
                lsq = ops._method_id(kw.get("method", "STE")) == ops.METHOD_IDS["LSQ"]
                kw["noise"] = None if lsq else pick(x)
                return real(x, *a, **kw)
            return f
        for name, real in self._real.items():
            setattr(ops, name, wrap(real))
        return self

    def __exit__(self, *a):
        torch.randint_like = self._rl
        for name, real in self._real.items():
            setattr(self.ops, name, real)


def _scalar_floor(n, gmax, vmax, smax):
    return 2e-7 * math.sqrt(n) * gmax * (vmax + 4 + 0.5 * smax)


@pytest.mark.parametrize("seed", range(N_LAYER_CASES))
def test_fuzz_noisy_act_layer(fq, ref, seed):
    """NoisyAct (log-domain parameters, signed / unsigned, training forward + backward, eval forward
    and `bw`) at random shapes and parameter values, same noise on both sides."""
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
    rng = random.Random(9000 + seed)
    g = torch.Generator(device="cuda").manual_seed(9000 + seed)
    shape = rng.choice([(2, 16, 14, 14), (1, 3, 7, 9), (5, 33, 8, 8), (64, 50), (4096 * 3 + 17,), (2, 8, 31, 33)])
    signed = rng.random() < 0.5
    log_s = float(rng.choice([-6, -4, -3, -2, -1.5, 0]))
    bits = rng.choice([1, 2, 3, 4, 8])
    log_q = log_s + bits + rng.choice([0.0, 0.0, 0.25])            # q = 2^bits * s (sometimes off-grid)
    b = -(2.0 ** (log_q - 1)) * rng.choice([1.0, 0.8]) if signed else 0.0
    x = torch.randn(shape, device="cuda", generator=g) * (2.0 ** (log_q - 1.5))
    if not signed:
        x = x.abs()
    if len(shape) == 4 and rng.random() < 0.5:
        x = x.contiguous(memory_format=torch.channels_last)
    go = torch.randn(shape, device="cuda", generator=g)
    ours = NoisyAct(signed=signed).cuda()
    theirs = ref.NoisyAct(signed=signed).cuda()
    for m in (ours, theirs):
        with torch.no_grad():
            m.log_act_s.fill_(log_s); m.log_act_q.fill_(log_q); m.act_b.fill_(b)
        m.train()
    r = _kernel_noise(fq, x, torch.ones(1, device="cuda"), 21, seed)
    xo = x.detach().clone().requires_grad_(True)
    xr = x.detach().clone().requires_grad_(True)
    with _SameNoise(r):
        yr = theirs(xr); yr.backward(go)
        yo = ours(xo); yo.backward(go)
    tag = f"seed {seed}: {shape} signed={signed} log_s={log_s} log_q={log_q} b={b}"
    C.assert_bit_exact(yo, yr, "y " + tag)
    C.assert_bit_exact(xo.grad, xr.grad, "gx " + tag)
    s = 2.0 ** log_s
    floor = _scalar_floor(x.numel(), float(go.abs().max()), 2.0 ** (log_q - log_s), s) * s * math.log(2) * 4
    for name in ("log_act_s", "log_act_q") + (("act_b",) if signed else ()):
        a, e = getattr(ours, name).grad, getattr(theirs, name).grad
        C.assert_close_rel(a, e, REL, f"g_{name} " + tag, abs_floor=floor)
    # eval: y, bw
    ours.eval(); theirs.eval()
    with torch.no_grad():
        ye_o, ye_r = ours(x), theirs(x)
    C.assert_bit_exact(ye_o, ye_r, "y eval " + tag)
    C.assert_bit_exact(ours.bw.reshape(-1), theirs.bw.reshape(-1), "bw " + tag)


def _exact_aewgs_weight_grad(w, log_s, G):
    """d loss / d weight of the per-channel AEWGS weight path (gdnsq_conv2d.py:72-98 with
    QNAEWGS.backward, gdnsq.py:113-147) in fp64, on the reference's own fp32-valued operands
    (u, v, e and g = G*s are formed in fp32 exactly as the reference forms them; the per-channel
    means, delta, gamma, the division by s and the amin scatter are fp64).  G = d loss / d weight_q."""
    O_ = w.shape[0]
    w2, G2 = w.detach().reshape(O_, -1), G.reshape(O_, -1)
    s = torch.exp2(log_s.detach()).reshape(O_, 1)
    zp = w2.amin(1, keepdim=True)
    v = (w2 - zp) / s
    e = torch.round(v) - v
    g = G2 * s
    e64, g64, s64 = e.double(), g.double(), s.double()
    sg = torch.sign(g64)
    num, e2, me = (sg * e64).mean(1, keepdim=True), (e64 * e64).mean(1, keepdim=True), e64.mean(1, keepdim=True)
    delta = num / (e2 - me * me).clamp_min(1e-3)
    gamma = (delta * (sg * e64)).clamp_max(1 - 0.01)
    du = (g64 - g64 * gamma) / s64
    dzp = G2.double().sum(1, keepdim=True) - du.sum(1, keepdim=True)
    at_min = (w2 == zp)
    return (du + at_min * (dzp / at_min.sum(1, keepdim=True))).reshape(w.shape)


@pytest.mark.parametrize("seed", range(N_LAYER_CASES))
def test_fuzz_noisy_conv2d_layer(fq, ref, seed):
    """NoisyConv2d (per-channel / per-tensor, STE / LSQ / AEWGS, optional quantized bias): the quantized
    weight the convolution sees, and the gradients of weight and log_wght_s, same noise on both
    sides.  cuDNN runs the identical convolution on both sides (deterministic, TF32 off)."""
    from mhaq_b200.aux.types import QScheme
    from mhaq_b200.quantization.gdnsq.gdnsq_utils import QNMethod
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
    rng = random.Random(12000 + seed)
    torch.manual_seed(12000 + seed)
    cin, cout = rng.choice([1, 3, 8, 16, 50]), rng.choice([1, 4, 16, 48, 130])
    k = rng.choice([1, 3, 3, 5])
    per_channel = rng.random() < 0.7
    method = rng.choice(["STE", "LSQ", "AEWGS"])
    bias = rng.random() < 0.5
    quant_bias = bias and per_channel and rng.random() < 0.5
    log_s = float(rng.choice([-7, -5, -4, -3]))
    kw = dict(padding=k // 2, bias=bias)
    ours = NoisyConv2d(cin, cout, k, qscheme=QScheme.PER_CHANNEL if per_channel else QScheme.PER_TENSOR,
                       qnmethod=QNMethod[method], quant_bias=quant_bias, **kw).cuda()
    theirs = ref.NoisyConv2d(cin, cout, k, qscheme=ref.QScheme.PER_CHANNEL if per_channel else ref.QScheme.PER_TENSOR,
                             qnmethod=ref.QNMethod[method], quant_bias=quant_bias, **kw).cuda()
    with torch.no_grad():
        theirs.weight.copy_(ours.weight)
        if bias:
            theirs.bias.copy_(ours.bias)
        for m in (ours, theirs):
            m.log_wght_s.fill_(log_s)
    x = torch.randn(2, cin, 9, 9, device="cuda")
    go = torch.randn(2, cout, 9, 9, device="cuda")
    rw = (torch.randint(0, 2, tuple(ours.weight.shape), device="cuda").float() - 0.5)
    rb = (torch.randint(0, 2, (cout,), device="cuda").float() - 0.5)
    flags = (torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = False, True, False
    try:
        ours.train(); theirs.train()
        with _SameNoise(rw, rb):
            yr = theirs(x); yr.backward(go)
        with _SameNoise(rw, rb):
            yo = ours(x); yo.backward(go)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = flags
    tag = f"seed {seed}: conv {cin}->{cout} k{k} {'pc' if per_channel else 'pt'} {method} bias={bias} qbias={quant_bias} log_s={log_s}"
    C.assert_bit_exact(yo, yr, "conv output " + tag)                  # same quantized weight => same cuDNN result
    if method == "AEWGS" and per_channel and not quant_bias:
        # the input gradient depends on per-channel means which the reference takes in fp32
        # (gdnsq.py:118-124) — over a few hundred elements they carry ~1e-4 relative noise, more
        # than the 1e-5 bar; so: within 1e-5 of the reference, OR at least as close as the
        # reference to the fp64 evaluation of its own formula
        wq = ours.quantized_weight()[0].detach().requires_grad_(True)
        G, = torch.autograd.grad(torch.nn.functional.conv2d(x, wq, None, padding=k // 2), wq, go)
        ex = _exact_aewgs_weight_grad(ours.weight, ours.log_wght_s, G)
        C.assert_param_grad(ours.weight.grad, theirs.weight.grad, ex, REL, "g_weight " + tag,
                            4e-7 * float(theirs.weight.grad.abs().max()))
    elif method == "AEWGS":
        # per-tensor (statistics over dim 0 only: 1-130 elements per mean) or with the bias
        # quantizer sharing the row minimum: no closed form at hand; where 1 - gamma is small the
        # fp32 means of the reference show at a few 1e-5 relative
        # (the row / tensor minimum also receives d/d zero_point = sum(G) - sum(du), a difference of
        # two large sums the reference forms in fp32: checked by the exact rule above, skipped here)
        wd = ours.weight.detach()
        zp = wd.amin((1, 2, 3), keepdim=True) if per_channel else wd.amin()
        keep = (wd != zp)
        C.assert_close_rel(ours.weight.grad[keep], theirs.weight.grad[keep], 1e-4, "g_weight " + tag,
                           abs_floor=1e-6 * float(theirs.weight.grad.abs().max()))
    else:
        C.assert_bit_exact(ours.weight.grad, theirs.weight.grad, "g_weight " + tag)
    n_per = ours.weight[0].numel() if per_channel else ours.weight.numel()
    gmax = float(theirs.weight.grad.abs().max()) + 1e-30
    s = 2.0 ** log_s
    wmax = float(ours.weight.detach().abs().max())
    floor = _scalar_floor(n_per, gmax, 2 * wmax / s, s) * s * math.log(2) * 4
    gs_r = theirs.log_wght_s.grad
    C.assert_close_rel(ours.log_wght_s.grad, gs_r, REL, "g_log_wght_s " + tag, abs_floor=floor)
    if bias:
        C.assert_close_rel(ours.bias.grad, theirs.bias.grad, 1e-5, "g_bias " + tag, abs_floor=1e-6 * float(go.abs().sum(dim=(0, 2, 3)).max()))


@pytest.mark.parametrize("seed", range(N_LAYER_CASES))
def test_fuzz_noisy_linear_layer(fq, ref, seed):
    """NoisyLinear (per-tensor, STE / LSQ) against the live
    reference's layer: output of F.linear on the quantized weight, weight / log_wght_s gradients."""
    from mhaq_b200.aux.types import QScheme
    from mhaq_b200.quantization.gdnsq.gdnsq_utils import QNMethod
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_linear import NoisyLinear
    rng = random.Random(15000 + seed)
    torch.manual_seed(15000 + seed)
    fin, fout = rng.choice([1, 7, 64, 300, 1000]), rng.choice([1, 10, 100, 257])
    # (the reference's per-channel NoisyLinear cannot run: gdnsq_linear.py:71 takes amin((1, 2, 3))
    # of a 2-D weight — IndexError; per-tensor is the only form there is to compare with)
    per_channel = False
    method = rng.choice(["STE", "LSQ"])
    bias = rng.random() < 0.6
    log_s = float(rng.choice([-7, -5, -4, -3]))
    mk = lambda cls, qs, qn: cls(fin, fout, bias=bias, qscheme=qs.PER_CHANNEL if per_channel else qs.PER_TENSOR,
                                 qnmethod=qn[method]).cuda()
    ours, theirs = mk(NoisyLinear, QScheme, QNMethod), mk(ref.NoisyLinear, ref.QScheme, ref.QNMethod)
    with torch.no_grad():
        theirs.weight.copy_(ours.weight)
        if bias:
            theirs.bias.copy_(ours.bias)
        for m in (ours, theirs):
            m.log_wght_s.fill_(log_s)
    x = torch.randn(5, fin, device="cuda")
    go = torch.randn(5, fout, device="cuda")
    rw = (torch.randint(0, 2, tuple(ours.weight.shape), device="cuda").float() - 0.5)
    rb = (torch.randint(0, 2, (fout,), device="cuda").float() - 0.5)
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ours.train(); theirs.train()
        with _SameNoise(rw, rb):
            yr = theirs(x); yr.backward(go)
        with _SameNoise(rw, rb):
            yo = ours(x); yo.backward(go)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    tag = f"seed {seed}: linear {fin}->{fout} {'pc' if per_channel else 'pt'} {method} bias={bias} log_s={log_s}"
    C.assert_bit_exact(yo, yr, "output " + tag)
    C.assert_bit_exact(ours.weight.grad, theirs.weight.grad, "g_weight " + tag)
    n_per = fin if per_channel else fin * fout
    s = 2.0 ** log_s
    floor = _scalar_floor(n_per, float(theirs.weight.grad.abs().max()) + 1e-30,
                          2 * float(ours.weight.detach().abs().max()) / s, s) * s * math.log(2) * 4
    C.assert_close_rel(ours.log_wght_s.grad, theirs.log_wght_s.grad, REL, "g_log_wght_s " + tag, abs_floor=floor)
