"""GPU parity against the LIVE reference (oracle/_ref, the unmodified reference sources staged by
oracle/make_ref.py) running ON THE SAME GPU, at the configurations the benchmarks measure.  Where
it is not staged, the same tests run against oracle/ref_port.py, the reference's API restated on
the golden-pinned oracle.

Bars (BASELINE.json north_star): fake-quant outputs / codes and STE / LSQ input gradients
bit-exact; AEWGS input gradients 1e-5 relative (they depend on per-channel fp32 means);
parameter gradients by the rule of oracle/checks.py:assert_param_grad — within 1e-5 of the
reference's fp32 value, or at least as close as the reference itself to `exact` = the fp64 sum of
the reference's own fp32 per-element terms (for AEWGS, where no per-element decomposition
exists: the reference evaluated in fp64 on the same fp32-valued operands, SURVEY.md §7).
"""
import math
import types

import pytest
import torch

from oracle import checks as C
from oracle import fq_oracle as O
from oracle import ref_loader, ref_port

pytestmark = pytest.mark.gpu

REL = 1e-5


@pytest.fixture(scope="module")
def ref():
    # the live reference where oracle/_ref/ is staged, else its restatement on the oracle
    return ref_loader.load_ops() if ref_loader.available() else ref_port.load()


@pytest.fixture(scope="module")
def fq():
    import mhaq_b200
    return mhaq_b200


class _Noise:
    """Feed the reference the noise the kernels draw: torch.randint_like -> (r + 0.5)."""

    def __init__(self, r):
        self.r, self._orig = r, torch.randint_like

    def __enter__(self):
        def fake(t, high, **kw):
            assert high == 2 and t.shape == self.r.shape
            return (self.r.to(t.dtype) + 0.5)
        if self.r is not None:
            torch.randint_like = fake
        return self

    def __exit__(self, *a):
        torch.randint_like = self._orig


def _ref_fake_quant(ref, x, scale, zp, lo, hi, method, noise):
    """Q.dequantize(Q.quantize(x)) of the live reference (gdnsq.py:189-229)."""
    mod = types.SimpleNamespace(training=True)
    Q = ref.Quantizer(mod, scale, zp, lo, hi, qnmethod=ref.QNMethod[method])
    return Q.dequantize(Q.quantize(x))


def _run_ref(ref, x, go, scale, zp, method, r, dtype=torch.float32):
    xs = x.detach().to(dtype).clone().requires_grad_(True)
    s_, z_ = scale.detach().clone().requires_grad_(True), zp.detach().clone().requires_grad_(True)
    with _Noise(None if method == "LSQ" else r):
        y = _ref_fake_quant(ref, xs, s_, z_, -math.inf, math.inf, method, r)
        y.backward(go.detach().to(dtype))
    return y.detach(), xs.grad, s_.grad, z_.grad


def _per_channel_case(C_, inner, bits, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(C_, inner, device="cuda", generator=g)
    go = torch.randn(C_, inner, device="cuda", generator=g)
    mn, mx = x.amin(1, keepdim=True), x.amax(1, keepdim=True)
    scale = (mx - mn) / (2 ** bits - 1)              # calibration formula, minmaxobserver.py:82
    return x, go, scale, mn


def _exact_per_channel(x, go, scale, zp, method, r):
    """fp64 per-channel sums of the reference's own fp32 per-element terms (gdnsq.py:197-229 and
    torch's Mul / Div / Sub backward), each term formed in fp32 exactly as the reference forms it:
        d/ds  = sum[ go*code ]  -  sum[ g * ((u/s)/s) ]  +  sum[ estimator term ],   g = go*s
        d/dzp = sum[ go ]       -  sum[ g/s ]
    (Summing an expanded-parameter autograd run instead would add the three contributions per
    element in fp32 in autograd's arrival order — a rounding at the magnitude of go*code that is
    not part of the reference's arithmetic.)"""
    u = x - zp
    v = u / scale
    e = torch.round(v) - v
    code = v + e
    g = go * scale
    t_mul = go * code
    t_div = g * (v / scale)
    if method == "LSQ":
        t_est = g * e                                   # gdnsq.py:81-82
    else:
        t_est = ((3.0 ** -0.5) * g) * r                 # gdnsq.py:54-55
    ds = (t_mul.double() - t_div.double() + t_est.double()).sum(1, keepdim=True)
    dz = (go.double() - (g / scale).double()).sum(1, keepdim=True)
    return ds.cpu(), dz.cpu()


def _exact_per_channel_aewgs(x, go, scale, zp, r):
    """QNAEWGS (gdnsq.py:113-147) evaluated in fp64 on the reference's own fp32-valued operands:
    v, e = round(v) - v, codes and g = go*s are formed in fp32 exactly as the reference forms them
    (so no code moves across a rounding tie, which an all-fp64 run of the reference would do);
    the per-channel statistics, delta, the estimator and every sum are then fp64."""
    u = x - zp
    v = u / scale
    e = torch.round(v) - v
    code = v + e
    g = go * scale
    e64, g64, v64, s64 = e.double(), g.double(), v.double(), scale.double()
    sg = torch.sign(g64)
    num = (sg * e64).mean(1, keepdim=True)
    e2 = (e64 * e64).mean(1, keepdim=True)
    me = e64.mean(1, keepdim=True)
    delta = num / (e2 - me * me).clamp_min(1e-3)
    gamma = (delta * (sg * e64)).clamp_max(1 - 0.01)
    gv = g64 - g64 * gamma
    ds = (go.double() * code.double() - gv * (v64 / s64) + (3.0 ** -0.5) * g64 * r.double()).sum(1, keepdim=True)
    dz = (go.double() - gv / s64).sum(1, keepdim=True)
    return ds.cpu(), dz.cpu()


def _check_per_channel(fq, ref, x, go, scale, zp, method, bits, philox=(7, 11)):
    n_inner = x.shape[1]
    r = None if method == "LSQ" else fq.philox_noise(x, scale, seed=philox[0], offset=philox[1])
    y_r, gx_r, gs_r, gz_r = _run_ref(ref, x, go, scale, zp, method, r)
    xs = x.detach().clone().requires_grad_(True)
    s_, z_ = scale.detach().clone().requires_grad_(True), zp.detach().clone().requires_grad_(True)
    y = fq.fake_quant(xs, s_, z_, -math.inf, math.inf, method=method, philox=philox)   # in-kernel Philox
    y.backward(go)
    assert torch.equal(y, y_r), "y not bit-exact"
    if method == "AEWGS":
        C.assert_close_rel(xs.grad, gx_r, REL, "gx", abs_floor=1e-7)
        exact_s, exact_z = _exact_per_channel_aewgs(x, go, scale, zp, r)
    else:
        assert torch.equal(xs.grad, gx_r), "gx not bit-exact"
        exact_s, exact_z = _exact_per_channel(x, go, scale, zp, method, r)
    # fp32 accumulation noise of an N-term sum whose terms are O(|go|): what separates two correct
    # summation orders (the reference's own value sits this far from `exact` too)
    floor = 4e-7 * math.sqrt(n_inner)
    if method == "AEWGS":
        # the fp64 `exact` above does not contain the per-element fp32 roundings of go*code and
        # gv*(v/s) (half an ulp of a number as large as the widest code, times |go|) that BOTH the
        # reference and the kernels commit, identically, before summing: a random walk of
        # ~2^-24 * 2^bits * sqrt(N) — and the assertion takes the worst of up to 4096 channels
        floor = 2.0 ** -24 * 2 ** bits * math.sqrt(n_inner)
    C.assert_param_grad(s_.grad, gs_r, exact_s, REL, f"g_scale[{method},{bits}b]", floor)
    C.assert_param_grad(z_.grad, gz_r, exact_z, REL, f"g_zp[{method},{bits}b]", 4 * floor)


def test_bench_workload_per_channel_512_by_2p19_ste_philox_4bit(fq, ref):
    """The exact BENCH workload (bench.py default): [512, 2^19] fp32, GDNSQ/STE with the in-kernel
    Philox stream, 4 bits; rows of 128 sub-tiles -> the backward's 2-sub-tile task policy."""
    x, go, scale, zp = _per_channel_case(512, 1 << 19, 4, seed=0)
    _check_per_channel(fq, ref, x, go, scale, zp, "STE", 4)


@pytest.mark.parametrize("method", ["LSQ", "AEWGS"])
@pytest.mark.parametrize("C_,log2inner", [(512, 17), (4096, 14)])
def test_large_per_channel_lsq_and_aewgs(fq, ref, C_, log2inner, method):
    x, go, scale, zp = _per_channel_case(C_, 1 << log2inner, 4, seed=C_ + log2inner)
    _check_per_channel(fq, ref, x, go, scale, zp, method, 4)


@pytest.mark.parametrize("bits", [1, 2, 3, 4, 5, 6, 7, 8])
def test_bits_sweep_with_backward_per_channel_2p22(fq, ref, bits):
    x, go, scale, zp = _per_channel_case(64, 1 << 16, bits, seed=100 + bits)
    _check_per_channel(fq, ref, x, go, scale, zp, "STE", bits)


@pytest.mark.parametrize("inner", [3 * 4096 + 1000, 3 * 4096 + 1001])
def test_two_subtile_tasks_with_ragged_last_subtile(fq, ref, inner):
    """2400 rows x 4 sub-tiles >= 2 x 4736: the backward takes 2 sub-tiles per task; the last
    sub-tile of every row is ragged (1000 valid elements), and with an odd row length every row
    base is misaligned (predicated scalar path)."""
    x, go, scale, zp = _per_channel_case(2400, inner, 4, seed=inner)
    _check_per_channel(fq, ref, x, go, scale, zp, "STE", 4)


@pytest.mark.parametrize("n", [2048 * 740 * 3 + 2048 * 5 + 12, 2048 * 9, 2044, 6422528])
@pytest.mark.parametrize("method", ["STE", "LSQ"])
def test_flat_per_tensor_backward_vs_live_reference(fq, ref, n, method):
    """Per-tensor clamped activations (one kernel: persistent balanced grid, operands staged by
    TMA, reduction finished in-kernel): uneven batch counts per block, a ragged tail, fewer
    elements than one batch, and a real ResNet-18 activation size."""
    g = torch.Generator(device="cuda").manual_seed(n % 9973)
    x = torch.randn(n, device="cuda", generator=g) * 1.5
    go = torch.randn(n, device="cuda", generator=g)
    b = torch.tensor([-2.0], device="cuda")
    s = torch.tensor([0.25], device="cuda")
    hi = b + 4.0 - s
    r = None if method == "LSQ" else fq.philox_noise(x, None, seed=5, offset=9)

    def run(fn, noise_kw):
        xs = x.clone().requires_grad_(True)
        s_, b_, h_ = (t.clone().requires_grad_(True) for t in (s, b, hi))
        y = fn(xs, s_, b_, b_, h_, **noise_kw)
        y.backward(go)
        return y.detach(), xs.grad, s_.grad, b_.grad, h_.grad

    with _Noise(r):
        y_r, gx_r, gs_r, gb_r, gh_r = run(lambda xs, s_, b_, l_, h_: _ref_fake_quant(ref, xs, s_, b_, l_, h_, method, r), {})
    y, gx, gs, gb, gh = run(fq.fake_quant, dict(method=method, philox=(5, 9)))
    assert torch.equal(y, y_r) and torch.equal(gx, gx_r)
    # b is zero_point AND min_val here: its exact gradient is the sum of the two leaves' exacts
    ex = C.exact_param_grads(O.fake_quant, x, go, s, b, b, hi, method, r)
    floor = 2e-7 * math.sqrt(n) * 4
    C.assert_param_grad(gs, gs_r, ex[0], REL, "g_scale", floor)
    C.assert_param_grad(gb, gb_r, ex[1] + ex[2], REL, "g_zp+g_lo", floor)
    C.assert_param_grad(gh, gh_r, ex[3], REL, "g_hi", floor)


def test_noisy_act_with_aewgs_estimator_matches_the_live_reference(fq, ref):
    """NoisyAct(qnmethod=AEWGS) — reachable through the public constructor (gdnsq_act.py:17);
    the per-tensor AEWGS statistics follow reduce_to_shape's dim-0 quirk (gdnsq.py:150-152)."""
    from mhaq_b200.quantization.gdnsq.gdnsq_utils import QNMethod
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct
    torch.manual_seed(3)
    x = torch.randn(16, 8, 12, 12, device="cuda") * 2
    go = torch.randn_like(x)
    ours = NoisyAct(signed=True, qnmethod=QNMethod.AEWGS).cuda()
    theirs = ref.NoisyAct(signed=True, qnmethod=ref.QNMethod.AEWGS).cuda()
    for m in (ours, theirs):
        with torch.no_grad():
            m.log_act_s.fill_(-2.0); m.log_act_q.fill_(2.0); m.act_b.fill_(-2.0)
        m.train()
    r = torch.randint(0, 2, x.shape, device="cuda").float() - 0.5
    xr = x.clone().requires_grad_(True)
    with _Noise(r):
        yr = theirs(xr)
        yr.backward(go)
    from mhaq_b200 import ops
    real = ops.fake_quant

    def with_noise(*a, **k):
        k["noise"] = r
        return real(*a, **k)
    xo = x.clone().requires_grad_(True)
    ops.fake_quant = with_noise
    try:
        yo = ours(xo)
        yo.backward(go)
    finally:
        ops.fake_quant = real
    assert torch.equal(yo, yr)
    C.assert_close_rel(xo.grad, xr.grad, REL, "gx", abs_floor=1e-7)
    for name in ("log_act_s", "log_act_q", "act_b"):
        C.assert_close_rel(getattr(ours, name).grad, getattr(theirs, name).grad, REL, name, abs_floor=2e-5)


@pytest.mark.parametrize("method", ["STE", "LSQ", "EWGS", "AEWGS"])
@pytest.mark.parametrize("per_channel", [False, True])
def test_rounding_noise_functions_match_the_live_reference(fq, ref, method, per_channel):
    """QNSTE / QNLSQ / QNAEWGS.apply(v, s) (gdnsq.py:32-147) through ops.rounding_noise: value
    round(v) - v bit-exact, gradients w.r.t. v and s like the reference's backward.  (QNEWGS cannot
    run in the reference, gdnsq.py:102: checked against the oracle's restatement of its intent.)"""
    from mhaq_b200.quantization.gdnsq import gdnsq as G
    torch.manual_seed(11)
    v = (torch.randn(24, 40, 3, 3, device="cuda") * 6)
    go = torch.randn_like(v)
    s = (torch.rand(24, 1, 1, 1, device="cuda") + 0.5) if per_channel else torch.tensor([0.75], device="cuda")
    r = torch.randint(0, 2, v.shape, device="cuda").float() - 0.5
    ours_fn = {"STE": G.QNSTE, "LSQ": G.QNLSQ, "EWGS": G.QNEWGS, "AEWGS": G.QNAEWGS}[method]
    vo, so = v.clone().requires_grad_(True), s.clone().requires_grad_(True)
    from mhaq_b200 import ops
    noise = None if method == "LSQ" else r
    out = ops.rounding_noise(vo, so, method=method, noise=noise)
    out.backward(go)
    assert torch.equal(ours_fn.apply(v, s), out.detach())
    vr, sr = v.clone().requires_grad_(True), s.clone().requires_grad_(True)
    if method == "EWGS":
        e = torch.round(vr) - vr
        ref_out = e.detach()
        gv_ref = -(go.abs()) * e.detach() * 0.01                       # gdnsq.py:96-100 (intent)
        gs_ref = ((3.0 ** -0.5) * go * r)
    else:
        theirs = {"STE": ref.gdnsq.QNSTE, "LSQ": ref.gdnsq.QNLSQ, "AEWGS": ref.gdnsq.QNAEWGS}[method]
        with _Noise(noise):
            ref_out = theirs.apply(vr, sr)
            ref_out.backward(go)
        gv_ref, gs_ref = vr.grad, sr.grad
        ref_out = ref_out.detach()
    assert torch.equal(out.detach(), ref_out)
    if method == "EWGS":
        gs_ref = gs_ref.sum((1, 2, 3), keepdim=True) if per_channel else gs_ref.sum().reshape(1)
    C.assert_close_rel(vo.grad, gv_ref, REL, "grad_v", abs_floor=1e-6)
    C.assert_close_rel(so.grad, gs_ref, REL, "grad_s", abs_floor=2e-5)


def test_noisy_linear_matches_the_live_reference_on_device(fq, ref):
    """NoisyLinear per-tensor LSQ (the only scheme the reference's NoisyLinear can run,
    gdnsq_linear.py:56,71), both on this GPU: same exp2, same cuBLAS — tight bars."""
    from mhaq_b200.aux.types import QScheme
    from mhaq_b200.quantization.gdnsq.gdnsq_utils import QNMethod
    from mhaq_b200.quantization.gdnsq.layers.gdnsq_linear import NoisyLinear
    torch.manual_seed(5)
    ours = NoisyLinear(96, 40, bias=True, qscheme=QScheme.PER_TENSOR, qnmethod=QNMethod.LSQ).cuda()
    theirs = ref.NoisyLinear(96, 40, bias=True, qscheme=ref.QScheme.PER_TENSOR, qnmethod=ref.QNMethod.LSQ).cuda()
    with torch.no_grad():
        theirs.weight.copy_(ours.weight); theirs.bias.copy_(ours.bias)
        ours.log_wght_s.fill_(-4.3); theirs.log_wght_s.fill_(-4.3)
    x = torch.randn(32, 96, device="cuda")
    go = torch.randn(32, 40, device="cuda")
    outs = []
    for m in (ours, theirs):
        m.train()
        xi = x.clone().requires_grad_(True)
        y = m(xi)
        y.backward(go)
        outs.append((y.detach(), xi.grad, m.weight.grad, m.bias.grad, m.log_wght_s.grad))
    (y, gx, gw, gb, gs), (yr, gxr, gwr, gbr, gsr) = outs
    assert torch.equal(y, yr) and torch.equal(gx, gxr) and torch.equal(gb, gbr)
    C.assert_close_rel(gw, gwr, REL, "g_weight", abs_floor=2e-6)
    # exact d/d log_wght_s from the reference's own per-element terms (fp64 sum)
    w = ours.weight.detach()
    s = torch.exp2(ours.log_wght_s.detach())
    g_wq = go.t() @ x                                        # d loss / d weight_q
    ex = C.exact_param_grads(O.fake_quant, w, g_wq, s, w.amin().reshape(1), None, None, "LSQ", None)
    exact = ex[0].double() * s.double().cpu() * math.log(2.0)
    C.assert_param_grad(gs, gsr, exact, REL, "g_log_wght_s", 1e-7)
