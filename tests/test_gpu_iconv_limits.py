"""GPU: the integer layers (include/mhaq_fq.h "Integer layers") at the edges of what they accept.

- fq_iconv_kernel over the N tiling (1 to 2048 output channels), the K pipeline (1 to 72 stages,
  partly zero-filled last stages), the M tiling (1 row to several waves of CTAs), the int32 bound
  with every code at 255, and the stores of y inside a larger buffer.  Each result is held to the
  operator bar of tests/test_gpu_iconv.py against the fp64 convolution of the exact dequantized
  values, or compared bit for bit.
- fq_act_codes_kernel against a numpy fp32 restatement of the forward's codes that shares no code
  with the kernel, at special values, misaligned inputs, scales outside the fast path and an input
  large enough for the grid-stride loop.
- The fused epilogue's general code path, its scalar residual load and its 64-bit offsets, each
  bit for bit against int_conv2d -> + residual -> activation -> act_codes."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mhaq_b200 import ops
from tests.test_gpu_iconv import _act_operands, _check_bar, _random_layer

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _i32(t):
    return t.contiguous(memory_format=torch.channels_last).view(torch.int32)


def _codes(ca, cp):
    """uint8 codes [B, H, W, cp] of integer activation codes ca [B, C, H, W], padding channels 0."""
    codes = torch.zeros(ca.shape[0], ca.shape[2], ca.shape[3], cp, dtype=torch.uint8, device=DEV)
    codes[..., :ca.shape[1]] = ca.permute(0, 2, 3, 1).to(torch.uint8)
    return codes


def _conv_bar(bsz, h, w, c, n, k, stride, pad, w_bits, levels, seed):
    L, cw, sw, zpw, sa, zpa, b = _random_layer(n, c, k, w_bits, levels, True, True, True, seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    ca = torch.randint(0, levels, (bsz, c, h, w), generator=g, device=DEV)
    y = ops.int_conv2d(_codes(ca, L.cp), L, stride, pad)
    _check_bar(y, ca, L, cw, sw, zpw, sa, zpa, b, stride, pad)
    return L


def _linear_bar(m, c, n, w_bits, levels, seed):
    L, cw, sw, zpw, sa, zpa, b = _random_layer(n, c, 1, w_bits, levels, True, True, True, seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    ca = torch.randint(0, levels, (m, c), generator=g, device=DEV)
    codes = torch.zeros(m, L.cp, dtype=torch.uint8, device=DEV)
    codes[:, :c] = ca.to(torch.uint8)
    y = ops.int_linear(codes, L)
    assert y.shape == (m, n)
    _check_bar(y[:, :, None, None], ca[:, :, None, None], L, cw, sw, zpw, sa, zpa, b, (1, 1), (0, 0))
    return L


# ---------------------------------------------------------------------------------------------
# N, K and M tiling
# ---------------------------------------------------------------------------------------------
# 1: tile_n 16 (32 TMEM columns); 256 / 257: two tiles of 128 / 129; 510: two full 255-channel
# tiles; 1000: four tiles of 250; 2048: nine tiles of 228, the last one 224
N_SWEEP = [1, 2, 15, 17, 254, 255, 256, 257, 509, 510, 511, 1000, 2048]


@pytest.mark.parametrize("n", N_SWEEP)
def test_n_sweep_linear(n):
    _linear_bar(130, 40, n, 4, 16, n)


@pytest.mark.parametrize("n", N_SWEEP)
def test_n_sweep_conv3x3(n):
    _conv_bar(2, 7, 6, 24, n, (3, 3), (1, 1), (1, 1), 8, 256, 7 * n + 1)


@pytest.mark.parametrize("stages", [1, 2, 3, 4, 5, 8, 9, 16, 17])
@pytest.mark.parametrize("last_stage", ["full", "one_chunk"])
def test_k_sweep_1x1(stages, last_stage):
    """K = Cp bytes of a 1x1 conv: whole stages, or a last stage holding one 16-byte chunk of K and
    seven zero-filled ones (C not a multiple of 16: padding channels as well).  Depths 1 and 2 run
    only the producers' tail arrivals; 4, 8, 16 end on an empty-barrier phase flip, 5, 9, 17 one
    stage after it."""
    c = 128 * stages if last_stage == "full" else 128 * stages - 117
    cp = ops.code_channels(c)
    assert ops.iconv_layout(64, cp)[4] == stages
    _conv_bar(2, 9, 9, c, 64, (1, 1), (1, 1), (0, 0), 8, 256, 100 * stages + len(last_stage))


@pytest.mark.parametrize("c,stages", [(16, 2), (48, 4), (100, 8), (1024, 72)])
def test_k_sweep_3x3(c, stages):
    """3x3 taps across stage boundaries: K = 9 Cp = 144 (9 chunks), 432 (27), 1008 (63), 9216."""
    assert ops.iconv_layout(48, 9 * ops.code_channels(c))[4] == stages
    _conv_bar(2, 8, 7, c, 48, (3, 3), (1, 1), (1, 1), 4, 16, c)


@pytest.mark.parametrize("m", [1, 127, 128, 129, 255, 257])
def test_m_sweep_linear(m):
    _linear_bar(m, 48, 20, 4, 16, m)


def test_several_waves_of_ctas():
    """M = 65536 rows: 512 M tiles, more than three waves of one CTA per SM on 148 SMs."""
    assert 4 * 128 * 128 > 148 * 128 * 3
    _conv_bar(4, 128, 128, 16, 32, (3, 3), (1, 1), (1, 1), 4, 16, 77)


# ---------------------------------------------------------------------------------------------
# the stores of y stay inside y
# ---------------------------------------------------------------------------------------------
SENTINEL = 0x7FBADBAD        # a NaN bit pattern no kernel result has


@pytest.mark.parametrize("offset,n", [(4, 64), (1, 64), (4, 300), (1, 300), (0, 10), (3, 1)])
def test_stores_stay_inside_y(offset, n):
    """y is a view at ``offset`` floats into a buffer filled with a sentinel: 16-byte aligned
    (float4 stores where n % 4 == 0) or not (offset 1 / 3: the scalar stores).  Every word outside
    y keeps the sentinel and y equals the result written to a fresh tensor, bit for bit.  M = 189
    leaves a partial last M tile; n = 300 has two N tiles of 150."""
    bsz, h, w, c = 3, 9, 7, 16
    L, *_ = _random_layer(n, c, (3, 3), 4, 16, True, True, True, offset + n)
    ca = torch.randint(0, 16, (bsz, c, h, w), generator=torch.Generator(device=DEV).manual_seed(n), device=DEV)
    codes = _codes(ca, L.cp)
    ref = ops.int_conv2d(codes, L, (1, 1), (1, 1))
    total = ref.numel()
    buf = torch.full((offset + total + 4096,), SENTINEL, dtype=torch.int32, device=DEV)
    y = buf.view(torch.float32)[offset:offset + total]
    assert y.data_ptr() % 16 == 4 * offset % 16
    ops._iconv(codes, L, y, bsz, h, w, (1, 1), (1, 1))
    assert bool((buf[:offset] == SENTINEL).all()) and bool((buf[offset + total:] == SENTINEL).all())
    assert torch.equal(buf[offset:offset + total], ref.permute(0, 2, 3, 1).reshape(-1).view(torch.int32))


# ---------------------------------------------------------------------------------------------
# the int32 bound: every code at 255 at the largest accepted K
# ---------------------------------------------------------------------------------------------
# (kernel, C = Cp, padding, (B, H, W)): K = 33024 resp. 9 * 3664 = 32976, K * 255 * 255 < 2^31
BOUND = [((1, 1), 33024, (0, 0), (2, 5, 13)), ((3, 3), 3664, (1, 2), (2, 6, 5))]


@pytest.mark.parametrize("k,c,pad,shape", BOUND)
@pytest.mark.parametrize("pattern", ["all_255", "mixed_0_255"])
def test_int32_bound_is_exact(k, c, pad, shape, pattern):
    """Channel 0 has alpha * S + beta * SA = 2^-18 (S - 255 SA), channel 1 2^-18 (S - 254 SA), both
    exact in fp64 (alpha = 2^-18, beta = -255 / -254 * 2^-18, C = 0).  With every code at 255,
    S = 255 SA at every pixel, so channel 0 is exactly 0 and channel 1 exactly 2^-18 SA with
    SA = 255 * (valid taps) * C: at an interior pixel S = K * 255 * 255, the largest sum the bound
    admits.  The other channels have random operands and the mixed pattern random 0 / 255 codes:
    the operator bar."""
    (kh, kw), (bsz, h, w), n = k, shape, 16
    kk = kh * kw * c
    assert ops.int32_bound_ok(kk, 255, 255) and not ops.int32_bound_ok(kh * kw * (c + 16), 255, 255)
    g = torch.Generator(device=DEV).manual_seed(c)
    if pattern == "all_255":
        cw = torch.full((n, c, kh, kw), 255, device=DEV)
        ca = torch.full((bsz, c, h, w), 255, device=DEV)
    else:
        cw = torch.randint(0, 2, (n, c, kh, kw), generator=g, device=DEV) * 255
        ca = torch.randint(0, 2, (bsz, c, h, w), generator=g, device=DEV) * 255
    f64 = dict(dtype=torch.float64, device=DEV)
    sw = torch.exp2(torch.randint(-12, -8, (n,), generator=g, device=DEV).to(torch.float64)
                    + torch.rand(n, generator=g, device=DEV, dtype=torch.float64))
    zpw = -torch.rand(n, generator=g, device=DEV, dtype=torch.float64) * 0.2
    sw[:2] = 2.0 ** -10
    zpw[0], zpw[1] = -255 * 2.0 ** -10, -254 * 2.0 ** -10
    sa, zpa = 2.0 ** -8, 0.0
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, None, 255, 255)
    assert L.cp == c
    y = ops.int_conv2d(_codes(ca, c), L, (1, 1), pad)
    _check_bar(y, ca, L, cw, sw, zpw, sa, zpa, None, (1, 1), pad)
    if pattern == "all_255":
        taps = F.conv2d(torch.ones(bsz, 1, h, w, **f64), torch.ones(1, 1, kh, kw, **f64), padding=pad)[:, 0]
        sa_ref = 255 * c * taps
        assert bool((taps == kh * kw).any()) and (kh == 1 or bool((taps < kh * kw).any()))
        assert bool((y[:, 0] == 0).all()), "S != 255 SA"
        assert torch.equal(y[:, 1].double(), 2.0 ** -18 * sa_ref), "SA wrong"
        # at an interior pixel: S = 255 * SA = K * 255 * 255
        assert float(255 * sa_ref.max()) == kk * 65025 < 2 ** 31


@pytest.mark.parametrize("k,c,pad,shape", BOUND)
def test_int32_bound_refuses_one_step_above(k, c, pad, shape):
    (kh, kw) = k
    cw = torch.zeros(2, c + 16, kh, kw, dtype=torch.int64)
    with pytest.raises(ValueError, match="int32 accumulator"):
        ops.int_layer_operands(cw, 2.0 ** -10, 0.0, 2.0 ** -8, 0.0, None, 255, 255)
    ops.int_layer_operands(cw[:, :c], 2.0 ** -10, 0.0, 2.0 ** -8, 0.0, None, 255, 255)


# ---------------------------------------------------------------------------------------------
# act_codes against a numpy restatement of the forward's codes
# ---------------------------------------------------------------------------------------------
def _np_codes(x, s, zp, hi):
    """oracle.fq_oracle.quantize in eval mode restated in numpy fp32 (lo = zp, as act_codes passes
    it): rint((clip(x, lo, hi) - zp) / s), saturated to [0, 255] with NaN -> 0, and the number of
    codes outside [0, 255] (NaN included).  x: fp32 [..., C]."""
    s, zp, hi = np.float32(s), np.float32(zp), np.float32(hi)
    with np.errstate(invalid="ignore", over="ignore"):
        v = np.rint((np.clip(x, zp, hi) - zp) / s)
        bad = int((~((v >= 0) & (v <= 255))).sum())
        codes = np.where(np.isnan(v), np.float32(0), np.clip(v, 0, 255)).astype(np.uint8)
    return codes, bad


def _special_input(shape, s, zp, hi, levels, seed):
    """fp32 NHWC values zp + v * s, v uniform in [-20, levels + 40], with special values spread
    over the tensor: +-0, +-inf, NaN, subnormals, exactly lo and hi, exact (k + 0.5) * s ties and
    +-1e30 (beyond the fast path's |x| <= 2^80)."""
    rng = np.random.default_rng(seed)
    x = (np.float32(zp) + rng.uniform(-20, levels + 40, size=shape).astype(np.float32) * np.float32(s))
    flat = x.reshape(-1)
    specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1e-39, -1e-39, 2.0 ** -149,
                         zp, hi, 1e30, -1e30], dtype=np.float32)
    idx = rng.permutation(flat.size)
    k = min(flat.size, 6 * specials.size)
    flat[idx[:k]] = np.resize(specials, k)
    ties = idx[k:k + flat.size // 4]
    flat[ties] = np.float32(zp) + (rng.integers(0, levels, ties.size) + 0.5).astype(np.float32) * np.float32(s)
    return x.astype(np.float32)


# (levels, signed, top code): max_val = zp + top * s; top > 255 saturates codes above 255
ACT_PARAMS = [(16, True, 15), (256, False, 255), (256, True, 300)]


def _act_codes_case(x_nhwc, s, zp, hi, offset=0):
    b, h, w, c = x_nhwc.shape
    flat = torch.from_numpy(x_nhwc).reshape(-1).to(DEV)
    buf = torch.empty(flat.numel() + offset, device=DEV)
    buf[offset:] = flat
    x = buf[offset:].view(b, h, w, c).permute(0, 3, 1, 2)          # channels_last NCHW
    assert x.is_contiguous(memory_format=torch.channels_last) and x.data_ptr() % 16 == 4 * offset
    t = lambda v: torch.tensor([v], dtype=torch.float32, device=DEV)     # noqa: E731
    codes, n_bad = ops.act_codes(x, t(s), t(zp), t(hi))
    want, bad = _np_codes(x_nhwc, s, zp, hi)
    got = codes.cpu().numpy()
    assert got.shape == (b, h, w, ops.code_channels(c))
    mism = np.argwhere(got[..., :c] != want)
    assert mism.size == 0, f"{len(mism)} codes differ, first at {mism[0]}: x = {x_nhwc[tuple(mism[0])]!r}, " \
                           f"got {got[tuple(mism[0])]}, want {want[tuple(mism[0])]}"
    assert not got[..., c:].any()
    assert int(n_bad) == bad


@pytest.mark.parametrize("c", [1, 3, 4, 17, 255, 256])
@pytest.mark.parametrize("s_exp,params", [(-5, p) for p in ACT_PARAMS] + [(-40, ACT_PARAMS[2]), (40, ACT_PARAMS[2])])
def test_act_codes_equal_numpy_restatement(c, s_exp, params):
    """Scales 2^-40 and 2^40 lie outside [2^-32, 2^32] and take the general path throughout."""
    levels, signed, top = params
    s = 2.0 ** s_exp
    zp = -(levels // 2) * s if signed else 0.0
    hi = zp + top * s
    x = _special_input((3, 5, 7, c), s, zp, hi, levels, c * 1000 + s_exp + top)
    _act_codes_case(x, s, zp, hi)


@pytest.mark.parametrize("offset", [1, 2, 3])
@pytest.mark.parametrize("c", [4, 64])
def test_act_codes_of_a_misaligned_input(offset, c):
    """C % 4 == 0 but x off a 16-byte boundary: the scalar loads."""
    s, zp = 2.0 ** -4, -8 * 2.0 ** -4
    x = _special_input((2, 6, 5, c), s, zp, zp + 15 * s, 16, offset * 100 + c)
    _act_codes_case(x, s, zp, zp + 15 * s, offset)


def test_act_codes_grid_stride_loop():
    """[64, 64, 56, 56]: 12.8 M codes, 3.2 M 4-code groups, more than the 148 * 64 CTAs of 128
    threads cover in one pass."""
    s, zp = 2.0 ** -5, -128 * 2.0 ** -5
    x = _special_input((64, 56, 56, 64), s, zp, zp + 255 * s, 256, 5)
    assert x.size // 4 > 148 * 64 * 128
    _act_codes_case(x, s, zp, zp + 255 * s)


# ---------------------------------------------------------------------------------------------
# fused epilogue limits
# ---------------------------------------------------------------------------------------------
def _fused_layer(n, seed):
    bsz, h, w, c = 2, 9, 8, 16
    L, *_ = _random_layer(n, c, (3, 3), 4, 16, True, True, True, seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    ca = torch.randint(0, 16, (bsz, c, h, w), generator=g, device=DEV)
    return L, _codes(ca, L.cp)


def _composition(plain, r, activation, slope):
    ref = plain if r is None else plain + r
    if activation == "relu":
        return torch.relu(ref)
    if activation == "leaky_relu":
        return F.leaky_relu(ref, slope)
    return ref


@pytest.mark.parametrize("activation", [None, "relu", "leaky_relu"])
@pytest.mark.parametrize("case", ["huge_residual", "scale_2^-40", "scale_2^40"])
def test_fused_codes_general_path(case, activation):
    """The next layer's codes from fwd_elem: residuals of +-1e30 and +-inf put |t| above 2^80, and
    scales 2^-40 / 2^40 lie outside the fast path's range (the layer scaled by a folded 4 s, so
    that t spans the codes).  fp32 and codes equal the composition bit for bit, and the codes equal
    the numpy restatement."""
    n = 64
    L, codes = _fused_layer(n, 7)
    s_exp = {"huge_residual": -5, "scale_2^-40": -40, "scale_2^40": 40}[case]
    s = 2.0 ** s_exp
    if s_exp != -5:
        L = L.fold_affine(torch.full((n,), 4 * s, dtype=torch.float64), 0.0)
    zp, hi = -128 * s, 127 * s
    plain = ops.int_conv2d(codes, L, (1, 1), (1, 1))
    g = torch.Generator(device=DEV).manual_seed(3)
    r = torch.randn(plain.shape, generator=g, device=DEV) * plain.abs().amax()
    flat = r.view(-1)
    if case == "huge_residual":
        flat[0::5], flat[1::5], flat[2::11], flat[3::13] = 1e30, -1e30, float("inf"), float("-inf")
    r = r.contiguous(memory_format=torch.channels_last)
    slope = 0.125 if activation == "leaky_relu" else None
    prm = tuple(torch.tensor([v], device=DEV) for v in (s, zp, hi))
    y, cod = ops.int_conv2d_fused(codes, L, (1, 1), (1, 1), residual=r, activation=activation,
                                  negative_slope=slope, code_params=prm)
    ref = _composition(plain, r, activation, slope)
    assert torch.equal(_i32(y), _i32(ref))
    assert torch.equal(cod, ops.act_codes(ref, *prm)[0])
    want, _ = _np_codes(ref.permute(0, 2, 3, 1).cpu().numpy(), s, zp, hi)
    assert np.array_equal(cod[..., :n].cpu().numpy(), want)
    assert 0 < int((cod[..., :n] > 0).sum()) and 0 < int((cod[..., :n] < 255).sum())


@pytest.mark.parametrize("activation", [None, "relu"])
@pytest.mark.parametrize("n", [64, 300])
def test_fused_misaligned_residual(n, activation):
    """A channels_last residual one float off a 16-byte boundary with n % 4 == 0: int_conv2d_fused
    passes it as it is and the epilogue takes the scalar residual loads."""
    L, codes = _fused_layer(n, 11)
    plain = ops.int_conv2d(codes, L, (1, 1), (1, 1))
    b, _, ho, wo = plain.shape
    buf = torch.randn(plain.numel() + 1, generator=torch.Generator(device=DEV).manual_seed(n), device=DEV)
    r = buf[1:].view(b, ho, wo, n).permute(0, 3, 1, 2)
    assert r.is_contiguous(memory_format=torch.channels_last) and r.data_ptr() % 16 == 4
    s, zb, hi = _act_operands(16, True, seed=n)
    y, cod = ops.int_conv2d_fused(codes, L, (1, 1), (1, 1), residual=r, activation=activation,
                                  code_params=(s, zb, hi))
    ref = _composition(plain, r, activation, None)
    assert torch.equal(_i32(y), _i32(ref))
    assert torch.equal(cod, ops.act_codes(ref, s, zb, hi)[0])


def test_fused_more_than_2p31_elements():
    """64-bit offsets of the residual and the codes: a fused 1x1 layer over M rows with
    M * N > 2^31 residual elements and M * code_channels(N) > 2^31 code bytes, codes only.
    Sampled rows (the first and last 3000 among them) equal the same fused call on the gathered
    rows, which equals the composition (each output row depends on its own row alone)."""
    n, c = 20, 16
    m = (1 << 31) // n + 4097
    L, *_ = _random_layer(n, c, 1, 4, 16, True, True, True, 9)
    g = torch.Generator(device=DEV).manual_seed(9)
    codes = torch.randint(0, 16, (m, 1, 1, L.cp), generator=g, dtype=torch.uint8, device=DEV)
    r = torch.randn(m, n, 1, 1, generator=g, device=DEV)
    assert r.numel() > 1 << 31 and m * ops.code_channels(n) > 1 << 31
    s, zb, hi = _act_operands(16, True, seed=9)
    y, cod = ops.int_conv2d_fused(codes, L, residual=r, activation="relu", out_fp32=False, code_params=(s, zb, hi))
    assert y is None and cod.shape == (m, 1, 1, 32)
    rows = torch.cat([torch.arange(0, 3000, device=DEV), torch.arange(m - 3000, m, device=DEV),
                      torch.randint(0, m, (3000,), generator=g, device=DEV)])
    got = cod[rows]
    sub_codes, sub_r = codes[rows], r[rows]
    del cod, codes, r
    torch.cuda.empty_cache()
    _, want = ops.int_conv2d_fused(sub_codes, L, residual=sub_r, activation="relu", out_fp32=False,
                                   code_params=(s, zb, hi))
    assert torch.equal(got, want)
    ref = torch.relu(ops.int_conv2d(sub_codes, L) + sub_r)
    assert torch.equal(got, ops.act_codes(ref, s, zb, hi)[0])
    assert 0 < int((got[..., :n] > 0).sum()) and not got[..., n:].any()
