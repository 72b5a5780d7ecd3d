"""The grouped, depthwise and dilated integer convolutions (mhaq_fq_iconv_grouped_u8) at the edges
of what they accept.

- The block-diagonal tile plan of fq_iconv_kernel<true, true> (igroup_plan): a 256-row tile whose
  ones rows fill its upper half, tile_out + gpt = 256 exactly, 2 to 16 tiles, groups split into
  2, 3 and 9 parts, and a short last tile.  Each row's plan is pinned (on the CPU as well).
- The K pipeline (1 to 72 stages, a last stage holding one 16-byte chunk, tiles of different K
  widths), the M tiling (1 row to several waves of CTAs) and the depthwise kernel's grid-stride loop.
- The per-group int32 bound with every code at 255, at the largest accepted size and one step above.
- Bit-for-bit identities between the kernels, which all form exact int32 S and SA and the same fp64
  epilogue RN32(fma(alpha, S, fma(beta, SA, C))): the grouped kernel at groups = 1 against the dense
  kernel, a grouped layer against its groups run as dense layers, and a channel multiplier on the
  tensor cores against interleaved depthwise layers on the CUDA cores.  Each first asserts that the
  per-channel operands are equal, so that a difference points at a kernel."""
import pytest
import torch
import torch.nn.functional as F

from mhaq_b200 import ops
from tests.test_gpu_iconv import OP_CASES
from tests.test_gpu_iconv_limits import N_SWEEP
from tests.test_gpu_igroup import (DW_CASES, GCASES, _act_operands, _check_bar, _check_epilogue, _codes,
                                   _grouped_launch, _i32, _layer, _pair2)

DEV = torch.device("cuda")
gpu = pytest.mark.gpu


def _plan(c, n, kh, kw, groups):
    """(n_tiles, tile_n, tile_out, gpt, parts), k_stages of a grouped layer."""
    layout = ops.iconv_grouped_layout(c, n, kh, kw, groups)
    return layout[1:6], layout[6]


def _tile_chunks(c, n, kh, kw, groups):
    """16-channel input chunks of each N tile."""
    (nt, _, tile_out, gpt, parts), _ = _plan(c, n, kh, kw, groups)
    return [ops.grouped_tile(t, groups, c // groups, n // groups, tile_out, gpt, parts)[5] for t in range(nt)]


def _bar(bsz, h, w, c, n, groups, k, stride, pad, dil, w_bits, levels, seed):
    L, cw = _layer(n, c, groups, k, dil, w_bits, levels, seed)
    ca, codes = _codes(bsz, h, w, c, levels, seed + 1)
    y = ops.int_conv2d(codes, L, stride, pad)
    _check_bar(y, ca, L, cw, stride, pad)
    return L, codes


# ---------------------------------------------------------------------------------------------
# the tile plan
# ---------------------------------------------------------------------------------------------
PLAN_CASES = [  # (C, N, groups, dilation, (n_tiles, tile_n, tile_out, gpt, parts), fused), 3x3 kernels
    (256, 128, 128, 1, (1, 256, 128, 128, 1), True),     # cout_g = 1, cin_g = 2: sas fills all 4 A stages
    (32, 480, 32, 1, (2, 256, 240, 16, 1), False),       # tile_out + gpt = 256
    (16, 1008, 16, 1, (4, 256, 252, 4, 1), False),       # tile_out + gpt = 256
    (32, 4064, 32, 1, (16, 256, 254, 2, 1), False),      # 16 tiles
    (4, 1020, 4, 1, (4, 256, 255, 1, 1), False),         # one 255-channel group per full tile
    (4, 1024, 4, 1, (8, 144, 128, 1, 2), True),          # cout_g = 256: two parts
    (2, 1022, 2, 1, (6, 176, 171, 1, 3), True),          # three parts; n_base = 171, 342
    (8, 2048, 1, 2, (9, 240, 228, 1, 9), False),         # nine parts, the last one short (224)
    (258, 258, 129, 1, (2, 208, 130, 65, 1), True),      # a short last tile (65 + 64 groups)
]


@pytest.mark.parametrize("c,n,groups,dil,plan,fused", PLAN_CASES)
def test_plan_of_the_sweep_rows(c, n, groups, dil, plan, fused):
    assert _plan(c, n, 3, 3, groups)[0] == plan


@gpu
@pytest.mark.parametrize("c,n,groups,dil,plan,fused", PLAN_CASES)
def test_tile_plan_sweep(c, n, groups, dil, plan, fused):
    """The operator bar on every row; on the rows marked fused also the epilogue (residual,
    LeakyReLU, fp32 and codes; then codes alone) bit for bit against the composition."""
    assert _plan(c, n, 3, 3, groups)[0] == plan
    seed = c * 7 + n
    L, codes = _bar(2, 6, 5, c, n, groups, 3, 1, dil, dil, 4, 16, seed)
    if fused:
        _check_epilogue(L, codes, 1, dil, True, "leaky_relu", "both", (16, True), seed)
        _check_epilogue(L, codes, 1, dil, False, None, "codes", (256, False), seed + 1)


# ---------------------------------------------------------------------------------------------
# K pipeline, M tiling, waves and the depthwise grid-stride loop
# ---------------------------------------------------------------------------------------------
K_STAGES = [1, 2, 3, 4, 5, 8, 9, 16, 17]


def _k_sweep_cin_g(stages, last_stage):
    """Two groups of 128 output channels (one tile each) with ``stages`` K stages: whole stages,
    or tile 0's last stage holding one 16-byte chunk (cin_g % 16 = 11: its groups straddle chunks)."""
    return 128 * stages if last_stage == "full" else 128 * stages - 117


@pytest.mark.parametrize("stages", K_STAGES)
@pytest.mark.parametrize("last_stage", ["full", "one_chunk"])
def test_plan_of_the_k_sweep(stages, last_stage):
    cin_g = _k_sweep_cin_g(stages, last_stage)
    assert _plan(2 * cin_g, 256, 1, 1, 2) == ((2, 144, 128, 1, 1), stages)
    assert _tile_chunks(2 * cin_g, 256, 1, 1, 2)[0] == (8 * stages if last_stage == "full" else 8 * stages - 7)


@gpu
@pytest.mark.parametrize("stages", K_STAGES)
@pytest.mark.parametrize("last_stage", ["full", "one_chunk"])
def test_k_sweep_grouped_1x1(stages, last_stage):
    """Depths 1 and 2 run only the producers' tail arrivals; 4, 8, 16 end on an empty-barrier phase
    flip, 5, 9, 17 one stage after it."""
    cin_g = _k_sweep_cin_g(stages, last_stage)
    assert _plan(2 * cin_g, 256, 1, 1, 2)[1] == stages
    _bar(2, 5, 4, 2 * cin_g, 256, 2, 1, 1, 0, 1, 8, 256, 100 * stages + len(last_stage))


K_3X3 = [  # (C, N, groups, k_stages, chunks of each tile)
    (2048, 256, 2, 72, [64, 64]),                        # 9 taps x 64 chunks: 72 stages
    (492, 512, 4, 11, [8, 9, 9, 8]),                     # cin_g = 123: tiles 0 and 3 end in zero-filled stages
]


@pytest.mark.parametrize("c,n,groups,stages,chunks", K_3X3)
def test_plan_of_the_3x3_k_rows(c, n, groups, stages, chunks):
    assert _plan(c, n, 3, 3, groups)[1] == stages and _tile_chunks(c, n, 3, 3, groups) == chunks


@gpu
@pytest.mark.parametrize("c,n,groups,stages,chunks", K_3X3)
def test_k_sweep_grouped_3x3(c, n, groups, stages, chunks):
    assert _plan(c, n, 3, 3, groups)[1] == stages and _tile_chunks(c, n, 3, 3, groups) == chunks
    _bar(2, 5, 6, c, n, groups, 3, 1, 1, 1, 4, 16, c)


@gpu
@pytest.mark.parametrize("m", [1, 127, 128, 129, 255, 257])
def test_m_sweep_grouped(m):
    """A 1 x M image with a 3x3 kernel: M output rows, four N tiles (cout_g = 130)."""
    assert _plan(16, 520, 3, 3, 4)[0] == (4, 144, 130, 1, 1)
    _bar(1, 1, m, 16, 520, 4, 3, 1, 1, 1, 4, 16, m)


@gpu
def test_several_waves_of_grouped_ctas():
    """M = 65536 rows: 512 M tiles times 2 N tiles, several waves of one CTA per SM on 148 SMs."""
    assert _plan(16, 256, 3, 3, 2)[0][0] == 2
    _bar(4, 128, 128, 16, 256, 2, 3, 1, 1, 1, 4, 16, 77)


@gpu
def test_depthwise_grid_stride_loop():
    """M * Cp / 16 = 148 * 64 * 256 + 1 items: the capped grid's threads take one item each and
    exactly one thread a second."""
    w = 148 * 64 * 256 + 1
    _bar(1, 1, w, 16, 16, 16, (1, 3), 1, (0, 1), 1, 4, 16, 5)


# ---------------------------------------------------------------------------------------------
# the per-group int32 bound: every code at 255 at the largest accepted size
# ---------------------------------------------------------------------------------------------
BOUND = [  # (C, N, groups, (kh, kw), dilation, padding, (B, H, W)); kh * kw * C / groups * 255^2 < 2^31
    (2 * 3669, 32, 2, (3, 3), 1, (1, 2), (2, 6, 5)),     # 33021 terms; 3669 % 16 = 5: the groups straddle chunks
    (33025, 16, 1, (1, 1), 2, (0, 0), (2, 5, 13)),       # dilated 1x1 (the dense bound counts Cp = 33040)
    (16, 16, 16, (1, 33025), 1, (0, 0), (2, 1, 33025)),  # depthwise: one output pixel, every tap valid
]


def _bound_weights(c, n, groups, k, dev):
    return torch.full((n, c // groups, *k), 255, device=dev)


@pytest.mark.parametrize("c,n,groups,k,dil,pad,shape", BOUND)
def test_int32_bound_refuses_one_step_above(c, n, groups, k, dil, pad, shape):
    """One more input channel per group (one more tap for the depthwise layer) is refused; a dense
    layer with these channels would count its padding channels."""
    cw = _bound_weights(c, n, groups, k, "cpu")
    big = torch.cat([cw, cw[..., -1:]], -1) if groups == c else torch.cat([cw, cw[:, :1]], 1)
    with pytest.raises(ValueError, match="int32 accumulator"):
        ops.int_layer_operands(big, 2.0 ** -10, 0.0, 2.0 ** -8, 0.0, None, 255, 255, groups, dil)
    assert ops.int_layer_operands(cw, 2.0 ** -10, 0.0, 2.0 ** -8, 0.0, None, 255, 255, groups, dil).groups == groups
    if groups == 1:
        with pytest.raises(ValueError, match="int32 accumulator"):
            ops.int_layer_operands(cw, 2.0 ** -10, 0.0, 2.0 ** -8, 0.0, None, 255, 255, 1, 1)


@gpu
@pytest.mark.parametrize("c,n,groups,k,dil,pad,shape", BOUND)
@pytest.mark.parametrize("pattern", ["all_255", "mixed_0_255"])
def test_group_int32_bound_is_exact(c, n, groups, k, dil, pad, shape, pattern):
    """The first two channels of each group (every channel of the depthwise layer) have
    alpha = 2^-18 and beta = -(255 - n % 2) 2^-18, C = 0: with every code at 255, S = 255 SA, so
    even channels are exactly 0 and odd ones exactly 2^-18 SA, SA = 255 * valid taps * cin_g; at
    a pixel with every tap valid S is the largest sum the bound admits.  A weight or ones row that
    leaks into a neighbouring group's channels makes SA inexact.  All channels, and the random
    0 / 255 codes of the mixed pattern, are held to the operator bar."""
    (kh, kw), (bsz, h, w) = k, shape
    cin_g, cout_g = c // groups, n // groups
    g = torch.Generator(device=DEV).manual_seed(c)
    if pattern == "all_255":
        cw = _bound_weights(c, n, groups, k, DEV)
        ca = torch.full((bsz, c, h, w), 255, device=DEV)
    else:
        cw = torch.randint(0, 2, (n, cin_g, kh, kw), generator=g, device=DEV) * 255
        ca = torch.randint(0, 2, (bsz, c, h, w), generator=g, device=DEV) * 255
    f64 = dict(dtype=torch.float64, device=DEV)
    sw = torch.exp2(torch.randint(-12, -8, (n,), generator=g, device=DEV).to(torch.float64)
                    + torch.rand(n, generator=g, device=DEV, dtype=torch.float64))
    zpw = -torch.rand(n, generator=g, device=DEV, dtype=torch.float64) * 0.2
    ch = torch.arange(n, device=DEV)
    exact = ch % cout_g < 2
    sw[exact] = 2.0 ** -10
    zpw[exact] = -(255 - (ch[exact] % 2)).double() * 2.0 ** -10
    L = ops.int_layer_operands(cw, sw, zpw, 2.0 ** -8, 0.0, None, 255, 255, groups, dil)
    codes = torch.zeros(bsz, h, w, L.cp, dtype=torch.uint8, device=DEV)
    codes[..., :c] = ca.permute(0, 2, 3, 1).to(torch.uint8)
    y = ops.int_conv2d(codes, L, 1, pad)
    _check_bar(y, ca, L, cw, 1, pad)
    if pattern == "all_255":
        taps = F.conv2d(torch.ones(bsz, 1, h, w, **f64), torch.ones(1, 1, kh, kw, **f64), padding=pad,
                        dilation=dil)[:, 0]
        sa_ref = 255 * cin_g * taps
        assert float(255 * sa_ref.max()) == kh * kw * cin_g * 65025 < 2 ** 31
        even, odd = exact & (ch % 2 == 0), exact & (ch % 2 == 1)
        assert bool((y[:, even] == 0).all()), "S != 255 SA"
        assert torch.equal(y[:, odd].double(), (2.0 ** -18 * sa_ref)[:, None].expand(-1, int(odd.sum()), -1, -1)), \
            "SA wrong"


# ---------------------------------------------------------------------------------------------
# bit-for-bit identities between the kernels
# ---------------------------------------------------------------------------------------------
def _epilogue_args(shape, seed, fused):
    """(residual, activation, code operands) of the plain or the fused comparison."""
    if not fused:
        return dict(residual=None, activation=None, code_params=None)
    b, n, ho, wo = shape
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = torch.randn(b, ho, wo, n, generator=g, device=DEV).permute(0, 3, 1, 2)
    return dict(residual=r, activation="leaky_relu", code_params=_act_operands(16, True, seed))


def _fused(codes, L, stride, pad, e):
    slope = 0.125 if e["activation"] == "leaky_relu" else None
    return ops.int_conv2d_fused(codes, L, stride, pad, residual=e["residual"], activation=e["activation"],
                                negative_slope=slope, code_params=e["code_params"])


def _assert_same(got, want):
    assert torch.equal(_i32(got[0]), _i32(want[0]))
    assert (got[1] is None) == (want[1] is None)
    if got[1] is not None:
        assert torch.equal(got[1], want[1])


def _same_operands(La, Lb, idx, h, w, stride, pad):
    """Channels ``idx`` of La have Lb's alpha, beta and constant table, bit for bit."""
    assert torch.equal(La.alpha[idx], Lb.alpha) and torch.equal(La.beta[idx], Lb.beta)
    ta, tb = La.pattern_tables(h, w, stride, pad), Lb.pattern_tables(h, w, stride, pad)
    assert torch.equal(ta[0], tb[0]) and torch.equal(ta[1], tb[1]) and ta[2] == tb[2]
    assert torch.equal(ta[3][:, idx], tb[3])


DENSE_CASES = OP_CASES + [(2, 7, 6, 24, n, (3, 3), (1, 1), (1, 1), 8, 256) for n in N_SWEEP]


@gpu
@pytest.mark.parametrize("case", DENSE_CASES)
@pytest.mark.parametrize("fused", [False, True])
def test_grouped_kernel_equals_dense_kernel(case, fused):
    """groups = 1, dilation = 1 through mhaq_fq_iconv_grouped_u8 with the grouped weight operand,
    against the dense entries (fq_iconv_kernel<false> plain, <true> fused) on the same operands."""
    bsz, h, w, c, n, k, stride, pad, w_bits, levels = case
    seed = hash(case) & 0xFFFF
    L, cw = _layer(n, c, 1, k, 1, w_bits, levels, seed)
    assert L.dense
    _, codes = _codes(bsz, h, w, c, levels, seed + 1)
    ho, wo = L.out_size(h, w, stride, pad)
    e = _epilogue_args((bsz, n, ho, wo), seed, fused)
    want = _fused(codes, L, stride, pad, e) if fused else (ops.int_conv2d(codes, L, stride, pad), None)
    y = torch.empty_like(want[0])
    cod = torch.empty_like(want[1]) if fused else None
    _grouped_launch(codes, L, ops.iconv_grouped_weight_operand(cw, 1), stride, pad, y, cod, e["residual"],
                    e["activation"], e["code_params"])
    _assert_same((y, cod), want)


SPLIT_CASES = [case[:9] + case[10:] for case in GCASES if _pair2(case[9]) == (1, 1)] + [
    (2, 6, 5, c, n, groups, 3, 1, 1, 4, 16) for c, n, groups, dil, *_ in PLAN_CASES if dil == 1]


@gpu
@pytest.mark.parametrize("case", SPLIT_CASES)
@pytest.mark.parametrize("fused", [False, True])
def test_grouped_layer_equals_its_groups_as_dense_layers(case, fused):
    """Each group run as a dense layer on its slice of the input codes (repacked to
    code_channels(cin_g)), the outputs concatenated along N."""
    bsz, h, w, c, n, groups, k, stride, pad, w_bits, levels = case
    stride, pad = _pair2(stride), _pair2(pad)
    seed = hash(case) & 0xFFFF
    L, cw = _layer(n, c, groups, k, 1, w_bits, levels, seed)
    _, codes = _codes(bsz, h, w, c, levels, seed + 1)
    ho, wo = L.out_size(h, w, stride, pad)
    e = _epilogue_args((bsz, n, ho, wo), seed, fused)
    got = _fused(codes, L, stride, pad, e)
    cin_g, cout_g = c // groups, n // groups
    ys, cods = [], []
    for gi in range(groups):
        sl = slice(gi * cout_g, (gi + 1) * cout_g)
        Lg = ops.int_layer_operands(cw[sl], L.sw[sl], L.zpw[sl], L.sa, L.zpa, L.bias[sl], L.a_top, L.w_top)
        assert Lg.dense
        _same_operands(L, Lg, sl, h, w, stride, pad)
        cg = torch.zeros(bsz, h, w, ops.code_channels(cin_g), dtype=torch.uint8, device=DEV)
        cg[..., :cin_g] = codes[..., gi * cin_g:(gi + 1) * cin_g]
        eg = dict(e, residual=None if e["residual"] is None else e["residual"][:, sl])
        yg, cdg = _fused(cg, Lg, stride, pad, eg)
        ys.append(yg)
        cods.append(None if cdg is None else cdg[..., :cout_g])
    want_codes = None
    if fused:
        want_codes = torch.zeros_like(got[1])
        want_codes[..., :n] = torch.cat(cods, -1)
    _assert_same(got, (torch.cat(ys, 1), want_codes))


MULT_CASES = [case for case in DW_CASES if not hasattr(case, "id")]       # the per-axis depthwise rows


@gpu
@pytest.mark.parametrize("ci", range(len(MULT_CASES)))
@pytest.mark.parametrize("fused", [False, True])
def test_channel_multiplier_equals_interleaved_depthwise_layers(ci, fused):
    """groups = C, N = mult * C on the tensor cores against mult depthwise layers on the CUDA cores
    with weights cw[j::mult], output channel g * mult + j = channel g of layer j."""
    bsz, h, w, c, k, stride, pad, dil, w_bits, levels = MULT_CASES[ci]
    mult = 2 + ci % 2
    n = mult * c
    seed = 4000 + ci
    L, cw = _layer(n, c, c, k, dil, w_bits, levels, seed)
    assert _plan(c, n, *k, c)[0][0] >= 1                              # the tensor-core kernel
    _, codes = _codes(bsz, h, w, c, levels, seed + 1)
    ho, wo = L.out_size(h, w, stride, pad)
    e = _epilogue_args((bsz, n, ho, wo), seed, fused)
    got = _fused(codes, L, stride, pad, e)
    want_y = torch.empty_like(got[0])
    want_codes = torch.zeros_like(got[1]) if fused else None
    for j in range(mult):
        Lj = ops.int_layer_operands(cw[j::mult], L.sw[j::mult], L.zpw[j::mult], L.sa, L.zpa, L.bias[j::mult],
                                    L.a_top, L.w_top, c, dil)
        assert _plan(c, c, *k, c)[0][0] == 0                          # the CUDA-core kernel
        _same_operands(L, Lj, slice(j, None, mult), h, w, stride, pad)
        ej = dict(e, residual=None if e["residual"] is None else e["residual"][:, j::mult])
        yj, cj = _fused(codes, Lj, stride, pad, ej)
        want_y[:, j::mult] = yj
        if fused:
            want_codes[..., j:n:mult] = cj[..., :c]
    _assert_same(got, (want_y, want_codes))
