// fq_igemm.cuh — integer layers: activation codes and an int8 tensor-core implicit-GEMM convolution
// (included by mhaq_fq.cu after fq_pack.cuh).
//
// fq_act_codes_kernel: fp32 activations (channels_last NCHW, i.e. storage order NHWC, or a
// [B, in] matrix) -> uint8 codes [pixels][cp], cp = round_up(C, 16), padding channels code 0.  Each
// code is the forward's own rint(v) (fwd_pair_fast / fwd_elem with the forward's fast / general
// split), saturated to [0, 255] and counted like fq_pack_kernel.  Flat grid: one thread per 4
// consecutive output codes, which always share a pixel (cp % 16 == 0).
//
// fq_iconv_kernel: y[m][n] = alpha[n] * S[m][n] + beta[n] * SA[m] + ctab[p(m)][n] (DESIGN §3,
// "Integer layers"), with S = sum_k ca_k * cw_nk on the tensor cores (tcgen05.mma kind::i8,
// unsigned x unsigned -> int32 in tensor memory) and SA = sum_k ca_k from an all-ones row that
// every N tile of the weight operand carries after its real output channels.
//   M = output pixels (128 per CTA), K = (kh, kw, cp) with the channels contiguous, 128 bytes
//   per pipeline stage, N = one tile of the weight operand (tile_n <= 256 rows, see
//   iconv_layout).  Grid (ceil(M / 128), n_tiles), 160 threads:
//     warps 0-3  producers: gather the A rows of a stage with 16-byte cp.async (src-size 0
//                zero-fills padding taps and rows past M) and copy the stage's B block; after
//                cp.async.wait_group each thread fences the writes into the async proxy and
//                arrives on the stage's "full" barrier.  Then they are the epilogue: one TMEM lane
//                (= one output pixel) per thread, 16 columns per tcgen05.ld.
//     warp 4     allocates the accumulator columns; one lane waits "full", issues the stage's
//                4 MMAs (K = 32 bytes each) and tcgen05.commits to the stage's "empty" barrier,
//                and after the last stage to the "accumulator ready" barrier.
//   Shared-memory operands use the no-swizzle K-major canonical layout: 8 rows x 16 bytes core
//   matrices, offset(r, c) = (r / 8) * 1024 + c * 128 + (r % 8) * 16 for row r and 16-byte K
//   chunk c of a stage (LBO = 128 B between K-adjacent core matrices, SBO = 1024 B between 8-row
//   groups).  The weight operand is stored in global memory already in this order, one
//   [tile_n x 128 B] block per (tile, stage), so its copy is a linear one.  A producer warp's
//   16-byte writes land in four 128-byte core matrices: conflict-free, no swizzle needed.
// No host synchronisation, allocation or atomic in either kernel (graph-capturable); 64-bit offsets.
// Included inside the anonymous namespace of mhaq_fq.cu: uses fwd_pair_fast / fwd_elem / absmax4,
// sat_code and flush_count.

constexpr int kIcTileM = 128;          // output pixels per CTA (MMA M)
constexpr int kIcStageK = 128;         // bytes of K per stage (8 chunks of 16)
constexpr int kIcStages = 4;
constexpr int kIcLag = 2;              // stages a producer keeps in flight before it signals one
constexpr int kIcThreads = 160;        // 4 producer / epilogue warps + 1 MMA warp
constexpr int kIcMaxTileN = 256;
constexpr int kIcAStage = kIcTileM * kIcStageK;   // 16 KiB

// N tiling of the weight operand: n_tiles tiles of tile_n rows; tile t holds output channels
// [t * tile_out, min(n_out, (t + 1) * tile_out)) (tile_out <= 255, no tile empty), then the
// all-ones row at local row tile_out, then zero rows up to tile_n (a multiple of 16, <= 256: the
// MMA's N).
struct IcLayout {
    int n_tiles, tile_n, tile_out;
    int64_t k_stages;
};
__host__ __device__ inline IcLayout iconv_layout(int64_t n_out, int64_t k_bytes) {
    IcLayout l;
    // at most kIcMaxTileN - 1 output channels per tile, so the ones row always fits; then as
    // few tiles of that width as cover n_out (none of them empty)
    const int64_t n_min = (n_out + kIcMaxTileN - 2) / (kIcMaxTileN - 1);
    l.tile_out = (int)((n_out + n_min - 1) / n_min);
    l.n_tiles = (int)((n_out + l.tile_out - 1) / l.tile_out);
    l.tile_n = (l.tile_out + 1 + 15) / 16 * 16;
    l.k_stages = (k_bytes + kIcStageK - 1) / kIcStageK;
    return l;
}

// N tiling of a grouped (or dilated, one-group) weight operand: a pure function of (n_out, groups,
// cin_g, kh, kw).  When a group and its ones row fit one tile (cout_g + 1 <= 256), a tile holds gpt
// whole groups: tile_out = gpt * cout_g output channels, then gpt ones rows (local row tile_out + i
// for the tile's i-th group), tile_out + gpt <= 256 rounded up to 16.  Otherwise every group spans
// `parts` tiles of at most 255 channels and one ones row, one group per tile (gpt = 1).  A tile's K
// is (kh, kw, its groups' input channels rounded out to 16-channel chunks), so the tiles' K widths
// differ; every tile runs the widest tile's k_stages with the rest zero-filled.
struct IgPlan {
    int n_tiles, tile_n, tile_out, gpt, parts;
    int64_t k_stages;
};
// Output channels [n_base, n_base + n_here), groups [g_lo, g_lo + n_grp) and 16-channel input chunks
// [c_lo, c_lo + kc) of one tile.
struct IgTile {
    int64_t n_base, n_here, g_lo, c_lo, kc;
    int n_grp;
};
__host__ __device__ inline IgTile igroup_tile(int64_t groups, int64_t cin_g, int64_t cout_g, int tile_out, int gpt,
                                              int parts, int tile) {
    IgTile t;
    int64_t g_hi, n_end;
    if (parts == 1) {
        t.g_lo = (int64_t)tile * gpt;
        g_hi = t.g_lo + gpt < groups ? t.g_lo + gpt : groups;
        t.n_base = t.g_lo * cout_g;
        n_end = g_hi * cout_g;
    } else {
        t.g_lo = tile / parts;
        g_hi = t.g_lo + 1;
        t.n_base = t.g_lo * cout_g + (int64_t)(tile % parts) * tile_out;
        n_end = t.n_base + tile_out < g_hi * cout_g ? t.n_base + tile_out : g_hi * cout_g;
    }
    t.n_here = n_end - t.n_base;
    t.n_grp = (int)(g_hi - t.g_lo);
    t.c_lo = t.g_lo * cin_g / 16;
    t.kc = (g_hi * cin_g + 15) / 16 - t.c_lo;
    return t;
}
inline IgPlan igroup_plan(int64_t n_out, int64_t groups, int64_t cin_g, int kh, int kw) {
    IgPlan l;
    const int64_t cout_g = n_out / groups;
    if (cout_g + 1 <= kIcMaxTileN) {
        // as many whole groups as fit, then as few tiles of that many groups as cover them all
        int64_t gpt = kIcMaxTileN / (cout_g + 1);
        if (gpt > groups) gpt = groups;
        const int64_t nt = (groups + gpt - 1) / gpt;
        l.gpt = (int)((groups + nt - 1) / nt);
        l.n_tiles = (int)((groups + l.gpt - 1) / l.gpt);
        l.parts = 1;
        l.tile_out = (int)(l.gpt * cout_g);
    } else {
        const int64_t p_min = (cout_g + kIcMaxTileN - 2) / (kIcMaxTileN - 1);
        l.tile_out = (int)((cout_g + p_min - 1) / p_min);
        l.parts = (int)((cout_g + l.tile_out - 1) / l.tile_out);
        l.gpt = 1;
        l.n_tiles = (int)(groups * l.parts);
    }
    l.tile_n = (l.tile_out + l.gpt + 15) / 16 * 16;
    int64_t kc_max = 0;
    for (int t = 0; t < l.n_tiles; ++t) {
        const IgTile g = igroup_tile(groups, cin_g, cout_g, l.tile_out, l.gpt, l.parts, t);
        if (g.kc > kc_max) kc_max = g.kc;
    }
    l.k_stages = ((int64_t)kh * kw * kc_max + 7) / 8;
    return l;
}

// ---------------------------------------------------------------------------------------------
// activation codes
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
fq_act_codes_kernel(const float *__restrict__ x, uint8_t *__restrict__ codes, QParams prm,
                    int64_t n_pix, int64_t c, int64_t cp, bool vec, unsigned long long *__restrict__ n_oor) {
    const QConst q = load_qconst(prm, 0);
    const Div2 dv = make_div2(q.s, __frcp_rn(q.s));
    const f32x2 zpn = bc2(-q.zp), zp2 = bc2(q.zp);
    const bool fast_ok = scale_fast_ok(q.s);
    const int64_t groups_per_pix = cp / 4;
    const int64_t n_groups = n_pix * groups_per_pix;
    uint32_t bad = 0;
    for (int64_t g = (int64_t)blockIdx.x * kThreads + threadIdx.x; g < n_groups;
         g += (int64_t)gridDim.x * kThreads) {
        const int64_t pix = g / groups_per_pix;
        const int64_t ch = (g - pix * groups_per_pix) * 4;
        const float *xp = x + pix * c + ch;
        const int nv = ch + 4 <= c ? 4 : (ch < c ? (int)(c - ch) : 0);
        float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (vec && nv == 4) {
            xv = ld_stream4(xp);
        } else {
            if (nv > 0) xv.x = __ldg(xp);
            if (nv > 1) xv.y = __ldg(xp + 1);
            if (nv > 2) xv.z = __ldg(xp + 2);
            if (nv > 3) xv.w = __ldg(xp + 3);
        }
        float4 cv, yv;
        if (fast_ok && !(absmax4(0.f, xv) > kXHi)) {
            fwd_pair_fast<true>(xv.x, xv.y, q, dv, zpn, zp2, yv.x, yv.y, cv.x, cv.y);
            fwd_pair_fast<true>(xv.z, xv.w, q, dv, zpn, zp2, yv.z, yv.w, cv.z, cv.w);
        } else {
            (void)fwd_elem(xv.x, q, cv.x);
            (void)fwd_elem(xv.y, q, cv.y);
            (void)fwd_elem(xv.z, q, cv.z);
            (void)fwd_elem(xv.w, q, cv.w);
        }
        (void)yv;
        const uint32_t c0 = nv > 0 ? sat_code<8>(cv.x, bad) : 0u;
        const uint32_t c1 = nv > 1 ? sat_code<8>(cv.y, bad) : 0u;
        const uint32_t c2 = nv > 2 ? sat_code<8>(cv.z, bad) : 0u;
        const uint32_t c3 = nv > 3 ? sat_code<8>(cv.w, bad) : 0u;
        *reinterpret_cast<uint32_t *>(codes + pix * cp + ch) = (uint32_t)pack4<8>(c0, c1, c2, c3);
    }
    flush_count(bad, n_oor);
}

// ---------------------------------------------------------------------------------------------
// tcgen05 / cp.async primitives (the mbarrier helpers are mhaq_fq.cu's)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// shared-memory matrix descriptor: K-major, no swizzle (layout type 0), version 1 (bit 46)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor of kind::i8: D = s32 (bits 4-5 = 2), A = B = u8 (bits 7-9, 10-12 = 0),
// both K-major, N >> 3 at bits 17-22, M >> 4 at bits 24-28
__host__ __device__ constexpr uint32_t idesc_i8(int m, int n) {
    return (2u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
        "l"(a), "l"(b), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, uint32_t &v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// implicit-GEMM convolution
// ---------------------------------------------------------------------------------------------
struct IConvArgs {
    const uint8_t *a;          // codes [batch * h * w][cp]
    const uint8_t *b;          // weight operand [n_tiles][k_stages][tile_n * 128]
    const float *alpha, *beta; // [n_out]
    const float *ctab;         // [n_hcls * n_wcls][n_out]
    const int32_t *hcls, *wcls;   // [ho], [wo]
    float *y;                  // [m][n_out]
    int64_t m, h, w, cp, n_out, ho, wo, k_chunks, k_stages;
    int kh, kw, sh, sw, ph, pw, n_wcls, tile_n, tile_out, tmem_cols;
    int vec_out;               // y 16-byte aligned and n_out % 4 == 0: float4 stores
    // fused epilogue (fq_iconv_kernel<true> only)
    const float *res;          // residual [m][n_out] or NULL
    uint8_t *codes;            // next layer's codes [m][cp_out] or NULL (y may then be NULL)
    const float *code_s, *code_zp, *code_hi;   // its per-tensor LINEAR operands
    int64_t cp_out;
    float slope;               // LeakyReLU negative slope
    int act;                   // kIcAct*
    int vec_res;               // res 16-byte aligned and n_out % 4 == 0: float4 loads
    // grouped / dilated layers (fq_iconv_kernel<true, true>, fq_idw_kernel)
    int dh, dw;                // dilation
    int64_t groups, cin_g, cout_g;
    int gpt, parts;            // IgPlan
};

constexpr int kIcActNone = 0, kIcActRelu = 1, kIcActLeaky = 2;   // = MHAQ_FQ_ACT_*

// Fused epilogue of one 16-column chunk: t = out (+ residual), activation, then fp32 and / or the
// next layer's codes.  relu keeps NaN and is fmaxf(t, 0) otherwise, as torch's CUDA clamp_min;
// LeakyReLU is t > 0 ? t : t * slope, as torch's CUDA leaky_relu.  The codes are the forward's
// rint(v) of t exactly as fq_act_codes_kernel forms them (fwd_pair_fast where its guard allows it,
// fwd_elem otherwise: bit-identical), saturated to [0, 255] with NaN -> 0 and not counted.
// The residual of a chunk, loaded before its accumulator columns are read so that the two
// latencies overlap (0 where nv or the row ends).
__device__ __forceinline__ void iconv_load_res(const IConvArgs &p, float (&r)[16], int64_t m, int64_t n0, int nv) {
    const float *rrow = p.res + m * p.n_out + n0;
    if (p.vec_res && (n0 & 3) == 0 && nv == 16) {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(rrow + i));
            r[i] = v.x; r[i + 1] = v.y; r[i + 2] = v.z; r[i + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = i < nv ? __ldg(rrow + i) : 0.f;
    }
}

__device__ __forceinline__ void iconv_fused_chunk(const IConvArgs &p, float (&out)[16], const float (&r)[16],
                                                  int64_t m, int64_t n0, int nv, bool vec, const QConst &q,
                                                  const Div2 &dv, f32x2 zpn, f32x2 zp2, bool fast_ok) {
    if (p.res) {
#pragma unroll
        for (int i = 0; i < 16; ++i) out[i] = __fadd_rn(out[i], r[i]);
    }
    if (p.act == kIcActRelu) {
#pragma unroll
        for (int i = 0; i < 16; ++i) out[i] = isnan(out[i]) ? out[i] : fmaxf(out[i], 0.f);
    } else if (p.act == kIcActLeaky) {
#pragma unroll
        for (int i = 0; i < 16; ++i) out[i] = out[i] > 0.f ? out[i] : __fmul_rn(out[i], p.slope);
    }
    if (p.y) {
        float *yrow = p.y + m * p.n_out + n0;
        if (vec && nv == 16) {
#pragma unroll
            for (int i = 0; i < 16; i += 4)
                *reinterpret_cast<float4 *>(yrow + i) = make_float4(out[i], out[i + 1], out[i + 2], out[i + 3]);
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < nv) yrow[i] = out[i];
        }
    }
    if (p.codes) {
        uint32_t c[16], bad = 0;
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
            float c0, c1, y0, y1;
            if (fast_ok && !(fmaxf(fabsf(out[i]), fabsf(out[i + 1])) > kXHi)) {
                fwd_pair_fast<true>(out[i], out[i + 1], q, dv, zpn, zp2, y0, y1, c0, c1);
            } else {
                (void)fwd_elem(out[i], q, c0);
                (void)fwd_elem(out[i + 1], q, c1);
            }
            c[i] = sat_code<8>(c0, bad);
            c[i + 1] = sat_code<8>(c1, bad);
        }
        uint8_t *crow = p.codes + m * p.cp_out + n0;
        if (nv == 16 && (n0 & 15) == 0) {
            uint4 w;
            w.x = (uint32_t)pack4<8>(c[0], c[1], c[2], c[3]);
            w.y = (uint32_t)pack4<8>(c[4], c[5], c[6], c[7]);
            w.z = (uint32_t)pack4<8>(c[8], c[9], c[10], c[11]);
            w.w = (uint32_t)pack4<8>(c[12], c[13], c[14], c[15]);
            *reinterpret_cast<uint4 *>(crow) = w;
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < nv) crow[i] = (uint8_t)c[i];
        }
    }
}

// FUSED = false: y = alpha * S + beta * SA + C, fp32 only (mhaq_fq_iconv_u8).  FUSED = true: the
// same value through iconv_fused_chunk (mhaq_fq_iconv_fused_u8); the tile holding the last output
// channels also writes the codes' padding channels [n_out, cp_out) as 0.
// GROUPED = true (with FUSED, mhaq_fq_iconv_grouped_u8): block-diagonal N tiles of IgPlan.  The
// producers gather only the tile's input chunks [c_lo, c_lo + kc) of each tap, at dilated tap
// offsets; the epilogue reads channel n's SA from the ones column of its group, which it first
// copies from tensor memory into the (then idle) A stages, [group][row].
template <bool FUSED, bool GROUPED = false>
__global__ void __launch_bounds__(kIcThreads, 1)
fq_iconv_kernel(const IConvArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int b_stage = p.tile_n * kIcStageK;
    uint8_t *sa = smem;                                   // kIcStages x 16 KiB
    uint8_t *sb = smem + kIcStages * kIcAStage;           // kIcStages x tile_n * 128
    uint64_t *bars = reinterpret_cast<uint64_t *>(sb + kIcStages * b_stage);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kIcStages + 1);
    uint64_t *full = bars, *empty = bars + kIcStages, *accum = bars + 2 * kIcStages;
    const int64_t m0 = (int64_t)blockIdx.x * kIcTileM;
    const int tile = blockIdx.y;

    if (tid == 0) {
        for (int s = 0; s < kIcStages; ++s) {
            mbar_init(full + s, 128);
            mbar_init(empty + s, 1);
        }
        mbar_init(accum, 1);
        mbar_fence_init();
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp < 4) {
        // ---------------- producers ----------------
        // thread -> rows rr and rr + 64, 16-byte chunks 2j + sub (j = 0..3) of each stage: a warp's
        // accesses are 16 rows x 32 contiguous bytes in global memory, four whole core matrices in
        // shared memory
        const int sub = tid & 1, rr = tid >> 1;
        const uint8_t *row_base[2];
        int64_t hi0[2], wi0[2];
        bool row_ok[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int64_t m = m0 + rr + 64 * i;
            row_ok[i] = m < p.m;
            const int64_t mm = row_ok[i] ? m : 0;
            const int64_t img = mm / (p.ho * p.wo), rem = mm - img * (p.ho * p.wo);
            const int64_t oh = rem / p.wo, ow = rem - oh * p.wo;
            hi0[i] = oh * p.sh - p.ph;
            wi0[i] = ow * p.sw - p.pw;
            row_base[i] = p.a + img * p.h * p.w * p.cp;
        }
        [[maybe_unused]] IgTile gt{};
        if constexpr (GROUPED) gt = igroup_tile(p.groups, p.cin_g, p.cout_g, p.tile_out, p.gpt, p.parts, tile);
        const int64_t cpc = GROUPED ? gt.kc : p.cp / 16;        // 16-byte chunks per tap
        [[maybe_unused]] const int64_t g_chunks = GROUPED ? (int64_t)p.kh * p.kw * gt.kc : 0;
        const uint8_t *bsrc = p.b + (int64_t)tile * p.k_stages * b_stage;
        for (int64_t kt = 0; kt < p.k_stages; ++kt) {
            const int s = (int)(kt % kIcStages);
            if (kt >= kIcStages) mbar_wait(empty + s, (uint32_t)((kt / kIcStages - 1) & 1));
            const uint32_t a_dst = smem_u32(sa + s * kIcAStage), b_dst = smem_u32(sb + s * b_stage);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = 2 * j + sub;
                const int64_t q = kt * 8 + c;               // global 16-byte chunk of K
                const int64_t tap = q / cpc, cc = q - tap * cpc + (GROUPED ? gt.c_lo : 0);
                const int64_t tkh = tap / p.kw, tkw = tap - tkh * p.kw;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int r = rr + 64 * i;
                    const int64_t ih = hi0[i] + (GROUPED ? tkh * p.dh : tkh), iw = wi0[i] + (GROUPED ? tkw * p.dw : tkw);
                    const bool ok = row_ok[i] && q < (GROUPED ? g_chunks : p.k_chunks) && ih >= 0 && ih < p.h &&
                                    iw >= 0 && iw < p.w;
                    const uint8_t *src = ok ? row_base[i] + ((ih * p.w + iw) * p.cp + cc * 16) : p.a;
                    cp_async16(a_dst + (r >> 3) * 1024 + c * 128 + (r & 7) * 16, src, ok ? 16 : 0);
                }
            }
            const uint8_t *bs = bsrc + kt * b_stage;
            for (int o = tid * 16; o < b_stage; o += 128 * 16) cp_async16(b_dst + o, bs + o, 16);
            cp_async_commit();
            if (kt >= kIcLag) {
                cp_async_wait<kIcLag>();
                fence_proxy_async();
                mbar_arrive(full + (kt - kIcLag) % kIcStages);
            }
        }
        cp_async_wait<0>();
        fence_proxy_async();
        for (int64_t kt = p.k_stages > kIcLag ? p.k_stages - kIcLag : 0; kt < p.k_stages; ++kt)
            mbar_arrive(full + kt % kIcStages);

        // ---------------- epilogue ----------------
        mbar_wait(accum, 0);
        tc_fence_after();
        const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
        [[maybe_unused]] uint32_t sa_u;
        [[maybe_unused]] uint32_t *sas = reinterpret_cast<uint32_t *>(sa);
        if constexpr (GROUPED) {
            // the ones columns tile_out + [0, n_grp) -> sas[group][row]; the MMAs that read the A
            // stages are complete (accum), so the stages are free.  A 16-column load starts at most
            // at tile_n - 16 so that it stays inside the tile's columns.
            for (int g0 = 0; g0 < gt.n_grp; g0 += 16) {
                const int base = p.tile_out + g0 < p.tile_n - 16 ? p.tile_out + g0 : p.tile_n - 16;
                uint32_t v[16];
                tmem_ld16(lane_addr + base, v);
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int g = base - p.tile_out + i;
                    if (g >= g0 && g < gt.n_grp) sas[g * kIcTileM + tid] = v[i];
                }
            }
        } else {
            tmem_ld1(lane_addr + p.tile_out, sa_u);
            tmem_wait_ld();
        }
        const int64_t m = m0 + tid;                  // TMEM lane tid = row tid of the tile
        const bool live = m < p.m;
        int64_t ctab_row = 0;
        if (live) {
            const int64_t rem = m % (p.ho * p.wo);
            const int64_t oh = rem / p.wo, ow = rem - oh * p.wo;
            ctab_row = ((int64_t)__ldg(p.hcls + oh) * p.n_wcls + __ldg(p.wcls + ow)) * p.n_out;
        }
        [[maybe_unused]] const double sa_d = GROUPED ? 0.0 : (double)sa_u;
        const int64_t n_base = GROUPED ? gt.n_base : (int64_t)tile * p.tile_out;
        const int64_t n_here =
            GROUPED ? gt.n_here : ((p.n_out - n_base) < p.tile_out ? (p.n_out - n_base) : p.tile_out);
        float *yrow = p.y + m * p.n_out + n_base;
        const bool vec = p.vec_out && (n_base & 3) == 0;
        QConst cq{};
        Div2 cdv{};
        f32x2 czpn{}, czp2{};
        bool cfast = false;
        if constexpr (FUSED) {
            if (p.codes) {
                const QParams prm = {p.code_s, p.code_zp, p.code_zp, p.code_hi, 0, 0, 0, 0, PARAMS_LINEAR};
                cq = load_qconst(prm, 0);
                cdv = make_div2(cq.s, __frcp_rn(cq.s));
                czpn = bc2(-cq.zp);
                czp2 = bc2(cq.zp);
                cfast = scale_fast_ok(cq.s);
            }
        }
        for (int col = 0; col < n_here; col += 16) {
            uint32_t v[16];
            [[maybe_unused]] float rv[16];
            if constexpr (FUSED) {
                if (p.res && live) iconv_load_res(p, rv, m, n_base + col, n_here - col < 16 ? (int)(n_here - col) : 16);
            }
            tmem_ld16(lane_addr + col, v);
            tmem_wait_ld();
            if (!live) continue;
            float out[16];
            [[maybe_unused]] int64_t gq = 0, gr = 0;     // the column's group within the tile, and its rank in it
            if constexpr (GROUPED) {
                gq = col / p.cout_g;
                gr = col - gq * p.cout_g;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int64_t n = n_base + col + i;
                if (col + i < n_here) {
                    // fp64: alpha * S and beta * SA carry at most one rounding each, the result one
                    const double sa_n = GROUPED ? (double)sas[gq * kIcTileM + tid] : sa_d;
                    const double t = __fma_rn((double)__ldg(p.beta + n), sa_n, (double)__ldg(p.ctab + ctab_row + n));
                    out[i] = __double2float_rn(__fma_rn((double)__ldg(p.alpha + n), (double)(int32_t)v[i], t));
                } else {
                    out[i] = 0.f;
                }
                if constexpr (GROUPED) {
                    if (++gr == p.cout_g) {
                        gr = 0;
                        ++gq;
                    }
                }
            }
            if constexpr (FUSED) {
                const int nv = n_here - col < 16 ? (int)(n_here - col) : 16;
                iconv_fused_chunk(p, out, rv, m, n_base + col, nv, vec, cq, cdv, czpn, czp2, cfast);
            } else if (vec && col + 16 <= n_here) {
#pragma unroll
                for (int i = 0; i < 16; i += 4)
                    *reinterpret_cast<float4 *>(yrow + col + i) = make_float4(out[i], out[i + 1], out[i + 2], out[i + 3]);
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (col + i < n_here) yrow[col + i] = out[i];
            }
        }
        if constexpr (FUSED) {
            if (p.codes && live && tile == (int)gridDim.y - 1)
                for (int64_t n = p.n_out; n < p.cp_out; ++n) p.codes[m * p.cp_out + n] = 0;
        }
    } else if (tid == 128) {
        // ---------------- MMA issuer ----------------
        const uint32_t idesc = idesc_i8(kIcTileM, p.tile_n);
        for (int64_t kt = 0; kt < p.k_stages; ++kt) {
            const int s = (int)(kt % kIcStages);
            mbar_wait(full + s, (uint32_t)((kt / kIcStages) & 1));
            tc_fence_after();
            const uint32_t a_addr = smem_u32(sa + s * kIcAStage), b_addr = smem_u32(sb + s * b_stage);
#pragma unroll
            for (int j = 0; j < kIcStageK / 32; ++j)
                mma_i8(tmem, smem_desc(a_addr + j * 256, 128, 1024), smem_desc(b_addr + j * 256, 128, 1024),
                       idesc, (kt > 0 || j > 0) ? 1u : 0u);
            mma_commit(empty + s);
        }
        mma_commit(accum);
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(p.tmem_cols) : "memory");
    }
}

inline size_t iconv_smem_bytes(int tile_n) {
    return (size_t)kIcStages * (kIcAStage + tile_n * kIcStageK) + (2 * kIcStages + 1) * 8 + 16;
}

// ---------------------------------------------------------------------------------------------
// depthwise convolution on the CUDA cores (groups == cin == n_out)
// ---------------------------------------------------------------------------------------------
// One channel's sum has only kh * kw terms, so block-diagonal MMA tiles would multiply zeros almost
// everywhere.  Instead one thread per (output pixel, 16-channel chunk) loads one 16-byte code
// vector and one 16-byte weight vector per valid tap and accumulates S and SA of its 16 channels
// in int32; the weight operand is u8 [kh * kw][cp].  Consecutive threads take consecutive chunks
// of one pixel, so a warp's code loads are contiguous.  The epilogue is fq_iconv_kernel<true>'s:
// the same fp64 sum, then iconv_fused_chunk.  Grid-stride, 64-bit offsets; no host
// synchronisation, allocation or atomic.
constexpr int kDwThreads = 256;

__device__ __forceinline__ void dw_acc4(uint32_t a, uint32_t w, int32_t *s, int32_t *sa) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int32_t av = (int32_t)((a >> (8 * j)) & 0xffu), wv = (int32_t)((w >> (8 * j)) & 0xffu);
        s[j] += av * wv;
        sa[j] += av;
    }
}

__global__ void __launch_bounds__(kDwThreads)
fq_idw_kernel(const IConvArgs p) {
    const int64_t cpc = p.cp / 16;
    const int64_t total = p.m * cpc;
    QConst cq{};
    Div2 cdv{};
    f32x2 czpn{}, czp2{};
    bool cfast = false;
    if (p.codes) {
        const QParams prm = {p.code_s, p.code_zp, p.code_zp, p.code_hi, 0, 0, 0, 0, PARAMS_LINEAR};
        cq = load_qconst(prm, 0);
        cdv = make_div2(cq.s, __frcp_rn(cq.s));
        czpn = bc2(-cq.zp);
        czp2 = bc2(cq.zp);
        cfast = scale_fast_ok(cq.s);
    }
    for (int64_t t = (int64_t)blockIdx.x * kDwThreads + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * kDwThreads) {
        const int64_t m = t / cpc, ck = t - m * cpc;
        const int64_t img = m / (p.ho * p.wo), rem = m - img * (p.ho * p.wo);
        const int64_t oh = rem / p.wo, ow = rem - oh * p.wo;
        const int64_t hi0 = oh * p.sh - p.ph, wi0 = ow * p.sw - p.pw;
        const uint8_t *abase = p.a + img * p.h * p.w * p.cp + ck * 16;
        const uint8_t *wbase = p.b + ck * 16;
        int32_t s[16], sa[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) s[i] = sa[i] = 0;
        for (int th = 0; th < p.kh; ++th) {
            const int64_t ih = hi0 + (int64_t)th * p.dh;
            if (ih < 0 || ih >= p.h) continue;
            for (int tw = 0; tw < p.kw; ++tw) {
                const int64_t iw = wi0 + (int64_t)tw * p.dw;
                if (iw < 0 || iw >= p.w) continue;
                const uint4 av = __ldg(reinterpret_cast<const uint4 *>(abase + (ih * p.w + iw) * p.cp));
                const uint4 wv = __ldg(reinterpret_cast<const uint4 *>(wbase + (int64_t)(th * p.kw + tw) * p.cp));
                dw_acc4(av.x, wv.x, s, sa);
                dw_acc4(av.y, wv.y, s + 4, sa + 4);
                dw_acc4(av.z, wv.z, s + 8, sa + 8);
                dw_acc4(av.w, wv.w, s + 12, sa + 12);
            }
        }
        const int64_t n0 = ck * 16;
        const int nv = p.n_out - n0 < 16 ? (int)(p.n_out - n0) : 16;
        float rv[16];
        if (p.res) iconv_load_res(p, rv, m, n0, nv);
        const int64_t ctab_row = ((int64_t)__ldg(p.hcls + oh) * p.n_wcls + __ldg(p.wcls + ow)) * p.n_out;
        float out[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int64_t n = n0 + i;
            if (i < nv) {
                const double u = __fma_rn((double)__ldg(p.beta + n), (double)sa[i], (double)__ldg(p.ctab + ctab_row + n));
                out[i] = __double2float_rn(__fma_rn((double)__ldg(p.alpha + n), (double)s[i], u));
            } else {
                out[i] = 0.f;
            }
        }
        iconv_fused_chunk(p, out, rv, m, n0, nv, p.vec_out, cq, cdv, czpn, czp2, cfast);
        if (p.codes)
            for (int i = nv; i < 16; ++i) p.codes[m * p.cp_out + n0 + i] = 0;
    }
}
