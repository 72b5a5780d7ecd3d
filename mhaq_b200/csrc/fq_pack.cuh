// fq_pack.cuh — packed low-bit integer codes (included by mhaq_fq.cu after the forward kernel).
//
// Format (include/mhaq_fq.h, "Packed codes"): row r of the [n_rows][n_inner] storage-order view
// starts at byte r * row_stride, row_stride = round_up(ceil(n_inner * b / 8), 16); for b <= 8 code
// j sits in bits [(j*b) mod 8, +b) of byte floor(j*b/8), least-significant bit first; for b = 16
// it is a little-endian uint16 at byte 2j; padding is zero.
//
// fq_pack_kernel uses the forward's decomposition (make_task, load_qconst, 4096-element sub-tiles,
// the fast / general split with the |x| > 2^80 guard) and the forward's own device functions
// (fwd_pair_fast / fwd_elem), so a stored code IS the forward's rint(v).  In a warp iteration
// each lane holds 4 consecutive codes = 4b bits: b = 16 one 64-bit store, b = 8 one 32-bit store,
// b = 4 one 16-bit store, b = 2 one byte; b = 1 pairs neighbouring lanes with one shuffle and the
// even lane stores the byte.  Ragged tails, unaligned rows and unaligned code buffers take the
// byte-granular general path.  A code outside [0, 2^b - 1] (NaN included) is stored saturated
// (NaN -> 0) and counted; each CTA adds its count to the caller's counter with one integer atomic
// (no floating-point atomics anywhere).
// Included inside the anonymous namespace of mhaq_fq.cu: uses fwd_pair_fast / fwd_elem / absmax4.

__host__ __device__ constexpr int64_t packed_row_bytes(int64_t n_inner, int bits) {
    return ((n_inner * bits + 7) / 8 + 15) / 16 * 16;
}

// saturate a code to [0, 2^BITS - 1] (NaN -> 0: fmaxf returns the non-NaN operand); `bad`
// counts the codes that needed it
template <int BITS>
__device__ __forceinline__ uint32_t sat_code(float c, uint32_t &bad) {
    constexpr float kMax = (float)((1u << BITS) - 1u);
    bad += (c >= 0.f && c <= kMax) ? 0u : 1u;
    return (uint32_t)fminf(fmaxf(c, 0.f), kMax);
}

// 4 consecutive codes -> 4 * BITS bits, code 0 in the lowest bits
template <int BITS>
__device__ __forceinline__ uint64_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return (uint64_t)a | ((uint64_t)b << BITS) | ((uint64_t)c << (2 * BITS)) |
           ((uint64_t)d << (3 * BITS));
}

// Fast-path store of the 4 codes of element position p (p % 4 == 0) into a 16-byte aligned row.
// Every lane of the warp must call it (b = 1 shuffles).
template <int BITS>
__device__ __forceinline__ void store_packed4(uint8_t *pr, int64_t p, uint64_t w) {
    if (BITS == 16) {
        *reinterpret_cast<unsigned long long *>(pr + 2 * p) = w;
    } else if (BITS == 8) {
        *reinterpret_cast<uint32_t *>(pr + p) = (uint32_t)w;
    } else if (BITS == 4) {
        *reinterpret_cast<uint16_t *>(pr + p / 2) = (uint16_t)w;
    } else if (BITS == 2) {
        pr[p / 4] = (uint8_t)w;
    } else {
        const uint32_t hi = __shfl_down_sync(0xffffffffu, (uint32_t)w, 1);
        if (((threadIdx.x & 31) & 1) == 0) pr[p / 8] = (uint8_t)((uint32_t)w | (hi << 4));
    }
}

// General-path store: byte by byte, only the bytes holding one of the nv valid codes (the codes
// of invalid elements are 0, so a partly valid last byte gets zero bits).  All lanes call it.
template <int BITS>
__device__ __forceinline__ void store_packed4_bytes(uint8_t *pr, int64_t p, uint64_t w, int nv) {
    if constexpr (BITS == 1) {
        const uint32_t hi = __shfl_down_sync(0xffffffffu, (uint32_t)w, 1);
        if (((threadIdx.x & 31) & 1) == 0 && nv > 0) pr[p / 8] = (uint8_t)((uint32_t)w | (hi << 4));
    } else {
#pragma unroll
        for (int k = 0; k < BITS / 2; ++k)
            if (8 * k < nv * BITS) pr[p * BITS / 8 + k] = (uint8_t)(w >> (8 * k));
    }
}

__device__ __forceinline__ void flush_count(uint32_t bad, unsigned long long *n_oor) {
    __shared__ uint32_t s_bad[kThreads / 32];
    const uint32_t wsum = __reduce_add_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) s_bad[threadIdx.x >> 5] = wsum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long tot = 0;
        for (int w = 0; w < kThreads / 32; ++w) tot += s_bad[w];
        if (tot && n_oor) atomicAdd(n_oor, tot);
    }
}

template <int BITS, bool VEC, bool CLAMP>
__global__ void __launch_bounds__(kThreads)
fq_pack_kernel(const float *__restrict__ x, uint8_t *__restrict__ packed, QParams prm, Geom g,
               int64_t row_stride, unsigned long long *__restrict__ n_oor) {
    const int tid = threadIdx.x;
    uint32_t bad = 0;
    const int64_t data_bytes = (g.n_inner * BITS + 7) / 8;
    for (int64_t t = blockIdx.x; t < g.n_tasks; t += gridDim.x) {
        const Task k = make_task(g, t);
        const QConst q = load_qconst(prm, k.ch);
        const Div2 dv = make_div2(q.s, __frcp_rn(q.s));
        const f32x2 zpn = bc2(-q.zp), zp2 = bc2(q.zp);
        const bool fast_ok = VEC && scale_fast_ok(q.s);
        const float *xr = x + k.row_off;
        uint8_t *pr = packed + k.row * row_stride;
        for (int64_t sub = k.q0; sub < k.q1; ++sub) {
            const int64_t base = sub * kSubElems + tid * 4;
            const bool full = (sub + 1) * kSubElems <= g.n_inner;
            if (fast_ok && full) {
#pragma unroll
                for (int b = 0; b < kSubIters / kU; ++b) {
                    float4 xv[kU];
#pragma unroll
                    for (int u = 0; u < kU; ++u)
                        xv[u] = ld_stream4(xr + base + (b * kU + u) * kIterElems);
                    float mx = 0.f;
#pragma unroll
                    for (int u = 0; u < kU; ++u) mx = absmax4(mx, xv[u]);
                    const bool huge = mx > kXHi;
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        float4 cv, yv;
                        if (!huge) {
                            fwd_pair_fast<CLAMP>(xv[u].x, xv[u].y, q, dv, zpn, zp2, yv.x, yv.y, cv.x, cv.y);
                            fwd_pair_fast<CLAMP>(xv[u].z, xv[u].w, q, dv, zpn, zp2, yv.z, yv.w, cv.z, cv.w);
                        } else {
                            yv.x = fwd_elem(xv[u].x, q, cv.x);
                            yv.y = fwd_elem(xv[u].y, q, cv.y);
                            yv.z = fwd_elem(xv[u].z, q, cv.z);
                            yv.w = fwd_elem(xv[u].w, q, cv.w);
                        }
                        (void)yv;
                        const uint64_t w = pack4<BITS>(sat_code<BITS>(cv.x, bad), sat_code<BITS>(cv.y, bad),
                                                       sat_code<BITS>(cv.z, bad), sat_code<BITS>(cv.w, bad));
                        store_packed4<BITS>(pr, base + (b * kU + u) * kIterElems, w);
                    }
                }
                continue;
            }
            // ---------------- general path: ragged / unaligned / out-of-range scale ----------------
#pragma unroll 1
            for (int it = 0; it < kSubIters; ++it) {
                const int64_t p = base + (int64_t)it * kIterElems;
                if (p - 4 * (tid & 31) >= g.n_inner) break;       // the whole warp is past the row end
                const int nv = full ? 4 : valid4<VEC>(p, g.n_inner);
                const float4 xv = nv ? load4<VEC>(xr, p, g.n_inner) : make_float4(0.f, 0.f, 0.f, 0.f);
                float c[4];
                (void)fwd_elem(xv.x, q, c[0]);
                (void)fwd_elem(xv.y, q, c[1]);
                (void)fwd_elem(xv.z, q, c[2]);
                (void)fwd_elem(xv.w, q, c[3]);
                uint32_t cu[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) cu[e] = e < nv ? sat_code<BITS>(c[e], bad) : 0u;
                store_packed4_bytes<BITS>(pr, p, pack4<BITS>(cu[0], cu[1], cu[2], cu[3]), nv);
            }
        }
        // zero padding after the row's last code byte, written by the task holding its end
        if (k.q1 == g.subs_per_row) {
            const int64_t pad = row_stride - data_bytes;
            if (tid < pad) pr[data_bytes + tid] = 0;
        }
    }
    flush_count(bad, n_oor);
}

// scale / zero point of the dequantization in every parameter mode (the forward's load_qconst
// without the clamp bounds, which dequantization does not use)
__device__ __forceinline__ void unpack_const(const QParams &p, int64_t ch, float &s, float &zp) {
    if (p.mode == PARAMS_UNIT) {
        s = 1.f;
        zp = 0.f;
        return;
    }
    const float sv = __ldg(p.scale + ch * p.ss);
    s = (p.mode == PARAMS_LINEAR) ? sv : exp2f(sv);
    zp = __ldg(p.zp + ch * p.zs);
}

// the 4 codes of element position p (p % 4 == 0) from a 16-byte aligned row
template <int BITS>
__device__ __forceinline__ uint64_t load_packed4(const uint8_t *pr, int64_t p) {
    if (BITS == 16) return __ldg(reinterpret_cast<const unsigned long long *>(pr + 2 * p));
    if (BITS == 8) return __ldg(reinterpret_cast<const unsigned int *>(pr + p));
    if (BITS == 4) return __ldg(reinterpret_cast<const unsigned short *>(pr + p / 2));
    if (BITS == 2) return __ldg(pr + p / 4);
    return (uint64_t)(__ldg(pr + p / 8) >> (((p >> 2) & 1) * 4)) & 0xFu;
}
// byte-granular form for the general path (any alignment; positions beyond the row read as 0)
template <int BITS>
__device__ __forceinline__ uint32_t load_code(const uint8_t *pr, int64_t j, int64_t n_inner) {
    if (j >= n_inner) return 0u;
    if (BITS == 16) return (uint32_t)__ldg(pr + 2 * j) | ((uint32_t)__ldg(pr + 2 * j + 1) << 8);
    const int64_t bit = j * BITS;
    return ((uint32_t)__ldg(pr + (bit >> 3)) >> (bit & 7)) & ((1u << BITS) - 1u);
}

__device__ __forceinline__ float dequant(uint32_t code, float s, float zp) {
    return f_add(f_mul((float)code, s), zp);        // code*s, then + zp (two roundings)
}

template <int BITS, bool VEC>
__global__ void __launch_bounds__(kThreads)
fq_unpack_kernel(const uint8_t *__restrict__ packed, float *__restrict__ y, QParams prm, Geom g,
                 int64_t row_stride) {
    const int tid = threadIdx.x;
    constexpr uint64_t kMask = (BITS == 16) ? 0xFFFFull : ((1ull << BITS) - 1ull);
    for (int64_t t = blockIdx.x; t < g.n_tasks; t += gridDim.x) {
        const Task k = make_task(g, t);
        float s, zp;
        unpack_const(prm, k.ch, s, zp);
        const uint8_t *pr = packed + k.row * row_stride;
        float *yr = y + k.row_off;
        for (int64_t sub = k.q0; sub < k.q1; ++sub) {
            const int64_t base = sub * kSubElems + tid * 4;
            const bool full = (sub + 1) * kSubElems <= g.n_inner;
            if (VEC && full) {
#pragma unroll
                for (int b = 0; b < kSubIters / kU; ++b) {
                    uint64_t w[kU];
#pragma unroll
                    for (int u = 0; u < kU; ++u) w[u] = load_packed4<BITS>(pr, base + (b * kU + u) * kIterElems);
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        float4 yv;
                        yv.x = dequant((uint32_t)(w[u] & kMask), s, zp);
                        yv.y = dequant((uint32_t)((w[u] >> BITS) & kMask), s, zp);
                        yv.z = dequant((uint32_t)((w[u] >> (2 * BITS)) & kMask), s, zp);
                        yv.w = dequant((uint32_t)((w[u] >> (3 * BITS)) & kMask), s, zp);
                        st_stream4(yr + base + (b * kU + u) * kIterElems, yv);
                    }
                }
                continue;
            }
#pragma unroll 1
            for (int it = 0; it < kSubIters; ++it) {
                const int64_t p = base + (int64_t)it * kIterElems;
                if (p >= g.n_inner) break;
                float4 yv;
                yv.x = dequant(load_code<BITS>(pr, p + 0, g.n_inner), s, zp);
                yv.y = dequant(load_code<BITS>(pr, p + 1, g.n_inner), s, zp);
                yv.z = dequant(load_code<BITS>(pr, p + 2, g.n_inner), s, zp);
                yv.w = dequant(load_code<BITS>(pr, p + 3, g.n_inner), s, zp);
                store4<VEC>(yr, p, g.n_inner, yv);
            }
        }
    }
}
