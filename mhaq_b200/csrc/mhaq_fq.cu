// mhaq_fq.cu — sm_100a fake-quantization kernels + the C ABI of include/mhaq_fq.h.
//
// Replaces, per quantized tensor, the ~8 (forward) and ~19-27 (backward)
// separate ATen elementwise/reduction launches of the reference
// (src/quantization/gdnsq/gdnsq.py:189-229 and the QN*.backward functions)
// with ONE forward kernel (8 B/element) and ONE backward kernel
// (12 B/element) plus a tiny deterministic finalize.  HBM-bandwidth bound by
// design: 128-bit coalesced streaming accesses, per-channel constants in
// registers, fp32 per-thread partial sums -> warp shuffle -> fp64 across
// warps / tasks, no atomics.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo
#include "fq_common.cuh"
#include "../../include/mhaq_fq.h"
#include <cstdlib>

using namespace mhaq;

namespace {

// float32(3.0 ** -0.5): the GDNSQ scale-gradient factor (gdnsq.py:55).
__device__ constexpr float kInvSqrt3 = 0.57735026918962584f;
__device__ constexpr float kEwgsDelta = 0.01f;   // gdnsq.py:99
__device__ constexpr float kAewgsEps = 1e-3f;    // gdnsq.py:131
__device__ constexpr float kAewgsCap = 0.99f;    // 1 - gap, gdnsq.py:136-139

enum { NOISE_PHILOX = 0, NOISE_EXPLICIT = 1, NOISE_NONE = 2 };

// resident CTAs per SM the backward kernel is compiled for (register cap = 65536/(128*N))
#ifndef MHAQ_BWD_MIN_CTAS
#define MHAQ_BWD_MIN_CTAS 5
#endif

// ===========================================================================
// Forward
// ===========================================================================
// Eval-mode statistics (STATS): min / max CODE (NoisyAct.bw, gdnsq_act.py:51-54; the eval asserts
// of gdnsq.py:211-217 reduce to "every code finite") and min / max INPUT (what MinMaxObserver
// takes from the same tensor during calibration, calib/minmaxobserver.py:28-37) in the same pass.
// NaN-propagating min / max, like torch.min / torch.max / aminmax.
struct FwdStat {
    float cmin, cmax, xmin, xmax;
};
__device__ __forceinline__ float min_nan(float a, float b) {
    float d;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ float max_nan(float a, float b) {
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ void stat_push(FwdStat &st, float x, float c) {
    st.cmin = min_nan(st.cmin, c);
    st.cmax = max_nan(st.cmax, c);
    st.xmin = min_nan(st.xmin, x);
    st.xmax = max_nan(st.xmax, x);
}
__device__ __forceinline__ float warp_min_nan(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min_nan(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max_nan(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max_nan(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// General path: true IEEE division, any operand (also the ragged / unaligned tiles).
__device__ __forceinline__ float fwd_elem(float x, const QConst &q, float &code) {
    float c = f_clamp(x, q.lo, q.hi);            // gdnsq.py:197
    float u = f_sub(c, q.zp);                    // gdnsq.py:199
    float v = f_div(u, q.s);                     // gdnsq.py:204
    float nz = f_sub(rintf(v), v);               // QNoise.forward, gdnsq.py:15
    code = f_add(v, nz);                         // gdnsq.py:208 (== rint(v); NaN for v = +-inf)
    return f_add(f_mul(code, q.s), q.zp);        // gdnsq.py:229 (two roundings)
}
// Fast path: same roundings, the division by the channel-invariant scale done with the
// hoisted reciprocal (bit-identical, see div_exact).  For |v| < 0.5 the value of v is
// irrelevant to code = v + (rint(v) - v) = 0, so tiny / denormal u need no guard; huge
// |x| (> 2^80, incl. inf) is sent to the general path by the caller.
template <bool CLAMP>
__device__ __forceinline__ void fwd_pair_fast(float x0, float x1, const QConst &q, const Div2 &d,
                                              f32x2 zpn, f32x2 zp2, float &y0, float &y1, float &c0,
                                              float &c1) {
    const float a0 = CLAMP ? f_clamp(x0, q.lo, q.hi) : x0;
    const float a1 = CLAMP ? f_clamp(x1, q.lo, q.hi) : x1;
    const f32x2 u = add2(pk2(a0, a1), zpn);              // c - zp
    const f32x2 v = div2_quot(u, d);                     // u / s
    float v0, v1;
    upk2(v, v0, v1);
    const f32x2 nz = sub2(pk2(rintf(v0), rintf(v1)), v); // round(v) - v
    const f32x2 code = add2(v, nz);                      // v + noise
    const f32x2 y = add2(mul2_rounded(code, d.s), zp2);  // code*s, then + zp (two roundings)
    upk2(y, y0, y1);
    upk2(code, c0, c1);
}

__device__ __forceinline__ float absmax4(float m, const float4 &v) {
    return fmaxf(fmaxf(fmaxf(m, fabsf(v.x)), fmaxf(fabsf(v.y), fabsf(v.z))), fabsf(v.w));
}

// One CTA per task (grid = n_tasks) in both modes; the hardware block scheduler balances the SMs.
// STATS = true additionally keeps running min / max of codes and inputs per task and writes one
// 16-byte record {cmin, cmax, xmin, xmax} per task (min / max are exact and order-free).  A
// persistent variant (one record per CTA, 148 x 8 CTAs) was measured at 0.82-0.86 of the copy
// peak against 1.03 for the plain forward (profiles/r02_exp_eval_persistent.txt) and dropped.
// ---- programmatic dependent launch (PDL) of the eval-statistics finalize kernel ----
// fq_minmax_finalize_kernel is launched with cudaLaunchAttributeProgrammaticStreamSerialization: it
// may become resident while the forward kernel's last CTAs are still running, and calls pdl_wait()
// (griddepcontrol.wait: the prerequisite grid has completed and its memory is visible) before
// it touches a record — its launch latency overlaps the producer's tail instead of following it
// (-0.4 ... -0.7 us per eval forward at every size).  The STATS forward calls pdl_trigger() on
// entry; after a kernel that never triggers (anything else in the stream) the launch degrades to
// ordinary stream order.  Works under stream capture.  Measured and NOT kept for the backward's
// finalize and the AEWGS statistics finalize: +1 ... +3 us with 64-512 channels
// (profiles/r02_exp_pdl.txt).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <bool VEC, bool CLAMP, bool STATS>
__global__ void __launch_bounds__(kThreads)
fq_fwd_kernel(const float *__restrict__ x, float *__restrict__ y, float *__restrict__ codes,
              QParams prm, Geom g, double *__restrict__ mm_ws) {
    const int tid = threadIdx.x;
    if (STATS) pdl_trigger();                        // the statistics finalize may start launching
    __shared__ float s_red[4][kThreads / 32];
    for (int64_t t = blockIdx.x; t < g.n_tasks; t += gridDim.x) {
        FwdStat st = {INFINITY, -INFINITY, INFINITY, -INFINITY};
        const Task k = make_task(g, t);
        const QConst q = load_qconst(prm, k.ch);
        const Div2 dv = make_div2(q.s, __frcp_rn(q.s));
        const f32x2 zpn = bc2(-q.zp), zp2 = bc2(q.zp);
        const bool fast_ok = VEC && scale_fast_ok(q.s);
        const float *xr = x + k.row_off;
        float *yr = y ? y + k.row_off : nullptr;
        float *cr = codes ? codes + k.row_off : nullptr;
        for (int64_t sub = k.q0; sub < k.q1; ++sub) {
            const int64_t base = sub * kSubElems + tid * 4;
            const bool full = (sub + 1) * kSubElems <= g.n_inner;
            if (fast_ok && full) {
                // ---------------- fast path: full, aligned sub-tile ----------------
#pragma unroll
                for (int b = 0; b < kSubIters / kU; ++b) {
                    float4 xv[kU];
#pragma unroll
                    for (int u = 0; u < kU; ++u)
                        xv[u] = ld_stream4(xr + base + (b * kU + u) * kIterElems);
                    float mx = 0.f;
#pragma unroll
                    for (int u = 0; u < kU; ++u) mx = absmax4(mx, xv[u]);
                    const bool huge = mx > kXHi;      // NaN never sets it; NaN is fine on the fast path
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
                        const int64_t p = base + (b * kU + u) * kIterElems;
                        if (yr) st_stream4(yr + p, yv);
                        if (cr) st_stream4(cr + p, cv);
                        if (STATS) {
                            stat_push(st, xv[u].x, cv.x);
                            stat_push(st, xv[u].y, cv.y);
                            stat_push(st, xv[u].z, cv.z);
                            stat_push(st, xv[u].w, cv.w);
                        }
                    }
                }
                continue;
            }
            // ---------------- general path: ragged / unaligned / out-of-range scale ----------------
#pragma unroll 1
            for (int b = 0; b < kSubIters / kU; ++b) {
                float4 xv[kU];
                int nv[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int64_t p = base + (int64_t)(b * kU + u) * kIterElems;
                    nv[u] = full ? 4 : valid4<VEC>(p, g.n_inner);
                    xv[u] = nv[u] ? load4<VEC>(xr, p, g.n_inner) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    if (!nv[u]) continue;
                    const int64_t p = base + (int64_t)(b * kU + u) * kIterElems;
                    float4 cv, yv;
                    yv.x = fwd_elem(xv[u].x, q, cv.x);
                    yv.y = fwd_elem(xv[u].y, q, cv.y);
                    yv.z = fwd_elem(xv[u].z, q, cv.z);
                    yv.w = fwd_elem(xv[u].w, q, cv.w);
                    if (yr) store4<VEC>(yr, p, g.n_inner, yv);
                    if (cr) store4<VEC>(cr, p, g.n_inner, cv);
                    if (STATS) {
                        const float ce[4] = {cv.x, cv.y, cv.z, cv.w};
                        const float xe[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (e < nv[u]) stat_push(st, xe[e], ce[e]);
                    }
                }
            }
        }
            if (STATS) {
            const float a = warp_min_nan(st.cmin), b = warp_max_nan(st.cmax);
            const float c = warp_min_nan(st.xmin), d = warp_max_nan(st.xmax);
            if ((tid & 31) == 0) {
                s_red[0][tid >> 5] = a; s_red[1][tid >> 5] = b;
                s_red[2][tid >> 5] = c; s_red[3][tid >> 5] = d;
            }
            __syncthreads();
            if (tid == 0) {
                float r0 = s_red[0][0], r1 = s_red[1][0], r2 = s_red[2][0], r3 = s_red[3][0];
                for (int w = 1; w < kThreads / 32; ++w) {
                    r0 = min_nan(r0, s_red[0][w]); r1 = max_nan(r1, s_red[1][w]);
                    r2 = min_nan(r2, s_red[2][w]); r3 = max_nan(r3, s_red[3][w]);
                }
                reinterpret_cast<float4 *>(mm_ws)[t] = make_float4(r0, r1, r2, r3);
            }
            __syncthreads();
        }
    }
}

// out5 = {min code, max code, non-finite flag, min input, max input} from the per-task records
// (one 128-bit load per record, every load of a thread independent of the others)
constexpr int kMmThreads = 1024;
__global__ void __launch_bounds__(kMmThreads)
fq_minmax_finalize_kernel(const double *ws, int64_t n_rec, float *__restrict__ out5) {
    __shared__ float s[4][kMmThreads / 32];
    pdl_wait();                                      // the forward kernel's records are complete and visible
    const float4 *rec = reinterpret_cast<const float4 *>(ws);
    float v[4] = {INFINITY, -INFINITY, INFINITY, -INFINITY};
    for (int64_t t = threadIdx.x; t < n_rec; t += kMmThreads) {
        const float4 r = __ldcg(rec + t);
        v[0] = min_nan(v[0], r.x); v[1] = max_nan(v[1], r.y);
        v[2] = min_nan(v[2], r.z); v[3] = max_nan(v[3], r.w);
    }
    v[0] = warp_min_nan(v[0]); v[1] = warp_max_nan(v[1]);
    v[2] = warp_min_nan(v[2]); v[3] = warp_max_nan(v[3]);
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int m = 0; m < 4; ++m) s[m][threadIdx.x >> 5] = v[m];
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int l = threadIdx.x;
        const float a = warp_min_nan(s[0][l]), b = warp_max_nan(s[1][l]);
        const float c = warp_min_nan(s[2][l]), d = warp_max_nan(s[3][l]);
        if (l == 0) {
            out5[0] = a;
            out5[1] = b;
            // every code is finite  <=>  both extremes are (NaN propagates into both)
            out5[2] = (fabsf(a) < INFINITY && fabsf(b) < INFINITY) ? 0.f : 1.f;
            out5[3] = c;
            out5[4] = d;
        }
    }
}

// ===========================================================================
// Backward
// ===========================================================================
struct Acc {
    float se;  // sum [go*code - gv*((u/s)/s)]        -> d/d scale via dequant-mul and div
    float sn;  // estimator's own scale gradient (GDNSQ noise term / LSQ)
    float sz;  // sum (go - g_u)                      -> d/d zero_point
    float sl;  // sum g_u [x < lo]                    -> d/d min_val
    float sh;  // sum g_u [x > hi]                    -> d/d max_val
};

struct BwdConst {
    float smul;      // s (grad w.r.t. y) or 1 (grad w.r.t. codes)
    float rcp;       // RN(1/s) for the fast division sequences
    float delta;     // AEWGS per-channel delta
    bool lo_lt_hi, lo_gt_hi;
};

// The estimator: gradient w.r.t. v given g = gradient w.r.t. the codes (QN*.backward).
template <int METHOD>
__device__ __forceinline__ float estimator_gv(float g, float e, float delta) {
    if (METHOD == MHAQ_FQ_STE || METHOD == MHAQ_FQ_LSQ) {
        return __fmaf_rn(g, 0.f, g);                         // g + g*0   (gdnsq.py:50,78)
    } else if (METHOD == MHAQ_FQ_EWGS) {
        const float gi = f_mul(f_mul(-fabsf(g), e), kEwgsDelta);   // gdnsq.py:100
        return f_add(g, gi);
    } else {                                                 // AEWGS, gdnsq.py:118-141
        const float sg = (g > 0.f) ? 1.f : ((g < 0.f) ? -1.f : 0.f);
        const float nf = f_mul(sg, e);
        float gs = f_mul(delta, nf);
        gs = (gs > kAewgsCap) ? kAewgsCap : gs;              // clamp_max(1-gap)
        return f_add(g, f_mul(-g, gs));
    }
}

template <int METHOD, bool CLAMP, int NOISE, bool FAST, bool CODEGRAD>
__device__ __forceinline__ float bwd_elem(float x, float go, float rv, uint32_t sign_flip,
                                          const QConst &q, const BwdConst &bc, Acc &acc) {
    // ---- recompute the forward (gdnsq.py:197-208) ----
    float c;
    bool in, lo_m = false, hi_m = false;
    if (CLAMP && FAST) {
        // fast path is only entered with lo < hi: the clamp_backward_min_max predicate is
        // then constant-true and the masks collapse to the two comparisons
        lo_m = x < q.lo;
        hi_m = x > q.hi;
        c = hi_m ? q.hi : (lo_m ? q.lo : x);
        in = (c == x);                                   // == (x >= lo && x <= hi); false for NaN
    } else if (CLAMP) {
        const bool p_lt = x < q.lo, p_gt = x > q.hi;
        const float c1 = p_lt ? q.lo : x;
        c = (c1 > q.hi) ? q.hi : c1;
        in = (x >= q.lo) && (x <= q.hi);                 // clamp_backward mask
        lo_m = p_lt && bc.lo_lt_hi;                      // clamp_backward_min_max
        hi_m = p_gt || (p_lt && bc.lo_gt_hi);
    } else {
        c = x;
        in = (x == x);
    }
    const float u = f_sub(c, q.zp);
    const float v = FAST ? div_exact(u, q.s, bc.rcp) : f_div(u, q.s);
    const float e = f_sub(rintf(v), v);                  // round(v) - v, exact
    const float code = f_add(v, e);
    // ---- gradient w.r.t. codes, then the estimator ----
    const float g = f_mul(go, bc.smul);                  // MulBackward of code*s
    float gv, gu;                                        // gu = DivBackward (self): gv / s
    if (FAST && (METHOD == MHAQ_FQ_STE || METHOD == MHAQ_FQ_LSQ) && !CODEGRAD) {
        // g + g*0 == g bit for bit unless g is inf (-> NaN); div_of_product maps an
        // infinite g to NaN as well (inf*s - inf), so gx matches the reference either way
        gv = g;
        gu = div_of_product(go, gv, q.s, bc.rcp);        // gv == RN(go*s)
    } else {
        gv = estimator_gv<METHOD>(g, e, bc.delta);
        gu = FAST ? div_exact(gv, q.s, bc.rcp) : f_div(gv, q.s);
    }
    const float gx = in ? gu : 0.f;                      // ClampBackward
    // ---- parameter-gradient partial sums ----
    // d/ds: the reference's own fp32 per-element terms — MulBackward go*code and
    // DivBackward -gv*((u/s)/s) — differenced per element (they nearly cancel, so the
    // difference is all but exact) and only then accumulated: same terms as the
    // reference, summed without its catastrophic cancellation between two big fp32 sums.
    const float t2 = f_mul(gv, FAST ? div_exact(v, q.s, bc.rcp) : f_div(v, q.s));
    if (!CODEGRAD) {
        acc.se += f_sub(f_mul(go, code), t2);
        acc.sz += f_sub(go, gu);                         // (+zp of dequant) - (sub zp)
    } else {
        acc.se -= t2;
        acc.sz -= gu;
    }
    if (METHOD == MHAQ_FQ_LSQ) {
        acc.sn = __fmaf_rn(g, e, acc.sn);                // gdnsq.py:81-82
    } else if (NOISE == NOISE_EXPLICIT) {
        acc.sn += f_mul(f_mul(kInvSqrt3, g), rv);        // gdnsq.py:54-55
    } else {
        const float t = f_mul(kInvSqrt3, g);
        const float ts = __uint_as_float(__float_as_uint(t) ^ (sign_flip & 0x80000000u));
        acc.sn = __fmaf_rn(ts, 0.5f, acc.sn);            // r = bit - 0.5
    }
    if (CLAMP) {
        if (lo_m) acc.sl += gu;
        if (hi_m) acc.sh += gu;
    }
    return gx;
}

// Packed (two elements per FP instruction) version of bwd_elem<.., FAST=true, CODEGRAD=false>
// for the STE / LSQ estimators — the hot variants (every activation, most weights).
// Same fp32 operations element by element; g is carried NEGATED (gn = go*(-s) == -RN(go*s)
// exactly) so that no operand-negate modifier is needed:
//   r  = go*s - g           = fma2(go, s, gn)            (exact)
//   gu = RN(g/s)            = fma2(r, -y, go)            (div_of_product, zero signs included)
//   t2 = -RN(g*RN(v/s))     = mul2(gn, div2_quot(v))
// The noise / LSQ sum is accumulated with the opposite sign and negated at the flush.
struct Acc2 {
    f32x2 se, sn, sz;
};
struct PairConst {
    Div2 d;
    f32x2 zpn, c, half;
};

template <int METHOD, bool CLAMP, int NOISE>
__device__ __forceinline__ void bwd_pair_fast(float x0, float x1, float go0, float go1, float rn0,
                                              float rn1, uint32_t sf0, uint32_t sf1, const QConst &q,
                                              const PairConst &pc, Acc2 &a2, Acc &acc, float &o0,
                                              float &o1) {
    float c0, c1;
    bool in0, in1, lo0 = false, lo1 = false, hi0 = false, hi1 = false;
    if (CLAMP) {        // lo < hi on this path (see bwd_elem)
        lo0 = x0 < q.lo; hi0 = x0 > q.hi;
        lo1 = x1 < q.lo; hi1 = x1 > q.hi;
        c0 = hi0 ? q.hi : (lo0 ? q.lo : x0);
        c1 = hi1 ? q.hi : (lo1 ? q.lo : x1);
        in0 = (c0 == x0); in1 = (c1 == x1);
    } else {
        c0 = x0; c1 = x1;
        in0 = (x0 == x0); in1 = (x1 == x1);
    }
    const f32x2 go = pk2(go0, go1);
    const f32x2 u = add2(pk2(c0, c1), pc.zpn);
    const f32x2 v = div2_quot(u, pc.d);
    float v0, v1;
    upk2(v, v0, v1);
    const f32x2 e = sub2(pk2(rintf(v0), rintf(v1)), v);
    const f32x2 code = add2(v, e);
    const f32x2 gn = mul2(go, pc.d.sn);                  // -g
    const f32x2 r = fma2(go, pc.d.s, gn);                // go*s - g, exact
    const f32x2 gu = fma2(r, pc.d.yn, go);               // RN(g / s)
    float gu0, gu1;
    upk2(gu, gu0, gu1);
    o0 = in0 ? gu0 : 0.f;
    o1 = in1 ? gu1 : 0.f;
    const f32x2 t2n = mul2_rounded(gn, div2_quot(v, pc.d));       // -fl(g * fl(v/s))
    a2.se = add2(a2.se, add2(mul2_rounded(go, code), t2n));       // fl(go*code) - fl(g*fl(v/s))
    a2.sz = add2(a2.sz, sub2(go, gu));
    if (METHOD == MHAQ_FQ_LSQ) {
        a2.sn = fma2(gn, e, a2.sn);                      // -(g*e)
    } else if (NOISE == NOISE_EXPLICIT) {
        a2.sn = add2(a2.sn, mul2_rounded(mul2(gn, pc.c), pk2(rn0, rn1)));   // -fl(fl(c*g)*r)
    } else {
        float t0, t1;
        upk2(mul2(gn, pc.c), t0, t1);                    // -fl(c*g)
        t0 = __uint_as_float(__float_as_uint(t0) ^ (sf0 & 0x80000000u));
        t1 = __uint_as_float(__float_as_uint(t1) ^ (sf1 & 0x80000000u));
        a2.sn = fma2(pk2(t0, t1), pc.half, a2.sn);       // -(c*g)*r,  r = bit - 0.5
    }
    if (CLAMP) {
        if (lo0) acc.sl += gu0;
        if (lo1) acc.sl += gu1;
        if (hi0) acc.sh += gu0;
        if (hi1) acc.sh += gu1;
    }
}

// Guard fall-back of the fast path (rare: tiny non-zero / huge gradients): recompute the
// input gradient of one 16-element thread batch with true IEEE divisions, RE-LOADING the
// operands (L2 hits) so that nothing of this path stays live in the streaming loop, and
// overwrite what the fast path stored (same thread, program order).
template <int METHOD, bool CLAMP>
__device__ __noinline__ void fix_batch_exact(const float *xr, const float *gr, float *gxr, int64_t p0,
                                             QConst q, float smul, float delta) {
#pragma unroll 1
    for (int u = 0; u < kU; ++u) {
        const int64_t p = p0 + u * kIterElems;
        const float4 xv = *reinterpret_cast<const float4 *>(xr + p);
        const float4 gv = *reinterpret_cast<const float4 *>(gr + p);
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float x = xs[i];
            const float c = CLAMP ? f_clamp(x, q.lo, q.hi) : x;
            const bool in = CLAMP ? ((x >= q.lo) && (x <= q.hi)) : (x == x);
            const float v = f_div(f_sub(c, q.zp), q.s);
            const float e = f_sub(rintf(v), v);
            const float gvv = estimator_gv<METHOD>(f_mul(gs[i], smul), e, delta);
            o[i] = in ? f_div(gvv, q.s) : 0.f;
        }
        *reinterpret_cast<float4 *>(gxr + p) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// min over the 4 components of (bits<<1)-1: zero maps to 0xffffffff (never the minimum),
// anything else orders by magnitude -> "smallest non-zero |go|" with 2 integer ops/element.
__device__ __forceinline__ uint32_t nzmin4(uint32_t m, const float4 &v) {
    const uint32_t a = (__float_as_uint(v.x) << 1) - 1u, b = (__float_as_uint(v.y) << 1) - 1u;
    const uint32_t c = (__float_as_uint(v.z) << 1) - 1u, d = (__float_as_uint(v.w) << 1) - 1u;
    return min(min(min(m, a), min(b, c)), d);
}

// Per-task epilogue of the backward kernel: fp32 partials -> warp shuffle -> fp64 sum over
// the 4 warps -> one record per task.  No fences, no atomics: the kernel boundary orders the
// records before the finalize kernel, so the streaming kernel's CTAs retire immediately.
template <bool CLAMP>
__device__ __forceinline__ void flush_record(const Acc &acc, int64_t t, double *__restrict__ ws) {
    __shared__ float s_red[5][kThreads / 32];
    const int tid = threadIdx.x;
    float v0 = warp_sum(acc.se), v1 = warp_sum(acc.sn), v2 = warp_sum(acc.sz);
    float v3 = CLAMP ? warp_sum(acc.sl) : 0.f, v4 = CLAMP ? warp_sum(acc.sh) : 0.f;
    if ((tid & 31) == 0) {
        const int w = tid >> 5;
        s_red[0][w] = v0; s_red[1][w] = v1; s_red[2][w] = v2; s_red[3][w] = v3; s_red[4][w] = v4;
    }
    __syncthreads();
    if (tid < 5) {
        double a = 0.0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) a += (double)s_red[tid][w];
        ws[t * kNPart + tid] = a;
    }
    __syncthreads();
}

// Deterministic second stage, ONE launch for any record count.
// grid = (slices, n_ch).  CTA (sl, ch) sums records [sl*kSliceRecs, ...) of channel ch in a
// fixed order (thread-strided, then a fixed tree) -> slice record.  The last CTA of a channel
// to finish (ticket) sums the channel's slice records in index order and writes the
// gradients.  Which CTA performs the last step varies run to run; the summation order, hence
// the result, does not.  Tickets are zero on entry and restored to zero.
// one record per thread in the first stage: every load of a stage is issued at once
// (a serial loop over records pays a full memory latency per iteration — measured 15-22 us
// for 4096-8192 records in one CTA vs ~3 us with 256-record slices)
constexpr int kSliceRecs = 256;
constexpr int kFinThreads = 256;

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// Fixed-shape tree: 5 shuffle levels inside each warp, then the warp sums (in warp-id order)
// reduced by warp 0.  The result is valid in thread 0.  One barrier.
template <int NCOL>
__device__ __forceinline__ void block_sum_cols(double (&a)[NCOL], double (*s)[kFinThreads / 32]) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int m = 0; m < NCOL; ++m) {
        a[m] = warp_sum_f64(a[m]);
        if (lane == 0) s[m][w] = a[m];
    }
    __syncthreads();
    if (w == 0) {
#pragma unroll
        for (int m = 0; m < NCOL; ++m) a[m] = warp_sum_f64(lane < nw ? s[m][lane] : 0.0);
    }
    __syncthreads();
}

// record index of the i-th record of channel ch (rows r = ch + k*n_ch, tasks_per_row each)
__device__ __forceinline__ int64_t chan_record(const Geom &g, int64_t ch, int64_t i) {
    const int64_t rr = i / g.tasks_per_row;
    return (rr * g.n_ch + ch) * g.tasks_per_row + (i - rr * g.tasks_per_row);
}

template <int NCOL, typename Emit>
__device__ __forceinline__ void finalize_channel(const double *ws, double *slice_ws,
                                                 unsigned int *tickets, const Geom &g, int64_t n_sl,
                                                 Emit emit) {
    __shared__ double s[NCOL][kFinThreads / 32];
    __shared__ int s_last;
    const int tid = threadIdx.x;
    const int nthr = blockDim.x;
    // 1-D grid of n_ch * n_sl CTAs (the channel count is not limited by gridDim.y)
    const int64_t ch = (int64_t)blockIdx.x / n_sl, sl = (int64_t)blockIdx.x - ch * n_sl;
    const int64_t recs = (g.n_rows / g.n_ch) * g.tasks_per_row;
    const int64_t i0 = sl * kSliceRecs;
    const int64_t i1 = (i0 + kSliceRecs < recs) ? i0 + kSliceRecs : recs;
    double a[NCOL];
#pragma unroll
    for (int m = 0; m < NCOL; ++m) a[m] = 0.0;
    for (int64_t i = i0 + tid; i < i1; i += nthr) {
        const double *rec = ws + chan_record(g, ch, i) * kNPart;
#pragma unroll
        for (int m = 0; m < NCOL; ++m) a[m] += __ldcg(rec + m);
    }
    block_sum_cols<NCOL>(a, s);
    if (n_sl == 1) {
        if (tid == 0) emit(ch, a);
        return;
    }
    if (tid == 0) {
        double *o = slice_ws + (ch * n_sl + sl) * kNPart;
#pragma unroll
        for (int m = 0; m < NCOL; ++m) o[m] = a[m];
        __threadfence();
        s_last = (atomicAdd(&tickets[ch], 1u) == (unsigned)(n_sl - 1));
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
#pragma unroll
    for (int m = 0; m < NCOL; ++m) a[m] = 0.0;
    for (int64_t i = tid; i < n_sl; i += nthr) {
        const double *o = slice_ws + (ch * n_sl + i) * kNPart;
#pragma unroll
        for (int m = 0; m < NCOL; ++m) a[m] += __ldcg(o + m);
    }
    block_sum_cols<NCOL>(a, s);
    if (tid == 0) {
        emit(ch, a);
        tickets[ch] = 0u;
    }
}

// Outputs by parameter mode (a[] = {S_e, S_noise, S_zp, S_lo, S_hi} of the channel):
//   LINEAR    : o0 = d/d scale, o1 = d/d zero_point, o2 = d/d min_val, o3 = d/d max_val
//   ACT_LOG   : o0 = d/d log_act_s = (d/ds - S_hi) * s * ln2      (hi contains -s)
//               o1 = d/d act_b     = S_zp + S_lo + S_hi           (zp, lo and hi all contain act_b)
//               o2 = d/d log_act_q = S_hi * q * ln2
//   WEIGHT_LOG: o0 = d/d log_wght_s = d/ds * s * ln2,  o1 = d/d zero_point
//   UNIT      : o0 = S_noise alone: the estimator's own scale gradient (QN*.backward's grad_scale,
//               gdnsq.py:54-55, 81-82) — the unit divisor is not a parameter
// i.e. the Exp2Backward / AddBackward / SubBackward nodes autograd would run on the tiny
// parameter tensors (gdnsq_act.py:42-48), folded into the last thread of the reduction.
__device__ __forceinline__ void emit_param_grads(const QParams &prm, int64_t ch, const double (&a)[5],
                                                 float *o0, float *o1, float *o2, float *o3) {
    const double ds = a[0] + a[1];
    constexpr double kLn2 = 0.693147180559945309417;
    // (+ prm.accK: the gradient the same parameter receives along the caller's other paths, added in
    // fp32 exactly as autograd's AccumulateGrad would add the two contributions)
    const bool log1 = (prm.mode == PARAMS_ACT_LOG);
    auto put = [&](float *o, const float *acc, double v) {
        if (!o) return;
        const int64_t i = log1 ? 0 : ch;
        const float f = (float)v;
        o[i] = acc ? __fadd_rn(f, acc[i]) : f;
    };
    if (prm.mode == PARAMS_ACT_LOG) {
        const double s = (double)exp2f(prm.scale[0]), q = (double)exp2f(prm.lo[0]);
        put(o0, prm.acc0, (ds - a[4]) * s * kLn2);
        put(o1, prm.acc1, a[2] + a[3] + a[4]);
        put(o2, prm.acc2, a[4] * q * kLn2);
    } else if (prm.mode == PARAMS_WEIGHT_LOG) {
        const double s = (double)exp2f(prm.scale[ch * prm.ss]);
        put(o0, prm.acc0, ds * s * kLn2);
        put(o1, prm.acc1, a[2]);
    } else if (prm.mode == PARAMS_UNIT) {
        put(o0, prm.acc0, a[1]);
    } else {
        put(o0, prm.acc0, ds);
        put(o1, prm.acc1, a[2]);
        put(o2, prm.acc2, a[3]);
        put(o3, prm.acc3, a[4]);
    }
}

__global__ void __launch_bounds__(kFinThreads)
fq_bwd_finalize_kernel(const double *ws, double *slice_ws, unsigned int *tickets,
                       Geom g, int64_t n_sl, QParams prm, float *__restrict__ o0,
                       float *__restrict__ o1, float *__restrict__ o2, float *__restrict__ o3) {
    finalize_channel<5>(ws, slice_ws, tickets, g, n_sl, [=](int64_t ch, const double (&a)[5]) {
        emit_param_grads(prm, ch, a, o0, o1, o2, o3);
    });
}

template <int METHOD, bool CLAMP, int NOISE, bool VEC, bool CODEGRAD>
__global__ void __launch_bounds__(kThreads, MHAQ_BWD_MIN_CTAS)
fq_bwd_kernel(const float *__restrict__ go, const float *__restrict__ x, float *__restrict__ gx,
              QParams prm, Geom g, const float *__restrict__ r, uint64_t seed,
              uint64_t offset, const uint64_t *__restrict__ philox_dev,
              const float *__restrict__ aewgs_stats, double *__restrict__ ws) {
    const int tid = threadIdx.x;
    PhiloxKey key = {0, 0, 0, 0};
    if (NOISE == NOISE_PHILOX) key = make_key(seed, offset, philox_dev);
    const int64_t supers_per_row = (g.n_inner + kSuperElems - 1) / kSuperElems;
    constexpr bool kProductDiv = (METHOD == MHAQ_FQ_STE || METHOD == MHAQ_FQ_LSQ);

    for (int64_t t = blockIdx.x; t < g.n_tasks; t += gridDim.x) {
        const Task k = make_task(g, t);
        const QConst q = load_qconst(prm, k.ch);
        BwdConst bc;
        bc.smul = CODEGRAD ? 1.f : q.s;
        bc.rcp = __frcp_rn(q.s);
        bc.lo_lt_hi = q.lo < q.hi;
        bc.lo_gt_hi = q.lo > q.hi;
        bc.delta = 0.f;
        if (METHOD == MHAQ_FQ_AEWGS) {
            const float num = __ldg(aewgs_stats + 0 * g.n_ch + k.ch);
            const float e2 = __ldg(aewgs_stats + 1 * g.n_ch + k.ch);
            const float me = __ldg(aewgs_stats + 2 * g.n_ch + k.ch);
            float den = f_sub(e2, f_mul(me, me));            // gdnsq.py:132
            den = (den < kAewgsEps) ? kAewgsEps : den;       // clamp_min(eps)
            bc.delta = f_div(num, den);                      // gdnsq.py:134
        }
        const bool fast_ok = VEC && scale_fast_ok(q.s) && (!CLAMP || bc.lo_lt_hi);
        const float *xr = x + k.row_off;
        const float *gr = go + k.row_off;
        const float *rr = (NOISE == NOISE_EXPLICIT) ? r + k.row_off : nullptr;
        float *gxr = gx ? gx + k.row_off : nullptr;
        Acc acc = {0.f, 0.f, 0.f, 0.f, 0.f};
        Acc2 a2 = {0ull, 0ull, 0ull};
        PairConst pc;
        pc.d = make_div2(q.s, bc.rcp);
        pc.zpn = bc2(-q.zp);
        pc.c = bc2(kInvSqrt3);
        pc.half = bc2(0.5f);
        uint4 rnd = make_uint4(0, 0, 0, 0);
        int64_t curT = -1;

        for (int64_t sub = k.q0; sub < k.q1; ++sub) {
            const int64_t base = sub * kSubElems + tid * 4;
            const bool full = (sub + 1) * kSubElems <= g.n_inner;
            const int it0 = (int)(sub & (kSuperSubs - 1)) * kSubIters;
            if (NOISE == NOISE_PHILOX) {
                const int64_t T = sub / kSuperSubs;
                if (T != curT) {
                    rnd = noise_block(key, k.row, supers_per_row, T, tid);
                    curT = T;
                }
            }
            if (fast_ok && full) {
                // ---------------- fast path: full, aligned sub-tile ----------------
                // one Philox word (32 bits) covers the 8 iterations x 4 elements of a sub-tile
                uint32_t nw = 0;
                if (NOISE == NOISE_PHILOX) {
                    const int wi = (int)(sub & (kSuperSubs - 1));
                    nw = ~((wi < 2) ? ((wi == 0) ? rnd.x : rnd.y) : ((wi == 2) ? rnd.z : rnd.w));
                }
#pragma unroll
                for (int b = 0; b < kSubIters / kU; ++b) {
                    float4 xv[kU], gv[kU], rv4[kU];
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        const int64_t p = base + (b * kU + u) * kIterElems;
                        xv[u] = ld_stream4(xr + p);
                        gv[u] = ld_stream4(gr + p);
                        rv4[u] = (NOISE == NOISE_EXPLICIT) ? ld_stream4(rr + p)
                                                           : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    // guard of the gradient division: smallest non-zero |go| >= 2^-56
                    // (and, off the product shortcut, largest |go| <= 2^80)
                    uint32_t mn = 0xffffffffu;
                    float mx = 0.f;
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        mn = nzmin4(mn, gv[u]);
                        if (!kProductDiv || CODEGRAD) mx = absmax4(mx, gv[u]);
                    }
                    const bool odd = (mn < kGoLoBits2m1) || (mx > kGvHi);
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        const int64_t p = base + (b * kU + u) * kIterElems;
                        constexpr int kTop = 31;
                        const int sh = (b * kU + u) * 4;     // compile-time after unrolling
                        float4 o;
                        if (kProductDiv && !CODEGRAD) {
                            bwd_pair_fast<METHOD, CLAMP, NOISE>(xv[u].x, xv[u].y, gv[u].x, gv[u].y, rv4[u].x, rv4[u].y,
                                                                nw << (kTop - sh - 0), nw << (kTop - sh - 1), q, pc, a2, acc, o.x, o.y);
                            bwd_pair_fast<METHOD, CLAMP, NOISE>(xv[u].z, xv[u].w, gv[u].z, gv[u].w, rv4[u].z, rv4[u].w,
                                                                nw << (kTop - sh - 2), nw << (kTop - sh - 3), q, pc, a2, acc, o.z, o.w);
                        } else {
                            o.x = bwd_elem<METHOD, CLAMP, NOISE, true, CODEGRAD>(xv[u].x, gv[u].x, rv4[u].x, nw << (kTop - sh - 0), q, bc, acc);
                            o.y = bwd_elem<METHOD, CLAMP, NOISE, true, CODEGRAD>(xv[u].y, gv[u].y, rv4[u].y, nw << (kTop - sh - 1), q, bc, acc);
                            o.z = bwd_elem<METHOD, CLAMP, NOISE, true, CODEGRAD>(xv[u].z, gv[u].z, rv4[u].z, nw << (kTop - sh - 2), q, bc, acc);
                            o.w = bwd_elem<METHOD, CLAMP, NOISE, true, CODEGRAD>(xv[u].w, gv[u].w, rv4[u].w, nw << (kTop - sh - 3), q, bc, acc);
                        }
                        if (gxr) st_stream4(gxr + p, o);
                    }
                    if (odd && gxr)   // rare: exact IEEE division for the input gradient
                        fix_batch_exact<METHOD, CLAMP>(xr, gr, gxr, base + (b * kU) * kIterElems, q,
                                                       bc.smul, bc.delta);
                }
                continue;
            }
            // ---------------- general path: ragged / unaligned / out-of-range scale ----------------
#pragma unroll 1
            for (int b = 0; b < kSubIters / kU; ++b) {
                float4 xv[kU], gv[kU], rv4[kU];
                int nv[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int64_t p = base + (int64_t)(b * kU + u) * kIterElems;
                    nv[u] = full ? 4 : valid4<VEC>(p, g.n_inner);
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    xv[u] = nv[u] ? load4<VEC>(xr, p, g.n_inner) : z;
                    gv[u] = nv[u] ? load4<VEC>(gr, p, g.n_inner) : z;
                    rv4[u] = z;
                    if (NOISE == NOISE_EXPLICIT && nv[u]) rv4[u] = load4<VEC>(rr, p, g.n_inner);
                }
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    if (!nv[u]) continue;
                    const int64_t p = base + (int64_t)(b * kU + u) * kIterElems;
                    uint32_t inv = 0;
                    if (NOISE == NOISE_PHILOX) inv = ~noise_nibble(rnd, it0 + b * kU + u);
                    float4 o;
                    o.x = bwd_elem<METHOD, CLAMP, NOISE, false, CODEGRAD>(xv[u].x, gv[u].x, rv4[u].x, inv << 31, q, bc, acc);
                    o.y = bwd_elem<METHOD, CLAMP, NOISE, false, CODEGRAD>(xv[u].y, gv[u].y, rv4[u].y, inv << 30, q, bc, acc);
                    o.z = bwd_elem<METHOD, CLAMP, NOISE, false, CODEGRAD>(xv[u].z, gv[u].z, rv4[u].z, inv << 29, q, bc, acc);
                    o.w = bwd_elem<METHOD, CLAMP, NOISE, false, CODEGRAD>(xv[u].w, gv[u].w, rv4[u].w, inv << 28, q, bc, acc);
                    if (gxr) store4<VEC>(gxr, p, g.n_inner, o);
                }
            }
        }
        if (kProductDiv && !CODEGRAD) {   // fold the packed lanes (fixed order) into the record
            float l, h;
            upk2(a2.se, l, h); acc.se += l + h;
            upk2(a2.sn, l, h); acc.sn -= l + h;          // accumulated with the opposite sign
            upk2(a2.sz, l, h); acc.sz += l + h;
        }
        flush_record<CLAMP>(acc, t, ws);
    }
}

// ===========================================================================
// Flat (per-tensor) backward: persistent, balanced, reduction finished in-kernel
// ===========================================================================
// Activation tensors of real models are per-tensor and mid-sized (1-50 M elements): a few waves of
// CTAs, where a second (finalize) launch and per-task flushes are a visible fraction of the
// kernel.  This variant is launched with at most `cap` = SMs x resident-CTAs blocks; block b owns
// the contiguous range of `per_cta` 2048-element batches [b*per_cta, ...) — every block resident at
// once with (almost) the same amount of work, no waves — folds its fp32 per-thread partials into
// per-warp fp64 accumulators every 4 batches (64 elements per thread, like a 2-sub-tile task of
// the streaming kernel), publishes ONE self-validating record, and block 0 sums the <= cap
// records in index order and applies emit_param_grads.  Deterministic: the partition and both
// summation orders are functions of the shape only.
// The noise stream is the streaming kernel's (a function of the element position only).
// No fence, no atomic: the record words are their own "ready" flags (see flat_enc below).
constexpr int kBatchElems = kIterElems * kU;      // 2048
constexpr int kFlatGroup = 4;                     // batches between fp32 -> fp64 folds
constexpr int kFlatCapMax = 2048;                 // upper bound on the grid (workspace sizing)

struct FlatGeom {
    int64_t n;          // elements
    int64_t full;       // whole 2048-element batches
    int64_t k;          // batches per block (the last block may own fewer)
    int64_t rest0;      // first element of the ragged tail (= full * 2048)
    int64_t rest_iters; // 512-element iterations of the tail (0..4, the last may be ragged)
    int grid;           // blocks == records
    // interleaved mode (large tensors): block b owns the 4-batch chunks b, b + grid, b + 2 grid, ...
    // so the resident blocks sweep the tensor as ONE moving band of addresses (DRAM-page friendly,
    // like the dynamically scheduled streaming kernel) instead of `grid` far-apart streams
    int interleave;
    int64_t chunks;     // ceil(full / 4)
};
// Batch-granular balance: k = ceil(full / cap) batches per block, grid = ceil(full / k) blocks, so
// every block but the last owns exactly k batches.  (Balancing the remainder at 512-element
// granularity through a separate direct-load path was measured and rejected: the extra
// un-pipelined phase per block cost more than the evened-out batch bought,
// profiles/r02_midsize.md.)
__host__ __device__ inline FlatGeom make_flat_geom(int64_t n, int cap, int interleave = 0) {
    FlatGeom f;
    f.n = n;
    if (cap > kFlatCapMax) cap = kFlatCapMax;
    if (cap < 1) cap = 1;
    f.full = n / kBatchElems;
    f.interleave = interleave;
    f.chunks = (f.full + kFlatGroup - 1) / kFlatGroup;
    if (interleave) {
        int64_t kc = (f.chunks + cap - 1) / cap;          // chunks per block
        if (kc < 1) kc = 1;
        int64_t gsz = (f.chunks + kc - 1) / kc;
        if (gsz < 1) gsz = 1;
        f.grid = (int)gsz;
        f.k = kc * kFlatGroup;                            // upper bound of batches per block
    } else {
        f.k = (f.full + cap - 1) / cap;
        if (f.k < 1) f.k = 1;
        int64_t gsz = (f.full + f.k - 1) / f.k;
        if (gsz < 1) gsz = 1;
        f.grid = (int)gsz;
    }
    f.rest0 = f.full * kBatchElems;
    f.rest_iters = (n - f.rest0 + kIterElems - 1) / kIterElems;
    return f;
}

template <bool CLAMP>
__device__ __forceinline__ void flat_fold(Acc &acc, Acc2 &a2, double (*s_acc)[kThreads / 32]) {
    float l, h;
    upk2(a2.se, l, h); acc.se += l + h;
    upk2(a2.sn, l, h); acc.sn -= l + h;          // accumulated with the opposite sign
    upk2(a2.sz, l, h); acc.sz += l + h;
    const float v0 = warp_sum(acc.se), v1 = warp_sum(acc.sn), v2 = warp_sum(acc.sz);
    const float v3 = CLAMP ? warp_sum(acc.sl) : 0.f, v4 = CLAMP ? warp_sum(acc.sh) : 0.f;
    if ((threadIdx.x & 31) == 0) {               // each warp owns its slot: no barrier needed
        const int w = threadIdx.x >> 5;
        s_acc[0][w] += (double)v0; s_acc[1][w] += (double)v1; s_acc[2][w] += (double)v2;
        if (CLAMP) { s_acc[3][w] += (double)v3; s_acc[4][w] += (double)v4; }
    }
    acc = {0.f, 0.f, 0.f, 0.f, 0.f};
    a2 = {0ull, 0ull, 0ull};
}

// ---- TMA (bulk async copy) + mbarrier helpers: global -> shared staging of the operands ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// 1-D bulk copy global -> shared; completion (bytes landed) is signalled on the mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- per-block records of the flat backward, published without fence or ticket ----
// A record is 3 x 16 bytes {v0,v1} {v2,v3} {v4,1}; every 64-bit word is stored ENCODED so that it
// is never zero (bits(v + 0.0) ^ sign bit: +0.0 -> 0x8000..., -0.0 cannot occur after "+ 0.0"),
// and zero means "not written yet".  The reader (block 0) polls the words
// themselves, so no ordering between data and a flag is needed — the data IS the flag — and
// writes zero back after it has read a record (the region lives in the zero-initialised ticket
// buffer, which every launch leaves zero: include/mhaq_fq.h).
constexpr int kFlatRecWords = 6;                  // 64-bit words per record (48 bytes)
constexpr int kFlatRecOffsetU32 = 4;              // records start 16 bytes into the ticket buffer
__device__ __forceinline__ unsigned long long flat_enc(double v) {
    return (unsigned long long)__double_as_longlong(v + 0.0) ^ 0x8000000000000000ull;
}
__device__ __forceinline__ double flat_dec(unsigned long long b) {
    return __longlong_as_double((long long)(b ^ 0x8000000000000000ull));
}
__device__ __forceinline__ void st_rec2(unsigned long long *p, unsigned long long a, unsigned long long b) {
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void ld_rec2(const unsigned long long *p, unsigned long long &a, unsigned long long &b) {
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}

// operand staging ring: kFlatStages x (8 KB x + 8 KB go) per CTA (dynamic shared memory)
#ifndef MHAQ_FLAT_STAGES
#define MHAQ_FLAT_STAGES 2
#endif
constexpr int kFlatStages = MHAQ_FLAT_STAGES;
// 4 compute warps + 1 auxiliary warp: the auxiliary warp's lane 0 drives the TMA ring and
// publishes the block's record.  It never stores gradients, so its release fence before the
// ticket has nothing to wait for — a compute thread's fence would sit out the L2 round trip of
// the gradient stores it has just issued, on the critical path of the last block.
constexpr int kFlatThreads = kThreads + 32;
constexpr int kFlatSmemBytes = kFlatStages * 2 * kBatchElems * (int)sizeof(float);
constexpr int kFlatCtasPerSm = 4;

template <int METHOD, bool CLAMP, int NOISE, bool MBAR>
__global__ void __launch_bounds__(kFlatThreads, kFlatCtasPerSm)
fq_bwd_flat_kernel(const float *__restrict__ go, const float *__restrict__ x, float *__restrict__ gx,
                   QParams prm, FlatGeom f, const float *__restrict__ r, uint64_t seed,
                   uint64_t offset, const uint64_t *__restrict__ philox_dev, double *__restrict__ ws,
                   unsigned int *ticket, float *__restrict__ o0, float *__restrict__ o1,
                   float *__restrict__ o2, float *__restrict__ o3, int exp_flags) {
    static_assert(METHOD == MHAQ_FQ_STE || METHOD == MHAQ_FQ_LSQ, "flat backward: STE / LSQ only");
    const int tid = threadIdx.x;
    const bool aux = tid >= kThreads;                 // warp 4: TMA producer + record publisher
    // Operands arrive through the TMA engine (cp.async.bulk, 8 KB per operand per batch) into a
    // shared-memory ring guarded by mbarriers: the copies of the next batches are in flight while
    // batch i is computed, whatever the register budget — a short kernel has no steady state in
    // which resident CTAs would drift apart and overlap each other's load and compute phases.
    extern __shared__ __align__(128) unsigned char flat_smem[];
    float *const s_x = reinterpret_cast<float *>(flat_smem);                   // [stages][2048]
    float *const s_g = s_x + kFlatStages * kBatchElems;                         // [stages][2048]
    __shared__ __align__(8) uint64_t s_bar[kFlatStages];      // the stage's bytes have landed
    __shared__ __align__(8) uint64_t s_emp[kFlatStages];      // MBAR: all 4 compute warps have copied it to registers
    __shared__ double s_acc[5][kThreads / 32];
    __shared__ double s_fin[5][kFinThreads / 32];
    constexpr uint32_t kOpBytes = kBatchElems * sizeof(float);   // 8192
    const int64_t b0 = (int64_t)blockIdx.x * f.k;
    int nb;                                                       // batches of this block
    if (f.interleave) {
        const int64_t mine = f.chunks > blockIdx.x ? (f.chunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
        nb = (int)(mine * kFlatGroup);
        // the tensor's last chunk may be short; it belongs to block (chunks - 1) % grid
        if (mine > 0 && (f.chunks - 1) % gridDim.x == blockIdx.x) nb -= (int)(f.chunks * kFlatGroup - f.full);
    } else {
        nb = (int)(f.full - b0 < f.k ? (f.full > b0 ? f.full - b0 : 0) : f.k);
    }
    // i-th batch of this block -> batch index in the tensor
    auto batch_of = [&](int i) -> int64_t {
        if (!f.interleave) return b0 + i;
        return ((int64_t)(i / kFlatGroup) * gridDim.x + blockIdx.x) * kFlatGroup + (i % kFlatGroup);
    };
    // i-th batch of this block -> stage i % kFlatStages (armed with the byte count, then two copies)
    auto issue = [&](int i) {
        const int sg = i % kFlatStages;
        const int64_t Bs = batch_of(i);
        mbar_expect_tx(&s_bar[sg], 2 * kOpBytes);
        bulk_g2s(s_x + sg * kBatchElems, x + Bs * kBatchElems, kOpBytes, &s_bar[sg]);
        bulk_g2s(s_g + sg * kBatchElems, go + Bs * kBatchElems, kOpBytes, &s_bar[sg]);
    };
    if (aux) {
        // ---- auxiliary warp: first thing, get the first batches moving; then refill a stage one
        // full iteration after its last shared-memory read (every compute thread is past the
        // compute of batch i-1 when it arrives at the barrier of iteration i)
        if (tid == kThreads && nb > 0) {
#pragma unroll
            for (int sg = 0; sg < kFlatStages; ++sg) {
                mbar_init(&s_bar[sg], 1);
                if (MBAR) mbar_init(&s_emp[sg], kThreads / 32);
            }
            mbar_fence_init();
            for (int i = 0; i < kFlatStages && i < nb; ++i) issue(i);
        }
        if (nb > 0) __syncthreads();                              // the mbarriers are initialised
        // (Releasing a stage through an "empty" mbarrier as soon as the four warps have copied it
        // to registers — two batches in flight during every compute phase — was measured: neutral
        // below 2^24 elements, 15-18 % SLOWER above, like a third stage or a fifth block per SM:
        // more requests in flight break up the moving band of DRAM pages.  profiles/r02_midsize.md)
        // Refill point: batch i+1 is issued once every compute warp has READ batch i (so exactly one
        // batch is in flight during a compute phase).  Two ways to learn that, chosen by size:
        //   block barrier per batch            — best below 2^26 elements (short kernels)
        //   "empty" mbarrier, warps never wait — 3 % faster from 2^27 (478 vs 495 us at 2^28),
        //     for each other (MBAR)              0.3-1.5 us slower below 2^26 (r02_exp_flat5.txt)
        if (MBAR) {
            if (tid == kThreads)
                for (int i = 1; i - 1 + kFlatStages < nb; ++i) {
                    mbar_wait(&s_emp[i % kFlatStages], (uint32_t)(i / kFlatStages) & 1u);
                    issue(i - 1 + kFlatStages);
                }
            __syncwarp();
        } else {
            for (int i = 0; i < nb; ++i) {
                __syncthreads();
                if (tid == kThreads && i >= 1 && i - 1 + kFlatStages < nb) issue(i - 1 + kFlatStages);
            }
        }
    } else {
    if ((tid & 31) == 0) {
#pragma unroll
        for (int m = 0; m < 5; ++m) s_acc[m][tid >> 5] = 0.0;
    }
    // the ragged tail (< one batch, up to 4 iterations) belongs to the last block: its loads are
    // in flight next to the TMA copies
    const bool owns_tail = (blockIdx.x == gridDim.x - 1) && f.rest_iters > 0;
    const int64_t r_it0 = owns_tail ? 0 : f.rest_iters;
    float4 rx[4], rg[4], rr4[4];
    bool rvalid[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int64_t it = r_it0 + u;
        const int64_t p = f.rest0 + it * kIterElems + tid * 4;
        rvalid[u] = (it < f.rest_iters) && (p < f.n);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        rx[u] = rvalid[u] ? ld_stream4(x + p) : z;
        rg[u] = rvalid[u] ? ld_stream4(go + p) : z;
        rr4[u] = (NOISE == NOISE_EXPLICIT && rvalid[u]) ? ld_stream4(r + p) : z;
    }
    PhiloxKey key = {0, 0, 0, 0};
    if (NOISE == NOISE_PHILOX) key = make_key(seed, offset, philox_dev);
    const int64_t supers_per_row = (f.n + kSuperElems - 1) / kSuperElems;
    const QConst q = load_qconst(prm, 0);
    BwdConst bc;
    bc.smul = q.s;
    bc.rcp = __frcp_rn(q.s);
    bc.lo_lt_hi = q.lo < q.hi;
    bc.lo_gt_hi = q.lo > q.hi;
    bc.delta = 0.f;
    const bool fast_ok = scale_fast_ok(q.s) && (!CLAMP || bc.lo_lt_hi);
    PairConst pc;
    pc.d = make_div2(q.s, bc.rcp);
    pc.zpn = bc2(-q.zp);
    pc.c = bc2(kInvSqrt3);
    pc.half = bc2(0.5f);
    Acc acc = {0.f, 0.f, 0.f, 0.f, 0.f};
    Acc2 a2 = {0ull, 0ull, 0ull};
    uint4 rnd = make_uint4(0, 0, 0, 0);
    int64_t curT = -1;
    int in_group = 0;

    // ---- ragged tail: up to 4 single iterations (the element position decides the noise) ----
    {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (!rvalid[u]) continue;
            const int64_t p = f.rest0 + (r_it0 + u) * kIterElems + tid * 4;
            const int64_t git = (f.rest0 >> 9) + r_it0 + u;          // global iteration index (512 elements)
            uint32_t inv = 0;
            if (NOISE == NOISE_PHILOX) {
                const int64_t T = git >> 5;                          // 32 iterations per super-tile
                if (T != curT) {
                    rnd = noise_block(key, 0, supers_per_row, T, tid);
                    curT = T;
                }
                inv = ~noise_nibble(rnd, (int)(git & 31));
            }
            float4 o;
            // (smallest non-zero |go| >= 2^-56, else the exact IEEE division: same guard as a batch)
            const bool odd = nzmin4(0xffffffffu, rg[u]) < kGoLoBits2m1;
            if (fast_ok && !odd) {
                bwd_pair_fast<METHOD, CLAMP, NOISE>(rx[u].x, rx[u].y, rg[u].x, rg[u].y, rr4[u].x, rr4[u].y,
                                                    inv << 31, inv << 30, q, pc, a2, acc, o.x, o.y);
                bwd_pair_fast<METHOD, CLAMP, NOISE>(rx[u].z, rx[u].w, rg[u].z, rg[u].w, rr4[u].z, rr4[u].w,
                                                    inv << 29, inv << 28, q, pc, a2, acc, o.z, o.w);
            } else {
                o.x = bwd_elem<METHOD, CLAMP, NOISE, false, false>(rx[u].x, rg[u].x, rr4[u].x, inv << 31, q, bc, acc);
                o.y = bwd_elem<METHOD, CLAMP, NOISE, false, false>(rx[u].y, rg[u].y, rr4[u].y, inv << 30, q, bc, acc);
                o.z = bwd_elem<METHOD, CLAMP, NOISE, false, false>(rx[u].z, rg[u].z, rr4[u].z, inv << 29, q, bc, acc);
                o.w = bwd_elem<METHOD, CLAMP, NOISE, false, false>(rx[u].w, rg[u].w, rr4[u].w, inv << 28, q, bc, acc);
            }
            if (gx) st_stream4(gx + p, o);
        }
        // BLOCK-uniform (never per-thread: the fold below runs full-mask warp shuffles)
        if (owns_tail) ++in_group;
    }

    // ---- main region: nb aligned batches through the TMA ring ----
    if (nb > 0) __syncthreads();                                 // the mbarriers are initialised
    for (int i = 0; i < nb; ++i) {
        const int64_t B = batch_of(i);
        const int st = i % kFlatStages;
        const int64_t base = B * kBatchElems + tid * 4;
        const int it0 = (int)(B & 7) * kU;                       // iteration index inside the super-tile
        uint32_t nw = 0;
        if (NOISE == NOISE_PHILOX) {
            const int64_t T = B >> 3;                            // 8 batches per 16384-element super-tile
            if (T != curT) {
                rnd = noise_block(key, 0, supers_per_row, T, tid);
                curT = T;
            }
            const int wi = it0 >> 3;                             // 32-bit word of the 128-bit block
            nw = ~((wi < 2) ? ((wi == 0) ? rnd.x : rnd.y) : ((wi == 2) ? rnd.z : rnd.w));
            if (it0 & 4) nw >>= 16;                              // second half of the word's 8 iterations
        }
        mbar_wait(&s_bar[st], (uint32_t)(i / kFlatStages) & 1u);
        float4 xv[kU], gv[kU], rv4[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            xv[u] = *reinterpret_cast<const float4 *>(s_x + st * kBatchElems + u * kIterElems + tid * 4);
            gv[u] = *reinterpret_cast<const float4 *>(s_g + st * kBatchElems + u * kIterElems + tid * 4);
            rv4[u] = (NOISE == NOISE_EXPLICIT) ? ld_stream4(r + base + u * kIterElems)
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        // (!MBAR) every thread is past the compute of batch i-1 here: the auxiliary warp refills
        // that batch's stage behind this barrier
        if (!MBAR) __syncthreads();
        if (fast_ok) {
            uint32_t mn = 0xffffffffu;
#pragma unroll
            for (int u = 0; u < kU; ++u) mn = nzmin4(mn, gv[u]);
            const bool odd = mn < kGoLoBits2m1;
            if (MBAR) {      // the staged operands are in registers (mn depends on the last load issued)
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&s_emp[st]);
            }
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const int64_t p = base + u * kIterElems;
                constexpr int kTop = 31;
                const int sh = u * 4;
                float4 o;
                bwd_pair_fast<METHOD, CLAMP, NOISE>(xv[u].x, xv[u].y, gv[u].x, gv[u].y, rv4[u].x, rv4[u].y,
                                                    nw << (kTop - sh - 0), nw << (kTop - sh - 1), q, pc, a2, acc, o.x, o.y);
                bwd_pair_fast<METHOD, CLAMP, NOISE>(xv[u].z, xv[u].w, gv[u].z, gv[u].w, rv4[u].z, rv4[u].w,
                                                    nw << (kTop - sh - 2), nw << (kTop - sh - 3), q, pc, a2, acc, o.z, o.w);
                if (gx) st_stream4(gx + p, o);
            }
            if (odd && gx)   // rare: exact IEEE division for the input gradient
                fix_batch_exact<METHOD, CLAMP>(x, go, gx, base, q, bc.smul, bc.delta);
        } else {
            // out-of-range scale / lo >= hi: true IEEE division on the staged operands
#pragma unroll 1
            for (int u = 0; u < kU; ++u) {
                const int64_t p = base + (int64_t)u * kIterElems;
                uint32_t inv = 0;
                if (NOISE == NOISE_PHILOX) inv = ~noise_nibble(rnd, it0 + u);
                const float4 xe = *reinterpret_cast<const float4 *>(s_x + st * kBatchElems + u * kIterElems + tid * 4);
                const float4 ge = *reinterpret_cast<const float4 *>(s_g + st * kBatchElems + u * kIterElems + tid * 4);
                float4 re = make_float4(0.f, 0.f, 0.f, 0.f);
                if (NOISE == NOISE_EXPLICIT) re = ld_stream4(r + p);
                float4 o;
                o.x = bwd_elem<METHOD, CLAMP, NOISE, false, false>(xe.x, ge.x, re.x, inv << 31, q, bc, acc);
                o.y = bwd_elem<METHOD, CLAMP, NOISE, false, false>(xe.y, ge.y, re.y, inv << 30, q, bc, acc);
                o.z = bwd_elem<METHOD, CLAMP, NOISE, false, false>(xe.z, ge.z, re.z, inv << 29, q, bc, acc);
                o.w = bwd_elem<METHOD, CLAMP, NOISE, false, false>(xe.w, ge.w, re.w, inv << 28, q, bc, acc);
                if (gx) st_stream4(gx + p, o);
            }
            if (MBAR) {
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&s_emp[st]);
            }
        }
        if (++in_group == kFlatGroup) {
            flat_fold<CLAMP>(acc, a2, s_acc);
            in_group = 0;
        }
    }
    if (in_group) flat_fold<CLAMP>(acc, a2, s_acc);
    }   // compute warps
    // (exp_flags: timing experiments only — MHAQ_FQ_FLAT_EXP=1 skips the reduction epilogue, the
    // parameter gradients are then NOT produced; never set in production)
    if (exp_flags & 1) return;
    __syncthreads();
    // ---- records without fence or ticket: every block but block 0 stores its encoded record and
    // leaves; block 0 polls the record words until they are non-zero, sums them in index order
    // (thread t takes records t, t + 160, ...) and writes zero back.  One store -> load hand-over
    // on the critical path instead of store, fence, atomic, load: 1.6-1.9 us less per call
    // (profiles/r02_midsize.md).  Block 0 owns a full share of the work, so it starts polling
    // when the other blocks are finishing too: a reader that polls EARLY (the last block, which
    // owns the short remainder, was tried) pulls the record lines towards itself and slows the
    // hand-over down (+4 us at 12.8 M elements).  The grid is at most SMs x 4 blocks, all
    // resident together; were it ever not, block 0 holds one slot while every other block runs
    // to completion, so the wait ends — and a bounded spin traps instead of hanging.
    unsigned long long *recs = reinterpret_cast<unsigned long long *>(ticket + kFlatRecOffsetU32);
    const int last = (int)gridDim.x - 1;
    constexpr int reader = 0;
    if ((int)blockIdx.x != reader) {
        if (tid == kThreads) {
            double v[5];
#pragma unroll
            for (int m = 0; m < 5; ++m) {
                double a = 0.0;
#pragma unroll
                for (int w = 0; w < kThreads / 32; ++w) a += s_acc[m][w];
                v[m] = a;
            }
            unsigned long long *rec = recs + (int64_t)blockIdx.x * kFlatRecWords;
            st_rec2(rec + 0, flat_enc(v[0]), flat_enc(v[1]));
            st_rec2(rec + 2, flat_enc(v[2]), flat_enc(v[3]));
            st_rec2(rec + 4, flat_enc(v[4]), 1ull);
        }
        return;
    }
    double a[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    constexpr int kPerThread = (kFlatCapMax + kFlatThreads - 1) / kFlatThreads;
    for (int k0 = 0; k0 < kPerThread; k0 += 4) {
        if (tid + k0 * kFlatThreads > last) break;
        unsigned long long w[4][kFlatRecWords];
        // first pass: all loads of up to 4 records in flight at once
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = tid + (k0 + k) * kFlatThreads;
            if (i <= last && i != reader) {
                const unsigned long long *rec = recs + (int64_t)i * kFlatRecWords;
                ld_rec2(rec + 0, w[k][0], w[k][1]);
                ld_rec2(rec + 2, w[k][2], w[k][3]);
                ld_rec2(rec + 4, w[k][4], w[k][5]);
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = tid + (k0 + k) * kFlatThreads;
            if (i <= last && i != reader) {
                unsigned long long *rec = recs + (int64_t)i * kFlatRecWords;
                unsigned int spins = 0;
                while (!(w[k][0] && w[k][1] && w[k][2] && w[k][3] && w[k][4] && w[k][5])) {
                    if (++spins > (1u << 24)) __trap();      // a lost block: fail loudly, never hang
                    ld_rec2(rec + 0, w[k][0], w[k][1]);
                    ld_rec2(rec + 2, w[k][2], w[k][3]);
                    ld_rec2(rec + 4, w[k][4], w[k][5]);
                }
                st_rec2(rec + 0, 0ull, 0ull);                // leave the region zero for the next launch
                st_rec2(rec + 2, 0ull, 0ull);
                st_rec2(rec + 4, 0ull, 0ull);
#pragma unroll
                for (int m = 0; m < 5; ++m) a[m] += flat_dec(w[k][m]);
            } else if (i == reader) {                        // this block's own record: from shared memory
#pragma unroll
                for (int m = 0; m < 5; ++m) {
                    double b = 0.0;
#pragma unroll
                    for (int ww = 0; ww < kThreads / 32; ++ww) b += s_acc[m][ww];
                    a[m] += b;
                }
            }
        }
    }
    block_sum_cols<5>(a, s_fin);
    if (tid == 0) emit_param_grads(prm, 0, a, o0, o1, o2, o3);
}

// ===========================================================================
// AEWGS statistics (gdnsq.py:118-124)
// ===========================================================================
template <bool VEC>
__global__ void __launch_bounds__(kThreads)
fq_aewgs_stats_kernel(const float *__restrict__ go, const float *__restrict__ x, QParams prm, Geom g,
                      int codegrad, double *__restrict__ ws) {
    const int tid = threadIdx.x;
    __shared__ float s_red[3][kThreads / 32];
    for (int64_t t = blockIdx.x; t < g.n_tasks; t += gridDim.x) {
        const Task k = make_task(g, t);
        const QConst q = load_qconst(prm, k.ch);
        const float smul = codegrad ? 1.f : q.s;
        const float rcp = __frcp_rn(q.s);
        const bool fast_ok = VEC && scale_fast_ok(q.s);
        const float *xr = x + k.row_off;
        const float *gr = go + k.row_off;
        float a_num = 0.f, a_e2 = 0.f, a_e = 0.f;
        for (int64_t sub = k.q0; sub < k.q1; ++sub) {
            const int64_t base = sub * kSubElems + tid * 4;
            const bool full = (sub + 1) * kSubElems <= g.n_inner;
            if (fast_ok && full) {
                // ---- fast path: full aligned sub-tile, division by the hoisted reciprocal
                // (bit-identical to IEEE division, see div_exact; |x| > 2^80 -> general path) ----
#pragma unroll
                for (int b = 0; b < kSubIters / kU; ++b) {
                    float4 xv[kU], gv[kU];
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        const int64_t p = base + (b * kU + u) * kIterElems;
                        xv[u] = ld_stream4(xr + p);
                        gv[u] = ld_stream4(gr + p);
                    }
                    float mx = 0.f;
#pragma unroll
                    for (int u = 0; u < kU; ++u) mx = absmax4(mx, xv[u]);
                    const bool huge = mx > kXHi;
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        const float xe[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
                        const float ge[4] = {gv[u].x, gv[u].y, gv[u].z, gv[u].w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float uu = f_sub(f_clamp(xe[i], q.lo, q.hi), q.zp);
                            const float v = huge ? f_div(uu, q.s) : div_exact(uu, q.s, rcp);
                            const float e = f_sub(rintf(v), v);
                            const float gg = f_mul(ge[i], smul);
                            const float sg = (gg > 0.f) ? 1.f : ((gg < 0.f) ? -1.f : 0.f);
                            a_num += f_mul(sg, e);
                            a_e2 += f_mul(e, e);
                            a_e += e;
                        }
                    }
                }
                continue;
            }
#pragma unroll 1
            for (int b = 0; b < kSubIters / kU; ++b) {
                float4 xv[kU], gv[kU];
                int nv[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int64_t p = base + (int64_t)(b * kU + u) * kIterElems;
                    nv[u] = full ? 4 : valid4<VEC>(p, g.n_inner);
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    xv[u] = nv[u] ? load4<VEC>(xr, p, g.n_inner) : z;
                    gv[u] = nv[u] ? load4<VEC>(gr, p, g.n_inner) : z;
                }
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const float xe[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
                    const float ge[4] = {gv[u].x, gv[u].y, gv[u].z, gv[u].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (i < nv[u]) {
                            const float c = f_clamp(xe[i], q.lo, q.hi);
                            const float v = f_div(f_sub(c, q.zp), q.s);
                            const float e = f_sub(rintf(v), v);
                            const float gg = f_mul(ge[i], smul);
                            const float sg = (gg > 0.f) ? 1.f : ((gg < 0.f) ? -1.f : 0.f);
                            a_num += f_mul(sg, e);
                            a_e2 += f_mul(e, e);
                            a_e += e;
                        }
                    }
                }
            }
        }
        float v0 = warp_sum(a_num), v1 = warp_sum(a_e2), v2 = warp_sum(a_e);
        if ((tid & 31) == 0) {
            const int w = tid >> 5;
            s_red[0][w] = v0; s_red[1][w] = v1; s_red[2][w] = v2;
        }
        __syncthreads();
        if (tid < 3) {
            double a = 0.0;
#pragma unroll
            for (int w = 0; w < kThreads / 32; ++w) a += (double)s_red[tid][w];
            ws[t * kNPart + tid] = a;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
fq_aewgs_stats_finalize_kernel(const double *ws, Geom g, float *__restrict__ stats) {
    __shared__ double s[3][256];

    const int64_t ch = blockIdx.x;
    const int64_t rows_per_ch = g.n_rows / g.n_ch;
    const int64_t recs = rows_per_ch * g.tasks_per_row;
    double a[3] = {0, 0, 0};
    for (int64_t i = threadIdx.x; i < recs; i += 256) {
        const int64_t rr = i / g.tasks_per_row;
        const int64_t j = i - rr * g.tasks_per_row;
        const int64_t t = (rr * g.n_ch + ch) * g.tasks_per_row + j;
#pragma unroll
        for (int m = 0; m < 3; ++m) a[m] += __ldcg(ws + t * kNPart + m);
    }
#pragma unroll
    for (int m = 0; m < 3; ++m) s[m][threadIdx.x] = a[m];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
#pragma unroll
            for (int m = 0; m < 3; ++m) s[m][threadIdx.x] += s[m][threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double cnt = (double)rows_per_ch * (double)g.n_inner;
#pragma unroll
        for (int m = 0; m < 3; ++m) stats[m * g.n_ch + ch] = (float)(s[m][0] / cnt);
    }
}

// ===========================================================================
// Noise materialisation (tests / parity): r = bit - 0.5
// ===========================================================================
__global__ void __launch_bounds__(kThreads)
fq_noise_kernel(float *__restrict__ r, Geom g, uint64_t seed, uint64_t offset,
                const uint64_t *__restrict__ philox_dev) {
    const int tid = threadIdx.x;
    const PhiloxKey key = make_key(seed, offset, philox_dev);
    const int64_t supers_per_row = (g.n_inner + kSuperElems - 1) / kSuperElems;
    for (int64_t t = blockIdx.x; t < g.n_tasks; t += gridDim.x) {
        const Task k = make_task(g, t);
        float *rr = r + k.row_off;
        for (int64_t sub = k.q0; sub < k.q1; ++sub) {
            const uint4 rnd = noise_block(key, k.row, supers_per_row, sub / kSuperSubs, tid);
            const int it0 = (int)(sub & (kSuperSubs - 1)) * kSubIters;
            for (int it = 0; it < kSubIters; ++it) {
                const int64_t p = sub * kSubElems + (int64_t)it * kIterElems + tid * 4;
                const uint32_t nib = noise_nibble(rnd, it0 + it);
                for (int e = 0; e < 4; ++e)
                    if (p + e < g.n_inner) rr[p + e] = ((nib >> e) & 1u) ? 0.5f : -0.5f;
            }
        }
    }
}

// ===========================================================================
// Row statistics (amin / amax with tie counts) and their backward
// ===========================================================================
struct RowStat {
    float mn, mx, cmn, cmx;
};
__device__ __forceinline__ void rs_push(RowStat &a, float v) {
    if (v < a.mn) { a.mn = v; a.cmn = 1.f; } else if (v == a.mn) { a.cmn += 1.f; }
    if (v > a.mx) { a.mx = v; a.cmx = 1.f; } else if (v == a.mx) { a.cmx += 1.f; }
}
__device__ __forceinline__ void rs_merge(RowStat &a, const RowStat &b) {
    if (b.mn < a.mn) { a.mn = b.mn; a.cmn = b.cmn; } else if (b.mn == a.mn) { a.cmn += b.cmn; }
    if (b.mx > a.mx) { a.mx = b.mx; a.cmx = b.cmx; } else if (b.mx == a.mx) { a.cmx += b.cmx; }
}

// One CTA per row (rows are weight rows: short).  Deterministic: the merge is
// associative and commutative on (value, count) pairs.
__global__ void __launch_bounds__(kThreads)
fq_rowstat_kernel(const float *__restrict__ x, int64_t n_rows, int64_t n_inner,
                  float *__restrict__ row_min, float *__restrict__ row_max,
                  float *__restrict__ n_at_min, float *__restrict__ n_at_max) {
    __shared__ RowStat s[kThreads / 32];
    const int tid = threadIdx.x;
    for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const float *xr = x + row * n_inner;
        RowStat a = {INFINITY, -INFINITY, 0.f, 0.f};
        const bool vec = ((n_inner & 3) == 0) && ((reinterpret_cast<uintptr_t>(xr) & 15) == 0);
        if (vec) {
            for (int64_t p = tid * 4; p < n_inner; p += kIterElems) {
                const float4 v = ld_stream4(xr + p);
                rs_push(a, v.x); rs_push(a, v.y); rs_push(a, v.z); rs_push(a, v.w);
            }
        } else {
            for (int64_t p = tid; p < n_inner; p += kThreads) rs_push(a, __ldg(xr + p));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            RowStat b;
            b.mn = __shfl_xor_sync(0xffffffffu, a.mn, o);
            b.mx = __shfl_xor_sync(0xffffffffu, a.mx, o);
            b.cmn = __shfl_xor_sync(0xffffffffu, a.cmn, o);
            b.cmx = __shfl_xor_sync(0xffffffffu, a.cmx, o);
            rs_merge(a, b);
        }
        if ((tid & 31) == 0) s[tid >> 5] = a;
        __syncthreads();
        if (tid == 0) {
            RowStat z = s[0];
            for (int w = 1; w < kThreads / 32; ++w) rs_merge(z, s[w]);
            if (row_min) row_min[row] = z.mn;
            if (row_max) row_max[row] = z.mx;
            if (n_at_min) n_at_min[row] = z.cmn;
            if (n_at_max) n_at_max[row] = z.cmx;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kThreads)
fq_rowstat_bwd_kernel(const float *__restrict__ gx, const float *__restrict__ x, int64_t n_rows,
                      int64_t n_inner, const float *__restrict__ row_min,
                      const float *__restrict__ n_at_min, const float *__restrict__ g_min,
                      const float *__restrict__ row_max, const float *__restrict__ n_at_max,
                      const float *__restrict__ g_max, float *__restrict__ out) {
    const int tid = threadIdx.x;
    for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const int64_t off = row * n_inner;
        float mn = 0.f, mx = 0.f, dmn = 0.f, dmx = 0.f;
        const bool has_mn = g_min != nullptr, has_mx = g_max != nullptr;
        if (has_mn) { mn = row_min[row]; dmn = f_div(g_min[row], n_at_min[row]); }
        if (has_mx) { mx = row_max[row]; dmx = f_div(g_max[row], n_at_max[row]); }
        for (int64_t p = tid; p < n_inner; p += kThreads) {
            const float xv = __ldg(x + off + p);
            float o = gx ? __ldg(gx + off + p) : 0.f;
            if (has_mn && xv == mn) o = f_add(o, dmn);
            if (has_mx && xv == mx) o = f_add(o, dmx);
            out[off + p] = o;
        }
    }
}

#include "fq_wrow.cuh"
#include "fq_loss.cuh"
#include "fq_pack.cuh"
#include "fq_igemm.cuh"

// ===========================================================================
// Host-side launch helpers
// ===========================================================================
inline int check_common(const void *x, const float *scale, const float *zp, int64_t n_rows,
                        int64_t n_inner, int64_t n_ch) {
    if (!x || !scale || !zp) return MHAQ_FQ_ENULL;
    if (n_rows < 0 || n_inner < 0 || n_ch < 1) return MHAQ_FQ_EINVAL;
    if (n_rows > 0 && (n_rows % n_ch) != 0) return MHAQ_FQ_EINVAL;
    return 0;
}
inline bool stride_ok(int s) { return s == 0 || s == 1; }
inline bool mode_ok(int m) { return m >= PARAMS_LINEAR && m <= PARAMS_UNIT; }
// ACT_LOG needs all of log_act_s (scale), act_b (zp) and log_act_q (lo) and is per-tensor
inline int check_mode(int mode, const float *lo, int64_t n_ch) {
    if (!mode_ok(mode)) return MHAQ_FQ_EINVAL;
    if (mode == PARAMS_ACT_LOG && !lo) return MHAQ_FQ_ENULL;
    if (mode == PARAMS_ACT_LOG && n_ch != 1) return MHAQ_FQ_EINVAL;
    return 0;
}
inline bool has_clamp(int mode, const float *lo, const float *hi) {
    return mode == PARAMS_ACT_LOG || (mode == PARAMS_LINEAR && (lo != nullptr || hi != nullptr));
}
inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

inline int grid_for(int64_t n_tasks) {
    // Non-persistent: one CTA per task, hardware block scheduler balances the
    // SMs.  (Tasks are >= 4096 elements so a 2^31-1 grid covers 8 Ti elements.)
    const int64_t cap = 0x7fffffffLL;
    return (int)(n_tasks < cap ? n_tasks : cap);
}

// experiment knob (not part of the ABI): MHAQ_FQ_BWD_SPT / MHAQ_FQ_FWD_SPT force the
// sub-tiles-per-task of the reducing / streaming kernels (power of two).
inline int env_int(const char *name) {
    const char *e = getenv(name);
    return e ? atoi(e) : 0;
}
inline Geom stream_geom(int64_t n_rows, int64_t n_inner, int64_t n_ch) {
    static const int ov = env_int("MHAQ_FQ_FWD_SPT");
    return make_geom(n_rows, n_inner, n_ch, GEOM_STREAM, ov);
}
inline Geom reduce_geom(int64_t n_rows, int64_t n_inner, int64_t n_ch) {
    static const int ov = env_int("MHAQ_FQ_BWD_SPT");
    return make_geom(n_rows, n_inner, n_ch, GEOM_REDUCE, ov);
}

inline int last_error() {
    cudaError_t e = cudaGetLastError();
    return (int)e;
}

// Launch a finalize kernel as a programmatic dependent of the kernel before it in the stream
// (see pdl_wait / pdl_trigger).  MHAQ_FQ_NO_PDL=1 falls back to an ordinary launch.
template <typename... KArgs, typename... Args>
int launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t st, Args... args) {
    static const int no_pdl = env_int("MHAQ_FQ_NO_PDL");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = no_pdl ? 0 : 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
    if (e != cudaSuccess) return (int)e;
    return last_error();
}

template <int METHOD, bool CLAMP, int NOISE>
int launch_bwd(bool vec, int grid, cudaStream_t st, const float *go, const float *x, float *gx,
               const QParams &prm, const Geom &g, int codegrad, const float *r, uint64_t seed,
               uint64_t offset, const uint64_t *philox_dev, const float *stats, double *ws) {
#define MHAQ_LAUNCH(V, C)                                                             \
    fq_bwd_kernel<METHOD, CLAMP, NOISE, V, C><<<grid, kThreads, 0, st>>>(             \
        go, x, gx, prm, g, r, seed, offset, philox_dev, stats, ws)
    if (vec && !codegrad) MHAQ_LAUNCH(true, false);
    else if (vec) MHAQ_LAUNCH(true, true);
    else if (!codegrad) MHAQ_LAUNCH(false, false);
    else MHAQ_LAUNCH(false, true);
#undef MHAQ_LAUNCH
    return last_error();
}

template <int METHOD, bool CLAMP>
int launch_bwd_noise(bool explicit_r, bool vec, int grid, cudaStream_t st, const float *go,
                     const float *x, float *gx, const QParams &prm, const Geom &g, int codegrad,
                     const float *r, uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                     const float *stats, double *ws) {
    if (METHOD == MHAQ_FQ_LSQ)
        return launch_bwd<METHOD, CLAMP, NOISE_NONE>(vec, grid, st, go, x, gx, prm, g, codegrad, r,
                                                     seed, offset, philox_dev, stats, ws);
    if (explicit_r)
        return launch_bwd<METHOD, CLAMP, NOISE_EXPLICIT>(vec, grid, st, go, x, gx, prm, g, codegrad,
                                                         r, seed, offset, philox_dev, stats, ws);
    return launch_bwd<METHOD, CLAMP, NOISE_PHILOX>(vec, grid, st, go, x, gx, prm, g, codegrad, r,
                                                   seed, offset, philox_dev, stats, ws);
}

template <int METHOD, int NOISE>
int launch_wrow_bwd(bool vec, int grid, cudaStream_t st, const float *go, const float *w,
                    const WRowArgs &a, const float *row_min, const float *row_max, const float *g_lr,
                    const float *g_mn, const float *g_mx, const float *r, uint64_t seed,
                    uint64_t offset, const uint64_t *philox_dev, float *gw, float *g_log_s) {
    if (vec)
        fq_wrow_bwd_kernel<METHOD, NOISE, true><<<grid, kThreads, 0, st>>>(
            go, w, a, row_min, row_max, g_lr, g_mn, g_mx, r, seed, offset, philox_dev, gw, g_log_s);
    else
        fq_wrow_bwd_kernel<METHOD, NOISE, false><<<grid, kThreads, 0, st>>>(
            go, w, a, row_min, row_max, g_lr, g_mn, g_mx, r, seed, offset, philox_dev, gw, g_log_s);
    return last_error();
}

// blocks the flat backward may use: SMs x resident CTAs (MHAQ_FQ_FLAT_CTAS_PER_SM overrides the
// per-SM factor for experiments)
inline int flat_cap() {
    static int cap = 0;
    if (cap == 0) {
        int dev = 0, sms = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
            sms = 148;
        // 4 blocks per SM measured best (profiles/r02_midsize.md): 5 fit, but the fifth adds
        // DRAM / L2 contention, not bandwidth
        const int per_sm = env_int("MHAQ_FQ_FLAT_CTAS_PER_SM");
        cap = sms * (per_sm > 0 ? per_sm : kFlatCtasPerSm);
    }
    return cap;
}
// Largest tensor (elements) the flat backward takes.  With the interleaved partition and the
// mbarrier-released ring it beats the dynamically scheduled streaming kernel + finalize launch at
// every size measured (2^30: 1877 vs 1981 us), so there is no upper limit in practice.
// MHAQ_FQ_FLAT_MAX_LOG2 overrides (0 disables the flat kernel).
inline int64_t flat_max_elems() {
    static int64_t mx = -1;
    if (mx < 0) {
        const char *e = getenv("MHAQ_FQ_FLAT_MAX_LOG2");
        const int l2 = e ? atoi(e) : 40;
        mx = l2 <= 0 ? 0 : (int64_t)1 << (l2 > 62 ? 62 : l2);
    }
    return mx;
}
// Tensors of at least this many elements use the interleaved (moving band) partition.
inline int64_t flat_interleave_min() {
    static int64_t mn = -1;
    if (mn < 0) {
        const char *e = getenv("MHAQ_FQ_FLAT_INTERLEAVE_LOG2");
        const int l2 = e ? atoi(e) : 24;
        mn = (int64_t)1 << (l2 < 0 ? 0 : (l2 > 62 ? 62 : l2));
    }
    return mn;
}
// Tensors of at least this many elements release the staging ring through mbarriers instead of a
// block barrier per batch (see the kernel).
inline int64_t flat_mbar_min() {
    static int64_t mn = -1;
    if (mn < 0) {
        const char *e = getenv("MHAQ_FQ_FLAT_MBAR_LOG2");
        const int l2 = e ? atoi(e) : 26;
        mn = (int64_t)1 << (l2 < 0 ? 0 : (l2 > 62 ? 62 : l2));
    }
    return mn;
}
inline int flat_exp_flags() {
    static const int v = env_int("MHAQ_FQ_FLAT_EXP");
    return v;
}
inline bool flat_shape_ok(int64_t n_rows, int64_t n_inner, int64_t n_ch, int method, int codegrad) {
    return n_rows == 1 && n_ch == 1 && !codegrad && (n_inner % 4 == 0) && n_inner <= flat_max_elems() &&
           (method == MHAQ_FQ_STE || method == MHAQ_FQ_LSQ);
}

template <int METHOD, bool CLAMP>
int launch_bwd_flat(bool explicit_r, const FlatGeom &f, cudaStream_t st, const float *go, const float *x,
                    float *gx, const QParams &prm, const float *r, uint64_t seed, uint64_t offset,
                    const uint64_t *philox_dev, double *ws, unsigned int *ticket, float *o0, float *o1,
                    float *o2, float *o3) {
#define MHAQ_FLAT2(N, M)                                                                          \
    do {                                                                                          \
        static bool attr_set = false;                                                             \
        if (!attr_set) {                                                                          \
            cudaFuncSetAttribute(fq_bwd_flat_kernel<METHOD, CLAMP, N, M>,                         \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, kFlatSmemBytes);    \
            attr_set = true;                                                                      \
        }                                                                                         \
        fq_bwd_flat_kernel<METHOD, CLAMP, N, M><<<f.grid, kFlatThreads, kFlatSmemBytes, st>>>(    \
            go, x, gx, prm, f, r, seed, offset, philox_dev, ws, ticket, o0, o1, o2, o3,           \
            flat_exp_flags());                                                                    \
    } while (0)
#define MHAQ_FLAT(N)                                                                              \
    do {                                                                                          \
        if (f.n >= flat_mbar_min()) MHAQ_FLAT2(N, true);                                          \
        else MHAQ_FLAT2(N, false);                                                                \
    } while (0)
    if (METHOD == MHAQ_FQ_LSQ) MHAQ_FLAT(NOISE_NONE);
    else if (explicit_r) MHAQ_FLAT(NOISE_EXPLICIT);
    else MHAQ_FLAT(NOISE_PHILOX);
#undef MHAQ_FLAT2
#undef MHAQ_FLAT
    return last_error();
}

// shared by the multi-tensor backward and the multi-tensor AEWGS statistics: validate, chunk, pack
template <typename Launch>
int wrow_multi_bwd_chunks(const mhaq_fq_wrow_bwd_desc *descs, int n_tensors, Launch launch) {
    int64_t row_base = 0;
    for (int c0 = 0; c0 < n_tensors; c0 += kWRowMultiBwdMax) {
        WRowBwdMulti m;
        m.n = 0;
        m.row0[0] = 0;
        // (every tensor of the chunk keeps a slot, empty ones included: slot index == noise stream index)
        for (int i = c0; i < n_tensors && m.n < kWRowMultiBwdMax; ++i) {
            const mhaq_fq_wrow_bwd_desc &d = descs[i];
            const int k = m.n++;
            m.d[k] = {d.g_wq, d.w, d.log_scale, d.row_min, d.row_max, d.g_log_range, d.g_row_min,
                      d.g_row_max, d.r, d.g_w, d.g_log_scale, d.n_inner, d.g_log_scale_acc};
            m.vec[k] = (d.n_inner % 4 == 0) && aligned16(d.w) && aligned16(d.g_wq) &&
                       (!d.g_w || aligned16(d.g_w)) && (!d.r || aligned16(d.r));
            m.row0[k + 1] = m.row0[k] + (int)d.n_rows;
        }
        if (m.row0[m.n] > 0) {
            const int rc = launch(m, c0, row_base);
            if (rc) return rc;
        }
        row_base += m.row0[m.n];
    }
    return 0;
}

int wrow_multi_check(const mhaq_fq_wrow_bwd_desc *descs, int n_tensors, bool *explicit_r) {
    for (int i = 0; i < n_tensors; ++i) {
        const mhaq_fq_wrow_bwd_desc &d = descs[i];
        if (!d.g_wq || !d.w || !d.log_scale || !d.row_min || !d.row_max) return MHAQ_FQ_ENULL;
        if (d.n_rows < 0 || d.n_inner <= 0 || d.n_rows > 0x3fffffff) return MHAQ_FQ_EINVAL;
        if (i == 0) *explicit_r = d.r != nullptr;
        else if ((d.r != nullptr) != *explicit_r) return MHAQ_FQ_EINVAL;   // all explicit or all in-kernel
    }
    return 0;
}

// ---- packed codes (fq_pack.cuh) ----
inline bool pack_bits_ok(int bits) {
    return bits == 1 || bits == 2 || bits == 4 || bits == 8 || bits == 16;
}

template <int BITS>
void launch_pack(bool vec, bool clamp, int grid, cudaStream_t st, const float *x, uint8_t *packed,
                 const QParams &prm, const Geom &g, int64_t row_stride, unsigned long long *n_oor) {
    if (vec && clamp)
        fq_pack_kernel<BITS, true, true><<<grid, kThreads, 0, st>>>(x, packed, prm, g, row_stride, n_oor);
    else if (vec)
        fq_pack_kernel<BITS, true, false><<<grid, kThreads, 0, st>>>(x, packed, prm, g, row_stride, n_oor);
    else
        fq_pack_kernel<BITS, false, true><<<grid, kThreads, 0, st>>>(x, packed, prm, g, row_stride, n_oor);
}

template <int BITS>
void launch_unpack(bool vec, int grid, cudaStream_t st, const uint8_t *packed, float *y, const QParams &prm,
                   const Geom &g, int64_t row_stride) {
    if (vec)
        fq_unpack_kernel<BITS, true><<<grid, kThreads, 0, st>>>(packed, y, prm, g, row_stride);
    else
        fq_unpack_kernel<BITS, false><<<grid, kThreads, 0, st>>>(packed, y, prm, g, row_stride);
}

// ---- integer layers (fq_igemm.cuh) ----
// The iconv kernel needs more than 48 KiB of dynamic shared memory: opt in once per device and
// instantiation.
template <bool FUSED, bool GROUPED = false>
inline int iconv_smem_opt_in() {
    static bool done[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 64 && done[dev]) return 0;
    e = cudaFuncSetAttribute(fq_iconv_kernel<FUSED, GROUPED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)iconv_smem_bytes(kIcMaxTileN));
    if (e != cudaSuccess) return (int)e;
    if (dev < 64) done[dev] = true;
    return 0;
}

// Argument checks and kernel arguments shared by mhaq_fq_iconv_u8 and mhaq_fq_iconv_fused_u8 (no
// CUDA call); the epilogue fields of `a` are left zero and y to the caller.
inline int iconv_args(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                      const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                      int64_t batch, int64_t height, int64_t width, int64_t cp, int64_t n_out, int kernel_h,
                      int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int act_max_code,
                      int weight_max_code, IConvArgs &a, dim3 &grid) {
    if (!codes || !weights || !alpha || !beta || !ctab || !h_class || !w_class) return MHAQ_FQ_ENULL;
    if (batch < 1 || height < 1 || width < 1 || cp < 16 || cp % 16 != 0 || n_out < 1 || n_w_classes < 1)
        return MHAQ_FQ_EINVAL;
    if (kernel_h < 1 || kernel_w < 1 || stride_h < 1 || stride_w < 1 || pad_h < 0 || pad_w < 0)
        return MHAQ_FQ_EINVAL;
    if (act_max_code < 1 || act_max_code > 255 || weight_max_code < 1 || weight_max_code > 255)
        return MHAQ_FQ_EINVAL;
    if (!aligned16(codes) || !aligned16(weights)) return MHAQ_FQ_EINVAL;
    const int64_t ho = (height + 2 * pad_h - kernel_h) / stride_h + 1;
    const int64_t wo = (width + 2 * pad_w - kernel_w) / stride_w + 1;
    if (height + 2 * pad_h < kernel_h || width + 2 * pad_w < kernel_w) return MHAQ_FQ_EINVAL;
    const int64_t k_bytes = (int64_t)kernel_h * kernel_w * cp;
    // the int32 accumulator holds sum_k ca_k * cw_nk <= K * act_max_code * weight_max_code
    if (k_bytes > (int64_t)1 << 31 || k_bytes * act_max_code * weight_max_code >= ((int64_t)1 << 31))
        return MHAQ_FQ_EINVAL;
    const IcLayout l = iconv_layout(n_out, k_bytes);
    if (l.tile_n > kIcMaxTileN) return MHAQ_FQ_EINVAL;
    const int64_t m = batch * ho * wo;
    const int64_t m_tiles = (m + kIcTileM - 1) / kIcTileM;
    if (m_tiles > 0x7fffffffLL) return MHAQ_FQ_EINVAL;
    a = IConvArgs{};
    a.a = codes; a.b = weights; a.alpha = alpha; a.beta = beta; a.ctab = ctab;
    a.hcls = h_class; a.wcls = w_class;
    a.m = m; a.h = height; a.w = width; a.cp = cp; a.n_out = n_out; a.ho = ho; a.wo = wo;
    a.k_chunks = k_bytes / 16; a.k_stages = l.k_stages;
    a.kh = kernel_h; a.kw = kernel_w; a.sh = stride_h; a.sw = stride_w; a.ph = pad_h; a.pw = pad_w;
    a.n_wcls = n_w_classes; a.tile_n = l.tile_n; a.tile_out = l.tile_out;
    a.tmem_cols = 32;
    while (a.tmem_cols < l.tile_n) a.tmem_cols <<= 1;
    grid = dim3((unsigned)m_tiles, (unsigned)l.n_tiles);
    return 0;
}

// Checks of a fused epilogue (no CUDA call).
inline int iconv_epilogue_check(const mhaq_fq_iconv_epilogue *epilogue) {
    if (!epilogue) return MHAQ_FQ_ENULL;
    const mhaq_fq_iconv_epilogue &e = *epilogue;
    if (!e.y && !e.codes) return MHAQ_FQ_EINVAL;
    if (e.codes && (!e.code_scale || !e.code_zero_point || !e.code_max_val)) return MHAQ_FQ_ENULL;
    if (e.codes && !aligned16(e.codes)) return MHAQ_FQ_EINVAL;
    if (e.activation != MHAQ_FQ_ACT_NONE && e.activation != MHAQ_FQ_ACT_RELU &&
        e.activation != MHAQ_FQ_ACT_LEAKY_RELU)
        return MHAQ_FQ_EINVAL;
    return 0;
}

// The epilogue's fields of `a` (after iconv_epilogue_check; a.n_out is set).
inline void iconv_epilogue_set(const mhaq_fq_iconv_epilogue &e, IConvArgs &a) {
    a.y = e.y;
    a.vec_out = e.y && aligned16(e.y) && a.n_out % 4 == 0;
    a.res = e.residual;
    a.vec_res = e.residual && aligned16(e.residual) && a.n_out % 4 == 0;
    a.act = e.activation;
    a.slope = e.negative_slope;
    a.codes = e.codes;
    a.code_s = e.code_scale; a.code_zp = e.code_zero_point; a.code_hi = e.code_max_val;
    a.cp_out = (a.n_out + 15) / 16 * 16;
}

inline bool igroup_depthwise(int64_t n_in, int64_t n_out, int groups) { return groups == n_in && groups == n_out; }

// Geometry checks of a grouped / dilated layer (no CUDA call).
inline int igroup_geometry_ok(int64_t n_in, int64_t n_out, const mhaq_fq_iconv_geometry &g) {
    if (n_in < 1 || n_out < 1 || g.groups < 1 || n_in % g.groups != 0 || n_out % g.groups != 0) return 0;
    if (g.kernel_h < 1 || g.kernel_w < 1 || g.stride_h < 1 || g.stride_w < 1 || g.pad_h < 0 || g.pad_w < 0)
        return 0;
    return g.dilation_h >= 1 && g.dilation_w >= 1;
}

// Argument checks and kernel arguments of mhaq_fq_iconv_grouped_u8 (no CUDA call).
inline int igroup_args(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                       const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                       int64_t batch, int64_t height, int64_t width, int64_t n_in, int64_t n_out,
                       const mhaq_fq_iconv_geometry *geometry, int act_max_code, int weight_max_code,
                       const mhaq_fq_iconv_epilogue *epilogue, IConvArgs &a, IgPlan &l) {
    const int rc = iconv_epilogue_check(epilogue);
    if (rc) return rc;
    if (!codes || !weights || !alpha || !beta || !ctab || !h_class || !w_class || !geometry) return MHAQ_FQ_ENULL;
    const mhaq_fq_iconv_geometry g = *geometry;
    if (!igroup_geometry_ok(n_in, n_out, g)) return MHAQ_FQ_EINVAL;
    if (batch < 1 || height < 1 || width < 1 || n_w_classes < 1) return MHAQ_FQ_EINVAL;
    if (act_max_code < 1 || act_max_code > 255 || weight_max_code < 1 || weight_max_code > 255)
        return MHAQ_FQ_EINVAL;
    if (!aligned16(codes) || !aligned16(weights)) return MHAQ_FQ_EINVAL;
    // extent of the dilated kernel
    const int64_t eh = (int64_t)g.dilation_h * (g.kernel_h - 1) + 1, ew = (int64_t)g.dilation_w * (g.kernel_w - 1) + 1;
    if (height + 2 * g.pad_h < eh || width + 2 * g.pad_w < ew) return MHAQ_FQ_EINVAL;
    const int64_t ho = (height + 2 * g.pad_h - eh) / g.stride_h + 1;
    const int64_t wo = (width + 2 * g.pad_w - ew) / g.stride_w + 1;
    const int64_t cin_g = n_in / g.groups;
    // one channel's int32 sums: kh * kw * cin_g products, each at most act_max_code * weight_max_code
    const int64_t terms = (int64_t)g.kernel_h * g.kernel_w * cin_g;
    if (terms > (int64_t)1 << 31 || terms * act_max_code * weight_max_code >= ((int64_t)1 << 31))
        return MHAQ_FQ_EINVAL;
    a = IConvArgs{};
    const int64_t m = batch * ho * wo;
    const int64_t cp = (n_in + 15) / 16 * 16;
    if (igroup_depthwise(n_in, n_out, g.groups)) {
        l = IgPlan{};
    } else {
        l = igroup_plan(n_out, g.groups, cin_g, g.kernel_h, g.kernel_w);
        if ((m + kIcTileM - 1) / kIcTileM > 0x7fffffffLL || l.n_tiles > 65535) return MHAQ_FQ_EINVAL;
    }
    a.a = codes; a.b = weights; a.alpha = alpha; a.beta = beta; a.ctab = ctab;
    a.hcls = h_class; a.wcls = w_class;
    a.m = m; a.h = height; a.w = width; a.cp = cp; a.n_out = n_out; a.ho = ho; a.wo = wo;
    a.k_stages = l.k_stages;
    a.kh = g.kernel_h; a.kw = g.kernel_w; a.sh = g.stride_h; a.sw = g.stride_w; a.ph = g.pad_h; a.pw = g.pad_w;
    a.dh = g.dilation_h; a.dw = g.dilation_w;
    a.groups = g.groups; a.cin_g = cin_g; a.cout_g = n_out / g.groups;
    a.n_wcls = n_w_classes; a.tile_n = l.tile_n; a.tile_out = l.tile_out; a.gpt = l.gpt; a.parts = l.parts;
    a.tmem_cols = 32;
    while (a.tmem_cols < l.tile_n) a.tmem_cols <<= 1;
    iconv_epilogue_set(*epilogue, a);
    return 0;
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int mhaq_fq_abi_version(void) { return MHAQ_FQ_ABI_VERSION; }

unsigned long long mhaq_fq_stream_capture_id(void *stream) {
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    unsigned long long id = 0;
    if (cudaStreamGetCaptureInfo((cudaStream_t)stream, &status, &id) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return status == cudaStreamCaptureStatusActive ? id : 0;
}

const char *mhaq_fq_build_info(void) {
    return "mhaq_fq sm_100a fp32 fake-quant; cuda " __DATE__ " " __TIME__;
}

int64_t mhaq_fq_num_tasks(int64_t n_rows, int64_t n_inner) {
    if (n_rows <= 0 || n_inner <= 0) return 0;
    return stream_geom(n_rows, n_inner, 1).n_tasks;   // the finest decomposition any kernel uses
}

static inline int64_t n_slices_of(const Geom &g) {
    const int64_t recs = (g.n_rows / g.n_ch) * g.tasks_per_row;
    return (recs + kSliceRecs - 1) / kSliceRecs;
}

int64_t mhaq_fq_workspace_bytes(int64_t n_rows, int64_t n_inner) {
    if (n_rows <= 0 || n_inner <= 0) return (1 + kFlatCapMax) * kNPart * (int64_t)sizeof(double);
    const Geom gs = stream_geom(n_rows, n_inner, 1), gr = reduce_geom(n_rows, n_inner, 1);
    const int64_t tasks = gs.n_tasks > gr.n_tasks ? gs.n_tasks : gr.n_tasks;
    // records + slice records (at most one slice record per kSliceRecs records, >= 1 per row)
    const int64_t slices = tasks / kSliceRecs + n_rows + 1;
    // (the flat backward and the eval forward write at most kFlatCapMax per-CTA records)
    return (tasks + slices + kFlatCapMax) * kNPart * (int64_t)sizeof(double);
}

int64_t mhaq_fq_ticket_count(int64_t n_rows, int64_t n_inner, int64_t n_ch) {
    (void)n_rows; (void)n_inner;
    // per-channel tickets, then (16-byte aligned) the flat backward's self-validating records
    return (n_ch > 0 ? n_ch : 1) + kFlatRecOffsetU32 + (int64_t)kFlatCapMax * kFlatRecWords * 2;
}

int mhaq_fq_fwd_f32(const float *x, float *y, float *codes, const float *scale, const float *zp,
                    const float *lo, const float *hi, int scale_stride, int zp_stride,
                    int lo_stride, int hi_stride, int param_mode, int64_t n_rows, int64_t n_inner,
                    int64_t n_ch, double *minmax_ws, void *stream) {
    int rc = check_common(x, scale, zp, n_rows, n_inner, n_ch);
    if (rc) return rc;
    if ((rc = check_mode(param_mode, lo, n_ch)) != 0) return rc;
    if (!stride_ok(scale_stride) || !stride_ok(zp_stride) || !stride_ok(lo_stride) ||
        !stride_ok(hi_stride))
        return MHAQ_FQ_EINVAL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const Geom g = stream_geom(n_rows, n_inner, n_ch);
    const QParams prm = {scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride, param_mode};
    const bool vec = (n_inner % 4 == 0) && aligned16(x) && (!y || aligned16(y)) &&
                     (!codes || aligned16(codes));
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(g.n_tasks);
    const bool clamp = has_clamp(param_mode, lo, hi);
    if (minmax_ws) {      // eval statistics: one 16-byte record per task
        if (vec && clamp)
            fq_fwd_kernel<true, true, true><<<grid, kThreads, 0, st>>>(x, y, codes, prm, g, minmax_ws);
        else if (vec)
            fq_fwd_kernel<true, false, true><<<grid, kThreads, 0, st>>>(x, y, codes, prm, g, minmax_ws);
        else
            fq_fwd_kernel<false, true, true><<<grid, kThreads, 0, st>>>(x, y, codes, prm, g, minmax_ws);
        return last_error();
    }
    if (vec && clamp)
        fq_fwd_kernel<true, true, false><<<grid, kThreads, 0, st>>>(x, y, codes, prm, g, nullptr);
    else if (vec)
        fq_fwd_kernel<true, false, false><<<grid, kThreads, 0, st>>>(x, y, codes, prm, g, nullptr);
    else
        fq_fwd_kernel<false, true, false><<<grid, kThreads, 0, st>>>(x, y, codes, prm, g, nullptr);
    return last_error();
}

int mhaq_fq_minmax_finalize(const double *minmax_ws, int64_t n_rows, int64_t n_inner, float *out5,
                            void *stream) {
    if (!minmax_ws || !out5) return MHAQ_FQ_ENULL;
    const int64_t n_tasks = mhaq_fq_num_tasks(n_rows, n_inner);
    if (n_tasks <= 0) return MHAQ_FQ_EINVAL;
    return launch_pdl(fq_minmax_finalize_kernel, 1, kMmThreads, (cudaStream_t)stream, minmax_ws, n_tasks, out5);
}

int mhaq_fq_bwd_f32(const float *go, const float *x, float *gx, const float *scale,
                    const float *zp, const float *lo, const float *hi, int scale_stride,
                    int zp_stride, int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                    int64_t n_inner, int64_t n_ch, int method, int go_is_code_grad, const float *r,
                    uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                    const float *aewgs_stats, double *ws, void *stream) {
    int rc = check_common(x, scale, zp, n_rows, n_inner, n_ch);
    if (rc) return rc;
    if ((rc = check_mode(param_mode, lo, n_ch)) != 0) return rc;
    if (!go || !ws) return MHAQ_FQ_ENULL;
    if (!stride_ok(scale_stride) || !stride_ok(zp_stride) || !stride_ok(lo_stride) ||
        !stride_ok(hi_stride))
        return MHAQ_FQ_EINVAL;
    if (method < 0 || method > 3) return MHAQ_FQ_EINVAL;
    if (method == MHAQ_FQ_AEWGS && !aewgs_stats) return MHAQ_FQ_ENULL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const Geom g = reduce_geom(n_rows, n_inner, n_ch);
    const QParams prm = {scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride, param_mode};
    const bool vec = (n_inner % 4 == 0) && aligned16(x) && aligned16(go) &&
                     (!gx || aligned16(gx)) && (!r || aligned16(r));
    const bool clamp = has_clamp(param_mode, lo, hi);
    const bool er = (r != nullptr);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(g.n_tasks);
#define MHAQ_BWD(M)                                                                              \
    (clamp ? launch_bwd_noise<M, true>(er, vec, grid, st, go, x, gx, prm, g, go_is_code_grad, r, \
                                       seed, offset, philox_dev, aewgs_stats, ws)                \
           : launch_bwd_noise<M, false>(er, vec, grid, st, go, x, gx, prm, g, go_is_code_grad,   \
                                        r, seed, offset, philox_dev, aewgs_stats, ws))
    switch (method) {
        case MHAQ_FQ_STE: return MHAQ_BWD(MHAQ_FQ_STE);
        case MHAQ_FQ_EWGS: return MHAQ_BWD(MHAQ_FQ_EWGS);
        case MHAQ_FQ_AEWGS: return MHAQ_BWD(MHAQ_FQ_AEWGS);
        default: return MHAQ_BWD(MHAQ_FQ_LSQ);
    }
#undef MHAQ_BWD
}

static int bwd_finalize_impl(double *ws, unsigned int *tickets, const float *scale, const float *zp,
                             const float *lo, const float *hi, int scale_stride, int zp_stride,
                             int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                             int64_t n_inner, int64_t n_ch, float *g_scale, float *g_zp, float *g_lo,
                             float *g_hi, const float *const acc[4], void *stream) {
    if (!ws || !tickets) return MHAQ_FQ_ENULL;
    if (n_rows <= 0 || n_inner <= 0 || n_ch < 1 || (n_rows % n_ch) != 0) return MHAQ_FQ_EINVAL;
    int rc = check_mode(param_mode, lo, n_ch);
    if (rc) return rc;
    if (param_mode != PARAMS_LINEAR && !scale) return MHAQ_FQ_ENULL;
    const QParams prm = {scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride, param_mode,
                         acc ? acc[0] : nullptr, acc ? acc[1] : nullptr, acc ? acc[2] : nullptr,
                         acc ? acc[3] : nullptr};
    const Geom g = reduce_geom(n_rows, n_inner, n_ch);
    const int64_t n_sl = n_slices_of(g);
    if (n_sl * n_ch > 0x7fffffffLL) return MHAQ_FQ_EINVAL;
    const unsigned grid = (unsigned)(n_sl * n_ch);
    double *slice_ws = ws + g.n_tasks * kNPart;
    const int64_t recs = (g.n_rows / g.n_ch) * g.tasks_per_row;
    const int threads = recs <= 64 ? 64 : (recs <= 128 ? 128 : kFinThreads);
    fq_bwd_finalize_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(ws, slice_ws, tickets, g, n_sl,
                                                                    prm, g_scale, g_zp, g_lo, g_hi);
    return last_error();
}

int mhaq_fq_bwd_finalize_f32(double *ws, unsigned int *tickets, const float *scale, const float *zp,
                             const float *lo, const float *hi, int scale_stride, int zp_stride,
                             int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                             int64_t n_inner, int64_t n_ch, float *g_scale, float *g_zp, float *g_lo,
                             float *g_hi, void *stream) {
    return bwd_finalize_impl(ws, tickets, scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride,
                             param_mode, n_rows, n_inner, n_ch, g_scale, g_zp, g_lo, g_hi, nullptr, stream);
}

int mhaq_fq_bwd_single_launch(int64_t n_rows, int64_t n_inner, int64_t n_ch, int method,
                                 int go_is_code_grad) {
    return flat_shape_ok(n_rows, n_inner, n_ch, method, go_is_code_grad) ? 1 : 0;
}

static int bwd_fused_impl(const float *go, const float *x, float *gx, const float *scale,
                          const float *zp, const float *lo, const float *hi, int scale_stride,
                          int zp_stride, int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                          int64_t n_inner, int64_t n_ch, int method, int go_is_code_grad, const float *r,
                          uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                          const float *aewgs_stats, double *ws, unsigned int *tickets, float *g_scale,
                          float *g_zp, float *g_lo, float *g_hi, const float *const acc[4], void *stream) {
    int rc = check_common(x, scale, zp, n_rows, n_inner, n_ch);
    if (rc) return rc;
    if ((rc = check_mode(param_mode, lo, n_ch)) != 0) return rc;
    if (!go || !ws || !tickets) return MHAQ_FQ_ENULL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const bool aligned = aligned16(x) && aligned16(go) && (!gx || aligned16(gx)) && (!r || aligned16(r));
    // (an UNCLAMPED per-tensor tensor of 2^26 elements or more — never an activation — is the one
    // case the streaming kernel still wins: 466 vs 498 us at 2^28, tools/exp_flat_unclamped2.py)
    const bool flat_wins = has_clamp(param_mode, lo, hi) || n_inner < flat_mbar_min();
    if (aligned && flat_wins && flat_shape_ok(n_rows, n_inner, n_ch, method, go_is_code_grad)) {
        if (!stride_ok(scale_stride) || !stride_ok(zp_stride) || !stride_ok(lo_stride) ||
            !stride_ok(hi_stride))
            return MHAQ_FQ_EINVAL;
        const QParams prm = {scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride, param_mode,
                             acc ? acc[0] : nullptr, acc ? acc[1] : nullptr, acc ? acc[2] : nullptr,
                             acc ? acc[3] : nullptr};
        const FlatGeom f = make_flat_geom(n_inner, flat_cap(), n_inner >= flat_interleave_min());
        const bool clamp = has_clamp(param_mode, lo, hi);
        cudaStream_t st = (cudaStream_t)stream;
        const bool er = (r != nullptr);
        if (method == MHAQ_FQ_STE)
            return clamp ? launch_bwd_flat<MHAQ_FQ_STE, true>(er, f, st, go, x, gx, prm, r, seed, offset, philox_dev,
                                                              ws, tickets, g_scale, g_zp, g_lo, g_hi)
                         : launch_bwd_flat<MHAQ_FQ_STE, false>(er, f, st, go, x, gx, prm, r, seed, offset, philox_dev,
                                                               ws, tickets, g_scale, g_zp, g_lo, g_hi);
        return clamp ? launch_bwd_flat<MHAQ_FQ_LSQ, true>(er, f, st, go, x, gx, prm, r, seed, offset, philox_dev,
                                                          ws, tickets, g_scale, g_zp, g_lo, g_hi)
                     : launch_bwd_flat<MHAQ_FQ_LSQ, false>(er, f, st, go, x, gx, prm, r, seed, offset, philox_dev,
                                                           ws, tickets, g_scale, g_zp, g_lo, g_hi);
    }
    rc = mhaq_fq_bwd_f32(go, x, gx, scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride,
                         param_mode, n_rows, n_inner, n_ch, method, go_is_code_grad, r, seed, offset,
                         philox_dev, aewgs_stats, ws, stream);
    if (rc) return rc;
    return bwd_finalize_impl(ws, tickets, scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride,
                             param_mode, n_rows, n_inner, n_ch, g_scale, g_zp, g_lo, g_hi, acc, stream);
}

int mhaq_fq_bwd_fused_f32(const float *go, const float *x, float *gx, const float *scale,
                          const float *zp, const float *lo, const float *hi, int scale_stride,
                          int zp_stride, int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                          int64_t n_inner, int64_t n_ch, int method, int go_is_code_grad, const float *r,
                          uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                          const float *aewgs_stats, double *ws, unsigned int *tickets, float *g_scale,
                          float *g_zp, float *g_lo, float *g_hi, void *stream) {
    return bwd_fused_impl(go, x, gx, scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride,
                          param_mode, n_rows, n_inner, n_ch, method, go_is_code_grad, r, seed, offset,
                          philox_dev, aewgs_stats, ws, tickets, g_scale, g_zp, g_lo, g_hi, nullptr, stream);
}

int mhaq_fq_bwd_fused_acc_f32(const float *go, const float *x, float *gx, const float *scale,
                              const float *zp, const float *lo, const float *hi, int scale_stride,
                              int zp_stride, int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                              int64_t n_inner, int64_t n_ch, int method, int go_is_code_grad, const float *r,
                              uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                              const float *aewgs_stats, double *ws, unsigned int *tickets, float *g_scale,
                              float *g_zp, float *g_lo, float *g_hi, const float *acc_scale,
                              const float *acc_zp, const float *acc_lo, const float *acc_hi, void *stream) {
    const float *const acc[4] = {acc_scale, acc_zp, acc_lo, acc_hi};
    return bwd_fused_impl(go, x, gx, scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride,
                          param_mode, n_rows, n_inner, n_ch, method, go_is_code_grad, r, seed, offset,
                          philox_dev, aewgs_stats, ws, tickets, g_scale, g_zp, g_lo, g_hi, acc, stream);
}

int mhaq_fq_aewgs_stats_f32(const float *go, const float *x, const float *scale, const float *zp,
                            const float *lo, const float *hi, int scale_stride, int zp_stride,
                            int lo_stride, int hi_stride, int param_mode, int64_t n_rows,
                            int64_t n_inner, int64_t n_ch, int go_is_code_grad, double *ws,
                            void *stream) {
    int rc = check_common(x, scale, zp, n_rows, n_inner, n_ch);
    if (rc) return rc;
    if ((rc = check_mode(param_mode, lo, n_ch)) != 0) return rc;
    if (!go || !ws) return MHAQ_FQ_ENULL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const Geom g = stream_geom(n_rows, n_inner, n_ch);
    const QParams prm = {scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride, param_mode};
    const bool vec = (n_inner % 4 == 0) && aligned16(x) && aligned16(go);
    const int grid = grid_for(g.n_tasks);
    cudaStream_t st = (cudaStream_t)stream;
    if (vec)
        fq_aewgs_stats_kernel<true><<<grid, kThreads, 0, st>>>(go, x, prm, g, go_is_code_grad, ws);
    else
        fq_aewgs_stats_kernel<false><<<grid, kThreads, 0, st>>>(go, x, prm, g, go_is_code_grad, ws);
    return last_error();
}

int mhaq_fq_aewgs_stats_finalize_f32(const double *ws, int64_t n_rows, int64_t n_inner,
                                     int64_t n_ch, float *stats, void *stream) {
    if (!ws || !stats) return MHAQ_FQ_ENULL;
    if (n_rows <= 0 || n_inner <= 0 || n_ch < 1 || (n_rows % n_ch) != 0) return MHAQ_FQ_EINVAL;
    const Geom g = stream_geom(n_rows, n_inner, n_ch);
    fq_aewgs_stats_finalize_kernel<<<(int)n_ch, 256, 0, (cudaStream_t)stream>>>(ws, g, stats);
    return last_error();
}

int mhaq_fq_rowstat_f32(const float *x, int64_t n_rows, int64_t n_inner, float *row_min,
                        float *row_max, float *n_at_min, float *n_at_max, void *stream) {
    if (!x) return MHAQ_FQ_ENULL;
    if (n_rows < 0 || n_inner <= 0) return MHAQ_FQ_EINVAL;
    if (n_rows == 0) return 0;
    const int grid = grid_for(n_rows);
    fq_rowstat_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(x, n_rows, n_inner, row_min,
                                                                  row_max, n_at_min, n_at_max);
    return last_error();
}

int mhaq_fq_rowstat_bwd_f32(const float *gx, const float *x, int64_t n_rows, int64_t n_inner,
                            const float *row_min, const float *n_at_min, const float *g_min,
                            const float *row_max, const float *n_at_max, const float *g_max,
                            float *out, void *stream) {
    if (!x || !out) return MHAQ_FQ_ENULL;
    if ((g_min && (!row_min || !n_at_min)) || (g_max && (!row_max || !n_at_max)))
        return MHAQ_FQ_ENULL;
    if (n_rows < 0 || n_inner <= 0) return MHAQ_FQ_EINVAL;
    if (n_rows == 0) return 0;
    const int grid = grid_for(n_rows);
    fq_rowstat_bwd_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        gx, x, n_rows, n_inner, row_min, n_at_min, g_min, row_max, n_at_max, g_max, out);
    return last_error();
}

int mhaq_fq_wrow_fwd_f32(const float *w, float *wq, const float *log_scale, int64_t n_rows,
                         int64_t n_inner, float *row_min, float *row_max, float *log_range,
                         void *stream) {
    if (!w || !log_scale) return MHAQ_FQ_ENULL;
    if (n_rows < 0 || n_inner <= 0) return MHAQ_FQ_EINVAL;
    if (n_rows == 0) return 0;
    const WRowArgs a = {log_scale, 1, n_rows, n_inner};
    const bool vec = (n_inner % 4 == 0) && aligned16(w) && (!wq || aligned16(wq));
    const int grid = grid_for(n_rows);
    cudaStream_t st = (cudaStream_t)stream;
    if (vec)
        fq_wrow_fwd_kernel<true><<<grid, kThreads, 0, st>>>(w, wq, a, row_min, row_max, log_range);
    else
        fq_wrow_fwd_kernel<false><<<grid, kThreads, 0, st>>>(w, wq, a, row_min, row_max, log_range);
    return last_error();
}

int mhaq_fq_wrow_bwd_f32(const float *g_wq, const float *w, const float *log_scale,
                         const float *row_min, const float *row_max, const float *g_log_range,
                         const float *g_row_min, const float *g_row_max, int64_t n_rows,
                         int64_t n_inner, int method, const float *r, uint64_t seed, uint64_t offset,
                         const uint64_t *philox_dev, float *g_w, float *g_log_scale, void *stream) {
    if (!g_wq || !w || !log_scale || !row_min || !row_max) return MHAQ_FQ_ENULL;
    if (n_rows < 0 || n_inner <= 0) return MHAQ_FQ_EINVAL;
    // AEWGS needs its statistics all-reduced between two passes: streaming kernels only
    if (method != MHAQ_FQ_STE && method != MHAQ_FQ_EWGS && method != MHAQ_FQ_LSQ) return MHAQ_FQ_EINVAL;
    if (n_rows == 0) return 0;
    const WRowArgs a = {log_scale, 1, n_rows, n_inner};
    const bool vec = (n_inner % 4 == 0) && aligned16(w) && aligned16(g_wq) && (!g_w || aligned16(g_w)) &&
                     (!r || aligned16(r));
    const int grid = grid_for(n_rows);
    cudaStream_t st = (cudaStream_t)stream;
#define MHAQ_WROW(M, N)                                                                             \
    launch_wrow_bwd<M, N>(vec, grid, st, g_wq, w, a, row_min, row_max, g_log_range, g_row_min,     \
                          g_row_max, r, seed, offset, philox_dev, g_w, g_log_scale)
    if (method == MHAQ_FQ_LSQ) return MHAQ_WROW(MHAQ_FQ_LSQ, NOISE_NONE);
    if (method == MHAQ_FQ_STE)
        return r ? MHAQ_WROW(MHAQ_FQ_STE, NOISE_EXPLICIT) : MHAQ_WROW(MHAQ_FQ_STE, NOISE_PHILOX);
    return r ? MHAQ_WROW(MHAQ_FQ_EWGS, NOISE_EXPLICIT) : MHAQ_WROW(MHAQ_FQ_EWGS, NOISE_PHILOX);
#undef MHAQ_WROW
}

int mhaq_fq_wrow_multi_fwd_f32(const mhaq_fq_wrow_fwd_desc *descs, int n_tensors, void *stream) {
    if (n_tensors < 0) return MHAQ_FQ_EINVAL;
    if (n_tensors == 0) return 0;
    if (!descs) return MHAQ_FQ_ENULL;
    cudaStream_t st = (cudaStream_t)stream;
    for (int c0 = 0; c0 < n_tensors; c0 += kWRowMultiMax) {
        WRowFwdMulti m;
        m.n = 0;
        m.row0[0] = 0;
        for (int i = c0; i < n_tensors && m.n < kWRowMultiMax; ++i) {
            const mhaq_fq_wrow_fwd_desc &d = descs[i];
            if (!d.w || !d.log_scale) return MHAQ_FQ_ENULL;
            if (d.n_rows < 0 || d.n_inner <= 0 || d.n_rows > 0x3fffffff) return MHAQ_FQ_EINVAL;
            if (d.n_rows == 0) continue;
            const int k = m.n++;
            m.d[k] = {d.w, d.log_scale, d.wq, d.row_min, d.row_max, d.log_range, d.n_inner};
            m.vec[k] = (d.n_inner % 4 == 0) && aligned16(d.w) && (!d.wq || aligned16(d.wq));
            m.row0[k + 1] = m.row0[k] + (int)d.n_rows;
        }
        if (m.n == 0) continue;
        fq_wrow_multi_fwd_kernel<<<grid_for(m.row0[m.n]), kThreads, 0, st>>>(m);
        const int rc = last_error();
        if (rc) return rc;
    }
    return 0;
}

int mhaq_fq_wrow_multi_aewgs_stats_f32(const mhaq_fq_wrow_bwd_desc *descs, int n_tensors, float *stats,
                                       int64_t total_rows, void *stream) {
    if (n_tensors < 0 || total_rows < 0) return MHAQ_FQ_EINVAL;
    if (n_tensors == 0) return 0;
    if (!descs || !stats) return MHAQ_FQ_ENULL;
    bool er = false;
    int rc = wrow_multi_check(descs, n_tensors, &er);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    return wrow_multi_bwd_chunks(descs, n_tensors, [&](const WRowBwdMulti &m, int, int64_t row_base) {
        if (row_base + m.row0[m.n] > total_rows) return (int)MHAQ_FQ_EINVAL;
        fq_wrow_multi_aewgs_stats_kernel<<<grid_for(m.row0[m.n]), kThreads, 0, st>>>(m, stats, row_base, total_rows);
        return last_error();
    });
}

int mhaq_fq_wrow_multi_bwd_f32(const mhaq_fq_wrow_bwd_desc *descs, int n_tensors, int method,
                               uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                               const float *aewgs_stats, int64_t total_rows, void *stream) {
    if (n_tensors < 0) return MHAQ_FQ_EINVAL;
    if (n_tensors == 0) return 0;
    if (!descs) return MHAQ_FQ_ENULL;
    if (method < 0 || method > 3) return MHAQ_FQ_EINVAL;
    if (method == MHAQ_FQ_AEWGS && !aewgs_stats) return MHAQ_FQ_ENULL;
    bool explicit_r = false;
    int rc = wrow_multi_check(descs, n_tensors, &explicit_r);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    return wrow_multi_bwd_chunks(descs, n_tensors, [&](const WRowBwdMulti &m, int c0, int64_t row_base) {
        const int grid = grid_for(m.row0[m.n]);
        const uint64_t off = offset + (uint64_t)c0;
        if (method == MHAQ_FQ_AEWGS && row_base + m.row0[m.n] > total_rows) return (int)MHAQ_FQ_EINVAL;
#define MHAQ_WMULTI(M, N)                                                                        \
    fq_wrow_multi_bwd_kernel<M, N><<<grid, kThreads, 0, st>>>(m, seed, off, philox_dev, aewgs_stats, \
                                                             row_base, total_rows)
        if (method == MHAQ_FQ_LSQ) MHAQ_WMULTI(MHAQ_FQ_LSQ, NOISE_NONE);
        else if (method == MHAQ_FQ_STE) {
            if (explicit_r) MHAQ_WMULTI(MHAQ_FQ_STE, NOISE_EXPLICIT); else MHAQ_WMULTI(MHAQ_FQ_STE, NOISE_PHILOX);
        } else if (method == MHAQ_FQ_EWGS) {
            if (explicit_r) MHAQ_WMULTI(MHAQ_FQ_EWGS, NOISE_EXPLICIT); else MHAQ_WMULTI(MHAQ_FQ_EWGS, NOISE_PHILOX);
        } else {
            if (explicit_r) MHAQ_WMULTI(MHAQ_FQ_AEWGS, NOISE_EXPLICIT); else MHAQ_WMULTI(MHAQ_FQ_AEWGS, NOISE_PHILOX);
        }
#undef MHAQ_WMULTI
        return last_error();
    });
}

int mhaq_fq_potential_loss_fwd_f32(const float *log_act_s, const float *log_act_q, int64_t n_act,
                                   const float *log_wght_s, const float *log_w_range, int64_t n_wght,
                                   const float *base_loss, float *loss_sum, float *cnt, float w_target,
                                   float a_target, float eps, float t, int lossless, int training,
                                   float *out, void *stream) {
    if (!log_act_s || !log_act_q || !log_wght_s || !log_w_range || !base_loss || !loss_sum || !cnt || !out)
        return MHAQ_FQ_ENULL;
    if (n_act < 0 || n_wght < 0) return MHAQ_FQ_EINVAL;
    const PLossArgs a = {log_act_s, log_act_q, log_wght_s, log_w_range, n_act, n_wght,
                         w_target, a_target, eps, t, lossless, training};
    fq_potential_loss_fwd_kernel<<<1, kLossThreads, 0, (cudaStream_t)stream>>>(a, base_loss, loss_sum, cnt, out);
    return last_error();
}

int mhaq_fq_potential_loss_bwd_f32(const float *log_act_s, const float *log_act_q, int64_t n_act,
                                   const float *log_wght_s, const float *log_w_range, int64_t n_wght,
                                   const float *saved, const float *g_loss, float w_target, float a_target,
                                   float eps, float *g_log_act_s, float *g_log_act_q, float *g_log_wght_s,
                                   float *g_log_w_range, float *g_base_loss, void *stream) {
    if (!log_act_s || !log_act_q || !log_wght_s || !log_w_range || !saved || !g_loss) return MHAQ_FQ_ENULL;
    if (n_act < 0 || n_wght < 0) return MHAQ_FQ_EINVAL;
    const PLossArgs a = {log_act_s, log_act_q, log_wght_s, log_w_range, n_act, n_wght,
                         w_target, a_target, eps, 0.f, 0, 0};
    const int64_t n = n_wght > n_act ? n_wght : n_act;
    int grid = (int)((n + kLossThreads - 1) / kLossThreads);
    if (grid < 1) grid = 1;
    if (grid > 1024) grid = 1024;
    fq_potential_loss_bwd_kernel<<<grid, kLossThreads, 0, (cudaStream_t)stream>>>(
        a, saved, g_loss, g_log_act_s, g_log_act_q, g_log_wght_s, g_log_w_range, g_base_loss);
    return last_error();
}

int64_t mhaq_fq_packed_row_bytes(int64_t n_inner, int bits) {
    if (n_inner < 0 || !pack_bits_ok(bits)) return -1;
    return packed_row_bytes(n_inner, bits);
}

int mhaq_fq_pack_f32(const float *x, uint8_t *packed, int bits, const float *scale, const float *zp,
                     const float *lo, const float *hi, int scale_stride, int zp_stride, int lo_stride,
                     int hi_stride, int param_mode, int64_t n_rows, int64_t n_inner, int64_t n_ch,
                     unsigned long long *n_out_of_range, void *stream) {
    int rc = check_common(x, scale, zp, n_rows, n_inner, n_ch);
    if (rc) return rc;
    if (!packed) return MHAQ_FQ_ENULL;
    if (!pack_bits_ok(bits)) return MHAQ_FQ_EINVAL;
    if ((rc = check_mode(param_mode, lo, n_ch)) != 0) return rc;
    if (!stride_ok(scale_stride) || !stride_ok(zp_stride) || !stride_ok(lo_stride) ||
        !stride_ok(hi_stride))
        return MHAQ_FQ_EINVAL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const Geom g = stream_geom(n_rows, n_inner, n_ch);
    const QParams prm = {scale, zp, lo, hi, scale_stride, zp_stride, lo_stride, hi_stride, param_mode};
    const bool vec = (n_inner % 4 == 0) && aligned16(x) && aligned16(packed);
    const bool clamp = has_clamp(param_mode, lo, hi);
    const int64_t rs = packed_row_bytes(n_inner, bits);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(g.n_tasks);
    switch (bits) {
        case 1: launch_pack<1>(vec, clamp, grid, st, x, packed, prm, g, rs, n_out_of_range); break;
        case 2: launch_pack<2>(vec, clamp, grid, st, x, packed, prm, g, rs, n_out_of_range); break;
        case 4: launch_pack<4>(vec, clamp, grid, st, x, packed, prm, g, rs, n_out_of_range); break;
        case 8: launch_pack<8>(vec, clamp, grid, st, x, packed, prm, g, rs, n_out_of_range); break;
        default: launch_pack<16>(vec, clamp, grid, st, x, packed, prm, g, rs, n_out_of_range); break;
    }
    return last_error();
}

int mhaq_fq_unpack_f32(const uint8_t *packed, int bits, float *y, const float *scale, const float *zp,
                       int scale_stride, int zp_stride, int param_mode, int64_t n_rows, int64_t n_inner,
                       int64_t n_ch, void *stream) {
    int rc = check_common(packed, scale, zp, n_rows, n_inner, n_ch);
    if (rc) return rc;
    if (!y) return MHAQ_FQ_ENULL;
    if (!pack_bits_ok(bits) || !mode_ok(param_mode)) return MHAQ_FQ_EINVAL;
    if (param_mode == PARAMS_ACT_LOG && n_ch != 1) return MHAQ_FQ_EINVAL;
    if (!stride_ok(scale_stride) || !stride_ok(zp_stride)) return MHAQ_FQ_EINVAL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const Geom g = stream_geom(n_rows, n_inner, n_ch);
    const QParams prm = {scale, zp, nullptr, nullptr, scale_stride, zp_stride, 0, 0, param_mode};
    const bool vec = (n_inner % 4 == 0) && aligned16(y) && aligned16(packed);
    const int64_t rs = packed_row_bytes(n_inner, bits);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(g.n_tasks);
    switch (bits) {
        case 1: launch_unpack<1>(vec, grid, st, packed, y, prm, g, rs); break;
        case 2: launch_unpack<2>(vec, grid, st, packed, y, prm, g, rs); break;
        case 4: launch_unpack<4>(vec, grid, st, packed, y, prm, g, rs); break;
        case 8: launch_unpack<8>(vec, grid, st, packed, y, prm, g, rs); break;
        default: launch_unpack<16>(vec, grid, st, packed, y, prm, g, rs); break;
    }
    return last_error();
}

int mhaq_fq_noise_f32(float *r, int64_t n_rows, int64_t n_inner, uint64_t seed, uint64_t offset,
                      const uint64_t *philox_dev, void *stream) {
    if (!r) return MHAQ_FQ_ENULL;
    if (n_rows < 0 || n_inner < 0) return MHAQ_FQ_EINVAL;
    if (n_rows == 0 || n_inner == 0) return 0;
    const Geom g = stream_geom(n_rows, n_inner, 1);
    fq_noise_kernel<<<grid_for(g.n_tasks), kThreads, 0, (cudaStream_t)stream>>>(r, g, seed, offset,
                                                                               philox_dev);
    return last_error();
}

int64_t mhaq_fq_iconv_weight_bytes(int64_t n_out, int64_t k_bytes, int *n_tiles, int *tile_n, int *tile_out,
                                   int64_t *k_stages) {
    if (n_out < 1 || k_bytes < 16 || k_bytes % 16 != 0) return -1;
    const IcLayout l = iconv_layout(n_out, k_bytes);
    if (n_tiles) *n_tiles = l.n_tiles;
    if (tile_n) *tile_n = l.tile_n;
    if (tile_out) *tile_out = l.tile_out;
    if (k_stages) *k_stages = l.k_stages;
    return (int64_t)l.n_tiles * l.k_stages * l.tile_n * kIcStageK;
}

int mhaq_fq_act_codes_f32(const float *x, uint8_t *codes, const float *scale, const float *zero_point,
                          const float *max_val, int64_t n_pixels, int64_t n_channels, int64_t cp,
                          unsigned long long *n_out_of_range, void *stream) {
    if (!x || !codes || !scale || !zero_point || !max_val) return MHAQ_FQ_ENULL;
    if (n_pixels < 0 || n_channels < 1 || cp < n_channels || cp % 16 != 0 || !aligned16(codes))
        return MHAQ_FQ_EINVAL;
    if (n_pixels == 0) return 0;
    const QParams prm = {scale, zero_point, zero_point, max_val, 0, 0, 0, 0, PARAMS_LINEAR};
    const bool vec = n_channels % 4 == 0 && aligned16(x);
    const int64_t groups = n_pixels * (cp / 4);
    const int64_t blocks = (groups + kThreads - 1) / kThreads;
    const int grid = (int)(blocks < 148 * 64 ? blocks : 148 * 64);
    fq_act_codes_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(x, codes, prm, n_pixels, n_channels, cp, vec,
                                                                      n_out_of_range);
    return last_error();
}

int mhaq_fq_iconv_u8(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                     const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                     float *y, int64_t batch, int64_t height, int64_t width, int64_t cp, int64_t n_out,
                     int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                     int act_max_code, int weight_max_code, void *stream) {
    if (!y) return MHAQ_FQ_ENULL;
    IConvArgs a;
    dim3 grid;
    int rc = iconv_args(codes, weights, alpha, beta, ctab, h_class, w_class, n_w_classes, batch, height, width, cp,
                        n_out, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, act_max_code, weight_max_code,
                        a, grid);
    if (rc) return rc;
    rc = iconv_smem_opt_in<false>();
    if (rc) return rc;
    a.y = y;
    a.vec_out = aligned16(y) && n_out % 4 == 0;
    fq_iconv_kernel<false><<<grid, kIcThreads, iconv_smem_bytes(a.tile_n), (cudaStream_t)stream>>>(a);
    return last_error();
}

int mhaq_fq_iconv_fused_u8(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                           const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                           int64_t batch, int64_t height, int64_t width, int64_t cp, int64_t n_out,
                           int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                           int act_max_code, int weight_max_code, const mhaq_fq_iconv_epilogue *epilogue,
                           void *stream) {
    int rc = iconv_epilogue_check(epilogue);
    if (rc) return rc;
    IConvArgs a;
    dim3 grid;
    rc = iconv_args(codes, weights, alpha, beta, ctab, h_class, w_class, n_w_classes, batch, height, width, cp,
                    n_out, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, act_max_code, weight_max_code,
                    a, grid);
    if (rc) return rc;
    rc = iconv_smem_opt_in<true>();
    if (rc) return rc;
    iconv_epilogue_set(*epilogue, a);
    fq_iconv_kernel<true><<<grid, kIcThreads, iconv_smem_bytes(a.tile_n), (cudaStream_t)stream>>>(a);
    return last_error();
}

int64_t mhaq_fq_iconv_grouped_weight_bytes(int64_t n_in, int64_t n_out, const mhaq_fq_iconv_geometry *geometry,
                                           int *n_tiles, int *tile_n, int *tile_out, int *groups_per_tile,
                                           int *tiles_per_group, int64_t *k_stages) {
    if (!geometry || !igroup_geometry_ok(n_in, n_out, *geometry)) return -1;
    const mhaq_fq_iconv_geometry &g = *geometry;
    const int64_t cp = (n_in + 15) / 16 * 16;
    IgPlan l{};
    int64_t bytes = (int64_t)g.kernel_h * g.kernel_w * cp;
    if (!igroup_depthwise(n_in, n_out, g.groups)) {
        l = igroup_plan(n_out, g.groups, n_in / g.groups, g.kernel_h, g.kernel_w);
        bytes = (int64_t)l.n_tiles * l.k_stages * l.tile_n * kIcStageK;
    }
    if (n_tiles) *n_tiles = l.n_tiles;
    if (tile_n) *tile_n = l.tile_n;
    if (tile_out) *tile_out = l.tile_out;
    if (groups_per_tile) *groups_per_tile = l.gpt;
    if (tiles_per_group) *tiles_per_group = l.parts;
    if (k_stages) *k_stages = l.k_stages;
    return bytes;
}

int mhaq_fq_iconv_grouped_u8(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                             const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                             int64_t batch, int64_t height, int64_t width, int64_t n_in, int64_t n_out,
                             const mhaq_fq_iconv_geometry *geometry, int act_max_code, int weight_max_code,
                             const mhaq_fq_iconv_epilogue *epilogue, void *stream) {
    IConvArgs a;
    IgPlan l;
    int rc = igroup_args(codes, weights, alpha, beta, ctab, h_class, w_class, n_w_classes, batch, height, width,
                         n_in, n_out, geometry, act_max_code, weight_max_code, epilogue, a, l);
    if (rc) return rc;
    if (igroup_depthwise(n_in, n_out, geometry->groups)) {
        const int64_t blocks = (a.m * (a.cp / 16) + kDwThreads - 1) / kDwThreads;
        const int grid = (int)(blocks < 148 * 64 ? blocks : 148 * 64);
        fq_idw_kernel<<<grid, kDwThreads, 0, (cudaStream_t)stream>>>(a);
        return last_error();
    }
    rc = iconv_smem_opt_in<true, true>();
    if (rc) return rc;
    const dim3 grid((unsigned)((a.m + kIcTileM - 1) / kIcTileM), (unsigned)l.n_tiles);
    fq_iconv_kernel<true, true><<<grid, kIcThreads, iconv_smem_bytes(a.tile_n), (cudaStream_t)stream>>>(a);
    return last_error();
}

}  // extern "C"
