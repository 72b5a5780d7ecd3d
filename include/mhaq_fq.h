/*
 * mhaq_fq.h — C ABI of the B200 (sm_100a) fake-quantization hot path.
 *
 * This is the drop-in boundary for MHAQ's QAT quantizer ops.  Every entry
 * point replaces a piece of the reference's PyTorch implementation (paths are
 * relative to the reference checkout):
 *
 *   mhaq_fq_fwd_f32            Quantizer.quantize + Quantizer.dequantize
 *                              src/quantization/gdnsq/gdnsq.py:189-229
 *                              (+ QNoise.forward, gdnsq.py:13-16)
 *   mhaq_fq_bwd_f32            autograd of the above: QNSTE/QNLSQ/QNEWGS/QNAEWGS
 *                              .backward (gdnsq.py:35-57, 63-84, 90-107, 113-147)
 *                              fused with torch's clamp/sub/div/mul/add backward
 *   mhaq_fq_bwd_finalize_f32   the broadcast "sum_to_size" reductions autograd
 *                              performs for scale / zero_point / min_val / max_val
 *   mhaq_fq_bwd_fused_f32      the two calls above as ONE entry point (and, for per-tensor
 *                              tensors, ONE kernel: the reduction is finished in-kernel)
 *   mhaq_fq_aewgs_stats_f32    reduce_to_shape(num/e2/me) of QNAEWGS.backward
 *   + _finalize                gdnsq.py:118-124, 150-152 (the caller all-reduces
 *                              the packed [3*n_ch] buffer once, gdnsq.py:126-129)
 *   mhaq_fq_rowstat_f32        weight.amin((1,2,3)) / amax of NoisyConv2d.forward
 *                              (layers/gdnsq_conv2d.py:80-84) and
 *                              ModelHelper.get_model_values (utils/model_helper.py:24-25)
 *   mhaq_fq_wrow_fwd_f32 /     the whole per-channel weight path of NoisyConv2d / NoisyLinear.forward
 *   mhaq_fq_wrow_bwd_f32       (gdnsq_conv2d.py:72-98) plus ModelHelper's log2(max-min+2^log_s)
 *                              (utils/model_helper.py:24-25,44) and their autograd, one launch each
 *   mhaq_fq_minmax_finalize    q.aminmax() of NoisyAct.forward (layers/gdnsq_act.py:51-54),
 *                              the eval-mode asserts (gdnsq.py:211-217) and the input min / max
 *                              MinMaxObserver takes during calibration
 *                              (calib/minmaxobserver.py:28-37) — all from the forward's own pass
 *   mhaq_fq_noise_f32          torch.randint_like(input, 2).sub_(0.5)  (gdnsq.py:54)
 *   mhaq_fq_pack_f32           the forward's integer codes stored at their real width (1, 2, 4, 8
 *                              or 16 bits, "Packed codes" below): the low-bit artifact of QAT
 *   mhaq_fq_unpack_f32         its inverse, code * s + zero_point, in every parameter mode
 *   mhaq_fq_packed_row_bytes   the row stride of the packed format
 *   mhaq_fq_act_codes_f32      the activation codes of an eval-mode NoisyAct as uint8, channels padded
 *                              to 16: the input of the integer layers ("Integer layers" below)
 *   mhaq_fq_iconv_u8           a quantized convolution / linear layer on integer codes: int8
 *                              tensor-core implicit GEMM (tcgen05.mma kind::i8), fp32 output
 *   mhaq_fq_iconv_weight_bytes the size and tiling of the weight operand mhaq_fq_iconv_u8 reads
 *   mhaq_fq_iconv_fused_u8     mhaq_fq_iconv_u8 with an eval BatchNorm folded into its operands and
 *                              the residual add, ReLU / LeakyReLU and the next layer's codes in its
 *                              epilogue
 *   mhaq_fq_iconv_grouped_u8   a grouped, depthwise or dilated integer convolution with the fused
 *                              epilogue: depthwise on the CUDA cores, the rest on the tensor cores
 *   mhaq_fq_iconv_grouped_weight_bytes  the size and tiling of its weight operand
 *   mhaq_fq_potential_loss_*   PotentialLoss.forward's constraint arithmetic and its autograd
 *                              (gdnsq_loss.py:32-86, 114-168), one launch each way
 *
 * Conventions
 *   - fp32 only, CUDA only, contiguous tensors only.  No CPU fallback exists.
 *   - All pointers are DEVICE pointers unless stated otherwise.  The caller
 *     owns every buffer, including workspaces; nothing here allocates.
 *   - A tensor is viewed as [n_rows][n_inner]; row r belongs to quantization
 *     channel (r % n_ch).  Per-tensor: n_rows=1, n_ch=1.  Conv weight
 *     (O,I,kh,kw) per-channel: n_rows=O, n_inner=I*kh*kw, n_ch=O.
 *   - Each of scale / zp / lo / hi is an array indexed [ch * stride] with
 *     stride 0 (one broadcast value) or 1 (one value per channel).  lo / hi may
 *     be NULL meaning -inf / +inf (the weight quantizer).
 *   - Every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 *     stateless and re-entrant.  Return value: 0 on success, otherwise the
 *     cudaError_t of the failed launch / a negative MHAQ_FQ_E* argument error.
 *     No exceptions cross this boundary.
 */
#ifndef MHAQ_FQ_H_
#define MHAQ_FQ_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MHAQ_FQ_ABI_VERSION 7

/* gradient estimators — numeric values follow the reference enum
 * QNMethod (src/quantization/gdnsq/gdnsq_utils.py:9-13). */
#define MHAQ_FQ_STE 0
#define MHAQ_FQ_EWGS 1
#define MHAQ_FQ_AEWGS 2
#define MHAQ_FQ_LSQ 3

/* How the parameter pointers are interpreted (`param_mode`).
 *   LINEAR     scale, zp, lo, hi as described under Conventions.
 *   ACT_LOG    the NoisyAct parameters (layers/gdnsq_act.py:42-48), one float each:
 *              scale -> log_act_s, zp -> act_b, lo -> log_act_q, hi unused (n_ch must be 1);
 *              the kernels form s = exp2(log_act_s), q = exp2(log_act_q), zero_point =
 *              min_val = act_b, max_val = (act_b + q) - s themselves, and the finalize returns
 *              g_scale = d/d log_act_s, g_zp = d/d act_b, g_lo = d/d log_act_q (g_hi unused).
 *   WEIGHT_LOG scale -> log_wght_s[ch] (layers/gdnsq_conv2d.py:72), zp -> zero point per
 *              channel, lo = hi = NULL; the finalize returns g_scale = d/d log_wght_s,
 *              g_zp = d/d zero_point.
 * The log modes remove the ~25 tiny elementwise launches autograd otherwise runs per quantizer
 * for exp2 / add / sub and their backward.
 *   UNIT       the value is already scaled — the reference's two-step form
 *              `v + QN*.apply(v, s)` (gdnsq.py:204-208, `scaled_noise`): s = 1, zero_point = 0, no
 *              clamp; `scale` (and `zp`, any non-NULL pointer) only fix the channel layout.  The
 *              finalize returns g_scale = the estimator's own scale gradient (QN*.backward's
 *              grad_scale: the GDNSQ noise term, gdnsq.py:54-55, or LSQ's, :81-82) and nothing else. */
#define MHAQ_FQ_PARAMS_LINEAR 0
#define MHAQ_FQ_PARAMS_ACT_LOG 1
#define MHAQ_FQ_PARAMS_WEIGHT_LOG 2
#define MHAQ_FQ_PARAMS_UNIT 3

/* argument errors */
#define MHAQ_FQ_EINVAL (-1)
#define MHAQ_FQ_ENULL (-2)

/* doubles per record in the backward / stats workspace */
#define MHAQ_FQ_NPART 8

int mhaq_fq_abi_version(void);
const char *mhaq_fq_build_info(void);

/* Workspaces (caller-owned device memory) for a [n_rows][n_inner] tensor:
 *   ws      : mhaq_fq_workspace_bytes() bytes of scratch, contents irrelevant.
 *   tickets : mhaq_fq_ticket_count() unsigned ints, 16-byte aligned, used by the deterministic
 *             reductions: one ticket per channel for the finalize, followed by the region in
 *             which the single-launch per-tensor backward hands its per-block records to the
 *             summing block (every 64-bit word doubles as its own "ready" flag: zero = not
 *             written).  The buffer MUST be zero on entry; every launch leaves it zero
 *             again, so one zero-initialised buffer can be reused forever by calls that are
 *             ordered on one stream (allocate one per stream).
 * mhaq_fq_num_tasks: number of records the streaming kernels write (informational). */
int64_t mhaq_fq_num_tasks(int64_t n_rows, int64_t n_inner);
int64_t mhaq_fq_workspace_bytes(int64_t n_rows, int64_t n_inner);
int64_t mhaq_fq_ticket_count(int64_t n_rows, int64_t n_inner, int64_t n_ch);
/* Id of the CUDA-graph capture `stream` is currently recording into, 0 when it is not capturing
 * (cudaStreamGetCaptureInfo).  A host layer that keeps one ticket buffer per stream uses it to
 * give every capture its own buffer: a graph may later be replayed on any stream, concurrently
 * with eager launches on the stream it was captured from. */
unsigned long long mhaq_fq_stream_capture_id(void *stream);

/* Forward: y = rint((clamp(x,lo,hi) - zp) / s) * s + zp, each step one IEEE
 * fp32 rounding (no FMA contraction, true division, round-half-even).
 *   y      : fake-quantized output, or NULL
 *   codes  : integer-valued fp32 codes rint(v), or NULL
 *   minmax_ws : NULL, or a workspace (mhaq_fq_workspace_bytes) that receives one 16-byte
 *            {min code, max code, min input, max input} record per task for
 *            mhaq_fq_minmax_finalize (eval mode / calibration; NaN-propagating like
 *            torch.aminmax).  The statistics ride the same packed fast path as the plain forward. */
int mhaq_fq_fwd_f32(const float *x, float *y, float *codes,
                    const float *scale, const float *zp, const float *lo, const float *hi,
                    int scale_stride, int zp_stride, int lo_stride, int hi_stride, int param_mode,
                    int64_t n_rows, int64_t n_inner, int64_t n_ch,
                    double *minmax_ws, void *stream);

/* out5[0]=min code, out5[1]=max code, out5[2]= 0 if every code is finite else 1 (the eval
 * asserts of gdnsq.py:211-217 can only fail on non-finite codes), out5[3]=min input,
 * out5[4]=max input, over the whole tensor. */
int mhaq_fq_minmax_finalize(const double *minmax_ws, int64_t n_rows, int64_t n_inner,
                            float *out5, void *stream);

/* Backward of the fake-quant op: input gradient plus one fp64 record of partial
 * parameter-gradient sums per task (fp32 per thread -> warp shuffle -> fp64 per CTA).
 *   go      : gradient w.r.t. y (go_is_code_grad=0) or w.r.t. the codes
 *             returned by quantize() (go_is_code_grad=1)
 *   x       : the forward input (the only tensor saved for backward)
 *   gx      : gradient w.r.t. x, or NULL
 *   method  : MHAQ_FQ_STE / EWGS / AEWGS / LSQ
 *   r       : explicit noise tensor in {-0.5,+0.5} (parity runs), or NULL to
 *             draw it in-kernel from Philox4x32-10 keyed by (seed, offset);
 *             if philox_dev != NULL the kernel reads seed=philox_dev[0] and
 *             adds philox_dev[1] to offset (CUDA-graph friendly).
 *   aewgs_stats : [3*n_ch] per-channel means {num, e2, me} (AEWGS only)
 *   ws      : workspace, consumed by mhaq_fq_bwd_finalize_f32. */
int mhaq_fq_bwd_f32(const float *go, const float *x, float *gx,
                    const float *scale, const float *zp, const float *lo, const float *hi,
                    int scale_stride, int zp_stride, int lo_stride, int hi_stride, int param_mode,
                    int64_t n_rows, int64_t n_inner, int64_t n_ch,
                    int method, int go_is_code_grad,
                    const float *r, uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                    const float *aewgs_stats, double *ws, void *stream);

/* Deterministic second stage, one launch whatever the record count: per-channel sums in
 * a fixed order in fp64 (slices of 256 records in parallel, then a ticketed last-CTA sum
 * of the slice sums in index order; no floating-point atomics, bitwise reproducible).
 * Each output is [n_ch] floats (or NULL to skip):
 *   g_scale = d/d scale,  g_zp = d/d zero_point,  g_lo = d/d min_val,  g_hi = d/d max_val. */
int mhaq_fq_bwd_finalize_f32(double *ws, unsigned int *tickets,
                             const float *scale, const float *zp, const float *lo, const float *hi,
                             int scale_stride, int zp_stride, int lo_stride, int hi_stride,
                             int param_mode,     /* parameters only read in the log modes */
                             int64_t n_rows, int64_t n_inner, int64_t n_ch,
                             float *g_scale, float *g_zp, float *g_lo, float *g_hi,
                             void *stream);

/* mhaq_fq_bwd_f32 + mhaq_fq_bwd_finalize_f32 as one entry point (same arguments, the union of
 * the two lists).  For a per-tensor tensor (n_rows = n_ch = 1: every activation) with the
 * STE / LSQ estimator and the gradient w.r.t. y it is ONE kernel: a
 * persistent, balanced grid (<= SMs x 4 blocks; operands staged through a TMA bulk-copy ring;
 * each block one contiguous range, or — from 2^24 elements — every grid-th 8 Ki-element chunk)
 * whose block 0 sums the per-block fp64 records in index order (handed over through
 * self-validating words in `tickets`: no fence, no atomic) and writes the gradients — no second
 * launch, no per-task flushes; bitwise reproducible on a given device.
 * Everything else runs the two launches above (also an unclamped per-tensor tensor of 2^26 elements
 * or more).  mhaq_fq_bwd_single_launch() tells which (for 16-byte aligned, clamped operands). */
int mhaq_fq_bwd_fused_f32(const float *go, const float *x, float *gx,
                          const float *scale, const float *zp, const float *lo, const float *hi,
                          int scale_stride, int zp_stride, int lo_stride, int hi_stride, int param_mode,
                          int64_t n_rows, int64_t n_inner, int64_t n_ch,
                          int method, int go_is_code_grad,
                          const float *r, uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                          const float *aewgs_stats, double *ws, unsigned int *tickets,
                          float *g_scale, float *g_zp, float *g_lo, float *g_hi, void *stream);
int mhaq_fq_bwd_single_launch(int64_t n_rows, int64_t n_inner, int64_t n_ch, int method,
                              int go_is_code_grad);
/* mhaq_fq_bwd_fused_f32 that also ADDS acc_scale / acc_zp / acc_lo / acc_hi (one value per channel,
 * each may be NULL) to the gradient it writes for the corresponding parameter (in the log-domain
 * modes: to the gradient of log_act_s / act_b / log_act_q, resp. log_wght_s / zero_point).  They are
 * the gradients the same parameters receive along other paths of the caller's graph (PotentialLoss
 * reads log_act_s and log_act_q, gdnsq_loss.py:114-168): with them folded in here autograd sees ONE
 * gradient per parameter and the accumulation kernels it would otherwise launch (2 per activation
 * quantizer per step) disappear.  The sum is the fp32 sum autograd would have formed. */
int mhaq_fq_bwd_fused_acc_f32(const float *go, const float *x, float *gx,
                              const float *scale, const float *zp, const float *lo, const float *hi,
                              int scale_stride, int zp_stride, int lo_stride, int hi_stride, int param_mode,
                              int64_t n_rows, int64_t n_inner, int64_t n_ch,
                              int method, int go_is_code_grad,
                              const float *r, uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                              const float *aewgs_stats, double *ws, unsigned int *tickets,
                              float *g_scale, float *g_zp, float *g_lo, float *g_hi,
                              const float *acc_scale, const float *acc_zp, const float *acc_lo,
                              const float *acc_hi, void *stream);

/* AEWGS statistics: per-channel sums of sign(g)*e, e*e, e  (e = rint(v)-v). */
int mhaq_fq_aewgs_stats_f32(const float *go, const float *x,
                            const float *scale, const float *zp, const float *lo, const float *hi,
                            int scale_stride, int zp_stride, int lo_stride, int hi_stride,
                            int param_mode, int64_t n_rows, int64_t n_inner, int64_t n_ch,
                            int go_is_code_grad, double *ws, void *stream);

/* stats[0*n_ch+c]=mean num, stats[1*n_ch+c]=mean e2, stats[2*n_ch+c]=mean e. */
int mhaq_fq_aewgs_stats_finalize_f32(const double *ws, int64_t n_rows, int64_t n_inner,
                                     int64_t n_ch, float *stats, void *stream);

/* Per-row min / max / number of elements equal to the row min / to the row max
 * (what amin/amax backward needs for its even split among ties).
 * Any output may be NULL.  One pass over x. */
int mhaq_fq_rowstat_f32(const float *x, int64_t n_rows, int64_t n_inner,
                        float *row_min, float *row_max, float *n_at_min, float *n_at_max,
                        void *stream);

/* out[i] = gx[i] + (x[i]==row_min ? g_min[row]/n_at_min[row] : 0)
 *                + (x[i]==row_max ? g_max[row]/n_at_max[row] : 0)
 * — amin / amax backward fused into one pass (g_min / g_max may be NULL). */
int mhaq_fq_rowstat_bwd_f32(const float *gx, const float *x, int64_t n_rows, int64_t n_inner,
                            const float *row_min, const float *n_at_min, const float *g_min,
                            const float *row_max, const float *n_at_max, const float *g_max,
                            float *out, void *stream);

/* Row-resident fused WEIGHT quantizer (per-channel, channel = row, short rows: conv / linear
 * weights).  One CTA per row, one launch:
 *   row_min / row_max  = weight.amin / amax over the row  (gdnsq_conv2d.py:80-81,
 *                        utils/model_helper.py:24-25)
 *   wq        = fake_quant(w; s = exp2(log_scale[row]), zero_point = row_min)   (gdnsq_conv2d.py:72-98)
 *   log_range = log2((row_max - row_min) + s)     (ModelHelper.get_model_values, model_helper.py:44)
 * Any of wq / row_min / row_max / log_range may be NULL. */
int mhaq_fq_wrow_fwd_f32(const float *w, float *wq, const float *log_scale,
                         int64_t n_rows, int64_t n_inner,
                         float *row_min, float *row_max, float *log_range, void *stream);

/* Backward of mhaq_fq_wrow_fwd_f32 in one launch (methods STE / EWGS / LSQ; AEWGS needs an
 * all-reduce between its two passes and stays on the streaming kernels):
 *   g_w         = d/d w: the quantizer's input gradient plus the amin / amax backward (even split
 *                 among ties) of everything that flowed into row_min / row_max — the zero-point
 *                 gradient, g_row_min / g_row_max (NULL = none) and log_range's own dependence
 *   g_log_scale = d/d log_scale[row], through the quantizer and through log_range
 *   g_log_range : gradient w.r.t. the log_range output, or NULL
 *   r / seed / offset / philox_dev : as mhaq_fq_bwd_f32 (same noise stream for the same shape). */
int mhaq_fq_wrow_bwd_f32(const float *g_wq, const float *w, const float *log_scale,
                         const float *row_min, const float *row_max,
                         const float *g_log_range, const float *g_row_min, const float *g_row_max,
                         int64_t n_rows, int64_t n_inner, int method,
                         const float *r, uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                         float *g_w, float *g_log_scale, void *stream);

/* Multi-tensor forms of the two entry points above: EVERY per-channel weight tensor of a model in
 * one launch each way (SURVEY.md §8 row (f)-4: CIFAR-sized models are bound by launch count, not
 * by any kernel).  `descs` is a HOST array; the descriptors travel in the kernel's parameter
 * space (the library splits more than 32 / 24 tensors over several launches).  Fields have the
 * meaning of the same-named arguments of mhaq_fq_wrow_fwd_f32 / mhaq_fq_wrow_bwd_f32; tensor i of
 * the backward draws its in-kernel noise from Philox stream (seed, offset + i) — what a
 * per-tensor call with that offset would read; `r` must be NULL for all tensors or for none. */
typedef struct {
    const float *w, *log_scale;
    float *wq, *row_min, *row_max, *log_range;      /* any may be NULL */
    int64_t n_rows, n_inner;
} mhaq_fq_wrow_fwd_desc;
typedef struct {
    const float *g_wq, *w, *log_scale, *row_min, *row_max;
    const float *g_log_range, *g_row_min, *g_row_max, *r;   /* any may be NULL */
    float *g_w, *g_log_scale;                               /* either may be NULL */
    int64_t n_rows, n_inner;
    /* optional (NULL = none): the gradient log_scale[row] receives along OTHER paths of the caller's
     * graph (PotentialLoss reads log_wght_s directly); added to g_log_scale in the kernel so that
     * autograd sees one gradient per parameter and launches no accumulation kernel */
    const float *g_log_scale_acc;
} mhaq_fq_wrow_bwd_desc;
int mhaq_fq_wrow_multi_fwd_f32(const mhaq_fq_wrow_fwd_desc *descs, int n_tensors, void *stream);
/* AEWGS (the one estimator with an exchange step) in the multi-tensor form: first
 * mhaq_fq_wrow_multi_aewgs_stats_f32 writes the per-row means of sign(g)*e, e*e, e of EVERY tensor
 * into one packed buffer stats[3][total_rows] (rows of tensor 0, then tensor 1, ...); the caller
 * all-reduces (AVG) that buffer ONCE for the whole model — the reference issues three all-reduces per
 * weight tensor, gdnsq.py:126-129 — and passes it to mhaq_fq_wrow_multi_bwd_f32(method = AEWGS).
 * For the other methods aewgs_stats is NULL and total_rows ignored. */
int mhaq_fq_wrow_multi_aewgs_stats_f32(const mhaq_fq_wrow_bwd_desc *descs, int n_tensors,
                                       float *stats, int64_t total_rows, void *stream);
int mhaq_fq_wrow_multi_bwd_f32(const mhaq_fq_wrow_bwd_desc *descs, int n_tensors, int method,
                               uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                               const float *aewgs_stats, int64_t total_rows, void *stream);

/* PotentialLoss's bit-width constraint (gdnsq_loss.py:32-86 / 114-168, exponent p = 1 as
 * GDNSQQuant passes it, gdnsq_quant.py:90-102) in ONE launch:
 *   ploss = (loss_sum/cnt) * l1 * (wmul * wloss + amul * aloss) + l2 * base_loss,
 *   wloss = mean(max(0, (log_w_range - log_wght_s) - (w_target - eps))),  aloss likewise with
 *   (log_act_q - log_act_s, a_target); wmul / amul from the numbers of active constraints;
 *   (l1, l2) = lossless ? (1, t) : (t, 1); when `training`, loss_sum += base_loss and cnt += 1
 *   (device scalars, updated in place — CUDA-graph friendly).
 * out: MHAQ_FQ_PLOSS_NOUT floats = {ploss, wloss, aloss, rloss, -mean(log_wght_s),
 *   mean(log_w_range), -mean(log_act_s), mean(log_act_q), max(log_w_range - log_wght_s), wact, aact,
 *   cw, ca, l2}; the last three are what the backward needs (pass `out` back as `saved`). */
#define MHAQ_FQ_PLOSS_NOUT 14
int mhaq_fq_potential_loss_fwd_f32(const float *log_act_s, const float *log_act_q, int64_t n_act,
                                   const float *log_wght_s, const float *log_w_range, int64_t n_wght,
                                   const float *base_loss, float *loss_sum, float *cnt,
                                   float w_target, float a_target, float eps, float t,
                                   int lossless, int training, float *out, void *stream);
/* Gradients of ploss (times g_loss[0]) w.r.t. the four vectors and the base loss; any output may
 * be NULL.  torch.max(0, x) semantics: full gradient where x > 0, half on a tie. */
int mhaq_fq_potential_loss_bwd_f32(const float *log_act_s, const float *log_act_q, int64_t n_act,
                                   const float *log_wght_s, const float *log_w_range, int64_t n_wght,
                                   const float *saved, const float *g_loss,
                                   float w_target, float a_target, float eps,
                                   float *g_log_act_s, float *g_log_act_q, float *g_log_wght_s,
                                   float *g_log_w_range, float *g_base_loss, void *stream);

/* Materialise the in-kernel noise stream: r[i] in {-0.5,+0.5}, identical to what
 * mhaq_fq_bwd_f32 draws for the same (seed, offset, philox_dev, shape). */
int mhaq_fq_noise_f32(float *r, int64_t n_rows, int64_t n_inner,
                      uint64_t seed, uint64_t offset, const uint64_t *philox_dev,
                      void *stream);

/* Packed codes.
 *   Width b in {1, 2, 4, 8, 16}.  A learned width of 3, 5, 6 or 7 is stored in the next supported
 *   width (the true width is the caller's to record).
 *   The tensor is the usual [n_rows][n_inner] storage-order view, row r quantized with channel
 *   r % n_ch; the stored value is the code rint(v) the forward computes (the same device
 *   functions, so it is identical to mhaq_fq_fwd_f32's `codes` by construction).
 *   Row r starts at byte r * row_stride, row_stride = round_up(ceil(n_inner * b / 8), 16), so every
 *   row is 16-byte aligned (relative to the buffer).  For b <= 8, code j of a row occupies bits
 *   [(j*b) mod 8, +b) of byte floor(j*b / 8), least-significant bit first; for b = 16 it is a
 *   little-endian uint16 at byte 2j.  Padding bits and bytes are 0.
 *   A code outside [0, 2^b - 1] (a NaN code included) is stored saturated (NaN as 0) and counted.
 *   Only the generic operator can produce one: weight codes are >= 0 because the zero point is
 *   the row minimum, and clamped activation codes are >= 0 as well.
 *   Dequantization is y = code * s, then + zero_point: two roundings, as in the forward.  For every
 *   in-range element y equals the forward's output bit for bit.  (A zero code is always +0 in the
 *   forward too: v + (rint(v) - v) rounds to +0 for every v in (-0.5, 0], so a zero point of -0.0
 *   gives +0 on both sides.)
 *
 * mhaq_fq_packed_row_bytes: row_stride for (n_inner, b), or -1 for a bad width / n_inner < 0. */
int64_t mhaq_fq_packed_row_bytes(int64_t n_inner, int bits);

/* Pack x's codes into `packed` (n_rows * mhaq_fq_packed_row_bytes(n_inner, bits) bytes, every byte
 * written).  Parameters, strides, param_mode and the geometry are those of mhaq_fq_fwd_f32.
 * n_out_of_range: NULL, or one device counter to which the number of saturated codes is ADDED
 * (one integer atomic per CTA that saw any; the caller zeroes it).  No host synchronisation and
 * no allocation: safe under CUDA-graph capture. */
int mhaq_fq_pack_f32(const float *x, uint8_t *packed, int bits,
                     const float *scale, const float *zp, const float *lo, const float *hi,
                     int scale_stride, int zp_stride, int lo_stride, int hi_stride, int param_mode,
                     int64_t n_rows, int64_t n_inner, int64_t n_ch,
                     unsigned long long *n_out_of_range, void *stream);

/* y = code * s + zp from packed codes, with s and zp as the forward forms them in `param_mode`
 * (ACT_LOG: scale -> log_act_s, zp -> act_b; WEIGHT_LOG: scale -> log_wght_s[ch]; UNIT: y = code).
 * Capture-safe like mhaq_fq_pack_f32. */
int mhaq_fq_unpack_f32(const uint8_t *packed, int bits, float *y,
                       const float *scale, const float *zp,
                       int scale_stride, int zp_stride, int param_mode,
                       int64_t n_rows, int64_t n_inner, int64_t n_ch, void *stream);

/* Integer layers.
 *   A quantized layer y = conv(a, w) + bias (a Linear is the case H = W = kh = kw = 1) with
 *   a = ca * sa + zpa (activation code ca in [0, act_max_code]) and w_nk = cw_nk * sw_n + zpw_n
 *   (weight code cw in [0, weight_max_code]) is evaluated as
 *     y[m][n] = alpha[n] * S[m][n] + beta[n] * SA[m] + ctab[p(m)][n]
 *   with S = sum over the valid taps k of ca_k * cw_nk and SA = sum of ca_k (both int32, exact),
 *   alpha = sa * sw, beta = sa * zpw and ctab[p][n] = zpa * (sw_n * sum_{k in p} cw_nk + zpw_n * |p|)
 *   + bias_n for the pixel's tap-validity pattern p(m) = h_class[ho] * n_w_classes + w_class[wo]
 *   (DESIGN.md §3).  A padding tap is the value 0, so it adds nothing to any of the three terms.
 *   The epilogue evaluates the sum in fp64 and rounds once to fp32.
 *
 * mhaq_fq_act_codes_f32: codes[pixel][c] = the forward's code of x[pixel][c] (clamped to
 *   [zero_point, max_val], per-tensor LINEAR parameters, one float each), saturated to [0, 255]
 *   (NaN -> 0) and counted into *n_out_of_range (NULL = not counted) like mhaq_fq_pack_f32;
 *   channels [n_channels, cp) are 0.  x is [n_pixels][n_channels] (channels_last NCHW storage or a
 *   [B, in] matrix); codes is [n_pixels][cp], cp % 16 == 0, 16-byte aligned.
 *
 * mhaq_fq_iconv_weight_bytes: bytes of the weight operand for n_out output channels and K =
 *   k_bytes = kh * kw * cp; -1 for a bad size.  The operand holds n_tiles tiles of tile_n rows
 *   (tile_n % 16 == 0, <= 256): tile t has output channels [t * tile_out, min(n_out, (t+1) *
 *   tile_out)), tile_out <= 255 and no tile empty, then one row of ones (it yields SA), then zero
 *   rows.  A row is K bytes in
 *   (kh, kw, cp) order, zero-padded to k_stages * 128.  Storage: [tile][stage][tile_n * 128], the
 *   byte of row r and K position 16 * c + j (0 <= c < 8, 0 <= j < 16) of a stage at
 *   (r / 8) * 1024 + c * 128 + (r % 8) * 16 + j.  Any output pointer may be NULL.
 *
 * mhaq_fq_iconv_u8: codes from mhaq_fq_act_codes_f32 ([batch][height][width][cp], 16-byte
 *   aligned), the weight operand above (16-byte aligned), alpha / beta [n_out], ctab
 *   [n_h_classes * n_w_classes][n_out], h_class [ho], w_class [wo] (int32); y is fp32
 *   [batch * ho * wo][n_out] (a channels_last [batch, n_out, ho, wo] or a [batch, n_out] tensor).
 *   Errors (before any CUDA call): cp % 16 != 0, bad sizes, a code bound outside [1, 255], and
 *   kh * kw * cp * act_max_code * weight_max_code >= 2^31 (the int32 accumulator could overflow).
 *   Capture-safe: no host synchronisation, allocation or atomic. */
int64_t mhaq_fq_iconv_weight_bytes(int64_t n_out, int64_t k_bytes, int *n_tiles, int *tile_n, int *tile_out,
                                   int64_t *k_stages);
int mhaq_fq_act_codes_f32(const float *x, uint8_t *codes, const float *scale, const float *zero_point,
                          const float *max_val, int64_t n_pixels, int64_t n_channels, int64_t cp,
                          unsigned long long *n_out_of_range, void *stream);
int mhaq_fq_iconv_u8(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                     const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                     float *y, int64_t batch, int64_t height, int64_t width, int64_t cp, int64_t n_out,
                     int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                     int act_max_code, int weight_max_code, void *stream);

/* Fused epilogue of an integer convolution.
 *   t = RN32(alpha * S + beta * SA + C) as in mhaq_fq_iconv_u8 (an eval BatchNorm k * y + shift is
 *   folded into alpha, beta and C by the caller: DESIGN.md §3 "Fused epilogue"), then
 *     residual   (optional) t = t + residual[m][n], one fp32 rounding; residual is fp32 [m][n_out],
 *                the same storage-order view as y;
 *     activation MHAQ_FQ_ACT_NONE; MHAQ_FQ_ACT_RELU: t unchanged if NaN, else fmaxf(t, 0) (torch's
 *                CUDA relu); MHAQ_FQ_ACT_LEAKY_RELU: t > 0 ? t : t * negative_slope (fp32);
 *   and writes any non-empty combination of
 *     y          fp32 [m][n_out], or NULL;
 *     codes      uint8 [m][cp_out], cp_out = round_up(n_out, 16), 16-byte aligned, or NULL: the
 *                forward's code of t under the next quantizer's per-tensor LINEAR operands
 *                (code_scale, code_zero_point, code_max_val; one float each), exactly as
 *                mhaq_fq_act_codes_f32 forms it, saturated to [0, 255] (NaN -> 0), not counted;
 *                channels [n_out, cp_out) are 0. */
#define MHAQ_FQ_ACT_NONE 0
#define MHAQ_FQ_ACT_RELU 1
#define MHAQ_FQ_ACT_LEAKY_RELU 2

typedef struct mhaq_fq_iconv_epilogue {
    const float *residual;
    int activation;
    float negative_slope;
    float *y;
    uint8_t *codes;
    const float *code_scale;
    const float *code_zero_point;
    const float *code_max_val;
} mhaq_fq_iconv_epilogue;

/* mhaq_fq_iconv_u8's arguments without y, plus the epilogue above.  Errors (before any CUDA call):
 * those of mhaq_fq_iconv_u8, no output, codes without all three code operands, an unknown
 * activation and a misaligned codes buffer.  Capture-safe like mhaq_fq_iconv_u8. */
int mhaq_fq_iconv_fused_u8(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                           const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                           int64_t batch, int64_t height, int64_t width, int64_t cp, int64_t n_out,
                           int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                           int act_max_code, int weight_max_code, const mhaq_fq_iconv_epilogue *epilogue,
                           void *stream);

/* Grouped and dilated integer convolutions (DESIGN.md §3 "Grouped and dilated layers").
 *   The layer has n_in input and n_out output channels in `groups` groups (both divisible by it);
 *   output channel n of group g(n) = n / (n_out / groups) sums over the cin_g = n_in / groups input
 *   channels of its group and the valid taps, tap (i, j) reading input position
 *   (o_h * stride_h - pad_h + i * dilation_h, o_w * stride_w - pad_w + j * dilation_w).  The output is
 *   ((height + 2 pad_h - dilation_h (kernel_h - 1) - 1) / stride_h + 1) x (... w ...).  The epilogue
 *   is that of mhaq_fq_iconv_u8 with SA[m][g(n)] the sum of the group's codes and |p| counting
 *   valid taps x cin_g.
 *
 * mhaq_fq_iconv_grouped_weight_bytes: bytes of the weight operand; -1 for a bad geometry.
 *   Depthwise (groups == n_in == n_out): u8 [kernel_h * kernel_w][cp], cp = round_up(n_in, 16),
 *   padding channels 0; *n_tiles = *tile_n = *tile_out = *groups_per_tile = *tiles_per_group =
 *   *k_stages = 0.  Otherwise N tiles as in mhaq_fq_iconv_weight_bytes, block-diagonal: when a group
 *   with its ones row fits a tile, tile t holds groups_per_tile whole groups
 *   [t * groups_per_tile, ...) (tiles_per_group = 1), their tile_out = groups_per_tile * cout_g
 *   channels, then one ones row per group (row tile_out + i for the tile's i-th group); otherwise
 *   each group spans tiles_per_group tiles of at most tile_out channels and one ones row
 *   (groups_per_tile = 1).  Tile t's K is (kh, kw, chunks [c_lo, c_hi)) with
 *   c_lo = floor(first group * cin_g / 16), c_hi = ceil(end group * cin_g / 16): a row holds its
 *   channel's weights at its own group's channels and 0 elsewhere, a ones row is 1 exactly at its
 *   group's channels.  Each row is zero-padded to k_stages * 128 bytes (the widest tile's K) and
 *   stored like mhaq_fq_iconv_weight_bytes' operand.  Any output pointer may be NULL.
 *
 * mhaq_fq_iconv_grouped_u8: codes [batch][height][width][cp] (16-byte aligned), the weight operand
 *   above (16-byte aligned), alpha / beta [n_out], ctab [n_h_classes * n_w_classes][n_out] and
 *   h_class / w_class of the dilated tap patterns; the outputs as in mhaq_fq_iconv_fused_u8 (an
 *   epilogue with y alone is the plain layer).  Depthwise layers run on the CUDA cores, all others
 *   on the tensor cores.  Errors (before any CUDA call): those of mhaq_fq_iconv_fused_u8, groups
 *   that do not divide n_in and n_out, a dilation below 1, and
 *   kernel_h * kernel_w * cin_g * act_max_code * weight_max_code >= 2^31.  Capture-safe. */
typedef struct mhaq_fq_iconv_geometry {
    int kernel_h, kernel_w;
    int stride_h, stride_w;
    int pad_h, pad_w;
    int dilation_h, dilation_w;
    int groups;
} mhaq_fq_iconv_geometry;

int64_t mhaq_fq_iconv_grouped_weight_bytes(int64_t n_in, int64_t n_out, const mhaq_fq_iconv_geometry *geometry,
                                           int *n_tiles, int *tile_n, int *tile_out, int *groups_per_tile,
                                           int *tiles_per_group, int64_t *k_stages);
int mhaq_fq_iconv_grouped_u8(const uint8_t *codes, const uint8_t *weights, const float *alpha, const float *beta,
                             const float *ctab, const int32_t *h_class, const int32_t *w_class, int n_w_classes,
                             int64_t batch, int64_t height, int64_t width, int64_t n_in, int64_t n_out,
                             const mhaq_fq_iconv_geometry *geometry, int act_max_code, int weight_max_code,
                             const mhaq_fq_iconv_epilogue *epilogue, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MHAQ_FQ_H_ */
