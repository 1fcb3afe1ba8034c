/*
 * rnnt_b200.h -- C ABI of the B200-native RNN-Transducer loss (librnnt_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of 1ytic/warp-rnnt: the loss + gradient
 * behind warp_rnnt.rnnt_loss(..., gather=, compact=).  Plain pointers and sizes only -- no
 * torch / ATen types.  All pointers are DEVICE pointers owned by the caller; every call is
 * asynchronous on `stream` (a cudaStream_t passed as void*) and never synchronises the host.
 *
 * Two groups of entry points:
 *
 *  (A) rnnt_b200_*  -- the native interface (what warp_rnnt_b200/csrc/binding.cpp binds).
 *      It fuses what the reference spreads over ATen ops + kernels: the dense zero-fill
 *      (pytorch_binding/binding.cpp:58), the python-level log-prob gather and its autograd
 *      scatter (pytorch_binding/warp_rnnt/__init__.py:118-128), the in-place grad_output
 *      scaling (__init__.py:21-24) and the compact prefix sums (binding.cpp:141-158).
 *      Scratch lives in one caller-provided workspace (size from rnnt_b200_workspace_bytes);
 *      outputs are fully written (no pre-zeroing contract).
 *
 *  (B) run_warp_rnnt / run_warp_rnnt_gather / run_gather_for_compact / run_warp_rnnt_compact /
 *      run_scatter_grad_for_compact -- the reference's own C ABI, /root/reference/core.h:29-60,
 *      same names, argument order and meaning, so the reference's pytorch_binding/binding.cpp
 *      and tensorflow_binding/binding.cpp link against librnnt_b200.so unchanged
 *      (see INTEGRATION.md).  `counts` is accepted and ignored: the global-memory polling
 *      scheduler (core.cu:64-78,136-140) is replaced by on-chip warp/cluster hand-off.
 */
#ifndef RNNT_B200_H
#define RNNT_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Status codes.  Values 0-4 are the reference's rnntStatus_t (core.h:16-22). */
typedef enum {
    RNNT_STATUS_SUCCESS = 0,
    RNNT_STATUS_WARP_FAILED = 1,        /* alpha/beta wavefront kernel */
    RNNT_STATUS_GRADS_BLANK_FAILED = 2, /* gradient kernels (blank and label are one kernel here) */
    RNNT_STATUS_GRADS_LABEL_FAILED = 3,
    RNNT_STATUS_COSTS_FAILED = 4,
    RNNT_STATUS_INVALID_ARGUMENT = 5,
    RNNT_STATUS_WORKSPACE_TOO_SMALL = 6,
    RNNT_STATUS_GATHER_FAILED = 7
} rnntStatus_t;

/* Numerics of the log-sum-exp on the wavefront's dependent chain (core.cu:26-39).
 *   RNNT_LSE_EXACT : max + log1pf(expf(d)) in the reference's operation order; alpha, beta,
 *                    costs and gradients are bit-identical to the reference kernels.
 *   RNNT_LSE_FAST  : max + ln2*lg2.approx(1 + ex2.approx(d*log2e)); ~3x shorter dependent chain,
 *                    |error| < 4e-7 per step (measured against the fp64 oracle in tests/).
 *   RNNT_LSE_AUTO  : the library default = RNNT_LSE_EXACT (parity first; see DESIGN.md section 4). */
typedef enum { RNNT_LSE_AUTO = 0, RNNT_LSE_EXACT = 1, RNNT_LSE_FAST = 2 } rnntLseMode_t;

/* Process-wide default for calls that do not pass a mode (the compat ABI (B)); initialised from
 * the environment variable RNNT_B200_LSE = auto|exact|fast. */
void rnnt_b200_set_lse_mode(int mode);
int rnnt_b200_get_lse_mode(void);

const char *rnnt_b200_version(void);
const char *rnnt_b200_status_string(int status);

/* Number of kernels this library has launched since load (all streams); bench.py reports the
 * delta over the timed region as "gpu_launches". */
uint64_t rnnt_b200_launch_count(void);

/* Diagnostics: when `buf` is non-NULL the fused small-lattice kernel records, per CTA (grid order
 * blockIdx.y * gridDim.x + blockIdx.x), sixteen clock64() stamps (latest arrival of each phase):
 * 0 start, 1 sentinels set, 2 gather done, 3 wavefront start, 4 alpha done, 5 beta done, 6 zero-fill
 * done, 7 kernel end (8..15 reserved).  `buf` is device memory, 16 * CTAs int64, zeroed by the caller.  NULL = off. */
void rnnt_b200_debug_fused_trace(void *buf);

/* Diagnostics (tests only): add `delta` to the alpha-side log-likelihood of sample `n` right before the
 * forward/backward mismatch guard (core.cu:346-367) compares it with beta[0,0], so that the guard's FIRED branch
 * (warning, zeroed gradient slab, cost = -(a+b)/2) can be exercised on well-formed input.  n < 0 = off (default).
 * Process-wide; affects the dense and gathered layouts (the compact reference has no guard). */
void rnnt_b200_debug_guard_poison(int n, float delta);

/* Diagnostics (tests only): the exact LSE's log1p is libdevice's main path restated without its unreachable tail
 * (csrc/common.cuh).  This kernel compares it with libdevice's log1pf on EVERY float in [+0, 1] (the range of
 * expf(d <= 0)), on NaN, and the complete exact LSE flavours on pseudo-random operand pairs; it ADDS the number of
 * bit mismatches to *mismatches (device memory, zeroed by the caller).  Must stay 0. */
int rnnt_b200_debug_lse_selfcheck(void *stream, unsigned long long *mismatches);

/* ------------------------------------------------------------------------------------------
 * (A) native interface
 * ------------------------------------------------------------------------------------------ */

/* Workspace bytes for a problem with `cells` lattice cells (dense: N*T*U incl. padding;
 * compact: STU = sum xn*(yn+1)) and N lattices.  Valid for every rnnt_b200_* call below. */
size_t rnnt_b200_workspace_bytes(int64_t cells, int N);

/* Dense layout.  Replaces run_warp_rnnt (core.h:29-33) + zeros_like (binding.cpp:58) and,
 * when grad_scale != NULL, RNNTLoss.backward's mul_ (__init__.py:21-24).
 *   log_probs (N,T,U,V) f32 log-softmaxed; labels (N,U-1) i32; xn,yn (N) i32
 *   costs (N) f32 out;  grads (N,T,U,V) f32 out, every element written (NULL = forward only)
 *   grad_scale (N) f32 or NULL: grads[n] *= grad_scale[n]
 *   blank in [0,V).  fastemit_lambda scales label gradients only (core.cu:327-329).
 * Lengths are NOT validated on the host (that would need a device->host copy): a sample with xn outside [1,T] or
 * yn+1 outside [1,U] gets cost NaN and an all-zero gradient slab, the call still returns RNNT_STATUS_SUCCESS (the
 * reference reads out of bounds in that case).  Callers that cannot trust their lengths check costs for NaN. */
int rnnt_b200_loss_dense(void *stream, void *workspace, size_t workspace_bytes,
                         const float *log_probs, const int *labels, const int *xn, const int *yn,
                         float *costs, float *grads, const float *grad_scale,
                         int N, int T, int U, int V, int blank, float fastemit_lambda, int lse_mode);

/* rnnt_b200_loss_dense plus the reduction of the python API (__init__.py:132-143) fused in:
 *   loss_sum (1) f32 out or NULL: sum_n costs[n] * (grad_scale ? grad_scale[n] : 1), summed in a fixed order
 *     (deterministic; lane-strided partials + shuffle tree, so the low bits differ from torch.sum's order).
 *     With grad_scale[n] = 1/N ('mean'), 1/xn[n] (average_frames) or their product this is the reduced loss and
 *     `grads` is already d loss / d log_probs -- one launch for what the reference does in
 *     zeros_like + 4 kernels + sum/mean + mul_.
 *   sync_counter: one device `unsigned`, 0 on entry, left at 0 on exit (self-resetting ticket for the
 *     last-CTA reduction of the single-kernel path; one counter per concurrently running call).  NULL: the
 *     reduction runs as a second tiny launch instead. */
int rnnt_b200_loss_dense_reduced(void *stream, void *workspace, size_t workspace_bytes,
                                 const float *log_probs, const int *labels, const int *xn, const int *yn,
                                 float *costs, float *grads, const float *grad_scale, float *loss_sum,
                                 unsigned int *sync_counter, int N, int T, int U, int V, int blank,
                                 float fastemit_lambda, int lse_mode);

/* In-place grads[n, :] *= grad_out[n * grad_out_stride] / (applied ? applied[n] : 1) for the samples where the two
 * differ (stride 0: one upstream scalar for all samples).  Replaces RNNTLoss.backward's dense mul_
 * (__init__.py:21-24): when the upstream gradient equals what the forward already multiplied in (the usual
 * loss.backward()), no memory is touched.  With applied == NULL the product is exactly the reference's. */
int rnnt_b200_rescale(void *stream, void *grads, const float *grad_out, int grad_out_stride,
                      const float *applied, int N, int64_t elems_per_sample, int elem_bytes /* 4 = f32, 2 = bf16 */);

/* Half-precision I/O (SURVEY.md 8(f)2; the reference is fp32-only, binding.cpp:17-19, __init__.py:111):
 * rnnt_b200_loss_dense_reduced with log_probs (N,T,U,V) and grads (N,T,U,V) in bfloat16.  alpha, beta, costs and all
 * arithmetic stay fp32 (the gradient is rounded to bf16 once, on the final store), so costs equal the fp32 path's on
 * the same (bf16-representable) inputs and the gradient is within bf16 rounding (2^-9 relative) of it.  Halves both
 * the algorithmic and the physical bytes of the path; grads is required (forward-only callers use the fp32 entry). */
int rnnt_b200_loss_dense_bf16(void *stream, void *workspace, size_t workspace_bytes,
                              const void *log_probs_bf16, const int *labels, const int *xn, const int *yn,
                              float *costs, void *grads_bf16, const float *grad_scale, float *loss_sum,
                              unsigned int *sync_counter, int N, int T, int U, int V, int blank,
                              float fastemit_lambda, int lse_mode);

/* Gathered layout (N,T,U,2) = [blank, label] per cell.  Replaces run_warp_rnnt_gather
 * (core.h:35-39).  pair_grads (N,T,U,2) out, fully written (zeros on padding); NULL = fwd only. */
int rnnt_b200_loss_pairs(void *stream, void *workspace, size_t workspace_bytes,
                         const float *pairs, const int *xn, const int *yn,
                         float *costs, float *pair_grads,
                         int N, int T, int U, float fastemit_lambda, int lse_mode);

/* Memory-saving path of rnnt_loss(gather=True): gather fused into the forward
 * (__init__.py:118-128 without the int64 index tensor), gradients kept as (N,T,U,2). */
int rnnt_b200_gather_forward(void *stream, void *workspace, size_t workspace_bytes,
                             const float *log_probs, const int *labels, const int *xn, const int *yn,
                             float *costs, float *pair_grads,
                             int N, int T, int U, int V, int blank, float fastemit_lambda, int lse_mode);

/* ... and its backward: out (N,T,U,V) = scatter of pair_grads * grad_out[n], zeros elsewhere,
 * every element written (replaces mul_ + GatherBackward's zeros + scatter_add_).
 * accumulate != 0: a label equal to blank adds both gradients (torch scatter_add_, gather=True);
 * accumulate == 0: the label gradient overrides (core.cu launches the label kernel last).
 * yn: with the label lengths a label slot is taken as real iff u < yn[n] (structural); with NULL every u < U-1 is,
 * and in override mode a label gradient of exactly 0 is read as "no transition" (padded labels may equal blank). */
int rnnt_b200_gather_backward(void *stream, const float *pair_grads, const int *labels,
                              const float *grad_out, float *out,
                              int N, int T, int U, int V, int blank, int accumulate,
                              const int *yn /* (N) label lengths, or NULL */);

/* Loss straight from un-normalised logits (the reference needs log-softmaxed input, README.md:59, and its
 * benchmark times F.log_softmax with the loss, pytorch_binding/benchmark.py:65): log_softmax's forward and backward
 * are fused into the two dense passes this path needs anyway.
 *   forward : one read of logits (N,T,U,V) -> lse (N,T,U) f32 out [the per-cell normaliser], costs (N), and
 *             pair_grads (N,T,U,2) out = d cost / d (blank, label) LOG-PROB per cell (NULL = costs only)
 *   backward: out (N,T,U,V) = d sum_n grad_out[n] cost[n] / d logits
 *                           = [v==blank] gb + [v==label] gl - exp(logit[v] - lse) (gb + gl), times grad_out[n]
 *             (grad_out NULL = ones); every element written; a label equal to blank adds both (autograd semantics).
 * Not bit-identical to torch.log_softmax + the reference (the normaliser is summed in a different order):
 * costs agree to 1e-5 relative, gradients to 1e-4 absolute (tests/test_gpu_logits.py). */
int rnnt_b200_logits_forward(void *stream, void *workspace, size_t workspace_bytes, const float *logits,
                             const int *labels, const int *xn, const int *yn, float *costs, float *lse,
                             float *pair_grads, int N, int T, int U, int V, int blank, float fastemit_lambda,
                             int lse_mode);
int rnnt_b200_logits_backward(void *stream, const float *logits, const float *lse, const float *pair_grads,
                              const int *labels, const float *grad_out, float *out, int N, int T, int U, int V,
                              int blank);

/* The same two calls with bfloat16 logits (N,T,U,V) and a bfloat16 logit gradient `out`; lse, costs, pair_grads and
 * grad_out stay fp32.  Every bf16 value is converted exactly to fp32 and all arithmetic is the fp32 calls', in their
 * order (the same elements are summed by the same lanes in the same order), so for bf16 logits x:
 *   costs, lse and pair_grads are bit for bit those of rnnt_b200_logits_forward on x converted to fp32, in either LSE
 *   mode, and out is that of rnnt_b200_logits_backward rounded once to bf16 (round to nearest even).
 * Halves the bytes of the two dense passes.  An odd logits / out address returns RNNT_STATUS_INVALID_ARGUMENT
 * (tests/test_gpu_logits_bf16.py). */
int rnnt_b200_logits_forward_bf16(void *stream, void *workspace, size_t workspace_bytes, const void *logits_bf16,
                                  const int *labels, const int *xn, const int *yn, float *costs, float *lse,
                                  float *pair_grads, int N, int T, int U, int V, int blank, float fastemit_lambda,
                                  int lse_mode);
int rnnt_b200_logits_backward_bf16(void *stream, const void *logits_bf16, const float *lse, const float *pair_grads,
                                   const int *labels, const float *grad_out, void *out_bf16, int N, int T, int U,
                                   int V, int blank);

/* Compact (ragged) layout.  xs (STU,V), ys (sum yn), STU = sum xn*(yn+1).
 * Replaces run_gather_for_compact + run_warp_rnnt_compact (core.h:41-55) and the host-side
 * prefix sums / .item() syncs of binding.cpp:132-158 (prefix sums are computed on device).
 *   pair_grads (STU,2) out or NULL (forward only = the reference's required_grad=false)
 *   loc (STU) i64 out or NULL: label id per cell, blank on each sample's last column
 *   totals (4) i32 out or NULL: {sum xn*(yn+1), sum yn, max xn, max yn+1} for host validation
 *   max_T, max_U: launch-shaping hints, UPPER BOUNDS of xn and yn+1 (0 = unknown: general kernels).  With
 *   hints small lattices take the single fused kernel; a sample exceeding the hints gets cost NaN. */
int rnnt_b200_compact_forward(void *stream, void *workspace, size_t workspace_bytes,
                              const float *xs, const int *ys, const int *xn, const int *yn,
                              float *costs, float *pair_grads, int64_t *loc, int *totals,
                              int64_t STU, int N, int V, int blank, float fastemit_lambda,
                              int lse_mode, int max_T, int max_U);

/* totals (4) i32 out = {sum xn*(yn+1), sum yn, max xn, max yn+1} (each clamped to INT32_MAX):
 * lets a binding validate shapes with ONE small device->host copy instead of the reference's
 * four .item() syncs (binding.cpp:132,137,138,146).  scratch: 2*N int64 of device memory. */
int rnnt_b200_compact_totals(void *stream, const int *xn, const int *yn, int N, int64_t *scratch,
                             int *totals);

/* Compact packing of the joint network's INPUT -- the caller side of the compact layout (SURVEY.md 8(f)3;
 * the reference's benchmark does it with a python loop, 2N host syncs and a cat, benchmark2.py:37-50):
 *   x[row(n,t,u), :] = f[n,t,:] + g[n,u,:]   for t < lf[n], u <= lg[n],   row(n,t,u) = mem_pref[n] + t*(lg[n]+1) + u
 * f (N,T,H) encoder output, g (N,U1,H) predictor output (U1 = max labels + 1), lf / lg (N) i32 = the loss'
 * frames_lengths / labels_lengths, x (STU,H) out, H the joint dimension.  scratch: 2*N int64 of device memory; on
 * return scratch[0..N) = mem_pref (kept by the caller for the backward).  totals (4) i32 out or NULL as in
 * rnnt_b200_compact_totals (totals[0] = STU).  x == NULL: prefix sums / totals only (to size x).
 * stu_hint: STU if known (launch shaping only), else 0. */
int rnnt_b200_joint_pack(void *stream, const float *f, const float *g, const int *lf, const int *lg,
                         int64_t *scratch, int *totals, float *x, int N, int T, int U1, int H, int64_t stu_hint);
/* ... and its backward: df (N,T,H) = sum over u of dx rows, dg (N,U1,H) = sum over t; zeros on padding; fixed
 * summation order (deterministic).  df or dg may be NULL. */
int rnnt_b200_joint_pack_backward(void *stream, const float *dx, const int *lf, const int *lg,
                                  const int64_t *mem_pref, float *df, float *dg, int N, int T, int U1, int H);

/* Compact backward: out (STU,V) fully written.  Replaces torch::zeros (binding.cpp:239) +
 * run_scatter_grad_for_compact (core.h:56-60).  cum_lens (N) i32 inclusive cumsum. */
int rnnt_b200_compact_backward(void *stream, const float *grad_cost, const float *pair_grads,
                               const int64_t *loc, const int *cum_lens, float *out,
                               int64_t STU, int N, int V, int blank);

/* ------------------------------------------------------------------------------------------
 * (B) the reference's C ABI, /root/reference/core.h:29-60 (argument-for-argument)
 * ------------------------------------------------------------------------------------------ */
#ifndef RNNT_CORE_H /* do not clash if the reference's core.h is also included */
int run_warp_rnnt(void *stream, unsigned int *counts, float *alphas, float *betas,
                  const int *labels, const float *log_probs, float *grads, float *costs,
                  const int *xn, const int *yn, int N, int T, int U, int V, int blank,
                  float fastemit_lambda);

int run_warp_rnnt_gather(void *stream, unsigned int *counts, float *alphas, float *betas,
                         const float *log_probs, float *grads, float *costs, const int *xn,
                         const int *yn, int N, int T, int U, float fastemit_lambda);

void run_gather_for_compact(const float *xs, const int *ys, const unsigned int *xn,
                            const unsigned int *yn, float *gather_xs, long *loc,
                            const unsigned int *memPref, const unsigned int *labelPref,
                            unsigned int N, unsigned int T, unsigned int U, unsigned int V,
                            unsigned int blank);

void run_warp_rnnt_compact(unsigned int *counts, float *alphas, float *betas,
                           const float *log_probs, float *grads, float *costs,
                           const unsigned int *xn, const unsigned int *yn,
                           const unsigned int *memPref, const unsigned int *labelPref,
                           unsigned int N, unsigned int T, unsigned int U, float fastemit_lambda,
                           bool required_grad);

void run_scatter_grad_for_compact(const float *grad_cost, const float *gather_grad,
                                  const long *loc, const int *cum_lens, float *scatter_grad,
                                  unsigned int STU, unsigned int N, unsigned int V,
                                  unsigned int blank);
#endif

#ifdef __cplusplus
}
#endif
#endif /* RNNT_B200_H */
