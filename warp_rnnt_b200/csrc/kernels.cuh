// kernels.cuh -- host-side launch entry points shared between the .cu files and api.cu.
#pragma once
#include "common.cuh"

namespace rnnt {

void count_launch();   // api.cu: bumps the library-wide launch counter
// api.cu: test hook (rnnt_b200_debug_guard_poison): sample index whose alpha-side log-likelihood gets `delta` added
// in front of the forward/backward mismatch guard; n < 0 = off
struct GuardPoison { int n; float delta; };
GuardPoison guard_poison();

cudaError_t launch_prefix(cudaStream_t s, const int *xn, const int *yn, int N, int64_t *mem_pref,
                          int64_t *lab_pref, int *totals);
cudaError_t launch_gather(cudaStream_t s, const Problem &p, const void *lp, const int *labels, int V, int blank,
                          float2 *pairs, int64_t *loc, int64_t cells_hint, int io_bf16 = 0);
cudaError_t launch_wavefront(cudaStream_t s, int kind, const Problem &p, const float2 *pairs, float *alphas,
                             float *betas, float *ws_ll, int *bad, float *costs, int beta_only, int guard,
                             int t_hint, int u_hint);
cudaError_t launch_grads_pairs(cudaStream_t s, const Problem &p, const float2 *pairs, const float *alphas,
                               const float *betas, const int *bad, float fastemit_lambda, float2 *out,
                               int64_t cells_hint);

// expand.cu -- dense gradient emit (every element of `out` is written)
struct ExpandSrc {
    // source A: alpha/beta/pairs (forward, dense layout)      -> pg == nullptr
    // source B: pair grads (cells,2) (+ per-sample scale)     -> pg != nullptr
    const float2 *pairs;
    const float *alphas;
    const float *betas;
    const int *bad;
    const float2 *pg;
    const float *scale;      // (N) or nullptr
    const int *labels;       // dense: (N,U-1)
    const int64_t *loc;      // compact backward: label id per cell (blank on the last column)
    const int *cum_lens;     // compact backward: inclusive cumsum of xn*(yn+1), (N)
    float fastemit_lambda;
    int label_adds;          // 1: label == blank accumulates (torch scatter_add semantics of gather=True)
};
cudaError_t launch_expand(cudaStream_t s, const Problem &p, const ExpandSrc &src, void *out, int64_t cells,
                          int V, int blank, bool retire_early = false, int io_bf16 = 0);   // io_bf16: bf16 output (forward emit)

// logits.cu -- loss from un-normalised logits (fused log_softmax forward / backward); io_bf16: x (and out) bf16
cudaError_t launch_lse_pairs(cudaStream_t s, const void *x, const int *labels, int N, int T, int U, int V, int blank,
                             float2 *pairs, float *lse, int io_bf16 = 0);
cudaError_t launch_expand_logits(cudaStream_t s, const void *x, const float *lse, const float2 *pg, const int *labels,
                                 const float *grad_out, void *out, int N, int T, int U, int V, int blank,
                                 int io_bf16 = 0);

// joint.cu -- compact packing of the joint network's input (caller side of compact=True)
cudaError_t launch_joint_pack(cudaStream_t s, const float *f, const float *g, const int *lf, const int *lg,
                              const int64_t *mem_pref, float *x, int N, int T, int U1, int H, int64_t stu_hint);
cudaError_t launch_joint_grads(cudaStream_t s, const float *dx, const int *lf, const int *lg, const int64_t *mem_pref,
                               float *df, float *dg, int N, int T, int U1, int H);

// One loss call: its inputs, shape, numerics and outputs.  api.cu fills one per call and runs it either through
// launch_fused or through the general sequence (gather, wavefront, gradient stage).
struct LossJob {
    // inputs
    const void *lp;            // dense (N,T,U,V) log-probs, f32 or (io_bf16) bf16; pairs_in: (cells,2) f32
    const int *labels;         // dense: (N,U-1); compact: (sum yn); pairs_in: unused
    const int *xn, *yn;
    const int64_t *mem_pref, *lab_pref;   // compact layout: first cell / first label of lattice n; dense: null
    int pairs_in;              // lp is already the (cells,2) {blank, label} layout: no gather, V = 2, blank = 0
    int io_bf16;               // lp and grads are bf16 (dense gradient only)
    // shape
    int N, T, U, V, blank;     // compact: T, U = upper bounds of the lengths, or 0 when unknown
    int64_t cells;             // dense: N*T*U; compact: cells of the packed layout (or a bound on them)
    // numerics
    int kind;                  // LSE flavour (kExactDense, kExactCompact, kFast)
    int guard;                 // forward/backward mismatch guard on
    float lam;                 // FastEmit lambda
    // outputs
    float *costs;              // (N)
    void *grads;               // dense gradient (N,T,U,V), or null
    float2 *pair_grads;        // (cells,2) gradient, or null; with neither: loss only
    const float *scale;        // (N) per-sample factor of the dense gradient and of loss_sum, or null
    int64_t *loc;              // compact layout: label id per cell, written by the gather; or null
    float *loss_sum;           // sum_n costs[n] * scale[n], or null
    unsigned *sync_counter;    // with loss_sum: zeroed device counter that lets the fused kernel write the sum itself
};

// fused.cu -- single-kernel path for lattices that fit shared memory
struct FusedPlan { int W, ring, nw, slices; size_t smem; };
bool fused_plan(int N, int T, int U, FusedPlan *plan);
void set_fused_trace(long long *buf);   // diagnostics: per-CTA phase stamps of k_fused (8 x clock64 per CTA)
cudaError_t launch_fused(cudaStream_t s, const LossJob &job, const FusedPlan &plan);

// expand.cu -- small helpers of the python-level API
cudaError_t launch_loss_sum(cudaStream_t s, const float *costs, const float *scale, int N, float *loss_sum);
cudaError_t launch_rescale(cudaStream_t s, void *grads, const float *grad_out, int grad_out_stride,
                           const float *applied, int N, int64_t elems_per_sample, int io_bf16 = 0);

}  // namespace rnnt
