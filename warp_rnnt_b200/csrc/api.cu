// api.cu -- the extern "C" surface of librnnt_b200.so (declared in include/rnnt_b200.h).
//
// (A) rnnt_b200_*: native interface bound by csrc/binding.cpp.
// (B) run_warp_rnnt & co: the reference's C ABI (/root/reference/core.h:29-60) implemented on top
//     of (A)'s kernels so the reference's own bindings link against this library unchanged.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "kernels.cuh"

namespace rnnt {

static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static std::atomic<int> g_poison_n{-1};
static std::atomic<float> g_poison_delta{0.0f};
GuardPoison guard_poison() { return {g_poison_n.load(std::memory_order_relaxed), g_poison_delta.load(std::memory_order_relaxed)}; }

static int env_lse_mode() {
    const char *e = getenv("RNNT_B200_LSE");
    if (!e) return RNNT_LSE_AUTO;
    if (!strcmp(e, "exact")) return RNNT_LSE_EXACT;
    if (!strcmp(e, "fast")) return RNNT_LSE_FAST;
    return RNNT_LSE_AUTO;
}
static std::atomic<int> g_lse_mode{-1};

static int default_lse_mode() {
    int m = g_lse_mode.load(std::memory_order_relaxed);
    if (m < 0) {
        m = env_lse_mode();
        g_lse_mode.store(m, std::memory_order_relaxed);
    }
    return m;
}

// AUTO policy (DESIGN.md "numerics"): AUTO = exact, i.e. results are bit-identical to the reference
// kernels unless the caller opts out.  Parity is the first gate: at BASELINE cfg 2 the fast flavour
// differs from the reference by up to 1.2e-4 on a gradient (pure fp32 noise -- the reference itself is
// 1.25e-4 away from fp64 there), which is outside the stated 1e-4.  The exact chain is ~2x longer per
// anti-diagonal; it costs ~10 us at cfg 2 and nothing measurable where the dense write dominates
// (cfg 3-5).  RNNT_LSE_FAST / RNNT_B200_LSE=fast selects the short chain.
static int resolve_kind(int lse_mode, bool compact) {
    if (lse_mode == RNNT_LSE_AUTO) lse_mode = default_lse_mode();
    if (lse_mode == RNNT_LSE_FAST) return kFast;
    return compact ? kExactCompact : kExactDense;
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// RNNT_B200_PATH = auto | fused | general  (tests exercise both paths on the same inputs)
static int forced_path() {
    static const int path = [] {
        const char *e = getenv("RNNT_B200_PATH");
        return (e && !strcmp(e, "general")) ? 2 : (e && !strcmp(e, "fused")) ? 1 : 0;
    }();
    return path;
}

struct Workspace {
    float2 *pairs;
    float *alphas, *betas, *ll;
    int *bad;
    int64_t *mem_pref, *lab_pref;
    int *totals;
    size_t bytes;
};

// Sections of a workspace.  The native entry points take all of them (rnnt_b200_workspace_bytes); the
// reference-ABI shims leave out what their call does not use, e.g. alphas and betas, which their caller owns.
enum : unsigned { kWsPairs = 1, kWsLattices = 2, kWsLL = 4, kWsBad = 8, kWsPrefix = 16, kWsAll = 31 };

static Workspace carve(void *base, int64_t cells, int N, unsigned parts = kWsAll) {
    Workspace w;
    size_t off = 0;
    auto take = [&](unsigned part, size_t bytes) {
        if (!(parts & part)) return (void *)nullptr;
        void *p = base ? (void *)((char *)base + off) : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    const size_t c = (size_t)(cells > 0 ? cells : 0), n = (size_t)(N > 0 ? N : 0);
    w.pairs = (float2 *)take(kWsPairs, c * sizeof(float2));
    w.alphas = (float *)take(kWsLattices, c * sizeof(float));
    w.betas = (float *)take(kWsLattices, c * sizeof(float));
    w.ll = (float *)take(kWsLL, 2 * n * sizeof(float));
    w.bad = (int *)take(kWsBad, n * sizeof(int));
    w.mem_pref = (int64_t *)take(kWsPrefix, n * sizeof(int64_t));
    w.lab_pref = (int64_t *)take(kWsPrefix, n * sizeof(int64_t));
    w.totals = (int *)take(kWsPrefix, 4 * sizeof(int));
    w.bytes = off;
    return w;
}

static bool dense_args_ok(int N, int T, int U, int V) {
    if (N < 0 || T < 1 || U < 1 || V < 1) return false;
    if ((int64_t)T * U >= (int64_t)1 << 31) return false;
    if ((int64_t)N * T * U >= (int64_t)1 << 31) return false;   // cell ids are 32-bit in the emit kernel
    if (V >= (1 << 22)) return false;
    return true;
}
// (cells,2) float2 buffers must be 8-byte aligned; null passes
static bool f2_aligned(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }
// A dense-layout call: its shape, its blank id, and its (cells,2) gradient buffer (if any) aligned.
static bool dense_call_ok(int N, int T, int U, int V, int blank, const void *pair_grads = nullptr) {
    return dense_args_ok(N, T, U, V) && blank >= 0 && blank < V && f2_aligned(pair_grads);
}

// Internal streams for the pipelined general path: one for gathers, one for emits, four
// high-priority ones for wavefronts (their CTAs are few and long-lived; priority lets them take the
// SMs that free up at every gather / emit kernel boundary).  Created once per process and device.
struct Pipeline {
    static constexpr int kWave = 4, kGroups = 8;
    cudaStream_t gather_s, expand_s, wave_s[kWave];
    cudaEvent_t fork, gathered[kGroups], swept[kGroups], join[2 + kWave];
    int device;
};
static bool pipeline_enabled() {
    // on by default (RNNT_B200_PIPELINE=0 disables).  Measured on B200, same box: cfg 5 micro-batch
    // 2.23 ms pipelined vs 2.38 ms serial, cfg 4 2.85 vs 2.94 ms.  It only pays off with the
    // early-retiring emit grid (launch_expand retire_early): persistent emit CTAs hold every SM
    // until their kernel ends and the high-priority wavefront CTAs never get in (2.96 vs 2.90 ms).
    static const bool on = !env_is("RNNT_B200_PIPELINE", '0');
    return on;
}
// One pipeline per device (streams and events belong to a device); created on first use under g_pipe_mu,
// which also serialises the calls that use a pipeline's shared events.
static std::mutex g_pipe_mu;
static Pipeline *get_pipeline_locked() {
    static Pipeline *pipes[kMaxDevices] = {};
    const int dev = current_device();
    if (dev >= kMaxDevices) return nullptr;
    if (pipes[dev]) return pipes[dev];
    Pipeline *p = new Pipeline();
    p->device = dev;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = numerically lowest = highest priority
    bool ok = cudaStreamCreateWithPriority(&p->gather_s, cudaStreamNonBlocking, lo) == cudaSuccess &&
              cudaStreamCreateWithPriority(&p->expand_s, cudaStreamNonBlocking, lo) == cudaSuccess;
    for (int i = 0; i < Pipeline::kWave && ok; ++i)
        ok = cudaStreamCreateWithPriority(&p->wave_s[i], cudaStreamNonBlocking, hi) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&p->fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < Pipeline::kGroups && ok; ++i)
        ok = cudaEventCreateWithFlags(&p->gathered[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&p->swept[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 2 + Pipeline::kWave && ok; ++i)
        ok = cudaEventCreateWithFlags(&p->join[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { cudaGetLastError(); delete p; return nullptr; }
    pipes[dev] = p;
    return p;
}

// Self-check of the restated log1pf (common.cuh:log1pf_unit) against libdevice: every float in [+0, 1], a NaN, and the
// complete exact LSE (both flavours) on pseudo-random operand pairs.  counts[0] += mismatches.
__global__ void k_lse_selfcheck(unsigned long long *counts) {
    unsigned long long bad = 0;
    const uint32_t top = 0x3f800000u;                       // 1.0f
    for (uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; b <= top; b += (uint64_t)gridDim.x * blockDim.x) {
        const float x = __uint_as_float((uint32_t)b);
        const uint32_t r0 = __float_as_uint(log1pf(x)), r1 = __float_as_uint(log1pf_unit(x));
        bad += (r0 != r1);
    }
    // NaN in, NaN out (the guard lives in lse_tail); NaN / inf - inf operands of the whole LSE stay NaN like the reference's
    { const float n = lse_tail(-1.0f, __uint_as_float(0x7fc00000u + threadIdx.x)); bad += !(n != n); }
    {
        const float qn = __uint_as_float(0x7fc00000u), inf = __uint_as_float(0x7f800000u);
        const float A4[8] = {qn, 1.0f, -inf, inf, -3.0f, 0.0f, -inf, -2.5f}, B4[8] = {1.0f, qn, -inf, inf, -3.0f, -0.0f, -7.0f, -inf};
        for (int k = 0; k < 8; ++k) {
            const float a = A4[k], b2 = B4[k];
            float mx, df;
            if (a > b2) { mx = a; df = b2 - a; } else { mx = b2; df = a - b2; }
            const float ref = mx + log1pf(expf(df)), got = lse<kExactDense>(a, b2);
            bad += ((ref != ref) != (got != got)) || (ref == ref && __float_as_uint(ref) != __float_as_uint(got));
            const float tmp = a - b2;
            const float refc = (a == b2) ? (float)(a + M_LN2) : (tmp > 0) ? a + log1pf(expf(-tmp)) : (tmp <= 0) ? b2 + log1pf(expf(tmp)) : tmp;
            const float gotc = lse<kExactCompact>(a, b2);
            bad += ((refc != refc) != (gotc != gotc)) || (refc == refc && __float_as_uint(refc) != __float_as_uint(gotc));
        }
    }
    // -0 as the larger operand: (-0) + log1p(e) and (+0) + log1p(e) are the same float for every e in [0, 1]
    { const float r0 = lse<kExactDense>(-0.0f, -3.0f), r1 = -0.0f + log1pf(expf(-3.0f)); bad += (__float_as_uint(r0) != __float_as_uint(r1));
      const float r2 = lse<kExactDense>(-0.0f, -__uint_as_float(0x7f800000u)), r3 = -0.0f + log1pf(0.0f); bad += (__float_as_uint(r2) != __float_as_uint(r3)); }
    // the whole LSE on operand pairs spread over the magnitudes the lattices see (a hash of the thread index)
    uint32_t h = 0x9e3779b9u * ((uint32_t)blockIdx.x * blockDim.x + threadIdx.x + 1u);
    for (int k = 0; k < 64; ++k) {
        h = h * 1664525u + 1013904223u;
        const float a = -(float)(h >> 8) * (1.0f / 65536.0f) * 40.0f;       // [-10240, 0]
        h = h * 1664525u + 1013904223u;
        const float d = ((float)(h >> 8) * (1.0f / 16777216.0f) - 0.5f) * ((k & 1) ? 40.0f : 2.0f);
        const float b2 = a + d;
        float mx, df;
        if (a > b2) { mx = a; df = b2 - a; } else { mx = b2; df = a - b2; }
        const float ref = mx + log1pf(expf(df));
        bad += (__float_as_uint(ref) != __float_as_uint(lse<kExactDense>(a, b2)));
        const float tmp = a - b2;
        float refc = (a == b2) ? (float)(a + M_LN2) : ((tmp > 0) ? a + log1pf(expf(-tmp)) : b2 + log1pf(expf(tmp)));
        bad += (__float_as_uint(refc) != __float_as_uint(lse<kExactCompact>(a, b2)));
    }
    if (bad) atomicAdd(counts, bad);
}

#define RNNT_TRY(expr, code)                                            \
    do {                                                                \
        cudaError_t e__ = (expr);                                       \
        if (e__ != cudaSuccess) {                                       \
            fprintf(stderr, "rnnt_b200: %s failed: %s\n", #expr, cudaGetErrorString(e__)); \
            return (code);                                              \
        }                                                               \
    } while (0)

// The general sequence over the scratch in `w`: gather (unless the input already is pairs), the wavefront (beta
// only when no gradient is asked for), then the dense emit or the (cells,2) gradients.
static int run_general(cudaStream_t s, const LossJob &j, const Workspace &w) {
    const int compact = j.mem_pref != nullptr;
    const Problem p = {j.xn, j.yn, j.mem_pref, j.lab_pref, j.N, compact ? 0 : j.T, compact ? 0 : j.U, compact};
    const float2 *pairs = j.pairs_in ? static_cast<const float2 *>(j.lp) : w.pairs;
    // without the guard, `bad` would only mark the lattices that are not L.ok, which every later kernel checks itself
    int *bad = j.guard ? w.bad : nullptr;
    if (!j.pairs_in)
        RNNT_TRY(launch_gather(s, p, j.lp, j.labels, j.V, j.blank, w.pairs, j.loc, j.cells, j.io_bf16),
                 RNNT_STATUS_GATHER_FAILED);
    RNNT_TRY(launch_wavefront(s, j.kind, p, pairs, w.alphas, w.betas, w.ll, bad, j.costs, !j.grads && !j.pair_grads,
                              j.guard, j.T, j.U),
             RNNT_STATUS_WARP_FAILED);
    if (j.grads) {
        ExpandSrc src = {};
        src.pairs = pairs; src.alphas = w.alphas; src.betas = w.betas; src.bad = bad;
        src.scale = j.scale; src.labels = j.labels; src.fastemit_lambda = j.lam;
        RNNT_TRY(launch_expand(s, p, src, j.grads, j.cells, j.V, j.blank, false, j.io_bf16),
                 RNNT_STATUS_GRADS_BLANK_FAILED);
    } else if (j.pair_grads) {
        RNNT_TRY(launch_grads_pairs(s, p, pairs, w.alphas, w.betas, bad, j.lam, j.pair_grads, j.cells),
                 RNNT_STATUS_GRADS_BLANK_FAILED);
    }
    return RNNT_STATUS_SUCCESS;
}

// The general sequence of a dense job with gradients, pipelined.  Returns false, having launched nothing, when the
// batch is not pipelined; else true with the status in *status.
static bool run_pipelined(cudaStream_t s, const LossJob &j, const Workspace &w, int *status) {
    const int N = j.N, T = j.T, U = j.U, V = j.V, blank = j.blank, io_bf16 = j.io_bf16;
    const int64_t cells = j.cells;
    const void *grads = j.grads;
    const size_t esz = io_bf16 ? 2 : 4;
    auto lp_at = [&](int64_t cell0) { return (const void *)((const char *)j.lp + (size_t)cell0 * V * esz); };
    auto g_at = [&](int64_t cell0) { return (void *)((char *)j.grads + (size_t)cell0 * V * esz); };
    // Large batches of large lattices: software-pipeline lattice groups over internal streams so that the
    // latency-bound wavefront of group g overlaps the bandwidth-bound gather of g+1 and emit of g-1.
    // ... which only pays when the wavefront (a per-lattice latency chain of T+U-1 steps, ~0.45 us each, that does not
    // shrink with the group) is short against the bandwidth-bound emit: measured on B200, cfg 5 micro-batch (chain
    // 0.34 ms, emit 2.1 ms) 2.14 ms pipelined vs 2.39 ms serial; cfg 4 (chain 0.8 ms, emit 1.05 ms) 2.96 vs 2.70 ms.
    const double wave_us = 0.45 * (T + U), emit_us = (double)cells * V * (io_bf16 ? 2 : 4) / 5.5e6;
    const int groups = (grads && N >= 8 && (int64_t)cells * V * 4 >= ((int64_t)512 << 20) && pipeline_enabled() &&
                        wave_us < 0.4 * emit_us)
                           ? (N >= 32 ? 8 : 4) : 1;
    if (groups <= 1) return false;
    std::lock_guard<std::mutex> lock(g_pipe_mu);    // the pipeline's events are shared by all calls on this device
    Pipeline *pl = get_pipeline_locked();
    if (!pl) return false;
    *status = RNNT_STATUS_SUCCESS;
    cudaEventRecord(pl->fork, s);
    cudaStreamWaitEvent(pl->gather_s, pl->fork, 0);
    cudaStreamWaitEvent(pl->expand_s, pl->fork, 0);
    for (int i = 0; i < Pipeline::kWave; ++i) cudaStreamWaitEvent(pl->wave_s[i], pl->fork, 0);
    for (int g = 0; g < groups && !*status; ++g) {
        const int n0 = (int)((int64_t)N * g / groups), n1 = (int)((int64_t)N * (g + 1) / groups);
        const int ng = n1 - n0;
        const int64_t c0 = (int64_t)n0 * T * U, cg = (int64_t)ng * T * U;
        Problem p = {j.xn + n0, j.yn + n0, nullptr, nullptr, ng, T, U, 0};
        const int *lab_g = j.labels + (int64_t)n0 * (U - 1);
        cudaStream_t ws = pl->wave_s[g % Pipeline::kWave];
        if (launch_gather(pl->gather_s, p, lp_at(c0), lab_g, V, blank, w.pairs + c0, nullptr, cg, io_bf16) != cudaSuccess)
            *status = RNNT_STATUS_GATHER_FAILED;
        cudaEventRecord(pl->gathered[g], pl->gather_s);
        cudaStreamWaitEvent(ws, pl->gathered[g], 0);
        if (!*status && launch_wavefront(ws, j.kind, p, w.pairs + c0, w.alphas + c0, w.betas + c0, w.ll + 2 * n0,
                                         w.bad + n0, j.costs + n0, 0, 1, T, U) != cudaSuccess)
            *status = RNNT_STATUS_WARP_FAILED;
        cudaEventRecord(pl->swept[g], ws);
        cudaStreamWaitEvent(pl->expand_s, pl->swept[g], 0);
        ExpandSrc src = {};
        src.pairs = w.pairs + c0; src.alphas = w.alphas + c0; src.betas = w.betas + c0; src.bad = w.bad + n0;
        src.scale = j.scale ? j.scale + n0 : nullptr; src.labels = lab_g; src.fastemit_lambda = j.lam;
        if (!*status && launch_expand(pl->expand_s, p, src, g_at(c0), cg, V, blank, true, io_bf16) != cudaSuccess)
            *status = RNNT_STATUS_GRADS_BLANK_FAILED;
    }
    cudaEventRecord(pl->join[0], pl->gather_s);
    cudaEventRecord(pl->join[1], pl->expand_s);
    cudaStreamWaitEvent(s, pl->join[0], 0);
    cudaStreamWaitEvent(s, pl->join[1], 0);
    for (int i = 0; i < Pipeline::kWave; ++i) {
        cudaEventRecord(pl->join[2 + i], pl->wave_s[i]);
        cudaStreamWaitEvent(s, pl->join[2 + i], 0);
    }
    return true;
}

// A native entry point's job: the fused kernel when its plan takes the shape (never for a compact job without
// length bounds, T = U = 0) and RNNT_B200_PATH does not force the general path; else the general sequence over the
// caller's workspace, pipelined where that pays.  Then the loss sum: inside the fused kernel when a counter is
// given, else one more launch.
static int dispatch(cudaStream_t s, const LossJob &j, void *workspace, size_t workspace_bytes) {
    FusedPlan plan;
    const bool fused = forced_path() < 2 && fused_plan(j.N, j.T, j.U, &plan);
    if (fused) {
        RNNT_TRY(launch_fused(s, j, plan), RNNT_STATUS_WARP_FAILED);
    } else {
        const Workspace w = carve(workspace, j.cells, j.N);
        if (!workspace || workspace_bytes < w.bytes) return RNNT_STATUS_WORKSPACE_TOO_SMALL;
        int status;
        if (!run_pipelined(s, j, w, &status)) status = run_general(s, j, w);
        if (status) return status;
    }
    if (j.loss_sum && !(fused && j.sync_counter))
        RNNT_TRY(launch_loss_sum(s, j.costs, j.scale, j.N, j.loss_sum), RNNT_STATUS_COSTS_FAILED);
    return RNNT_STATUS_SUCCESS;
}

}  // namespace rnnt

using namespace rnnt;

// dense layout, log_probs / grads of 4-byte (f32) or 2-byte (bf16) elements
static int loss_dense_any(void *stream, void *workspace, size_t workspace_bytes, const void *log_probs,
                          const int *labels, const int *xn, const int *yn, float *costs, void *grads,
                          const float *grad_scale, float *loss_sum, unsigned int *sync_counter, int N, int T,
                          int U, int V, int blank, float fastemit_lambda, int lse_mode, int io_bf16) {
    if (io_bf16 && !grads) return RNNT_STATUS_INVALID_ARGUMENT;
    if (!dense_call_ok(N, T, U, V, blank)) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    LossJob j = {};
    j.lp = log_probs; j.labels = labels; j.xn = xn; j.yn = yn; j.io_bf16 = io_bf16;
    j.N = N; j.T = T; j.U = U; j.V = V; j.blank = blank; j.cells = (int64_t)N * T * U;
    j.kind = resolve_kind(lse_mode, false); j.guard = 1; j.lam = fastemit_lambda;
    j.costs = costs; j.grads = grads; j.scale = grad_scale; j.loss_sum = loss_sum; j.sync_counter = sync_counter;
    return dispatch((cudaStream_t)stream, j, workspace, workspace_bytes);
}

// loss from logits of 4-byte (f32) or 2-byte (bf16) elements; lse, costs and pair gradients are f32 either way
static int logits_forward_any(void *stream, void *workspace, size_t workspace_bytes, const void *logits,
                              const int *labels, const int *xn, const int *yn, float *costs, float *lse,
                              float *pair_grads, int N, int T, int U, int V, int blank, float fastemit_lambda,
                              int lse_mode, int io_bf16) {
    if (!dense_call_ok(N, T, U, V, blank, pair_grads) || !lse) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    const Workspace w = carve(workspace, (int64_t)N * T * U, N);
    if (!workspace || workspace_bytes < w.bytes) return RNNT_STATUS_WORKSPACE_TOO_SMALL;
    // one pass over the logits: normaliser per cell + the two normalised log-probs the recurrence needs
    RNNT_TRY(launch_lse_pairs((cudaStream_t)stream, logits, labels, N, T, U, V, blank, w.pairs, lse, io_bf16),
             RNNT_STATUS_GATHER_FAILED);
    // the (cells,2) layout from here on: the job of rnnt_b200_loss_pairs over the workspace's pairs
    return rnnt_b200_loss_pairs(stream, workspace, workspace_bytes, reinterpret_cast<const float *>(w.pairs), xn, yn,
                                costs, pair_grads, N, T, U, fastemit_lambda, lse_mode);
}

static int logits_backward_any(void *stream, const void *logits, const float *lse, const float *pair_grads,
                               const int *labels, const float *grad_out, void *out, int N, int T, int U, int V,
                               int blank, int io_bf16) {
    if (!dense_call_ok(N, T, U, V, blank, pair_grads)) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    RNNT_TRY(launch_expand_logits((cudaStream_t)stream, logits, lse, reinterpret_cast<const float2 *>(pair_grads), labels,
                                  grad_out, out, N, T, U, V, blank, io_bf16),
             RNNT_STATUS_GRADS_BLANK_FAILED);
    return RNNT_STATUS_SUCCESS;
}

static bool bf16_aligned(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 1u) == 0; }

extern "C" {

const char *rnnt_b200_version(void) { return "0.1.0 (sm_100a)"; }

const char *rnnt_b200_status_string(int s) {
    switch (s) {
        case RNNT_STATUS_SUCCESS: return "success";
        case RNNT_STATUS_WARP_FAILED: return "alpha/beta wavefront kernel failed";
        case RNNT_STATUS_GRADS_BLANK_FAILED: return "gradient kernel failed";
        case RNNT_STATUS_GRADS_LABEL_FAILED: return "gradient kernel (label) failed";
        case RNNT_STATUS_COSTS_FAILED: return "cost kernel failed";
        case RNNT_STATUS_INVALID_ARGUMENT: return "invalid argument";
        case RNNT_STATUS_WORKSPACE_TOO_SMALL: return "workspace too small";
        case RNNT_STATUS_GATHER_FAILED: return "gather kernel failed";
        default: return "unknown status";
    }
}

void rnnt_b200_set_lse_mode(int mode) {
    if (mode < RNNT_LSE_AUTO || mode > RNNT_LSE_FAST) mode = RNNT_LSE_AUTO;
    g_lse_mode.store(mode, std::memory_order_relaxed);
}
int rnnt_b200_get_lse_mode(void) { return default_lse_mode(); }

uint64_t rnnt_b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
void rnnt_b200_debug_guard_poison(int n, float delta) {
    g_poison_delta.store(delta, std::memory_order_relaxed);
    g_poison_n.store(n, std::memory_order_relaxed);
}
int rnnt_b200_debug_lse_selfcheck(void *stream, unsigned long long *mismatches) {
    if (!mismatches) return RNNT_STATUS_INVALID_ARGUMENT;
    rnnt::k_lse_selfcheck<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(mismatches);
    return cudaGetLastError() == cudaSuccess ? RNNT_STATUS_SUCCESS : RNNT_STATUS_WARP_FAILED;
}
void rnnt_b200_debug_fused_trace(void *buf) { rnnt::set_fused_trace(static_cast<long long *>(buf)); }

size_t rnnt_b200_workspace_bytes(int64_t cells, int N) { return carve(nullptr, cells, N).bytes; }

int rnnt_b200_loss_dense(void *stream, void *workspace, size_t workspace_bytes, const float *log_probs,
                         const int *labels, const int *xn, const int *yn, float *costs, float *grads,
                         const float *grad_scale, int N, int T, int U, int V, int blank, float fastemit_lambda,
                         int lse_mode) {
    return rnnt_b200_loss_dense_reduced(stream, workspace, workspace_bytes, log_probs, labels, xn, yn, costs, grads,
                                        grad_scale, nullptr, nullptr, N, T, U, V, blank, fastemit_lambda, lse_mode);
}

int rnnt_b200_loss_dense_reduced(void *stream, void *workspace, size_t workspace_bytes, const float *log_probs,
                                 const int *labels, const int *xn, const int *yn, float *costs, float *grads,
                                 const float *grad_scale, float *loss_sum, unsigned int *sync_counter, int N, int T,
                                 int U, int V, int blank, float fastemit_lambda, int lse_mode) {
    return loss_dense_any(stream, workspace, workspace_bytes, log_probs, labels, xn, yn, costs, grads, grad_scale,
                          loss_sum, sync_counter, N, T, U, V, blank, fastemit_lambda, lse_mode, 0);
}

int rnnt_b200_loss_dense_bf16(void *stream, void *workspace, size_t workspace_bytes, const void *log_probs_bf16,
                              const int *labels, const int *xn, const int *yn, float *costs, void *grads_bf16,
                              const float *grad_scale, float *loss_sum, unsigned int *sync_counter, int N, int T,
                              int U, int V, int blank, float fastemit_lambda, int lse_mode) {
    if ((reinterpret_cast<uintptr_t>(log_probs_bf16) | reinterpret_cast<uintptr_t>(grads_bf16)) & 1u)
        return RNNT_STATUS_INVALID_ARGUMENT;
    return loss_dense_any(stream, workspace, workspace_bytes, log_probs_bf16, labels, xn, yn, costs, grads_bf16,
                          grad_scale, loss_sum, sync_counter, N, T, U, V, blank, fastemit_lambda, lse_mode, 1);
}

int rnnt_b200_rescale(void *stream, void *grads, const float *grad_out, int grad_out_stride, const float *applied,
                      int N, int64_t elems_per_sample, int elem_bytes) {
    if (N < 0 || elems_per_sample < 0 || grad_out_stride < 0 || grad_out_stride > 1 || !grads || !grad_out ||
        (elem_bytes != 4 && elem_bytes != 2))
        return RNNT_STATUS_INVALID_ARGUMENT;
    RNNT_TRY(launch_rescale((cudaStream_t)stream, grads, grad_out, grad_out_stride, applied, N, elems_per_sample,
                            elem_bytes == 2),
             RNNT_STATUS_GRADS_BLANK_FAILED);
    return RNNT_STATUS_SUCCESS;
}

int rnnt_b200_loss_pairs(void *stream, void *workspace, size_t workspace_bytes, const float *pairs, const int *xn,
                         const int *yn, float *costs, float *pair_grads, int N, int T, int U,
                         float fastemit_lambda, int lse_mode) {
    if (!dense_call_ok(N, T, U, 2, 0, pair_grads) || !f2_aligned(pairs)) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    LossJob j = {};
    j.lp = pairs; j.xn = xn; j.yn = yn; j.pairs_in = 1;
    j.N = N; j.T = T; j.U = U; j.V = 2; j.blank = 0; j.cells = (int64_t)N * T * U;
    j.kind = resolve_kind(lse_mode, false); j.guard = 1; j.lam = fastemit_lambda;
    j.costs = costs; j.pair_grads = reinterpret_cast<float2 *>(pair_grads);
    return dispatch((cudaStream_t)stream, j, workspace, workspace_bytes);
}

int rnnt_b200_gather_forward(void *stream, void *workspace, size_t workspace_bytes, const float *log_probs,
                             const int *labels, const int *xn, const int *yn, float *costs, float *pair_grads,
                             int N, int T, int U, int V, int blank, float fastemit_lambda, int lse_mode) {
    if (!dense_call_ok(N, T, U, V, blank, pair_grads)) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    LossJob j = {};
    j.lp = log_probs; j.labels = labels; j.xn = xn; j.yn = yn;
    j.N = N; j.T = T; j.U = U; j.V = V; j.blank = blank; j.cells = (int64_t)N * T * U;
    j.kind = resolve_kind(lse_mode, false); j.guard = 1; j.lam = fastemit_lambda;
    j.costs = costs; j.pair_grads = reinterpret_cast<float2 *>(pair_grads);
    return dispatch((cudaStream_t)stream, j, workspace, workspace_bytes);
}

int rnnt_b200_logits_forward(void *stream, void *workspace, size_t workspace_bytes, const float *logits,
                              const int *labels, const int *xn, const int *yn, float *costs, float *lse,
                              float *pair_grads, int N, int T, int U, int V, int blank, float fastemit_lambda,
                              int lse_mode) {
    return logits_forward_any(stream, workspace, workspace_bytes, logits, labels, xn, yn, costs, lse, pair_grads, N, T,
                              U, V, blank, fastemit_lambda, lse_mode, 0);
}

int rnnt_b200_logits_forward_bf16(void *stream, void *workspace, size_t workspace_bytes, const void *logits_bf16,
                                  const int *labels, const int *xn, const int *yn, float *costs, float *lse,
                                  float *pair_grads, int N, int T, int U, int V, int blank, float fastemit_lambda,
                                  int lse_mode) {
    if (!bf16_aligned(logits_bf16)) return RNNT_STATUS_INVALID_ARGUMENT;
    return logits_forward_any(stream, workspace, workspace_bytes, logits_bf16, labels, xn, yn, costs, lse, pair_grads,
                              N, T, U, V, blank, fastemit_lambda, lse_mode, 1);
}

int rnnt_b200_logits_backward(void *stream, const float *logits, const float *lse, const float *pair_grads,
                              const int *labels, const float *grad_out, float *out, int N, int T, int U, int V,
                              int blank) {
    return logits_backward_any(stream, logits, lse, pair_grads, labels, grad_out, out, N, T, U, V, blank, 0);
}

int rnnt_b200_logits_backward_bf16(void *stream, const void *logits_bf16, const float *lse, const float *pair_grads,
                                   const int *labels, const float *grad_out, void *out_bf16, int N, int T, int U,
                                   int V, int blank) {
    if (!bf16_aligned(logits_bf16) || !bf16_aligned(out_bf16)) return RNNT_STATUS_INVALID_ARGUMENT;
    return logits_backward_any(stream, logits_bf16, lse, pair_grads, labels, grad_out, out_bf16, N, T, U, V, blank, 1);
}

int rnnt_b200_gather_backward(void *stream, const float *pair_grads, const int *labels, const float *grad_out,
                              float *out, int N, int T, int U, int V, int blank, int accumulate, const int *yn) {
    if (!dense_call_ok(N, T, U, V, blank, pair_grads)) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    Problem p = {nullptr, yn, nullptr, nullptr, N, T, U, 0};     // yn (optional): which labels are real
    ExpandSrc src = {};
    src.pg = reinterpret_cast<const float2 *>(pair_grads);
    src.scale = grad_out;
    src.labels = labels;
    src.label_adds = accumulate ? 1 : 0;
    RNNT_TRY(launch_expand((cudaStream_t)stream, p, src, out, (int64_t)N * T * U, V, blank),
             RNNT_STATUS_GRADS_BLANK_FAILED);
    return RNNT_STATUS_SUCCESS;
}

int rnnt_b200_compact_forward(void *stream, void *workspace, size_t workspace_bytes, const float *xs, const int *ys,
                              const int *xn, const int *yn, float *costs, float *pair_grads, int64_t *loc,
                              int *totals, int64_t STU, int N, int V, int blank, float fastemit_lambda,
                              int lse_mode, int max_T, int max_U) {
    if (N < 0 || STU < 0 || V < 1 || V >= (1 << 22) || blank < 0 || blank >= V || !f2_aligned(pair_grads))
        return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    cudaStream_t s = (cudaStream_t)stream;
    const Workspace w = carve(workspace, STU, N);
    if (!workspace || workspace_bytes < w.bytes) return RNNT_STATUS_WORKSPACE_TOO_SMALL;
    RNNT_TRY(launch_prefix(s, xn, yn, N, w.mem_pref, w.lab_pref, totals ? totals : w.totals), RNNT_STATUS_GATHER_FAILED);
    // the fused kernel (when max_T, max_U > 0 and it fits) also writes loc; no mismatch guard in the compact
    // reference (core_compact.cu:347-358)
    LossJob j = {};
    j.lp = xs; j.labels = ys; j.xn = xn; j.yn = yn; j.mem_pref = w.mem_pref; j.lab_pref = w.lab_pref;
    j.N = N; j.T = max_T; j.U = max_U; j.V = V; j.blank = blank; j.cells = STU;
    j.kind = resolve_kind(lse_mode, true); j.guard = 0; j.lam = fastemit_lambda;
    j.costs = costs; j.pair_grads = reinterpret_cast<float2 *>(pair_grads); j.loc = loc;
    return dispatch(s, j, workspace, workspace_bytes);
}

int rnnt_b200_compact_totals(void *stream, const int *xn, const int *yn, int N, int64_t *scratch, int *totals) {
    if (N <= 0 || !scratch || !totals) return RNNT_STATUS_INVALID_ARGUMENT;
    RNNT_TRY(launch_prefix((cudaStream_t)stream, xn, yn, N, scratch, scratch + N, totals), RNNT_STATUS_GATHER_FAILED);
    return RNNT_STATUS_SUCCESS;
}

int rnnt_b200_joint_pack(void *stream, const float *f, const float *g, const int *lf, const int *lg, int64_t *scratch,
                         int *totals, float *x, int N, int T, int U1, int H, int64_t stu_hint) {
    if (N < 0 || T < 1 || U1 < 1 || H < 1 || !scratch) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    cudaStream_t s = (cudaStream_t)stream;
    // mem_pref[n] = first packed row of lattice n: the same device prefix sums as the compact loss (lf = xn, lg = yn)
    RNNT_TRY(launch_prefix(s, lf, lg, N, scratch, scratch + N, totals), RNNT_STATUS_GATHER_FAILED);
    if (x) RNNT_TRY(launch_joint_pack(s, f, g, lf, lg, scratch, x, N, T, U1, H, stu_hint), RNNT_STATUS_GATHER_FAILED);
    return RNNT_STATUS_SUCCESS;
}

int rnnt_b200_joint_pack_backward(void *stream, const float *dx, const int *lf, const int *lg, const int64_t *mem_pref,
                                  float *df, float *dg, int N, int T, int U1, int H) {
    if (N < 0 || T < 1 || U1 < 1 || H < 1 || !mem_pref || !dx) return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    RNNT_TRY(launch_joint_grads((cudaStream_t)stream, dx, lf, lg, mem_pref, df, dg, N, T, U1, H),
             RNNT_STATUS_GRADS_BLANK_FAILED);
    return RNNT_STATUS_SUCCESS;
}

int rnnt_b200_compact_backward(void *stream, const float *grad_cost, const float *pair_grads, const int64_t *loc,
                               const int *cum_lens, float *out, int64_t STU, int N, int V, int blank) {
    if (N < 0 || STU < 0 || V < 1 || V >= (1 << 22) || blank < 0 || blank >= V || !f2_aligned(pair_grads))
        return RNNT_STATUS_INVALID_ARGUMENT;
    if (N == 0 || STU == 0) return RNNT_STATUS_SUCCESS;
    Problem p = {nullptr, nullptr, nullptr, nullptr, N, 0, 0, 1};
    ExpandSrc src = {};
    src.pg = reinterpret_cast<const float2 *>(pair_grads);
    src.scale = grad_cost;
    src.loc = loc;
    src.cum_lens = cum_lens;
    RNNT_TRY(launch_expand((cudaStream_t)stream, p, src, out, STU, V, blank), RNNT_STATUS_GRADS_BLANK_FAILED);
    return RNNT_STATUS_SUCCESS;
}

// ------------------------------------------------------------------------------------------
// (B) the reference's C ABI.  Scratch that the reference signatures have no room for comes
// from the stream-ordered allocator (cudaMallocAsync / cudaFreeAsync on the same stream).
// ------------------------------------------------------------------------------------------
static void compat_die(const char *what, int status) {
    // the reference's CHECK_KERNEL_STAT prints and exit(-1)s (core.h:7-14)
    fprintf(stderr, "%s error: %s\n", what, rnnt_b200_status_string(status));
    exit(-1);
}

// The `parts` of a workspace in one cudaMallocAsync block on `s`, or null; the caller frees it with cudaFreeAsync on `s`.
static void *compat_scratch(cudaStream_t s, int64_t cells, int N, unsigned parts, Workspace *w) {
    void *block = nullptr;
    if (cudaMallocAsync(&block, carve(nullptr, cells, N, parts).bytes, s) != cudaSuccess) return nullptr;
    *w = carve(block, cells, N, parts);
    return block;
}

// The shims return alphas and betas, so they run the general sequence (never the fused kernel) with the caller's.
int run_warp_rnnt(void *stream, unsigned int *counts, float *alphas, float *betas, const int *labels,
                  const float *log_probs, float *grads, float *costs, const int *xn, const int *yn, int N, int T,
                  int U, int V, int blank, float fastemit_lambda) {
    (void)counts;
    if (!dense_call_ok(N, T, U, V, blank)) return RNNT_STATUS_WARP_FAILED;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    cudaStream_t s = (cudaStream_t)stream;
    LossJob j = {};
    j.lp = log_probs; j.labels = labels; j.xn = xn; j.yn = yn;
    j.N = N; j.T = T; j.U = U; j.V = V; j.blank = blank; j.cells = (int64_t)N * T * U;
    j.kind = resolve_kind(RNNT_LSE_AUTO, false); j.guard = 1; j.lam = fastemit_lambda;
    j.costs = costs; j.grads = grads;
    Workspace w;
    void *tmp = compat_scratch(s, j.cells, N, kWsPairs | kWsLL | kWsBad, &w);
    if (!tmp) return RNNT_STATUS_WARP_FAILED;
    w.alphas = alphas; w.betas = betas;
    const int status = run_general(s, j, w);
    cudaFreeAsync(tmp, s);
    return status == RNNT_STATUS_GATHER_FAILED ? RNNT_STATUS_WARP_FAILED : status;   // the reference's statuses have no gather
}

int run_warp_rnnt_gather(void *stream, unsigned int *counts, float *alphas, float *betas, const float *log_probs,
                         float *grads, float *costs, const int *xn, const int *yn, int N, int T, int U,
                         float fastemit_lambda) {
    (void)counts;
    if (!dense_call_ok(N, T, U, 2, 0)) return RNNT_STATUS_WARP_FAILED;
    if (N == 0) return RNNT_STATUS_SUCCESS;
    cudaStream_t s = (cudaStream_t)stream;
    LossJob j = {};
    j.lp = log_probs; j.xn = xn; j.yn = yn; j.pairs_in = 1;
    j.N = N; j.T = T; j.U = U; j.V = 2; j.blank = 0; j.cells = (int64_t)N * T * U;
    j.kind = resolve_kind(RNNT_LSE_AUTO, false); j.guard = 1; j.lam = fastemit_lambda;
    j.costs = costs; j.pair_grads = reinterpret_cast<float2 *>(grads);
    Workspace w;
    void *tmp = compat_scratch(s, j.cells, N, kWsLL | kWsBad, &w);
    if (!tmp) return RNNT_STATUS_WARP_FAILED;
    w.alphas = alphas; w.betas = betas;
    const int status = run_general(s, j, w);
    cudaFreeAsync(tmp, s);
    return status;
}

// compact variants run on the legacy default stream like the reference (core.h:41-60 has no stream)
void run_gather_for_compact(const float *xs, const int *ys, const unsigned int *xn, const unsigned int *yn,
                            float *gather_xs, long *loc, const unsigned int *memPref, const unsigned int *labelPref,
                            unsigned int N, unsigned int T, unsigned int U, unsigned int V, unsigned int blank) {
    (void)memPref; (void)labelPref;   // recomputed on device in 64-bit
    if (N == 0) return;
    cudaStream_t s = 0;
    Workspace w;
    void *tmp = compat_scratch(s, 0, (int)N, kWsPrefix, &w);
    if (!tmp) compat_die("rnnt loss gather for compact", RNNT_STATUS_GATHER_FAILED);
    const int *xi = (const int *)xn, *yi = (const int *)yn;
    bool ok = launch_prefix(s, xi, yi, (int)N, w.mem_pref, w.lab_pref, w.totals) == cudaSuccess;
    Problem p = {xi, yi, w.mem_pref, w.lab_pref, (int)N, 0, 0, 1};
    ok = ok && launch_gather(s, p, xs, ys, (int)V, (int)blank, reinterpret_cast<float2 *>(gather_xs),
                             reinterpret_cast<int64_t *>(loc), (int64_t)N * T * U) == cudaSuccess;
    cudaFreeAsync(tmp, s);
    if (!ok) compat_die("rnnt loss gather for compact", RNNT_STATUS_GATHER_FAILED);
}

void run_warp_rnnt_compact(unsigned int *counts, float *alphas, float *betas, const float *log_probs, float *grads,
                           float *costs, const unsigned int *xn, const unsigned int *yn, const unsigned int *memPref,
                           const unsigned int *labelPref, unsigned int N, unsigned int T, unsigned int U,
                           float fastemit_lambda, bool required_grad) {
    (void)counts; (void)memPref; (void)labelPref;
    if (N == 0) return;
    cudaStream_t s = 0;
    Workspace w;
    void *tmp = compat_scratch(s, 0, (int)N, kWsLL | kWsPrefix, &w);
    if (!tmp) compat_die("rnnt loss compact betas", RNNT_STATUS_WARP_FAILED);
    w.alphas = alphas; w.betas = betas;
    LossJob j = {};
    j.lp = log_probs; j.xn = (const int *)xn; j.yn = (const int *)yn; j.mem_pref = w.mem_pref; j.lab_pref = w.lab_pref;
    j.pairs_in = 1;
    j.N = (int)N; j.T = (int)T; j.U = (int)U; j.V = 2; j.blank = 0; j.cells = (int64_t)N * T * U;
    j.kind = resolve_kind(RNNT_LSE_AUTO, true); j.guard = 0; j.lam = fastemit_lambda;
    j.costs = costs; j.pair_grads = required_grad ? reinterpret_cast<float2 *>(grads) : nullptr;
    const bool ok = launch_prefix(s, j.xn, j.yn, j.N, w.mem_pref, w.lab_pref, w.totals) == cudaSuccess &&
                    run_general(s, j, w) == RNNT_STATUS_SUCCESS;
    cudaFreeAsync(tmp, s);
    if (!ok) compat_die("rnnt loss compact", RNNT_STATUS_WARP_FAILED);
}

void run_scatter_grad_for_compact(const float *grad_cost, const float *gather_grad, const long *loc,
                                  const int *cum_lens, float *scatter_grad, unsigned int STU, unsigned int N,
                                  unsigned int V, unsigned int blank) {
    const int st = rnnt_b200_compact_backward(nullptr, grad_cost, gather_grad, reinterpret_cast<const int64_t *>(loc),
                                              cum_lens, scatter_grad, (int64_t)STU, (int)N, (int)V, (int)blank);
    if (st != RNNT_STATUS_SUCCESS) compat_die("rnnt loss filling scatter grad", st);
}

}  // extern "C"
