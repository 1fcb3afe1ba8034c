// logits.cu -- the step BEFORE the reference's path, fused in: the loss straight from un-normalised joint-network
// logits (SURVEY.md 8(f)1).
//
// The reference requires log-softmaxed input (/root/reference/README.md:59) and its benchmark times F.log_softmax with
// the loss (pytorch_binding/benchmark.py:65): log_softmax forward (read + write of (N,T,U,V)), the loss (read + dense
// gradient write, + mul_) and log_softmax backward (two reads + one write) -- seven dense passes.  Here:
//
//   k_lse_pairs      one read of the logits: per cell the normaliser lse = max + log(sum exp(x - max)) and the two
//                    normalised log-probs the recurrence needs, pairs[cell] = (x[blank] - lse, x[label] - lse)
//   (wavefront)      the existing kernels on the (cells,2) layout -> (cells,2) gradients w.r.t. the log-probs
//   k_expand_logits  one read of the logits + one write: the gradient w.r.t. the LOGITS,
//                        g[v] = [v == blank] gb + [v == label] gl - exp(x[v] - lse) (gb + gl),
//                    i.e. log_softmax's backward applied to the loss' (blank, label) gradient on the fly, times grad_out[n]
//
// three dense passes in total.  A label equal to blank: the two gradients add (what autograd through torch.gather /
// log_softmax does).  Padded cells carry zero pair gradients and get exact zeros.  Logits (and the logit gradient) are
// float32 or bfloat16; lse, pairs and the pair gradients are float32 either way.
#include "common.cuh"
#include "kernels.cuh"

namespace rnnt {

constexpr int kLogitThreads = 256;

// Element types IO: float, or bf16 (bf16 logits in, bf16 logit gradient out).  Every bf16 value is converted exactly to
// float on load and all arithmetic is the f32 path's, in the f32 path's order: both instantiations of a kernel give the
// same lse / pairs bits on the same values, and the bf16 gradient is the f32 one rounded once (RNE) on the store.

// the q-th 4-element vector of a 4-element-aligned row: one 16-byte (f32) or 8-byte (bf16) load
__device__ __forceinline__ float4 ld4(const float *row, int q) { return __ldg(reinterpret_cast<const float4 *>(row) + q); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16 *row, int q) {
    const uint2 t = __ldg(reinterpret_cast<const uint2 *>(row) + q);
    float4 a;
    bf16x2_to_float(t.x, a.x, a.y);
    bf16x2_to_float(t.y, a.z, a.w);
    return a;
}

// iterations of the vec4 loop whose loads are issued ahead of their math: a bf16 lane loads 8 bytes per iteration,
// half of what an f32 lane does, so it keeps four iterations in flight; f32 keeps its one 16-byte load per iteration.
template <typename IO> constexpr int kLseIlp = sizeof(IO) == 2 ? 4 : 1;

// SUB lanes cooperate on one cell (SUB in {1, 8, 32}); online max / sum so the row is read once.  VEC4: rows are whole
// 4-element vectors at 4-element-aligned addresses -> the SUB lanes stride over vectors (V = 28: 7 of 8 lanes load one
// vector each, a warp reads 4 consecutive rows = 448 contiguous bytes in f32).  Lane `sub` sums vectors sub, sub + SUB,
// ... in that order for either element type.
template <typename IO, int SUB, bool VEC4>
__global__ void __launch_bounds__(kLogitThreads)
k_lse_pairs(const IO *__restrict__ x, const int *__restrict__ labels, int64_t cells, int V, int blank, int U,
            FastDiv divU, FastDiv divTU, float2 *__restrict__ pairs, float *__restrict__ lse_out) {
    const int sub = threadIdx.x % SUB;
    const int64_t per_block = kLogitThreads / SUB;
    for (int64_t base = (int64_t)blockIdx.x * per_block; base < cells; base += (int64_t)gridDim.x * per_block) {   // block-uniform trip count
        const int64_t cell = min(base + threadIdx.x / SUB, cells - 1);          // surplus groups redo the last cell (shuffles need every lane)
        const IO *row = x + cell * V;
        float m = -INFINITY, s = 0.0f;
        auto add = [&](float a) {
            if (a > m) { s = s * expf(m - a); m = a; }        // (m == -inf: s is 0, exp(-inf) = 0)
            s += expf(a - m);
        };
        if (VEC4 && (V >> 2) <= SUB) {
            // the whole row is one vector per lane: max first (shuffles only), then ONE exp per element -- the online
            // merge below would spend two more exp per lane and shuffle round
            const bool has = sub < (V >> 2);
            const float4 a = has ? ld4(row, sub) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
            m = fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w));
#pragma unroll
            for (int o = SUB / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            s = has ? (expf(a.x - m) + expf(a.y - m)) + (expf(a.z - m) + expf(a.w - m)) : 0.0f;
#pragma unroll
            for (int o = SUB / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        } else if (VEC4) {
            auto add4 = [&](const float4 a) {
                const float mx = fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w));
                if (mx > m) { s = s * expf(m - mx); m = mx; }
                s += (expf(a.x - m) + expf(a.y - m)) + (expf(a.z - m) + expf(a.w - m));
            };
            constexpr int ILP = kLseIlp<IO>;
            int q0 = sub;
            if constexpr (ILP > 1) {
                for (; q0 + (ILP - 1) * SUB < (V >> 2); q0 += ILP * SUB) {
                    float4 a[ILP];
#pragma unroll
                    for (int k = 0; k < ILP; ++k) a[k] = ld4(row, q0 + k * SUB);
#pragma unroll
                    for (int k = 0; k < ILP; ++k) add4(a[k]);
                }
            }
            for (int q = q0; q < (V >> 2); q += SUB) add4(ld4(row, q));
        } else if (SUB == 1) {
            // short unaligned rows: one thread per cell; neighbouring threads' rows share cache lines, so the pass over
            // v is served from L1 after the first touch
            for (int v = 0; v < V; ++v) m = fmaxf(m, io_load<IO>(row + v));
            for (int v = 0; v < V; ++v) s += expf(io_load<IO>(row + v) - m);
        } else {
            for (int v = sub; v < V; v += SUB) add(io_load<IO>(row + v));
        }
        if (SUB > 1 && !(VEC4 && (V >> 2) <= SUB)) {
#pragma unroll
            for (int o = SUB / 2; o > 0; o >>= 1) {
                const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
                const float mm = fmaxf(m, m2);
                s = (m == mm ? s : s * expf(m - mm)) + (m2 == mm ? s2 : s2 * expf(m2 - mm));
                m = mm;
            }
        }
        if (sub == 0) {
            const float l = m + logf(s);
            uint32_t n, rem, t, u;
            divTU.divmod((uint32_t)cell, n, rem);
            divU.divmod(rem, t, u);
            const int lab = ((int)u < U - 1) ? labels[(int64_t)n * (U - 1) + u] : blank;
            pairs[cell] = make_float2(io_load<IO>(row + blank) - l, io_load<IO>(row + lab) - l);
            lse_out[cell] = l;
        }
    }
}

// flat stream of the (cells, V) output in vectors of VEC elements (the widest of at most 16 bytes that divides V and
// the alignment of both pointers): a vector never straddles a row, so one (gb, gl, lse, label) fetch serves it.  The
// arithmetic is per element, so VEC does not change the values.
template <typename IO, int VEC>
__global__ void __launch_bounds__(kLogitThreads)
k_expand_logits(const IO *__restrict__ x, const float *__restrict__ lse, const float2 *__restrict__ pg,
                const int *__restrict__ labels, const float *__restrict__ grad_out, IO *__restrict__ out,
                int64_t cells, int V, int blank, int U, FastDiv divU, FastDiv divTU, int64_t stride_rows,
                int stride_v) {
    const int64_t total = cells * (int64_t)V;
    int64_t f = ((int64_t)blockIdx.x * kLogitThreads + threadIdx.x) * VEC;
    if (f >= total) return;
    // (row, v0) of the thread's vector: one 64-bit division here, then a running cursor (the grid stride is
    // stride_rows whole rows + stride_v elements)
    int64_t row = f / V;
    int v0 = (int)(f - row * V);
    const int64_t stride = stride_rows * V + stride_v;
    for (; f < total; f += stride, row += stride_rows, v0 += stride_v) {
        if (v0 >= V) { v0 -= V; ++row; }
        const float2 q = pg[row];
        float e[VEC];
        if (q.x == 0.0f && q.y == 0.0f) {
#pragma unroll
            for (int k = 0; k < VEC; ++k) e[k] = 0.0f;            // padding (or a dead cell): exact zeros
        } else {
            uint32_t n, rem, t, u;
            divTU.divmod((uint32_t)row, n, rem);
            divU.divmod(rem, t, u);
            const int lab = ((int)u < U - 1) ? labels[(int64_t)n * (U - 1) + u] : -1;
            const float sc = grad_out ? grad_out[n] : 1.0f;
            const float l = lse[row], tot = q.x + q.y;
            float xv[VEC];
            ld_vec<VEC>(x + f, xv);
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                float gsel = (v0 + k == blank) ? q.x : 0.0f;
                if (v0 + k == lab) gsel += q.y;
                e[k] = (gsel - expf(xv[k] - l) * tot) * sc;
            }
        }
        st_cs_vec<VEC>(out + f, e);
    }
}

template <typename IO>
static void lse_pairs_io(cudaStream_t s, int grid, bool vec4, int sub, const IO *x, const int *labels, int64_t cells,
                         int V, int blank, int U, FastDiv divU, FastDiv divTU, float2 *pairs, float *lse) {
#define RNNT_LSE_LAUNCH(SUB, VEC) k_lse_pairs<IO, SUB, VEC><<<grid, kLogitThreads, 0, s>>>(x, labels, cells, V, blank, U, divU, divTU, pairs, lse)
    if (vec4) { if (sub == 8) RNNT_LSE_LAUNCH(8, true); else RNNT_LSE_LAUNCH(32, true); }
    else if (sub == 1) RNNT_LSE_LAUNCH(1, false);
    else if (sub == 8) RNNT_LSE_LAUNCH(8, false);
    else RNNT_LSE_LAUNCH(32, false);
#undef RNNT_LSE_LAUNCH
}

cudaError_t launch_lse_pairs(cudaStream_t s, const void *x, const int *labels, int N, int T, int U, int V, int blank,
                             float2 *pairs, float *lse, int io_bf16) {
    const int64_t cells = (int64_t)N * T * U;
    if (cells <= 0) return cudaSuccess;
    const FastDiv divU((uint32_t)U), divTU((uint32_t)(T * U));
    const int sms = sm_count(current_device());
    // variant chosen in elements, the same for both element types (it fixes which lane sums which elements)
    const uintptr_t vec_bytes = 4 * (io_bf16 ? sizeof(__nv_bfloat16) : sizeof(float));
    const bool vec4 = (V % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & (vec_bytes - 1)) == 0);
    const int sub = vec4 ? (V <= 32 ? 8 : 32) : (V <= 12 ? 1 : (V <= 512 ? 8 : 32));
    const int64_t per_block = kLogitThreads / sub;
    const int grid = (int)min((cells + per_block - 1) / per_block, (int64_t)sms * 16);
    if (io_bf16)
        lse_pairs_io(s, grid, vec4, sub, static_cast<const __nv_bfloat16 *>(x), labels, cells, V, blank, U, divU, divTU, pairs, lse);
    else
        lse_pairs_io(s, grid, vec4, sub, static_cast<const float *>(x), labels, cells, V, blank, U, divU, divTU, pairs, lse);
    count_launch();
    return cudaGetLastError();
}

template <typename IO>
static void expand_logits_io(cudaStream_t s, int grid, int vec, const IO *x, const float *lse, const float2 *pg,
                             const int *labels, const float *grad_out, IO *out, int64_t cells, int V, int blank, int U,
                             FastDiv divU, FastDiv divTU, int64_t srows, int sv) {
#define RNNT_EXPAND_LAUNCH(VEC) k_expand_logits<IO, VEC><<<grid, kLogitThreads, 0, s>>>(x, lse, pg, labels, grad_out, out, cells, V, blank, U, divU, divTU, srows, sv)
    if constexpr (sizeof(IO) == 2) { if (vec == 8) { RNNT_EXPAND_LAUNCH(8); return; } }
    if (vec == 4) RNNT_EXPAND_LAUNCH(4);
    else if (vec == 2) RNNT_EXPAND_LAUNCH(2);
    else RNNT_EXPAND_LAUNCH(1);
#undef RNNT_EXPAND_LAUNCH
}

cudaError_t launch_expand_logits(cudaStream_t s, const void *x, const float *lse, const float2 *pg, const int *labels,
                                 const float *grad_out, void *out, int N, int T, int U, int V, int blank, int io_bf16) {
    const int64_t cells = (int64_t)N * T * U;
    if (cells <= 0) return cudaSuccess;
    const FastDiv divU((uint32_t)U), divTU((uint32_t)(T * U));
    const int sms = sm_count(current_device());
    // the widest vector of at most 16 bytes that divides V and to which both pointers are aligned
    const size_t esz = io_bf16 ? sizeof(__nv_bfloat16) : sizeof(float);
    const uintptr_t addr = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out);
    int vec = (int)(16 / esz);
    while (vec > 1 && (V % vec != 0 || (addr & (vec * esz - 1)) != 0)) vec >>= 1;
    const int64_t total = cells * (int64_t)V / vec;
    const int grid = (int)min((total + kLogitThreads - 1) / kLogitThreads, (int64_t)sms * 32);
    const int64_t stride = (int64_t)grid * kLogitThreads * vec;
    const int64_t srows = stride / V;
    const int sv = (int)(stride - srows * V);
    if (io_bf16)
        expand_logits_io(s, grid, vec, static_cast<const __nv_bfloat16 *>(x), lse, pg, labels, grad_out,
                         static_cast<__nv_bfloat16 *>(out), cells, V, blank, U, divU, divTU, srows, sv);
    else
        expand_logits_io(s, grid, vec, static_cast<const float *>(x), lse, pg, labels, grad_out, static_cast<float *>(out),
                         cells, V, blank, U, divU, divTU, srows, sv);
    count_launch();
    return cudaGetLastError();
}

}  // namespace rnnt
