// expand.cu -- dense gradient emit: every element of the (cells, V) output is written exactly once
// (zeros + the <= 2 non-zeros of each row), with 128-bit streaming stores.
//
// What it replaces in the reference (/root/reference):
//   at::zeros_like(xs) dense memset                 pytorch_binding/binding.cpp:58
//   kernel_grads_blank / kernel_grads_label         core.cu:260-332  (4-byte stores at stride U*V)
//   RNNTLoss.backward grads.mul_(grad_output)       pytorch_binding/warp_rnnt/__init__.py:21-24
//   torch GatherBackward (zeros + scatter_add_)     __init__.py:118-128 (python-level gather=True)
//   torch::zeros({STU,V}) + kernel_fill_scatter_grad   binding.cpp:239, core_compact.cu:456-484
//
// The output is treated as one flat float stream cut into chunks of R consecutive rows; a CTA
// first stages the R rows' (blank grad, label grad, label id) in shared memory (coalesced reads
// of alpha/beta/pairs or of the (cells,2) pair grads), then all its threads sweep the chunk with
// float4 stores, composing each vector from the staged values.  HBM traffic = 4*V bytes written
// + <= 24 bytes read per row; no pre-zeroing pass, no second pass.
#include "common.cuh"
#include "kernels.cuh"

namespace rnnt {

constexpr int kExpandThreads = 256;
constexpr int kExpandMaxRows = 256;

// same arithmetic as k_grads_pairs (core.cu:284-294, :319-331)
__device__ __forceinline__ float2 cell_grads_ab(const Lattice &L, const ExpandSrc &src, int t, int u, float b00) {
    const int64_t c = L.base + (int64_t)t * L.stride + u;
    const float2 w = src.pairs[c];
    const float al = src.alphas[c];
    float gb = 0.0f, gl = 0.0f;
    const bool last_t = (t == L.Tn - 1), last_u = (u == L.Un - 1);
    if (!(last_t && !last_u)) {
        float a = al;
        if (!last_t) a += src.betas[c + L.stride];
        a = expf(a + w.x - b00);
        gb = -a;
    }
    if (!last_u) {
        float a = al + src.betas[c + 1];
        a = expf(a + w.y - b00);
        a = (float)((1.0 + (double)src.fastemit_lambda) * (double)a);
        gl = -a;
    }
    return make_float2(gb, gl);
}

// (blank grad, label grad, label id or -1) of output row c -- the two non-zeros every emit flavour places
template <int MODE>
__device__ __forceinline__ void stage_row(const Problem &p, const ExpandSrc &src, int64_t c, int blank,
                                          const FastDiv &divU, const FastDiv &divTU, float2 &g, int &lab) {
    g = make_float2(0.0f, 0.0f);
    lab = -1;
    if (MODE == 2) {
        // which sample? binary search in the inclusive cumsum (core_compact.cu:465-477)
        int lo = 0, hi = p.N - 1;
        while (lo <= hi) {
            const int mid = lo + (hi - lo) / 2;
            if (c >= (int64_t)src.cum_lens[mid]) lo = mid + 1; else hi = mid - 1;
        }
        const int n = min(lo, p.N - 1);
        const float sc = src.scale ? src.scale[n] : 1.0f;
        const float2 q = src.pg[c];
        g = make_float2(q.x * sc, q.y * sc);
        const int64_t l = src.loc[c];
        lab = (l != (int64_t)blank) ? (int)l : -1;
    } else {
        uint32_t n, rem, t, u;
        divTU.divmod((uint32_t)c, n, rem);
        divU.divmod(rem, t, u);
        if (MODE == 1) {
            const float sc = src.scale ? src.scale[n] : 1.0f;
            const float2 q = src.pg[c];
            g = make_float2(q.x * sc, q.y * sc);
            // label transition out of (t,u) exists iff u < yn[n]; without lengths (p.yn == null) every u < U-1 is taken
            // and the sweep falls back to "a zero label gradient means none" in override mode
            if ((int)u < (p.yn ? min(p.yn[n], p.U - 1) : p.U - 1)) lab = src.labels[(int64_t)n * (p.U - 1) + u];
        } else {
            const Lattice L = get_lattice(p, (int)n);
            const bool live = L.ok && !(src.bad && src.bad[n]);
            if (live && (int)t < L.Tn && (int)u < L.Un) {
                g = cell_grads_ab(L, src, (int)t, (int)u, src.betas[L.base]);
                if (src.scale) { const float sc = src.scale[n]; g.x *= sc; g.y *= sc; }
                if ((int)u < L.Un - 1) lab = src.labels[L.lab_base + u];
            }
        }
    }
}

__device__ __forceinline__ void st_one(float *p, float v) { st_cs(p, v); }
__device__ __forceinline__ void st_one(__nv_bfloat16 *p, float v) { *p = __float2bfloat16_rn(v); }

// MODE 0: dense layout, source = alpha/beta/pairs (forward)            label overrides blank
// MODE 1: dense layout, source = pair grads (gather=True backward)     label adds to blank (scatter_add)
// MODE 2: compact layout, source = pair grads + loc (compact backward) label written iff loc != blank
// OUT: element type of the dense output (float; __nv_bfloat16 for the bf16 i/o forward, MODE 0)
template <int MODE, typename OUT = float>
__global__ void __launch_bounds__(kExpandThreads)
k_expand(Problem p, ExpandSrc src, OUT *__restrict__ out, int64_t cells, int V, int blank, int rows_per_chunk,
         FastDiv divV, FastDiv divU, FastDiv divTU, int vec_ok, FastDiv divG) {
    constexpr int VEC = 16 / (int)sizeof(OUT);          // output elements per 16-byte vector
    __shared__ float2 s_g[kExpandMaxRows];
    __shared__ int s_lab[kExpandMaxRows];
    // V % 4 == 2 (float output): two consecutive rows are V/2 whole vectors.  Per row (blank grad, label grad, label
    // position or a far-away "none"), with the label-equals-blank rules already applied, so that the sweep of a
    // row pair is four compare/selects per float and nothing else (see below).
    __shared__ __align__(16) float4 s_q[(VEC == 4) ? kExpandMaxRows + 2 : 1];
    constexpr int kNoLabel = -(1 << 24);
    const bool pair_path = (VEC == 4) && ((V & 3) == 2) && vec_ok && ((rows_per_chunk & 1) == 0);
    const int64_t nchunks = (cells + rows_per_chunk - 1) / rows_per_chunk;
    for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        const int64_t r0 = chunk * rows_per_chunk;
        const int rows = (int)min((int64_t)rows_per_chunk, cells - r0);
        __syncthreads();  // previous chunk's sweep is done with s_g / s_lab
        // ---- phase 1: stage the rows' non-zeros
        for (int r = threadIdx.x; r < rows; r += kExpandThreads) {
            float2 g;
            int lab;
            stage_row<MODE>(p, src, r0 + r, blank, divU, divTU, g, lab);
            s_g[r] = g;
            s_lab[r] = lab;
            if (VEC == 4 && pair_path) {
                const bool adds = (MODE == 1) && src.label_adds;
                float gb = g.x;
                int le = lab;
                if (lab < 0 || (MODE == 1 && !adds && !p.yn && g.y == 0.0f)) le = kNoLabel;    // no label transition here
                else if (adds && lab == blank) { gb += g.y; le = kNoLabel; }                   // scatter_add semantics
                s_q[r] = make_float4(gb, g.y, __int_as_float(le), 0.0f);
            }
        }
        if (VEC == 4 && pair_path && threadIdx.x < 2) s_q[rows + threadIdx.x] = make_float4(0.0f, 0.0f, __int_as_float(kNoLabel), 0.0f);
        __syncthreads();
        // ---- phase 2: sweep the chunk's floats [f0, f1)
        const int64_t f0 = r0 * (int64_t)V;
        const int64_t f1 = f0 + (int64_t)rows * V;
        auto value = [&](int row, int v) -> float {
            const float2 g = s_g[row];
            const int lab = s_lab[row];
            float x = (v == blank) ? g.x : 0.0f;
            // override mode: a zero label gradient marks "no label transition here" (padded labels may equal blank)
            if (v == lab) x = (MODE == 1 && src.label_adds) ? x + g.y : ((MODE == 1 && !p.yn && g.y == 0.0f) ? x : g.y);
            return x;
        };
        int64_t a0 = vec_ok ? min(f1, (f0 + VEC - 1) & ~(int64_t)(VEC - 1)) : f1;
        int64_t a1 = vec_ok ? max(a0, f1 & ~(int64_t)(VEC - 1)) : f1;
        // head and tail scalars (fewer than VEC each when vec_ok)
        for (int64_t f = f0 + threadIdx.x; f < a0; f += kExpandThreads) {
            const uint32_t local = (uint32_t)(f - f0);
            const uint32_t row = divV.div(local);
            st_one(out + f, value((int)row, (int)(local - row * V)));
        }
        for (int64_t f = a1 + threadIdx.x; f < f1; f += kExpandThreads) {
            const uint32_t local = (uint32_t)(f - f0);
            const uint32_t row = divV.div(local);
            st_one(out + f, value((int)row, (int)(local - row * V)));
        }
        if (VEC == 4 && pair_path) {
            // rows come in pairs of G = V/2 vectors (r0 is even, so a0 == f0): vector k of pair q covers positions
            // [4k, 4k+4) of the pair's 2V floats; the four candidate non-zeros sit at blank, label(row0), V + blank,
            // V + label(row1).  The label is applied after its row's blank (it overrides, core.cu:383-390).
            const uint32_t nvec = (uint32_t)((a1 - a0) >> 2), G = (uint32_t)V >> 1;
            float *o4 = reinterpret_cast<float *>(out) + a0;
            for (uint32_t i = threadIdx.x; i < nvec; i += kExpandThreads) {
                const uint32_t q = divG.div(i);
                const int p0 = (int)(4u * (i - q * G));
                const float4 A = s_q[2 * q], B = s_q[2 * q + 1];
                const int ab = blank - p0, al = __float_as_int(A.z) - p0, bb = ab + V, bl = __float_as_int(B.z) - p0 + V;
                float e[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float x = (ab == k) ? A.x : 0.0f;
                    x = (al == k) ? A.y : x;
                    x = (bb == k) ? B.x : x;
                    x = (bl == k) ? B.y : x;
                    e[k] = x;
                }
                st_cs_v4(o4 + 4 * (size_t)i, make_float4(e[0], e[1], e[2], e[3]));
            }
        } else
        for (int64_t f = a0 + VEC * (int64_t)threadIdx.x; f < a1; f += VEC * kExpandThreads) {
            const uint32_t local = (uint32_t)(f - f0);
            uint32_t row = divV.div(local);
            int v = (int)(local - row * V);
            float e[VEC];
            if ((V & (VEC - 1)) == 0) {
                // rows are whole vectors: one staged-row fetch, four compare/selects.  (Kernel-uniform
                // test on purpose: a per-vector "does it straddle a row end" branch makes nearly every
                // warp run both paths -- measured 15 % slower at V = 50.  Also tried and dropped: composing
                // 16 KB tiles in shared memory and streaming them out, 40 % slower at V = 50 because the
                // per-chunk barriers and staging latency are amortised over too few bytes.)
                const float2 g = s_g[row];
                const int lab = s_lab[row];
                const int pb = blank - v, pl = lab - v;
                const bool adds = (MODE == 1) && src.label_adds;
                const bool lab_live = (MODE != 1) || adds || p.yn || (g.y != 0.0f);
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    float x = (k == pb) ? g.x : 0.0f;
                    if (k == pl && lab_live) x = adds ? x + g.y : g.y;
                    e[k] = x;
                }
            } else {
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    e[k] = value((int)row, v);
                    if (++v == V) { v = 0; ++row; }
                }
            }
            st_cs_vec(out + f, e);            // 16 bytes: 4 floats or 8 bf16
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_loss_sum: loss = sum_n costs[n] * scale[n] in a fixed order (general path; the fused kernel does this itself).
// k_rescale : grads[n] *= grad_out[n] / applied[n] where they differ -- RNNTLoss.backward's mul_
//             (__init__.py:21-24) reduced to a no-op for the usual case that the upstream gradient is what the
//             forward already multiplied in (a CTA whose sample needs no change returns at once, no memory traffic).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_loss_sum(const float *__restrict__ costs, const float *__restrict__ scale, int N,
                                                 float *__restrict__ loss_sum) {
    const int lane = threadIdx.x;
    float acc = 0.0f;
    for (int i = lane; i < N; i += 32) acc += scale ? costs[i] * scale[i] : costs[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) *loss_sum = acc;
}

constexpr int kRescaleThreads = 256;
__global__ void __launch_bounds__(kRescaleThreads)
k_rescale_bf16(__nv_bfloat16 *__restrict__ grads, const float *__restrict__ grad_out, int go_stride,
               const float *__restrict__ applied, int64_t elems) {
    const int n = blockIdx.y;
    const float target = grad_out[(int64_t)n * go_stride];
    const float cur = applied ? applied[n] : 1.0f;
    if (target == cur) return;
    const float f = (cur == 1.0f) ? target : target / cur;
    __nv_bfloat16 *g = grads + (int64_t)n * elems;
    for (int64_t i = (int64_t)blockIdx.x * kRescaleThreads + threadIdx.x; i < elems; i += (int64_t)gridDim.x * kRescaleThreads)
        g[i] = __float2bfloat16_rn(__bfloat162float(g[i]) * f);
}

__global__ void __launch_bounds__(kRescaleThreads)
k_rescale(float *__restrict__ grads, const float *__restrict__ grad_out, int go_stride, const float *__restrict__ applied,
          int64_t elems) {
    const int n = blockIdx.y;
    const float target = grad_out[(int64_t)n * go_stride];
    const float cur = applied ? applied[n] : 1.0f;
    if (target == cur) return;                              // already what the forward multiplied in
    const float f = (cur == 1.0f) ? target : target / cur;  // cur == 1: exactly the reference's grads * grad_output
    float *g = grads + (int64_t)n * elems;
    const bool vec = ((reinterpret_cast<uintptr_t>(g) & 15u) == 0);
    const int64_t n4 = vec ? elems / 4 : 0;
    float4 *g4 = reinterpret_cast<float4 *>(g);
    for (int64_t i = (int64_t)blockIdx.x * kRescaleThreads + threadIdx.x; i < n4; i += (int64_t)gridDim.x * kRescaleThreads) {
        float4 v = g4[i];
        v.x *= f; v.y *= f; v.z *= f; v.w *= f;
        g4[i] = v;
    }
    for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * kRescaleThreads + threadIdx.x; i < elems; i += (int64_t)gridDim.x * kRescaleThreads)
        g[i] *= f;
}

cudaError_t launch_loss_sum(cudaStream_t s, const float *costs, const float *scale, int N, float *loss_sum) {
    k_loss_sum<<<1, 32, 0, s>>>(costs, scale, N, loss_sum);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_rescale(cudaStream_t s, void *grads, const float *grad_out, int grad_out_stride, const float *applied,
                           int N, int64_t elems_per_sample, int io_bf16) {
    if (N <= 0 || elems_per_sample <= 0) return cudaSuccess;
    const int sms = sm_count(current_device());
    int64_t gx = (elems_per_sample / 4 + kRescaleThreads * 8 - 1) / (kRescaleThreads * 8);
    const int64_t cap = ((int64_t)sms * 2 + N - 1) / N;      // few CTAs: in the usual case every one of them returns at once
    gx = max((int64_t)1, min(gx, cap));
    dim3 grid((unsigned)gx, (unsigned)N);
    if (io_bf16) k_rescale_bf16<<<grid, kRescaleThreads, 0, s>>>(static_cast<__nv_bfloat16 *>(grads), grad_out, grad_out_stride, applied, elems_per_sample);
    else k_rescale<<<grid, kRescaleThreads, 0, s>>>(static_cast<float *>(grads), grad_out, grad_out_stride, applied, elems_per_sample);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_expand(cudaStream_t s, const Problem &p, const ExpandSrc &src, void *out_v, int64_t cells,
                          int V, int blank, bool retire_early, int io_bf16) {
    float *out = static_cast<float *>(out_v);
    if (cells <= 0) return cudaSuccess;
    int rows = (int)(65536 / ((int64_t)V * (io_bf16 ? 2 : 4)));
    rows = max(1, min(rows, kExpandMaxRows));
    if (rows > 1) rows &= ~1;                          // whole row pairs per chunk (the V % 4 == 2 path pairs rows)
    const int64_t nchunks = (cells + rows - 1) / rows;
    const int sms = sm_count(current_device());
    // persistent CTAs by default; retire_early = one CTA per few chunks, so that SM resources keep freeing
    // up for the high-priority wavefront CTAs of the pipelined path
    const int64_t cap = retire_early ? (int64_t)sms * 64 : (int64_t)sms * 8;
    const int grid = (int)(nchunks < cap ? nchunks : cap);
    const FastDiv divV((uint32_t)V), divU((uint32_t)max(p.U, 1)), divTU((uint32_t)max(p.T * p.U, 1));
    const FastDiv divG((uint32_t)max(V / 2, 1));      // vectors per row pair when V % 4 == 2
    const int vec_ok = ((reinterpret_cast<uintptr_t>(out) & 15u) == 0) ? 1 : 0;
    const int mode = p.compact ? 2 : (src.pg ? 1 : 0);
    if (io_bf16) {
        if (mode != 0) return cudaErrorInvalidValue;    // bf16 output: the dense forward emit only
        k_expand<0, __nv_bfloat16><<<grid, kExpandThreads, 0, s>>>(p, src, static_cast<__nv_bfloat16 *>(out_v), cells, V, blank, rows, divV,
                                                               divU, divTU, vec_ok, divG);
        count_launch();
        return cudaGetLastError();
    }
    if (mode == 0) k_expand<0><<<grid, kExpandThreads, 0, s>>>(p, src, out, cells, V, blank, rows, divV, divU, divTU, vec_ok, divG);
    else if (mode == 1) k_expand<1><<<grid, kExpandThreads, 0, s>>>(p, src, out, cells, V, blank, rows, divV, divU, divTU, vec_ok, divG);
    else k_expand<2><<<grid, kExpandThreads, 0, s>>>(p, src, out, cells, V, blank, rows, divV, divU, divTU, vec_ok, divG);
    count_launch();
    return cudaGetLastError();
}

}  // namespace rnnt
