// fused.cu -- single-kernel loss + gradient for lattices that fit one SM's shared memory
// ((T+U)*U <~ 9k cells: BASELINE configs 1-3).  One launch does everything the reference spreads
// over zeros_like + 4 kernels (+ python gather / mul_):
//
//   phase 0  gather      gather warps stage the lattice's blank/label log-probs into shared memory ONCE, in
//                        diagonal-major form indexed the beta way (replaces the python-level gather,
//                        __init__.py:118-128, and the strided loads inside kernel_warp, core.cu:115-120): one TMA
//                        bulk copy per lattice row (U*V contiguous elements, f32 or bf16) into a row buffer -- two
//                        buffers per gather warp, so the next row is in flight while this one is picked apart -- then
//                        two LDS per cell pick blank and label (fallback: LDG picks in 128-cell chunks).  Rows are
//                        staged from both ends towards the middle and each warp publishes its progress (st.release),
//                        so the two wavefronts START WHILE THE GATHER IS STILL RUNNING and chase it (alpha needs the
//                        top rows first, beta the bottom rows)
//   phase 1  wavefront   ONE warp runs alpha and one runs beta: lane l owns C adjacent lattice columns, every
//                        anti-diagonal is one step = one shuffle + C independent LSE chains, operands and results
//                        move as C-wide vector LDS/STS (a diagonal's cells are contiguous in the staged layout; alpha
//                        walks the same planes as beta, backwards).  No inter-warp hand-off, no barrier, no atomics on
//                        the recurrence (replaces kernel_warp + the global-memory counts scheduler, core.cu:41-258)
//            zero-fill   when the gather is done, two warps' lane 0 issue TMA bulk stores of a zeroed shared-memory
//                        buffer (evict_last) over this CTA's slice of the dense gradient (replaces at::zeros_like,
//                        binding.cpp:58); fallback: 256-bit stores
//            chase       the other free warps follow the two wavefronts from the middle anti-diagonal outwards and
//                        replace each staged log-prob by (alpha + beta) + log-prob: all of the gradient that does not
//                        need beta[0,0]
//   phase 2  cost/guard  kernel_fill_costs (core.cu:334-370) + the reduced loss sum_n costs[n]*scale[n] by the last CTA
//            patch       expf(x - beta00) and <= 2 four-byte stores per cell into the freshly zeroed, still L2-resident
//                        lines (kernel_grads_blank/label, core.cu:260-332), or -- MODE 1 -- the gradients are emitted
//                        in (N,T,U,2) form for the deferred dense backward (+ loc for the compact layout, whose
//                        lattices are addressed through mem_pref / lab_pref).
//
// grid (S, N): S CTAs per lattice recompute the (cheap) wavefront redundantly and split the
// (bandwidth-bound) fill/patch of the lattice's rows, so small batches still use every SM.
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"

namespace rnnt {

constexpr int kFusedThreads = 512;
constexpr float kBigF = -1.0e30f;   // finite stand-in for -inf (see wavefront.cu)

// L2 residency control (B200: 126 MB L2).  The dense gradient slab is zero-filled while the
// wavefront runs and patched afterwards; the patch is a partial-sector write, so it must still HIT
// in L2 or ECC forces a DRAM read-modify-write per touched sector.  Filled lines are therefore
// stored evict_last (TMA bulk stores with an evict_last policy, or 256-bit STG.E.ELL2.256), and the
// one-pass log-prob gather is loaded evict_first so that it cannot displace them.
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float ldg_hint(const float *ptr, uint64_t pol) {
    float v;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(ptr), "l"(pol));
    return v;
}
template <typename IO> __device__ __forceinline__ float ldg_hint_io(const IO *ptr, uint64_t pol);
template <> __device__ __forceinline__ float ldg_hint_io<float>(const float *ptr, uint64_t pol) { return ldg_hint(ptr, pol); }
template <> __device__ __forceinline__ float ldg_hint_io<__nv_bfloat16>(const __nv_bfloat16 *ptr, uint64_t pol) {
    unsigned short v;
    asm volatile("ld.global.nc.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(v) : "l"(ptr), "l"(pol));
    return __uint_as_float((uint32_t)v << 16);
}
__device__ __forceinline__ float2 ldg_hint2(const float2 *ptr, uint64_t pol) {
    float2 v;
    asm volatile("ld.global.nc.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;" : "=f"(v.x), "=f"(v.y) : "l"(ptr), "l"(pol));
    return v;
}
__device__ __forceinline__ void stg_zero256_evict_last(float *ptr) {
    asm volatile("st.global.L2::evict_last.v8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"l"(ptr), "r"(0) : "memory");
}

// Zero-fill through the TMA engine: bulk shared->global copies of a zeroed shared-memory buffer,
// evict_last in L2.  One thread issues 8 KB per instruction, so the fill costs the SM no LSU / MIO
// queue slots -- with STG fills the queue stays full of back-pressured stores and the wavefront
// warps' LDS/STS wait behind them (measured: exact-LSE step 330 ns with STG fill running, 160 ns alone).
constexpr int kZeroBytes = 8192;
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_store(void *gdst, uint32_t ssrc, uint32_t bytes, uint64_t pol) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 ::"l"(gdst), "r"(ssrc), "r"(bytes), "l"(pol) : "memory");
}

// TMA row gather: one bulk global->shared copy per lattice row (U*V contiguous floats), completion
// on an mbarrier.  The whole row is read -- HBM has to deliver it anyway (64-byte atoms: the two
// 4-byte picks per 112-byte cell touch nearly every atom) -- but as full lines by the copy engine
// instead of as ~60 L1 line look-ups per 32 cells, which is what bounded the LDG gather.
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void bulk_load(uint32_t sdst, const void *gsrc, uint32_t bytes, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(sdst), "l"(gsrc), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
constexpr int kMaxRowBufs = 14;                               // one per gather warp

// chunk flags: gather warps publish, wavefront warps consume (same CTA, shared memory)
__device__ __forceinline__ void flag_release(int *f) {
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(f)), "r"(1) : "memory");
}
__device__ __forceinline__ int flag_acquire(const int *f) {
    int v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(f)) : "memory");
    return v;
}
constexpr int kChunkLog = 7, kChunkCells = 1 << kChunkLog;   // gather granule: 4 cells per lane
constexpr int kMaxChunks = 96;                                 // >= ceil(max staged cells / kChunkCells)

// Consumer side of the gather.  Order-row k: even k = top row k/2, odd k = bottom row Tn-1-(k-1)/2.
// A wavefront that is about to read lattice rows within m of its starting edge needs order-rows
// <= 2m+1 staged.
//   chunked LDG gather : chunk q holds order-space cells [128q, 128q+128); flag[q] set when staged
//   TMA row gather     : gather warp g stages order-rows g, g+gwn, ...; flag[g] counts its finished rows
struct GatherWait {
    const int *flag;
    int Un, Tn, lane, gwn;  // gwn > 0: TMA row gather with gwn warps
    int ready;              // chunks [0, ready) / order-rows [0, ready) are known complete
    int m_ok;               // rows(m) is known to hold for every m <= m_ok (one compare on the per-step path)
    __device__ __forceinline__ void ensure(int m) {
        if (m > m_ok) {
            rows(m);
            // order-rows known complete -> largest m with min(2m+1, Tn-1) < rows_done
            const int rows_done = gwn > 0 ? ready : min(Tn, (ready << kChunkLog) / Un);
            m_ok = (rows_done >= Tn) ? 0x7fffffff : ((rows_done - 2) >> 1);
        }
    }
    __device__ __forceinline__ void rows(int m) {
        const int k = min(2 * m + 1, Tn - 1);
        if (gwn > 0) {
            while (ready <= k) {
                int first_open = 0x7fffffff;          // this gather warp's first unfinished order-row
                if (lane < gwn) first_open = flag_acquire(flag + lane) * gwn + lane;
                ready = __reduce_min_sync(0xffffffffu, first_open);
            }
        } else {
            const int q = ((k + 1) * Un - 1) >> kChunkLog;
            while (ready <= q) {
                while (flag_acquire(flag + ready) == 0) {}
                ++ready;
            }
        }
    }
};

// C-wide shared-memory vector load / store (C in {1,2,4,8}); asm volatile keeps program order so
// the operand prefetch stays where it is written.
template <int C>
__device__ __forceinline__ void lds_vec(uint32_t a, float (&v)[C]) {
    if constexpr (C == 1) {
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v[0]) : "r"(a) : "memory");
    } else if constexpr (C == 2) {
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(a) : "memory");
    } else if constexpr (C == 4) {
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a) : "memory");
    } else {
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a) : "memory");
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(a + 16u) : "memory");
    }
}
template <int C>
__device__ __forceinline__ void sts_vec(uint32_t a, const float (&v)[C]) {
    if constexpr (C == 1) {
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v[0]) : "memory");
    } else if constexpr (C == 2) {
        asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(v[0]), "f"(v[1]) : "memory");
    } else if constexpr (C == 4) {
        asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
    } else {
        asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
        asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a + 16u), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
    }
}

// Fused loss reduction (replaces the separate costs.sum() pass of __init__.py:132-143 and, through `scale`,
// average_frames / 'mean'): every reporting CTA's warp 0 calls this after its thread 0 wrote costs[n]; the LAST caller
// (device counter) adds costs[0..N) * scale[0..N) in a fixed order -- lane-strided partial sums, then a shuffle tree --
// so the result is deterministic (no float atomics).  The counter is left at 0 for the next launch.
__device__ __forceinline__ void loss_reduce_last(const float *costs, const float *scale, int N, float *loss_sum,
                                                 unsigned *counter) {
    const int lane = threadIdx.x & 31;
    unsigned last = 0;
    if (lane == 0) {
        __threadfence();                                    // costs[n] before the ticket
        last = (atomicAdd(counter, 1u) == (unsigned)(N - 1)) ? 1u : 0u;
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();                                        // the other CTAs' costs after the ticket
    float acc = 0.0f;
    for (int i = lane; i < N; i += 32) {
        const float c = __ldcg(costs + i);
        acc += scale ? c * __ldcg(scale + i) : c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) { *loss_sum = acc; *counter = 0u; }
}

struct FusedArgs {
    const void *lp;         // dense (N,T,U,V) of the kernel's IO type (f32 / bf16) or, pairs_in, (N,T,U,2) f32
    const int *labels;      // (N,U-1); compact: (sum yn)
    const int64_t *mem_pref, *lab_pref;   // compact layout: first cell / first label of lattice n (else null)
    int64_t *loc;           // compact layout: label id per cell (core_compact.cu:424-431), or null
    const int *xn, *yn;
    float *costs;           // (N)
    void *grads;            // MODE 0: dense (N,T,U,V) of the kernel's IO type
    float2 *pair_grads;     // MODE 1: (N,T,U) float2
    const float *scale;     // (N) or null
    int N, T, U, V, blank;
    float lam;
    int pairs_in, guard, slices;
    int zoff;               // byte offset of the zero buffer in dynamic shared memory
    int nbuf, row_off, row_stride;   // TMA row gather: buffers (0 = LDG gather), their byte offset and stride
    int gwn, nb_per;        // TMA row gather: gather warps and row buffers per warp (nbuf = gwn * nb_per)
    int Wd;                 // staged row stride (floats) = C * ceil(U / C), even
    int nd;                 // staged rows (diagonals) allocated = T + Wd + 16
    int gw;                 // warps that gather (of the 14 non-wavefront warps); MODE 0: the rest start the zero-fill at once
    int tma_fill;           // MODE 0: zero-fill with bulk shared->global copies (else 256-bit STG)
    int fill_warps;         // MODE 0, bulk fill: how many of the 14 free warps issue it (the others chase at once)
    long long *trace;       // optional per-CTA phase stamps (clock64), 8 per CTA; null = off
    float *loss_sum;        // optional: sum_n costs[n] * (scale ? scale[n] : 1), written by the last CTA to finish
    unsigned *sync_counter; // with loss_sum: device counter, 0 on entry, left 0 (self-resetting)
    int poison_n;           // test hook: sample whose alpha-side ll gets poison_delta added before the guard (-1 = off)
    float poison_delta;
};

// One direction of one lattice, one warp.  Diagonal-major, target-indexed operands:
//   wb[d][j] = weight of the row edge    (i-1,j) -> (i,j)       with i = d - j
//   wl[d][j] = weight of the column edge (i,j-1) -> (i,j)
// and out[d][j] = val[i,j].  Slots outside the lattice hold wb = 0, wl = kBig, which makes the one
// uniform step below reproduce every edge rule of core.cu:64-134 / :171-239 without a branch:
//   row 0 (val starts at kBig -> skip vanishes), first column (wl = kBig -> emit vanishes),
//   cell (0,0) (val of the first real column starts at 0 and wb(0,0) carries the initial value),
//   cells past the last row / column only ever feed other out-of-lattice slots.
// Column j at diagonal d reads its own previous value (row edge) and column j-1's previous value
// (column edge): inside a lane that is a register, across lanes one __shfl_up of the lane's last column.
// __shfl_up_sync(full, v, 1) as a volatile asm: keeps the shuffle in program order with the (volatile)
// shared-memory loads/stores of the loop.  Left free, the compiler batches three steps' LDS/STS in front of
// the fourth shuffle and then copies the freshly loaded operands into place -- register moves that wait
// for the load they follow, on the dependent chain (exact LSE: 158 vs 125 ns per step).
__device__ __forceinline__ float shfl_up1_ordered(float v) {
    float r;
    asm volatile("shfl.sync.up.b32 %0, %1, 1, 0, 0xffffffff;" : "=f"(r) : "f"(v) : "memory");
    return r;
}

// ALPHA: the operands come from the BETA-side planes (one staged copy of the log-probs serves both directions; the
// shared memory this saves holds more TMA row buffers).  An anti-diagonal t+u = e is ONE row of the beta layout,
// r(e) = T1 + Wd - 1 - e, with the columns reversed (j' = Wd-1-u).  Alpha's step e needs the blank edges of the cells
// on diagonal e-1 -> row r(e)+1, walked DOWNWARDS (negative stride), the lane's C columns as one reversed vector; its
// label edges sit one column further (lp_l[t,u-1] at j'+1): the aligned vector supplies C-1 of them and the lane to
// the left the last one (one extra shuffle per step, off the dependent chain; lattice column 0 has no label edge).
// `prog`: diagonals completed so far, published (st.release) once per loop iteration for the warps that chase the
// wavefronts (see k_fused, "chase").
template <int KIND, int C, bool ALPHA>
__device__ __forceinline__ void sweep_diag(uint32_t wb, uint32_t wl, uint32_t out, int Wd, int ndiag, int lane,
                                           int first_col, const float *pre, int pre_rows, GatherWait gw,
                                           uint32_t scratch, int *prog, int row0) {
    constexpr int P = (C <= 2) ? 4 : 2;                       // diagonals of operand prefetch = steps per loop iteration
    float val[C];
#pragma unroll
    for (int c = 0; c < C; ++c) val[c] = (C * lane + c == first_col) ? 0.0f : kBigF;
    // The loop below is one long dependent chain (shuffle -> add -> LSE -> shuffle ...) on an in-order
    // pipeline: anything that stalls ISSUE stalls the chain.  So the row stride lives in a register the
    // compiler cannot rematerialise from the constant bank (a per-step LDC + dependent IMAD cost ~40
    // cycles), the exact-mode column override is a prefetched select instead of a divergent branch
    // around a shared-memory load, and the gather hand-shake is checked once per P steps.
    uint32_t stride = 4u * (uint32_t)Wd;
    asm volatile("" : "+r"(stride));
    const uint32_t off = 4u * (uint32_t)(C * lane);
    // operand addresses.  beta: row 0 upwards, columns C*lane..  alpha: row `row0` = T1 + Wd downwards, columns
    // Wd - C*(lane+1).. (reversed); lanes past the staged row read neighbouring rows (finite garbage, never used)
    const uint32_t opoff = ALPHA ? (uint32_t)(4 * (row0 * Wd + Wd - C * (lane + 1))) : off;
    uint32_t a_wb = wb + opoff, a_wl = wl + opoff, a_out = out + off;
    const uint32_t ostride = ALPHA ? (0u - stride) : stride;
    // one diagonal's operands into b[k], l[k] (alpha: reversed vector + the left lane's first element)
    auto fetch = [&](float (&bk)[C], float (&lk)[C]) {
        if constexpr (ALPHA) {
            float vb[C], vl[C];
            lds_vec<C>(a_wb, vb);
            lds_vec<C>(a_wl, vl);
            float edge;
            asm volatile("shfl.sync.up.b32 %0, %1, 1, 0, 0xffffffff;" : "=f"(edge) : "f"(vl[0]) : "memory");
            if (lane == 0) edge = kBigF;                       // lattice column 0: no label edge
#pragma unroll
            for (int c = 0; c < C; ++c) {
                bk[c] = vb[C - 1 - c];
                lk[c] = (c == 0) ? edge : vl[C - c];
            }
        } else {
            lds_vec<C>(a_wb, bk);
            lds_vec<C>(a_wl, lk);
        }
        a_wb += ostride;
        a_wl += ostride;
    };
    // exact mode: the first real column is taken from the reference-order prefix scan (core.cu:92-110)
    const int l0 = first_col / C, c0 = first_col - l0 * C;
    // Predicate registers are scarce (7 per thread) and each exact-LSE chain keeps 3 alive; with more in the
    // loop ptxas runs the lane's C chains one after the other instead of interleaved (160 vs 125 ns per step
    // at C = 2).  So the column override is a bitwise select on a mask, and lanes past the staged row store to a
    // scratch slot instead of being predicated off.
    uint32_t own[C];                                          // all-ones where this register holds the first real column
#pragma unroll
    for (int c = 0; c < C; ++c) own[c] = ((KIND != kFast) && lane == l0 && c == c0) ? 0xffffffffu : 0u;
    const uint32_t a_pre = (uint32_t)__cvta_generic_to_shared(pre);
    const uint32_t a_prog = (uint32_t)__cvta_generic_to_shared(prog);
    auto pre_at = [&](int d) -> float {                      // scan value for diagonal d (clamped; unused when out of range)
        const int i = min(max(d - first_col, 0), pre_rows - 1);
        float v;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a_pre + 4u * (uint32_t)i) : "memory");
        return v;
    };
    // results are written in place over operands (see k_fused): lanes past the staged row must not spill into
    // the next one -- they store to `scratch` (4*C bytes per lane) instead
    const bool in_row = C * lane < Wd;
    if (!in_row) a_out = scratch + off;
    uint32_t stride_out = in_row ? stride : 0u;
    asm volatile("" : "+r"(stride_out));
    float b[P][C], l[P][C], pv[P];
    gw.ensure(P - 1);                                         // diagonals 0..P-1 touch rows <= P-1
#pragma unroll
    for (int k = 0; k < P; ++k) {
        fetch(b[k], l[k]);
        if (KIND != kFast) pv[k] = pre_at(k);
    }
    // Exact LSE: ptxas interleaves the lane's C chains in every step of the unrolled body except the last one
    // before the back-edge (and in none of them if the loop also contains a conditional store, e.g. a trace
    // stamp) -- so the body is 2P steps long: 7 of 8 steps run at ~125 ns instead of 160 ns.
    // tools/sass_check.py watches this.
    constexpr int H = (KIND != kFast) ? 2 : 1;                 // groups of P steps per iteration
    for (int d00 = 0; d00 < ndiag; d00 += H * P) {
        gw.ensure(d00 + (H + 1) * P - 1);                      // the gather has staged every row this iteration prefetches
#pragma unroll
      for (int h = 0; h < H; ++h) {
        const int d0 = d00 + h * P;
#pragma unroll
        for (int k = 0; k < P; ++k) {
            const float left = shfl_up1_ordered(val[C - 1]);   // lane 0 gets its own value: wl = kBig there
            float nv[C], xs[C], ys[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                xs[c] = val[c] + b[k][c];                             // row edge
                ys[c] = (c == 0 ? left : val[c > 0 ? c - 1 : 0]) + l[k][c];   // column edge
            }
            lse_vec<KIND, C>(xs, ys, nv);
            if (KIND != kFast) {
                const int i = d0 + k - first_col;              // row of the first real column on this diagonal
                const uint32_t in = ((i >= 1) && (i < pre_rows)) ? 0xffffffffu : 0u;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const uint32_t m = own[c] & in;
                    nv[c] = __uint_as_float((__float_as_uint(nv[c]) & ~m) | (__float_as_uint(pv[k]) & m));
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c) val[c] = nv[c];
            sts_vec<C>(a_out, val);                          // (lanes past the staged row: scratch slot, stride 0)
            a_out += stride_out;
            fetch(b[k], l[k]);                                 // operands P diagonals ahead (rows past ndiag are allocated)
            if (KIND != kFast) pv[k] = pre_at(d0 + k + P);
        }
      }
        // progress for the chasing warps: diagonals < d00 + H*P are complete and their operands consumed (every lane
        // stores the same word: an unconditional store keeps the loop free of predicated side exits)
        asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(a_prog), "r"(d00 + H * P) : "memory");
    }
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(a_prog), "r"(0x3fffffff) : "memory");
}

// MODE 0: dense gradients (zero-fill + patch).  MODE 1: (N,T,U,2) gradients.  Both write costs.
// IO: element type of log_probs and of the dense gradient (float, or __nv_bfloat16 with MODE 0).
template <int KIND, int MODE, int C, typename IO = float>
__global__ void __launch_bounds__(kFusedThreads, 1) k_fused(FusedArgs A) {
    constexpr int ESZ = (int)sizeof(IO);
    const IO *const lp_io = static_cast<const IO *>(A.lp);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = blockIdx.y, slice = blockIdx.x;
    const int T = A.T, U = A.U, V = A.V, Wd = A.Wd;
    const int Tn = A.xn[n], Un = A.yn[n] + 1;
    const bool ok = (Tn >= 1 && Tn <= T && Un >= 1 && Un <= U);
    const int T1 = Tn - 1, U1 = Un - 1;

    // ---- shared memory carve-up: four diagonal-major planes [nd][Wd], prefix-scan columns, labels.
    // ONE staged copy of the log-probs (beta-side indexing) serves both wavefronts; alpha walks it backwards.
    // Plane order matters: alpha's prefetch past its last diagonal reads a few rows BELOW row 0 of WBb / WLb, which
    // must still be shared memory (it lands in the plane before; the values are never used).
    const size_t plane = (size_t)A.nd * Wd;
    float *AL = reinterpret_cast<float *>(smem_raw);    // alpha[t,u] at [t+u][u]
    float *BE = AL + plane;                             // beta[t,u]  at [d'][j'], j' = Wd-1-u, d' = (T1-t)+j'
    float *WBb = BE + plane;                            // blank edge out of (t,u) at [d'][j']; after the chase: alpha+beta+lp
    float *WLb = WBb + plane;                           // label edge out of (t,u) at [d'][j']; after the chase: alpha+beta+lp
    float *preA = WLb + plane;                          // [T] exact-mode column scans
    float *preB = preA + T;
    int *s_lab = reinterpret_cast<int *>(preB + T);     // [U]
    // zero buffer for the bulk fill: the last kZeroBytes of the dynamic allocation (128-byte aligned)
    float *zbuf = reinterpret_cast<float *>(smem_raw + A.zoff);
    __shared__ __align__(16) float s_scratch[2][256];   // wavefront lanes past the staged row store here
    __shared__ int s_next;                              // fill work counter
    __shared__ int s_bad;
    __shared__ int s_flag[kMaxChunks];                  // gather chunk q staged / rows finished by gather warp g
    __shared__ int s_prog[2];                           // diagonals completed by the alpha / beta wavefront
    __shared__ __align__(8) unsigned long long s_bar[2 * kMaxRowBufs];   // TMA row gather: one mbarrier per buffer
    long long *trace = A.trace ? A.trace + 16 * ((size_t)blockIdx.y * gridDim.x + blockIdx.x) : nullptr;
    auto stamp = [&](int slot) {                        // latest arrival per phase
        if (trace && lane == 0) atomicMax(reinterpret_cast<unsigned long long *>(trace) + slot, (unsigned long long)clock64());
    };
    stamp(0);
    auto idxA = [&](int t, int u) { return (t + u) * Wd + u; };
    auto idxB = [&](int t, int u) { const int jp = Wd - 1 - u; return (T1 - t + jp) * Wd + jp; };

    // rows of the padded slab this CTA fills / patches
    const int t0 = (int)((int64_t)T * slice / A.slices), t1 = (int)((int64_t)T * (slice + 1) / A.slices);
    // dense: lattice n is a padded (T,U) slab; compact: its Tn*Un cells are packed at mem_pref[n]
    const bool compact = (A.mem_pref != nullptr);
    const int64_t slab = compact ? A.mem_pref[n] : (int64_t)n * T * U;   // first cell of this lattice
    const int RS = compact ? Un : U;                    // cells per lattice row in memory
    const int64_t lab0 = compact ? A.lab_pref[n] : (int64_t)n * (U - 1);
    // TMA rows need 16-byte aligned, 16-byte multiple rows: always true when chosen for the dense layout,
    // per lattice in the compact layout
    const bool use_tma = A.nbuf > 0 && (!compact || ((((slab * V) | ((int64_t)Un * V)) & (16 / ESZ - 1)) == 0));

    // ---- phase 0: sentinels, labels, gather
    if (tid == 0) { s_next = 0; s_bad = ok ? 0 : 1; s_prog[0] = 0; s_prog[1] = 0; }
    if (tid < kMaxChunks) s_flag[tid] = 0;
    if (tid < A.nbuf) mbar_init((uint32_t)__cvta_generic_to_shared(&s_bar[tid]), 1);
    if (A.nbuf > 0) {                                   // make the initialised barriers visible to the async proxy (TMA)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (MODE == 0 && A.tma_fill) {
        for (int k = tid; k < kZeroBytes / 4; k += kFusedThreads) zbuf[k] = 0.0f;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy zeros -> async-proxy reads
    }
    if (ok) {
        const int used = (Tn + Wd + 16) * Wd;           // diagonals any sweep or its prefetch can touch
        const int lim4 = min((used + 3) >> 2, (int)(plane >> 2));   // planes are whole float4s (nd, Wd even)
        const float4 z4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), b4 = make_float4(kBigF, kBigF, kBigF, kBigF);
        for (int k = tid; k < lim4; k += kFusedThreads) {
            reinterpret_cast<float4 *>(WBb)[k] = z4;
            reinterpret_cast<float4 *>(WLb)[k] = b4;
        }
        if (!A.pairs_in)
            for (int u = tid; u < U1; u += kFusedThreads) s_lab[u] = A.labels[lab0 + u];
    }
    __syncthreads();
    stamp(1);
    // Roles go by a rotated warp index: the two wavefront warps are the HIGHEST-numbered hardware
    // warps (14 and 15, on different sub-partitions).  The SM's issue arbiter favours higher warp
    // ids, so the latency-critical recurrence is never starved by the fill / gather warps sharing its
    // scheduler (with the sweep on warps 0/1 the exact flavour measured anywhere from 65 to 250 us).
    //   logical warp 0 / 1      alpha / beta wavefront, chasing the gather chunk by chunk
    //   logical warps [2,2+GW)  gather, then (MODE 0) zero-fill
    //   the rest (MODE 0)       zero-fill from the start: HBM reads (gather) and writes (fill) overlap
    const int lw = (warp + 2) & (kFusedThreads / 32 - 1);
    const int GW = A.gw;
    const int cells_n = ok ? Tn * Un : 0;
    const int nchunks = (cells_n + kChunkCells - 1) >> kChunkLog;
    if (use_tma) {
        // TMA row gather: gather warp g of `gwn` stages order-rows g, g+gwn, ... through its own `nb_per` row buffers
        // (two when they fit: the next row is already in flight while this one is picked apart)
        if (ok && lw >= 2 && lw < 2 + A.gwn) {
            const int g = lw - 2, NB = A.nb_per;
            const uint64_t pol_first = policy_evict_first();
            const uint32_t bytes = ((uint32_t)(Un * V) * (uint32_t)ESZ + 15u) & ~15u;   // <= U*V*ESZ, which is a multiple of 16
            auto buf_of = [&](int slot) { return reinterpret_cast<const IO *>(smem_raw + A.row_off + (size_t)(g * NB + slot) * A.row_stride); };
            auto row_of = [&](int k) { return (k & 1) ? T1 - (k >> 1) : (k >> 1); };   // rows alternate: top, bottom, top, ...
            auto issue = [&](int k, int slot) {
                if (lane == 0) {
                    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar[g * NB + slot]);
                    mbar_expect_tx(bar, bytes);
                    bulk_load((uint32_t)__cvta_generic_to_shared(buf_of(slot)), lp_io + (slab + (int64_t)row_of(k) * RS) * V, bytes, bar, pol_first);
                }
            };
            for (int j = 0; j < NB; ++j)
                if (g + j * A.gwn < Tn) issue(g + j * A.gwn, j);
            uint32_t phases = 0;                        // bit `slot` = parity to wait for
            int done = 0, slot = 0;
            for (int k = g; k < Tn; k += A.gwn) {
                const int t = row_of(k);
                const IO *buf = buf_of(slot);
                const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar[g * NB + slot]);
                // lane 0 waits for the copy, the warp converges behind it (one poller per barrier)
                if (lane == 0) while (!mbar_try_wait(bar, (phases >> slot) & 1u)) {}
                __syncwarp();
                phases ^= 1u << slot;
                for (int u = lane; u < Un; u += 32) {
                    const float vb = io_to_float<IO>(buf[u * V + A.blank]);
                    const float vl = (u < U1) ? io_to_float<IO>(buf[u * V + s_lab[u]]) : kBigF;
                    const int ib = idxB(t, u);
                    WBb[ib] = vb;
                    WLb[ib] = vl;                       // kBig on the last column: beta's first column has no column edge
                }
                __syncwarp();                           // every lane is done with the buffer and has staged its cells
                const int kn = k + NB * A.gwn;          // refill this buffer with the row NB turns ahead
                if (kn < Tn) issue(kn, slot);
                if (lane == 0) {
                    ++done;
                    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_flag[g])), "r"(done) : "memory");
                }
                slot = (slot + 1 == NB) ? 0 : slot + 1;
            }
            stamp(2);
        }
        // the zero-fill starts when the whole gather is done (HBM serves the critical reads first)
        if (MODE == 0 && lw >= 2) asm volatile("bar.sync 1, %0;" ::"r"(kFusedThreads - 64) : "memory");
    } else if (ok && lw >= 2 && lw < 2 + GW) {
        const float inv = 1.0f / (float)Un;
        const uint64_t pol_first = policy_evict_first();
        constexpr int G = kChunkCells / 32;             // cells per lane per chunk: all loads first
        for (int q = lw - 2; q < nchunks; q += GW) {
            float vb[G], vl[G];
            int tt[G], uu[G];
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int c = (q << kChunkLog) + g * 32 + lane;   // cell index in order-space
                const bool in = c < cells_n;
                int k = (int)(((float)c + 0.5f) * inv);            // order-row
                int u = c - k * Un;
                if (u < 0) { --k; u += Un; } else if (u >= Un) { ++k; u -= Un; }
                int t = (k & 1) ? T1 - (k >> 1) : (k >> 1);        // rows alternate: top, bottom, top, ...
                if (!in) { t = 0; u = 0; }
                tt[g] = in ? t : -1;
                uu[g] = u;
                const int64_t cell = slab + (int64_t)t * RS + u;
                vl[g] = kBigF;
                if (A.pairs_in) {
                    const float2 w2 = ldg_hint2(static_cast<const float2 *>(A.lp) + cell, pol_first);
                    vb[g] = w2.x;
                    if (u < U1) vl[g] = w2.y;
                } else {
                    const IO *row = lp_io + cell * V;
                    vb[g] = ldg_hint_io<IO>(row + A.blank, pol_first);
                    if (u < U1) vl[g] = ldg_hint_io<IO>(row + s_lab[u], pol_first);
                }
            }
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int t = tt[g], u = uu[g];
                if (t >= 0) {
                    const int ib = idxB(t, u);
                    WBb[ib] = vb[g];
                    WLb[ib] = vl[g];                    // kBig on the last column: beta's first column has no column edge
                }
            }
            __syncwarp();
            if (lane == 0) flag_release(&s_flag[q]);
        }
        stamp(2);
    }

    // ---- phase 1: logical warp 0 = alpha, 1 = beta (then both help filling); other warps zero-fill
    if (ok && lw < 2) {
        const bool beta = (lw == 1);
        const int first_col = beta ? (Wd - Un) : 0;
        const int ndiag = beta ? (Tn + Wd - 1) : (Tn + Un - 1);
        float *pre = beta ? preB : preA;
        if (KIND != kFast) {
            // column 0 in the reference's summation order: 32-wide Kogge-Stone scan per tile + the tile's
            // base (core.cu:92-110 / :197-215), so that exact mode is bit-identical.  The column's blank
            // edges are fetched straight from HBM by this warp (the gather is still in flight):
            // pre[0] = base, pre[i] = edge into row i of the first column.
            for (int i0 = lane; i0 <= T1; i0 += 256) {  // eight loads in flight per lane
                float v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int i = min(i0 + 32 * k, T1);
                    const int64_t cell = slab + (beta ? ((int64_t)(T1 - i) * RS + U1) : ((int64_t)max(i - 1, 0) * RS));
                    v[k] = A.pairs_in ? __ldg(static_cast<const float2 *>(A.lp) + cell).x : io_load<IO>(lp_io + cell * V + A.blank);
                    if (!beta && i == 0) v[k] = 0.0f;
                }
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (i0 + 32 * k <= T1) pre[i0 + 32 * k] = v[k];
            }
            __syncwarp();
            float base = pre[0];
            for (int p0 = 0; p0 < T1; p0 += 32) {
                const int i = p0 + lane + 1;
                float bsum = 0.0f;
                if (i <= T1) bsum = pre[i];             // blank edge into row i of the first column
#pragma unroll
                for (int k = 1; k < 32; k <<= 1) {
                    const float a = __shfl_up_sync(0xffffffffu, bsum, k);
                    if (k <= lane) bsum += a;
                }
                const float v = base + bsum;
                if (i <= T1) pre[i] = v;
                base = __shfl_sync(0xffffffffu, v, 31);
            }
            __syncwarp();
        }
        const uint32_t wb_a = (uint32_t)__cvta_generic_to_shared(WBb);
        const uint32_t wl_a = (uint32_t)__cvta_generic_to_shared(WLb);
        const uint32_t out_a = (uint32_t)__cvta_generic_to_shared(beta ? BE : AL);
        GatherWait gwait;
        gwait.flag = s_flag; gwait.Un = Un; gwait.Tn = Tn; gwait.ready = 0; gwait.lane = lane; gwait.gwn = use_tma ? A.gwn : 0; gwait.m_ok = -1;
        stamp(3);
        const uint32_t scr = (uint32_t)__cvta_generic_to_shared(&s_scratch[lw][0]);
        if (beta) sweep_diag<KIND, C, false>(wb_a, wl_a, out_a, Wd, ndiag, lane, first_col, pre, Tn, gwait, scr, &s_prog[1], 0);
        else sweep_diag<KIND, C, true>(wb_a, wl_a, out_a, Wd, ndiag, lane, first_col, pre, Tn, gwait, scr, &s_prog[0], T1 + Wd);
        stamp(beta ? 5 : 4);
    }
    if (MODE == 0) {
        // zero-fill rows [t0,t1) of this lattice's slab: elements [f0,f1); 32 KB chunks handed out by
        // s_next; 256-bit evict_last stores (or bulk copies) on the 32-byte aligned interior
        const int64_t f0 = (slab + (int64_t)t0 * U) * V, f1 = (slab + (int64_t)t1 * U) * V;
        IO *g = static_cast<IO *>(A.grads);
        constexpr int EPV = 32 / ESZ;                   // elements per 32 bytes
        const bool vec = ((reinterpret_cast<uintptr_t>(g) & 31u) == 0);
        const int64_t a0 = vec ? min(f1, (f0 + EPV - 1) & ~(int64_t)(EPV - 1)) : f1;
        const int64_t a1 = vec ? max(a0, f1 & ~(int64_t)(EPV - 1)) : f1;
        constexpr int kChunk = 32768 / ESZ;             // elements per chunk
        const int64_t nfill = (a1 - a0 + kChunk - 1) / kChunk;
        if (A.tma_fill) {
            // the bulk-copy issue blocks when the SM's copy queue is full (the zeros drain at HBM speed), so only
            // `fill_warps` warps issue -- one instruction per 8 KB keeps the queue full -- and the others chase at once
            if (lane == 0 && (lw < 2 || lw >= 2 + (kFusedThreads / 32 - 2) - A.fill_warps)) {
                const uint64_t pol = policy_evict_last();
                const uint32_t zs = (uint32_t)__cvta_generic_to_shared(zbuf);
                constexpr int piece = kZeroBytes / ESZ; // elements per bulk copy
                for (;;) {
                    const int c = atomicAdd(&s_next, 1);
                    if (c >= nfill) break;
                    const int64_t b = a0 + (int64_t)c * kChunk;
                    const int64_t e = min(a1, b + kChunk);
                    for (int64_t f = b; f < e; f += piece)
                        bulk_store(g + f, zs, (uint32_t)(min(e - f, (int64_t)piece) * ESZ), pol);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
            __syncwarp();
        } else {
            for (;;) {
                int c = 0;
                if (lane == 0) c = atomicAdd(&s_next, 1);
                c = __shfl_sync(0xffffffffu, c, 0);
                if (c >= nfill) break;
                const int64_t b = a0 + (int64_t)c * kChunk;
                const int64_t e = min(a1, b + kChunk);
#pragma unroll 4
                for (int64_t f = b + EPV * lane; f < e; f += 32 * EPV) stg_zero256_evict_last(reinterpret_cast<float *>(g + f));
            }
        }
        if (lw == kFusedThreads / 32 - 1) {             // unaligned head / tail (< 32 bytes each, or everything if !vec)
            for (int64_t f = f0 + lane; f < a0; f += 32) g[f] = io_from_float<IO>(0.0f);
            for (int64_t f = a1 + lane; f < f1; f += 32) g[f] = io_from_float<IO>(0.0f);
        }
        stamp(6);
        // ---- chase: while the zeros drain and the two wavefronts run their last diagonals, the 14 free warps follow
        // them from the MIDDLE anti-diagonal outwards (alpha has passed it from above, beta from below: the cells of
        // diagonal e are final once alpha is past e+1 and beta past e+1 from the other side) and replace each staged
        // log-prob by the exponent's variable part, in the reference's operation order (core.cu:284-294, :319-331):
        //   WBb[cell] <- (alpha[t,u] + beta[t+1,u]) + lp_blank        WLb[cell] <- (alpha[t,u] + beta[t,u+1]) + lp_label
        // What is left for after beta[0,0] is known is expf(x - beta00) and the store.
        if (ok && lw >= 2) {
            const int CW = kFusedThreads / 32 - 2, cw = lw - 2;
            const int r0 = t0, r1 = min(t1, Tn);        // rows this CTA patches
            const int Elast = T1 + U1, mid = Elast >> 1, E0 = T1 + Wd - 1;
            int pa = 0, pb = 0;                         // cached progress of the alpha / beta wavefront
            for (int k = cw; k <= Elast && r1 > r0; k += CW) {
                const int e = (k & 1) ? mid + ((k + 1) >> 1) : mid - (k >> 1);
                const int ulo = max(0, e - r1 + 1), uhi = min(U1, e - r0);
                if (ulo > uhi) continue;
                // alpha: steps <= e+1 done (it reads diagonal e's staged log-probs at step e+1);
                // beta: anti-diagonal e+1 done = its steps <= E0-e-1, whose operand prefetch covers diagonal e
                while (pa < e + 2) { pa = flag_acquire(&s_prog[0]); if (pa < e + 2) __nanosleep(100); }
                while (pb < E0 - e) { pb = flag_acquire(&s_prog[1]); if (pb < E0 - e) __nanosleep(100); }
                for (int u = ulo + lane; u <= uhi; u += 32) {
                    const int t = e - u;
                    const int ib = idxB(t, u);
                    const float a0v = AL[idxA(t, u)];
                    const bool last_t = (t == T1), last_u = (u == U1);
                    if (!(last_t && !last_u)) {
                        float a = a0v;
                        if (!last_t) a += BE[ib - Wd];  // beta[t+1,u]: one diagonal earlier, same column
                        WBb[ib] = a + WBb[ib];
                    }
                    if (!last_u) {
                        const float a = a0v + BE[ib - Wd - 1];   // beta[t,u+1]: previous diagonal, previous primed column
                        WLb[ib] = a + WLb[ib];
                    }
                }
            }
            stamp(8);
        }
        if (A.tma_fill && lane == 0) {
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the zeros have landed ...
            asm volatile("fence.proxy.async;" ::: "memory");            // ... before anyone patches them
        }
        stamp(9);
    }
    __syncthreads();

    // ---- phase 2: cost (+ mismatch guard, core.cu:346-367), gradients
    if (tid == 0) {
        float cost = NAN;
        if (ok) {
            float b = BE[idxB(0, 0)];                   // beta[0,0]
            if (A.guard) {
                // alpha-side ll = alpha[T-1,U-1] + blank[T-1,U-1] (core.cu:346); MODE 0: the chase has left exactly this sum
                float a = (MODE == 0 && t0 <= T1 && T1 < t1) ? WBb[idxB(T1, U1)] : AL[idxA(T1, U1)] + WBb[idxB(T1, U1)];
                if (n == A.poison_n) a += A.poison_delta;              // test hook, see rnnt_b200_debug_guard_poison
                const float ratio = fabsf(a - b) / fabsf(fmaxf(a, b));
                if (ratio > 0.001f) {
                    if (slice == 0)
                        printf("\nWARNING: sample %d [%d, %d] has a forward/backward mismatch %f / %f\n", n, Tn, Un - 1, a, b);
                    b = (a + b) / 2.0f;
                    s_bad = 1;
                }
            }
            cost = -b;
        }
        if (slice == 0) A.costs[n] = cost;
    }
    if (A.loss_sum && slice == 0 && warp == 0) loss_reduce_last(A.costs, A.scale, A.N, A.loss_sum, A.sync_counter);
    __syncthreads();
    stamp(10);
    const bool live = ok && !s_bad;
    const float b00 = live ? BE[idxB(0, 0)] : 0.0f;
    const float sc = A.scale ? A.scale[n] : 1.0f;
    const bool has_lam = (A.lam != 0.0f);
    auto cell_grad = [&](int t, int u) -> float2 {
        // same operation order as core.cu:284-294 and :319-331
        const int ib = idxB(t, u);
        const float a0v = AL[idxA(t, u)];
        float gb = 0.0f, gl = 0.0f;
        const bool last_t = (t == T1), last_u = (u == U1);
        if (!(last_t && !last_u)) {
            float a = a0v;
            if (!last_t) a += BE[ib - Wd];              // beta[t+1,u]: one diagonal earlier, same column
            a = expf(a + WBb[ib] - b00);
            gb = -a;
        }
        if (!last_u) {
            float a = a0v + BE[ib - Wd - 1];            // beta[t,u+1]: previous diagonal, previous primed column
            a = expf(a + WLb[ib] - b00);
            // (1. + lambda) * a is a double multiply in the reference (core.cu:327-329); with lambda == 0
            // it returns a unchanged, so the fp64 round trip is skipped without changing a bit
            if (has_lam) a = (float)((1.0 + (double)A.lam) * (double)a);
            gl = -a;
        }
        if (A.scale) { gb *= sc; gl *= sc; }
        return make_float2(gb, gl);
    };
    if (MODE == 0) {
        if (live) {
            // Items (t, u, blank|label) of rows [r0,r1) in row-major order, thread i takes items i, i+512, ...: lanes
            // (2k,2k+1) = (blank,label) of one cell, a store instruction covers 16 adjacent cells.  The chase has left
            // x = alpha + beta + lp in the staged planes; here: expf(x - beta00), FastEmit, scale, store.  The item
            // index walks (row, rest) incrementally -- one division per thread, none per item.
            const int r0 = t0, r1 = min(t1, Tn);
            const int rows = r1 - r0, per = 2 * Un;
            const int dq = kFusedThreads / per, dr = kFusedThreads - dq * per;   // both even: the parity of `r` never changes
            const int which = tid & 1;                  // 0 = blank, 1 = label
            const float *wplane = which ? WLb : WBb;
            int tt = tid / per, r = tid - tt * per;
            // running staged index and output offset of the item: a pass moves dq rows down and dr/2 columns right,
            // a wrap (r >= per) one more row down and Un columns back
            int ib = idxB(r0 + tt, r >> 1);
            const int dib = -dq * Wd - (dr >> 1) * (Wd + 1), wib = -Wd + Un * (Wd + 1);
            int64_t off = (slab + (int64_t)(r0 + tt) * RS + (r >> 1)) * V;
            const int64_t doff = ((int64_t)dq * RS + (dr >> 1)) * V, woff = (int64_t)(RS - Un) * V;
            IO *const g = static_cast<IO *>(A.grads);
            const double lam1 = 1.0 + (double)A.lam;
            auto patch = [&](auto with_lam) {
                while (tt < rows) {
                    const int u = r >> 1;
                    const bool last_t = (r0 + tt == T1), last_u = (u == U1);
                    const int lab = last_u ? -1 : s_lab[u];
                    // blank: every cell except the last row's inner cells (core.cu:284), and not where the label
                    // store lands on the same element (label == blank: the label gradient wins, core.cu:383-390)
                    const bool go = which ? !last_u : (!(last_t && !last_u) && lab != A.blank);
                    if (go) {
                        float a = expf(wplane[ib] - b00);
                        // (1. + lambda) * a is a double multiply in the reference (core.cu:327-329); with lambda == 0
                        // it returns a unchanged, so the fp64 round trip is skipped without changing a bit
                        if (decltype(with_lam)::value && which) a = (float)(lam1 * (double)a);
                        float v = -a;
                        if (A.scale) v *= sc;
                        g[off + (which ? lab : A.blank)] = io_from_float<IO>(v);
                    }
                    r += dr; tt += dq; ib += dib; off += doff;
                    if (r >= per) { r -= per; ++tt; ib += wib; off += woff; }
                }
            };
            if (has_lam) patch(std::true_type{}); else patch(std::false_type{});
        }
    } else if (A.pair_grads || A.loc) {
        // dense: every cell of rows [t0,t1) incl. padding (zeros); compact: the packed cells of rows < Tn
        const int ncol = compact ? Un : U;
        const int cells = ok ? max((compact ? min(t1, Tn) : t1) - t0, 0) * ncol : (compact ? 0 : (t1 - t0) * ncol);
#pragma unroll 4
        for (int c = tid; c < cells; c += kFusedThreads) {
            const int tt = c / ncol, u = c - tt * ncol;
            const int t = t0 + tt;
            float2 gq = make_float2(0.0f, 0.0f);
            if (live && t < Tn && u < Un) gq = cell_grad(t, u);
            const int64_t cell = slab + (int64_t)t * RS + u;
            if (A.pair_grads) A.pair_grads[cell] = gq;
            if (A.loc) A.loc[cell] = (u < U1) ? s_lab[u] : A.blank;   // last column: the blank (core_compact.cu:424-431)
        }
    }
    stamp(7);
}

// ---- host side -------------------------------------------------------------------------------
constexpr int kFusedMaxDynSmem = 223 * 1024;           // 227 KB per CTA minus the kernel's static shared memory
static long long *g_fused_trace = nullptr;             // diagnostics: see rnnt_b200_debug_fused_trace
void set_fused_trace(long long *buf) { g_fused_trace = buf; }

static size_t fused_zero_offset(int T, int U, int Wd, int nd) {
    const size_t used = sizeof(float) * ((size_t)4 * nd * Wd + (size_t)2 * T) + sizeof(int) * (size_t)U;
    return (used + 127) / 128 * 128;
}
static size_t fused_smem_bytes(int T, int U, int Wd, int nd) {
    return fused_zero_offset(T, U, Wd, nd) + kZeroBytes;
}

// Can the fused kernel take this shape?  Fills `plan` with the derived launch parameters.
bool fused_plan(int N, int T, int U, FusedPlan *plan) {
    if (N < 1 || T < 1 || U < 1 || U > 256) return false;
    const int C = U <= 32 ? 1 : (U <= 64 ? 2 : (U <= 128 ? 4 : 8));
    int Wd = (U + C - 1) / C * C;
    if (Wd & 1) ++Wd;                                   // C == 1: keep the diagonal stride even
    const int nd = (T + Wd + 16 + 1) & ~1;              // diagonals + prefetch overshoot; even, so a plane is whole float4s
    const size_t smem = fused_smem_bytes(T, U, Wd, nd);
    if (smem > 220 * 1024) return false;
    if (((int64_t)T * U + kChunkCells - 1) / kChunkCells > kMaxChunks) return false;
    const int sms = sm_count(current_device());
    // CTAs per lattice: fill every SM (two CTAs per SM when two staged lattices fit in its shared memory)
    const int per_sm = (smem <= 110 * 1024) ? 2 : 1;
    int slices = (per_sm * sms) / N;
    slices = max(1, min(slices, T));
    plan->W = Wd; plan->ring = nd; plan->nw = C; plan->slices = slices; plan->smem = smem;
    return true;
}

template <int KIND, int MODE, int C, typename IO = float>
static cudaError_t launch_fused_kmc(cudaStream_t s, FusedArgs a, size_t smem) {
    static std::atomic<bool> attr_done[kMaxDevices];
    {
        const cudaError_t e = ensure_dyn_smem(k_fused<KIND, MODE, C, IO>, attr_done, kFusedMaxDynSmem);
        if (e != cudaSuccess) return e;
    }
    if (a.slices > 1) {
        // CTAs per lattice: fill every SM with what is actually co-resident (registers can forbid the second
        // CTA that shared memory would allow; a second, partial wave costs more than it brings).  Cached per device.
        struct Occ { size_t smem = ~(size_t)0; int occ = 1; };
        static Occ cache[kMaxDevices];
        static std::mutex mu;
        const int dev = current_device();
        int occ = 1;
        {
            std::lock_guard<std::mutex> lock(mu);
            Occ local;
            Occ &o = dev < kMaxDevices ? cache[dev] : local;
            if (o.smem != smem) {
                int n = 1;
                o.occ = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_fused<KIND, MODE, C, IO>, kFusedThreads, smem) == cudaSuccess && n >= 1) ? n : 1;
                o.smem = smem;
            }
            occ = o.occ;
        }
        a.slices = max(1, min(a.slices, (occ * sm_count(dev)) / a.N));
    }
    dim3 grid(a.slices, a.N);
    k_fused<KIND, MODE, C, IO><<<grid, kFusedThreads, smem, s>>>(a);
    count_launch();
    return cudaGetLastError();
}

template <int KIND, int MODE, typename IO = float>
static cudaError_t launch_fused_km(cudaStream_t s, const FusedArgs &a, size_t smem, int C) {   // (a is copied per launch)
    switch (C) {
        case 1: return launch_fused_kmc<KIND, MODE, 1, IO>(s, a, smem);
        case 2: return launch_fused_kmc<KIND, MODE, 2, IO>(s, a, smem);
        case 4: return launch_fused_kmc<KIND, MODE, 4, IO>(s, a, smem);
        default: return launch_fused_kmc<KIND, MODE, 8, IO>(s, a, smem);
    }
}

cudaError_t launch_fused(cudaStream_t s, const LossJob &j, const FusedPlan &plan) {
    FusedArgs a;
    if (j.io_bf16 && (!j.grads || j.pairs_in || j.mem_pref)) return cudaErrorInvalidValue;   // bf16 i/o: dense gradients only
    a.loss_sum = j.sync_counter ? j.loss_sum : nullptr; a.sync_counter = j.sync_counter;
    a.mem_pref = j.mem_pref; a.lab_pref = j.lab_pref; a.loc = j.loc;
    a.lp = j.lp; a.labels = j.labels; a.xn = j.xn; a.yn = j.yn; a.costs = j.costs; a.grads = j.grads;
    a.pair_grads = j.pair_grads; a.scale = j.scale; a.N = j.N; a.T = j.T; a.U = j.U; a.V = j.V; a.blank = j.blank;
    a.lam = j.lam; a.pairs_in = j.pairs_in; a.guard = j.guard;
    a.slices = (j.grads || j.pair_grads) ? plan.slices : 1; a.Wd = plan.W; a.nd = plan.ring;
    {
        static const int gw_raw = env_int("RNNT_B200_GATHER_WARPS", 0);   // tuning knob, in [1,14]
        const int gw_env = (gw_raw < 1 || gw_raw > kFusedThreads / 32 - 2) ? 0 : gw_raw;
        // fast LSE: the fill (HBM-write bound) outlasts the wavefront, so start it during the gather;
        // exact LSE: the wavefront outlasts the fill, so let every free warp gather and feed it sooner
        // (measured with the TMA fill: starting the fill only when the gather is done is best in both modes)
        a.gw = gw_env ? gw_env : kFusedThreads / 32 - 2;
        if (!j.grads) a.gw = kFusedThreads / 32 - 2;      // nothing to fill: everyone gathers
    }
    a.zoff = (int)(plan.smem - kZeroBytes);
    // TMA row gather when a lattice row (U*V floats) is a 16-byte multiple at a 16-byte aligned address and
    // at least four row buffers fit behind the planes (RNNT_B200_GATHER=ldg forces the LDG gather)
    size_t smem = plan.smem;
    a.nbuf = 0; a.row_off = 0; a.row_stride = 0; a.gwn = 0; a.nb_per = 1;
    {
        static const bool want_tma = !env_is("RNNT_B200_GATHER", 'l');
        static const int nb_env = env_int("RNNT_B200_ROW_BUFS", 0);     // tuning knob: row buffers per gather warp (1 or 2)
        const size_t row = (size_t)j.U * j.V * (j.io_bf16 ? 2 : sizeof(float));
        const size_t stride = (row + 127) / 128 * 128;
        // keep two CTAs per SM where the plan counted on them
        const size_t cap = (plan.smem <= 110 * 1024) ? (size_t)113 * 1024 : (size_t)kFusedMaxDynSmem;
        if (want_tma && !j.pairs_in && (row % 16) == 0 && (reinterpret_cast<uintptr_t>(j.lp) % 16) == 0 && row <= 32 * 1024 &&
            plan.smem + 4 * stride <= cap) {
            const int fit = (int)((cap - plan.smem) / stride);
            // two buffers per gather warp once at least 8 fit (the copy of the next row overlaps the picking of this one
            // and more bytes stay in flight per SM: the gather is bound by that, not by HBM, up to ~20 rows); else one
            a.nb_per = (nb_env == 1 || nb_env == 2) ? nb_env : (fit >= 8 ? 2 : 1);
            if (a.nb_per == 2 && fit < 2) a.nb_per = 1;
            a.gwn = min(kMaxRowBufs, fit / a.nb_per);
            a.nbuf = a.gwn * a.nb_per;
            a.row_off = (int)(plan.smem);
            a.row_stride = (int)stride;
            smem = plan.smem + (size_t)a.nbuf * stride;
        }
    }
    {
        static const bool tma = !env_is("RNNT_B200_FILL", 's');   // RNNT_B200_FILL=stg selects the 256-bit store fill
        a.tma_fill = tma ? 1 : 0;
        static const int fw = env_int("RNNT_B200_FILL_WARPS", 2);
        a.fill_warps = max(1, min(fw, kFusedThreads / 32 - 2));
    }
    a.trace = g_fused_trace;
    { const GuardPoison gp = guard_poison(); a.poison_n = gp.n; a.poison_delta = gp.delta; }
    const bool dense = j.grads != nullptr;
    const int C = plan.nw, kind = j.kind;
    if (j.io_bf16)
        return kind == kFast ? launch_fused_km<kFast, 0, __nv_bfloat16>(s, a, smem, C)
                             : launch_fused_km<kExactDense, 0, __nv_bfloat16>(s, a, smem, C);
    if (kind == kFast)
        return dense ? launch_fused_km<kFast, 0>(s, a, smem, C) : launch_fused_km<kFast, 1>(s, a, smem, C);
    if (kind == kExactCompact)                          // compact layout: (cells,2) gradients only
        return launch_fused_km<kExactCompact, 1>(s, a, smem, C);
    return dense ? launch_fused_km<kExactDense, 0>(s, a, smem, C) : launch_fused_km<kExactDense, 1>(s, a, smem, C);
}

}  // namespace rnnt
