// binding.cpp -- the `_C` operator module: PyTorch tensors in, librnnt_b200.so (C ABI) underneath.
//
// Mirrors the reference's operator boundary /root/reference/pytorch_binding/binding.cpp:
//   rnnt_loss                  (:28-106, pybind :250-254)   same kwargs, checks, messages, returns
//   rnnt_loss_compact          (:109-207, pybind :256-262)
//   rnnt_loss_compact_backward (:209-247, pybind :264-268)
// Differences that are deliberate: a device guard and the *current* stream are used everywhere
// (the reference sets no guard for the dense path, :77, and launches compact kernels on the legacy
// default stream, core.h:41-60); no dense zeros_like / torch::zeros passes (the kernels write every
// element); compact shapes are validated with one small device->host copy instead of four .item()s.
// Extra entry points (rnnt_loss_dense, rnnt_gather_forward/backward) serve the fused python-level
// paths of warp_rnnt_b200/__init__.py.
#include <algorithm>
#include <mutex>
#include <string>
#include <tuple>

#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include "../../include/rnnt_b200.h"

namespace {

void check4(const at::Tensor &xs, const at::Tensor &ys, const at::Tensor &xn, const at::Tensor &yn,
            bool allow_bf16 = false) {
    // order as in the reference (binding.cpp:31-46): contiguity, then dtypes, then device
    TORCH_CHECK(xs.is_contiguous(), "xs must be contiguous");
    TORCH_CHECK(ys.is_contiguous(), "ys must be contiguous");
    TORCH_CHECK(xn.is_contiguous(), "xn must be contiguous");
    TORCH_CHECK(yn.is_contiguous(), "yn must be contiguous");
    TORCH_CHECK(xs.scalar_type() == at::ScalarType::Float || (allow_bf16 && xs.scalar_type() == at::ScalarType::BFloat16),
                "xs must be a Float tensor");
    TORCH_CHECK(ys.scalar_type() == at::ScalarType::Int, "ys must be a Int tensor");
    TORCH_CHECK(xn.scalar_type() == at::ScalarType::Int, "xn must be a Int tensor");
    TORCH_CHECK(yn.scalar_type() == at::ScalarType::Int, "yn must be a Int tensor");
    TORCH_CHECK(xs.device().is_cuda(), "xs must be located in the CUDA");
    TORCH_CHECK(ys.device().is_cuda(), "ys must be located in the CUDA");
    TORCH_CHECK(xn.device().is_cuda(), "xn must be located in the CUDA");
    TORCH_CHECK(yn.device().is_cuda(), "yn must be located in the CUDA");
}

void check_dense_shapes(const at::Tensor &xs, const at::Tensor &ys, const at::Tensor &xn, const at::Tensor &yn) {
    TORCH_CHECK(xs.dim() == 4, "xs must have 4 dimensions");
    TORCH_CHECK(xn.numel() == xs.size(0), "xn shape must be equal (N,)");
    TORCH_CHECK(yn.numel() == xs.size(0), "yn shape must be equal (N,)");
    TORCH_CHECK(ys.dim() == 2 && xs.size(2) == ys.size(1) + 1, "ys shape (N, U-1) mismatched with xs (N, T, U, V)");
}

at::Tensor workspace_for(const at::Tensor &like, int64_t cells, int64_t N) {
    const size_t bytes = rnnt_b200_workspace_bytes(cells, (int)N);
    return at::empty({(int64_t)bytes}, like.options().dtype(at::kByte));
}

void check_status(int status) {
    TORCH_CHECK(status == RNNT_STATUS_SUCCESS, "rnnt_loss status " + std::to_string(status) + " (" +
                                                   rnnt_b200_status_string(status) + ")");
}

void *current_stream(const at::Tensor &t) {
    return (void *)c10::cuda::getCurrentCUDAStream(t.device().index()).stream();
}

// Tickets for the in-kernel loss reduction (rnnt_b200_loss_dense_reduced): a small ring of self-resetting device
// counters per device, zeroed once; consecutive calls take consecutive slots so that calls running concurrently
// on different streams (or captured into different CUDA graphs) never share one.
unsigned int *next_sync_counter(const at::Tensor &like) {
    constexpr int kSlots = 256, kMaxDev = 64;
    static std::mutex mu;
    static at::Tensor ring[kMaxDev];
    static unsigned next[kMaxDev] = {};
    const int dev = like.device().index();
    if (dev < 0 || dev >= kMaxDev) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!ring[dev].defined()) ring[dev] = at::zeros({kSlots}, like.options().dtype(at::kInt));
    return reinterpret_cast<unsigned int *>(ring[dev].data_ptr<int>()) + (next[dev]++ % kSlots);
}

// dense forward (+ gradients), optional per-sample scale, explicit LSE mode; loss_sum: (1) tensor or undefined
std::tuple<at::Tensor, at::Tensor> loss_dense_impl(const at::Tensor &xs, const at::Tensor &ys, const at::Tensor &xn,
                                                   const at::Tensor &yn, int blank, float fastemit_lambda,
                                                   const c10::optional<at::Tensor> &scale, bool want_grads,
                                                   int lse_mode, at::Tensor loss_sum = at::Tensor(),
                                                   bool allow_bf16 = false) {
    check4(xs, ys, xn, yn, allow_bf16);
    check_dense_shapes(xs, ys, xn, yn);
    const c10::cuda::CUDAGuard guard(xs.device());
    const int64_t N = xs.size(0), T = xs.size(1), U = xs.size(2), V = xs.size(3);
    const bool bf16 = xs.scalar_type() == at::ScalarType::BFloat16;
    at::Tensor costs = at::empty({N}, xs.options().dtype(at::kFloat));
    at::Tensor grads = want_grads ? at::empty_like(xs) : at::empty({0}, xs.options());
    if (N == 0) return std::make_tuple(costs, grads);
    TORCH_CHECK(!bf16 || (want_grads && blank != -1), "bfloat16 xs: dense (N,T,U,V) layout with gradients only");
    const float *sc = nullptr;
    if (scale.has_value() && scale->defined()) {
        TORCH_CHECK(scale->is_contiguous() && scale->scalar_type() == at::ScalarType::Float &&
                        scale->device() == xs.device() && scale->numel() == N,
                    "grad_scale must be a contiguous Float tensor of shape (N,) on the device of xs");
        sc = scale->data_ptr<float>();
    }
    int status;
    if (blank == -1) {
        // gathered (N,T,U,2) form, binding.cpp:81-90
        TORCH_CHECK(V == 2, "xs must have values only for blank and label");
        at::Tensor ws = workspace_for(xs, N * T * U, N);
        status = rnnt_b200_loss_pairs(current_stream(xs), ws.data_ptr(), (size_t)ws.numel(), xs.data_ptr<float>(),
                                      xn.data_ptr<int>(), yn.data_ptr<int>(), costs.data_ptr<float>(),
                                      want_grads ? grads.data_ptr<float>() : nullptr, (int)N, (int)T, (int)U,
                                      fastemit_lambda, lse_mode);
        check_status(status);
        if (want_grads && sc) grads.mul_(scale->view({-1, 1, 1, 1}));
    } else {
        TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V) (or -1 for the gathered layout)");
        at::Tensor ws = workspace_for(xs, N * T * U, N);
        float *ls = loss_sum.defined() ? loss_sum.data_ptr<float>() : nullptr;
        if (bf16)
            status = rnnt_b200_loss_dense_bf16(current_stream(xs), ws.data_ptr(), (size_t)ws.numel(), xs.data_ptr(),
                                               ys.data_ptr<int>(), xn.data_ptr<int>(), yn.data_ptr<int>(),
                                               costs.data_ptr<float>(), grads.data_ptr(), sc, ls,
                                               ls ? next_sync_counter(xs) : nullptr, (int)N, (int)T, (int)U, (int)V,
                                               blank, fastemit_lambda, lse_mode);
        else
        status = rnnt_b200_loss_dense_reduced(current_stream(xs), ws.data_ptr(), (size_t)ws.numel(), xs.data_ptr<float>(),
                                              ys.data_ptr<int>(), xn.data_ptr<int>(), yn.data_ptr<int>(),
                                              costs.data_ptr<float>(), want_grads ? grads.data_ptr<float>() : nullptr,
                                              sc, ls, ls ? next_sync_counter(xs) : nullptr, (int)N, (int)T, (int)U,
                                              (int)V, blank, fastemit_lambda, lse_mode);
        check_status(status);
    }
    return std::make_tuple(costs, grads);
}

// ---- reference-compatible entry points --------------------------------------------------

std::tuple<at::Tensor, at::Tensor> rnnt_loss(const at::Tensor &xs, const at::Tensor &ys, const at::Tensor &xn,
                                             const at::Tensor &yn, const int blank, const float fastemit_lambda) {
    return loss_dense_impl(xs, ys, xn, yn, blank, fastemit_lambda, c10::nullopt, true, RNNT_LSE_AUTO);
}

std::tuple<at::Tensor, at::Tensor, at::Tensor> rnnt_loss_compact(const at::Tensor &xs, const at::Tensor &ys,
                                                                 const at::Tensor &xn, const at::Tensor &yn,
                                                                 const int blank, const float fastemit_lambda,
                                                                 const bool required_grad, int hint_T, int hint_U) {
    check4(xs, ys, xn, yn);
    TORCH_CHECK(xs.dim() == 2, "xs must have 2 dimensions");
    TORCH_CHECK(xn.dim() == 1 && yn.dim() == 1 && xn.size(0) == yn.size(0), "xn and yn shape must be equal (N,)");
    const c10::cuda::CUDAGuard guard(xs.device());
    const int64_t N = xn.size(0), STU = xs.size(0), V = xs.size(1);
    TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V)");
    void *stream = current_stream(xs);
    at::Tensor costs = at::empty({N}, xs.options());
    at::Tensor loc = at::empty({STU}, xs.options().dtype(at::kLong));
    // like the reference (binding.cpp:196-201): without required_grad the returned "grads" is a
    // placeholder the caller must not use
    at::Tensor grads = required_grad ? at::empty({STU, 2}, xs.options()) : at::empty({0}, xs.options());
    if (N == 0) return std::make_tuple(costs, grads, loc);
    int max_T = 0, max_U = 0;
    // shape validation: one 16-byte device->host copy (the reference needs four .item() syncs) -- or none at all
    // when the caller vouches for upper bounds of xn and yn+1 (sync-free, CUDA-graph capturable)
    if (hint_T > 0 && hint_U > 0) {
        max_T = hint_T;
        max_U = hint_U;
    } else {
        at::Tensor scratch = at::empty({2 * N}, xs.options().dtype(at::kLong));
        at::Tensor totals = at::empty({4}, xs.options().dtype(at::kInt));
        check_status(rnnt_b200_compact_totals(stream, xn.data_ptr<int>(), yn.data_ptr<int>(), (int)N,
                                              scratch.data_ptr<int64_t>(), totals.data_ptr<int>()));
        at::Tensor h = totals.cpu();
        const int *t = h.data_ptr<int>();
        TORCH_CHECK(ys.numel() == t[1], "ys shape must be equal to (sum(yn), )");
        TORCH_CHECK(STU == t[0], "xs shape mismatch with (\\sum{xn*(yn+1)}, )");
        max_T = t[2];
        max_U = t[3];
    }
    at::Tensor ws = workspace_for(xs, STU, N);
    check_status(rnnt_b200_compact_forward(stream, ws.data_ptr(), (size_t)ws.numel(), xs.data_ptr<float>(),
                                           ys.data_ptr<int>(), xn.data_ptr<int>(), yn.data_ptr<int>(),
                                           costs.data_ptr<float>(), required_grad ? grads.data_ptr<float>() : nullptr,
                                           loc.data_ptr<int64_t>(), nullptr, STU, (int)N, (int)V, blank,
                                           fastemit_lambda, RNNT_LSE_AUTO, max_T, max_U));
    return std::make_tuple(costs, grads, loc);
}

at::Tensor rnnt_loss_compact_backward(const at::Tensor &grad_cost, const at::Tensor &grad_xs,
                                      const at::Tensor &cum_lens, const at::Tensor &loc, int64_t V, int blank) {
    TORCH_CHECK(grad_cost.is_contiguous(), "grad_cost must be contiguous");
    TORCH_CHECK(grad_xs.is_contiguous(), "grad_xs must be contiguous");
    TORCH_CHECK(loc.is_contiguous(), "loc must be contiguous");
    TORCH_CHECK(grad_cost.scalar_type() == at::ScalarType::Float, "grad_cost must be a Float tensor");
    TORCH_CHECK(grad_xs.scalar_type() == at::ScalarType::Float, "grad_xs must be a Float tensor");
    TORCH_CHECK(loc.scalar_type() == at::ScalarType::Long, "loc must be a Long tensor");
    TORCH_CHECK(grad_cost.device().is_cuda(), "grad_cost must be located in the CUDA");
    TORCH_CHECK(grad_xs.device().is_cuda(), "grad_xs must be located in the CUDA");
    TORCH_CHECK(cum_lens.device().is_cuda(), "cum_lens must be located in the CUDA");
    TORCH_CHECK(loc.device().is_cuda(), "loc must be located in the CUDA");
    TORCH_CHECK(grad_cost.dim() == 1, "grad_cost must have 1 dimensions");
    TORCH_CHECK(grad_xs.dim() == 2, "grad must have 2 dimensions");
    TORCH_CHECK(grad_xs.size(0) == loc.size(0), "grad and loc must be equal in dim=0");
    TORCH_CHECK(cum_lens.is_contiguous() && cum_lens.scalar_type() == at::ScalarType::Int &&
                    cum_lens.numel() == grad_cost.size(0),
                "cum_lens must be a contiguous Int tensor of shape (N,)");
    TORCH_CHECK(grad_xs.size(1) == 2, "grad must have shape (STU, 2)");
    TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V)");
    const c10::cuda::CUDAGuard guard(grad_cost.device());
    const int64_t N = grad_cost.size(0), STU = grad_xs.size(0);
    at::Tensor out = at::empty({STU, V}, grad_cost.options());
    check_status(rnnt_b200_compact_backward(current_stream(grad_cost), grad_cost.data_ptr<float>(),
                                            grad_xs.data_ptr<float>(), loc.data_ptr<int64_t>(),
                                            cum_lens.data_ptr<int>(), out.data_ptr<float>(), STU, (int)N, (int)V,
                                            blank));
    return out;
}

// ---- native extras used by warp_rnnt_b200/__init__.py ------------------------------------

std::tuple<at::Tensor, at::Tensor> rnnt_loss_dense(const at::Tensor &xs, const at::Tensor &ys, const at::Tensor &xn,
                                                   const at::Tensor &yn, int blank, float fastemit_lambda,
                                                   const c10::optional<at::Tensor> &grad_scale, bool want_grads,
                                                   int lse_mode) {
    return loss_dense_impl(xs, ys, xn, yn, blank, fastemit_lambda, grad_scale, want_grads, lse_mode);
}

// loss + dense gradients + reduced loss in one call: (costs (N), grads like xs or empty, loss (1) = sum costs*scale)
std::tuple<at::Tensor, at::Tensor, at::Tensor> rnnt_loss_fused(const at::Tensor &xs, const at::Tensor &ys,
                                                               const at::Tensor &xn, const at::Tensor &yn, int blank,
                                                               float fastemit_lambda,
                                                               const c10::optional<at::Tensor> &grad_scale,
                                                               bool want_grads, int lse_mode) {
    TORCH_CHECK(blank >= 0, "rnnt_loss_fused takes the dense (N,T,U,V) layout");
    TORCH_CHECK(xs.device().is_cuda(), "xs must be located in the CUDA");
    const c10::cuda::CUDAGuard guard(xs.device());
    at::Tensor loss = at::empty({1}, xs.options().dtype(at::kFloat));
    if (xs.dim() == 4 && xs.size(0) == 0) loss.zero_();
    auto r = loss_dense_impl(xs, ys, xn, yn, blank, fastemit_lambda, grad_scale, want_grads, lse_mode, loss, true);
    return std::make_tuple(std::get<0>(r), std::get<1>(r), loss);
}

// in place: grads[n] *= grad_out[n] / applied[n] where they differ (grad_out with one element: one scalar for all)
void rnnt_rescale_(at::Tensor grads, const at::Tensor &grad_out, const c10::optional<at::Tensor> &applied) {
    const bool bf16 = grads.scalar_type() == at::ScalarType::BFloat16;
    TORCH_CHECK(grads.is_contiguous() && (grads.scalar_type() == at::ScalarType::Float || bf16) &&
                    grads.device().is_cuda() && grads.dim() >= 1,
                "grads must be a contiguous CUDA Float (or BFloat16) tensor");
    const int64_t N = grads.size(0);
    TORCH_CHECK(grad_out.is_contiguous() && grad_out.scalar_type() == at::ScalarType::Float &&
                    grad_out.device() == grads.device() && (grad_out.numel() == N || grad_out.numel() == 1),
                "grad_out must be a contiguous Float tensor with N elements (or one) on the device of grads");
    const float *ap = nullptr;
    if (applied.has_value() && applied->defined()) {
        TORCH_CHECK(applied->is_contiguous() && applied->scalar_type() == at::ScalarType::Float &&
                        applied->device() == grads.device() && applied->numel() == N,
                    "applied must be a contiguous Float tensor of shape (N,) on the device of grads");
        ap = applied->data_ptr<float>();
    }
    if (N == 0) return;
    const c10::cuda::CUDAGuard guard(grads.device());
    check_status(rnnt_b200_rescale(current_stream(grads), grads.data_ptr(), grad_out.data_ptr<float>(),
                                   (grad_out.numel() == 1 && N != 1) ? 0 : 1, ap, (int)N, grads.numel() / N,
                                   bf16 ? 2 : 4));
}

std::tuple<at::Tensor, at::Tensor> rnnt_gather_forward(const at::Tensor &xs, const at::Tensor &ys,
                                                       const at::Tensor &xn, const at::Tensor &yn, int blank,
                                                       float fastemit_lambda, bool want_grads, int lse_mode) {
    check4(xs, ys, xn, yn);
    check_dense_shapes(xs, ys, xn, yn);
    const c10::cuda::CUDAGuard guard(xs.device());
    const int64_t N = xs.size(0), T = xs.size(1), U = xs.size(2), V = xs.size(3);
    TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V)");
    at::Tensor costs = at::empty({N}, xs.options());
    at::Tensor pg = want_grads ? at::empty({N, T, U, 2}, xs.options()) : at::empty({0}, xs.options());
    if (N == 0) return std::make_tuple(costs, pg);
    at::Tensor ws = workspace_for(xs, N * T * U, N);
    check_status(rnnt_b200_gather_forward(current_stream(xs), ws.data_ptr(), (size_t)ws.numel(),
                                          xs.data_ptr<float>(), ys.data_ptr<int>(), xn.data_ptr<int>(),
                                          yn.data_ptr<int>(), costs.data_ptr<float>(),
                                          want_grads ? pg.data_ptr<float>() : nullptr, (int)N, (int)T, (int)U, (int)V,
                                          blank, fastemit_lambda, lse_mode));
    return std::make_tuple(costs, pg);
}

// loss from un-normalised logits, float32 or bfloat16: (costs (N), lse (N,T,U), pair_grads (N,T,U,2) or empty), all
// three float32
std::tuple<at::Tensor, at::Tensor, at::Tensor> rnnt_logits_forward(const at::Tensor &xs, const at::Tensor &ys,
                                                                   const at::Tensor &xn, const at::Tensor &yn,
                                                                   int blank, float fastemit_lambda, bool want_grads,
                                                                   int lse_mode) {
    check4(xs, ys, xn, yn, true);
    check_dense_shapes(xs, ys, xn, yn);
    const c10::cuda::CUDAGuard guard(xs.device());
    const int64_t N = xs.size(0), T = xs.size(1), U = xs.size(2), V = xs.size(3);
    TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V)");
    const at::TensorOptions f32 = xs.options().dtype(at::kFloat);
    at::Tensor costs = at::empty({N}, f32);
    at::Tensor lse = at::empty({N, T, U}, f32);
    at::Tensor pg = want_grads ? at::empty({N, T, U, 2}, f32) : at::empty({0}, f32);
    if (N == 0) return std::make_tuple(costs, lse, pg);
    at::Tensor ws = workspace_for(xs, N * T * U, N);
    float *pgp = want_grads ? pg.data_ptr<float>() : nullptr;
    if (xs.scalar_type() == at::ScalarType::BFloat16)
        check_status(rnnt_b200_logits_forward_bf16(current_stream(xs), ws.data_ptr(), (size_t)ws.numel(), xs.data_ptr(),
                                                   ys.data_ptr<int>(), xn.data_ptr<int>(), yn.data_ptr<int>(),
                                                   costs.data_ptr<float>(), lse.data_ptr<float>(), pgp, (int)N, (int)T,
                                                   (int)U, (int)V, blank, fastemit_lambda, lse_mode));
    else
        check_status(rnnt_b200_logits_forward(current_stream(xs), ws.data_ptr(), (size_t)ws.numel(), xs.data_ptr<float>(),
                                              ys.data_ptr<int>(), xn.data_ptr<int>(), yn.data_ptr<int>(),
                                              costs.data_ptr<float>(), lse.data_ptr<float>(), pgp, (int)N, (int)T,
                                              (int)U, (int)V, blank, fastemit_lambda, lse_mode));
    return std::make_tuple(costs, lse, pg);
}

// d loss / d logits, of the dtype of xs (float32 or bfloat16); lse, pair_grads and grad_out float32
at::Tensor rnnt_logits_backward(const at::Tensor &xs, const at::Tensor &lse, const at::Tensor &pair_grads,
                                const at::Tensor &ys, const at::Tensor &grad_out, int blank) {
    const bool bf16 = xs.scalar_type() == at::ScalarType::BFloat16;
    TORCH_CHECK(xs.is_contiguous() && (xs.scalar_type() == at::ScalarType::Float || bf16) && xs.device().is_cuda() &&
                    xs.dim() == 4,
                "xs must be a contiguous CUDA Float tensor of shape (N, T, U, V)");
    const int64_t N = xs.size(0), T = xs.size(1), U = xs.size(2), V = xs.size(3);
    TORCH_CHECK(lse.is_contiguous() && lse.scalar_type() == at::ScalarType::Float && lse.device() == xs.device() &&
                    lse.numel() == N * T * U,
                "lse must be a contiguous Float tensor of shape (N, T, U) on the device of xs");
    TORCH_CHECK(pair_grads.is_contiguous() && pair_grads.scalar_type() == at::ScalarType::Float &&
                    pair_grads.device() == xs.device() && pair_grads.numel() == N * T * U * 2,
                "pair_grads must be a contiguous Float tensor of shape (N, T, U, 2) on the device of xs");
    TORCH_CHECK(ys.is_contiguous() && ys.scalar_type() == at::ScalarType::Int && ys.device() == xs.device() &&
                    ys.dim() == 2 && ys.size(0) == N && ys.size(1) + 1 == U,
                "ys must be a contiguous Int tensor of shape (N, U-1) on the device of xs");
    TORCH_CHECK(grad_out.is_contiguous() && grad_out.scalar_type() == at::ScalarType::Float &&
                    grad_out.device() == xs.device() && grad_out.numel() == N,
                "grad_out must be a contiguous Float tensor of shape (N,)");
    TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V)");
    const c10::cuda::CUDAGuard guard(xs.device());
    at::Tensor out = at::empty_like(xs);
    if (bf16)
        check_status(rnnt_b200_logits_backward_bf16(current_stream(xs), xs.data_ptr(), lse.data_ptr<float>(),
                                                    pair_grads.data_ptr<float>(), ys.data_ptr<int>(),
                                                    grad_out.data_ptr<float>(), out.data_ptr(), (int)N, (int)T, (int)U,
                                                    (int)V, blank));
    else
        check_status(rnnt_b200_logits_backward(current_stream(xs), xs.data_ptr<float>(), lse.data_ptr<float>(),
                                               pair_grads.data_ptr<float>(), ys.data_ptr<int>(), grad_out.data_ptr<float>(),
                                               out.data_ptr<float>(), (int)N, (int)T, (int)U, (int)V, blank));
    return out;
}

// compact packing of the joint input: (x (STU,H), mem_pref (N) int64).  stu < 0: STU is read back from the device
// (one 16-byte copy); stu >= 0: trusted, no host sync.
std::tuple<at::Tensor, at::Tensor> rnnt_joint_pack(const at::Tensor &f, const at::Tensor &g, const at::Tensor &lf,
                                                   const at::Tensor &lg, int64_t stu) {
    TORCH_CHECK(f.is_contiguous() && g.is_contiguous() && lf.is_contiguous() && lg.is_contiguous(), "inputs must be contiguous");
    TORCH_CHECK(f.scalar_type() == at::ScalarType::Float && g.scalar_type() == at::ScalarType::Float,
                "f and g must be Float tensors");
    TORCH_CHECK(lf.scalar_type() == at::ScalarType::Int && lg.scalar_type() == at::ScalarType::Int,
                "lf and lg must be Int tensors");
    TORCH_CHECK(f.device().is_cuda() && g.device() == f.device() && lf.device() == f.device() && lg.device() == f.device(),
                "f, g, lf, lg must be on the same CUDA device");
    TORCH_CHECK(f.dim() == 3 && g.dim() == 3 && f.size(0) == g.size(0) && f.size(2) == g.size(2),
                "f must be (N, T, H) and g (N, U+1, H)");
    const int64_t N = f.size(0), T = f.size(1), U1 = g.size(1), H = f.size(2);
    TORCH_CHECK(lf.numel() == N && lg.numel() == N, "lf and lg must have N elements");
    const c10::cuda::CUDAGuard guard(f.device());
    void *stream = current_stream(f);
    at::Tensor scratch = at::empty({2 * std::max<int64_t>(N, 1)}, f.options().dtype(at::kLong));
    if (N == 0) return std::make_tuple(at::empty({0, H}, f.options()), scratch);
    if (stu < 0) {
        at::Tensor totals = at::empty({4}, f.options().dtype(at::kInt));
        check_status(rnnt_b200_joint_pack(stream, nullptr, nullptr, lf.data_ptr<int>(), lg.data_ptr<int>(),
                                          scratch.data_ptr<int64_t>(), totals.data_ptr<int>(), nullptr, (int)N, (int)T,
                                          (int)U1, (int)H, 0));
        at::Tensor h = totals.cpu();
        const int *t = h.data_ptr<int>();
        TORCH_CHECK(t[2] <= T && t[3] <= U1, "lf / lg exceed the shapes of f / g");
        stu = t[0];
    }
    at::Tensor x = at::empty({stu, H}, f.options());
    check_status(rnnt_b200_joint_pack(stream, f.data_ptr<float>(), g.data_ptr<float>(), lf.data_ptr<int>(),
                                      lg.data_ptr<int>(), scratch.data_ptr<int64_t>(), nullptr, x.data_ptr<float>(), (int)N,
                                      (int)T, (int)U1, (int)H, stu));
    return std::make_tuple(x, scratch.narrow(0, 0, N));
}

std::tuple<at::Tensor, at::Tensor> rnnt_joint_pack_backward(const at::Tensor &dx, const at::Tensor &lf,
                                                            const at::Tensor &lg, const at::Tensor &mem_pref,
                                                            int64_t T, int64_t U1) {
    TORCH_CHECK(dx.is_contiguous() && dx.scalar_type() == at::ScalarType::Float && dx.device().is_cuda() && dx.dim() == 2,
                "dx must be a contiguous CUDA Float tensor of shape (STU, H)");
    TORCH_CHECK(mem_pref.is_contiguous() && mem_pref.scalar_type() == at::ScalarType::Long && mem_pref.device() == dx.device(),
                "mem_pref must be a contiguous Long tensor on the device of dx");
    const int64_t N = mem_pref.numel(), H = dx.size(1);
    TORCH_CHECK(lf.numel() == N && lg.numel() == N && lf.is_contiguous() && lg.is_contiguous() &&
                    lf.scalar_type() == at::ScalarType::Int && lg.scalar_type() == at::ScalarType::Int,
                "lf and lg must be contiguous Int tensors with N elements");
    const c10::cuda::CUDAGuard guard(dx.device());
    at::Tensor df = at::empty({N, T, H}, dx.options()), dg = at::empty({N, U1, H}, dx.options());
    check_status(rnnt_b200_joint_pack_backward(current_stream(dx), dx.data_ptr<float>(), lf.data_ptr<int>(),
                                               lg.data_ptr<int>(), mem_pref.data_ptr<int64_t>(), df.data_ptr<float>(),
                                               dg.data_ptr<float>(), (int)N, (int)T, (int)U1, (int)H));
    return std::make_tuple(df, dg);
}

at::Tensor rnnt_gather_backward(const at::Tensor &pair_grads, const at::Tensor &ys, const at::Tensor &grad_out,
                                int64_t V, int blank, bool accumulate, const c10::optional<at::Tensor> &yn) {
    TORCH_CHECK(pair_grads.is_contiguous() && pair_grads.scalar_type() == at::ScalarType::Float &&
                    pair_grads.device().is_cuda() && pair_grads.dim() == 4 && pair_grads.size(3) == 2,
                "pair_grads must be a contiguous CUDA Float tensor of shape (N, T, U, 2)");
    TORCH_CHECK(ys.is_contiguous() && ys.scalar_type() == at::ScalarType::Int && ys.device() == pair_grads.device(),
                "ys must be a contiguous Int tensor on the device of pair_grads");
    TORCH_CHECK(grad_out.is_contiguous() && grad_out.scalar_type() == at::ScalarType::Float &&
                    grad_out.device() == pair_grads.device() && grad_out.numel() == pair_grads.size(0),
                "grad_out must be a contiguous Float tensor of shape (N,)");
    const int64_t N = pair_grads.size(0), T = pair_grads.size(1), U = pair_grads.size(2);
    TORCH_CHECK(ys.dim() == 2 && ys.size(0) == N && ys.size(1) + 1 == U, "ys shape (N, U-1) mismatched");
    TORCH_CHECK(blank >= 0 && blank < V, "blank must be in [0, V)");
    const int *ynp = nullptr;
    if (yn.has_value() && yn->defined()) {
        TORCH_CHECK(yn->is_contiguous() && yn->scalar_type() == at::ScalarType::Int && yn->device() == pair_grads.device() &&
                        yn->numel() == N,
                    "yn must be a contiguous Int tensor of shape (N,) on the device of pair_grads");
        ynp = yn->data_ptr<int>();
    }
    const c10::cuda::CUDAGuard guard(pair_grads.device());
    at::Tensor out = at::empty({N, T, U, V}, pair_grads.options());
    check_status(rnnt_b200_gather_backward(current_stream(pair_grads), pair_grads.data_ptr<float>(),
                                           ys.data_ptr<int>(), grad_out.data_ptr<float>(), out.data_ptr<float>(),
                                           (int)N, (int)T, (int)U, (int)V, blank, accumulate ? 1 : 0, ynp));
    return out;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    namespace py = pybind11;
    m.def("rnnt_loss", &rnnt_loss, "B200 RNN-Transducer loss (forward and gradients).", py::arg("xs"), py::arg("ys"),
          py::arg("xn"), py::arg("yn"), py::arg("blank") = 0, py::arg("fastemit_lambda") = 0.0);
    m.def("rnnt_loss_compact", &rnnt_loss_compact, "B200 RNN-Transducer loss in compact layout.", py::arg("xs"),
          py::arg("ys"), py::arg("xn"), py::arg("yn"), py::arg("blank") = 0, py::arg("fastemit_lambda") = 0.0,
          py::arg("required_grad") = true, py::arg("max_T") = 0, py::arg("max_U") = 0);
    m.def("rnnt_loss_compact_backward", &rnnt_loss_compact_backward,
          "B200 RNN-Transducer loss backward for compact layout", py::arg("grad_costs"), py::arg("grad_xs"),
          py::arg("cumSum"), py::arg("loc"), py::arg("V"), py::arg("blank") = 0);
    m.def("rnnt_loss_dense", &rnnt_loss_dense, py::arg("xs"), py::arg("ys"), py::arg("xn"), py::arg("yn"),
          py::arg("blank") = 0, py::arg("fastemit_lambda") = 0.0, py::arg("grad_scale") = py::none(),
          py::arg("want_grads") = true, py::arg("lse_mode") = 0);
    m.def("rnnt_loss_fused", &rnnt_loss_fused, py::arg("xs"), py::arg("ys"), py::arg("xn"), py::arg("yn"),
          py::arg("blank") = 0, py::arg("fastemit_lambda") = 0.0, py::arg("grad_scale") = py::none(),
          py::arg("want_grads") = true, py::arg("lse_mode") = 0);
    m.def("rnnt_rescale_", &rnnt_rescale_, py::arg("grads"), py::arg("grad_out"), py::arg("applied") = py::none());
    m.def("rnnt_logits_forward", &rnnt_logits_forward, py::arg("xs"), py::arg("ys"), py::arg("xn"), py::arg("yn"),
          py::arg("blank") = 0, py::arg("fastemit_lambda") = 0.0, py::arg("want_grads") = true, py::arg("lse_mode") = 0);
    m.def("rnnt_logits_backward", &rnnt_logits_backward, py::arg("xs"), py::arg("lse"), py::arg("pair_grads"),
          py::arg("ys"), py::arg("grad_out"), py::arg("blank") = 0);
    m.def("rnnt_joint_pack", &rnnt_joint_pack, py::arg("f"), py::arg("g"), py::arg("lf"), py::arg("lg"), py::arg("stu") = -1);
    m.def("rnnt_joint_pack_backward", &rnnt_joint_pack_backward, py::arg("dx"), py::arg("lf"), py::arg("lg"),
          py::arg("mem_pref"), py::arg("T"), py::arg("U1"));
    m.def("rnnt_gather_forward", &rnnt_gather_forward, py::arg("xs"), py::arg("ys"), py::arg("xn"), py::arg("yn"),
          py::arg("blank") = 0, py::arg("fastemit_lambda") = 0.0, py::arg("want_grads") = true,
          py::arg("lse_mode") = 0);
    m.def("rnnt_gather_backward", &rnnt_gather_backward, py::arg("pair_grads"), py::arg("ys"), py::arg("grad_out"),
          py::arg("V"), py::arg("blank") = 0, py::arg("accumulate") = false, py::arg("yn") = py::none());
    m.def("set_lse_mode", [](int mode) { rnnt_b200_set_lse_mode(mode); }, py::arg("mode"));
    m.def("get_lse_mode", []() { return rnnt_b200_get_lse_mode(); });
    m.def("launch_count", []() { return rnnt_b200_launch_count(); });
    m.def("version", []() { return std::string(rnnt_b200_version()); });
}
