"""rnnt_loss_from_logits with bfloat16 logits: bf16 in, bf16 logit gradient out, float32 costs / lse / pair gradients.

The contract: every bf16 value is converted exactly to float32 and the arithmetic is the float32 path's, in its order.
So on bf16 logits xb the bf16 path returns the float32 path's costs, lse and pair gradients for xb.float() bit for bit,
in both LSE modes and for every kernel variant, and its logit gradient is the float32 one rounded once to bf16.
Against the fp64 oracle on the same values: costs |d|/|ref| <= 1e-5, gradients |d| <= 2^-8 |g| + 1e-4 + 2 gtol(T,U)
(one bf16 rounding on top of the float32 path's tolerance in tests/test_gpu_logits.py).

The GPU tests are marked one by one: the C ABI validation test at the end runs without a GPU."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from tests.test_gpu_logits import SHAPES, make

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "warp_rnnt_b200", "lib", "librnnt_b200.so")
gpu = pytest.mark.gpu

# SHAPES plus a V = 1024 row (vec4 loop with whole load batches, 16-byte gradient vectors) and V = 1001 (32 lanes on
# scalar loads, one-element gradient vectors).  With SHAPES this covers every k_lse_pairs variant -- SUB 1 (V = 5, 6,
# 7), SUB 8 (V = 50), SUB 32 (V = 300, 1001, 1024, 5000), vec4 or not, one vector per lane (V = 28, 64) -- and every
# bf16 k_expand_logits width: V = 5, 7, 1001 -> 1; 6, 50 -> 2; 28, 300 -> 4; 64, 1024, 5000 -> 8.
BIT_SHAPES = SHAPES + [(2, 30, 12, 1024, 0, 0.0), (2, 20, 6, 1001, 0, 0.0)]


def gtol(T, U):
    return 2e-5 + 6e-6 * (T + U)


@pytest.fixture(scope="module")
def w():
    import warp_rnnt_b200
    return warp_rnnt_b200


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def same_bits(a, b):
    """dtype and every bit equal (also tells -0 from +0)."""
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    as_int = {torch.float32: torch.int32, torch.bfloat16: torch.int16}[a.dtype]
    return torch.equal(a.view(as_int), b.view(as_int))


def check_bits(w, xb, x32, args, blank, lam, go):
    """The operator pair on bf16 logits xb against the same on float32 logits x32 = the same values."""
    cb, lb, pb = w._C.rnnt_logits_forward(xb, *args, blank, lam, True, 0)
    c3, l3, p3 = w._C.rnnt_logits_forward(x32, *args, blank, lam, True, 0)
    assert same_bits(cb, c3) and same_bits(lb, l3) and same_bits(pb, p3)
    gb = w._C.rnnt_logits_backward(xb, lb, pb, args[0], go, blank)
    g3 = w._C.rnnt_logits_backward(x32, l3, p3, args[0], go, blank)
    assert gb.dtype == torch.bfloat16
    assert same_bits(gb, g3.to(torch.bfloat16))


@gpu
@pytest.mark.parametrize("mode", ["exact", "fast"])
@pytest.mark.parametrize("shape", BIT_SHAPES)
def test_bf16_bit_identical_to_f32_path(w, shape, mode):
    N, T, U, V, blank, lam = shape
    x, ys, xn, yn = make(N, T, U, V, seed=T + V + 1, blank=blank)
    xb = cu(x).to(torch.bfloat16)
    go = cu(np.linspace(0.5, 1.5, N).astype(np.float32))
    w.set_lse_mode(mode)
    try:
        check_bits(w, xb, xb.float(), (cu(ys), cu(xn), cu(yn)), blank, lam, go)
    finally:
        w.set_lse_mode("auto")


@gpu
@pytest.mark.parametrize("mode", ["exact", "fast"])
@pytest.mark.parametrize("shape", [(2, 16, 5, 64, 2, 0.0), (2, 31, 18, 7, 0, 0.1)])
def test_bf16_label_equal_to_blank(w, shape, mode):
    """A label equal to blank: its blank and label gradients add, in both paths alike."""
    N, T, U, V, blank, lam = shape
    x, ys, xn, yn = make(N, T, U, V, seed=7 + V, blank=blank)
    ys[:, ::2] = blank
    xb = cu(x).to(torch.bfloat16)
    w.set_lse_mode(mode)
    try:
        check_bits(w, xb, xb.float(), (cu(ys), cu(xn), cu(yn)), blank, lam, cu(np.ones(N, np.float32)))
    finally:
        w.set_lse_mode("auto")


@gpu
@pytest.mark.parametrize("shape", [(3, 12, 7, 28, 0, 0.0), (2, 16, 5, 64, 2, 0.0), (2, 30, 12, 1024, 0, 0.0)])
def test_bf16_unaligned_rows(w, shape):
    """Logits one element past an aligned address: bf16 and float32 both take the unvectorised variants."""
    N, T, U, V, blank, lam = shape
    x, ys, xn, yn = make(N, T, U, V, seed=3 + V, blank=blank)
    vals = cu(x).to(torch.bfloat16).reshape(-1)
    flat_b = torch.zeros(vals.numel() + 1, dtype=torch.bfloat16, device="cuda")
    flat_f = torch.zeros(vals.numel() + 1, dtype=torch.float32, device="cuda")
    flat_b[1:] = vals
    flat_f[1:] = vals.float()
    xb, x32 = flat_b[1:].view(N, T, U, V), flat_f[1:].view(N, T, U, V)
    assert xb.is_contiguous() and xb.data_ptr() % 4 != 0 and x32.data_ptr() % 8 != 0
    check_bits(w, xb, x32, (cu(ys), cu(xn), cu(yn)), blank, lam, cu(np.linspace(0.5, 1.5, N).astype(np.float32)))


@gpu
@pytest.mark.parametrize("shape", SHAPES)
def test_bf16_vs_oracle(w, shape):
    N, T, U, V, blank, lam = shape
    x, ys, xn, yn = make(N, T, U, V, seed=T + V, blank=blank)
    xb = cu(x).to(torch.bfloat16)
    go = np.linspace(0.5, 1.5, N)
    c0, g0 = oracle.from_logits(xb.float().cpu().numpy(), ys, xn, yn, blank, lam, grad_output=go)
    xt = xb.clone().requires_grad_(True)
    costs = w.rnnt_loss_from_logits(xt, cu(ys), cu(xn), cu(yn), blank=blank, fastemit_lambda=lam)
    assert costs.dtype == torch.float32
    (costs * cu(go.astype(np.float32))).sum().backward()
    np.testing.assert_allclose(costs.detach().cpu().numpy(), c0, rtol=1e-5)
    g = xt.grad
    assert g.dtype == torch.bfloat16
    err = np.abs(g.float().cpu().numpy() - g0) - (2.0 ** -8 * np.abs(g0) + 1e-4 + 2 * gtol(T, U))
    assert err.max() <= 0, err.max()
    for n in range(N):                                   # padded frames / labels: exact zeros
        if xn[n] < T:
            assert g[n, xn[n]:].abs().max().item() == 0
        if yn[n] + 1 < U:
            assert g[n, :, yn[n] + 1:].abs().max().item() == 0


@gpu
def test_bf16_python_api_reductions(w):
    """Every reduction, with and without average_frames, equals the float32 API on the same values; 257 and 259 frames
    are not bf16 numbers, so dividing by the frame counts in the logits' dtype would show here."""
    N, T, U, V = 3, 260, 6, 24
    x, ys, xn, yn = make(N, T, U, V, seed=21)
    xn[:] = [260, 257, 259]
    xb = cu(x).to(torch.bfloat16)
    args = (cu(ys), cu(xn), cu(yn))
    for reduction in ("none", "sum", "mean"):
        for avg in (False, True):
            xt, x32 = xb.clone().requires_grad_(True), xb.float().requires_grad_(True)
            lb = w.rnnt_loss_from_logits(xt, *args, average_frames=avg, reduction=reduction)
            l3 = w.rnnt_loss_from_logits(x32, *args, average_frames=avg, reduction=reduction)
            assert lb.dtype == torch.float32
            assert same_bits(lb.detach(), l3.detach()), (reduction, avg)
            lb.sum().backward()
            l3.sum().backward()
            assert xt.grad.dtype == torch.bfloat16
            assert same_bits(xt.grad, x32.grad.to(torch.bfloat16)), (reduction, avg)


@gpu
def test_bf16_autocast_linear(w):
    """A joint-network Linear under autocast hands the loss bf16 logits.  Its weight gradient is compared with the same
    model run in float32: bf16 matmul inputs and a bf16 logit gradient leave a relative error of the order of 2^-8;
    the bound, 3e-2 of the gradient's norm, is loose on purpose."""
    N, T, U, H, V = 2, 40, 10, 64, 128
    g = torch.Generator(device="cuda").manual_seed(0)
    h = torch.randn(N, T, U, H, device="cuda", generator=g)
    ys = torch.randint(1, V, (N, U - 1), device="cuda", dtype=torch.int32, generator=g)
    xn = torch.tensor([T, T - 7], device="cuda", dtype=torch.int32)
    yn = torch.tensor([U - 1, U - 3], device="cuda", dtype=torch.int32)
    torch.manual_seed(0)
    lin = torch.nn.Linear(H, V).cuda()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        logits = lin(h)
        assert logits.dtype == torch.bfloat16
        loss_b = w.rnnt_loss_from_logits(logits, ys, xn, yn, average_frames=True, reduction="mean")
    loss_b.backward()
    gw_b = lin.weight.grad.clone()
    lin.weight.grad = None
    loss_f = w.rnnt_loss_from_logits(lin(h), ys, xn, yn, average_frames=True, reduction="mean")
    loss_f.backward()
    gw_f = lin.weight.grad
    assert loss_b.dtype == torch.float32
    np.testing.assert_allclose(loss_b.item(), loss_f.item(), rtol=1e-2)
    assert ((gw_b - gw_f).norm() / gw_f.norm()).item() < 3e-2


@gpu
def test_bf16_empty_batch_and_other_dtypes(w):
    T, U, V = 5, 3, 8
    x = torch.zeros(0, T, U, V, dtype=torch.bfloat16, device="cuda", requires_grad=True)
    e = torch.zeros(0, dtype=torch.int32, device="cuda")
    costs = w.rnnt_loss_from_logits(x, torch.zeros(0, U - 1, dtype=torch.int32, device="cuda"), e, e)
    assert costs.shape == (0,) and costs.dtype == torch.float32
    costs.sum().backward()
    assert x.grad.shape == x.shape and x.grad.dtype == torch.bfloat16
    xs, ys, xn, yn = make(2, T, U, V, seed=1)
    args = (cu(ys), cu(xn), cu(yn))
    with pytest.raises(RuntimeError, match="xs must be a Float tensor"):
        w.rnnt_loss_from_logits(cu(xs).half(), *args)
    c, lse, pg = w._C.rnnt_logits_forward(cu(xs), *args, 0, 0.0, True, 0)
    with pytest.raises(RuntimeError, match="xs must be a contiguous CUDA Float tensor"):
        w._C.rnnt_logits_backward(cu(xs).half(), lse, pg, args[0], torch.ones_like(c), 0)


@gpu
def test_bf16_no_upcast_copy(w):
    """Peak memory of a bf16 forward + backward at V = 1024: the bf16 gradient and per-cell float32 state, no float32
    copy of the logits (that alone would be 4 N T U V bytes more)."""
    N, T, U, V = 4, 100, 50, 1024
    g = torch.Generator(device="cuda").manual_seed(1)
    xb = (torch.randn(N, T, U, V, device="cuda", generator=g) * 3).to(torch.bfloat16).requires_grad_(True)
    ys = torch.randint(1, V, (N, U - 1), device="cuda", dtype=torch.int32, generator=g)
    xn = torch.full((N,), T, device="cuda", dtype=torch.int32)
    yn = torch.full((N,), U - 1, device="cuda", dtype=torch.int32)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    m0 = torch.cuda.memory_allocated()
    w.rnnt_loss_from_logits(xb, ys, xn, yn, reduction="sum").backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - m0
    cells = N * T * U
    assert xb.grad.dtype == torch.bfloat16
    assert peak < 2 * cells * V + 64 * cells + (8 << 20), peak


@gpu
def test_bf16_step_graph_capture(w):
    """The whole bf16 step is capturable (no host sync) and its replay reproduces the eager result."""
    N, T, U, V = 2, 40, 20, 300
    x, ys, xn, yn = make(N, T, U, V, seed=17)
    xb = cu(x).to(torch.bfloat16).requires_grad_(True)
    args = (cu(ys), cu(xn), cu(yn))

    def step():
        xb.grad = None
        loss = w.rnnt_loss_from_logits(xb, *args, reduction="sum")
        loss.backward()
        return loss

    loss0 = step().detach().clone()
    grad0 = xb.grad.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    xb.grad = None
    with torch.cuda.graph(graph):
        loss = step()
    graph.replay()
    torch.cuda.synchronize()
    assert same_bits(loss.detach(), loss0) and same_bits(xb.grad, grad0)


def test_bf16_logits_entries_validate_on_host():
    """No GPU needed: the two bf16 entry points reject bad shapes, blank >= V and odd addresses (status 5) before any
    CUDA call.  The pointers are never dereferenced."""
    import warp_rnnt_b200  # noqa: F401  builds the extension if it is missing
    lib = ctypes.CDLL(LIB)
    P, ODD = ctypes.c_void_p(4096), ctypes.c_void_p(4097)
    fwd, bwd = lib.rnnt_b200_logits_forward_bf16, lib.rnnt_b200_logits_backward_bf16
    fwd.restype = bwd.restype = ctypes.c_int

    def f(logits, T, V, blank):        # (N, T, U, V) = (4, T, 3, V), no workspace
        return fwd(None, None, ctypes.c_size_t(0), logits, P, P, P, P, P, P, 4, T, 3, V, blank, ctypes.c_float(0.0), 0)

    def b(logits, out, T, V, blank):
        return bwd(None, logits, P, P, P, P, out, 4, T, 3, V, blank)

    assert f(P, 0, 5, 0) == 5                      # T == 0
    assert f(P, 2, 5, 5) == 5                      # blank >= V
    assert f(ODD, 2, 5, 0) == 5                    # odd bf16 address
    assert f(P, 2, 5, 0) == 6                      # valid: gets as far as the (missing) workspace, still on the host
    assert b(P, P, 0, 5, 0) == 5
    assert b(P, P, 2, 5, 5) == 5
    assert b(ODD, P, 2, 5, 0) == 5
    assert b(P, ODD, 2, 5, 0) == 5
