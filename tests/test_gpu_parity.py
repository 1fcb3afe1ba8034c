"""GPU parity tests (B200): the CUDA path against
  (1) the reference's golden vectors (tests/golden/reference_vectors.json),
  (2) the fp64 oracle (oracle/rnnt_oracle.c) on seeded random inputs,
  (3) the unmodified reference kernels: their recorded outputs (tests/golden/reference_outputs.json, see
      tests/common.py ReferenceOutputs) for the same seeded inputs.

Tolerances (BASELINE.md section 3): cost |d|/|ref| <= 1e-4, gradients max|d| <= 1e-4 (values lie in
[-(1+lambda), 0]); the assertions below use the much tighter bounds these sizes actually meet.
LSE mode 'exact' must be BIT-IDENTICAL to the reference kernels.
"""
import numpy as np
import pytest
import torch

from oracle import oracle
from tests.common import ReferenceOutputs, compact_defined, golden_case, make_inputs, to_compact, from_compact

pytestmark = pytest.mark.gpu

MODES = ["fast", "exact"]


def gtol(T, U):
    """fp32 alpha/beta carry ~ulp(|alpha|) rounding per anti-diagonal; the compiled reference shows the
    same distance to the fp64 oracle (see test_reference_noise_floor).  Grows with the path length."""
    return 2e-5 + 6e-6 * (T + U)


@pytest.fixture(scope="module")
def w():
    import warp_rnnt_b200
    return warp_rnnt_b200


@pytest.fixture
def reference(request):
    return ReferenceOutputs(request)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gather_np(lp, ys, blank):
    N, T, U, V = lp.shape
    index = np.full((N, T, U, 2), blank, dtype=np.int64)
    index[:, :, :U - 1, 1] = ys[:, None, :]
    return np.ascontiguousarray(np.take_along_axis(lp, index, axis=3))


# ------------------------------------------------------------------ (1) the reference's own tests
def test_shape_message(w):
    e = torch.tensor([], dtype=torch.float32).cuda()
    i = torch.tensor([], dtype=torch.int).cuda()
    with pytest.raises(RuntimeError, match="xs must have 4 dimensions"):
        w._C.rnnt_loss(e, i, i, i)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["test_one_to_many", "test_one_to_empty", "test_forward_single",
                                  "test_forward_batch"])
def test_golden_dense(w, name, mode):
    c = golden_case(name)
    w.set_lse_mode(mode)
    costs, grads = w._C.rnnt_loss(cu(c["lp"]), cu(c["ys"]), cu(c["xn"]), cu(c["yn"]))
    np.testing.assert_array_almost_equal(costs.cpu().numpy(), c["costs"], decimal=6)
    np.testing.assert_array_almost_equal(grads.cpu().numpy(), c["grads"], decimal=6)


@pytest.mark.parametrize("mode", MODES)
def test_golden_gather_boundary(w, mode):
    c = golden_case("test_forward_single_gather")
    w.set_lse_mode(mode)
    g = gather_np(c["lp"], c["ys"], 0)
    costs, grads = w._C.rnnt_loss(cu(g), cu(c["ys"]), cu(c["xn"]), cu(c["yn"]), blank=-1)
    np.testing.assert_array_almost_equal(costs.cpu().numpy(), c["costs"], decimal=6)
    np.testing.assert_array_almost_equal(grads.cpu().numpy(), c["grads"], decimal=6)


@pytest.mark.parametrize("mode", MODES)
def test_golden_compact(w, mode):
    c = golden_case("test_forward_batch_compact")
    w.set_lse_mode(mode)
    xs_c, ys_c = to_compact(c["lp"], c["ys"], c["xn"], c["yn"])
    costs, grads, loc = w._C.rnnt_loss_compact(cu(xs_c), cu(ys_c), cu(c["xn"]), cu(c["yn"]))
    np.testing.assert_array_almost_equal(costs.cpu().numpy(), c["costs"], decimal=6)
    cumlen = torch.cumsum(cu(c["xn"]) * (cu(c["yn"]) + 1), dim=0, dtype=torch.int32)
    g = w._C.rnnt_loss_compact_backward(torch.ones_like(costs).contiguous(), grads, cumlen, loc,
                                        c["lp"].shape[-1], 0)
    np.testing.assert_array_almost_equal(g.cpu().numpy(), c["grads"], decimal=6)


def test_golden_python_gather(w):
    """tensorflow_binding/warp_rnnt_tf/test.py:227-252 -- python-level gather=True."""
    c = golden_case("test_forward_single_inner_gather")
    w.set_lse_mode("fast")
    lp = cu(c["lp"]).requires_grad_(True)
    costs = w.rnnt_loss(lp, cu(c["ys"]), cu(c["xn"]), cu(c["yn"]), gather=True)
    costs.sum().backward()
    np.testing.assert_array_almost_equal(costs.detach().cpu().numpy(), c["costs"], decimal=6)
    np.testing.assert_array_almost_equal(lp.grad.cpu().numpy(), c["grads"], decimal=6)


def test_calls_smoke(w, capfd):
    """test.py:190-212: N=128,T=100,U=90,V=3, random label lengths; must not hang, crash or warn."""
    n, t, u, v = 128, 100, 90, 3
    w.set_lse_mode("fast")
    for i in range(2):
        rng = np.random.RandomState(i)
        xs = torch.log_softmax(torch.tensor(rng.randn(n, t, u, v), dtype=torch.float32), dim=-1)
        ys = torch.tensor(rng.randint(1, v, (n, u - 1)), dtype=torch.int)
        xn = torch.tensor([t] * n, dtype=torch.int)
        yn = torch.tensor(rng.randint(1, u, n), dtype=torch.int)
        costs, grads = w._C.rnnt_loss(xs.cuda(), ys.cuda(), xn.cuda(), yn.cuda())
        torch.cuda.synchronize()
        c0, g0 = oracle.dense(xs.numpy(), ys.numpy(), xn.numpy(), yn.numpy())
        np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=1e-5)
        np.testing.assert_allclose(grads.cpu().numpy(), g0, atol=1e-4)   # T+U = 190 fp32 steps
    assert "WARNING" not in capfd.readouterr().out


# ------------------------------------------------------------------ (2) fp64 oracle, random shapes
SHAPES = [
    # N, T, U, V, random_lengths, blank, lambda
    (1, 1, 1, 1, False, 0, 0.0),
    (2, 1, 5, 3, False, 0, 0.0),
    (2, 6, 1, 4, False, 0, 0.0),
    (3, 7, 5, 6, True, 0, 0.0),
    (4, 33, 34, 5, True, 2, 0.25),       # crosses one warp boundary
    (2, 40, 70, 3, True, 0, 0.0),        # three warps
    (3, 150, 40, 28, True, 0, 0.01),     # BASELINE cfg 1/2 shape
    (2, 70, 129, 7, False, 6, 0.0),      # 5 warps, blank = V-1
    (2, 300, 20, 50, True, 0, 0.0),
    (1, 64, 600, 4, True, 1, 0.0),       # U > 512: two column passes per CTA
    (5, 9, 9, 4101, True, 17, 0.0),      # big V, odd row length
]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", SHAPES)
def test_dense_vs_oracle(w, shape, mode):
    N, T, U, V, rl, blank, lam = shape
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=N + T + U, random_lengths=rl, blank=blank)
    w.set_lse_mode(mode)
    costs, grads = w._C.rnnt_loss(cu(lp), cu(ys), cu(xn), cu(yn), blank=blank, fastemit_lambda=lam)
    c0, g0 = oracle.dense(lp, ys, xn, yn, blank=blank, fastemit_lambda=lam)
    np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=2e-6)
    np.testing.assert_allclose(grads.cpu().numpy(), g0, atol=gtol(T, U))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", SHAPES[:9])
def test_gathered_input_vs_oracle(w, shape, mode):
    N, T, U, V, rl, blank, lam = shape
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=7 + T, random_lengths=rl, blank=blank)
    g = gather_np(lp, ys, blank)
    w.set_lse_mode(mode)
    costs, grads = w._C.rnnt_loss(cu(g), cu(ys), cu(xn), cu(yn), blank=-1, fastemit_lambda=lam)
    c0, g0 = oracle.dense(g, ys, xn, yn, blank=-1, fastemit_lambda=lam)
    np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=2e-6)
    np.testing.assert_allclose(grads.cpu().numpy(), g0, atol=gtol(T, U))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", SHAPES)
def test_compact_vs_oracle(w, shape, mode):
    N, T, U, V, rl, blank, lam = shape
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=11 + U, random_lengths=rl, blank=blank)
    xs_c, ys_c = to_compact(lp, ys, xn, yn)
    w.set_lse_mode(mode)
    costs, pg, loc = w._C.rnnt_loss_compact(cu(xs_c), cu(ys_c), cu(xn), cu(yn), blank=blank, fastemit_lambda=lam)
    c0, pg0, loc0 = oracle.compact(xs_c, ys_c, xn, yn, blank=blank, fastemit_lambda=lam)
    np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=2e-6)
    np.testing.assert_allclose(pg.cpu().numpy(), pg0, atol=gtol(T, U))
    assert np.array_equal(loc.cpu().numpy(), loc0)
    cum = np.cumsum(xn.astype(np.int64) * (yn + 1)).astype(np.int32)
    go = np.linspace(0.5, 2.0, N).astype(np.float32)
    out = w._C.rnnt_loss_compact_backward(cu(go), pg, cu(cum), loc, V, blank)
    out0 = oracle.compact_scatter(go, pg0, loc0, cum, V, blank)
    np.testing.assert_allclose(out.cpu().numpy(), out0, atol=2 * gtol(T, U))
    # forward only (required_grad=False, __init__.py:109-116)
    costs2, _, _ = w._C.rnnt_loss_compact(cu(xs_c), cu(ys_c), cu(xn), cu(yn), blank=blank,
                                          fastemit_lambda=lam, required_grad=False)
    assert torch.equal(costs, costs2)


def test_compact_shape_errors(w):
    lp, ys, xn, yn = make_inputs(2, 4, 3, 5, seed=0, random_lengths=False)
    xs_c, ys_c = to_compact(lp, ys, xn, yn)
    with pytest.raises(RuntimeError, match="xs shape mismatch"):
        w._C.rnnt_loss_compact(cu(xs_c[:-1]), cu(ys_c), cu(xn), cu(yn))
    with pytest.raises(RuntimeError, match="ys shape must be equal"):
        w._C.rnnt_loss_compact(cu(xs_c), cu(ys_c[:-1]), cu(xn), cu(yn))
    with pytest.raises(RuntimeError, match="xs must have 2 dimensions"):
        w._C.rnnt_loss_compact(cu(lp), cu(ys_c), cu(xn), cu(yn))


# ------------------------------------------------------------------ python API / autograd
@pytest.mark.parametrize("gather", [False, True])
@pytest.mark.parametrize("reduction,avg", [("none", False), ("mean", True), ("sum", False), ("none", True),
                                           ("sum", True), ("mean", False), (None, False)])
def test_python_api_autograd(w, gather, reduction, avg):
    N, T, U, V = 4, 21, 13, 9
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=3, random_lengths=True, blank=0)
    w.set_lse_mode("fast")
    x = cu(lp).requires_grad_(True)
    loss = w.rnnt_loss(x, cu(ys), cu(xn), cu(yn), average_frames=avg, reduction=reduction, gather=gather,
                       fastemit_lambda=0.1)
    go = np.linspace(1.0, 2.0, N)
    if reduction in ("none", None):
        (loss * cu(go.astype(np.float32))).sum().backward()
        loss0, g0 = oracle.rnnt_loss(lp, ys, xn, yn, avg, reduction, 0, gather, 0.1, grad_output=go)
    else:
        loss.backward()
        loss0, g0 = oracle.rnnt_loss(lp, ys, xn, yn, avg, reduction, 0, gather, 0.1)
    np.testing.assert_allclose(loss.detach().cpu().numpy(), loss0, rtol=1e-5)
    np.testing.assert_allclose(x.grad.cpu().numpy(), g0, atol=2 * gtol(T, U))


def test_python_api_one_launch_and_upstream_scaling(w):
    """rnnt_loss(reduction=...) + backward on the dense path: ONE fused kernel produces costs, the reduced loss and the
    final gradient; backward adds only the rescale check (which rescales when the upstream gradient is not 1)."""
    N, T, U, V = 5, 33, 17, 11
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=12, random_lengths=True)
    args = (cu(ys), cu(xn), cu(yn))
    w.set_lse_mode("exact")
    for reduction, avg in (("sum", False), ("mean", True)):
        loss0, g0 = oracle.rnnt_loss(lp, ys, xn, yn, avg, reduction)
        x = cu(lp).requires_grad_(True)
        torch.cuda.synchronize()
        n0 = w._C.launch_count()
        loss = w.rnnt_loss(x, *args, average_frames=avg, reduction=reduction)
        assert w._C.launch_count() - n0 == 1                       # k_fused: costs + loss + gradient
        loss.backward()
        assert w._C.launch_count() - n0 == 2                       # + k_rescale (returns at once: upstream == 1)
        np.testing.assert_allclose(loss.item(), loss0, rtol=1e-6)
        np.testing.assert_allclose(x.grad.cpu().numpy(), g0, atol=2 * gtol(T, U))
        g1 = x.grad.clone()
        # upstream gradient != 1: (3 * loss).backward() must give exactly 3 * the gradient above
        x2 = cu(lp).requires_grad_(True)
        (3.0 * w.rnnt_loss(x2, *args, average_frames=avg, reduction=reduction)).backward()
        assert torch.equal(x2.grad, g1 * 3.0)
        # reduced loss == reduction of the per-sample costs (fixed-order sum in the kernel vs torch's order)
        costs = w.rnnt_loss(cu(lp), *args, average_frames=avg, reduction="none")
        red = costs.sum() if reduction == "sum" else costs.mean()
        np.testing.assert_allclose(loss.item(), red.item(), rtol=2e-6)
    # a second backward through the same graph has no buffer left: clear error instead of a wrong gradient
    x = cu(lp).requires_grad_(True)
    loss = w.rnnt_loss(x, *args, reduction="sum")
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="second time"):
        loss.backward()
    w.set_lse_mode("auto")


def test_python_api_compact_autograd(w):
    N, T, U, V = 3, 12, 7, 6
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=4, random_lengths=True)
    xs_c, ys_c = to_compact(lp, ys, xn, yn)
    x = cu(xs_c).requires_grad_(True)
    loss = w.rnnt_loss(x, cu(ys_c), cu(xn), cu(yn), reduction="mean", compact=True)
    loss.backward()
    loss0, g0 = oracle.rnnt_loss(xs_c, ys_c, xn, yn, reduction="mean", compact_layout=True)
    np.testing.assert_allclose(loss.item(), loss0, rtol=1e-5)
    np.testing.assert_allclose(x.grad.cpu().numpy(), g0, atol=2e-5)
    with torch.no_grad():
        loss2 = w.rnnt_loss(cu(xs_c), cu(ys_c), cu(xn), cu(yn), reduction="mean", compact=True)
    np.testing.assert_allclose(loss2.item(), loss0, rtol=1e-5)


def test_eager_variant_and_no_grad(w):
    N, T, U, V = 3, 10, 6, 5
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=8, random_lengths=True)
    c0, g0 = oracle.dense(lp, ys, xn, yn)
    x = cu(lp).requires_grad_(True)
    costs = w.RNNTLossEager.apply(x, cu(ys), cu(xn), cu(yn), 0, 0.0)
    (2.0 * costs).sum().backward()
    np.testing.assert_allclose(x.grad.cpu().numpy(), 2.0 * g0, atol=2e-5)
    costs_ng = w.rnnt_loss(cu(lp), cu(ys), cu(xn), cu(yn))        # requires_grad=False: forward only
    np.testing.assert_allclose(costs_ng.cpu().numpy(), c0, rtol=1e-5)


def test_label_equal_to_blank_semantics(w):
    """Dense path: the label gradient overrides the blank one (core.cu launches the label kernel
    last); python-level gather=True adds them (torch scatter_add)."""
    N, T, U, V = 1, 4, 3, 4
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=1)
    ys[:] = 0
    c0, g0 = oracle.dense(lp, ys, xn, yn)                  # oracle = override
    costs, grads = w._C.rnnt_loss(cu(lp), cu(ys), cu(xn), cu(yn))
    np.testing.assert_allclose(grads.cpu().numpy(), g0, atol=1e-6)
    x = cu(lp).requires_grad_(True)
    w.rnnt_loss(x, cu(ys), cu(xn), cu(yn), gather=True).sum().backward()
    g = gather_np(lp, ys, 0)
    _, gp = oracle.dense(g, ys, xn, yn, blank=-1)
    expect = np.zeros_like(lp, dtype=np.float64)
    expect[..., 0] = gp[..., 0] + gp[..., 1]
    np.testing.assert_allclose(x.grad.cpu().numpy(), expect, atol=1e-6)


def test_non_default_stream_and_device_guard(w):
    lp, ys, xn, yn = make_inputs(2, 30, 10, 8, seed=2, random_lengths=True)
    c0, g0 = oracle.dense(lp, ys, xn, yn)
    s = torch.cuda.Stream()
    a, b, c, d = cu(lp), cu(ys), cu(xn), cu(yn)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        costs, grads = w._C.rnnt_loss(a, b, c, d)
    s.synchronize()
    np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=1e-5)
    np.testing.assert_allclose(grads.cpu().numpy(), g0, atol=2e-5)


# ------------------------------------------------------------------ (3) the compiled reference
REF_SHAPES = [(3, 7, 5, 6, True, 0, 0.0), (4, 33, 34, 5, True, 2, 0.25), (3, 150, 40, 28, True, 0, 0.01),
              (2, 70, 129, 7, False, 6, 0.0), (8, 100, 90, 3, True, 0, 0.0), (2, 300, 50, 50, True, 0, 0.0)]


@pytest.mark.parametrize("shape", REF_SHAPES)
def test_exact_mode_is_bit_identical_to_reference_dense(w, reference, shape):
    N, T, U, V, rl, blank, lam = shape
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=21 + T, random_lengths=rl, blank=blank)
    args = (cu(lp), cu(ys), cu(xn), cu(yn))
    w.set_lse_mode("exact")
    cm, gm = w._C.rnnt_loss(*args, blank=blank, fastemit_lambda=lam)
    reference.check("dense", (cm, gm), lambda ref: ref.rnnt_loss(*args, blank=blank, fastemit_lambda=lam), args)
    w.set_lse_mode("fast")                       # cm, gm are the reference's bits from here on
    cf, gf = w._C.rnnt_loss(*args, blank=blank, fastemit_lambda=lam)
    assert ((cf - cm).abs() / cm.abs()).max().item() <= 1e-5
    assert (gf - gm).abs().max().item() <= gtol(T, U)


def reference_compact_backward(cargs, go, blank, lam):
    """The reference's compact forward, then its backward on its own pair gradients (for ReferenceOutputs.check)."""
    def run(ref):
        _, gr, lr = ref.rnnt_loss_compact(*cargs, blank=blank, fastemit_lambda=lam)
        cumlen = torch.cumsum(cargs[2] * (cargs[3] + 1), dim=0, dtype=torch.int32)
        return (ref.rnnt_loss_compact_backward(go, gr, cumlen, lr, cargs[0].size(1), blank),)
    return run


@pytest.mark.parametrize("shape", REF_SHAPES)
def test_exact_mode_is_bit_identical_to_reference_gather_and_compact(w, reference, shape):
    N, T, U, V, rl, blank, lam = shape
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=31 + U, random_lengths=rl, blank=blank)
    w.set_lse_mode("exact")
    g = gather_np(lp, ys, blank)
    args = (cu(g), cu(ys), cu(xn), cu(yn))
    cm, gm = w._C.rnnt_loss(*args, blank=-1, fastemit_lambda=lam)
    reference.check("gathered", (cm, gm), lambda ref: ref.rnnt_loss(*args, blank=-1, fastemit_lambda=lam), args)
    xs_c, ys_c = to_compact(lp, ys, xn, yn)
    cargs = (cu(xs_c), cu(ys_c), cu(xn), cu(yn))
    cm, gm, lm = w._C.rnnt_loss_compact(*cargs, blank=blank, fastemit_lambda=lam)
    reference.check("compact", compact_defined(cm, gm, lm, blank),
                    lambda ref: compact_defined(*ref.rnnt_loss_compact(*cargs, blank=blank, fastemit_lambda=lam), blank),
                    cargs)
    assert torch.all(gm[:, 1][lm == blank] == 0)
    cumlen = torch.cumsum(cu(xn) * (cu(yn) + 1), dim=0, dtype=torch.int32)
    go = torch.linspace(0.5, 1.5, N).cuda()
    bm = w._C.rnnt_loss_compact_backward(go, gm, cumlen, lm, V, blank)
    reference.check("compact_backward", (bm,), reference_compact_backward(cargs, go, blank, lam), cargs)


# ------------------------------------------------------------------ drop-in at the C-ABI level
@pytest.fixture(scope="module")
def compat():
    # the reference's own binding.cpp, built by oracle/build_ref.py only where the reference's sources are present
    from oracle import build_ref
    return build_ref.load_compat()


@pytest.mark.parametrize("name", ["test_one_to_many", "test_one_to_empty", "test_forward_single", "test_forward_batch"])
def test_reference_binding_on_our_c_abi_golden(w, compat, name):
    """The reference's UNMODIFIED pytorch_binding/binding.cpp linked against librnnt_b200.so
    (run_warp_rnnt & co, core.h:29-60) reproduces the reference's own test vectors."""
    if compat is None:
        pytest.skip("oracle/_ref/warp_rnnt_compat_C.so not present")
    c = golden_case(name)
    costs, grads = compat.rnnt_loss(cu(c["lp"]), cu(c["ys"]), cu(c["xn"]), cu(c["yn"]))
    np.testing.assert_array_almost_equal(costs.cpu().numpy(), c["costs"], decimal=6)
    np.testing.assert_array_almost_equal(grads.cpu().numpy(), c["grads"], decimal=6)


def test_reference_binding_on_our_c_abi_all_layouts(w, compat, reference):
    if compat is None:
        pytest.skip("oracle/_ref/warp_rnnt_compat_C.so not present")
    N, T, U, V, blank, lam = 4, 45, 37, 11, 3, 0.2
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=77, random_lengths=True, blank=blank)
    w.set_lse_mode("exact")                      # compat ABI uses the process-wide LSE mode
    args = (cu(lp), cu(ys), cu(xn), cu(yn))
    cm, gm = compat.rnnt_loss(*args, blank=blank, fastemit_lambda=lam)
    reference.check("dense", (cm, gm), lambda ref: ref.rnnt_loss(*args, blank=blank, fastemit_lambda=lam), args)
    g = gather_np(lp, ys, blank)
    gargs = (cu(g), cu(ys), cu(xn), cu(yn))
    cm, gm = compat.rnnt_loss(*gargs, blank=-1, fastemit_lambda=lam)
    reference.check("gathered", (cm, gm), lambda ref: ref.rnnt_loss(*gargs, blank=-1, fastemit_lambda=lam), gargs)
    xs_c, ys_c = to_compact(lp, ys, xn, yn)
    cargs = (cu(xs_c), cu(ys_c), cu(xn), cu(yn))
    cm, gm, lm = compat.rnnt_loss_compact(*cargs, blank=blank, fastemit_lambda=lam)
    reference.check("compact", compact_defined(cm, gm, lm, blank),
                    lambda ref: compact_defined(*ref.rnnt_loss_compact(*cargs, blank=blank, fastemit_lambda=lam), blank),
                    cargs)
    cumlen = torch.cumsum(cu(xn) * (cu(yn) + 1), dim=0, dtype=torch.int32)
    go = torch.linspace(0.5, 1.5, N).cuda()
    bm = compat.rnnt_loss_compact_backward(go, gm, cumlen, lm, V, blank)
    reference.check("compact_backward", (bm,), reference_compact_backward(cargs, go, blank, lam), cargs)
    w.set_lse_mode("auto")


# ------------------------------------------------------------------ the emit's row-pair path (V % 4 == 2)
@pytest.mark.parametrize("V", [6, 10, 50])
def test_expand_row_pair_path_all_modes(w, reference, V):
    """k_expand sweeps two rows at a time when V % 4 == 2 (float output): dense forward (label overrides blank), python
    gather=True backward (label adds to blank), compact backward -- on a lattice too large for the fused kernel, with
    odd and even row counts per chunk, labels that equal the blank, and an output base that is only 16-byte aligned."""
    N, T, U = 3, 301, 47
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=V, random_lengths=True, blank=1)
    ys[0, :5] = 1                                                    # labels equal to blank = 1
    args = (cu(ys), cu(xn), cu(yn))
    w.set_lse_mode("exact")
    try:
        c0, g0 = oracle.dense(lp, ys, xn, yn, blank=1, fastemit_lambda=0.1)
        x0 = cu(lp)
        costs, grads = w._C.rnnt_loss(x0, *args, blank=1, fastemit_lambda=0.1)
        np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=1e-5)
        assert np.abs(grads.cpu().numpy() - g0).max() <= gtol(T, U)
        reference.check("dense", (costs, grads), lambda ref: ref.rnnt_loss(x0, *args, blank=1, fastemit_lambda=0.1),
                        (x0,) + args)
        # gather=True: torch.gather's backward adds the label gradient to the blank one where they coincide
        x = cu(lp).requires_grad_(True)
        go = cu(np.linspace(0.5, 1.5, N).astype(np.float32))
        (w.rnnt_loss(x, *args, blank=1, gather=True, fastemit_lambda=0.1) * go).sum().backward()
        g = gather_np(lp, ys, 1)
        _, gp = oracle.dense(g, ys, xn, yn, blank=-1, fastemit_lambda=0.1)
        expect = np.zeros_like(lp, dtype=np.float64)
        n_i, t_i, u_i = np.meshgrid(np.arange(N), np.arange(T), np.arange(U - 1), indexing="ij")
        np.add.at(expect, (n_i, t_i, u_i, ys[n_i, u_i]), gp[:, :, :U - 1, 1])
        expect[..., 1] += gp[..., 0]
        expect *= go.cpu().numpy().reshape(-1, 1, 1, 1)
        assert np.abs(x.grad.cpu().numpy() - expect).max() <= 2 * gtol(T, U)
        # compact backward
        xs_c, ys_c = to_compact(lp, ys, xn, yn)
        cargs = (cu(xs_c), cu(ys_c), cu(xn), cu(yn))
        cm, gm, lm = w._C.rnnt_loss_compact(*cargs, blank=1, fastemit_lambda=0.1)
        cumlen = torch.cumsum(cu(xn) * (cu(yn) + 1), dim=0, dtype=torch.int32)
        bm = w._C.rnnt_loss_compact_backward(go, gm, cumlen, lm, V, 1)
        c1, pg1, loc1 = oracle.compact(xs_c, ys_c, xn, yn, blank=1, fastemit_lambda=0.1)
        b1 = oracle.compact_scatter(go.cpu().numpy(), pg1, loc1, cumlen.cpu().numpy(), V, 1)
        assert np.abs(bm.cpu().numpy() - b1).max() <= 2 * gtol(T, U)
        # the reference's backward (scatter) on the same pair gradients
        reference.check("compact_backward", (bm,),
                        lambda ref: (ref.rnnt_loss_compact_backward(go, gm, cumlen, lm, V, 1),), cargs + (go,))
    finally:
        w.set_lse_mode("auto")
