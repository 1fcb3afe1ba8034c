"""GPU: rnnt_loss_from_logits (fused log_softmax + loss, SURVEY.md 8(f)1) against
  (1) the fp64 oracle (oracle.from_logits = log_softmax then the loss, differentiated through both),
  (2) torch.log_softmax + this library's rnnt_loss through autograd (same kernels, unfused),
  (3) torch.log_softmax + the reference kernels through autograd (their recorded outputs, tests/common.py
      ReferenceOutputs: this library's exact mode reproduces them bit for bit).

Not bit-identical by construction (the normaliser is summed in another order than torch's): stated tolerances are
costs |d|/|ref| <= 1e-5 and gradients max|d| <= 1e-4 + gtol(T,U) (values in [-(1+lambda), 1+lambda])."""
import numpy as np
import pytest
import torch

from oracle import oracle
from tests.common import ReferenceOutputs

pytestmark = pytest.mark.gpu


def gtol(T, U):
    return 2e-5 + 6e-6 * (T + U)


@pytest.fixture(scope="module")
def w():
    import warp_rnnt_b200
    return warp_rnnt_b200


@pytest.fixture
def reference(request):
    return ReferenceOutputs(request)


def make(N, T, U, V, seed, blank=0, scale=3.0):
    rng = np.random.RandomState(seed)
    x = (rng.randn(N, T, U, V) * scale).astype(np.float32)           # raw logits, NOT normalised
    ys = rng.randint(0, V - 1, (N, U - 1)).astype(np.int32)
    ys = np.where(ys >= blank, ys + 1, ys).astype(np.int32)
    xn = rng.randint(max(T // 2, 1), T + 1, (N,)).astype(np.int32)
    yn = (rng.randint(U // 2, U, (N,)) if U > 1 else np.zeros(N)).astype(np.int32)
    xn[0], yn[0] = T, U - 1
    return x, ys, xn, yn


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


SHAPES = [(3, 12, 7, 5, 0, 0.0), (2, 33, 34, 28, 3, 0.2), (4, 150, 40, 28, 0, 0.0), (2, 40, 20, 300, 7, 0.0),
          (2, 25, 9, 5000, 0, 0.1), (2, 400, 70, 50, 0, 0.0), (3, 20, 1, 6, 0, 0.0), (2, 31, 18, 7, 0, 0.0), (2, 16, 5, 64, 2, 0.0)]


@pytest.mark.parametrize("mode", ["exact", "fast"])
@pytest.mark.parametrize("shape", SHAPES)
def test_from_logits_vs_oracle(w, shape, mode):
    N, T, U, V, blank, lam = shape
    x, ys, xn, yn = make(N, T, U, V, seed=T + V, blank=blank)
    go = np.linspace(0.5, 1.5, N)
    c0, g0 = oracle.from_logits(x, ys, xn, yn, blank, lam, grad_output=go)
    w.set_lse_mode(mode)
    try:
        xt = cu(x).requires_grad_(True)
        costs = w.rnnt_loss_from_logits(xt, cu(ys), cu(xn), cu(yn), blank=blank, fastemit_lambda=lam)
        (costs * cu(go.astype(np.float32))).sum().backward()
        np.testing.assert_allclose(costs.detach().cpu().numpy(), c0, rtol=1e-5)
        err = np.abs(xt.grad.cpu().numpy() - g0).max()
        assert err <= 1e-4 + 2 * gtol(T, U), err
        # padded frames / labels: exact zeros
        g = xt.grad
        for n in range(N):
            assert g[n, xn[n]:].abs().max().item() == 0 if xn[n] < T else True
            assert g[n, :, yn[n] + 1:].abs().max().item() == 0 if yn[n] + 1 < U else True
        # every in-lattice row of the logit gradient sums to ~0 (softmax Jacobian annihilates constants)
        assert g.sum(-1).abs().max().item() <= 1e-4
    finally:
        w.set_lse_mode("auto")


@pytest.mark.parametrize("shape", [(4, 150, 40, 28, 0, 0.0), (2, 60, 33, 50, 0, 0.25), (2, 30, 12, 1024, 0, 0.0)])
def test_from_logits_vs_unfused_and_reference(w, reference, shape):
    N, T, U, V, blank, lam = shape
    x, ys, xn, yn = make(N, T, U, V, seed=11 + V, blank=blank)
    args = (cu(ys), cu(xn), cu(yn))
    xt = cu(x).requires_grad_(True)
    loss = w.rnnt_loss_from_logits(xt, *args, average_frames=True, reduction="mean", blank=blank, fastemit_lambda=lam)
    loss.backward()
    # unfused, same library
    xu = cu(x).requires_grad_(True)
    lu = w.rnnt_loss(torch.log_softmax(xu, -1), *args, average_frames=True, reduction="mean", blank=blank, fastemit_lambda=lam)
    lu.backward()
    np.testing.assert_allclose(loss.item(), lu.item(), rtol=1e-5)
    assert (xt.grad - xu.grad).abs().max().item() <= 1e-4 / N
    xr = cu(x).requires_grad_(True)
    lp = torch.log_softmax(xr, -1)
    lpd = lp.detach().contiguous()
    w.set_lse_mode("exact")
    costs, grads = w._C.rnnt_loss(lpd, *args, blank=blank, fastemit_lambda=lam)
    reference.check("dense", (costs, grads), lambda ref: ref.rnnt_loss(lpd, *args, blank=blank, fastemit_lambda=lam),
                    (lpd,) + args)
    w.set_lse_mode("auto")
    wgt = (1.0 / cu(xn).float() / N).view(-1, 1, 1, 1)
    lp.backward(grads * wgt)
    np.testing.assert_allclose(loss.item(), (costs / cu(xn).float()).mean().item(), rtol=1e-5)
    assert (xt.grad - xr.grad).abs().max().item() <= 1e-4 / N


def test_from_logits_no_grad_and_invariance(w):
    N, T, U, V = 2, 20, 8, 12
    x, ys, xn, yn = make(N, T, U, V, seed=5)
    args = (cu(ys), cu(xn), cu(yn))
    c1 = w.rnnt_loss_from_logits(cu(x), *args)                       # requires_grad False: forward only
    c2 = w.rnnt_loss_from_logits(cu(x + 7.5), *args)                 # shifting every logit row changes nothing
    c0, _ = oracle.from_logits(x, ys, xn, yn)
    np.testing.assert_allclose(c1.cpu().numpy(), c0, rtol=1e-5)
    np.testing.assert_allclose(c2.cpu().numpy(), c0, rtol=2e-5)
