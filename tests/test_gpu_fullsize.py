"""GPU, BASELINE.json's full sizes: size-independent properties of the domain + the reference kernels' recorded
outputs (tests/common.py ReferenceOutputs) where the reference finishes in seconds.

Properties (all follow from alpha/beta being a flow on the lattice, SURVEY.md section 0):
  * every anti-diagonal t+u = d < Tn+Un-2 carries total flow 1:  -sum_{t+u=d}(g_blank + g_label) == 1
    (lambda = 0), and the last cell's blank gradient is -1;
  * gradients are <= 0 and non-zero only in the blank column and the cell's label column;
  * padded frames / labels get exactly zero gradient;
  * lattices are independent: a batch equals the concatenation of its sub-batches, bit for bit
    (also exercises 64-bit offsets: N*T*U*V > 2^31 at cfg 5's micro-batch);
  * compact layout == dense layout on the unpadded cells.
"""
import numpy as np
import pytest
import torch

from tests.common import ReferenceOutputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def w():
    import warp_rnnt_b200
    return warp_rnnt_b200


@pytest.fixture
def reference(request):
    return ReferenceOutputs(request)


def synth(N, T, U, V, seed, random_lengths=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    xs = torch.log_softmax(torch.randn((N, T, U, V), device="cuda", generator=g), dim=-1)
    ys = torch.randint(1, V, (N, U - 1), dtype=torch.int, device="cuda", generator=g)
    if random_lengths:
        xn = torch.randint(T // 2, T + 1, (N,), dtype=torch.int, device="cuda", generator=g)
        yn = torch.randint(U // 2, U, (N,), dtype=torch.int, device="cuda", generator=g)
        xn = xn + T - xn.max()
        yn = yn + (U - 1) - yn.max()
    else:
        xn = torch.full((N,), T, dtype=torch.int, device="cuda")
        yn = torch.full((N,), U - 1, dtype=torch.int, device="cuda")
    return xs, ys, xn, yn


def check_properties(xs, ys, xn, yn, costs, grads, flow_tol):
    N, T, U, V = xs.shape
    assert torch.isfinite(costs).all()
    assert (grads <= 0).all()
    idx = torch.zeros((N, T, U, 2), dtype=torch.long, device="cuda")
    idx[:, :, :U - 1, 1] = ys.long().unsqueeze(1)
    pair = grads.gather(3, idx)                                  # (N,T,U,2): blank, label
    pair[:, :, U - 1, 1] = 0                                     # last column: index 1 re-reads the blank
    # nothing outside the two columns
    total = grads.double().sum()
    assert abs((pair.double().sum() - total).item()) <= 1e-6 * abs(total.item())
    # padding is exactly zero
    tmask = torch.arange(T, device="cuda")[None, :] >= xn[:, None]
    umask = torch.arange(U, device="cuda")[None, :] >= (yn + 1)[:, None]
    assert grads[tmask].abs().max().item() == 0 if tmask.any() else True
    assert grads.transpose(1, 2)[umask].abs().max().item() == 0 if umask.any() else True
    # flow conservation per anti-diagonal
    flow = -(pair.double().sum(-1))                              # (N,T,U)
    d = (torch.arange(T, device="cuda")[:, None] + torch.arange(U, device="cuda")[None, :]).reshape(-1)
    per = torch.zeros((N, T + U - 1), dtype=torch.double, device="cuda")
    per.index_add_(1, d, flow.reshape(N, -1))
    nd = (xn + yn).long()                                        # diagonals 0 .. Tn+Un-2 carry flow
    dd = torch.arange(T + U - 1, device="cuda")[None, :]
    live = dd < nd[:, None]
    assert (per[live] - 1.0).abs().max().item() <= flow_tol, (per[live] - 1.0).abs().max().item()
    assert per[~live].abs().max().item() <= flow_tol if (~live).any() else True


def test_cfg2_full(w, reference):
    xs, ys, xn, yn = synth(128, 150, 40, 28, seed=128)
    w.set_lse_mode("fast")
    cf, gf = w._C.rnnt_loss(xs, ys, xn, yn)
    check_properties(xs, ys, xn, yn, cf, gf, flow_tol=2e-3)
    w.set_lse_mode("exact")
    ce, ge = w._C.rnnt_loss(xs, ys, xn, yn)
    args = (xs, ys, xn, yn)
    reference.check("dense", (ce, ge), lambda ref: ref.rnnt_loss(*args), args)     # bit-identical at full size
    # the opt-in fast LSE: fp32 noise against the reference (= ce, ge; measured 1.2e-4 on one of 21.5M
    # gradient elements -- the reference itself is 1.25e-4 from the fp64 oracle at this shape).
    # This is why the library default is the exact flavour.
    assert ((cf - ce).abs() / ce.abs()).max().item() <= 1e-5
    assert (gf - ge).abs().max().item() <= 2.5e-4
    w.set_lse_mode("auto")


def test_cfg2_random_lengths_python_api(w, reference):
    xs, ys, xn, yn = synth(128, 150, 40, 28, seed=7, random_lengths=True)
    w.set_lse_mode("exact")
    x = xs.clone().requires_grad_(True)
    loss = w.rnnt_loss(x, ys, xn, yn, reduction="sum", gather=True)
    loss.backward()
    costs, grads = w._C.rnnt_loss(xs, ys, xn, yn)
    assert torch.equal(x.grad, grads)                              # deferred emit == eager emit, bit for bit
    check_properties(xs, ys, xn, yn, costs, grads, flow_tol=2e-3)
    args = (xs, ys, xn, yn)
    reference.check("dense", (costs, grads), lambda ref: ref.rnnt_loss(*args), args)
    w.set_lse_mode("auto")


def test_cfg3_full(w, reference):
    xs, ys, xn, yn = synth(32, 150, 20, 5000, seed=32)
    w.set_lse_mode("exact")
    ce, ge = w._C.rnnt_loss(xs, ys, xn, yn)
    check_properties(xs, ys, xn, yn, ce, ge, flow_tol=2e-3)
    args = (xs, ys, xn, yn)
    reference.check("dense", (ce, ge), lambda ref: ref.rnnt_loss(*args), args)
    w.set_lse_mode("auto")


def test_cfg4_full_dense_and_compact(w):
    """N=64 T=1500 U=300 V=50 (the reference needs 14 s per call on B200 here; properties instead)."""
    N, T, U, V = 64, 1500, 300, 50
    xs, ys, xn, yn = synth(N, T, U, V, seed=64, random_lengths=True)
    w.set_lse_mode("fast")
    costs, grads = w._C.rnnt_loss(xs, ys, xn, yn)
    check_properties(xs, ys, xn, yn, costs, grads, flow_tol=3e-2)     # 1800 fp32 steps at |alpha| ~ 6000 (ulp 5e-4)
    # compact layout on the same data
    xs_c = torch.cat([xs[i, :xn[i], :yn[i] + 1].reshape(-1, V) for i in range(N)], 0).contiguous()
    ys_c = torch.cat([ys[i, :yn[i]] for i in range(N)], 0).contiguous()
    cc, pg, loc = w._C.rnnt_loss_compact(xs_c, ys_c, xn, yn)
    assert ((cc - costs).abs() / costs.abs()).max().item() <= 1e-6
    cum = torch.cumsum(xn * (yn + 1), 0, dtype=torch.int32)
    gc = w._C.rnnt_loss_compact_backward(torch.ones_like(cc), pg, cum, loc, V, 0)
    off = 0
    for i in (0, N // 2, N - 1):                                      # spot-check three lattices against the dense path
        off = int(cum[i - 1]) if i > 0 else 0
        c = int(xn[i]) * (int(yn[i]) + 1)
        a = gc[off:off + c].reshape(int(xn[i]), int(yn[i]) + 1, V)
        b = grads[i, :xn[i], :yn[i] + 1]
        assert (a - b).abs().max().item() <= 1e-6
    w.set_lse_mode("auto")


def test_cfg5_microbatch_independence_and_64bit(w, reference):
    """N=32 T=600 U=150 V=1024: 2.9e9 gradient elements (> 2^31, the reference's int idx4 overflows
    beyond 23 lattices, core.cu:22-24).  A batch must equal its sub-batches bit for bit."""
    N, T, U, V = 32, 600, 150, 1024
    xs, ys, xn, yn = synth(N, T, U, V, seed=5, random_lengths=True)
    w.set_lse_mode("exact")
    costs, grads = w._C.rnnt_loss(xs, ys, xn, yn)
    for lo, hi in ((0, 16), (16, 32)):
        c2, g2 = w._C.rnnt_loss(xs[lo:hi].contiguous(), ys[lo:hi].contiguous(), xn[lo:hi].contiguous(),
                                yn[lo:hi].contiguous())
        assert torch.equal(costs[lo:hi], c2) and torch.equal(grads[lo:hi], g2)
        del c2, g2
    k = 4                                                              # the reference on the last 4 lattices
    args = tuple(t[N - k:].contiguous() for t in (xs, ys, xn, yn))
    reference.check("dense", (costs[N - k:], grads[N - k:]), lambda ref: ref.rnnt_loss(*args), args)
    w.set_lse_mode("auto")
