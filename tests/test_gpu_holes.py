"""GPU: the code paths round 1 left without an oracle / reference comparison (VERDICT r1, "what's weak" 1-3).

  * BASELINE cfg 4 (N=64 T=1500 U=300 V=50, random lengths) in EXACT mode, dense and compact=True, against the
    fp64 oracle on 8 lattices and bit-for-bit against the reference kernels on 2 lattices; the 8-group multi-stream
    pipeline of the general path on a shape that takes it;
  * ring back-pressure in k_wavefront (a lattice longer than the boundary ring, and the compact C ABI without
    max_T / max_U hints);
  * the forward/backward mismatch guard's FIRED branch (core.cu:349-367) through a test-only hook;
  * two devices in one process (per-device function attributes, occupancy cache, pipeline streams).

Tolerances: costs |d|/|ref| <= 1e-5 against fp64; gradients max|d| <= gtol(T,U) = 2e-5 + 6e-6 (T+U) (fp32 alpha/beta
round at ulp(|alpha|) per anti-diagonal; the compiled reference sits at the same distance from fp64); bit for bit
against the recorded outputs of the reference kernels (tests/common.py ReferenceOutputs).
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from tests.common import ReferenceOutputs, compact_defined, make_inputs, to_compact

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gtol(T, U):
    return 2e-5 + 6e-6 * (T + U)


@pytest.fixture(scope="module")
def w():
    import warp_rnnt_b200
    return warp_rnnt_b200


@pytest.fixture
def reference(request):
    return ReferenceOutputs(request)


@pytest.fixture(scope="module")
def lib(w):
    L = ctypes.CDLL(os.path.join(ROOT, "warp_rnnt_b200", "lib", "librnnt_b200.so"))
    L.rnnt_b200_workspace_bytes.restype = ctypes.c_size_t
    L.rnnt_b200_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int]
    L.rnnt_b200_debug_guard_poison.argtypes = [ctypes.c_int, ctypes.c_float]
    L.rnnt_b200_debug_guard_poison.restype = None
    return L


def p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def cu(a, dev="cuda"):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def synth(N, T, U, V, seed, dev="cuda"):
    """benchmark2.py:81-85 style random lengths on the device (cfg 4 is 5.8 GB: too big to make on the host)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    xs = torch.log_softmax(torch.randn((N, T, U, V), device=dev, generator=g), dim=-1)
    ys = torch.randint(1, V, (N, U - 1), dtype=torch.int, device=dev, generator=g)
    xn = torch.randint(T // 2, T + 1, (N,), dtype=torch.int, device=dev, generator=g)
    yn = torch.randint(U // 2, U, (N,), dtype=torch.int, device=dev, generator=g)
    return xs, ys, xn + T - xn.max(), yn + (U - 1) - yn.max()


def ragged(xs, ys, xn, yn, idx):
    V = xs.shape[-1]
    xs_c = torch.cat([xs[i, :xn[i], :yn[i] + 1].reshape(-1, V) for i in idx], 0).contiguous()
    ys_c = torch.cat([ys[i, :yn[i]] for i in idx], 0).contiguous()
    return xs_c, ys_c


# ------------------------------------------------------------------------------------------ cfg 4, exact, at size
def test_cfg4_exact_dense_and_compact_vs_oracle_and_reference(w, reference):
    N, T, U, V = 64, 1500, 300, 50
    xs, ys, xn, yn = synth(N, T, U, V, seed=64)
    w.set_lse_mode("exact")
    try:
        costs, grads = w._C.rnnt_loss(xs, ys, xn, yn)              # full batch (serial general path: see the pipeline test)
        assert torch.isfinite(costs).all()
        pick = [0, 7, 8, 21, 33, 40, 55, 63]                        # lattices from different pipeline groups
        sel = torch.tensor(pick, device="cuda")
        lp_h, ys_h = xs[sel].cpu().numpy(), ys[sel].cpu().numpy()
        xn_h, yn_h = xn[sel].cpu().numpy(), yn[sel].cpu().numpy()
        c0, g0 = oracle.dense(lp_h, ys_h, xn_h, yn_h)               # fp64
        np.testing.assert_allclose(costs[sel].cpu().numpy(), c0, rtol=1e-5)
        # |alpha| reaches ~6000 here (fp32 ulp 4.9e-4) and 1800 anti-diagonals accumulate it: ANY fp32 implementation
        # sits ~1e-2 from fp64 on single gradient elements (SURVEY.md section 7); the compiled reference has the
        # identical error because it is bit-identical to this path (checked below).  Bound: 2 * gtol = 2.2e-2.
        err = np.abs(grads[sel].cpu().numpy() - g0).max()
        assert err <= 2 * gtol(T, U), err
        del g0
        # compact=True on the same data, full batch
        xs_c, ys_c = ragged(xs, ys, xn, yn, range(N))
        cc, pg, loc = w._C.rnnt_loss_compact(xs_c, ys_c, xn, yn)
        assert torch.equal(cc, costs) or ((cc - costs).abs() / costs.abs()).max().item() <= 1e-6
        cum = torch.cumsum(xn * (yn + 1), 0, dtype=torch.int32)
        go = torch.linspace(0.5, 1.5, N, device="cuda")
        gc = w._C.rnnt_loss_compact_backward(go, pg, cum, loc, V, 0)
        xs_s, ys_s = to_compact(lp_h, ys_h, xn_h, yn_h)
        cs, pgs, locs = oracle.compact(xs_s, ys_s, xn_h, yn_h)
        starts = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"), cum.long()])[:-1]
        o = 0
        for k, i in enumerate(pick):
            c = int(xn_h[k]) * (int(yn_h[k]) + 1)
            s = int(starts[i])
            np.testing.assert_allclose(cc[i].item(), cs[k], rtol=1e-5)
            assert np.array_equal(loc[s:s + c].cpu().numpy(), locs[o:o + c])
            e = np.abs(pg[s:s + c].cpu().numpy() - pgs[o:o + c]).max()
            assert e <= 2 * gtol(T, U), e
            dense_i = oracle.compact_scatter(np.array([go[i].item()]), pgs[o:o + c], locs[o:o + c],
                                             np.array([c], dtype=np.int32), V, 0)
            e = np.abs(gc[s:s + c].cpu().numpy() - dense_i).max()
            assert e <= 4 * gtol(T, U), e
            o += c
        # the reference on two of the lattices (14 s for the full batch on a B200, seconds for two): lattices are
        # independent, so its rows must equal ours bit for bit
        two = [7, 40]
        t2 = torch.tensor(two, device="cuda")
        a2 = (xs[t2].contiguous(), ys[t2].contiguous(), xn[t2].contiguous(), yn[t2].contiguous())
        reference.check("dense", (costs[t2], grads[t2]), lambda ref: ref.rnnt_loss(*a2), a2)
        # the reference's compact kernels take max lengths from ITS batch: compare per defined entry
        xs2, ys2 = ragged(xs, ys, xn, yn, two)
        cm, gm, lm = w._C.rnnt_loss_compact(xs2, ys2, a2[2], a2[3])
        reference.check("compact", compact_defined(cm, gm, lm, 0),
                        lambda ref: compact_defined(*ref.rnnt_loss_compact(xs2, ys2, a2[2], a2[3]), 0),
                        (xs2, ys2, a2[2], a2[3]))
        # ... and our full-batch compact run holds the same bits for these two lattices
        o = 0
        for i in two:
            c = int(xn[i]) * (int(yn[i]) + 1)
            s = int(starts[i])
            assert torch.equal(cc[i], cm[two.index(i)])
            assert torch.equal(pg[s:s + c], gm[o:o + c])
            o += c
    finally:
        w.set_lse_mode("auto")


# ------------------------------------------------------------------------------------------ the stream pipeline
def test_pipelined_general_path_vs_oracle_and_reference(w, reference):
    """N=32 T=300 U=70 V=1200: too large for the fused kernel, and the emit (3.2 GB) is long against the wavefront, so
    rnnt_b200_loss_dense runs its 8-group multi-stream pipeline (api.cu).  cfg 4 itself takes the serial path since
    round 2 (its wavefront is as long as its emit)."""
    N, T, U, V = 32, 300, 70, 1200
    xs, ys, xn, yn = synth(N, T, U, V, seed=32)
    w.set_lse_mode("exact")
    try:
        n0 = w._C.launch_count()
        costs, grads = w._C.rnnt_loss(xs, ys, xn, yn)
        assert w._C.launch_count() - n0 == 24                        # 8 groups x (gather, wavefront, emit)
        pick = [0, 5, 17, 31]
        sel = torch.tensor(pick, device="cuda")
        c0, g0 = oracle.dense(xs[sel].cpu().numpy(), ys[sel].cpu().numpy(), xn[sel].cpu().numpy(), yn[sel].cpu().numpy())
        np.testing.assert_allclose(costs[sel].cpu().numpy(), c0, rtol=1e-5)
        assert np.abs(grads[sel].cpu().numpy() - g0).max() <= gtol(T, U)
        two = torch.tensor([5, 31], device="cuda")
        a2 = (xs[two].contiguous(), ys[two].contiguous(), xn[two].contiguous(), yn[two].contiguous())
        reference.check("dense", (costs[two], grads[two]), lambda ref: ref.rnnt_loss(*a2), a2)
    finally:
        w.set_lse_mode("auto")


# ------------------------------------------------------------------------------------------ ring back-pressure
@pytest.mark.parametrize("mode", ["exact", "fast"])
def test_ring_backpressure_long_lattice(w, reference, mode):
    """Dense N=2 T=2600 U=300 V=3: ten warps per direction, boundary ring of 2048 rows < T -> the producer warp
    must wait for the consumer (wavefront.cu ring_put / ring_get with backpressure)."""
    N, T, U, V = 2, 2600, 300, 3
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=91, random_lengths=False)
    xn[1] = 2300                                                    # one lattice just above the ring, one well above
    yn[1] = 180
    args = (cu(lp), cu(ys), cu(xn), cu(yn))
    w.set_lse_mode(mode)
    try:
        costs, grads = w._C.rnnt_loss(*args)
        c0, g0 = oracle.dense(lp, ys, xn, yn)
        np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=1e-5)
        err = np.abs(grads.cpu().numpy() - g0).max()
        assert err <= 2 * gtol(T, U), err                           # fp32 noise at this length, see the cfg-4 test
        if mode == "exact":
            reference.check("dense", (costs, grads), lambda ref: ref.rnnt_loss(*args), args)
    finally:
        w.set_lse_mode("auto")


def test_ring_backpressure_compact_without_hints(w, lib):
    """rnnt_b200_compact_forward with max_T = max_U = 0: the launcher cannot size the ring, takes 128 slots, and a
    T=300 lattice runs with back-pressure (this is what the reference-ABI shim run_warp_rnnt_compact-style callers hit)."""
    N, T, U, V = 3, 300, 80, 6
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=17, random_lengths=True, blank=1)
    xs_c, ys_c = to_compact(lp, ys, xn, yn)
    STU = xs_c.shape[0]
    xs, y, a, b = cu(xs_c), cu(ys_c), cu(xn), cu(yn)
    ws = torch.empty(lib.rnnt_b200_workspace_bytes(STU, N), dtype=torch.uint8, device="cuda")
    costs, pg = torch.empty(N, device="cuda"), torch.empty(STU, 2, device="cuda")
    loc = torch.empty(STU, dtype=torch.int64, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for mode in (1, 2):                                             # exact, fast
        st = lib.rnnt_b200_compact_forward(stream, p(ws), ctypes.c_size_t(ws.numel()), p(xs), p(y), p(a), p(b),
                                           p(costs), p(pg), p(loc), None, ctypes.c_int64(STU), N, V, 1,
                                           ctypes.c_float(0.1), mode, 0, 0)
        assert st == 0
        c0, pg0, loc0 = oracle.compact(xs_c, ys_c, xn, yn, blank=1, fastemit_lambda=0.1)
        np.testing.assert_allclose(costs.cpu().numpy(), c0, rtol=1e-5)
        assert np.abs(pg.cpu().numpy() - pg0).max() <= gtol(T, U)
        assert np.array_equal(loc.cpu().numpy(), loc0)


# ------------------------------------------------------------------------------------------ the guard, fired
@pytest.mark.parametrize("shape", [(3, 20, 9, 7), (3, 700, 40, 5)])   # fused kernel / general path
@pytest.mark.parametrize("pairs", [False, True])
def test_mismatch_guard_fired_branch(w, lib, shape, pairs, capfd):
    """core.cu:349-367: |a-b|/|max(a,b)| > 1e-3 -> WARNING line, the sample's whole gradient slab is zero and
    cost = -(a+b)/2; other samples are untouched."""
    N, T, U, V = shape
    lp, ys, xn, yn = make_inputs(N, T, U, V, seed=3, random_lengths=True)
    if pairs:
        index = np.zeros((N, T, U, 2), dtype=np.int64)
        index[:, :, :U - 1, 1] = ys[:, None, :]
        lp = np.ascontiguousarray(np.take_along_axis(lp, index, axis=3))
    blank = -1 if pairs else 0
    args = (cu(lp), cu(ys), cu(xn), cu(yn))
    w.set_lse_mode("exact")
    try:
        c_clean, g_clean = w._C.rnnt_loss(*args, blank=blank)
        torch.cuda.synchronize()
        capfd.readouterr()
        victim = 1
        delta = 0.5 * float(c_clean[victim])                        # a = b + delta: ratio ~ 0.5 >> 1e-3
        lib.rnnt_b200_debug_guard_poison(victim, ctypes.c_float(-delta))   # ll = -cost: make a more negative
        try:
            c_bad, g_bad = w._C.rnnt_loss(*args, blank=blank)
            torch.cuda.synchronize()
        finally:
            lib.rnnt_b200_debug_guard_poison(-1, ctypes.c_float(0.0))
        out = capfd.readouterr().out
        assert "WARNING: sample %d" % victim in out and "forward/backward mismatch" in out
        assert g_bad[victim].abs().max().item() == 0.0              # zeroed slab
        b = -float(c_clean[victim])
        a = b - delta
        np.testing.assert_allclose(float(c_bad[victim]), -(a + b) / 2.0, rtol=2e-4)
        keep = [i for i in range(N) if i != victim]
        assert torch.equal(c_bad[keep], c_clean[keep]) and torch.equal(g_bad[keep], g_clean[keep])
        # and the hook is off again
        c3, g3 = w._C.rnnt_loss(*args, blank=blank)
        assert torch.equal(c3, c_clean) and torch.equal(g3, g_clean)
    finally:
        w.set_lse_mode("auto")


# ------------------------------------------------------------------------------------------ two devices, one process
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_in_one_process(w):
    """cuda:0 first, then cuda:1, same process: function attributes / occupancy / pipeline streams are per device."""
    shapes = [(5, 150, 40, 28, "fused, > 48 KB dynamic shared memory"),
              (3, 300, 600, 4, "general path, > 48 KB ring"),
              (32, 300, 70, 1200, "general path, multi-stream pipeline (3.2 GB of gradients, short wavefront)"),
              (40, 30, 20, 4096, "fused, several CTAs per lattice (occupancy cache)")]
    w.set_lse_mode("exact")
    try:
        for N, T, U, V, what in shapes:
            xs, ys, xn, yn = synth(N, T, U, V, seed=N + T, dev="cuda:0")
            outs = []
            for d in (0, 1, 0):
                dev = "cuda:%d" % d
                a = tuple(t.to(dev) for t in (xs, ys, xn, yn))
                c, g = w._C.rnnt_loss(*a)
                x = a[0].clone().requires_grad_(True)
                w.rnnt_loss(x, *a[1:], reduction="sum").backward()
                xs_c, ys_c = ragged(a[0], a[1], a[2], a[3], range(N))
                cc, pg, loc = w._C.rnnt_loss_compact(xs_c, ys_c, a[2], a[3])
                torch.cuda.synchronize(dev)
                assert c.device.index == d and g.device.index == d
                outs.append((c.cpu(), g.cpu(), x.grad.cpu(), cc.cpu(), pg.cpu()))
            for o in outs[1:]:
                for t0, t1 in zip(outs[0], o):
                    assert torch.equal(t0, t1), what
            k = min(N, 2)
            c0, g0 = oracle.dense(xs[:k].cpu().numpy(), ys[:k].cpu().numpy(), xn[:k].cpu().numpy(), yn[:k].cpu().numpy())
            np.testing.assert_allclose(outs[1][0][:k].numpy(), c0, rtol=1e-5)
            assert np.abs(outs[1][1][:k].numpy() - g0).max() <= gtol(T, U), what
    finally:
        w.set_lse_mode("auto")


def test_exact_log1p_restatement_is_libdevice_bit_for_bit(lib):
    """The exact LSE's log1p is libdevice's main path without its unreachable tail (csrc/common.cuh:log1pf_unit).
    The library's self-check kernel compares it with log1pf on EVERY float in [+0, 1] (2^30 - 2^23 + 1 patterns: the
    whole range of expf(d <= 0)), on NaNs, and both exact LSE flavours on 2^24 operand pairs: zero bit mismatches."""
    bad = torch.zeros(1, dtype=torch.int64, device="cuda")
    st = lib.rnnt_b200_debug_lse_selfcheck(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), p(bad))
    torch.cuda.synchronize()
    assert st == 0 and int(bad.item()) == 0
