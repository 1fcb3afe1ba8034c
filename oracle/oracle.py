"""ctypes front end of oracle/rnnt_oracle.c + a numpy restatement (awni ref_transduce style).

TEST INFRASTRUCTURE ONLY -- this is the checker, never the product.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import it.
The product package (warp_rnnt_b200) never imports anything from oracle/.

Reference citations (/root/reference/...): core.cu:41-370 (alpha, beta, grads, costs),
core_gather.cu (V=2 form), core_compact.cu:29-484 (ragged form), pytorch_binding/warp_rnnt/
__init__.py:57-143 (python-level gather / average_frames / reduction).
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "librnnt_oracle.so")
_lib = None


def build(force=False):
    """gcc -> oracle/_build/librnnt_oracle.so (rebuilt when a source is newer); into a fresh temporary
    directory instead when oracle/ cannot be written (a read-only checkout)."""
    srcs = [os.path.join(_HERE, f) for f in ("rnnt_oracle.c", "rnnt_oracle_body.inc")]
    stale = force or not os.path.exists(_LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs)
    if not stale:
        return _LIB_PATH
    out = _LIB_PATH
    try:
        os.makedirs(os.path.dirname(_LIB_PATH), exist_ok=True)
    except OSError:
        pass
    if not os.access(os.path.dirname(_LIB_PATH), os.W_OK):
        out = os.path.join(tempfile.mkdtemp(prefix="rnnt_oracle_"), os.path.basename(_LIB_PATH))
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-o", out, srcs[0], "-lm"])
    return out


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.rnnt_oracle_num_threads.restype = ctypes.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _prep(lp, labels, xn, yn):
    lp = np.ascontiguousarray(lp, dtype=np.float32)
    labels = np.ascontiguousarray(labels, dtype=np.int32)
    xn = np.ascontiguousarray(xn, dtype=np.int32)
    yn = np.ascontiguousarray(yn, dtype=np.int32)
    return lp, labels, xn, yn


def num_threads():
    return lib().rnnt_oracle_num_threads()


def set_threads(n):
    lib().rnnt_oracle_set_threads(ctypes.c_int(int(n)))


def dense(lp, labels, xn, yn, blank=0, fastemit_lambda=0.0, dtype="f64", guard=False,
          want_grads=True, want_ab=False):
    """Dense (N,T,U,V) [or gathered (N,T,U,2) with blank=-1] loss + grads.

    Returns (costs (N,), grads like lp or None[, alphas, betas (N,T,U)])."""
    lp, labels, xn, yn = _prep(lp, labels, xn, yn)
    N, T, U, V = lp.shape
    real = np.float64 if dtype == "f64" else np.float32
    costs = np.zeros(N, dtype=real)
    grads = np.empty(lp.shape, dtype=real) if want_grads else None
    al = np.full((N, T, U), np.nan, dtype=real) if want_ab else None
    be = np.full((N, T, U), np.nan, dtype=real) if want_ab else None
    fn = getattr(lib(), "rnnt_oracle_dense_" + dtype)
    rc = fn(_p(lp), _p(labels), _p(xn), _p(yn), N, T, U, V, int(blank),
            ctypes.c_double(fastemit_lambda), int(bool(guard)), _p(costs), _p(grads), _p(al), _p(be))
    if rc != 0:
        raise ValueError("rnnt_oracle_dense: bad argument (lengths out of range?)")
    if want_ab:
        return costs, grads, al, be
    return costs, grads


def compact(xs, ys, xn, yn, blank=0, fastemit_lambda=0.0, dtype="f64", want_grads=True):
    """Compact forward: returns (costs (N,), pair_grads (STU,2) or None, loc (STU,) int64)."""
    xs, ys, xn, yn = _prep(xs, ys, xn, yn)
    STU, V = xs.shape
    N = xn.shape[0]
    assert STU == int((xn.astype(np.int64) * (yn.astype(np.int64) + 1)).sum())
    real = np.float64 if dtype == "f64" else np.float32
    costs = np.zeros(N, dtype=real)
    pg = np.empty((STU, 2), dtype=real) if want_grads else None
    loc = np.empty(STU, dtype=np.int64)
    fn = getattr(lib(), "rnnt_oracle_compact_" + dtype)
    rc = fn(_p(xs), _p(ys), _p(xn), _p(yn), N, V, int(blank), ctypes.c_double(fastemit_lambda),
            _p(costs), _p(pg), _p(loc))
    if rc != 0:
        raise ValueError("rnnt_oracle_compact: bad argument")
    return costs, pg, loc


def compact_scatter(grad_cost, pair_grads, loc, cum_lens, V, blank=0, dtype="f64"):
    """Compact backward: (STU,2) pair grads x grad_cost[n] scattered into zeros (STU,V)."""
    real = np.float64 if dtype == "f64" else np.float32
    grad_cost = np.ascontiguousarray(grad_cost, dtype=real)
    pair_grads = np.ascontiguousarray(pair_grads, dtype=real)
    loc = np.ascontiguousarray(loc, dtype=np.int64)
    cum_lens = np.ascontiguousarray(cum_lens, dtype=np.int32)
    STU = pair_grads.shape[0]
    out = np.empty((STU, V), dtype=real)
    fn = getattr(lib(), "rnnt_oracle_compact_scatter_" + dtype)
    fn(_p(grad_cost), _p(pair_grads), _p(loc), _p(cum_lens), ctypes.c_int64(STU),
       int(grad_cost.shape[0]), int(V), int(blank), _p(out))
    return out


def rnnt_loss(lp, labels, xn, yn, average_frames=False, reduction="none", blank=0, gather=False,
              fastemit_lambda=0.0, compact_layout=False, grad_output=None, dtype="f64"):
    """Python-level API restatement (__init__.py:57-143): returns (loss, d loss / d log_probs).

    grad_output: upstream gradient of the *returned* loss w.r.t. each per-sample cost is derived
    from reduction/average_frames; an explicit per-sample grad_output (N,) multiplies on top."""
    lp = np.asarray(lp)
    xn_ = np.asarray(xn)
    N = xn_.shape[0]
    if compact_layout:
        costs, pg, loc = compact(lp, labels, xn, yn, blank, fastemit_lambda, dtype)
    else:
        # gather=True is value-identical to the dense path (gather -> V=2 core -> scatter_add)
        costs, grads = dense(lp, labels, xn, yn, blank, fastemit_lambda, dtype)
    w = np.ones(N, dtype=np.float64)
    if average_frames:
        w = w / xn_.astype(np.float64)
    if reduction == "mean":
        w = w / N
    if grad_output is not None:
        w = w * np.asarray(grad_output, dtype=np.float64)
    per = costs.astype(np.float64) * (1.0 / xn_ if average_frames else 1.0)
    if reduction == "sum":
        loss = per.sum()
    elif reduction == "mean":
        loss = per.mean()
    else:
        loss = per
    if compact_layout:
        cum = np.cumsum(xn_.astype(np.int64) * (np.asarray(yn).astype(np.int64) + 1)).astype(np.int32)
        g = compact_scatter(w, pg, loc, cum, lp.shape[1], blank, dtype)
    else:
        g = grads * w.reshape(-1, 1, 1, 1)
    return loss, g


# --------------------------------------------------------------------------------------
# numpy restatement, per-sample double loop in fp64 (BASELINE config 1: "awni ref_transduce.py
# numpy forward/backward on CPU").  awni/transducer is not vendored in the reference
# (README.md:6,11 cite it by URL only), so this follows SURVEY.md section 0 = core.cu:41-332.
# --------------------------------------------------------------------------------------
def ref_transduce_np(lp, labels, blank=0, fastemit_lambda=0.0):
    """One lattice: lp (T,U,V) float, labels (U-1,) -> (cost, grads (T,U,V), alphas, betas)."""
    lp = np.asarray(lp, dtype=np.float64)
    T, U, V = lp.shape
    y = np.asarray(labels, dtype=np.int64)
    alphas = np.zeros((T, U))
    for t in range(1, T):
        alphas[t, 0] = alphas[t - 1, 0] + lp[t - 1, 0, blank]
    for u in range(1, U):
        alphas[0, u] = alphas[0, u - 1] + lp[0, u - 1, y[u - 1]]
    for t in range(1, T):
        for u in range(1, U):
            skip = alphas[t - 1, u] + lp[t - 1, u, blank]
            emit = alphas[t, u - 1] + lp[t, u - 1, y[u - 1]]
            alphas[t, u] = np.logaddexp(skip, emit)
    betas = np.zeros((T, U))
    betas[T - 1, U - 1] = lp[T - 1, U - 1, blank]
    for t in range(T - 2, -1, -1):
        betas[t, U - 1] = betas[t + 1, U - 1] + lp[t, U - 1, blank]
    for u in range(U - 2, -1, -1):
        betas[T - 1, u] = betas[T - 1, u + 1] + lp[T - 1, u, y[u]]
    for t in range(T - 2, -1, -1):
        for u in range(U - 2, -1, -1):
            skip = betas[t + 1, u] + lp[t, u, blank]
            emit = betas[t, u + 1] + lp[t, u, y[u]]
            betas[t, u] = np.logaddexp(skip, emit)
    ll = betas[0, 0]
    grads = np.zeros_like(lp)
    # blank: t < T-1 all u ; t == T-1 only u == U-1
    grads[:T - 1, :, blank] = -np.exp(alphas[:T - 1, :] + betas[1:, :] + lp[:T - 1, :, blank] - ll)
    grads[T - 1, U - 1, blank] = -np.exp(alphas[T - 1, U - 1] + lp[T - 1, U - 1, blank] - ll)
    for u in range(U - 1):
        grads[:, u, y[u]] = -(1.0 + fastemit_lambda) * np.exp(
            alphas[:, u] + betas[:, u + 1] + lp[:, u, y[u]] - ll)
    return -ll, grads, alphas, betas


def ref_transduce_np_batch(lp, labels, xn, yn, blank=0, fastemit_lambda=0.0):
    lp = np.asarray(lp)
    N, T, U, V = lp.shape
    costs = np.zeros(N)
    grads = np.zeros(lp.shape)
    for n in range(N):
        Tn, Un = int(xn[n]), int(yn[n]) + 1
        c, g, _, _ = ref_transduce_np(lp[n, :Tn, :Un], np.asarray(labels)[n, :Un - 1], blank,
                                      fastemit_lambda)
        costs[n] = c
        grads[n, :Tn, :Un] = g
    return costs, grads


# --------------------------------------------------------------------------------------
# Loss straight from un-normalised logits (the rebuild's fused log_softmax, SURVEY.md 8(f)1): the oracle composes
# the reference's own two steps in fp64 -- log_softmax (benchmark.py:65) then the loss -- and differentiates through
# both: d/d logit[v] = g_lp[v] - softmax[v] * sum_v' g_lp[v'].
# --------------------------------------------------------------------------------------
def from_logits(logits, labels, xn, yn, blank=0, fastemit_lambda=0.0, grad_output=None):
    """-> (costs (N,), d sum_n grad_output[n]*cost[n] / d logits (N,T,U,V)), fp64."""
    x = np.asarray(logits, dtype=np.float64)
    m = x.max(axis=-1, keepdims=True)
    lse = m + np.log(np.exp(x - m).sum(axis=-1, keepdims=True))
    lp = x - lse
    costs, g = dense(lp, labels, xn, yn, blank, fastemit_lambda)
    # a label equal to blank: dense() overrides (core.cu's launch order); autograd through log_softmax ADDS.  The
    # inputs of the tests avoid that case, as the reference's benchmark recipe does (labels in [1, V)).
    gl = g - np.exp(lp) * g.sum(axis=-1, keepdims=True)
    if grad_output is not None:
        gl = gl * np.asarray(grad_output, dtype=np.float64).reshape(-1, 1, 1, 1)
    return costs, gl
