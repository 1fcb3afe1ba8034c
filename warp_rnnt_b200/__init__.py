"""warp_rnnt_b200 -- B200-native RNN-Transducer loss, drop-in for 1ytic/warp-rnnt's
``warp_rnnt.rnnt_loss`` (reference: /root/reference/pytorch_binding/warp_rnnt/__init__.py).

Same public surface as the reference module (``__init__.py:9-143``):

    rnnt_loss(log_probs, labels, frames_lengths, labels_lengths, average_frames=False,
              reduction='none', blank=0, gather=False, fastemit_lambda=0.0, compact=False)
    RNNTLoss, RNNTLossCompact (autograd Functions), __version__, and the operator module ``_C``
    (rnnt_loss / rnnt_loss_compact / rnnt_loss_compact_backward, same kwargs and error strings).

Host code here is plumbing only (argument handling, autograd wiring); all arithmetic runs in the
hand-written sm_100a kernels of ``lib/librnnt_b200.so`` through ``lib/_C.so``.  There is no CPU or
eager-PyTorch fallback: importing this package without the built extension raises ImportError.
"""
import contextlib
import importlib.machinery
import importlib.util
import os
import sys
import threading

import torch

__version__ = "0.1.0"

_HERE = os.path.dirname(os.path.abspath(__file__))
_EXT_PATH = os.path.join(_HERE, "lib", "_C.so")
_LIB_PATH = os.path.join(_HERE, "lib", "librnnt_b200.so")


def _load_ext():
    # Stale binaries must not load silently: lib/sources.sha256 records the content hash of the sources the two
    # artefacts were built from; on a mismatch (edited sources, a pull) they are rebuilt -- or, with
    # RNNT_B200_NO_AUTOBUILD=1, the import fails.
    from . import build as _build
    if not _build.up_to_date():
        if os.environ.get("RNNT_B200_NO_AUTOBUILD") == "1":
            raise ImportError(
                "warp_rnnt_b200: the CUDA extension is missing or older than its sources (%s). "
                "Run `python -m warp_rnnt_b200.build`; there is no CPU fallback." % _EXT_PATH)
        _build.build_all()                   # builds the CUDA extension itself (nvcc + g++)
    name = __name__ + "._C"
    loader = importlib.machinery.ExtensionFileLoader(name, _EXT_PATH)
    spec = importlib.util.spec_from_file_location(name, _EXT_PATH, loader=loader)
    mod = importlib.util.module_from_spec(spec)
    loader.exec_module(mod)
    sys.modules[name] = mod
    return mod


_C = _load_ext()
core = _C

LSE_AUTO, LSE_EXACT, LSE_FAST = 0, 1, 2


def set_lse_mode(mode):
    """'auto' | 'exact' | 'fast' (see include/rnnt_b200.h rnntLseMode_t).  'exact' (= 'auto', the
    default) reproduces the reference kernels' alpha/beta/cost/gradient bits; 'fast' shortens the
    wavefront's dependent chain at the price of fp32-noise-level differences (<= ~1e-4 on gradients)."""
    _C.set_lse_mode({"auto": 0, "exact": 1, "fast": 2}[mode] if isinstance(mode, str) else int(mode))


class RNNTLoss(torch.autograd.Function):
    """Dense loss, ONE kernel launch per step.  Reference: ``RNNTLoss`` (__init__.py:9-24).

    Like the reference, forward produces the dense gradient; unlike it, the python-level reduction
    (average_frames, 'sum' / 'mean', __init__.py:132-143) is part of this Function: the per-sample weights
    ``weights[n]`` (1/N, 1/frames, ...) go into the kernel as ``grad_scale``, the kernel returns
    ``sum_n weights[n] * cost[n]`` itself (``reduce=True``) and the gradient it wrote already is
    d(loss)/d(log_probs).  Backward then only has to compare the upstream gradient with what was multiplied
    in (``rnnt_rescale_``: a tiny launch that touches no gradient memory when they agree -- the usual
    ``loss.backward()``) instead of the reference's dense ``mul_`` (two more passes over (N,T,U,V)).

    With ``blank == -1`` the input is the gathered (N,T,U,2) layout of the reference's operator boundary
    (binding.cpp:81-90); weights / reduce are not supported there."""

    @staticmethod
    def forward(ctx, log_probs, labels, frames_lengths, labels_lengths, blank=0, fastemit_lambda=0.0,
                weights=None, reduce=False):
        need = ctx.needs_input_grad[0]
        ctx.need = need
        if blank == -1:
            assert weights is None and not reduce
            costs, grads = _C.rnnt_loss_dense(log_probs, labels, frames_lengths, labels_lengths, -1,
                                              fastemit_lambda, None, need, 0)
            ctx.grads = grads if need else None
            return costs
        costs, grads, loss = _C.rnnt_loss_fused(log_probs, labels, frames_lengths, labels_lengths, blank,
                                                fastemit_lambda, weights, need, 0)
        ctx.grads = grads if need else None
        if reduce:
            return loss[0]
        return costs if weights is None else costs * weights

    @staticmethod
    def backward(ctx, grads_output):
        if not ctx.need:
            return None, None, None, None, None, None, None, None
        g, ctx.grads = ctx.grads, None       # hand the buffer over: autograd can then adopt it as .grad without a copy
        if g is None:
            raise RuntimeError("RNNTLoss: backward called a second time, but the gradient buffer produced by forward "
                               "has already been handed to autograd (run forward again)")
        go = grads_output.detach().reshape(-1).to(torch.float32).contiguous()
        _C.rnnt_rescale_(g, go, None)        # in place, like the reference's mul_ (__init__.py:23); no-op when go == 1
        return g, None, None, None, None, None, None, None


class RNNTLossGather(torch.autograd.Function):
    """``gather=True``: the reference's memory-saving mode (__init__.py:118-128).  Forward keeps the gradient in
    its (N,T,U,2) [blank,label] form -- the log-prob gather runs inside the forward kernel, without the int64
    index tensor -- and backward emits the dense (N,T,U,V) tensor once, already scaled by grad_output (replaces
    mul_ + GatherBackward's zeros + scatter_add_).  A label equal to ``blank`` adds both gradients, as
    torch.gather's backward does."""

    @staticmethod
    def forward(ctx, log_probs, labels, frames_lengths, labels_lengths, blank=0, fastemit_lambda=0.0):
        need = ctx.needs_input_grad[0]
        costs, pg = _C.rnnt_gather_forward(log_probs, labels, frames_lengths, labels_lengths, blank,
                                           fastemit_lambda, need, 0)
        ctx.grads = pg if need else None
        ctx.labels = labels
        ctx.yn = labels_lengths
        ctx.V = log_probs.size(3)
        ctx.blank = blank
        return costs

    @staticmethod
    def backward(ctx, grads_output):
        if ctx.grads is None:
            return None, None, None, None, None, None
        go = grads_output.contiguous().to(ctx.grads.dtype)
        g = _C.rnnt_gather_backward(ctx.grads, ctx.labels, go, ctx.V, ctx.blank, True, ctx.yn)
        return g, None, None, None, None, None


class RNNTLossFromLogits(torch.autograd.Function):
    """Loss straight from un-normalised joint-network logits: ``log_softmax`` fused into the loss (SURVEY.md 8(f)1).

    The reference needs log-softmaxed input (README.md:59; its benchmark times ``F.log_softmax`` with the loss,
    benchmark.py:65): seven dense passes over (N,T,U,V) per step.  Here forward reads the logits once (per-cell
    normaliser + the two log-probs the recurrence needs) and keeps a (N,T,U,2) gradient; backward reads them once more
    and writes d loss / d LOGITS, applying log_softmax's backward on the fly: three dense passes.

    Logits may be float32 or bfloat16 (e.g. a joint network run under ``torch.autocast(dtype=torch.bfloat16)``).  With
    bfloat16 the two dense passes move half the bytes, the costs are float32, and the gradient handed to autograd is
    bfloat16: all arithmetic is float32, and the results are bit for bit those of the float32 path on
    ``logits.float()``, with the gradient rounded once to bfloat16."""

    @staticmethod
    def forward(ctx, logits, labels, frames_lengths, labels_lengths, blank=0, fastemit_lambda=0.0):
        need = ctx.needs_input_grad[0]
        costs, lse, pg = _C.rnnt_logits_forward(logits, labels, frames_lengths, labels_lengths, blank,
                                                fastemit_lambda, need, 0)
        if need:
            ctx.save_for_backward(logits, lse, pg, labels)
            ctx.blank = blank
        return costs

    @staticmethod
    def backward(ctx, grads_output):
        logits, lse, pg, labels = ctx.saved_tensors
        go = grads_output.contiguous().to(torch.float32)
        return _C.rnnt_logits_backward(logits, lse, pg, labels, go, ctx.blank), None, None, None, None, None


def rnnt_loss_from_logits(logits, labels, frames_lengths, labels_lengths, average_frames=False, reduction="none",
                          blank=0, fastemit_lambda=0.0):
    """``rnnt_loss(log_softmax(logits, -1), ...)`` in three dense passes instead of seven; the gradient is w.r.t. the
    LOGITS.  Dense (N,T,U,V) layout, float32 or bfloat16 logits (bfloat16: float32 costs and arithmetic, bfloat16
    gradient, see ``RNNTLossFromLogits``); other arguments as in ``rnnt_loss``.  The loss is float32 for either dtype.
    Agrees with ``torch.log_softmax`` + the reference to 1e-5 (costs, relative) / 1e-4 (gradients), not bit for bit."""
    assert average_frames is None or isinstance(average_frames, bool)
    assert reduction is None or reduction in ("none", "mean", "sum")
    assert isinstance(blank, int)
    assert not labels.requires_grad and not frames_lengths.requires_grad and not labels_lengths.requires_grad
    costs = RNNTLossFromLogits.apply(logits, labels, frames_lengths, labels_lengths, blank, fastemit_lambda)
    if average_frames:
        costs = costs / frames_lengths.to(torch.float32)       # not the logits' dtype: bf16 would round 257 frames to 256
    if reduction == "sum":
        return costs.sum()
    if reduction == "mean":
        return costs.mean()
    return costs


class JointPack(torch.autograd.Function):
    """x[(n,t,u), :] = f[n,t,:] + g[n,u,:] in the compact (ragged) row order that ``rnnt_loss(compact=True)`` takes --
    the joint network's input without padding (the reference's benchmark2.py:37-50 builds it with a python loop over
    the batch).  One kernel forward, two deterministic reductions backward."""

    @staticmethod
    def forward(ctx, f, g, lf, lg, stu=-1):
        x, mem_pref = _C.rnnt_joint_pack(f.contiguous(), g.contiguous(), lf, lg, int(stu))
        ctx.save_for_backward(lf, lg, mem_pref)
        ctx.shape = (f.size(1), g.size(1))
        return x

    @staticmethod
    def backward(ctx, dx):
        lf, lg, mem_pref = ctx.saved_tensors
        df, dg = _C.rnnt_joint_pack_backward(dx.contiguous().float(), lf, lg, mem_pref, ctx.shape[0], ctx.shape[1])
        return df, dg, None, None, None


def joint_pack(f, g, frames_lengths, labels_lengths, stu=None):
    """f (N,T,H) encoder output, g (N,U+1,H) predictor output -> (STU,H), STU = sum frames_lengths*(labels_lengths+1):
    the packed input of the joint network whose (STU,V) log-softmax output goes to ``rnnt_loss(..., compact=True)``.
    ``stu``: pass STU when known to avoid the one device->host copy that sizes the output."""
    return JointPack.apply(f, g, frames_lengths, labels_lengths, -1 if stu is None else int(stu))


class RNNTLossEager(torch.autograd.Function):
    """Reference-shaped variant: dense gradients are produced in forward (one fused pass) and
    scaled in backward, exactly like the reference's RNNTLoss (__init__.py:11-24)."""

    @staticmethod
    def forward(ctx, log_probs, labels, frames_lengths, labels_lengths, blank=0, fastemit_lambda=0.0):
        costs, ctx.grads = _C.rnnt_loss(xs=log_probs, ys=labels, xn=frames_lengths, yn=labels_lengths,
                                        blank=blank, fastemit_lambda=fastemit_lambda)
        return costs

    @staticmethod
    def backward(ctx, grads_output):
        grads_output = grads_output.view(-1, 1, 1, 1).to(ctx.grads)
        return ctx.grads.mul_(grads_output), None, None, None, None, None


_tls = threading.local()


@contextlib.contextmanager
def compact_hints(max_T, max_U):
    """Inside this context ``rnnt_loss(compact=True)`` trusts the caller's upper bounds of ``frames_lengths`` and
    ``labels_lengths + 1`` and skips the shape validation that needs a device->host copy of the length sums (the
    reference does four ``.item()`` syncs there, binding.cpp:132-146): the forward then has no host sync at all
    and can be captured into a CUDA graph.  A sample exceeding the bounds gets cost NaN."""
    prev = getattr(_tls, "hints", None)
    _tls.hints = (int(max_T), int(max_U))
    try:
        yield
    finally:
        _tls.hints = prev


class RNNTLossCompact(torch.autograd.Function):
    """Compact (ragged) layout.  Reference: ``RNNTLossCompact`` (__init__.py:26-54)."""

    @staticmethod
    def forward(ctx, log_probs, labels, frames_lengths, labels_lengths, blank=0, fastemit_lambda=0.0,
                enable_grad: bool = True):
        hints = getattr(_tls, "hints", None) or (0, 0)
        costs, grads, loc = _C.rnnt_loss_compact(
            xs=log_probs, ys=labels, xn=frames_lengths, yn=labels_lengths, blank=blank,
            fastemit_lambda=fastemit_lambda, required_grad=enable_grad, max_T=hints[0], max_U=hints[1])
        if enable_grad:
            cumlen = torch.cumsum(frames_lengths * (labels_lengths + 1), dim=0, dtype=torch.int32)
            ctx.V = log_probs.size(-1)
            ctx.blank = blank
            ctx.save_for_backward(grads, loc, cumlen)
        return costs

    @staticmethod
    def backward(ctx, grads_output):
        grads, loc, cumlen = ctx.saved_tensors
        grads_input = _C.rnnt_loss_compact_backward(grads_output.contiguous().float(), grads, cumlen, loc,
                                                    ctx.V, ctx.blank)
        return grads_input, None, None, None, None, None, None


def rnnt_loss(log_probs, labels, frames_lengths, labels_lengths, average_frames=False, reduction="none",
              blank=0, gather=False, fastemit_lambda=0.0, compact=False):
    """The RNN-Transducer loss (same signature and semantics as the reference, __init__.py:57-143).

    Args:
        log_probs: (N, T, U, V) float32 log-softmaxed joint output; compact: (STU, V).  The dense path
            (gather=False, compact=False) also takes bfloat16: bf16 in, bf16 gradient out, float32 costs and
            arithmetic (the reference is float32-only, binding.cpp:17-19).
        labels: (N, U-1) int32; compact: (sum(labels_lengths),).
        frames_lengths, labels_lengths: (N,) int32.
        average_frames: divide each sample's loss by its number of frames.
        reduction: 'none' | 'mean' | 'sum' | None.
        blank: blank label id.
        gather: the reference's memory-saving mode: only a (N,T,U,2) gradient lives between forward and
            backward (the dense one is emitted by backward); follows torch.gather's backward for a label
            equal to ``blank`` (the two gradients add).  ``gather=False`` (default) is the fast path: one
            kernel launch produces loss and dense gradient.
        fastemit_lambda: FastEmit regularisation (scales label gradients by 1+lambda).
        compact: ragged layout, STU = sum(frames_lengths * (labels_lengths + 1)).
    """
    assert average_frames is None or isinstance(average_frames, bool)
    assert reduction is None or reduction in ("none", "mean", "sum")
    assert isinstance(blank, int)
    assert isinstance(gather, bool)

    assert not labels.requires_grad, "labels does not require gradients"
    assert not frames_lengths.requires_grad, "frames_lengths does not require gradients"
    assert not labels_lengths.requires_grad, "labels_lengths does not require gradients"

    if compact:
        costs = RNNTLossCompact.apply(log_probs.float(), labels, frames_lengths, labels_lengths, blank,
                                      fastemit_lambda,
                                      (log_probs.requires_grad and torch.is_grad_enabled()))
    elif gather:
        assert log_probs.dtype == torch.float32, "gather=True takes float32 log_probs (bfloat16: gather=False)"
        costs = RNNTLossGather.apply(log_probs, labels, frames_lengths, labels_lengths, blank, fastemit_lambda)
    else:
        # dense path: the reduction below is folded into the one kernel launch (see RNNTLoss)
        if reduction not in ("none", "mean", "sum", None):
            raise ValueError(
                f"Unknown reduction method: {reduction}, expected to be one of ['mean', 'sum', 'none']")
        reduce = reduction in ("mean", "sum")
        weights = None                                   # float32 also for bfloat16 log_probs (costs are float32)
        if average_frames:
            weights = 1.0 / frames_lengths.to(torch.float32)
        if reduction == "mean":
            n = max(int(log_probs.size(0)), 1)
            weights = torch.full((log_probs.size(0),), 1.0 / n, dtype=torch.float32, device=log_probs.device) \
                if weights is None else weights / n
        return RNNTLoss.apply(log_probs, labels, frames_lengths, labels_lengths, blank, fastemit_lambda, weights,
                              reduce)

    if average_frames:
        costs = costs / frames_lengths.to(log_probs)

    if reduction == "none" or reduction is None:
        return costs
    elif reduction == "sum":
        return costs.sum()
    elif reduction == "mean":
        return costs.mean()
    else:
        raise ValueError(
            f"Unknown reduction method: {reduction}, expected to be one of ['mean', 'sum', 'none']")


__all__ = ["rnnt_loss", "rnnt_loss_from_logits", "joint_pack", "JointPack", "RNNTLossFromLogits", "RNNTLoss", "RNNTLossGather", "RNNTLossEager", "RNNTLossCompact", "compact_hints", "set_lse_mode", "core", "_C",
           "__version__"]
