"""Shared helpers for the tests: golden vectors, synthetic inputs (the reference's recipe), the recorded outputs of
the reference kernels."""
import hashlib
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "reference_vectors.json")))
REFERENCE_OUTPUTS = os.path.join(HERE, "golden", "reference_outputs.json")
RECORD_ENV = "RNNT_B200_RECORD_REFERENCE"


def log_softmax(x, axis=-1):
    x = np.asarray(x, dtype=np.float64)
    m = x.max(axis=axis, keepdims=True)
    y = x - m
    return y - np.log(np.exp(y).sum(axis=axis, keepdims=True))


def golden_case(name):
    """-> dict(lp f32 (N,T,U,V) log-softmaxed, ys, xn, yn, costs, grads)."""
    r = GOLDEN[name]
    xs = np.asarray(r["xs"], dtype=np.float32)
    # the reference tests log_softmax in fp32 torch (test.py:42); fp64-then-round is within 1 ulp
    lp = log_softmax(xs).astype(np.float32)
    ys = np.asarray(r["ys"], dtype=np.int32).reshape(xs.shape[0], -1)
    costs = np.atleast_1d(np.asarray(r.get("expected_costs", r.get("expected_cost")), dtype=np.float64))
    return dict(lp=lp, ys=ys, xn=np.asarray(r["xn"], dtype=np.int32), yn=np.asarray(r["yn"], dtype=np.int32),
                costs=costs, grads=np.asarray(r["expected_grads"], dtype=np.float64))


def make_inputs(N, T, U, V, seed=0, random_lengths=False, blank=0, min_len=True):
    """Synthetic inputs following the reference's benchmark recipe (benchmark.py:11-27):
    randn -> log_softmax, labels in [1,V) (never blank when blank == 0), full or random lengths
    (random: benchmark.py:20-23, shifted so the max hits T / U-1)."""
    rng = np.random.RandomState(seed)
    xs = rng.randn(N, T, U, V).astype(np.float32)
    lp = log_softmax(xs).astype(np.float32)
    if V > 1:
        ys = rng.randint(0, V - 1, (N, max(U - 1, 0))).astype(np.int32)
        ys = np.where(ys >= blank, ys + 1, ys).astype(np.int32)     # skip the blank id
    else:
        ys = np.zeros((N, max(U - 1, 0)), dtype=np.int32)
    if random_lengths:
        xn = rng.randint(max(T // 2, 1), T + 1, (N,)).astype(np.int32)
        yn = rng.randint(U // 2, U, (N,)).astype(np.int32) if U > 1 else np.zeros(N, np.int32)
        xn = xn + T - xn.max()
        yn = yn + (U - 1) - yn.max()
    else:
        xn = np.full(N, T, dtype=np.int32)
        yn = np.full(N, U - 1, dtype=np.int32)
    return lp, ys, xn, yn


def to_compact(lp, ys, xn, yn):
    """Ragged concat as in the reference test (test.py:291-299)."""
    V = lp.shape[-1]
    xs_c = np.concatenate([lp[i, :xn[i], :yn[i] + 1].reshape(-1, V) for i in range(lp.shape[0])], axis=0)
    ys_c = np.concatenate([ys[i, :yn[i]] for i in range(ys.shape[0])], axis=0).astype(np.int32)
    return np.ascontiguousarray(xs_c), np.ascontiguousarray(ys_c)


def from_compact(flat, xn, yn, T, U):
    """(STU,V) -> padded (N,T,U,V) with zeros."""
    V = flat.shape[-1]
    N = len(xn)
    out = np.zeros((N, T, U, V), dtype=flat.dtype)
    o = 0
    for i in range(N):
        c = int(xn[i]) * (int(yn[i]) + 1)
        out[i, :xn[i], :yn[i] + 1] = flat[o:o + c].reshape(xn[i], yn[i] + 1, V)
        o += c
    return out


def compact_defined(costs, pair_grads, loc, blank):
    """The entries of a compact forward's result that the reference kernels define: the reference never writes the
    label slot of a sample's last column when that sample has the batch's maximum label length (grid.y = U-1 in
    core_compact.cu:392 never reaches u == yn[n]), so those entries of its torch::empty buffer are uninitialised; the
    backward ignores them (loc == blank, core_compact.cu:482)."""
    return costs, loc, pair_grads[:, 0], pair_grads[:, 1][loc != blank]


# ------------------------------------------------------------------------------ outputs of the reference kernels
# LSE mode 'exact' must reproduce the unmodified reference kernels (1ytic/warp-rnnt, compiled for sm_100a by
# oracle/build_ref.py) bit for bit.  What they returned for the tests' inputs on a B200 is stored in
# golden/reference_outputs.json as a SHA-256 digest per tensor (plus a few sampled non-zero values for the error
# message), so the comparison needs neither the reference's sources nor its build.
# RNNT_B200_RECORD_REFERENCE=<file.json> records instead: every check runs the reference (oracle/_ref must be built),
# asserts live equality with this library and writes the reference's digests to <file.json>.
def digest(t):
    a = t.detach().contiguous().cpu().numpy()
    flat = a.reshape(-1)
    nz = np.flatnonzero(flat)
    pick = np.sort(np.random.RandomState(0).choice(nz, min(8, nz.size), replace=False)) if nz.size else []
    return {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": hashlib.sha256(a.tobytes()).hexdigest(),
            "sample": [[int(i), float(flat[i])] for i in pick]}


def _differences(what, ours, stored):
    out = []
    for k, (t, d) in enumerate(zip(ours, stored)):
        o = digest(t)
        if o["sha256"] == d["sha256"]:
            continue
        flat = t.detach().contiguous().cpu().reshape(-1)
        seen = [(i, float(flat[i]) if i < flat.numel() else None, v) for i, v in d["sample"]]
        out.append("%s %d: shape/dtype %s %s, recorded %s %s; sampled [index, ours, recorded]: %s"
                   % (what, k, o["shape"], o["dtype"], d["shape"], d["dtype"], seen))
    return out


class ReferenceOutputs:
    """``check(label, ours, run_reference, inputs)``: the tensors ``ours`` must equal, bit for bit, what
    ``run_reference(ref)`` returned when the reference module ``ref`` ran on ``inputs`` (the inputs' digests are
    stored too, so that a change of the input generation is told apart from a change of the kernels)."""

    _ref = None

    def __init__(self, request):
        self.test = "%s::%s" % (os.path.basename(str(request.node.fspath)), request.node.name)

    def check(self, label, ours, run_reference, inputs=()):
        key = self.test + "/" + label
        ours = list(ours)
        path = os.environ.get(RECORD_ENV)
        if path:
            if ReferenceOutputs._ref is None:
                from oracle import build_ref
                ReferenceOutputs._ref = build_ref.load()
                assert ReferenceOutputs._ref is not None, "recording needs oracle/_ref (python oracle/build_ref.py)"
            theirs = list(run_reference(ReferenceOutputs._ref))
            import torch
            db = json.load(open(path)) if os.path.exists(path) else {
                "recorded_on": "%s, torch %s" % (torch.cuda.get_device_name(), torch.__version__), "outputs": {}}
            db["outputs"][key] = {"inputs": [digest(t) for t in inputs], "outputs": [digest(t) for t in theirs]}
            with open(path, "w") as f:                     # one line per check
                f.write('{"recorded_on": %s,\n "outputs": {\n' % json.dumps(db["recorded_on"]))
                f.write(",\n".join("  %s: %s" % (json.dumps(k), json.dumps(v)) for k, v in sorted(db["outputs"].items())))
                f.write("\n }\n}\n")
            assert len(theirs) == len(ours), key
            for k, (a, b) in enumerate(zip(ours, theirs)):
                assert torch.equal(a, b), "%s: output %d differs from the reference" % (key, k)
            return
        stored = _recorded()["outputs"].get(key)
        if stored is None:
            pytest.fail("no recorded reference outputs for %s (record them with %s)" % (key, RECORD_ENV))
        bad = _differences("input", list(inputs), stored["inputs"])
        if bad:
            pytest.fail("%s: the inputs are not the ones the reference outputs were recorded for (%s):\n%s"
                        % (key, _recorded()["recorded_on"], "\n".join(bad)))
        assert len(ours) == len(stored["outputs"]), key
        bad = _differences("output", ours, stored["outputs"])
        assert not bad, "%s: not bit-identical to the reference kernels:\n%s" % (key, "\n".join(bad))


_RECORDED = []


def _recorded():
    if not _RECORDED:
        _RECORDED.append(json.load(open(REFERENCE_OUTPUTS)))
    return _RECORDED[0]
