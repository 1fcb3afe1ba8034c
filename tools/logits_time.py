"""Time rnnt_loss_from_logits on float32 and on bfloat16 logits of the same values, in one process.

    python tools/logits_time.py [--json PATH] [--calls 20] [--warmup 3] [--rounds 3]

Shapes: c2l (128,150,40,28) and c5mbl (32,600,150,1024) of bench.py, full lengths.  Timed: the forward op
(_C.rnnt_logits_forward: k_lse_pairs + the recurrence), the backward op (_C.rnnt_logits_backward: k_expand_logits) and,
at c5mbl, the whole step rnnt_loss_from_logits(x, ..., reduction='sum').backward().

Protocol: CUDA events around blocks of `calls` back-to-back calls after `warmup` calls, float32 and bf16 blocks
alternating for `rounds` rounds; the median block is reported.  The calls rotate over input sets whose bf16 logits
alone exceed the 126 MB L2 (c5mbl: one set is 5.9 GB; two sets).  The float32 logits are the bf16 ones converted, so the
outputs are also compared at the timed size: costs, lse and pair gradients bit for bit, and the bf16 logit gradient
against the float32 one rounded to bf16.

Per dense pass, achieved GB/s = algorithmic bytes / kernel time: the lse pass reads esz*cells*V bytes, the expand pass
reads and writes 2*esz*cells*V (esz = 4 or 2).  Kernel times come from a torch.profiler run of their own, after the
timed blocks.  Shares are of bench.peaks(), whose source is named in the output.  The card's name, power limit and
maximum SM clock are read in the same run (nvidia-smi, read-only query).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch

import bench
import warp_rnnt_b200 as w

SHAPES = {"c2l": (128, 150, 40, 28), "c5mbl": (32, 600, 150, 1024)}
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16}


def card():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"]
    try:
        out = subprocess.run(q, capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except Exception as e:                                   # the timing does not depend on it
        out = ["nvidia-smi failed: %s" % e]
    return {"torch_device": torch.cuda.get_device_name(), "nvidia_smi": out,
            "cuda_visible_devices": os.environ.get("CUDA_VISIBLE_DEVICES")}


def make_sets(N, T, U, V, dev):
    per_set = 2 * 2 * N * T * U * V                          # bf16 logits + bf16 gradient
    R = max(2, bench.rotation(per_set))
    sets = []
    for i in range(R):
        g = torch.Generator(device=dev).manual_seed(100 + i)
        xb = (torch.randn((N, T, U, V), device=dev, generator=g) * 3).to(torch.bfloat16)
        ys = torch.randint(1, V, (N, U - 1), device=dev, dtype=torch.int32, generator=g)
        xn = torch.full((N,), T, device=dev, dtype=torch.int32)
        yn = torch.full((N,), U - 1, device=dev, dtype=torch.int32)
        sets.append({"bf16": (xb, ys, xn, yn), "f32": (xb.float(), ys, xn, yn)})
    return sets


def block(fn, n_sets, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(calls):
        fn(i % n_sets)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def alternate(fns, n_sets, args):
    """fns: dtype -> fn(set index).  Median ms per call of each, blocks alternating."""
    for fn in fns.values():
        for i in range(args.warmup):
            fn(i % n_sets)
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(args.rounds):
        for k, fn in fns.items():
            times[k].append(block(fn, n_sets, args.calls))
    return {k: statistics.median(v) for k, v in times.items()}, times


def bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16}[t.dtype])


def kernel_ms(sets, outs, go, calls=5):
    """Mean device time per launch of k_lse_pairs / k_expand_logits for each dtype, from a profiler run of its own."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for dt in DTYPES:
            for i in range(calls):
                s = sets[i % len(sets)][dt]
                w._C.rnnt_logits_forward(*s, 0, 0.0, True, 0)
                o = outs[dt][i % len(sets)]
                w._C.rnnt_logits_backward(s[0], o[1], o[2], s[1], go, 0)
        torch.cuda.synchronize()
    res = {}
    for e in prof.key_averages():
        for kern in ("k_lse_pairs", "k_expand_logits"):
            if kern in e.key:
                dt = "bf16" if "bfloat16" in e.key else "f32"
                total = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                res[(dt, kern)] = total / max(e.count, 1) / 1e3
    return res


def run_shape(name, args, dev, peak):
    N, T, U, V = SHAPES[name]
    cells = N * T * U
    sets = make_sets(N, T, U, V, dev)
    R = len(sets)
    go = torch.ones(N, device=dev)
    fwd = {dt: (lambda i, dt=dt: w._C.rnnt_logits_forward(*sets[i][dt], 0, 0.0, True, 0)) for dt in DTYPES}
    outs = {dt: [fwd[dt](i) for i in range(R)] for dt in DTYPES}

    # the outputs at this size: bf16 against float32 on the same values
    o3, ob = outs["f32"][0], outs["bf16"][0]
    g3 = w._C.rnnt_logits_backward(sets[0]["f32"][0], o3[1], o3[2], sets[0]["f32"][1], go, 0)
    gb = w._C.rnnt_logits_backward(sets[0]["bf16"][0], ob[1], ob[2], sets[0]["bf16"][1], go, 0)
    check = {"costs_lse_pairs_bit_identical": all(torch.equal(bits(a), bits(b)) for a, b in zip(o3, ob)),
             "grad_equals_f32_grad_rounded": bool(torch.equal(bits(gb), bits(g3.to(torch.bfloat16))))}
    del g3, gb

    bwd = {dt: (lambda i, dt=dt: w._C.rnnt_logits_backward(sets[i][dt][0], outs[dt][i][1], outs[dt][i][2],
                                                             sets[i][dt][1], go, 0)) for dt in DTYPES}
    res = {"shape": {"N": N, "T": T, "U": U, "V": V}, "input_sets": R,
           "l2_protocol": "%d rotating input sets, %.0f MB of bf16 logits (float32: twice that)" % (R, R * 2 * cells * V / 1e6),
           "output_check": check}
    fwd_ms, fwd_blocks = alternate(fwd, R, args)
    bwd_ms, bwd_blocks = alternate(bwd, R, args)
    res["blocks_ms"] = {"fwd": fwd_blocks, "bwd": bwd_blocks}
    step_ms = None
    if name == "c5mbl":
        leaves = [{dt: sets[i][dt][0].detach().requires_grad_(True) for dt in DTYPES} for i in range(R)]

        def step(i, dt):
            x = leaves[i][dt]
            x.grad = None
            w.rnnt_loss_from_logits(x, *sets[i][dt][1:], reduction="sum").backward()
        step_ms, step_blocks = alternate({dt: (lambda i, dt=dt: step(i, dt)) for dt in DTYPES}, R, args)
        res["blocks_ms"]["step"] = step_blocks
        for lv in leaves:
            for x in lv.values():
                x.grad = None
    kms = kernel_ms(sets, outs, go)
    for dt, esz in (("f32", 4), ("bf16", 2)):
        r = {"fwd_op_ms": fwd_ms[dt], "bwd_op_ms": bwd_ms[dt], "fwd_plus_bwd_ms": fwd_ms[dt] + bwd_ms[dt]}
        if step_ms:
            r["step_ms"] = step_ms[dt]
        for kern, nbytes in (("k_lse_pairs", esz * cells * V), ("k_expand_logits", 2 * esz * cells * V)):
            km = kms.get((dt, kern))
            gbs = nbytes / (km * 1e-3) / 1e9 if km else None
            r[kern] = {"algorithmic_bytes": nbytes, "kernel_ms": km, "gbs": gbs, "share_of_peak": gbs / peak if gbs else None}
        res[dt] = r
    res["bf16_over_f32"] = {"fwd_plus_bwd": res["bf16"]["fwd_plus_bwd_ms"] / res["f32"]["fwd_plus_bwd_ms"],
                            "fwd": fwd_ms["bf16"] / fwd_ms["f32"], "bwd": bwd_ms["bf16"] / bwd_ms["f32"]}
    if step_ms:
        res["bf16_over_f32"]["step"] = step_ms["bf16"] / step_ms["f32"]
    del sets, outs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None, help="also write the result to this file")
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--shapes", default="c2l,c5mbl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("logits_time.py: no CUDA device")
    args.calls, args.warmup = max(args.calls, 20), max(args.warmup, 3)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    w.set_lse_mode("auto")
    peak, peak_src = bench.peaks()
    out = {"tool": "tools/logits_time.py", "card": card(), "peak_gbs": peak, "peak_source": peak_src,
           "lse_mode": "auto (exact)", "protocol": {"calls_per_block": args.calls, "warmup": args.warmup,
                                                   "rounds": args.rounds, "statistic": "median block, ms per call"},
           "shapes": {}}
    for name in args.shapes.split(","):
        out["shapes"][name] = run_shape(name, args, dev, peak)
    out["card_after"] = card()
    print("card: %s | peak %.0f GB/s (%s)" % ("; ".join(out["card"]["nvidia_smi"][1:]), peak, peak_src))
    print("%-6s %-5s %9s %9s %9s %9s | %-26s | %-26s" % ("shape", "dtype", "fwd ms", "bwd ms", "f+b ms", "step ms",
                                                         "lse pass GB/s (share)", "expand pass GB/s (share)"))
    for name, r in out["shapes"].items():
        for dt in DTYPES:
            d = r[dt]
            cell = lambda k: ("%7.0f (%.3f)" % (d[k]["gbs"], d[k]["share_of_peak"])) if d[k]["gbs"] else "not measured"
            print("%-6s %-5s %9.3f %9.3f %9.3f %9s | %-26s | %-26s" % (
                name, dt, d["fwd_op_ms"], d["bwd_op_ms"], d["fwd_plus_bwd_ms"],
                "%.3f" % d["step_ms"] if "step_ms" in d else "-", cell("k_lse_pairs"), cell("k_expand_logits")))
        print("%-6s bf16/f32: %s | outputs: %s" % (name, json.dumps({k: round(v, 3) for k, v in r["bf16_over_f32"].items()}),
                                                   json.dumps(r["output_check"])))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
