"""Where the captured training step's time goes, layer by layer: torch.profiler (CUDA activities) over graph replays
of the benchmark step (bench.py config 2: 4 encoder layers, batch 64 x 201 frames, bf16 autocast, FusedAdamW).

    python tools/prof_step.py [--out DIR] [--replays 3] [--batch 64] [--frames 201]

Writes <out>/trace_<i>.pt.trace.json (one replay each; default: prof_step under the system's temporary directory) and
prints one JSON summary.  Inside a graph replay the profiler reports every kernel on the stream the graph was launched
on, so the streams of a fork cannot be told apart by their ids; the split below is by kernel kind instead.  Per layer and direction (forward / backward):

  span_us         from the layer's first kernel start to the next layer's first kernel start
  idle_us         time in the span with no kernel running (dependent-launch gaps)
  side_only_us    time with kernels running but none of the data chain: only weight / bias / LayerNorm parameter sums
                  (gemm_tn, tn_reduce, colsum, reduce).  That is the time the data chain waits on a join, plus the
                  parameter sums it runs itself (the LayerNorm dgamma / dbeta reduce of the sequenced Functions)
  weight_us       pack_kernel + cast_transpose_kernel time in the span
  weight_exposed_us  the part of weight_us with no other kernel running
  scan_bwd_us     scan_bwd_lane_kernel's duration (backward only)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bimamba_b200 as bm  # noqa: E402

SIDE = ("gemm_tn_kernel", "tn_reduce_kernel", "colsum_kernel", "reduce_kernel")
WEIGHT = ("pack_kernel", "cast_transpose_kernel")


def kind(name):
    for k in SIDE + WEIGHT + ("ln_fwd_kernel", "ln_bwd_kernel", "scan_bwd_lane_kernel", "sumsq_kernel"):
        if k in name and not (k == "reduce_kernel" and "reduce_rows32" in name):
            return k
    return "chain"


def union(iv):
    out = []
    for a, b in sorted(iv):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def measure(iv, lo, hi):
    return sum(max(0.0, min(b, hi) - max(a, lo)) for a, b in iv)


def subtract(iv, cover):
    """Parts of the (unioned) intervals iv not covered by the (unioned) intervals cover."""
    out = []
    for a, b in iv:
        cur = a
        for c, d in cover:
            if d <= cur or c >= b:
                continue
            if c > cur:
                out.append([cur, c])
            cur = max(cur, d)
        if cur < b:
            out.append([cur, b])
    return out


def analyse(kernels):
    """kernels: [(name, start_us, end_us)] of one step, sorted by start."""
    t0, t1 = kernels[0][1], max(k[2] for k in kernels)
    ln_f = [k for k in kernels if kind(k[0]) == "ln_fwd_kernel"]
    ln_b = [k for k in kernels if kind(k[0]) == "ln_bwd_kernel"]
    loss = [k for k in kernels if kind(k[0]) == "sumsq_kernel"]
    nl = len(ln_f) // 2
    # forward of layer i: from its norm1 to the next layer's norm1 (the last: to the loss kernel); backward of layer i:
    # from the end of the next layer's norm1 backward (the last layer: the end of the loss kernel) to the end of its own
    # norm1 backward.  The optimizer step follows the last one.
    fb = [ln_f[2 * i][1] for i in range(nl)] + [loss[0][1]]
    bb = [loss[0][2]] + [ln_b[2 * j + 1][2] for j in range(nl)]
    segs = [(f"fwd{i}", fb[i], fb[i + 1]) for i in range(nl)]
    segs += [(f"bwd{nl - 1 - j}", bb[j], bb[j + 1]) for j in range(nl)]
    segs.append(("optim", bb[-1], t1))
    allu = union([[k[1], k[2]] for k in kernels])
    chain = union([[k[1], k[2]] for k in kernels if kind(k[0]) not in SIDE])
    side_only = subtract(union([[k[1], k[2]] for k in kernels if kind(k[0]) in SIDE]), chain)
    nonweight = union([[k[1], k[2]] for k in kernels if kind(k[0]) not in WEIGHT])
    wt = [[k[1], k[2]] for k in kernels if kind(k[0]) in WEIGHT]
    wt_exposed = subtract(union(wt), nonweight)
    rows = []
    for name, lo, hi in segs:
        inside = [k for k in kernels if lo <= k[1] < hi]
        r = {"segment": name, "span_us": hi - lo, "idle_us": (hi - lo) - measure(allu, lo, hi),
             "side_only_us": measure(side_only, lo, hi),
             "weight_us": sum(k[2] - k[1] for k in inside if kind(k[0]) in WEIGHT),
             "weight_exposed_us": measure(wt_exposed, lo, hi), "kernels": len(inside)}
        sb = [k[2] - k[1] for k in inside if kind(k[0]) == "scan_bwd_lane_kernel"]
        if sb:
            r["scan_bwd_us"] = sum(sb)
        rows.append(r)
    tot = {"step_us": t1 - t0, "kernels": len(kernels), "idle_us": (t1 - t0) - measure(allu, t0, t1),
           "side_only_us": measure(side_only, t0, t1), "weight_us": sum(b - a for a, b in wt),
           "weight_exposed_us": measure(wt_exposed, t0, t1)}
    return {"total": tot, "segments": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "prof_step"))
    ap.add_argument("--replays", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", type=int, default=201)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    torch.manual_seed(1234)
    model = bm.BiMambaBackend(144, 4, 16).cuda()
    with torch.no_grad():
        for layer in model.backbone_layers:
            layer.mamba.A_log.add_(0.1 * torch.randn_like(layer.mamba.A_log))
    params = list(model.backbone_layers.parameters())
    opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)
    x = torch.randn(a.batch, a.frames, 144, generator=torch.Generator().manual_seed(1234)).cuda()

    def zero_grad():
        for p in params:
            p.grad = None

    def fwd_loss(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model.forward_features(x)
        return bm.ops.mean_square_loss(out)

    runner = bm.GraphedTrainStep(fwd_loss, x, zero_grad, opt, warmup=3)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(10):
        runner.run()
    torch.cuda.synchronize()
    steps = []
    for i in range(a.replays):
        flush.zero_()                    # as bench.py: L2 flushed before each step
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            runner.run()
            torch.cuda.synchronize()
        path = os.path.join(a.out, f"trace_{i}.pt.trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
        ks = sorted((e["name"], float(e["ts"]), float(e["ts"]) + float(e["dur"]))
                    for e in ev if e.get("cat") == "kernel" and e.get("ph") == "X")
        ks = sorted(ks, key=lambda k: k[1])
        ks = [k for k in ks if "elementwise" not in k[0] and "fill" not in k[0].lower()] or ks
        steps.append(analyse(ks))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi, "batch": a.batch, "frames": a.frames, "steps": steps}))


if __name__ == "__main__":
    main()
