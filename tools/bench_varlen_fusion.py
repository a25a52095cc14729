"""Variable-length model-tail throughput: DualStreamFusion -> the 4-layer Bi-Mamba backend -> scoring head on 256 clips
with seeded sample counts of 1-10 s (10 ms steps), mapped to per-utterance frame counts by the front ends' formulas
(WavLM (S - 400) // 320 + 1, at most 499; SincNet (S - 128) // 3 then // 3 six times, at most 73).  Random streams of
1024 and 64 channels stand in for the front ends.  Scored three ways, in bf16 (autocast) and fp32:

  padded   one (256, 499) / (256, 73) pair of streams with both length vectors through one captured CUDA graph
           (torch.cuda.graph over static streams and length buffers)
  grouped  the exact alternative without lengths: one eager pass per distinct (n1, n2) pair
  ceiling  the fixed-length 256 x 499 / 73 streams through one captured graph (every frame valid)

and one training row (bf16): the mask_padding=True forward + backward of the tail on the padded streams against the
fixed-length forward + backward at the same padded shape (eager, parameter gradients included, no optimizer).

Reported as VALID frames per second (the sum of the WavLM lengths, or 256 x 499 for the fixed-length rows, over the
device time of one pass; CUDA events around `reps` passes after `warmup` passes, no L2 flush: one pass's activations
are several times the 126 MB L2).  The GPU name and power limit are read in the same run.  Needs a CUDA device; prints
one JSON line per row and optionally writes them all to --out.

    python tools/bench_varlen_fusion.py [--reps 10] [--warmup 2] [--out profiles/varlen_fusion_b200.json]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bimamba_b200 as bm  # noqa: E402
from tools.bench_varlen import device_ms, gpu_info  # noqa: E402


def wavlm_frames(S):
    return (S - 400) // 320 + 1


def sinc_frames(S):
    n = (S - 128) // 3
    for _ in range(6):
        n //= 3
    return n


def captured(fn):
    """fn() captured once in a CUDA graph (after one warm-up pass on a side stream); returns replay, outputs."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph.replay, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--min-s", type=float, default=1.0)
    ap.add_argument("--max-s", type=float, default=10.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_varlen_fusion.py needs a CUDA device")
    gen = torch.Generator().manual_seed(args.seed)
    n = args.n
    S = torch.randint(int(args.min_s * 100), int(args.max_s * 100) + 1, (n,), generator=gen) * 160
    S[0] = int(args.max_s * 16000)                         # the padded shape is the longest clip
    l1 = [wavlm_frames(int(s)) for s in S]
    l2 = [sinc_frames(int(s)) for s in S]
    T1, T2 = max(l1), max(l2)
    fw = torch.randn(n, T1, 1024, generator=gen).cuda()
    fs = torch.randn(n, T2, 64, generator=gen).cuda()
    sl1 = torch.tensor(l1, dtype=torch.int32, device="cuda")
    sl2 = torch.tensor(l2, dtype=torch.int32, device="cuda")
    torch.manual_seed(args.seed)
    fus = bm.DualStreamFusion(1024, 64, 144).cuda().eval()
    net = bm.BiMambaBackend(144, 4, 16).cuda().eval()
    valid = sum(l1)
    pairs = sorted(set(zip(l1, l2)))
    groups = [(a, b, torch.tensor([i for i in range(n) if (l1[i], l2[i]) == (a, b)], device="cuda")) for a, b in pairs]
    info = gpu_info()
    base = {"utterances": n, "padded_frames": n * T1, "padded_shape": [T1, T2], "distinct_pairs": len(pairs),
            "clips": f"seeded uniform {args.min_s}..{args.max_s} s in 10 ms steps (seed {args.seed})", "gpu": info}
    rows = []

    def emit(row):
        row = {**row, **base}
        print(json.dumps(row), flush=True)
        rows.append(row)

    for name, dtype in (("bf16", torch.bfloat16), ("fp32", torch.float32)):
        ac = lambda: torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32, cache_enabled=False)  # noqa: E731
        with torch.no_grad(), ac():
            run_pad, out_pad = captured(lambda: net(fus(fw, fs, sl1, sl2), sl1))
            run_fix, _ = captured(lambda: net(fus(fw, fs)))

            def grouped():
                return [(idx, net(fus(fw[idx, :a], fs[idx, :b]))[1]) for a, b, idx in groups]

            ms = {"padded": device_ms(run_pad, args.reps, args.warmup),
                  "grouped": device_ms(grouped, args.reps, args.warmup),
                  "ceiling": device_ms(run_fix, args.reps, args.warmup)}
            run_pad()
            s_pad = out_pad[1].float().clone()
            s_grp = torch.empty_like(s_pad)
            for idx, lg in grouped():
                s_grp[idx] = lg.float()
        diff = float((s_pad - s_grp).abs().max())
        for mode, t in ms.items():
            frames = n * T1 if mode == "ceiling" else valid
            emit({"metric": "valid_frames_per_sec", "dtype": name, "mode": mode, "value": frames / (t * 1e-3),
                  "ms_per_pass": t, "valid_frames": frames, "padded_vs_grouped_max_abs_logit_diff": diff})
        del run_pad, run_fix, out_pad

    fus.train()
    net.train()
    params = list(fus.parameters()) + list(net.parameters())
    fwr, fsr = fw.clone().requires_grad_(True), fs.clone().requires_grad_(True)

    def train(lengths):
        for p in params:
            p.grad = None
        fwr.grad = fsr.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if lengths:
                feats, logits = net(fus(fwr, fsr, sl1, sl2, mask_padding=True), sl1, mask_padding=True)
            else:
                feats, logits = net(fus(fwr, fsr))
        (logits.float().sum() + feats.float().sum()).backward()

    for mode, lengths, frames in (("padded_mask_padding", True, valid), ("fixed_length", False, n * T1)):
        t = device_ms(lambda: train(lengths), args.reps, args.warmup)
        emit({"metric": "valid_frames_per_sec", "dtype": "bf16", "mode": "train_fwd_bwd_" + mode,
              "value": frames / (t * 1e-3), "ms_per_pass": t, "valid_frames": frames})
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
