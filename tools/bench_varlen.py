"""Variable-length scoring throughput: 256 utterances with seeded lengths spread over 50..499 frames, scored three ways

  padded   one (256, 499) batch with per-utterance lengths through one captured GraphedForward (conv, scan and head skip
           the padded frames; the products, LayerNorms and feed-forward still run on every padded row)
  grouped  the exact alternative without lengths: one eager forward per distinct length (every shape would need its
           own captured graph)
  ceiling  the fixed-length (256, 499) batch through a captured GraphedForward (every frame valid)

in bf16 (autocast) and fp32, reported as VALID frames per second (sum of the lengths, or 256 x 499 for the ceiling,
over the device time of one scoring pass; CUDA events around `reps` passes after `warmup` passes, no L2 flush: the
activations of one pass are several times the 126 MB L2).  The GPU name and power limit are read in the same run.
Needs a CUDA device; prints one JSON line per (dtype, mode) and optionally writes them all to --out.

    python tools/bench_varlen.py [--reps 20] [--warmup 3] [--out profiles/varlen_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bimamba_b200 as bm  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                                       "-i", str(torch.cuda.current_device())], text=True, timeout=30)
        pl, sm = [v.strip() for v in out.splitlines()[0].split(",")]
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(sm)
    except (OSError, subprocess.SubprocessError, ValueError, IndexError) as e:
        info["power_limit_error"] = str(e)
    return info


def device_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--min-frames", type=int, default=50)
    ap.add_argument("--max-frames", type=int, default=499)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_varlen.py needs a CUDA device")
    gen = torch.Generator().manual_seed(args.seed)
    n, T = args.n, args.max_frames
    lengths = torch.randint(args.min_frames, T + 1, (n,), generator=gen)
    lengths[0] = T                                          # the padded shape is the longest utterance
    x = torch.randn(n, T, 144, generator=gen).cuda()
    torch.manual_seed(args.seed)
    net = bm.BiMambaBackend(144, 4, 16).cuda().eval()
    valid = int(lengths.sum())
    groups = [(int(v), torch.nonzero(lengths == v).flatten().cuda()) for v in torch.unique(lengths)]
    info = gpu_info()
    rows = []
    for name, dtype in (("bf16", torch.bfloat16), ("fp32", torch.float32)):
        ac = lambda: torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32)  # noqa: E731

        def score_len(xx, ll):
            with ac():
                return net(xx, ll)

        def score_fixed(xx):
            with ac():
                return net(xx)

        padded = bm.GraphedForward(score_len, x, lengths=lengths)
        ceiling = bm.GraphedForward(score_fixed, x)

        def grouped():
            with torch.no_grad(), ac():
                return [(idx, net(x[idx, :v])[1]) for v, idx in groups]

        ms = {"padded": device_ms(lambda: padded.run(x, lengths), args.reps, args.warmup),
              "grouped": device_ms(grouped, args.reps, args.warmup),
              "ceiling": device_ms(lambda: ceiling.run(x), args.reps, args.warmup)}
        s_pad = padded.run(x, lengths)[1].float().clone()
        s_grp = torch.empty_like(s_pad)
        for idx, lg in grouped():
            s_grp[idx] = lg.float()
        diff = float((s_pad - s_grp).abs().max())
        for mode, t in ms.items():
            frames = n * T if mode == "ceiling" else valid
            row = {"metric": "valid_frames_per_sec", "dtype": name, "mode": mode, "value": frames / (t * 1e-3),
                   "ms_per_pass": t, "utterances": n, "valid_frames": frames, "padded_frames": n * T,
                   "distinct_lengths": len(groups), "lengths": f"seeded uniform {args.min_frames}..{T} (seed {args.seed})",
                   "padded_vs_grouped_max_abs_logit_diff": diff, "gpu": info}
            print(json.dumps(row), flush=True)
            rows.append(row)
        del padded, ceiling
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
