"""Variable-length training throughput: the benchmark's 4-layer backend (d_model 144, bf16 autocast, FusedAdamW), a batch
of 64 utterances with seeded lengths 50..201 padded to 201 frames, one training step (cross-entropy on the logits of
the training head, backward, AdamW) three ways

  padded   net(x, lengths, mask_padding=True) captured once in a GraphedTrainStep(..., lengths=...), replayed
  grouped  the exact alternative without lengths: per distinct length one eager forward + backward on its utterances
           (gradients accumulate), then one AdamW step (every shape would need its own captured graph)
  ceiling  the same padded shape at fixed length, every frame valid, captured in a GraphedTrainStep

reported as VALID frames per second (sum of the lengths, or 64 x 201 for the ceiling, over the device time of one step;
CUDA events around `reps` steps after `warmup` steps).  Dropout is left as the model has it (0.1, training mode).  The
GPU name and power limit are read in the same run.  Needs a CUDA device; prints one JSON line per mode and optionally
writes them all to --out.

    python tools/bench_varlen_train.py [--reps 20] [--warmup 3] [--out profiles/varlen_train_b200.json]
"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bimamba_b200 as bm  # noqa: E402
from tools.bench_varlen import device_ms, gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--min-frames", type=int, default=50)
    ap.add_argument("--max-frames", type=int, default=201)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_varlen_train.py needs a CUDA device")
    gen = torch.Generator().manual_seed(args.seed)
    n, T = args.batch, args.max_frames
    lengths = torch.randint(args.min_frames, T + 1, (n,), generator=gen)
    lengths[0] = T                                          # the padded shape is the longest utterance
    x = torch.randn(n, T, 144, generator=gen).cuda()
    labels = torch.randint(0, 2, (n,), generator=gen).cuda()
    torch.manual_seed(args.seed)
    net = bm.BiMambaBackend(144, 4, 16).cuda().train()
    params = list(net.parameters())
    opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)
    valid = int(lengths.sum())
    groups = [(int(v), torch.nonzero(lengths == v).flatten().cuda()) for v in torch.unique(lengths)]

    def zero_grad():
        for p in params:
            p.grad = None

    def step_len(xx, ll):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            _, logits = net(xx, ll, mask_padding=True)
        return F.cross_entropy(logits.float(), labels)

    def step_fixed(xx):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            _, logits = net(xx)
        return F.cross_entropy(logits.float(), labels)

    padded = bm.GraphedTrainStep(step_len, x, zero_grad, opt, lengths=lengths)
    ceiling = bm.GraphedTrainStep(step_fixed, x, zero_grad, opt)

    def grouped():
        zero_grad()
        for v, idx in groups:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                _, logits = net(x[idx, :v])
            (F.cross_entropy(logits.float(), labels[idx], reduction="sum") / n).backward()
        opt.step()

    info = gpu_info()
    ms = {"padded": device_ms(lambda: padded.run(x, lengths), args.reps, args.warmup),
          "grouped": device_ms(grouped, args.reps, args.warmup),
          "ceiling": device_ms(lambda: ceiling.run(x), args.reps, args.warmup)}
    rows = []
    for mode, t in ms.items():
        frames = n * T if mode == "ceiling" else valid
        row = {"metric": "valid_frames_per_sec", "dtype": "bf16", "mode": mode, "value": frames / (t * 1e-3),
               "ms_per_step": t, "utterances": n, "valid_frames": frames, "padded_frames": n * T,
               "distinct_lengths": len(groups), "lengths": f"seeded uniform {args.min_frames}..{T} (seed {args.seed})",
               "gpu": info}
        print(json.dumps(row), flush=True)
        rows.append(row)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
