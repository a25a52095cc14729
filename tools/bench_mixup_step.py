"""Cost of Mixup (src/main.py:1038-1046, :1070-1073) in the training step at the benchmark's config 2: the 4-layer backend,
batch 64 x 201 frames, d_model 144, fp16 autocast, cross-entropy on the logits against labels, DeviceGradScaler, clip
at 3.0 and FusedEMA 0.999 over FusedAdamW.

  A  GraphedTrainStep(..., labels=): the captured recipe without Mixup
  B  GraphedTrainStep(..., labels=, mixup_alpha=1.0): the same with Mixup (host draw, one 8 + 4B-byte copy and one
     bimamba_mixup_frames launch per step)
  C  eager Phase6TrainStep with Mixup and the same tail

Every arm copies a fresh batch and its labels into the step.  Times are CUDA events around `steps` optimizer steps
after `warmup`, the arms alternated round by round in one process; the median over rounds is reported.  The kernel
alone is timed over `steps` launches on the (64, 201, 144) fp16 batch.  The GPU name and power limit are read in the
same run.

    python tools/bench_mixup_step.py [--steps 50] [--warmup 5] [--rounds 5] [--out profiles/mixup_step_b200.json]
"""
import argparse
import importlib
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F
from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bimamba_b200 as bm  # noqa: E402
from tools.bench_varlen import gpu_info  # noqa: E402

tr = importlib.import_module("robust-audio-deepfake-evolution_b200.training")
B, L, D, LAYERS = 64, 201, 144, 4
DECAY, MAX_NORM = 0.999, 3.0


def _ce(logits, feats, y):
    return F.cross_entropy(logits.float(), y)


def _setup(seed=1234):
    torch.manual_seed(seed)
    model = bm.BiMambaBackend(D, LAYERS, 16).cuda()
    params = [p for p in model.parameters() if p.requires_grad]
    opt = bm.FusedAdamW(params, lr=1e-3, weight_decay=1e-4)
    avg = AveragedModel(model, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    return model, params, opt, bm.FusedEMA(avg, model, DECAY), bm.DeviceGradScaler()


def _zero(params):
    def z():
        for p in params:
            p.grad = None
    return z


def build_arms(x, y):
    arms = {}
    for name, alpha in (("A", 0.0), ("B", 1.0)):
        model, params, opt, ema, scaler = _setup()

        def step_fn(xs, ys, lengths, mix, model=model):
            with torch.autocast("cuda", dtype=torch.float16):
                if mix is None:
                    feats, out = model(xs)
                    return _ce(out, feats, ys)
            mx, ya, yb, lam = bm.mixup_batch(xs, ys, lam=mix.mix, index=mix.perm)
            with torch.autocast("cuda", dtype=torch.float16):
                feats, out = model(mx)
                return bm.mixup_loss(_ce, out, feats, ya, yb, lam)
        g = bm.GraphedTrainStep(step_fn, x, _zero(params), opt, scaler=scaler, max_norm=MAX_NORM, ema=ema, labels=y,
                                mixup_alpha=alpha, generator=torch.Generator().manual_seed(1))
        arms[name] = lambda run=g.run: run(x, y=y)
    model, params, opt, ema, scaler = _setup()
    step = bm.Phase6TrainStep(model, opt, _ce, scaler=scaler, mixup_alpha=1.0, max_norm=MAX_NORM, ema_model=ema)
    gen = torch.Generator().manual_seed(1)
    arms["C"] = lambda: step([(x, y)], generator=gen)
    return arms


def _time(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def kernel_us(steps, warmup):
    x = torch.randn(B, L, D, device="cuda").half()
    perm = torch.randperm(B, device="cuda").to(torch.int32)
    mix = tr.mix_record(0.3, "cuda")
    out = torch.empty_like(x)
    return 1e3 * _time(lambda: bm.ops.mixup_frames(x, perm, mix, None, out), steps, warmup)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mixup_step.py measures on a GPU; none is visible")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, L, D, generator=g).cuda()
    y = torch.randint(0, 2, (B,), generator=g).cuda()
    arms = build_arms(x, y)
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            times[k].append(_time(fn, args.steps, args.warmup))
    res = {"gpu": gpu_info(), "shape": {"batch": B, "frames": L, "d_model": D, "layers": LAYERS, "autocast": "float16"},
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
           "arms": {k: {"ms_per_step_median": round(statistics.median(v), 4), "ms_per_step_rounds": [round(t, 4) for t in v]}
                    for k, v in times.items()},
           "mixup_kernel_us_fp16_64x201x144": round(kernel_us(200, 20), 2)}
    a, b = res["arms"]["A"]["ms_per_step_median"], res["arms"]["B"]["ms_per_step_median"]
    res["mixup_cost_captured_ms"] = round(b - a, 4)
    res["mixup_cost_captured_pct"] = round(100 * (b - a) / a, 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
