"""Cost of the fp16 recipe's optimizer tail (GradScaler unscale -> clip_grad_norm_(3.0) -> skip-on-inf step -> scale update
-> EMA 0.999, src/main.py:1100-1117) at the benchmark's shape: the 4-layer backend, batch 64 x 201 frames, d_model 144,
fp16 autocast, mean-square loss, optimizer over the backbone parameters.

  A  GraphedTrainStep with FusedAdamW, no scaler / clip / EMA (today's capturable step, in fp16)
  B  GraphedTrainStep(..., scaler=DeviceGradScaler, max_norm=3.0, ema=FusedEMA): the captured recipe
  C  eager: torch GradScaler, unscale_, clip_grad_norm_, scaler.step(FusedAdamW) (its host-read branch), update,
     AveragedModel.update_parameters
  D  B with accumulation_steps=4 (FlatGradBucket(accumulate=True)), per optimizer step and per micro-batch
  E  torch.optim.AdamW(fused=True, capturable=True) with GradScaler, clip_grad_norm_ and AveragedModel, captured in one
     torch.cuda.CUDAGraph (tried in a child process; the error is recorded when it does not capture)

Times are CUDA events around `steps` optimizer steps after `warmup`, the arms alternated round by round in one process
(the L2 cache is not flushed; the step's activations exceed it).  A separate torch.profiler pass counts the kernels of
one eager optimizer tail per arm.  The GPU name and power limit are read in the same run.

    python tools/bench_amp_step.py [--steps 50] [--warmup 5] [--rounds 5] [--out profiles/amp_step_b200.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bimamba_b200 as bm  # noqa: E402
from tools.bench_varlen import gpu_info  # noqa: E402

B, L, D, LAYERS = 64, 201, 144, 4
DECAY, MAX_NORM = 0.999, 3.0


def _setup(seed=1234):
    torch.manual_seed(seed)
    model = bm.BiMambaBackend(D, LAYERS, 16).cuda()
    params = list(model.backbone_layers.parameters())
    avg = AveragedModel(model, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    return model, params, avg


def _loss_fn(model):
    def f(x):
        with torch.autocast("cuda", dtype=torch.float16):
            out = model.forward_features(x)
        return bm.ops.mean_square_loss(out)
    return f


def _zero(params):
    def z():
        for p in params:
            p.grad = None
    return z


def build_arms(x):
    arms, tails = {}, {}
    # A
    model, params, _ = _setup()
    opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)
    g = bm.GraphedTrainStep(_loss_fn(model), x, _zero(params), opt)
    arms["A"] = (g.run, 1)
    tails["A"] = lambda opt=opt: opt.step()
    # B
    model, params, avg = _setup()
    opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)
    scaler, ema = bm.DeviceGradScaler(), bm.FusedEMA(avg, model, DECAY)
    g = bm.GraphedTrainStep(_loss_fn(model), x, _zero(params), opt, scaler=scaler, max_norm=MAX_NORM, ema=ema)
    arms["B"] = (g.run, 1)
    tails["B"] = lambda opt=opt, s=scaler, e=ema: opt.step(scaler=s, max_norm=MAX_NORM, ema=e)
    # C
    model, params, avg = _setup()
    opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)
    tscaler = torch.amp.GradScaler("cuda")
    fwd = _loss_fn(model)

    def tail_c(opt=opt, s=tscaler, avg=avg, model=model, params=params):
        s.unscale_(opt)
        torch.nn.utils.clip_grad_norm_([p for p in params if p.grad is not None], MAX_NORM)
        s.step(opt)
        s.update()
        avg.update_parameters(model)

    def step_c(fwd=fwd, s=tscaler, params=params):
        _zero(params)()
        s.scale(fwd(x)).backward()
        tail_c()
    arms["C"] = (step_c, 1)
    tails["C"] = tail_c
    # D
    model, params, avg = _setup()
    opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)
    scaler, ema = bm.DeviceGradScaler(), bm.FusedEMA(avg, model, DECAY)
    bucket = bm.FlatGradBucket(params, accumulate=True)
    g = bm.GraphedTrainStep(_loss_fn(model), x, bucket.zero, opt, scaler=scaler, max_norm=MAX_NORM, ema=ema,
                            accumulation_steps=4)

    def step_d(run=g.run):
        for _ in range(4):
            run()
    arms["D"] = (step_d, 4)
    tails["D"] = lambda opt=opt, s=scaler, e=ema, b=bucket: (opt.step(scaler=s, max_norm=MAX_NORM, ema=e), b.zero())
    return arms, tails


def arm_e(x, steps, warmup):
    """The framework's own capturable arrangement; raises if it does not capture."""
    model, params, avg = _setup()
    opt = torch.optim.AdamW(params, lr=1e-5, weight_decay=1e-4, fused=True, capturable=True)
    s = torch.amp.GradScaler("cuda")
    fwd = _loss_fn(model)

    def step():
        opt.zero_grad(set_to_none=False)
        s.scale(fwd(x)).backward()
        s.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(params, MAX_NORM)
        s.step(opt)
        s.update()
        avg.update_parameters(model)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    return _time(graph.replay, steps, warmup)


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


def tail_kernels(tails, x):
    """Kernels of one eager optimizer tail per arm (gradients from one eager backward), from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    counts = {}
    for name, tail in tails.items():
        opt = tail.__defaults__[0]
        params = [p for g in opt.param_groups for p in g["params"]]
        for p in params:                                    # any gradient: the tail's kernels do not depend on it
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        tail()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            tail()
            torch.cuda.synchronize()
        ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        kernels = [e.name for e in ev if "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]
        counts[name] = {"kernels": len(kernels), "copies_and_sets": len(ev) - len(kernels),
                        "names": sorted(set(kernels))}
    return counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    ap.add_argument("--arm-e-only", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_amp_step.py needs a CUDA device")
    x = torch.randn(B, L, D, generator=torch.Generator().manual_seed(0)).cuda()
    if args.arm_e_only:
        print(json.dumps({"ms": arm_e(x, args.steps, args.warmup)}))
        return
    info = gpu_info()
    arms, tails = build_arms(x)
    per = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, (fn, _) in arms.items():
            per[k].append(_time(fn, args.steps, args.warmup))
    res = {"gpu": info, "shape": {"batch": B, "frames": L, "d_model": D, "layers": LAYERS, "autocast": "float16"},
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "arms": {}}
    for k, (_, micro) in arms.items():
        med = statistics.median(per[k])
        row = {"ms_per_optimizer_step": round(med, 4), "rounds_ms": [round(v, 4) for v in per[k]]}
        if micro > 1:
            row["ms_per_micro_batch"] = round(med / micro, 4)
        res["arms"][k] = row
    a, b = res["arms"]["A"]["ms_per_optimizer_step"], res["arms"]["B"]["ms_per_optimizer_step"]
    res["B_minus_A_ms"] = round(b - a, 4)
    res["B_minus_A_pct_of_A"] = round(100 * (b - a) / a, 2)
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--arm-e-only", "--steps", str(args.steps),
                            "--warmup", str(args.warmup)], capture_output=True, text=True, timeout=1200)
    if child.returncode == 0:
        res["arms"]["E"] = {"ms_per_optimizer_step": round(json.loads(child.stdout.strip().splitlines()[-1])["ms"], 4)}
    else:
        err = [ln for ln in child.stderr.strip().splitlines() if ln.strip()]
        res["arms"]["E"] = {"error": err[-1] if err else f"exit code {child.returncode}"}
    res["tail_kernels"] = tail_kernels(tails, x)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
