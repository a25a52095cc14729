#!/usr/bin/env python
"""Benchmark of the Bi-Mamba backend hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload at N = 1 is BASELINE.json configs[1]: the 4-layer Bi-Mamba backend (4 x
PN_BiMambas_Encoder, d_model 144, d_state 16) fwd + bwd (+ AdamW step), 201 frames, batch 64,
bf16 activations / fp32 state / fp32 master weights, synthetic WavLM-shaped features.  For N > 1
(launched with torchrun, one rank per GPU) every rank runs that same per-GPU batch (weak scaling)
and gradients are all-reduced over NCCL once per step.

One JSON line is printed by rank 0.  `value` is device-resident throughput (inputs already in HBM,
CUDA-graph replay, CUDA events, L2 flushed between steps); `e2e` is the same metric through the
public API with the step's input coming from pinned HOST memory and the loss read back to the host
every step.  `--impl reference` times the CPU oracle port of the reference's own path
(oracle/bimamba_oracle.py; the reference is a Python package whose /root/reference tree does not
exist on the GPU box) on all host threads.

`--dump-outputs DIR` writes what the last device-timed training step handed back to its caller, as
DIR/<name>.npy: `loss` (float64) and, for every backbone parameter, `param.<name>` (after that step's
AdamW update) and `grad.<name>` (the gradient it applied), float32, about 10 MB in all.  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark may run from a read-only tree; it writes nothing into it

import torch  # noqa: E402

D_MODEL, D_STATE, N_LAYERS = 144, 16, 4
D_INNER = 2 * D_MODEL
METRIC = "bimamba_backend_fwd_bwd_frames_per_sec"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="per-GPU batch (config 2: 64)")
    ap.add_argument("--frames", type=int, default=201)
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-native-block", action="store_true",
                    help="eager mode only: keep the block on the Python-sequenced autograd Function instead of the one-call "
                         "native entry points (A/B of the two eager arrangements; a captured step always replays the former)")
    ap.add_argument("--torch-adamw", action="store_true", help="torch.optim.AdamW(fused=True) instead of FusedAdamW")
    ap.add_argument("--no-sweep", action="store_true", help="skip the config-5 scan sweep points")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tune", default="", help="knob=value,... forwarded to bimamba_set_tuning (A/B measurements)")
    ap.add_argument("--comm", default="overlap", choices=["overlap", "graph", "eager"],
                    help="N > 1: gradient all-reduce per encoder layer inside the step graph, overlapping the remaining "
                         "backward (default); one all-reduce inside the graph; or launched after the graph (round 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the loss, parameters and gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def workload_config(args, world):
    return {
        "workload": f"Phase-6 Bi-Mamba backend ({N_LAYERS} x PN_BiMambas_Encoder, d_model {D_MODEL}, d_state {D_STATE}) "
                    f"fwd+bwd+AdamW training step, {args.frames} frames, batch {args.batch} per GPU "
                    f"(BASELINE.json configs[1])",
        "per_gpu_batch": args.batch, "global_batch": args.batch * world, "frames": args.frames,
        "parallelism": f"dp{world}" if world > 1 else "single",
    }


# --------------------------------------------------------------------------------------
# CPU oracle legs
# --------------------------------------------------------------------------------------
def oracle_step_fn(batch, frames):
    """fwd+bwd of the 4-layer backend with the oracle port (fp32, all host threads)."""
    from oracle import bimamba_oracle as orc
    torch.manual_seed(1234)                      # reference default seed, src/main.py:1145
    layers = []
    for i in range(N_LAYERS):
        p = orc.init_encoder_params(D_MODEL, D_STATE, seed=i, dtype=torch.float32)
        layers.append({k: v.requires_grad_(True) for k, v in p.items()})
    x = torch.randn(batch, frames, D_MODEL)

    def step():
        h = x
        for p in layers:
            h = orc.pn_bimamba_encoder_ref(p, h)
        loss = h.square().mean()
        loss.backward()
        for p in layers:
            for v in p.values():
                v.grad = None
        return float(loss.detach())
    return step


def run_cpu_baseline(frames, sample_batch=64, reps=2):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = oracle_step_fn(sample_batch, frames)
    step()                                        # warm-up
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        step()
        best = min(best, time.perf_counter() - t0)
    return {
        "value": sample_batch * frames / best, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
        "sample": f"oracle/bimamba_oracle.py (port of mamba_block.py + PN_BiMambas_Encoder), fp32, batch {sample_batch} "
                  f"(the workload's own batch), {frames} frames, {N_LAYERS} layers, fwd+bwd (no optimizer step), best of {reps} "
                  f"after 1 warm-up ({best:.2f} s per step)",
    }


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample_batch = args.batch                     # the benchmarked batch itself (config 2: 64), not a sub-sample
    step = oracle_step_fn(sample_batch, args.frames)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    value = sample_batch * args.frames * steps / dt
    sample = (f"oracle port of the reference's CPU path (the reference is Python and /root/reference is absent on the GPU "
              f"box), fp32, batch {sample_batch} (the workload's batch), {args.frames} frames, fwd+bwd, {steps} timed steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------
# GPU legs
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def ready(self, timeout=5.0):
        """Block until nvidia-smi has delivered its first sample (its start-up takes longer than a short timed run)."""
        t_end = time.perf_counter() + timeout
        while self.proc is not None and not self.lines and time.perf_counter() < t_end:
            time.sleep(0.01)

    def stop(self, windows):
        """Median SM clock / throttle reasons over the samples that fall inside the timed windows [(t0, t1), ...]."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        inside = [ln for t, ln in self.lines if any(a <= t <= b for a, b in windows)]
        sm, mx, reasons = [], [], set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class EventTimer:
    """kernel_timer hook: CUDA events on the launching stream around each enqueue of one kernel."""

    def __init__(self):
        self.pairs = {}

    def __call__(self, name):
        timer = self

        class _Ctx:
            def __enter__(self_inner):
                self_inner.s = torch.cuda.Event(enable_timing=True)
                self_inner.e = torch.cuda.Event(enable_timing=True)
                self_inner.s.record()
                return self_inner

            def __exit__(self_inner, *a):
                self_inner.e.record()
                timer.pairs.setdefault(name, []).append((self_inner.s, self_inner.e))
                return False
        return _Ctx()

    def summary(self):
        torch.cuda.synchronize()
        return {k: [s.elapsed_time(e) for s, e in v] for k, v in self.pairs.items()}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_step_outputs(directory, model, loss):
    """What a caller of the training step holds once it returns: the loss, every backbone parameter after the AdamW
    update and the gradient that update applied."""
    import numpy as np
    out = {"loss": loss.detach().double().cpu().numpy()}
    for name, p in model.backbone_layers.named_parameters(prefix="backbone_layers"):
        out["param." + name] = p.detach().float().cpu().numpy()
        out["grad." + name] = p.grad.detach().float().cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def scan_bytes(frames, ndir, esize, backward):
    """SURVEY 8(d): fwd (4 D + 2 N) s, bwd (7 D + 4 N) s bytes per frame per direction."""
    per = (7 * D_INNER + 4 * D_STATE) if backward else (4 * D_INNER + 2 * D_STATE)
    return frames * ndir * per * esize


def scan_sweep(bm, peak):
    """Config 5 (BASELINE.json configs[4]): the single-direction selective_scan op on 524 288 frames, D = 288, N = 16,
    every L in 64..8192, bf16 and fp32 I/O.  Three rows per point: `scan_fwd_infer` (torch.no_grad: nothing saved for a
    backward - the bytes the op-boundary figure describes), `scan_fwd` (training forward: also writes the fp32
    checkpoints every 8 steps and ypre) and `scan_bwd`; all against SURVEY 8(d)'s algorithmic bytes."""
    out = []
    g = torch.Generator(device="cuda").manual_seed(0)
    for dtype, name in ((torch.bfloat16, "bf16"), (torch.float32, "f32")):
        for L in (64, 128, 256, 512, 1024, 2048, 4096, 8192):
            Bsz = (1 << 19) // L
            mk = lambda *sh: torch.randn(*sh, device="cuda", generator=g)
            u = mk(Bsz, D_INNER, L).to(dtype).requires_grad_(True)
            delta = (0.5 * mk(Bsz, D_INNER, L)).to(dtype).requires_grad_(True)
            z = mk(Bsz, D_INNER, L).to(dtype).requires_grad_(True)
            Bm = mk(Bsz, D_STATE, L).to(dtype).requires_grad_(True)
            Cm = mk(Bsz, D_STATE, L).to(dtype).requires_grad_(True)
            A = (-torch.exp(torch.log(torch.arange(1, D_STATE + 1, device="cuda", dtype=torch.float32)).repeat(D_INNER, 1)
                            + 0.1 * mk(D_INNER, D_STATE))).requires_grad_(True)
            Dp = (1 + 0.1 * mk(D_INNER)).requires_grad_(True)
            dt0 = torch.exp(torch.rand(D_INNER, device="cuda", generator=g) * (math.log(0.1) - math.log(1e-3)) + math.log(1e-3))
            bias = (dt0 + torch.log(-torch.expm1(-dt0))).requires_grad_(True)     # mamba dt-bias init range
            cot = mk(Bsz, D_INNER, L).to(dtype)
            timer = EventTimer()
            bm._lib.kernel_timer = timer
            for it in range(5):
                o = bm.selective_scan_fn(u, delta, A, Bm, Cm, Dp, z, bias, True)
                o.backward(cot)
                for t in (u, delta, z, Bm, Cm, A, Dp, bias):
                    t.grad = None
            times = timer.summary()
            timer = EventTimer()
            bm._lib.kernel_timer = timer
            with torch.no_grad():
                for it in range(5):
                    o = bm.selective_scan_fn(u, delta, A, Bm, Cm, Dp, z, bias, True)
            bm._lib.kernel_timer = None
            times["scan_fwd_infer"] = timer.summary()["scan_fwd"]
            es = 4 if dtype == torch.float32 else 2
            nseg = bm._lib.scan_split_plan(Bsz, 1, L, D_INNER, bm._lib.F32 if dtype == torch.float32 else bm._lib.BF16)[0]
            for kname, bwd in (("scan_fwd_infer", False), ("scan_fwd", False), ("scan_bwd", True)):
                ms = statistics.median(times[kname][2:])
                gbs = scan_bytes(Bsz * L, 1, es, bwd) / (ms * 1e-3) / 1e9
                row = {"kernel": kname, "io": name, "L": L, "batch": Bsz, "ms": round(ms, 4),
                       "achieved_gbs": round(gbs, 1), "frac": round(gbs / peak, 4)}
                if nseg > 1 and not bwd:
                    row["time_segments"] = nseg      # time-parallel forward: carry pass + output pass (two launches)
                out.append(row)
            del u, delta, z, Bm, Cm, cot, o
            torch.cuda.empty_cache()
    return out


def gemm_roofline(bm, B, L, flush):
    """The in_proj GEMM of the block at the benchmark shape (M = B*L, K = 144, N = 576, bf16, fp32 accumulate) timed
    alone (CUDA events around each launch, L2 flushed before each): flops / t against the measured dense bf16 peak and
    bytes / t against the measured HBM peak (SURVEY 8d)."""
    M, K, N = B * L, D_MODEL, 2 * D_INNER
    a = torch.randn(M, K, device="cuda").to(torch.bfloat16)
    w = torch.randn(N, K, device="cuda").to(torch.bfloat16)
    ts = []
    for it in range(12):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        bm.ops.gemm_nt(a, w)
        e.record()
        ts.append((s, e))
    torch.cuda.synchronize()
    ms = statistics.median([s.elapsed_time(e) for s, e in ts[2:]])
    flops = 2.0 * M * K * N
    nbytes = 2.0 * (M * K + N * K + M * N)
    tf_peak, tf_src = 1642.8, "fallback"
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            tf_peak, tf_src = json.load(f).get("bf16_tflops", tf_peak), "measured (MEASURED_PEAKS.json bf16_tflops, burst: kernel timed alone)"
    hbm_peak, _ = load_peaks()
    return {"kernel": "gemm_nt_kernel<bf16> in_proj (M %d, K %d, N %d), tcgen05 + TMEM + TMA" % (M, K, N), "bound": "tensor",
            "achieved": flops / (ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / tf_peak,
            "peak_source": tf_src, "avg_launch_ms": ms, "flops_per_launch": flops, "algorithmic_bytes_per_launch": nbytes,
            "hbm_achieved_gbs": nbytes / (ms * 1e-3) / 1e9, "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / hbm_peak,
            "note": "arithmetic intensity %.0f flop/B is below the B200 ridge (~250): stand-alone the product is bound by memory "
                    "and launch latency, not by the tensor pipe (DESIGN.md 4.5)" % (flops / nbytes)}


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback for the Bi-Mamba path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import bimamba_b200 as bm
    for kv in filter(None, args.tune.split(",")):
        k, v = kv.split("=")
        bm._lib.load().bimamba_set_tuning(int(k), int(v))

    torch.manual_seed(1234)
    model = bm.BiMambaBackend(D_MODEL, N_LAYERS, D_STATE).cuda()
    with torch.no_grad():                         # trained-like A (no power structure), SURVEY 8d
        for layer in model.backbone_layers:
            layer.mamba.A_log.add_(0.1 * torch.randn_like(layer.mamba.A_log))
    params = list(model.backbone_layers.parameters())
    # BENCH_FORCE_BUCKET=1 (diagnostic): the multi-GPU gradient-bucket path on ONE GPU - hooks, per-layer packs, the same
    # graph structure, collectives degenerate to nothing - to separate the bucket's cost from the collectives'
    bucketed = world > 1 or os.environ.get("BENCH_FORCE_BUCKET") == "1"
    if bucketed:
        # one flat buffer; backward assigns the gradients, multi-tensor copies pack them, NCCL averages them
        bucket = bm.FlatGradBucket(params, accumulate=False)
        zero_grad = bucket.zero
        all_reduce = bucket.all_reduce_mean
        pack = bucket.pack
        if args.comm == "overlap":      # one collective per encoder layer, issued when that layer's backward is done
            bucket.enable_overlap([list(layer.parameters()) for layer in model.backbone_layers])
        if world > 1:
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)           # communicator set-up outside any capture
            torch.cuda.synchronize()
    else:                                       # single GPU: no collective, so no bucket; autograd assigns .grad

        def zero_grad():
            for p in params:
                p.grad = None

        def all_reduce():
            return None
        pack = None
    if args.torch_adamw:    # A/B only: the framework's fused multi-tensor AdamW
        opt = torch.optim.AdamW(params, lr=1e-5, weight_decay=1e-4, capturable=True, fused=True)
    else:                   # this repository's one-launch AdamW (csrc/optim.cu), same update rule
        opt = bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)

    B, L = args.batch, args.frames
    gen = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(B, L, D_MODEL, generator=gen).pin_memory()
    x_dev = x_host.cuda()

    def fwd_loss(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model.forward_features(x)
        return bm.ops.mean_square_loss(out)          # mean(out^2) in fp32 (one launch forward, one backward)

    use_graph = not args.no_graph
    if args.no_native_block:
        bm.ops.USE_NATIVE_BLOCK = False
    if use_graph and not bucketed:
        runner = bm.GraphedTrainStep(fwd_loss, x_dev, zero_grad, opt, warmup=3)

        def step(x=None):
            return runner.run(x)
    elif use_graph and args.comm != "eager":
        # multi-GPU: forward, backward, the per-layer gradient collectives (parallel branches that overlap the remaining
        # backward) and AdamW are ONE graph
        if args.comm == "overlap":
            post = bucket.finish_overlap
        else:
            def post():
                pack()
                all_reduce()
        runner = bm.GraphedTrainStep(fwd_loss, x_dev, zero_grad, opt, warmup=3, post_backward=post)

        def step(x=None):
            return runner.run(x)
    elif use_graph:
        # round-1 arrangement: the NCCL all-reduce and AdamW launched after the graph
        runner = bm.GraphedTrainStep(fwd_loss, x_dev, zero_grad, None, warmup=3, post_backward=pack)

        def step(x=None):
            loss = runner.run(x)
            all_reduce()
            opt.step()
            return loss
    else:
        def step(x=None):
            zero_grad()
            loss = fwd_loss(x_dev if x is None else x.cuda(non_blocking=True))
            loss.backward()
            if bucketed and args.comm == "overlap":
                bucket.finish_overlap()
            else:
                if pack is not None:
                    pack()
                all_reduce()
            opt.step()
            return loss

    # count our own kernels in one eager step of the sequenced arrangement (the graph replays exactly these)
    bm._lib.launch_count = 0
    with bm.ops.sequenced_block():
        zero_grad()
        fwd_loss(x_dev).backward()
        if bucketed and args.comm == "overlap":
            bucket.finish_overlap()
    torch.cuda.synchronize()
    launches_per_step = bm._lib.launch_count + (0 if args.torch_adamw else 2)   # + AdamW: step tick + update

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    if rank == 0:
        sampler.ready()
    barrier()

    # ---- device-resident timing: per-step CUDA events, L2 flushed (untimed) between steps ----
    K = args.steps
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    w0 = time.perf_counter()
    for s, e in evs:
        flush.zero_()
        s.record()
        loss = step()
        e.record()
    barrier()
    w1 = time.perf_counter()
    dev_ms = sum(s.elapsed_time(e) for s, e in evs)
    if rank == 0 and args.dump_outputs:
        dump_step_outputs(args.dump_outputs, model, loss)

    # ---- end to end: pinned host input -> H2D -> step -> loss.item() every step ----
    pipelined = use_graph and (world == 1 or args.comm != "eager")
    for _ in range(2):
        float(step(x_host).detach())
    barrier()
    t0 = time.perf_counter()
    if pipelined:      # public API: the H2D copy of batch i+1 overlaps step i; every step's loss is read back
        for loss_val in runner.run_pipelined(x_host for _ in range(K)):
            pass
    else:
        for _ in range(K):
            loss_val = float(step(x_host).detach())   # .item(): D2H read + host sync, like src/main.py:1123
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    e2e_ms = (t1 - t0) * 1e3
    clocks = sampler.stop([(w0, w1), (t0, t1)]) if rank == 0 else None   # both timed regions

    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = float(t[0]), float(t[1])

    frames_total = B * L * world * K
    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (scan backward), instrumented eager pass of the same steps ----
        peak, peak_src = load_peaks()
        timer = EventTimer()
        bm._lib.kernel_timer = timer
        if bucketed and args.comm == "overlap":
            bucket.disable_overlap()        # rank 0 alone runs this instrumented pass: no collectives
        for _ in range(3):
            flush.zero_()
            zero_grad()
            fwd_loss(x_dev).backward()
        bm._lib.kernel_timer = None
        times = timer.summary()
        bwd_ms = statistics.mean(times["scan_bwd"][N_LAYERS:])       # drop the first step's launches
        fwd_ms = statistics.mean(times["scan_fwd"][N_LAYERS:])
        alg = scan_bytes(B * L, 2, 2, True)
        achieved = alg / (bwd_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "scan_traffic.json")
        if os.path.exists(tpath) and (B, L) == (64, 201):
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_src = tj.get("scan_bwd_dram_bytes_per_launch"), tj.get("source")
        roofline = {
            "kernel": "scan_bwd_lane_kernel<bf16> (both directions, one launch per layer; the longest kernel of the step)",
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "avg_launch_ms": bwd_ms,
            "algorithmic_bytes_per_launch": alg,
            "note": "bf16 IO, (7D+4N)*2 B per frame per direction (SURVEY 8d) x 12864 frames x 2 directions.  The kernel is "
                    "latency-bound, not HBM-bound (DESIGN.md 4.2: the Phase-6 grid offers 7.8 warps per SM - 1152 one-warp CTAs; "
                    "ncu issue-active 40 %%, XU 29 %%, DRAM 9 %%; the config-2 working set also sits in the 126 MB L2), so the HBM "
                    "fraction is low by construction.  scan_fwd (MUFU-bound, DESIGN.md 4.1) avg launch %.4f ms = %.1f GB/s algorithmic"
                    % (fwd_ms, scan_bytes(B * L, 2, 2, False) / (fwd_ms * 1e-3) / 1e9),
            "kernels_ms": {k: round(statistics.mean(v[len(v) // 3:]), 4) for k, v in times.items()},
        }
        fwd_alg = scan_bytes(B * L, 2, 2, False)
        roofline_more = [
            {"kernel": "scan_fwd_warp_kernel<bf16> (training forward, both directions, one launch per layer)", "bound": "hbm",
             "achieved": fwd_alg / (fwd_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
             "frac": fwd_alg / (fwd_ms * 1e-3) / 1e9 / peak, "avg_launch_ms": fwd_ms, "algorithmic_bytes_per_launch": fwd_alg,
             "traffic": None, "note": "(4D+2N)*2 B per frame per direction (SURVEY 8d); MUFU-bound: 16 ex2 per element (DESIGN.md 4.1)"},
            gemm_roofline(bm, B, L, flush),
        ]
        sweep = None if args.no_sweep else scan_sweep(bm, peak)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = run_cpu_baseline(L, sample_batch=B)
        line = {
            "metric": METRIC, "value": frames_total / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": K, "warmup": max(3, args.warmup), "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict(workload_config(args, world), l2="flushed between steps (256 MB write, untimed); per-step CUDA events summed",
                           launch="CUDA-graph replay" if use_graph else ("eager, native one-call layer entry points" if bm.ops.USE_NATIVE_BLOCK
                                                                          else "eager, Python-sequenced launches"), state="fp32", weights="fp32 master, bf16 autocast",
                           gemm="tcgen05 (this repo)",
                           comm=(None if world == 1 else {"overlap": "NCCL all-reduce (AVG) per encoder layer inside the step "
                                 "graph, overlapping the remaining backward",
                                 "graph": "one NCCL all-reduce inside the step graph",
                                 "eager": "one NCCL all-reduce after the graph"}[args.comm]),
                           optimizer="torch.optim.AdamW(fused)" if args.torch_adamw else "AdamW, one-launch kernel (this repo)"),
            "clocks": clocks,
            "e2e": {"value": frames_total / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / K,
                    "api": ("bimamba_b200.GraphedTrainStep.run_pipelined(pinned host batches) -> float(loss) per step" if pipelined else
                            "bimamba_b200.GraphedTrainStep.run(pinned_host_x) -> loss.item()") if use_graph
                           else "BiMambaBackend.forward_features + backward, eager"},
            "gpu_launches": launches_per_step * K,
            "gpu_launches_per_step": launches_per_step,
            "roofline": roofline,
            "roofline_more": roofline_more,
            "cpu_baseline": cpu,
            "scan_sweep": sweep,
            "scan_sweep_note": ("config 5: single-direction selective_scan op, 524 288 frames, D 288, N 16; per point "
                                "scan_fwd_infer = no-grad forward (the op-boundary bytes), scan_fwd = training forward (also writes "
                                "the fp32 checkpoints every 8 steps and the ungated y), scan_bwd; frac = SURVEY 8(d) algorithmic "
                                "bytes / kernel time / measured HBM peak; rows with time_segments ran the time-parallel forward "
                                "(carry pass + output pass, both launches inside the timed interval)") if sweep else None,
            "loss": loss_val,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        # a CUDA graph that holds captured NCCL work keeps the communicator busy: release it before tearing the
        # process group down, and never let a stuck teardown outlive the measurement (the JSON line is already out)
        if use_graph:
            runner.graph.reset()
        guard = threading.Timer(20.0, lambda: os._exit(0))
        guard.daemon = True
        guard.start()
        dist.destroy_process_group()
        guard.cancel()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
