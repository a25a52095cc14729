"""CUDA-graph capture of one training / scoring step of the Bi-Mamba backend.

At the Phase-6 shapes (B <= 64, L = 201) a backend step is a few hundred short kernels, so it is
launch-latency bound (SURVEY 3.5, 7.2); capturing it once and replaying removes the host from the
loop.  This plays the role a tracing compiler would: explicit capture, static buffers."""
from __future__ import annotations

import contextlib
import copy
import inspect
from typing import Callable, Optional

import torch

from . import ops
from .ops import seqlens_tensor


def _as_captured():
    """The warm-up runs the arrangement the capture records: the native layer calls with their second stream, or, with
    the side stream switched off (BIMAMBA_SIDE_STREAM=0), the sequenced Functions."""
    return contextlib.nullcontext() if ops.SIDE_STREAM else ops.sequenced_block()


def _snapshot(optimizer):
    params = [p for g in optimizer.param_groups for p in g["params"]]
    return params, [p.detach().clone() for p in params], copy.deepcopy(optimizer.state_dict())


def _restore(optimizer, snap):
    """Undo the warm-up's optimizer steps: parameters back to their values, optimizer state back to what it was (or,
    if there was none yet, to the freshly initialised value: zero moments, step 0)."""
    params, values, sd = snap
    with torch.no_grad():
        for p, v in zip(params, values):
            p.copy_(v)
    if sd["state"] or hasattr(optimizer, "_export_state"):      # FusedAdamW also resets itself from an empty state
        optimizer.load_state_dict(sd)
    else:
        for st in optimizer.state.values():
            for v in st.values():
                if torch.is_tensor(v):
                    v.zero_()


class GraphedTrainStep:
    """Captures  zero-grad -> forward -> loss -> backward [-> post_backward] [-> optimizer.step]  for a fixed input
    shape (post_backward: e.g. FlatGradBucket.pack, so a multi-GPU step leaves the graph with the flat gradient ready
    for the all-reduce).

    step_fn(x) must return a scalar loss tensor and must be capture-safe (no host sync).
    `run(x)` copies x (host-pinned or device) into the static input, replays, and returns the static
    loss tensor (read it with .item() to synchronise).

    With `lengths` (an example (B,) vector of frame counts, see ops.seqlens_tensor) step_fn is called as
    step_fn(x, lengths) with the lengths in a static int32 device buffer, and run(x, lengths) copies both: one captured
    training step then serves every mix of utterance lengths padded to the example's shape (variable-length training,
    e.g. net(x, lengths, mask_padding=True)).

    The `warmup` iterations before the capture run real optimizer steps on the example batch (lazy initialisation of
    handles, function attributes and optimizer state must happen outside the capture); with restore_after_warmup
    (default) the parameters and the optimizer state are put back afterwards, so building the runner - e.g. right
    after loading a checkpoint - does not change the model, the moments, or the step count (nor the scaler's scale
    and growth tracker, the averaged parameters or n_averaged).

    The fp16 recipe (src/main.py:1049-1117), with a FusedAdamW:
      * scaler (DeviceGradScaler), max_norm, ema (FusedEMA): the loss is multiplied by the device scale before
        backward and the captured step is optimizer.step(scaler=..., max_norm=..., ema=...) - unscale, clip, the skip
        of an overflowing step, the scale update and the EMA, with no host read;
      * accumulation_steps = k > 1: the loss is divided by k and two graphs are captured, a micro-step (forward and
        backward, accumulating into the gradients) and the optimizer step ([post_backward ->] step -> zero_grad).
        `run` replays the micro-step, and the optimizer step after every k-th call.  The gradients must be static
        buffers zeroed in place by `zero_grad` (FlatGradBucket(accumulate=True).zero).
    `run` returns step_fn's loss, unscaled and undivided.  post_backward (e.g. the multi-GPU all-reduce) runs before the
    optimizer step, so the inf check and the norm see the global gradient; an inf or NaN survives the all-reduce, so
    every rank skips the same steps.

    Labels and Mixup (src/main.py:1038-1046, :1070-1073):
      * labels (an example (B,) label vector) gives a static label buffer, and step_fn is then called as
        step_fn(x, y, lengths, mix) - lengths the static frame counts or None, mix a training.MixState or None;
      * mixup_alpha > 0 (needs labels) gives static perm and mix buffers: every `run` (every micro-step) draws lam ~
        Beta(alpha, alpha) and a permutation on the host (training.draw_mixup, perm on `generator`), and copies them in
        one 8 + 4B-byte copy, without a device sync, so each replay mixes with its own draw.  step_fn mixes with
        training.mixup_batch(x, y, lam=mix.mix, lengths=lengths, index=mix.perm) and weights its loss with
        training.mixup_loss(..., lam=mix.mix).  `last_lam` holds the last draw's lam.
    run(x, lengths, y=y) copies whichever of them is given."""

    def __init__(self, step_fn: Callable[[torch.Tensor], torch.Tensor], example: torch.Tensor,
                 zero_grad: Callable[[], None], optimizer: Optional[torch.optim.Optimizer] = None,
                 warmup: int = 3, post_backward: Optional[Callable[[], None]] = None,
                 capture_error_mode: Optional[str] = None, restore_after_warmup: bool = True, lengths=None,
                 scaler=None, max_norm: Optional[float] = None, ema=None, accumulation_steps: int = 1,
                 labels: Optional[torch.Tensor] = None, mixup_alpha: float = 0.0,
                 generator: Optional[torch.Generator] = None):
        self.static_x = torch.empty_like(example, device="cuda")
        self.static_x.copy_(example)
        self.static_lengths = None
        args = (self.static_x,)
        if lengths is not None:
            self.static_lengths = seqlens_tensor(lengths, example.shape[0], example.shape[1], self.static_x.device).clone()
            args = (self.static_x, self.static_lengths)
        self.static_y = self.mix = None
        self.mixup_alpha, self.generator, self.last_lam = float(mixup_alpha), generator, None
        if self.mixup_alpha > 0 and labels is None:
            raise ValueError("mixup_alpha needs labels (the mixed batch is scored against both label sets)")
        if labels is not None:
            self.static_y = labels.to("cuda").view(-1).long().clone()
            if self.static_y.numel() != example.shape[0]:
                raise ValueError(f"labels must hold {example.shape[0]} entries, got {self.static_y.numel()}")
            if self.mixup_alpha > 0:
                # one buffer, one copy per run: [lam, 1 - lam] as fp32 bits, then the permutation; until the first run
                # the identity at lam = 1 (the warm-up and the capture see a valid draw)
                B = example.shape[0]
                self._draw = torch.empty(B + 2, dtype=torch.int32, device=self.static_x.device)
                self._draw.copy_(self._draw_host(1.0, torch.arange(B)))
                from .training import MixState
                self.mix = MixState(self._draw[2:], self._draw[:2].view(torch.float32))
            args = (self.static_x, self.static_y, self.static_lengths, self.mix)
        self.optimizer = optimizer
        k = self.accumulation_steps = int(accumulation_steps)
        if k < 1:
            raise ValueError("accumulation_steps must be >= 1")
        if scaler is not None and not scaler.is_enabled():
            scaler = None
        step_kw = {}
        if scaler is not None or max_norm is not None or ema is not None:
            if optimizer is None or "scaler" not in inspect.signature(optimizer.step).parameters:
                raise TypeError("scaler / max_norm / ema need an optimizer whose step takes them (FusedAdamW)")
            step_kw = dict(scaler=scaler, max_norm=max_norm, ema=ema)
            if scaler is not None:
                scaler._lazy_init(self.static_x.device)         # the record exists before the snapshot and the capture
        if k > 1 and optimizer is None:
            raise ValueError("accumulation_steps > 1 needs the optimizer")
        self._micro = 0
        snap = _snapshot(optimizer) if (optimizer is not None and restore_after_warmup) else None
        amp_snap = None
        if restore_after_warmup:
            amp_snap = (scaler._record.clone() if scaler is not None else None,
                        ema.snapshot() if ema is not None else None)

        def forward_backward():
            loss = step_fn(*args)
            scaled = loss / k if k > 1 else loss
            if scaler is not None:
                scaled = scaler.scale(scaled)
            scaled.backward()
            return loss

        def apply():
            if post_backward is not None:
                post_backward()
            if optimizer is not None:
                optimizer.step(**step_kw)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), _as_captured():
            for _ in range(max(1, warmup)):          # lazy inits (cuBLAS handles, func attributes) happen here
                zero_grad()
                forward_backward()
                apply()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if snap is not None:
            _restore(optimizer, snap)
        if amp_snap is not None:
            if amp_snap[0] is not None:
                scaler._record.copy_(amp_snap[0])
            if amp_snap[1] is not None:
                ema.restore(amp_snap[1])
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        self.apply_graph = None
        if capture_error_mode is None:
            # a process group's watchdog thread issues CUDA calls of its own: with NCCL collectives inside the capture
            # only this thread's calls may invalidate it
            import torch.distributed as dist
            capture_error_mode = "thread_local" if dist.is_available() and dist.is_initialized() else "global"
        if k == 1:
            with torch.cuda.graph(self.graph, capture_error_mode=capture_error_mode):
                zero_grad()
                self.static_loss = forward_backward()
                apply()
            return
        zero_grad()
        params = [p for g in optimizer.param_groups for p in g["params"] if p.requires_grad]
        if any(p.grad is None for p in params):
            raise ValueError("accumulation_steps > 1 accumulates into static gradient buffers: zero_grad must zero "
                             "them in place (e.g. FlatGradBucket(accumulate=True).zero), not set them to None")
        torch.cuda.synchronize()
        with torch.cuda.graph(self.graph, capture_error_mode=capture_error_mode):
            self.static_loss = forward_backward()
        self.apply_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.apply_graph, pool=self.graph.pool(), capture_error_mode=capture_error_mode):
            apply()
            zero_grad()

    def _replay(self):
        self.graph.replay()
        if self.apply_graph is not None:
            self._micro += 1
            if self._micro == self.accumulation_steps:
                self.apply_graph.replay()
                self._micro = 0

    @staticmethod
    def _draw_host(lam: float, perm: torch.Tensor) -> torch.Tensor:
        """The host image of the draw buffer: [lam, 1 - lam] (fp32, 1 - lam taken in double) | perm (int32)."""
        mix = torch.tensor([lam, 1.0 - lam], dtype=torch.float32).view(torch.int32)
        return torch.cat([mix, perm.to(torch.int32)])

    def _load(self, y=None, lengths=None):
        """Copy the labels and lengths given, and a fresh Mixup draw, into the static buffers (no device sync)."""
        if y is not None:
            if self.static_y is None:
                raise ValueError("this step was captured without labels")
            self.static_y.copy_(y.view(-1), non_blocking=True)
        if lengths is not None:
            if self.static_lengths is None:
                raise ValueError("this step was captured without lengths")
            B, T = self.static_x.shape[:2]
            self.static_lengths.copy_(seqlens_tensor(lengths, B, T, self.static_x.device), non_blocking=True)
        if self.mix is not None:
            from .training import draw_mixup
            self.last_lam, perm = draw_mixup(self.static_x.shape[0], self.mixup_alpha, self.generator)
            self._draw.copy_(self._draw_host(self.last_lam, perm), non_blocking=True)

    def run(self, x: Optional[torch.Tensor] = None, lengths=None, *, y: Optional[torch.Tensor] = None) -> torch.Tensor:
        if x is not None:
            self.static_x.copy_(x, non_blocking=True)
        self._load(y, lengths)
        self._replay()
        return self.static_loss

    def _host_parts(self, batch):
        """A host batch x or (x, y[, lengths]) -> its tensors in the order of self._statics (lengths as int32)."""
        if isinstance(batch, torch.Tensor):
            return [batch]
        parts = [batch[0]]
        if len(batch) > 1 and batch[1] is not None:
            if self.static_y is None:
                raise ValueError("this step was captured without labels")
            parts.append(batch[1].view(-1))
        if len(batch) > 2 and batch[2] is not None:
            if self.static_lengths is None or len(parts) < 2:
                raise ValueError("lengths in a pipelined batch need a step captured with labels and lengths")
            parts.append(seqlens_tensor(batch[2], *self.static_x.shape[:2], "cpu"))
        return parts

    def run_pipelined(self, host_batches):
        """Generator over pinned host batches, each x or (x, y[, lengths]): yields float(loss) of every step (a
        device->host read per step, like src/main.py:1123).  The host->device copy of batch i+1 runs on a copy stream
        while step i replays (double buffered staging + one device-to-device copy per tensor into the graph's static
        buffers), which is what a data loader with pinned memory does for the reference loop.  A Mixup draw is made
        for every step, as in run()."""
        statics = [t for t in (self.static_x, self.static_y, self.static_lengths) if t is not None]
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream()
            self._stage = [[torch.empty_like(t) for t in statics] for _ in range(2)]
            self._ready = [torch.cuda.Event() for _ in range(2)]
            self._consumed = [torch.cuda.Event() for _ in range(2)]
        copy, main = self._copy_stream, torch.cuda.current_stream()
        it = iter(host_batches)
        nxt = next(it, None)
        count = [0, 0]

        def stage(slot, batch):
            parts = self._host_parts(batch)
            for buf, part in zip(self._stage[slot], parts):
                buf.copy_(part, non_blocking=True)
            count[slot] = len(parts)
            self._ready[slot].record(copy)
        if nxt is not None:
            copy.wait_stream(main)
            with torch.cuda.stream(copy):
                stage(0, nxt)
        idx = 0
        while nxt is not None:
            cur = idx & 1
            main.wait_event(self._ready[cur])
            for dst, buf in zip(statics[:count[cur]], self._stage[cur]):
                dst.copy_(buf, non_blocking=True)
            self._consumed[cur].record(main)
            nxt = next(it, None)
            if nxt is not None:
                with torch.cuda.stream(copy):
                    if idx > 0:
                        copy.wait_event(self._consumed[1 - cur])
                    stage(1 - cur, nxt)
            self._load()
            self._replay()
            yield float(self.static_loss.detach())
            idx += 1


class GraphedForward:
    """Captures a no-grad forward (scoring, src/main.py:958-995) for a fixed input shape.

    With `lengths` (an example (B,) vector of frame counts, see ops.seqlens_tensor) `fn` is called as fn(x, lengths)
    with the lengths in a static int32 device buffer, and run(x, lengths) copies both: one captured graph then scores
    every mix of utterance lengths padded to the example's shape."""

    def __init__(self, fn: Callable[..., torch.Tensor], example: torch.Tensor, warmup: int = 2, lengths=None):
        self.static_x = torch.empty_like(example, device="cuda")
        self.static_x.copy_(example)
        self.static_lengths = None
        args = (self.static_x,)
        if lengths is not None:
            self.static_lengths = seqlens_tensor(lengths, example.shape[0], example.shape[1], self.static_x.device).clone()
            args = (self.static_x, self.static_lengths)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad(), _as_captured():
            for _ in range(max(1, warmup)):
                fn(*args)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph), torch.no_grad():
            self.static_out = fn(*args)

    def run(self, x: Optional[torch.Tensor] = None, lengths=None):
        if x is not None:
            self.static_x.copy_(x, non_blocking=True)
        if lengths is not None:
            if self.static_lengths is None:
                raise ValueError("this graph was captured without lengths")
            B, T = self.static_x.shape[:2]
            self.static_lengths.copy_(seqlens_tensor(lengths, B, T, self.static_x.device), non_blocking=True)
        self.graph.replay()
        return self.static_out
