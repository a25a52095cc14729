"""CUDA-graph capture of one training / scoring step of the Bi-Mamba backend.

At the Phase-6 shapes (B <= 64, L = 201) a backend step is a few hundred short kernels, so it is
launch-latency bound (SURVEY 3.5, 7.2); capturing it once and replaying removes the host from the
loop.  This plays the role a tracing compiler would: explicit capture, static buffers."""
from __future__ import annotations

import copy
from typing import Callable, Optional

import torch

from .ops import seqlens_tensor, sequenced_block


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
    after loading a checkpoint - does not change the model, the moments, or the step count."""

    def __init__(self, step_fn: Callable[[torch.Tensor], torch.Tensor], example: torch.Tensor,
                 zero_grad: Callable[[], None], optimizer: Optional[torch.optim.Optimizer] = None,
                 warmup: int = 3, post_backward: Optional[Callable[[], None]] = None,
                 capture_error_mode: Optional[str] = None, restore_after_warmup: bool = True, lengths=None):
        self.static_x = torch.empty_like(example, device="cuda")
        self.static_x.copy_(example)
        self.static_lengths = None
        args = (self.static_x,)
        if lengths is not None:
            self.static_lengths = seqlens_tensor(lengths, example.shape[0], example.shape[1], self.static_x.device).clone()
            args = (self.static_x, self.static_lengths)
        self.optimizer = optimizer
        snap = _snapshot(optimizer) if (optimizer is not None and restore_after_warmup) else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), sequenced_block():   # warm up what the capture records, not the eager fast path
            for _ in range(max(1, warmup)):          # lazy inits (cuBLAS handles, func attributes) happen here
                zero_grad()
                loss = step_fn(*args)
                loss.backward()
                if post_backward is not None:
                    post_backward()
                if optimizer is not None:
                    optimizer.step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if snap is not None:
            _restore(optimizer, snap)
            torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        if capture_error_mode is None:
            # a process group's watchdog thread issues CUDA calls of its own: with NCCL collectives inside the capture
            # only this thread's calls may invalidate it
            import torch.distributed as dist
            capture_error_mode = "thread_local" if dist.is_available() and dist.is_initialized() else "global"
        with torch.cuda.graph(self.graph, capture_error_mode=capture_error_mode):
            zero_grad()
            self.static_loss = step_fn(*args)
            self.static_loss.backward()
            if post_backward is not None:
                post_backward()
            if optimizer is not None:
                optimizer.step()

    def run(self, x: Optional[torch.Tensor] = None, lengths=None) -> torch.Tensor:
        if x is not None:
            self.static_x.copy_(x, non_blocking=True)
        if lengths is not None:
            if self.static_lengths is None:
                raise ValueError("this step was captured without lengths")
            B, T = self.static_x.shape[:2]
            self.static_lengths.copy_(seqlens_tensor(lengths, B, T, self.static_x.device), non_blocking=True)
        self.graph.replay()
        return self.static_loss

    def run_pipelined(self, host_batches):
        """Generator over pinned host batches: yields float(loss) of every step (a device->host read per step, like
        src/main.py:1123).  The host->device copy of batch i+1 runs on a copy stream while step i replays (double
        buffered staging + one device-to-device copy into the graph's static input), which is what a data loader
        with pinned memory does for the reference loop."""
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream()
            self._stage = [torch.empty_like(self.static_x) for _ in range(2)]
            self._ready = [torch.cuda.Event() for _ in range(2)]
            self._consumed = [torch.cuda.Event() for _ in range(2)]
        copy, main = self._copy_stream, torch.cuda.current_stream()
        it = iter(host_batches)
        nxt = next(it, None)
        if nxt is not None:
            copy.wait_stream(main)
            with torch.cuda.stream(copy):
                self._stage[0].copy_(nxt, non_blocking=True)
                self._ready[0].record(copy)
        idx = 0
        while nxt is not None:
            cur = idx & 1
            main.wait_event(self._ready[cur])
            self.static_x.copy_(self._stage[cur], non_blocking=True)
            self._consumed[cur].record(main)
            nxt = next(it, None)
            if nxt is not None:
                with torch.cuda.stream(copy):
                    if idx > 0:
                        copy.wait_event(self._consumed[1 - cur])
                    self._stage[1 - cur].copy_(nxt, non_blocking=True)
                    self._ready[1 - cur].record(copy)
            self.graph.replay()
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
        with torch.cuda.stream(side), torch.no_grad(), sequenced_block():
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
