"""Loss scaling and the parameter average of the fp16 recipe (src/main.py:486, :495, :1100-1117) with their state on the
device, for `FusedAdamW.step(scaler=..., max_norm=..., ema=...)`: no host read anywhere in the optimizer step, so the
step is CUDA-graph capturable (`GraphedTrainStep(..., scaler=..., max_norm=..., ema=...)`)."""
from __future__ import annotations

import torch
import torch.nn as nn

# struct bimamba_amp as int32 words: scale, growth_tracker, found_inf, total_norm, clip_coef, reserved[3]
_SCALE, _TRACKER, _FOUND_INF, _TOTAL_NORM, _CLIP_COEF, _WORDS = 0, 1, 2, 3, 4, 8


def new_amp_record(device, scale: float = 1.0, growth_tracker: int = 0) -> torch.Tensor:
    """A `struct bimamba_amp` in device memory, as 8 int32 words (fp32 fields are views through .view(float32))."""
    rec = torch.zeros(_WORDS, dtype=torch.int32, device=device)
    f = rec.view(torch.float32)
    f[_SCALE] = scale
    rec[_TRACKER] = growth_tracker
    f[_CLIP_COEF] = 1.0
    return rec


class DeviceGradScaler:
    """`torch.amp.GradScaler` whose scale, growth tracker and found-inf flag live in one device record
    (`struct bimamba_amp`), so unscale, the inf check, the skip and the scale update run inside
    `FusedAdamW.step(scaler=self)` without a host read.

    Same constructor arguments, defaults and checks as torch's; `state_dict()` / `load_state_dict()` use torch's format,
    so a checkpoint moves between the two either way.  `scale(loss)` is a device multiply (capturable); `get_scale()`
    reads the device and is meant for logging outside the training loop.  With `enabled=False` everything is the
    identity and `FusedAdamW.step(scaler=...)` ignores the scaler, as torch's `scaler.step` just calls `optimizer.step()`.
    There is no `unscale_` / `step` / `update`: `FusedAdamW.step(scaler=self, ...)` does all three."""

    def __init__(self, device: str = "cuda", init_scale: float = 2.0 ** 16, growth_factor: float = 2.0,
                 backoff_factor: float = 0.5, growth_interval: int = 2000, enabled: bool = True):
        self._device = device
        self._enabled = enabled
        if enabled:
            if growth_factor <= 1.0:
                raise AssertionError("The growth factor must be > 1.0.")
            if backoff_factor >= 1.0:
                raise AssertionError("The backoff factor must be < 1.0.")
        self._init_scale = init_scale
        self._growth_factor = growth_factor
        self._backoff_factor = backoff_factor
        self._growth_interval = growth_interval
        self._init_growth_tracker = 0
        self._record = None

    def is_enabled(self) -> bool:
        return self._enabled

    def _lazy_init(self, device=None) -> torch.Tensor:
        if self._record is None:
            dev = torch.device(device if device is not None else self._device)
            if dev.type == "cuda" and dev.index is None:
                dev = torch.device("cuda", torch.cuda.current_device())
            self._record = new_amp_record(dev, self._init_scale, self._init_growth_tracker)
        return self._record

    # 0-d device views of the record (as torch.amp.GradScaler's `_scale` / `_growth_tracker`)
    @property
    def _scale(self) -> torch.Tensor:
        return self._lazy_init().view(torch.float32)[_SCALE]

    @property
    def _growth_tracker(self) -> torch.Tensor:
        return self._lazy_init()[_TRACKER]

    @property
    def found_inf(self) -> torch.Tensor:
        """0-d fp32 on the device: 1 when the last step's gradient held an inf or NaN (that step was skipped)."""
        return self._lazy_init().view(torch.float32)[_FOUND_INF]

    def scale(self, outputs):
        """outputs * scale on the device (a tensor, or a list / tuple of tensors), as torch.amp.GradScaler.scale."""
        if not self._enabled:
            return outputs
        if isinstance(outputs, torch.Tensor):
            rec = self._lazy_init(outputs.device)
            return outputs * rec.view(torch.float32)[_SCALE].to(device=outputs.device, non_blocking=True)
        if isinstance(outputs, (list, tuple)):
            return type(outputs)(self.scale(o) for o in outputs)
        raise ValueError("outputs must be a Tensor or a list / tuple of Tensors")

    def get_scale(self) -> float:
        """The current scale as a Python float (a device read: for logging outside the loop)."""
        if not self._enabled:
            return 1.0
        return self._init_scale if self._record is None else float(self._scale.item())

    def get_growth_factor(self) -> float:
        return self._growth_factor

    def get_backoff_factor(self) -> float:
        return self._backoff_factor

    def get_growth_interval(self) -> int:
        return self._growth_interval

    def state_dict(self) -> dict:
        """torch.amp.GradScaler's format: scale, growth_factor, backoff_factor, growth_interval, _growth_tracker."""
        if not self._enabled:
            return {}
        tracker = self._init_growth_tracker if self._record is None else int(self._growth_tracker.item())
        return {"scale": self.get_scale(), "growth_factor": self._growth_factor, "backoff_factor": self._backoff_factor,
                "growth_interval": self._growth_interval, "_growth_tracker": tracker}

    def load_state_dict(self, state_dict: dict) -> None:
        """Loads a DeviceGradScaler or torch.amp.GradScaler state_dict (written into the live record, so a captured
        step keeps using it)."""
        if not self._enabled:
            return
        if len(state_dict) == 0:
            raise RuntimeError("The source state dict is empty, possibly because it was saved from a disabled instance "
                               "of GradScaler.")
        self._init_scale = float(state_dict["scale"])
        self._growth_factor = float(state_dict["growth_factor"])
        self._backoff_factor = float(state_dict["backoff_factor"])
        self._growth_interval = int(state_dict["growth_interval"])
        self._init_growth_tracker = int(state_dict["_growth_tracker"])
        if self._record is not None:
            self._scale.fill_(self._init_scale)
            self._growth_tracker.fill_(self._init_growth_tracker)


class FusedEMA:
    """Pairs a `torch.optim.swa_utils.AveragedModel` built with `multi_avg_fn=get_ema_multi_avg_fn(decay)` (src/main.py:495)
    with the model it averages, for `FusedAdamW.step(ema=...)`: the AdamW pass moves the average of every parameter it
    updates, a second launch of the same kernel averages the model's parameters the optimizer does not hold (frozen
    ones), buffers are copied, and `n_averaged` is incremented on the device.  The result equals
    `averaged.update_parameters(model)`; `averaged` stays the user's object, so evaluation code and its `module.*` /
    `n_averaged` state_dict keys are the reference's.

    Parameters are paired by name.  `n_averaged` is moved to the parameters' device if it is elsewhere (AveragedModel
    creates it on the CPU unless given a device)."""

    def __init__(self, averaged: nn.Module, model: nn.Module, decay: float = 0.999):
        if not 0.0 <= decay <= 1.0:
            raise ValueError(f"Invalid decay value {decay} provided. Please provide a value in [0,1] range.")
        if getattr(averaged, "use_buffers", False):
            raise NotImplementedError("AveragedModel(use_buffers=True) averages buffers too; FusedEMA pairs parameters "
                                      "and copies buffers (use_buffers=False, the reference's setting)")
        avg_params = dict(averaged.module.named_parameters())
        self.pairs = []
        for name, p in model.named_parameters():
            a = avg_params.get(name)
            if a is None or a.shape != p.shape:
                raise ValueError(f"the averaged model has no parameter {name!r} of shape {tuple(p.shape)}")
            for t in (p, a):
                if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
                    raise TypeError("FusedEMA averages contiguous fp32 CUDA parameters")
            self.pairs.append((p, a))
        if len(self.pairs) != len(avg_params):
            raise ValueError("the averaged model has parameters the model does not have")
        avg_bufs = dict(averaged.module.named_buffers())
        self.buffers = [(b, avg_bufs[n]) for n, b in model.named_buffers()]
        dev = self.pairs[0][0].device if self.pairs else torch.device("cuda")
        if averaged.n_averaged.device != dev:
            averaged.n_averaged = averaged.n_averaged.to(dev)
        self.averaged, self.model, self.decay = averaged, model, decay
        self.weight = 1.0 - decay          # torch._foreach_lerp_'s weight in get_ema_multi_avg_fn

    @property
    def n_averaged(self) -> torch.Tensor:
        return self.averaged.n_averaged

    def snapshot(self):
        return [a.detach().clone() for _, a in self.pairs], [b.detach().clone() for _, b in self.buffers], \
            self.n_averaged.detach().clone()

    def restore(self, snap):
        params, bufs, n = snap
        with torch.no_grad():
            for (_, a), v in zip(self.pairs, params):
                a.copy_(v)
            for (_, b), v in zip(self.buffers, bufs):
                b.copy_(v)
            self.n_averaged.copy_(n)
