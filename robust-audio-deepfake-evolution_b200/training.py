"""Training-loop pieces of the Phase-6 recipe around the Bi-Mamba backend (SURVEY 8 row f3): what `train_epoch`
(src/main.py:998-1126) does for one optimizer step - Mixup, fp16/bf16 autocast + GradScaler, FGM's second forward /
backward, gradient accumulation, the (new) data-parallel all-reduce, unscale + clip, optimizer step, EMA - plus the
minimal LoRA the reference gets from `peft` (not installed here) and the BatchNorm freeze.

Everything is plain PyTorch on top of the drop-in modules: the hot path is untouched, these are the callers on either
side of it.  Differences from the reference loop, all deliberate:
  * no host synchronisation inside a step: FGM's `if norm != 0 and not isnan(norm)` (main.py:92) is a device-side
    select, and the loss is returned as a tensor (main.py:1123 calls .item() per micro-batch);
  * gradients are averaged over ranks once per optimizer step, after FGM's second backward and before unscale / clip
    (main.py:1077, :1097 -> :1103-1104), through `FlatGradBucket` (one flat NCCL all-reduce).
"""
from __future__ import annotations

import math
from typing import Callable, Iterable, NamedTuple, Optional, Sequence

import torch
import torch.nn as nn


# ----------------------------------------------------------------------------------------------------------------------
# FGM (src/main.py:74-100)
# ----------------------------------------------------------------------------------------------------------------------
class FGM:
    """Fast Gradient Method on the parameters whose name contains `emb_name` (reference: WavLM's
    'feature_projection').  attack(): p += epsilon * grad / ||grad||; restore(): put the saved values back.
    The gradient may be GradScaler-scaled: the scale cancels in grad / ||grad|| (SURVEY appendix B)."""

    def __init__(self, model: nn.Module, emb_name: str = "feature_projection", epsilon: float = 1.0):
        self.model = model
        self.emb_name = emb_name
        self.epsilon = epsilon
        self.backup = {}

    def _targets(self):
        for name, param in self.model.named_parameters():
            if param.requires_grad and self.emb_name in name:
                yield name, param

    @torch.no_grad()
    def attack(self):
        for name, param in self._targets():
            self.backup[name] = param.detach().clone()
            if param.grad is None:
                continue
            g = param.grad
            norm = torch.linalg.vector_norm(g.float())
            ok = torch.isfinite(norm) & (norm > 0)                       # main.py:92, without the host round trip
            scale = torch.where(ok, self.epsilon / norm.clamp_min(1e-30), torch.zeros_like(norm))
            param.add_((g.float() * scale).to(param.dtype))

    @torch.no_grad()
    def restore(self):
        for name, param in self._targets():
            if name in self.backup:
                param.copy_(self.backup[name])
        self.backup = {}


# ----------------------------------------------------------------------------------------------------------------------
# Mixup (src/main.py:1038-1046, :1070-1075)
# ----------------------------------------------------------------------------------------------------------------------
class MixState(NamedTuple):
    """The device side of one Mixup draw, as the kernel reads it: perm (B,) int32 and mix (2,) fp32 = (lam, 1 - lam),
    both weights formed in double on the host and rounded to fp32 (as torch rounds a Python scalar for an fp32/16-bit
    tensor).  A captured step reads them from static buffers, so every replay mixes with that replay's draw."""
    perm: torch.Tensor
    mix: torch.Tensor


def mix_record(lam: float, device) -> torch.Tensor:
    """(2,) fp32 (lam, 1 - lam) on `device`: 1 - lam is taken in double before the rounding, as `(1.0 - lam) * x`."""
    return torch.tensor([lam, 1.0 - lam], dtype=torch.float32).to(device, non_blocking=True)


def draw_mixup(batch: int, alpha: float, generator: Optional[torch.Generator] = None):
    """The host draw of one Mixup step, in mixup_batch's order -> (lam, permutation as a CPU int64 tensor): lam ~
    Beta(alpha, alpha) from torch's global generator, then torch.randperm(batch) on `generator` (a CPU generator, or
    torch's global one)."""
    lam = float(torch.distributions.Beta(alpha, alpha).sample())
    return lam, torch.randperm(batch, generator=generator)


def _mix_cpu(x, index, lam, lengths):
    """The CPU form of the kernel's contract (the CPU tests' stand-ins): the same three roundings, by selection."""
    n = torch.as_tensor(lengths, device=x.device).long().clamp(0, x.size(1))
    t = torch.arange(x.size(1), device=x.device).view(1, -1, *([1] * (x.dim() - 2)))
    keep_a, keep_b = t < n.view(-1, *([1] * (x.dim() - 1))), t < n[index].view(-1, *([1] * (x.dim() - 1)))
    a = torch.where(keep_a, lam * x, torch.zeros((), dtype=x.dtype))
    c = torch.where(keep_b, (1.0 - lam) * x[index], torch.zeros((), dtype=x.dtype))
    return a + c, torch.maximum(n, n[index])


def mixup_batch(x: torch.Tensor, y: torch.Tensor, alpha: float = 1.0, generator: Optional[torch.Generator] = None,
                lam=None, lengths=None, *, index: Optional[torch.Tensor] = None):
    """-> (mixed_x, y_a, y_b, lam), and with `lengths` (mixed_x, y_a, y_b, lam, mixed_lengths): lam ~ Beta(alpha,
    alpha) and one permutation of the batch, drawn on the host unless given (`lam`, `index`).  Batches of one sample
    are returned unchanged with lam = 1 (main.py:1038, :1043-1046).

    CUDA tensors are mixed by one bimamba_mixup_frames launch: without lengths the bits of `lam * x + (1.0 - lam) *
    x[index]`; with lengths (per-utterance frame counts of the right-padded batch x, as ops.seqlens_tensor takes them)
    each clip adds only over its own frames, zero-padded, and mixed utterance b has max(n_b, n_index[b]) frames
    (returned as a (B,) int32 tensor on x's device).  The capture-safe form passes lam as the (2,) device record of
    mix_record and index as a device int32 tensor (a MixState's fields): nothing is read or drawn on the host, and the
    returned lam is that record, which mixup_loss takes."""
    B = x.size(0)
    if B <= 1 or alpha <= 0:
        return (x, y, y, 1.0) if lengths is None else (x, y, y, 1.0, lengths)
    if lam is None:
        lam = float(torch.distributions.Beta(alpha, alpha).sample())
    if index is None:
        index = torch.randperm(B, generator=generator, device=x.device if generator is None else generator.device)
    device_lam = isinstance(lam, torch.Tensor)
    if not x.is_cuda:
        if device_lam:
            raise ValueError("a device lam record needs CUDA tensors")
        index = index.to(x.device)
        if lengths is None:
            return lam * x + (1.0 - lam) * x[index], y, y[index], lam
        mx, ml = _mix_cpu(x, index, lam, lengths)
        return mx, y, y[index], lam, ml
    from .ops import mixup_frames, seqlens_tensor
    perm = index.to(device=x.device, dtype=torch.int32)
    mix = lam if device_lam else mix_record(lam, x.device)
    sl = None if lengths is None else seqlens_tensor(lengths, B, x.size(1), x.device)
    mx, ml = mixup_frames(x, perm, mix, sl)
    y_b = y[perm]
    return (mx, y, y_b, lam) if lengths is None else (mx, y, y_b, lam, ml)


def mixup_loss(loss_fn: Callable, out, feats, y_a, y_b, lam):
    """lam * L(out, y_a) + (1 - lam) * L(out, y_b) (main.py:1070-1073).  lam: a float; a 0-d device tensor (1 - lam is
    then taken on the device); or the (2,) record (lam, 1 - lam) of mix_record, whose weights give the bits of the
    float form, so a captured step with a device draw computes what the eager step computes with the host's float."""
    if isinstance(lam, torch.Tensor):
        w_a, w_b = (lam[0], lam[1]) if lam.dim() == 1 else (lam, 1.0 - lam)
        return w_a * loss_fn(out, feats, y_a) + w_b * loss_fn(out, feats, y_b)
    if lam == 1.0:
        return loss_fn(out, feats, y_a)
    return lam * loss_fn(out, feats, y_a) + (1.0 - lam) * loss_fn(out, feats, y_b)


# ----------------------------------------------------------------------------------------------------------------------
# minimal LoRA (what peft's get_peft_model does for src/main.py:103-158: r = 8, alpha = 32, dropout 0.1 on q_proj / v_proj)
# ----------------------------------------------------------------------------------------------------------------------
class LoRALinear(nn.Module):
    """y = base(x) + (alpha / r) * B(A(dropout(x))); base frozen, A ~ kaiming-uniform, B = 0 (the adapter starts as the
    identity update)."""

    def __init__(self, base: nn.Linear, r: int = 8, alpha: int = 32, dropout: float = 0.1):
        super().__init__()
        self.base = base
        for p in self.base.parameters():
            p.requires_grad_(False)
        self.scaling = alpha / r
        self.lora_dropout = nn.Dropout(dropout) if dropout > 0 else nn.Identity()
        self.lora_A = nn.Linear(base.in_features, r, bias=False)
        self.lora_B = nn.Linear(r, base.out_features, bias=False)
        nn.init.kaiming_uniform_(self.lora_A.weight, a=math.sqrt(5))
        nn.init.zeros_(self.lora_B.weight)
        self.lora_A.to(base.weight.device)
        self.lora_B.to(base.weight.device)

    def forward(self, x):
        return self.base(x) + self.lora_B(self.lora_A(self.lora_dropout(x))) * self.scaling

    # transformers' WavLM attention does not CALL q_proj / v_proj: it reads their .weight / .bias and hands them to
    # F.multi_head_attention_forward (modeling_wavlm.py).  Expose the merged weight W + (alpha / r) B A there, so the
    # adapter is active (and trained) on that path too (adapter dropout cannot apply to a merged weight).
    @property
    def weight(self):
        return self.base.weight + self.scaling * (self.lora_B.weight @ self.lora_A.weight)

    @property
    def bias(self):
        return self.base.bias

    @property
    def in_features(self):
        return self.base.in_features

    @property
    def out_features(self):
        return self.base.out_features


def apply_lora(module: nn.Module, target_modules: Sequence[str] = ("q_proj", "v_proj"), r: int = 8, alpha: int = 32,
               dropout: float = 0.1) -> int:
    """Freeze every parameter of `module` and wrap each nn.Linear whose attribute name is in `target_modules` with a
    LoRALinear (main.py:121-134).  Returns the number of adapted layers."""
    for p in module.parameters():
        p.requires_grad_(False)
    n = 0
    for parent in list(module.modules()):
        for name, child in list(parent.named_children()):
            if name in target_modules and isinstance(child, nn.Linear):
                setattr(parent, name, LoRALinear(child, r, alpha, dropout))
                n += 1
    return n


def freeze_batch_norm_stats(model: nn.Module) -> None:
    """BatchNorm layers to eval() while the model trains (main.py:44-51; `freeze_bn: true` in Phase 6)."""
    for m in model.modules():
        if isinstance(m, (nn.BatchNorm1d, nn.BatchNorm2d, nn.BatchNorm3d)):
            m.eval()


# ----------------------------------------------------------------------------------------------------------------------
# one optimizer step of train_epoch (src/main.py:1031-1116)
# ----------------------------------------------------------------------------------------------------------------------
class Phase6TrainStep:
    """One optimizer step over `accumulation_steps` micro-batches, as the reference's loop body:

        for each micro-batch:  [mixup] -> autocast forward -> loss / accumulation_steps -> scaler.scale(loss).backward()
                               [FGM: attack -> autocast forward -> loss -> backward -> restore]
        [all-reduce the flat gradient bucket over ranks]  -> scaler.unscale_ -> clip_grad_norm_(3.0) -> scaler.step
        -> scaler.update -> zero grads -> [EMA update] -> [scheduler.step]

    model(x) must return (features, logits) like the reference Model.forward, and model(x, lengths, mask_padding=True)
    too when micro-batches carry lengths.  `loss_fn(logits, feats, target)`.
    bucket: a FlatGradBucket(accumulate=True) over the trainable parameters when running data-parallel (its views ARE
    the .grad tensors, so both backward passes of FGM and every micro-batch accumulate into it), else None.

    With a DeviceGradScaler and a FusedAdamW the tail is one FusedAdamW.step(scaler=, max_norm=, ema=) on the device,
    with no host read in the step; ema_model is then a FusedEMA (the AveragedModel paired with the model) or None.
    With torch's GradScaler the tail is torch's calls above."""

    def __init__(self, model: nn.Module, optimizer: torch.optim.Optimizer, loss_fn: Callable, *,
                 scaler: Optional[torch.amp.GradScaler] = None, autocast_dtype: Optional[torch.dtype] = torch.float16,
                 fgm: Optional[FGM] = None, mixup_alpha: float = 0.0, accumulation_steps: int = 1, max_norm: float = 3.0,
                 ema_model=None, scheduler=None, bucket=None, freeze_bn: bool = False, model_kwargs: Optional[dict] = None):
        self.model, self.optimizer, self.loss_fn = model, optimizer, loss_fn
        self.scaler = scaler if scaler is not None else torch.amp.GradScaler("cuda", enabled=False)
        self.autocast_dtype = autocast_dtype
        self.fgm, self.mixup_alpha = fgm, mixup_alpha
        self.accumulation_steps = max(1, int(accumulation_steps))
        self.max_norm, self.ema_model, self.scheduler, self.bucket = max_norm, ema_model, scheduler, bucket
        self.freeze_bn = freeze_bn
        self.model_kwargs = model_kwargs or {}
        from .amp import DeviceGradScaler, FusedEMA
        from .optim import FusedAdamW
        self.fused = isinstance(self.scaler, DeviceGradScaler)
        if self.fused:
            if not isinstance(optimizer, FusedAdamW):
                raise TypeError("a DeviceGradScaler unscales inside FusedAdamW.step: the optimizer must be a FusedAdamW")
            if ema_model is not None and not isinstance(ema_model, FusedEMA):
                raise TypeError("with a DeviceGradScaler, pass the AveragedModel as FusedEMA(averaged, model, decay)")
        self._zero()

    def _zero(self):
        if self.bucket is not None:
            self.bucket.zero()
        else:
            self.optimizer.zero_grad(set_to_none=True)

    def _forward_loss(self, x, y_a, y_b, lam, lengths=None):
        dev = x.device.type
        with torch.autocast(dev, dtype=self.autocast_dtype, enabled=self.autocast_dtype is not None):
            if lengths is None:
                feats, out = self.model(x, **self.model_kwargs)
            else:
                feats, out = self.model(x, lengths, mask_padding=True, **self.model_kwargs)
            loss = mixup_loss(self.loss_fn, out, feats, y_a, y_b, lam)
        return loss / self.accumulation_steps

    def __call__(self, micro_batches: Iterable, generator: Optional[torch.Generator] = None, lam: Optional[float] = None):
        """micro_batches: iterable of (x, y) or (x, y, lengths) of length accumulation_steps.  With lengths (per-utterance
        frame counts of the right-padded x, see ops.seqlens_tensor) the batch is mixed on its own frames (mixup_batch)
        and both the clean and FGM's adversarial pass call model(x, mixed_lengths, mask_padding=True).  Returns the mean
        (un-divided) clean loss of the micro-batches as a 0-d tensor (no host sync)."""
        self.model.train()
        if self.freeze_bn:
            freeze_batch_norm_stats(self.model)
        total = None
        for mb in micro_batches:
            x, y = mb[0], mb[1].view(-1).long()
            lengths = mb[2] if len(mb) > 2 else None
            if lengths is not None and x.is_cuda:
                from .ops import seqlens_tensor
                lengths = seqlens_tensor(lengths, x.size(0), x.size(1), x.device)
            if self.mixup_alpha > 0:
                mixed = mixup_batch(x, y, self.mixup_alpha, generator, lam, lengths)
                mx, y_a, y_b, lam_i = mixed[:4]
                lengths = mixed[4] if lengths is not None else None
            else:
                mx, y_a, y_b, lam_i = x, y, y, 1.0
            loss = self._forward_loss(mx, y_a, y_b, lam_i, lengths)
            self.scaler.scale(loss).backward()                                        # main.py:1077
            if self.fgm is not None:                                                  # main.py:1080-1098
                self.fgm.attack()
                adv = self._forward_loss(mx, y_a, y_b, lam_i, lengths)
                self.scaler.scale(adv).backward()
                self.fgm.restore()
            total = loss.detach() if total is None else total + loss.detach()
        if self.bucket is not None:
            self.bucket.all_reduce_mean()                                             # global gradient before the clip
        if self.fused:                                                                # main.py:1103-1113 on the device
            self.optimizer.step(scaler=self.scaler, max_norm=self.max_norm, ema=self.ema_model)
            self._zero()
            if self.scheduler is not None:
                self.scheduler.step()
            return total
        self.scaler.unscale_(self.optimizer)                                          # main.py:1103
        params = [p for g in self.optimizer.param_groups for p in g["params"] if p.grad is not None]
        torch.nn.utils.clip_grad_norm_(params, max_norm=self.max_norm)                # main.py:1104
        self.scaler.step(self.optimizer)
        self.scaler.update()
        self._zero()
        if self.ema_model is not None:
            self.ema_model.update_parameters(self.model)                              # main.py:1112-1113
        if self.scheduler is not None:
            self.scheduler.step()
        return total
