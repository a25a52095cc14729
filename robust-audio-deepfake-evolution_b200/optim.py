"""AdamW for the training step: every parameter tensor updated by ONE launch of this library's kernel.

Reference: `torch.optim.AdamW` as the reference builds it (src/main.py:453; decoupled weight decay, no amsgrad).  A
`torch.optim.Optimizer` subclass, so `param_groups`, `zero_grad`, LR schedulers (src/main.py:468-483) and
`clip_grad_norm_` (:1104) work as with the stock optimizer.  Hyper-parameters and the step counter live on the
device: the step is CUDA-graph capturable (`GraphedTrainStep`), and a scheduler's new `lr` reaches a captured graph
through `hyper` without re-capturing.

`step(scaler=..., max_norm=..., ema=...)` is the fp16 recipe's whole optimizer tail (src/main.py:1100-1117) on the
device: unscale, clip_grad_norm_, the skip of a step with an inf / NaN gradient, the scale update and the EMA update, in
four to six launches and no host read, so it captures too."""
from typing import List, Optional

import numpy as np
import torch

from . import _lib
from .amp import DeviceGradScaler, FusedEMA, new_amp_record, _TOTAL_NORM


class FusedAdamW(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1) or weight_decay < 0:
            raise ValueError("invalid AdamW hyper-parameters")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._groups = None      # per param group: device buffers and cached tables
        self._keep: List[torch.Tensor] = []            # pinned tables of recent eager steps (async copies in flight)
        self._keep_captured: List[torch.Tensor] = []   # pinned tables a captured graph reads at every replay: never freed
        self._ema_tables = None                          # (FusedEMA, per-group EMA tables, EMA-only launch of the rest)
        self.total_norm = None     # after a step with scaler / max_norm / ema: the pre-clip gradient norm (0-d, device)

    def _build(self):
        lib = _lib.load()
        chunk = lib.bimamba_adamw_chunk()
        self._groups = []
        # one table for every group (each group's launch reads its own slice), so the gradient statistics of the amp
        # step walk all groups in one launch over a block map with table-wide tensor indices
        counts = [sum(1 for p in group["params"] if p.requires_grad) for group in self.param_groups]
        devs = [p.device for group in self.param_groups for p in group["params"] if p.requires_grad]
        table_all = torch.zeros(max(sum(counts), 1) * 5, device=devs[0] if devs else torch.device("cuda"),
                                dtype=torch.int64)
        toff, bmaps = 0, []
        for group in self.param_groups:
            ps = [p for p in group["params"] if p.requires_grad]
            for p in ps:
                if p.dtype != torch.float32 or not p.is_cuda or not p.is_contiguous():
                    raise TypeError("FusedAdamW updates contiguous fp32 CUDA parameters (the master weights)")
            dev = ps[0].device if ps else torch.device("cuda")
            total = sum(p.numel() for p in ps)
            m = torch.zeros(total, device=dev, dtype=torch.float32)
            v = torch.zeros(total, device=dev, dtype=torch.float32)
            offs = np.cumsum([0] + [p.numel() for p in ps])
            for p, o in zip(ps, offs):                      # state views, for state_dict() / inspection
                self.state[p]["exp_avg"] = m[o:o + p.numel()].view_as(p)
                self.state[p]["exp_avg_sq"] = v[o:o + p.numel()].view_as(p)
            bmap = np.array([(i, c) for i, p in enumerate(ps) for c in range((p.numel() + chunk - 1) // chunk)],
                            dtype=np.int32).reshape(-1, 2)
            bmaps.append(bmap + np.array([toff, 0], dtype=np.int32))
            self._groups.append(dict(
                params=ps, m=m, v=v, offs=offs, nblocks=int(bmap.shape[0]),
                bmap=torch.from_numpy(bmap).to(dev), hyper=torch.zeros(5, device=dev), hyper_host=None,
                state=torch.zeros(1, device=dev), table=table_all[5 * toff:5 * (toff + len(ps))], gptrs=None))
            toff += len(ps)
        bmap_all = np.concatenate(bmaps) if bmaps else np.zeros((0, 2), dtype=np.int32)
        self._all = dict(table=table_all, nblocks=int(bmap_all.shape[0]),
                         bmap=torch.from_numpy(np.ascontiguousarray(bmap_all)).to(table_all.device),
                         partials=torch.zeros(max(int(bmap_all.shape[0]), 1), device=table_all.device,
                                              dtype=torch.float64),
                         amp=new_amp_record(table_all.device))    # the record of a step without a scaler: scale 1

    def _sync_hyper(self, group, g):
        h = (float(group["lr"]), float(group["betas"][0]), float(group["betas"][1]), float(group["eps"]),
             float(group["weight_decay"]))
        if h != g["hyper_host"]:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("FusedAdamW: hyper-parameters changed inside a CUDA-graph capture; call "
                                   "sync_hyper() outside the capture (the captured step reads them from the device)")
            g["hyper"].copy_(torch.tensor(h, dtype=torch.float32))
            g["hyper_host"] = h

    def sync_hyper(self):
        """Push param_groups' lr / betas / eps / weight_decay to the device (call after a scheduler step when the
        optimizer step itself is replayed from a CUDA graph)."""
        if self._groups is None:
            self._build()
        for group, g in zip(self.param_groups, self._groups):
            self._sync_hyper(group, g)

    # ---- checkpoint / resume: torch.optim.AdamW's layout (state[p] = {step, exp_avg, exp_avg_sq}) ------------------
    def _export_state(self):
        """Refresh `self.state` so that `state_dict()` holds the live moments and the step counter."""
        if self._groups is None:
            return
        for g in self._groups:
            step = g["state"].detach().clone().reshape(())
            for p, o in zip(g["params"], g["offs"]):
                n = p.numel()
                self.state[p] = {"step": step, "exp_avg": g["m"][o:o + n].view_as(p), "exp_avg_sq": g["v"][o:o + n].view_as(p)}

    def state_dict(self):
        self._export_state()
        return super().state_dict()

    def load_state_dict(self, state_dict):
        """Loads a FusedAdamW or torch.optim.AdamW state_dict: moments are copied into the flat buffers the kernel
        reads and the step counter is restored (bias correction continues where it stopped).  An empty state resets
        the optimizer."""
        if self._groups is None:
            self._build()                                   # before the load: _build() re-points state at its own (zero) buffers
        super().load_state_dict(state_dict)
        for g in self._groups:
            g["hyper_host"] = None                          # param_groups may carry new hyper-parameters
            step = None
            for p, o in zip(g["params"], g["offs"]):
                n = p.numel()
                st = self.state.get(p, None)
                if st and "exp_avg" in st:
                    g["m"][o:o + n].copy_(st["exp_avg"].reshape(-1).to(torch.float32))
                    g["v"][o:o + n].copy_(st["exp_avg_sq"].reshape(-1).to(torch.float32))
                    if "step" in st:
                        step = float(st["step"]) if step is None else max(step, float(st["step"]))
                else:
                    g["m"][o:o + n].zero_()
                    g["v"][o:o + n].zero_()
            g["state"].fill_(0.0 if step is None else step)
        for group, g in zip(self.param_groups, self._groups):
            self._sync_hyper(group, g)
        self._export_state()

    def _upload(self, arr: np.ndarray, dst: torch.Tensor) -> None:
        """Host table -> device through pinned memory (legal inside a capture, which then replays the copy)."""
        host = torch.from_numpy(np.ascontiguousarray(arr).reshape(-1)).pin_memory()
        if torch.cuda.is_current_stream_capturing():
            self._keep_captured.append(host)
        else:
            self._keep.append(host)
            if len(self._keep) > 64:
                del self._keep[:32]
        dst.copy_(host, non_blocking=True)

    @staticmethod
    def _grad_ptrs(g):
        for p in g["params"]:
            if p.grad is not None and (p.grad.dtype != torch.float32 or not p.grad.is_contiguous()):
                p.grad = p.grad.to(torch.float32).contiguous()
        return tuple(0 if p.grad is None else p.grad.data_ptr() for p in g["params"])

    def _write_table(self, g, gptrs):
        # parameters without a gradient are skipped, as torch.optim.AdamW does (src/main.py:453 hands the optimizer
        # the whole model, including tensors that never receive one): their table entry has n = 0
        ps = g["params"]
        if gptrs != g["gptrs"]:       # gradients moved (first step, or freshly allocated by autograd)
            tab = np.empty((len(ps), 5), dtype=np.int64)
            for i, (p, o) in enumerate(zip(ps, g["offs"])):
                tab[i] = (p.data_ptr(), gptrs[i], g["m"].data_ptr() + 4 * int(o), g["v"].data_ptr() + 4 * int(o),
                          p.numel() if gptrs[i] else 0)
            self._upload(tab, g["table"])
            g["gptrs"] = gptrs

    @torch.no_grad()
    def step(self, closure=None, *, scaler: Optional[DeviceGradScaler] = None, max_norm: Optional[float] = None,
             ema: Optional[FusedEMA] = None):
        """One AdamW step.  With any of the keywords, the fp16 recipe's whole tail on the device; for the same
        gradients it equals  scaler.unscale_(opt); clip_grad_norm_(params, max_norm); scaler.step(opt);
        scaler.update(); averaged.update_parameters(model)  with torch.optim.AdamW:
          * scaler (DeviceGradScaler): the gradients are unscaled by the scale the loss was multiplied with; a step
            whose gradient holds an inf or NaN leaves parameters, moments and the step count untouched; the scale is
            then updated as GradScaler.update does.  A disabled scaler is ignored;
          * max_norm: the unscaled gradient is clipped to this global 2-norm over every group;
          * ema (FusedEMA): the average moves toward the model afterwards, also on a skipped step.
        A step with a non-finite gradient is skipped whenever one of the keywords is given (without a scaler,
        clip_grad_norm_ would have scaled every gradient by NaN).  The pre-clip norm is left in `self.total_norm`
        (a 0-d device tensor, clip_grad_norm_'s return value).  `.grad` is NOT unscaled or clipped in place: after the
        step it still holds the scaled gradient (zero it before the next backward, as the reference loop does)."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if self._groups is None:
            self._build()
        if scaler is not None and not scaler.is_enabled():
            scaler = None
        if scaler is not None or max_norm is not None or ema is not None:
            self._amp_step(scaler, max_norm, ema)
            return loss
        lib = _lib.load()
        stream = torch.cuda.current_stream().cuda_stream
        for group, g in zip(self.param_groups, self._groups):
            ps = g["params"]
            if not ps:
                continue
            self._sync_hyper(group, g)
            gptrs = self._grad_ptrs(g)
            if not any(gptrs):
                continue
            self._write_table(g, gptrs)
            _lib.check(lib.bimamba_adamw_step(g["table"].data_ptr(), g["bmap"].data_ptr(), g["nblocks"],
                                              g["hyper"].data_ptr(), g["state"].data_ptr(), stream),
                       "bimamba_adamw_step")
            _lib.launch_count += 1    # tick + update
        return loss

    def _ema_for(self, ema: FusedEMA):
        """Device tables of `ema` (built once per FusedEMA): per group, entry i = the average of the group's parameter
        i; and the EMA-only launch over the model's parameters no group holds."""
        if self._ema_tables is not None and self._ema_tables[0] is ema:
            return self._ema_tables
        avg_of = {id(p): a for p, a in ema.pairs}
        dev = self._all["table"].device
        per_group, held = [], set()
        for g in self._groups:
            tab = np.zeros((max(len(g["params"]), 1), 2), dtype=np.int64)
            for i, p in enumerate(g["params"]):
                held.add(id(p))
                a = avg_of.get(id(p))
                if a is not None:
                    tab[i] = (a.data_ptr(), a.numel())
            dst = torch.empty(tab.size, dtype=torch.int64, device=dev)
            self._upload(tab, dst)
            per_group.append(dst)
        rest = [(p, a) for p, a in ema.pairs if id(p) not in held]
        rest_launch = None
        if rest:
            chunk = _lib.load().bimamba_adamw_chunk()
            tab = np.array([(p.data_ptr(), 0, 0, 0, 0) for p, _ in rest], dtype=np.int64)
            etab = np.array([(a.data_ptr(), a.numel()) for _, a in rest], dtype=np.int64)
            bmap = np.array([(i, c) for i, (p, _) in enumerate(rest) for c in range((p.numel() + chunk - 1) // chunk)],
                            dtype=np.int32).reshape(-1, 2)
            bufs = [torch.empty(x.size, dtype=torch.int64 if x.dtype == np.int64 else torch.int32, device=dev)
                    for x in (tab, etab, bmap)]
            for x, d in zip((tab, etab, bmap), bufs):
                self._upload(x, d)
            rest_launch = (*bufs, int(bmap.shape[0]))
        self._ema_tables = (ema, per_group, rest_launch)
        return self._ema_tables

    def _amp_step(self, scaler, max_norm, ema):
        if max_norm is not None and not max_norm > 0:
            raise ValueError("max_norm must be positive (None: no clipping)")
        if ema is not None and not isinstance(ema, FusedEMA):
            raise TypeError("ema must be a FusedEMA (pairs the AveragedModel with the trained model)")
        lib = _lib.load()
        stream = torch.cuda.current_stream().cuda_stream
        a = self._all
        rec = scaler._lazy_init(a["table"].device) if scaler is not None else a["amp"]
        gptrs = [self._grad_ptrs(g) for g in self._groups]
        for g, gp in zip(self._groups, gptrs):
            if g["params"]:               # every group, also one without gradients: the statistics read every table
                self._write_table(g, gp)
        _lib.check(lib.bimamba_amp_grad_stats(a["table"].data_ptr(), a["bmap"].data_ptr(), a["nblocks"],
                                              float(max_norm or 0.0), a["partials"].data_ptr(), rec.data_ptr(), stream),
                   "bimamba_amp_grad_stats")
        _lib.launch_count += 1    # partial sums + final sum
        n_av, w, etabs, rest = None, 0.0, None, None
        if ema is not None:
            _, etabs, rest = self._ema_for(ema)
            n_av, w = ema.n_averaged.data_ptr(), ema.weight
        for i, (group, g) in enumerate(zip(self.param_groups, self._groups)):
            if not g["params"]:
                continue
            self._sync_hyper(group, g)
            et = etabs[i].data_ptr() if etabs is not None else None
            if any(gptrs[i]):
                _lib.check(lib.bimamba_adamw_amp_step(g["table"].data_ptr(), g["bmap"].data_ptr(), g["nblocks"],
                                                      g["hyper"].data_ptr(), g["state"].data_ptr(), rec.data_ptr(),
                                                      et, n_av, w, stream), "bimamba_adamw_amp_step")
                _lib.launch_count += 1    # tick + update
            elif et is not None:          # no gradient in the group: AdamW skips it, the average still moves
                _lib.check(lib.bimamba_adamw_amp_step(g["table"].data_ptr(), g["bmap"].data_ptr(), g["nblocks"],
                                                      None, None, None, et, n_av, w, stream), "bimamba_adamw_amp_step")
        if rest is not None:
            tab, etab, bmap, nb = rest
            _lib.check(lib.bimamba_adamw_amp_step(tab.data_ptr(), bmap.data_ptr(), nb, None, None, None,
                                                  etab.data_ptr(), n_av, w, stream), "bimamba_adamw_amp_step")
        if ema is not None and ema.buffers:
            torch._foreach_copy_([b for _, b in ema.buffers], [b for b, _ in ema.buffers])
        if scaler is not None or ema is not None:
            _lib.check(lib.bimamba_amp_update(rec.data_ptr() if scaler is not None else None,
                                              float(scaler._growth_factor) if scaler is not None else 2.0,
                                              float(scaler._backoff_factor) if scaler is not None else 0.5,
                                              int(scaler._growth_interval) if scaler is not None else 1, n_av, stream),
                       "bimamba_amp_update")
        self.total_norm = rec.view(torch.float32)[_TOTAL_NORM]
