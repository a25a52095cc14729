"""Drop-in `Mamba` with the constructor / forward / state_dict surface of
`mamba_ssm.modules.mamba_simple.Mamba`, the class the reference imports at
src/models/DualStreamSEMamba.py:43 and builds as `Mamba(d_model, n_state)` at :455.

Parameter names and shapes equal the reference's in-repo block
(src/models/modules/mamba_block.py:22-39):
  in_proj.weight (2*d_inner, d_model), conv1d.weight (d_inner, 1, d_conv), conv1d.bias (d_inner),
  x_proj.weight (dt_rank + 2*d_state, d_inner), dt_proj.weight (d_inner, dt_rank),
  dt_proj.bias (d_inner), A_log (d_inner, d_state), D (d_inner), out_proj.weight (d_model, d_inner)
so reference checkpoints load unchanged (`backbone_layers.{i}.mamba.*`).
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .ops import bimamba_inner_fn


class Mamba(nn.Module):
    def __init__(self, d_model, d_state=16, d_conv=4, expand=2, dt_rank="auto", dt_min=0.001, dt_max=0.1,
                 dt_init="random", dt_scale=1.0, dt_init_floor=1e-4, conv_bias=True, bias=False,
                 use_fast_path=True, layer_idx=None, device=None, dtype=None):
        factory = {"device": device, "dtype": dtype}
        super().__init__()
        if bias:
            raise NotImplementedError("bias=True is not used by the reference path (mamba_block.py:22,39)")
        if not conv_bias:
            raise NotImplementedError("conv_bias=False is not used by the reference path (mamba_block.py:27)")
        self.d_model = d_model
        self.d_state = d_state
        self.d_conv = d_conv
        self.expand = expand
        self.d_inner = int(self.expand * self.d_model)
        self.dt_rank = math.ceil(self.d_model / 16) if dt_rank == "auto" else dt_rank   # mamba_block.py:20
        self.use_fast_path = use_fast_path
        self.layer_idx = layer_idx

        self.in_proj = nn.Linear(self.d_model, self.d_inner * 2, bias=False, **factory)
        self.conv1d = nn.Conv1d(self.d_inner, self.d_inner, kernel_size=d_conv, groups=self.d_inner,
                                padding=d_conv - 1, bias=True, **factory)
        self.activation = "silu"
        self.act = nn.SiLU()
        self.x_proj = nn.Linear(self.d_inner, self.dt_rank + self.d_state * 2, bias=False, **factory)
        self.dt_proj = nn.Linear(self.dt_rank, self.d_inner, bias=True, **factory)

        # dt_proj init as in the upstream package: weight ~ U(+-dt_rank^-0.5 * dt_scale), bias = softplus^-1(dt),
        # dt ~ logU[dt_min, dt_max] clamped at dt_init_floor (SURVEY row a13).
        dt_init_std = self.dt_rank ** -0.5 * dt_scale
        if dt_init == "constant":
            nn.init.constant_(self.dt_proj.weight, dt_init_std)
        elif dt_init == "random":
            nn.init.uniform_(self.dt_proj.weight, -dt_init_std, dt_init_std)
        else:
            raise NotImplementedError
        dt = torch.exp(torch.rand(self.d_inner, **factory) * (math.log(dt_max) - math.log(dt_min))
                       + math.log(dt_min)).clamp(min=dt_init_floor)
        inv_dt = dt + torch.log(-torch.expm1(-dt))
        with torch.no_grad():
            self.dt_proj.bias.copy_(inv_dt)
        self.dt_proj.bias._no_reinit = True

        # A_log = log(1..N) per row, D = 1 (mamba_block.py:36-38)
        A = torch.arange(1, self.d_state + 1, dtype=torch.float32, device=device).repeat(self.d_inner, 1)
        self.A_log = nn.Parameter(torch.log(A))
        self.A_log._no_weight_decay = True
        self.D = nn.Parameter(torch.ones(self.d_inner, device=device))
        self.D._no_weight_decay = True
        self.out_proj = nn.Linear(self.d_inner, self.d_model, bias=False, **factory)

    def _run(self, hidden_states, bidirectional, lengths=None, mask_padding=False):
        return bimamba_inner_fn(
            hidden_states, self.in_proj.weight, self.conv1d.weight, self.conv1d.bias, self.x_proj.weight,
            self.dt_proj.weight, self.dt_proj.bias, self.A_log, self.D, self.out_proj.weight,
            bidirectional=bidirectional, lengths=lengths, mask_padding=mask_padding)

    def forward(self, hidden_states, inference_params=None):
        """hidden_states (B, L, d_model) -> (B, L, d_model); one (causal) direction, as upstream."""
        if inference_params is not None:
            raise NotImplementedError("step-wise decoding is not part of the reference's path")
        return self._run(hidden_states, False)

    def forward_bidirectional(self, hidden_states, lengths=None, *, mask_padding=False):
        """M(x) + flip(M(flip(x))) with these weights in one fused pass
        (src/models/DualStreamSEMamba.py:473-481).

        lengths (B,) (list, CPU or CUDA tensor; scoring only): utterance b is frames 0 .. lengths[b]-1 of the
        right-padded batch, and its flip is taken over those frames alone, so each valid output frame equals that of
        the utterance run by itself.  Output frames at padded positions are unspecified.
        mask_padding=True (with lengths) trains on the padded batch: padded input frames are replaced by zeros, padded
        output frames are zero, and the loss and gradients are those of each utterance run alone (bimamba_inner_fn)."""
        return self._run(hidden_states, True, lengths, mask_padding)
