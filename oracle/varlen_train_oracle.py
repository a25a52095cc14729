"""CPU oracle for variable-length training.  TEST INFRASTRUCTURE ONLY (see bimamba_oracle.py for the rules).

The ground truth for a right-padded batch with per-utterance frame counts is every utterance run alone at its own
length (varlen_oracle.py for the scores); for training it is the fp64 loss summed over the utterances and its gradients,
parameter gradients summed over the utterances as a batch sums them.  A new file: the existing oracle files stay as
they are."""
from __future__ import annotations

from typing import Dict

import torch

from .bimamba_oracle import backend_ref, bimamba_ref, pn_bimamba_encoder_ref

Tensor = torch.Tensor


def varlen_loss_and_grads_ref(fn, params: Dict[str, Tensor], x: Tensor, lengths, loss_fn):
    """fp64 loss and gradients of a right-padded batch x (B, T, C) whose utterance b is x[b, :lengths[b]], each utterance
    run alone at its own length: fn(params, x_n) on every distinct length n (one batched call per length), loss_fn(out,
    idx, n) -> a scalar for the utterances idx, summed over the lengths.  Returns (loss, {name: gradient summed over the
    utterances}, dx (B, T, C) with zeros at padded frames).  The padded frames of x are never read."""
    lengths = [int(v) for v in lengths]
    ps = {k: v.detach().double().clone().requires_grad_(True) for k, v in params.items()}
    xs = {}
    total = x.new_zeros((), dtype=torch.float64)
    for n in sorted(set(lengths)):
        idx = [b for b, v in enumerate(lengths) if v == n]
        if n == 0:
            continue
        xn = x[idx, :n].detach().double().clone().requires_grad_(True)
        xs[n] = (idx, xn)
        total = total + loss_fn(fn(ps, xn), idx, n)
    total.backward()
    dx = torch.zeros(x.shape, dtype=torch.float64, device=x.device)
    for n, (idx, xn) in xs.items():
        dx[idx, :n] = xn.grad
    return total.detach(), {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in ps.items()}, dx


def block_fn(p, x):
    return bimamba_ref(p, x)


def layer_fn(p, x, eps: float = 1e-5):
    return pn_bimamba_encoder_ref(p, x, eps)


def backend_logits_fn(n_layers: int, eps: float = 1e-5):
    """fn for varlen_loss_and_grads_ref over a flat parameter dict with the backend's state_dict names."""
    def fn(p, x):
        layers = [{k.split(".", 2)[2]: v for k, v in p.items() if k.startswith(f"backbone_layers.{i}.")}
                  for i in range(n_layers)]
        head = {k: v for k, v in p.items() if not k.startswith("backbone_layers.")}
        return backend_ref(layers, head, x, eps)[1]
    return fn
