"""CPU oracle for variable-length scoring.  TEST INFRASTRUCTURE ONLY (see bimamba_oracle.py for the rules).

The reference scores every clip on its own (its loaders crop or tile to one length, src/data_utils.py:107-127), so the
ground truth for a right-padded batch with per-utterance frame counts is bimamba_oracle.backend_ref run on each
utterance at its own length."""
from __future__ import annotations

from typing import Dict

import torch

from .bimamba_oracle import backend_ref

Tensor = torch.Tensor


def backend_varlen_ref(layers, head: Dict[str, Tensor], x: Tensor, lengths, eps: float = 1e-5):
    """Scores of a right-padded batch x (B, T, d_model) whose utterance b is x[b, :lengths[b]]: backend_ref run on every
    utterance at its own length (one batched call per distinct length).  Returns (features (B, d_model), logits (B, 2))."""
    lengths = [int(v) for v in lengths]
    feats = x.new_zeros((x.shape[0], x.shape[-1]))
    logits = x.new_zeros((x.shape[0], head["classifier.weight"].shape[0]))
    for n in sorted(set(lengths)):
        idx = torch.tensor([b for b, v in enumerate(lengths) if v == n], device=x.device)
        feats[idx], logits[idx] = backend_ref(layers, head, x[idx, :n], eps)
    return feats, logits
