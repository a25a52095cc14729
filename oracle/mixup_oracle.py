"""CPU oracle for Mixup of a right-padded batch.  TEST INFRASTRUCTURE ONLY (see bimamba_oracle.py for the rules).

The contract of bimamba_mixup_frames restated per utterance pair: mixed utterance b is lam * clip b + (1 - lam) * clip
p = perm[b], each clip zero-padded past its own length n (clamped to [0, T]), over max(n_b, n_p) frames, and exactly zero
after them.  A padded frame of a source is never read, so NaN or huge padding reaches no output.  A new file: the existing
oracle files stay as they are."""
from __future__ import annotations

import torch

Tensor = torch.Tensor


def mixup_ref(x: Tensor, perm, lam: float, lengths=None, *, exact: bool = True):
    """-> (mixed (B, T, ...), mixed lengths (B,) int64).  lengths None: every frame is valid.

    exact=True: fp64 ground truth (x converted to float64, one product and one sum per frame, no rounding of note).
    exact=False: the torch expression in x's dtype, the bits the kernel must give: a = lam * x_b and c = (1.0 - lam) *
    x_p each rounded to x's dtype, then a + c rounded, the terms taken only over their own clip's frames."""
    B, T = x.shape[0], x.shape[1]
    perm = [int(v) for v in torch.as_tensor(perm).tolist()]
    n = [T] * B if lengths is None else [min(max(int(v), 0), T) for v in torch.as_tensor(lengths).tolist()]
    xs = x.double() if exact else x
    out = torch.zeros_like(xs)
    m = torch.zeros(B, dtype=torch.int64)
    for b in range(B):
        p = perm[b]
        nb, np_ = n[b], n[p]
        m[b] = max(nb, np_)
        a = torch.zeros_like(xs[b])
        c = torch.zeros_like(xs[b])
        a[:nb] = lam * xs[b, :nb]
        c[:np_] = (1.0 - lam) * xs[p, :np_]
        out[b, :m[b]] = (a + c)[:m[b]]
    return out, m
