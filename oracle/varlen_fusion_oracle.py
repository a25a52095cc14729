"""CPU oracle for variable-length DualStreamFusion.  TEST INFRASTRUCTURE ONLY (see bimamba_oracle.py for the rules).

The reference fuses every clip on its own: its WavLM stream has n1 frames and its SincNet stream n2, and
DualStreamSEMamba.py:601-626 interpolates the SincNet branch from n2 onto n1 frames (no interpolation when n1 == n2,
nearest when n1 / n2 > 4.0, else linear with align_corners=False).  The ground truth for a right-padded pair of streams
with per-utterance frame counts is therefore fusion_ref's math run on every utterance alone, in fp64.

One exception to "fp64 everywhere": F.interpolate picks its source frames and weights in the tensor's own precision,
and the reference runs it on fp32 (or autocast bf16 / fp16, whose index arithmetic is fp32).  In fp64 the nearest rule
picks a different source frame for 940 (n2, n1) pairs with n2 < 80, n1 < 520, among them 76 pairs that real clips of
0.5-12 s produce.  So interp_index_fp32 restates ATen's fp32 index rule explicitly and the fp64 math takes its indices
and weights from there; F.interpolate is never called on fp64 tensors here."""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch
import torch.nn.functional as F

from .bimamba_oracle import backend_ref

Tensor = torch.Tensor


def interp_mode(n2: int, n1: int) -> str:
    """The reference's rule (DualStreamSEMamba.py:601-626) in integers: n1 / n2 > 4.0 <=> n1 > 4 n2."""
    return "copy" if n1 == n2 else ("nearest" if n1 > 4 * n2 else "linear")


def interp_index_fp32(n2: int, n1: int):
    """Source frames and weights with which F.interpolate maps n2 frames onto n1 in fp32 (ATen, CPU and CUDA): returns
    (mode, i0, i1, w0, w1), output frame t = w0[t] * x[i0[t]] + w1[t] * x[i1[t]] (int64 indices, float32 weights).
    scale = float32(n2) / float32(n1).  nearest: i0 = min(floor(float32(t) * scale), n2 - 1).  linear (align_corners
    False): src = max(scale * (t + 0.5) - 0.5, 0) rounded ONCE to float32 (ATen's compiled kernels fuse the
    multiply-subtract; rounding the product first disagrees with F.interpolate on 10 170 (n2, n1) pairs of the range
    tested), i0 = floor(src), i1 = i0 + (i0 < n2 - 1), w1 = src - i0, w0 = 1 - w1 in float32."""
    mode = interp_mode(n2, n1)
    t = np.arange(n1)
    if mode == "copy" or mode == "nearest":
        if mode == "copy":
            i0 = t.astype(np.int64)
        else:
            scale = np.float32(n2) / np.float32(n1)
            i0 = np.minimum(np.floor(t.astype(np.float32) * scale), n2 - 1).astype(np.int64)
        return mode, i0, i0.copy(), np.ones(n1, np.float32), np.zeros(n1, np.float32)
    scale = np.float32(n2) / np.float32(n1)
    # fp32 x fp32 is exact in fp64 and so is the subtraction of 0.5 at these sizes: one rounding, as a fused multiply-add
    src = (np.float64(scale) * (t.astype(np.float64) + 0.5) - 0.5).astype(np.float32)
    src = np.maximum(src, np.float32(0))
    i0 = np.floor(src).astype(np.int64)
    i1 = i0 + (i0 < n2 - 1)
    w1 = (src - i0.astype(np.float32)).astype(np.float32)
    w0 = (np.float32(1) - w1).astype(np.float32)
    return mode, i0, i1, w0, w1


def interp_ref(x: Tensor, n1: int) -> Tensor:
    """x (B, n2, C) -> (B, n1, C) with interp_index_fp32's indices and weights, arithmetic in x's dtype."""
    _, i0, i1, w0, w1 = interp_index_fp32(x.shape[1], n1)
    w0 = torch.from_numpy(w0).to(x.dtype).view(1, n1, 1)
    w1 = torch.from_numpy(w1).to(x.dtype).view(1, n1, 1)
    return w0 * x[:, torch.from_numpy(i0)] + w1 * x[:, torch.from_numpy(i1)]


def fusion_one_ref(p: Dict[str, Tensor], f_wavlm: Tensor, f_sinc: Tensor, eps: float = 1e-5) -> Tensor:
    """fusion_ref (bimamba_oracle.py) for utterances that share (n1, n2) = (f_wavlm.shape[1], f_sinc.shape[1]), with the
    interpolation taken from interp_index_fp32."""
    fw = F.layer_norm(f_wavlm, (f_wavlm.shape[-1],), p["ln_wavlm.weight"], p["ln_wavlm.bias"], eps)     # :591
    fs = F.layer_norm(f_sinc, (f_sinc.shape[-1],), p["ln_sinc.weight"], p["ln_sinc.bias"], eps)         # :592
    fw = fw @ p["wavlm_proj.weight"].t() + p["wavlm_proj.bias"]                                         # :595
    fs = fs @ p["sinc_proj.weight"].t() + p["sinc_proj.bias"]                                           # :596
    fs = interp_ref(fs, fw.shape[1])                                                                    # :601-626
    fused = torch.cat([fw, fs], dim=-1) @ p["fusion_proj.weight"].t() + p["fusion_proj.bias"]           # :629-630
    se = fused.mean(dim=1)                                                                              # :524-526
    se = torch.sigmoid(torch.relu(se @ p["se_layer.fc.0.weight"].t()) @ p["se_layer.fc.2.weight"].t())  # :527
    fused = fused * se.unsqueeze(1)                                                                     # :528
    return F.layer_norm(fused, (fused.shape[-1],), p["norm.weight"], p["norm.bias"], eps)               # :636


def _groups(lengths, sinc_lengths):
    pairs = [(int(a), int(b)) for a, b in zip(lengths, sinc_lengths)]
    for pr in sorted(set(pairs)):
        yield pr, [i for i, q in enumerate(pairs) if q == pr]


def fusion_varlen_ref(p: Dict[str, Tensor], f_wavlm: Tensor, f_sinc: Tensor, lengths, sinc_lengths,
                      eps: float = 1e-5) -> Tensor:
    """Right-padded streams f_wavlm (B, T1, .), f_sinc (B, T2, .) whose utterance b is f_wavlm[b, :lengths[b]] with
    f_sinc[b, :sinc_lengths[b]]: fusion_one_ref on every utterance alone (one call per distinct pair).  (B, T1, out_dim)
    with zeros at padded frames; the padded input frames are never read."""
    out = f_wavlm.new_zeros((f_wavlm.shape[0], f_wavlm.shape[1], p["norm.weight"].shape[0]))
    for (n1, n2), idx in _groups(lengths, sinc_lengths):
        out[idx, :n1] = fusion_one_ref(p, f_wavlm[idx, :n1], f_sinc[idx, :n2], eps)
    return out


def fusion_loss_and_grads_ref(fn, params: Dict[str, Tensor], f_wavlm: Tensor, f_sinc: Tensor, lengths, sinc_lengths,
                              loss_fn):
    """Two-stream varlen_loss_and_grads_ref (varlen_train_oracle.py): fp64 loss summed over the utterances, each run alone
    as fn(params, fw_n, fs_n) and scored by loss_fn(out, idx, n1, n2), one call per distinct (n1, n2).  Returns (loss,
    {name: gradient summed over the utterances}, d f_wavlm, d f_sinc) with zeros at padded frames."""
    ps = {k: v.detach().double().clone().requires_grad_(True) for k, v in params.items()}
    leaves = []
    total = torch.zeros((), dtype=torch.float64)
    for (n1, n2), idx in _groups(lengths, sinc_lengths):
        fw = f_wavlm[idx, :n1].detach().double().cpu().clone().requires_grad_(True)
        fs = f_sinc[idx, :n2].detach().double().cpu().clone().requires_grad_(True)
        leaves.append((idx, n1, n2, fw, fs))
        total = total + loss_fn(fn(ps, fw, fs), idx, n1, n2)
    total.backward()
    dfw = torch.zeros(f_wavlm.shape, dtype=torch.float64)
    dfs = torch.zeros(f_sinc.shape, dtype=torch.float64)
    for idx, n1, n2, fw, fs in leaves:
        dfw[idx, :n1] = fw.grad
        dfs[idx, :n2] = fs.grad
    return total.detach(), {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in ps.items()}, dfw, dfs


def split_tail_params(p: Dict[str, Tensor], n_layers: int):
    """A flat dict with the model's state_dict names (fusion.*, backbone_layers.i.*, norm_f / attention_pool /
    classifier) -> (fusion params, [layer params], head params)."""
    fus = {k[len("fusion."):]: v for k, v in p.items() if k.startswith("fusion.")}
    layers = [{k.split(".", 2)[2]: v for k, v in p.items() if k.startswith(f"backbone_layers.{i}.")}
              for i in range(n_layers)]
    head = {k: v for k, v in p.items() if not k.startswith(("fusion.", "backbone_layers."))}
    return fus, layers, head


def tail_fn(n_layers: int, eps: float = 1e-5):
    """fn(p, fw, fs) -> (features, logits): the model tail, fusion -> backend_ref (n_layers encoder layers, norm_f,
    attention pooling, classifier), for utterances sharing one (n1, n2)."""
    def fn(p, fw, fs):
        fus, layers, head = split_tail_params(p, n_layers)
        return backend_ref(layers, head, fusion_one_ref(fus, fw, fs, eps), eps)
    return fn


def tail_varlen_ref(p: Dict[str, Tensor], n_layers: int, f_wavlm: Tensor, f_sinc: Tensor, lengths, sinc_lengths,
                    eps: float = 1e-5):
    """Scores of the model tail on right-padded streams, every utterance alone: (features (B, d), logits (B, 2))."""
    fn = tail_fn(n_layers, eps)
    feats = logits = None
    for (n1, n2), idx in _groups(lengths, sinc_lengths):
        f, lg = fn(p, f_wavlm[idx, :n1], f_sinc[idx, :n2])
        if feats is None:
            feats = f.new_zeros((f_wavlm.shape[0], f.shape[1]))
            logits = lg.new_zeros((f_wavlm.shape[0], lg.shape[1]))
        feats[idx], logits[idx] = f, lg
    return feats, logits
