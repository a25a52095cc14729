"""`PN_BiMambas_Encoder` and the 4-layer backend with the reference's attribute names
(src/models/DualStreamSEMamba.py:445-486, :697-710, :755-767), on top of the fused Bi-Mamba block."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .mamba_simple import Mamba
from .ops import (_check_mask_padding, _forward_only, _wants_grad, encoder_layer_native, feed_forward_fn, head_fwd,
                  head_pool_fn, layer_norm_fn, mask_frames, native_layer_ok, seqlens_tensor)


class PN_BiMambas_Encoder(nn.Module):
    """Pre-norm Bi-Mamba layer.  Same constructor, attributes (`mamba`, `norm1`, `norm2`,
    `feed_forward`) and state_dict keys as DualStreamSEMamba.py:451-465."""

    def __init__(self, d_model, n_state):
        super().__init__()
        self.d_model = d_model
        self.mamba = Mamba(d_model, n_state)
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)
        self.feed_forward = nn.Sequential(
            nn.Linear(d_model, d_model * 4),
            nn.GELU(),
            nn.Linear(d_model * 4, d_model),
        )

    def forward(self, x, lengths=None, *, mask_padding=False):
        """x (B, T, d_model) -> (B, T, d_model).  lengths (B,) (list, CPU or CUDA tensor): per-utterance frame counts of a
        right-padded x; valid output frames equal the utterance's own, padded ones are unspecified.  Without
        mask_padding that is scoring only.  mask_padding=True (training): the padded input frames are replaced by zeros
        and the padded output frames are exactly zero, in the forward and (their gradients) in the backward, so the loss
        and every gradient are those of each utterance run alone whatever the padding holds."""
        _check_mask_padding(lengths, mask_padding)
        seqlens = None
        if lengths is not None:
            seqlens = seqlens_tensor(lengths, x.shape[0], x.shape[1], x.device)
            if not mask_padding:
                _forward_only(seqlens, x, *self.parameters())
        if native_layer_ok(x, self):
            # eager mode: the whole layer in one native call each way (same kernels, same order, same bits; a captured
            # step keeps the sequenced Functions below, which overlap the weight-gradient products on a second stream)
            return encoder_layer_native(x, self, seqlens, mask_padding)
        if mask_padding:
            x = mask_frames(x, seqlens)
        # :471-472; the residual branch leaves the LayerNorm Function as its second output, so its gradient is added to dx
        # inside the LayerNorm backward kernel (no separate autograd add)
        x_norm, residual = layer_norm_fn(x, self.norm1.weight, self.norm1.bias, self.norm1.eps, with_residual=True)
        mamba_out = self.mamba.forward_bidirectional(x_norm, seqlens, mask_padding=mask_padding)    # :473-481 in one fused pass
        mamba_out = layer_norm_fn(mamba_out, self.norm2.weight, self.norm2.bias, self.norm2.eps)    # :482
        if isinstance(self.feed_forward[1], nn.GELU) and self.feed_forward[1].approximate == "none":
            l1, l2 = self.feed_forward[0], self.feed_forward[2]
            out = feed_forward_fn(mamba_out, l1.weight, l1.bias, l2.weight, l2.bias, residual=residual)   # :483-485
        else:
            out = self.feed_forward(mamba_out) + residual
        # the feed-forward and the norms make padded rows non-zero: without this mask a loss that touches them would
        # reach the feed-forward's weight gradients
        return mask_frames(out, seqlens) if mask_padding else out


class BiMambaBackend(nn.Module):
    """The part of the reference `Model` after fusion (DualStreamSEMamba.py:697-710, :755-767):
    `backbone_layers`, `norm_f`, `attention_pool`, `dropout`, `classifier` with the same names."""

    def __init__(self, emb_size=144, num_encoders=4, d_state=16):
        super().__init__()
        self.backbone_layers = nn.ModuleList(
            [PN_BiMambas_Encoder(d_model=emb_size, n_state=d_state) for _ in range(num_encoders)])
        self.norm_f = nn.LayerNorm(emb_size)
        self.attention_pool = nn.Linear(emb_size, 1)
        self.dropout = nn.Dropout(0.1)
        self.classifier = nn.Linear(emb_size, 2)

    def forward_features(self, f_fused, lengths=None, *, mask_padding=False):
        """lengths (B,) (list, CPU or CUDA tensor): per-utterance frame counts of the right-padded f_fused.  Output
        frames at padded positions are unspecified; with mask_padding=True (training, see PN_BiMambas_Encoder.forward)
        they are zero."""
        _check_mask_padding(lengths, mask_padding)
        seqlens = seqlens_tensor(lengths, f_fused.shape[0], f_fused.shape[1], f_fused.device)
        for layer in self.backbone_layers:
            f_fused = layer(f_fused, seqlens, mask_padding=mask_padding)
        return f_fused

    def forward(self, f_fused, lengths=None, *, mask_padding=False):
        """f_fused (B, T, emb) -> (features, logits).  lengths (B,): see forward_features; every utterance is scored
        as if it ran alone at its own length (net(x, lengths) with x padded on the right).  mask_padding=True trains on
        such a batch: the loss and every gradient are those of each utterance run alone, summed over utterances."""
        _check_mask_padding(lengths, mask_padding)
        seqlens = seqlens_tensor(lengths, f_fused.shape[0], f_fused.shape[1], f_fused.device)
        return backend_head(self, self.forward_features(f_fused, seqlens, mask_padding=mask_padding), seqlens,
                            mask_padding=mask_padding)


def backend_head(m, f_fused, lengths=None, *, mask_padding=False):
    """norm_f -> attention pooling -> dropout -> classifier on a module that carries the reference's attribute names
    (`norm_f`, `attention_pool`, `dropout`, `classifier`; DualStreamSEMamba.py:759-767).  Returns (features, logits).
    lengths (B,) (list, CPU or CUDA tensor): norm, softmax and pooling over each utterance's first lengths[b] frames
    only; scoring only unless mask_padding=True, which also takes the gradient over those frames (zero at the others)."""
    _check_mask_padding(lengths, mask_padding)
    if lengths is not None:
        return _backend_head_varlen(m, f_fused, lengths, mask_padding)
    if not torch.is_grad_enabled() and not m.training and f_fused.shape[-1] <= 256:
        # scoring (src/main.py:958-995): norm_f, attention pooling and the classifier in one launch
        feats, logits = head_fwd(f_fused, m.norm_f.weight, m.norm_f.bias, m.attention_pool.weight,
                                 m.attention_pool.bias, m.classifier.weight, m.classifier.bias, m.norm_f.eps)
        return feats.to(f_fused.dtype), logits.to(f_fused.dtype)
    if f_fused.shape[-1] <= 256:
        # training: norm_f + attention pooling as one kernel forward and one backward (:759-763)
        features = head_pool_fn(f_fused, m.norm_f.weight, m.norm_f.bias, m.attention_pool.weight,
                                m.attention_pool.bias, m.norm_f.eps).to(f_fused.dtype)
    else:
        f_fused = layer_norm_fn(f_fused, m.norm_f.weight, m.norm_f.bias, m.norm_f.eps, out_dtype=f_fused.dtype)   # :759
        attn = F.softmax(m.attention_pool(f_fused), dim=1)                          # :762
        features = torch.matmul(attn.transpose(1, 2), f_fused).squeeze(1)           # :763
    features = m.dropout(features)                                                  # :764
    return features, m.classifier(features)                                         # :767


def _backend_head_varlen(m, f_fused, lengths, mask_padding):
    seqlens = seqlens_tensor(lengths, f_fused.shape[0], f_fused.shape[1], f_fused.device)
    ps = (f_fused, *m.norm_f.parameters(), *m.attention_pool.parameters(), *m.classifier.parameters())
    if not mask_padding:
        _forward_only(seqlens, *ps)
    if f_fused.shape[-1] <= 256 and _wants_grad(*ps):
        # training: norm_f + attention pooling over the valid frames as one kernel forward and one backward
        features = head_pool_fn(f_fused, m.norm_f.weight, m.norm_f.bias, m.attention_pool.weight, m.attention_pool.bias,
                                m.norm_f.eps, seqlens).to(f_fused.dtype)
    elif f_fused.shape[-1] <= 256:
        feats, logits = head_fwd(f_fused, m.norm_f.weight, m.norm_f.bias, m.attention_pool.weight,
                                 m.attention_pool.bias, m.classifier.weight, m.classifier.bias, m.norm_f.eps, seqlens)
        if not m.training:
            return feats.to(f_fused.dtype), logits.to(f_fused.dtype)
        features = feats.to(f_fused.dtype)
    else:
        # wider than the head kernel: the same three steps with the padded frames masked out of the softmax
        f_fused = layer_norm_fn(f_fused, m.norm_f.weight, m.norm_f.bias, m.norm_f.eps, out_dtype=f_fused.dtype)
        valid = torch.arange(f_fused.shape[1], device=f_fused.device).unsqueeze(0) < seqlens.unsqueeze(1)
        scores = m.attention_pool(f_fused).masked_fill(~valid.unsqueeze(-1), float("-inf"))
        attn = F.softmax(scores, dim=1).masked_fill(~valid.unsqueeze(-1), 0.0)   # zero-length: zero features
        features = torch.matmul(attn.transpose(1, 2), f_fused.masked_fill(~valid.unsqueeze(-1), 0.0)).squeeze(1)
    features = m.dropout(features)
    return features, m.classifier(features)
