"""`DualStreamFusion` and `SELayer` with the reference's constructor, attributes and state_dict keys
(src/models/DualStreamSEMamba.py:492-531, :537-637): the block that turns the WavLM stream (B, T1, 1024) and the SincNet
stream (B, T2, 64) into the (B, T1, 144) features the Bi-Mamba backend reads (SURVEY 8 row f4).

B200 path: both input LayerNorms and the final one are this repository's kernels; the three Linear layers run on the
tcgen05 GEMM with bias / addend epilogues (forward, data gradient, MN-major weight gradient).  Two identities remove
the (B, T1, 288) concatenation and move the interpolation to the short side:
  fusion_proj(cat[f_w, f_s]) = f_w Wa^T + f_s Wb^T + b          (Wa, Wb = the two column halves of fusion_proj.weight)
  interp_T(f_s) Wb^T = interp_T(f_s Wb^T)                        (interpolation acts on time, the projection on channels)
so the SincNet branch is projected at its own T2 = 29 frames and enters the WavLM-side GEMM as its addend.

Variable length (`lengths`, `sinc_lengths`): every utterance runs as if alone at its own (n1, n2) frames - the
interpolation mode and index map, the SE mean and the SE scale are per utterance, on this repository's kernels
(ops.interp_frames, frame_mean, frame_scale); the fixed-length path below is untouched.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .ops import (_check_mask_padding, _forward_only, frame_mean, frame_scale, interp_frames, layer_norm_fn, linear_fn,
                  mask_frames, seqlens_tensor)


class SELayer(nn.Module):
    """Squeeze-and-excitation over (B, T, C) sequences, DualStreamSEMamba.py:509-531."""

    def __init__(self, channel: int, reduction: int = 16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool1d(1)
        self.fc = nn.Sequential(
            nn.Linear(channel, channel // reduction, bias=False),
            nn.ReLU(inplace=True),
            nn.Linear(channel // reduction, channel, bias=False),
            nn.Sigmoid(),
        )

    def gate(self, x):
        """(B, T, C) -> (B, 1, C) channel weights (fp32 statistics)."""
        y = x.float().mean(dim=1)                                                   # :524-526
        return self.fc(y).unsqueeze(1)                                              # :527

    def forward(self, x):
        return x * self.gate(x).to(x.dtype)                                         # :528


class DualStreamFusion(nn.Module):
    def __init__(self, wavlm_dim: int, sinc_dim: int, out_dim: int, reduction: int = 16):
        super().__init__()
        self.ln_wavlm = nn.LayerNorm(wavlm_dim)
        self.ln_sinc = nn.LayerNorm(sinc_dim)
        self.wavlm_proj = nn.Linear(wavlm_dim, out_dim)
        self.sinc_proj = nn.Linear(sinc_dim, out_dim)
        self.fusion_proj = nn.Linear(out_dim * 2, out_dim)
        self.se_layer = SELayer(out_dim, reduction=reduction)
        self.norm = nn.LayerNorm(out_dim)
        self.dropout = nn.Dropout(0.1)

    def forward(self, f_wavlm, f_sinc, lengths=None, sinc_lengths=None, *, mask_padding=False):
        """f_wavlm (B, T1, 1024), f_sinc (B, T2, 64) -> (B, T1, out_dim).

        lengths, sinc_lengths (B,): utterance b is f_wavlm[b, :lengths[b]] with f_sinc[b, :sinc_lengths[b]] of the
        right-padded streams (both or neither; list, CPU or CUDA tensor, see ops.seqlens_tensor).  Every valid output
        frame equals the utterance run alone; padded output frames are unspecified.  Scoring only (autograd recording
        raises NotImplementedError) unless mask_padding=True, the training form: padded input frames are replaced by
        zeros before anything reads them, padded output frames are zero, and gradients are those of the utterances run
        alone (zero at padded input frames)."""
        if lengths is not None or sinc_lengths is not None or mask_padding:
            return self._forward_varlen(f_wavlm, f_sinc, lengths, sinc_lengths, mask_padding)
        D = self.wavlm_proj.out_features
        T1, T2 = f_wavlm.shape[1], f_sinc.shape[1]
        res_dtype = f_wavlm.dtype if f_wavlm.dtype == torch.float32 or not torch.is_autocast_enabled("cuda") else torch.float32
        fw = layer_norm_fn(f_wavlm, self.ln_wavlm.weight, self.ln_wavlm.bias, self.ln_wavlm.eps)        # :591
        fs = layer_norm_fn(f_sinc, self.ln_sinc.weight, self.ln_sinc.bias, self.ln_sinc.eps)            # :592
        f_w = linear_fn(fw, self.wavlm_proj.weight, self.wavlm_proj.bias)                               # :595
        f_s = linear_fn(fs, self.sinc_proj.weight, self.sinc_proj.bias)                                 # :596
        Wa, Wb = self.fusion_proj.weight[:, :D], self.fusion_proj.weight[:, D:]
        s2 = linear_fn(f_s, Wb)                                                     # SincNet half of :630, at T2 frames
        if T2 != T1:                                                                # :601-626
            mode = "nearest" if T1 / T2 > 4.0 else "linear"
            kw = {} if mode == "nearest" else {"align_corners": False}
            s2 = F.interpolate(s2.transpose(1, 2), size=T1, mode=mode, **kw).transpose(1, 2).contiguous()
        fused = linear_fn(f_w, Wa, self.fusion_proj.bias, addend=s2)                # :629-630
        fused = fused * self.se_layer.gate(fused).to(fused.dtype)                   # :633
        fused = layer_norm_fn(fused, self.norm.weight, self.norm.bias, self.norm.eps, out_dtype=res_dtype)   # :636
        return self.dropout(fused)                                                  # :637

    def _forward_varlen(self, f_wavlm, f_sinc, lengths, sinc_lengths, mask_padding):
        _check_mask_padding(lengths, mask_padding)
        if (lengths is None) != (sinc_lengths is None):
            raise ValueError("lengths and sinc_lengths go together: pass the WavLM and the SincNet frame counts of every "
                             "utterance, or neither")
        D = self.wavlm_proj.out_features
        Bsz, T1, T2 = f_wavlm.shape[0], f_wavlm.shape[1], f_sinc.shape[1]
        sl1 = seqlens_tensor(lengths, Bsz, T1, f_wavlm.device)
        sl2 = seqlens_tensor(sinc_lengths, Bsz, T2, f_sinc.device)
        if mask_padding:
            f_wavlm, f_sinc = mask_frames(f_wavlm, sl1), mask_frames(f_sinc, sl2)
        else:
            _forward_only(sl1, f_wavlm, f_sinc, *self.parameters())
        res_dtype = f_wavlm.dtype if f_wavlm.dtype == torch.float32 or not torch.is_autocast_enabled("cuda") else torch.float32
        fw = layer_norm_fn(f_wavlm, self.ln_wavlm.weight, self.ln_wavlm.bias, self.ln_wavlm.eps)        # :591
        fs = layer_norm_fn(f_sinc, self.ln_sinc.weight, self.ln_sinc.bias, self.ln_sinc.eps)            # :592
        f_w = linear_fn(fw, self.wavlm_proj.weight, self.wavlm_proj.bias)                               # :595
        f_s = linear_fn(fs, self.sinc_proj.weight, self.sinc_proj.bias)                                 # :596
        Wa, Wb = self.fusion_proj.weight[:, :D], self.fusion_proj.weight[:, D:]
        s2 = interp_frames(linear_fn(f_s, Wb), sl1, sl2, T1)                        # :601-626 per utterance
        fused = linear_fn(f_w, Wa, self.fusion_proj.bias, addend=s2)                # :629-630
        gate = self.se_layer.fc(frame_mean(fused, sl1)).to(fused.dtype)             # :524-527 over each utterance's frames
        fused = frame_scale(fused, gate.float(), sl1)                               # :528, zero at padded frames
        fused = layer_norm_fn(fused, self.norm.weight, self.norm.bias, self.norm.eps, out_dtype=res_dtype)   # :636
        fused = self.dropout(fused)                                                 # :637
        return mask_frames(fused, sl1) if mask_padding else fused
