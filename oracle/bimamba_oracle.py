"""CPU oracle for the Bi-Mamba hot path.  TEST INFRASTRUCTURE ONLY.

This file restates, in plain CPU PyTorch (any dtype, fp64 for ground truth), the
arithmetic of the reference's Bi-Mamba backend so the CUDA path can be checked
against it.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import it; the product package
never does (it raises if the CUDA library is missing instead of falling back).

Pinning status
--------------
The path the reference model really executes lives in the third-party package
``mamba-ssm`` (``requirements.txt:7``, ``>=1.0.0``, un-pinned, not vendored, not
installable offline) so the reference holds no golden vector for it: at that
boundary parity is *unpinned by the reference's own tests*.  What this oracle IS
pinned against (``tests/golden/make_golden.py`` -> ``tests/golden/*.npz``,
checked by ``tests/test_oracle_golden.py``):

* outputs and all parameter/input gradients of the reference's own pure-PyTorch
  ``MambaBlock`` (``/root/reference/src/models/modules/mamba_block.py:6-122``)
  and of the reference's ``PN_BiMambas_Encoder``
  (``/root/reference/src/models/DualStreamSEMamba.py:445-486``) run in this
  container with ``Mamba`` bound to that ``MambaBlock``;
* ``compute_eer`` (``/root/reference/src/evaluation.py:126-160``) on seeded
  score sets;
* the reference ``Model`` (``DualStreamSEMamba.py:643-769``) from the two streams'
  features on - ``DualStreamFusion`` (``:537-637``, both interpolation branches),
  the 4 backbone layers, ``norm_f``, attention pooling and the classifier
  (``:697-710``, ``:755-767``) - run through the reference's own ``Model.forward``
  with only the pretrained WavLM frontend stubbed (``model_tail_*.npz``).

Each function cites the reference lines it follows.  Nothing here is copied:
the reference is a ``nn.Module`` with a python loop; this is a functional
restatement over a plain dict of tensors.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor

PARAM_NAMES = (
    "in_proj.weight", "conv1d.weight", "conv1d.bias", "x_proj.weight",
    "dt_proj.weight", "dt_proj.bias", "A_log", "D", "out_proj.weight",
)


# --------------------------------------------------------------------------
# op-level references (signatures of mamba_ssm's selective_scan_ref and
# causal-conv1d's causal_conv1d_ref; math = mamba_block.py:52-55, 80-120)
# --------------------------------------------------------------------------
def causal_conv1d_ref(x: Tensor, weight: Tensor, bias: Optional[Tensor] = None,
                      activation: Optional[str] = None) -> Tensor:
    """x (B, D, L), weight (D, K), bias (D).  out[b,d,t] = act(bias[d] +
    sum_k weight[d,k] * x[b,d,t-(K-1)+k]) with zeros left of t=0.
    Follows mamba_block.py:52-55 (Conv1d padding=K-1, crop to L, SiLU)."""
    if activation not in (None, "silu", "swish"):
        raise NotImplementedError("activation must be None, silu, or swish")
    dtype_in = x.dtype
    x = x.to(weight.dtype)
    Bsz, D, L = x.shape
    K = weight.shape[1]
    xp = F.pad(x, (K - 1, 0))
    out = torch.zeros_like(x)
    for k in range(K):
        out = out + weight[:, k].view(1, D, 1) * xp[:, :, k:k + L]
    if bias is not None:
        out = out + bias.view(1, D, 1)
    if activation is not None:
        out = out * torch.sigmoid(out)
    return out.to(dtype_in)


def selective_scan_ref(u: Tensor, delta: Tensor, A: Tensor, B: Tensor, C: Tensor,
                       D: Optional[Tensor] = None, z: Optional[Tensor] = None,
                       delta_bias: Optional[Tensor] = None, delta_softplus: bool = False,
                       return_last_state: bool = False):
    """u, delta, z (B, D, L); A (D, N); B, C (B, N, L); D, delta_bias (D).
    h_t = exp(delta_t A) h_{t-1} + delta_t B_t u_t ; y_t = <h_t, C_t> + D u_t ;
    out = y * silu(z).  State in the wider of fp32 / the input dtype.
    Follows mamba_block.py:80 (softplus), :82 (A), :92-117 (scan), :120 (D skip),
    :61 (gate)."""
    dtype_in = u.dtype
    wide = torch.float64 if u.dtype == torch.float64 else torch.float32
    u = u.to(wide)
    delta = delta.to(wide)
    if delta_bias is not None:
        delta = delta + delta_bias.to(wide).view(1, -1, 1)
    if delta_softplus:
        delta = F.softplus(delta)
    A = A.to(wide)
    B = B.to(wide)
    C = C.to(wide)
    Bsz, Dm, L = u.shape
    N = A.shape[1]
    h = torch.zeros(Bsz, Dm, N, dtype=wide, device=u.device)
    ys = []
    for t in range(L):
        dt = delta[:, :, t].unsqueeze(-1)                     # (B, D, 1)
        decay = torch.exp(dt * A.unsqueeze(0))                # (B, D, N)
        inp = dt * B[:, :, t].unsqueeze(1) * u[:, :, t].unsqueeze(-1)
        h = decay * h + inp
        ys.append((h * C[:, :, t].unsqueeze(1)).sum(-1))
    y = torch.stack(ys, dim=2) if L > 0 else torch.zeros_like(u)
    if D is not None:
        y = y + u * D.to(wide).view(1, -1, 1)
    if z is not None:
        zz = z.to(wide)
        y = y * (zz * torch.sigmoid(zz))
    y = y.to(dtype_in)
    return (y, h) if return_last_state else y


def scan_inputs(Bsz: int, D: int, L: int, N: int = 16, seed: int = 0, dtype=torch.float32):
    """Seeded scan operands with SURVEY 8(d) config-5 distributions (trained-like A, mamba's dt-bias range):
    [u, delta, z, B, C] in `dtype` ((B, D, L) and (B, N, L)), then A (D, N), D (D) and delta_bias (D) in fp32."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(Bsz, D, L, generator=g)
    delta = 0.5 * torch.randn(Bsz, D, L, generator=g)
    z = torch.randn(Bsz, D, L, generator=g)
    Bm = torch.randn(Bsz, N, L, generator=g)
    Cm = torch.randn(Bsz, N, L, generator=g)
    A = -torch.exp(torch.log(torch.arange(1, N + 1, dtype=torch.float32)).repeat(D, 1)
                   + 0.1 * torch.randn(D, N, generator=g))
    Dp = 1 + 0.1 * torch.randn(D, generator=g)
    dt = torch.exp(torch.rand(D, generator=g) * (torch.log(torch.tensor(0.1)) - torch.log(torch.tensor(1e-3)))
                   + torch.log(torch.tensor(1e-3)))
    bias = dt + torch.log(-torch.expm1(-dt))
    act = [t.to(dtype) for t in (u, delta, z, Bm, Cm)]
    return act + [A, Dp, bias]


def selective_scan_split_ref(u: Tensor, delta: Tensor, A: Tensor, B: Tensor, C: Tensor,
                             D: Optional[Tensor] = None, z: Optional[Tensor] = None,
                             delta_bias: Optional[Tensor] = None, delta_softplus: bool = False,
                             seg_len: int = 16) -> Tensor:
    """The same scan as selective_scan_ref, evaluated the way the time-parallel CUDA forward does it
    (csrc/scan_fwd_split.cu): a carry pass gives every time segment's end state e_s from a ZERO state and its
    S_s = sum_t delta_t; the state entering segment s is the scan's associative rule applied to the earlier carries in
    order, h <- exp(A S_k) h + e_k for k < s (prod_t exp(delta_t A) = exp(A sum_t delta_t)); the output pass then walks the
    segment from that state.  Serial loop it restates: mamba_block.py:92-117."""
    dtype_in = u.dtype
    wide = torch.float64 if u.dtype == torch.float64 else torch.float32
    u_, d_ = u.to(wide), delta.to(wide)
    if delta_bias is not None:
        d_ = d_ + delta_bias.to(wide).view(1, -1, 1)
    if delta_softplus:
        d_ = F.softplus(d_)
    A_, B_, C_ = A.to(wide), B.to(wide), C.to(wide)
    Bsz, Dm, L = u_.shape
    N = A_.shape[1]

    def walk(h, t0, t1, emit):
        ys = []
        for t in range(t0, t1):
            dt = d_[:, :, t].unsqueeze(-1)
            h = torch.exp(dt * A_.unsqueeze(0)) * h + dt * B_[:, :, t].unsqueeze(1) * u_[:, :, t].unsqueeze(-1)
            if emit:
                ys.append((h * C_[:, :, t].unsqueeze(1)).sum(-1))
        return h, ys

    bounds = [(t0, min(L, t0 + seg_len)) for t0 in range(0, L, seg_len)]
    zero = torch.zeros(Bsz, Dm, N, dtype=wide, device=u.device)
    carries = [(walk(zero, t0, t1, False)[0], d_[:, :, t0:t1].sum(-1)) for t0, t1 in bounds[:-1]]      # carry pass
    ys = []
    for s_, (t0, t1) in enumerate(bounds):                                                              # output pass
        h = zero
        for e_k, S_k in carries[:s_]:
            h = torch.exp(S_k.unsqueeze(-1) * A_.unsqueeze(0)) * h + e_k
        ys += walk(h, t0, t1, True)[1]
    y = torch.stack(ys, dim=2) if L > 0 else torch.zeros_like(u_)
    if D is not None:
        y = y + u_ * D.to(wide).view(1, -1, 1)
    if z is not None:
        zz = z.to(wide)
        y = y * (zz * torch.sigmoid(zz))
    return y.to(dtype_in)


# --------------------------------------------------------------------------
# block-level references
# --------------------------------------------------------------------------
def mamba_dims(d_model: int, d_state: int = 16, d_conv: int = 4, expand: int = 2):
    """mamba_block.py:15-20."""
    d_inner = int(expand * d_model)
    dt_rank = math.ceil(d_model / 16)
    return d_inner, dt_rank


def init_mamba_params(d_model: int, d_state: int = 16, d_conv: int = 4, expand: int = 2,
                      seed: int = 0, dtype=torch.float32) -> Dict[str, Tensor]:
    """Seeded parameters with the shapes of mamba_block.py:22-39 (values are NOT the
    reference's init: parity tests always copy weights, SURVEY Appendix B)."""
    g = torch.Generator().manual_seed(seed)
    d_inner, dt_rank = mamba_dims(d_model, d_state, d_conv, expand)

    def uni(shape, bound):
        return (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * bound

    p = {
        "in_proj.weight": uni((2 * d_inner, d_model), d_model ** -0.5),
        "conv1d.weight": uni((d_inner, 1, d_conv), d_conv ** -0.5),
        "conv1d.bias": uni((d_inner,), d_conv ** -0.5),
        "x_proj.weight": uni((dt_rank + 2 * d_state, d_inner), d_inner ** -0.5),
        "dt_proj.weight": uni((d_inner, dt_rank), dt_rank ** -0.5),
        "A_log": torch.log(torch.arange(1, d_state + 1, dtype=torch.float64)).repeat(d_inner, 1)
        + 0.1 * torch.randn((d_inner, d_state), generator=g, dtype=torch.float64),
        "D": 1.0 + 0.1 * torch.randn((d_inner,), generator=g, dtype=torch.float64),
        "out_proj.weight": uni((d_model, d_inner), d_inner ** -0.5),
    }
    dt = torch.exp(torch.rand((d_inner,), generator=g, dtype=torch.float64)
                   * (math.log(0.1) - math.log(1e-3)) + math.log(1e-3)).clamp(min=1e-4)
    p["dt_proj.bias"] = dt + torch.log(-torch.expm1(-dt))
    return {k: v.to(dtype) for k, v in p.items()}


def mamba_block_ref(p: Dict[str, Tensor], x: Tensor) -> Tensor:
    """One direction of the block, x (B, L, d_model) -> (B, L, d_model).
    mamba_block.py:41-63 (forward) + :65-122 (ssm_step)."""
    d_inner = p["D"].shape[0]
    d_state = p["A_log"].shape[1]
    dt_rank = p["dt_proj.weight"].shape[1]
    xz = x @ p["in_proj.weight"].t()                                   # :48
    xs, z = xz[..., :d_inner], xz[..., d_inner:]                        # :49
    xc = causal_conv1d_ref(xs.transpose(1, 2), p["conv1d.weight"][:, 0, :],
                           p["conv1d.bias"], "silu")                    # :52-55, (B, D, L)
    x_dbl = xc.transpose(1, 2) @ p["x_proj.weight"].t()                 # :73
    dtr = x_dbl[..., :dt_rank]
    Bm = x_dbl[..., dt_rank:dt_rank + d_state]
    Cm = x_dbl[..., dt_rank + d_state:]                                 # :75
    delta = dtr @ p["dt_proj.weight"].t()                               # :80 (bias + softplus in scan)
    A = -torch.exp(p["A_log"])                                          # :82
    y = selective_scan_ref(xc, delta.transpose(1, 2), A, Bm.transpose(1, 2), Cm.transpose(1, 2),
                           p["D"], z.transpose(1, 2), p["dt_proj.bias"], True)
    return y.transpose(1, 2) @ p["out_proj.weight"].t()                 # :62


def bimamba_ref(p: Dict[str, Tensor], x_norm: Tensor) -> Tensor:
    """M(x) + flip(M(flip(x))) with shared weights, DualStreamSEMamba.py:473-481."""
    fwd = mamba_block_ref(p, x_norm)
    bwd = torch.flip(mamba_block_ref(p, torch.flip(x_norm, dims=[1])), dims=[1])
    return fwd + bwd


def init_encoder_params(d_model: int, d_state: int = 16, seed: int = 0,
                        dtype=torch.float32) -> Dict[str, Tensor]:
    """Parameters of one PN_BiMambas_Encoder, keyed like its state_dict
    (DualStreamSEMamba.py:451-465)."""
    g = torch.Generator().manual_seed(seed + 7919)
    p = {"mamba." + k: v for k, v in init_mamba_params(d_model, d_state, seed=seed, dtype=torch.float64).items()}

    def uni(shape, bound):
        return (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * bound

    p["norm1.weight"] = 1.0 + 0.1 * torch.randn((d_model,), generator=g, dtype=torch.float64)
    p["norm1.bias"] = 0.1 * torch.randn((d_model,), generator=g, dtype=torch.float64)
    p["norm2.weight"] = 1.0 + 0.1 * torch.randn((d_model,), generator=g, dtype=torch.float64)
    p["norm2.bias"] = 0.1 * torch.randn((d_model,), generator=g, dtype=torch.float64)
    p["feed_forward.0.weight"] = uni((4 * d_model, d_model), d_model ** -0.5)
    p["feed_forward.0.bias"] = uni((4 * d_model,), d_model ** -0.5)
    p["feed_forward.2.weight"] = uni((d_model, 4 * d_model), (4 * d_model) ** -0.5)
    p["feed_forward.2.bias"] = uni((d_model,), (4 * d_model) ** -0.5)
    return {k: v.to(dtype) for k, v in p.items()}


def pn_bimamba_encoder_ref(p: Dict[str, Tensor], x: Tensor, eps: float = 1e-5) -> Tensor:
    """DualStreamSEMamba.py:467-486: LN -> bi-Mamba -> LN -> FFN(GELU) -> + residual."""
    d_model = x.shape[-1]
    mp = {k[len("mamba."):]: v for k, v in p.items() if k.startswith("mamba.")}
    xn = F.layer_norm(x, (d_model,), p["norm1.weight"], p["norm1.bias"], eps)       # :472
    m = bimamba_ref(mp, xn)                                                          # :473-481
    m = F.layer_norm(m, (d_model,), p["norm2.weight"], p["norm2.bias"], eps)        # :482
    ff = F.gelu(m @ p["feed_forward.0.weight"].t() + p["feed_forward.0.bias"])
    ff = ff @ p["feed_forward.2.weight"].t() + p["feed_forward.2.bias"]              # :483
    return ff + x                                                                    # :485


def backend_ref(layers, head: Dict[str, Tensor], x: Tensor, eps: float = 1e-5):
    """4-layer stack + norm_f + attention pooling + classifier,
    DualStreamSEMamba.py:755-767 (dropout is identity in eval).  Returns
    (features (B, d_model), logits (B, 2))."""
    for p in layers:
        x = pn_bimamba_encoder_ref(p, x, eps)
    d_model = x.shape[-1]
    x = F.layer_norm(x, (d_model,), head["norm_f.weight"], head["norm_f.bias"], eps)   # :759
    a = torch.softmax(x @ head["attention_pool.weight"].t() + head["attention_pool.bias"], dim=1)  # :762
    feats = (a.transpose(1, 2) @ x).squeeze(1)                                          # :763
    logits = feats @ head["classifier.weight"].t() + head["classifier.bias"]            # :767
    return feats, logits


def fusion_ref(p: Dict[str, Tensor], f_wavlm: Tensor, f_sinc: Tensor, eps: float = 1e-5) -> Tensor:
    """DualStreamFusion.forward, DualStreamSEMamba.py:580-637 with SELayer :519-531 (eval: dropout = identity).
    f_wavlm (B, T1, 1024), f_sinc (B, T2, 64) -> (B, T1, out_dim).  Keys as in the module's state_dict
    (ln_wavlm, ln_sinc, wavlm_proj, sinc_proj, fusion_proj, se_layer.fc.{0,2}, norm)."""
    fw = F.layer_norm(f_wavlm, (f_wavlm.shape[-1],), p["ln_wavlm.weight"], p["ln_wavlm.bias"], eps)     # :591
    fs = F.layer_norm(f_sinc, (f_sinc.shape[-1],), p["ln_sinc.weight"], p["ln_sinc.bias"], eps)         # :592
    fw = fw @ p["wavlm_proj.weight"].t() + p["wavlm_proj.bias"]                                         # :595
    fs = fs @ p["sinc_proj.weight"].t() + p["sinc_proj.bias"]                                           # :596
    T1, T2 = fw.shape[1], fs.shape[1]
    if T1 != T2:                                                                                        # :601-626
        fs = fs.transpose(1, 2)
        if T1 / T2 > 4.0:
            fs = F.interpolate(fs, size=T1, mode="nearest")
        else:
            fs = F.interpolate(fs, size=T1, mode="linear", align_corners=False)
        fs = fs.transpose(1, 2)
    fused = torch.cat([fw, fs], dim=-1) @ p["fusion_proj.weight"].t() + p["fusion_proj.bias"]           # :629-630
    se = fused.mean(dim=1)                                                                              # :524-526
    se = torch.sigmoid(torch.relu(se @ p["se_layer.fc.0.weight"].t()) @ p["se_layer.fc.2.weight"].t())  # :527 (:512-517)
    fused = fused * se.unsqueeze(1)                                                                     # :528
    return F.layer_norm(fused, (fused.shape[-1],), p["norm.weight"], p["norm.bias"], eps)               # :636


def init_head_params(d_model: int, seed: int = 0, dtype=torch.float32) -> Dict[str, Tensor]:
    g = torch.Generator().manual_seed(seed + 104729)

    def uni(shape, bound):
        return (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * bound

    h = {
        "norm_f.weight": 1.0 + 0.1 * torch.randn((d_model,), generator=g, dtype=torch.float64),
        "norm_f.bias": 0.1 * torch.randn((d_model,), generator=g, dtype=torch.float64),
        "attention_pool.weight": uni((1, d_model), d_model ** -0.5),
        "attention_pool.bias": uni((1,), d_model ** -0.5),
        "classifier.weight": uni((2, d_model), d_model ** -0.5),
        "classifier.bias": uni((2,), d_model ** -0.5),
    }
    return {k: v.to(dtype) for k, v in h.items()}


# --------------------------------------------------------------------------
# metric (src/evaluation.py:126-160)
# --------------------------------------------------------------------------
def compute_eer_ref(target_scores: np.ndarray, nontarget_scores: np.ndarray):
    """Equal error rate and threshold.  evaluation.py:126-151 (DET curve: stable
    sort of pooled scores, cumulative miss / false-alarm rates) and :154-160 (EER =
    mean of FRR and FAR where |FRR - FAR| is smallest)."""
    tgt = np.asarray(target_scores)
    non = np.asarray(nontarget_scores)
    pooled = np.concatenate([tgt, non])
    is_tgt = np.concatenate([np.ones(tgt.size), np.zeros(non.size)])
    order = np.argsort(pooled, kind="mergesort")
    is_tgt = is_tgt[order]
    tgt_below = np.cumsum(is_tgt)
    non_above = non.size - (np.arange(1, pooled.size + 1) - tgt_below)
    frr = np.concatenate([[0.0], tgt_below / tgt.size])
    far = np.concatenate([[1.0], non_above / non.size])
    thr = np.concatenate([[pooled[order[0]] - 0.001], pooled[order]])
    k = int(np.argmin(np.abs(frr - far)))
    return float(np.mean((frr[k], far[k]))), float(thr[k])
