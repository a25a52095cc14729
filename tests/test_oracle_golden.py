"""Pin oracle/bimamba_oracle.py to fixtures produced by the reference's own code
(tests/golden/make_golden.py: MambaBlock mamba_block.py:6-122, PN_BiMambas_Encoder
DualStreamSEMamba.py:445-486, compute_eer evaluation.py:154-160), all in fp64."""
import os

import numpy as np
import pytest
import torch

from oracle import bimamba_oracle as orc
from oracle.compare import rel as _rel

RTOL = 2e-6   # fixtures store gradients as fp32 (6e-8 rounding); oracle runs in fp64


def _load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name)))


@pytest.mark.parametrize("tag", ["small", "phase6"])
def test_mamba_block_matches_reference(golden_dir, tag):
    g = _load(golden_dir, f"mamba_block_{tag}.npz")
    p = {k[len("param."):]: torch.tensor(v, dtype=torch.float64, requires_grad=True)
         for k, v in g.items() if k.startswith("param.")}
    assert set(p) == set(orc.PARAM_NAMES)
    x = torch.tensor(g["x"], dtype=torch.float64, requires_grad=True)
    out = orc.mamba_block_ref(p, x)
    assert _rel(out.detach().numpy(), g["out"]) < 1e-12
    (out * torch.tensor(g["cot"], dtype=torch.float64)).sum().backward()
    assert _rel(x.grad.numpy(), g["grad.x"]) < 1e-11
    for k, v in p.items():
        assert _rel(v.grad.numpy(), g["grad." + k]) < RTOL, k


def test_pn_bimamba_encoder_matches_reference(golden_dir):
    g = _load(golden_dir, "pn_bimamba_encoder_phase6.npz")
    p = {k[len("param."):]: torch.tensor(v, dtype=torch.float64, requires_grad=True)
         for k, v in g.items() if k.startswith("param.")}
    x = torch.tensor(g["x"], dtype=torch.float64, requires_grad=True)
    out = orc.pn_bimamba_encoder_ref(p, x)
    assert _rel(out.detach().numpy(), g["out"]) < 1e-12
    (out * torch.tensor(g["cot"], dtype=torch.float64)).sum().backward()
    assert _rel(x.grad.numpy(), g["grad.x"]) < 1e-11
    for k, v in p.items():
        assert _rel(v.grad.numpy(), g["grad." + k]) < RTOL, k


def test_compute_eer_matches_reference(golden_dir):
    g = _load(golden_dir, "compute_eer_cases.npz")
    for i in range(3):
        eer, thr = orc.compute_eer_ref(g[f"tgt{i}"], g[f"non{i}"])
        assert eer == float(g[f"eer{i}"])          # rank statistic: bit-identical
        assert thr == float(g[f"thr{i}"])


def test_op_refs_compose_to_block():
    """selective_scan_ref / causal_conv1d_ref in fp32 agree with fp64 to fp32 noise
    (SURVEY 8c: oracle self-noise ~7e-7 rel at L=201)."""
    torch.manual_seed(0)
    p64 = orc.init_mamba_params(48, 16, seed=3, dtype=torch.float64)
    x64 = torch.randn(2, 40, 48, dtype=torch.float64)
    y64 = orc.bimamba_ref(p64, x64)
    y32 = orc.bimamba_ref({k: v.float() for k, v in p64.items()}, x64.float())
    assert _rel(y32.numpy(), y64.numpy()) < 2e-5


def test_scan_ref_empty_and_edge():
    u = torch.zeros(1, 3, 0)
    y = orc.selective_scan_ref(u, u, -torch.ones(3, 4), torch.zeros(1, 4, 0), torch.zeros(1, 4, 0))
    assert y.shape == (1, 3, 0)
    # L = 1: y = (delta*B*u)*C + D*u
    u = torch.tensor([[[2.0]]]); d = torch.tensor([[[0.5]]])
    y = orc.selective_scan_ref(u, d, -torch.ones(1, 1), torch.tensor([[[3.0]]]), torch.tensor([[[4.0]]]),
                               D=torch.tensor([1.0]))
    assert torch.allclose(y, torch.tensor([[[0.5 * 3 * 2 * 4 + 2.0]]]))


def _tail_params(g, dtype=torch.float64, grad=True):
    P = {k[len("param."):]: torch.tensor(v, dtype=dtype, requires_grad=grad) for k, v in g.items() if k.startswith("param.")}
    fusion = {k[len("fusion."):]: v for k, v in P.items() if k.startswith("fusion.")}
    head = {k: v for k, v in P.items() if k.startswith(("norm_f.", "attention_pool.", "classifier."))}
    nl = 1 + max([int(k.split(".")[1]) for k in P if k.startswith("backbone_layers.")], default=-1)
    layers = [{k[len(f"backbone_layers.{i}."):]: v for k, v in P.items() if k.startswith(f"backbone_layers.{i}.")}
              for i in range(nl)]
    return P, fusion, layers, head


def test_fusion_matches_reference_linear_branch(golden_dir):
    """DualStreamFusion with T1 / T2 <= 4 (linear interpolation, DualStreamSEMamba.py:617-623): the fixture's
    grad.f_fused is the cotangent, so the fusion block's gradients are reproduced without the backbone."""
    g = _load(golden_dir, "model_tail_linear.npz")
    P, fusion, _, _ = _tail_params(g)
    fw = torch.tensor(g["f_wavlm"], dtype=torch.float64, requires_grad=True)
    fs = torch.tensor(g["f_sinc"], dtype=torch.float64, requires_grad=True)
    out = orc.fusion_ref(fusion, fw, fs)
    assert _rel(out.detach().numpy(), g["f_fused"]) < 1e-12
    (out * torch.tensor(g["grad.f_fused"])).sum().backward()
    assert _rel(fw.grad.numpy(), g["grad.f_wavlm"]) < RTOL
    assert _rel(fs.grad.numpy(), g["grad.f_sinc"]) < 1e-11
    for k, v in fusion.items():
        assert _rel(v.grad.numpy(), g["grad.fusion." + k]) < RTOL, k


def test_model_tail_matches_reference(golden_dir):
    """Fusion (nearest branch, the Phase-6 shape 201 vs 29 frames) -> 4 backbone layers -> norm_f -> attention
    pooling -> classifier against the reference Model.forward run (WavLM frontend stubbed)."""
    g = _load(golden_dir, "model_tail_nearest.npz")
    P, fusion, layers, head = _tail_params(g)
    assert len(layers) == 4
    fw = torch.tensor(g["f_wavlm"], dtype=torch.float64, requires_grad=True)
    fs = torch.tensor(g["f_sinc"], dtype=torch.float64, requires_grad=True)
    fused = orc.fusion_ref(fusion, fw, fs)
    assert _rel(fused.detach().numpy(), g["f_fused"]) < 1e-12
    feats, logits = orc.backend_ref(layers, head, fused)
    assert _rel(feats.detach().numpy(), g["features"]) < 1e-11
    assert _rel(logits.detach().numpy(), g["logits"]) < 1e-11
    ((logits * torch.tensor(g["cot_logits"])).sum() + (feats * torch.tensor(g["cot_features"])).sum()).backward()
    assert _rel(fw.grad.numpy().reshape(-1)[::5], g["grad5.f_wavlm"]) < RTOL
    assert _rel(fs.grad.numpy(), g["grad.f_sinc"]) < 1e-10
    for k, v in P.items():
        if k.startswith("backbone_layers."):
            assert _rel(v.grad.numpy().reshape(-1)[::5], g["grad5." + k]) < RTOL, k
        elif k == "attention_pool.bias":      # softmax over time is shift invariant: the true gradient is 0
            assert np.abs(v.grad.numpy()).max() < 1e-10 and np.abs(g["grad." + k]).max() < 1e-10
        else:
            assert _rel(v.grad.numpy(), g["grad." + k]) < RTOL, k


def test_time_split_carry_rule_equals_the_serial_scan():
    """The associative carry rule the time-parallel CUDA forward uses (csrc/scan_fwd_split.cu; oracle restatement
    selective_scan_split_ref) against the serial loop of mamba_block.py:92-117, in fp64: equal to rounding for every
    segmentation, including ragged last segments and a single segment."""
    g = torch.Generator().manual_seed(5)
    Bsz, D, N, L = 2, 5, 16, 77
    u, delta, z = (torch.randn(Bsz, D, L, generator=g, dtype=torch.float64) for _ in range(3))
    Bm, Cm = (torch.randn(Bsz, N, L, generator=g, dtype=torch.float64) for _ in range(2))
    A = -torch.exp(torch.log(torch.arange(1, N + 1, dtype=torch.float64)).repeat(D, 1) + 0.1 * torch.randn(D, N, generator=g, dtype=torch.float64))
    Dp = 1 + 0.1 * torch.randn(D, generator=g, dtype=torch.float64)
    bias = 0.05 * torch.randn(D, generator=g, dtype=torch.float64) - 2.0
    ref = orc.selective_scan_ref(u, 0.5 * delta, A, Bm, Cm, Dp, z, bias, delta_softplus=True)
    for seg_len in (16, 32, 48, 64, 80, 1024):
        out = orc.selective_scan_split_ref(u, 0.5 * delta, A, Bm, Cm, Dp, z, bias, delta_softplus=True, seg_len=seg_len)
        assert float((out - ref).abs().max() / ref.abs().max()) < 1e-12, seg_len
