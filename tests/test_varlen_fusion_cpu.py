"""Host-side checks of variable-length DualStreamFusion (no device needed): the oracle's fp32 interpolation index rule
against F.interpolate, why it is not the fp64 rule, the oracle at full lengths against fusion_ref, the module's keyword
checks before any device work, and the argument errors of the new C entries."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bimamba_b200 as bm
from oracle import bimamba_oracle as orc
from oracle.varlen_fusion_oracle import fusion_varlen_ref, interp_index_fp32

FAKE = 4096          # a non-null device address: every call below must fail (or return) before touching it


def _weights(n2, n1):
    """(n2, n1) float32 matrix W with output frame t = sum_j W[j, t] x[j], from interp_index_fp32."""
    _, i0, i1, w0, w1 = interp_index_fp32(n2, n1)
    W = np.zeros((n2, n1), np.float32)
    t = np.arange(n1)
    W[i0, t] = w0
    W[i1, t] = W[i1, t] + w1          # i0 == i1 at the last source frame: w0 + w1 in float32, as F.interpolate adds them
    return W


def test_fp32_index_rule_equals_f_interpolate_on_every_pair():
    """For every n2 in 1..80 and n1 in 1..520 the rule gives F.interpolate's fp32 output bit for bit: interpolating the
    identity (n2 channels of one-hot frames) reads the weight matrix out."""
    bad = []
    for n2 in range(1, 81):
        eye = torch.eye(n2).view(1, n2, n2)
        for n1 in range(1, 521):
            if n1 == n2:
                continue
            kw = {"mode": "nearest"} if n1 > 4 * n2 else {"mode": "linear", "align_corners": False}
            ref = F.interpolate(eye, size=n1, **kw)[0].numpy()
            if not np.array_equal(_weights(n2, n1), ref):
                bad.append((n2, n1))
    assert not bad, bad[:10]
    mode, i0, i1, w0, w1 = interp_index_fp32(29, 29)
    assert mode == "copy" and (i0 == np.arange(29)).all() and (w0 == 1).all() and (w1 == 0).all()
    assert interp_index_fp32(29, 116)[0] == "linear" and interp_index_fp32(29, 117)[0] == "nearest"


def test_fp64_rule_picks_another_frame_for_a_real_clip():
    """A 2.21 s clip (35 360 samples) has n1 = (35360 - 400) // 320 + 1 = 110 WavLM frames and n2 = 16 SincNet frames
    ((S - 128) // 3, then // 3 six times).  Frame 55 is exactly 55 * 16 / 110 = 8 in exact arithmetic; in fp32
    scale = 16 / 110 rounds down and F.interpolate reads frame 7, in fp64 it reads frame 8."""
    S = 35360
    n1, n2 = (S - 400) // 320 + 1, (S - 128) // 3
    for _ in range(6):
        n2 //= 3
    assert (n1, n2) == (110, 16)
    src = torch.arange(n2, dtype=torch.float64).view(1, 1, n2)
    assert int(F.interpolate(src.float(), size=n1, mode="nearest")[0, 0, 55]) == 7
    assert int(F.interpolate(src, size=n1, mode="nearest")[0, 0, 55]) == 8
    assert interp_index_fp32(n2, n1)[1][55] == 7


def _fixture_fusion(tag):
    g = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", f"model_tail_{tag}.npz")))
    p = {k[len("param.fusion."):]: torch.tensor(v, dtype=torch.float64) for k, v in g.items()
         if k.startswith("param.fusion.")}
    return p, torch.tensor(g["f_wavlm"], dtype=torch.float64), torch.tensor(g["f_sinc"], dtype=torch.float64)


@pytest.mark.parametrize("tag", ["nearest", "linear"])
def test_varlen_oracle_at_full_length_equals_fusion_ref(tag):
    """Full lengths (201 / 29 nearest, 60 / 14 linear): the per-utterance oracle is fusion_ref.  At these two pairs the
    fp32 and fp64 index rules agree, so only the weights' fp32 rounding separates them (linear)."""
    p, fw, fs = _fixture_fusion(tag)
    B, T1, T2 = fw.shape[0], fw.shape[1], fs.shape[1]
    ref = orc.fusion_ref(p, fw, fs)
    out = fusion_varlen_ref(p, fw, fs, [T1] * B, [T2] * B)
    err = float((out - ref).abs().max() / ref.abs().max())
    assert err < (1e-14 if tag == "nearest" else 1e-6), err


def test_varlen_oracle_padding_is_never_read():
    p, fw, fs = _fixture_fusion("linear")
    fw2, fs2 = fw.clone(), fs.clone()
    fw2[0, 40:] = float("nan")
    fs2[0, 9:] = float("nan")
    a = fusion_varlen_ref(p, fw2, fs2, [40, 60], [9, 14])
    assert torch.isfinite(a).all() and bool((a[0, 40:] == 0).all())
    b = fusion_varlen_ref(p, fw[:1, :40], fs[:1, :9], [40], [9])
    assert torch.equal(a[0, :40], b[0])


def test_module_keyword_checks_come_before_any_device_work():
    fus = bm.DualStreamFusion(1024, 64, 144)
    fw, fs = torch.randn(2, 20, 1024), torch.randn(2, 4, 64)
    with pytest.raises(ValueError, match="go together"):
        fus(fw, fs, [20, 10])
    with pytest.raises(ValueError, match="go together"):
        fus(fw, fs, None, [4, 2])
    with pytest.raises(ValueError, match="mask_padding=True needs lengths"):
        fus(fw, fs, mask_padding=True)
    with pytest.raises(ValueError, match="1..20"):
        fus(fw, fs, [21, 10], [4, 2], mask_padding=True)
    with pytest.raises(ValueError, match="1..4"):
        fus(fw, fs, [20, 10], [4, 5], mask_padding=True)


def test_fusion_entry_argument_errors_are_codes():
    lib = bm._lib.load()
    for fn in (lib.bimamba_interp_frames_fwd, lib.bimamba_interp_frames_bwd):
        assert fn(None, FAKE, FAKE, FAKE, 2, 20, 4, 144, 1, None) == -1
        assert fn(FAKE, FAKE, FAKE, None, 2, 20, 4, 144, 1, None) == -1
        assert fn(FAKE, FAKE, FAKE, FAKE, 2, 20, 4, 144, 7, None) == -3
        assert fn(FAKE, FAKE, FAKE, FAKE, -1, 20, 4, 144, 1, None) == -3
        assert fn(None, None, None, None, 0, 20, 4, 144, 1, None) == 0               # empty batch: a no-op
    assert b"interp_frames_bwd: bad sizes" in lib.bimamba_last_error()
    assert lib.bimamba_frame_mean(None, FAKE, FAKE, 2, 20, 144, 0, None) == -1
    assert lib.bimamba_frame_mean(FAKE, FAKE, FAKE, 2, 20, 144, 3, None) == -3
    assert lib.bimamba_frame_mean(None, None, None, 0, 20, 144, 0, None) == 0
    assert lib.bimamba_frame_mean_bwd(FAKE, None, FAKE, 2, 20, 144, 0, None) == -1
    assert lib.bimamba_frame_mean_bwd(None, None, None, 0, 20, 144, 0, None) == 0
    assert lib.bimamba_frame_scale(FAKE, None, FAKE, FAKE, 2, 20, 144, 1, None) == -1
    assert lib.bimamba_frame_scale(FAKE, FAKE, FAKE, FAKE, 2, 20, 144, -1, None) == -3
    assert lib.bimamba_frame_scale(None, None, None, None, 0, 20, 144, 1, None) == 0
    assert lib.bimamba_frame_scale_bwd(FAKE, FAKE, FAKE, FAKE, None, FAKE, 2, 20, 144, 1, None) == -1
    assert b"frame_scale_bwd: null operand" in lib.bimamba_last_error()
    assert lib.bimamba_frame_scale_bwd(None, None, None, None, None, None, 0, 20, 144, 1, None) == 0
    assert [lib.bimamba_frame_scale_bwd_slices(n) for n in (0, 1, 64, 65, 499)] == [1, 1, 1, 2, 8]
