"""GPU parity of the Bi-Mamba block / encoder / backend against the oracle and the golden
fixtures generated from the reference (tests/golden/make_golden.py).

Tolerance (north_star): <= 1e-4 relative fp32, <= 2e-2 bf16, outputs AND every gradient, measured per slice
(oracle/compare.py): activations per utterance and per 8-frame chunk, each parameter gradient per its own blocks
(x_proj rows dt | B | C, in_proj halves, conv taps, dt_proj rank columns, 32-row groups, channels, states).
"""
import copy
import os
import pickle

import numpy as np
import pytest
import torch

import bimamba_b200 as bm
from oracle import bimamba_oracle as orc
from oracle import compare as cmp

pytestmark = pytest.mark.gpu


def _check_params(named, want, tol):
    """Every parameter gradient of `named` (name, parameter) against want[name], sliced by the parameter's blocks."""
    for name, p in named:
        cmp.check(name, p.grad, want[name], tol, cmp.param(name, p.shape))


def _load_mamba(m, params):
    sd = {k: torch.as_tensor(np.asarray(v)).float() for k, v in params.items()}
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected


@pytest.mark.parametrize("tag", ["small", "phase6"])
def test_mamba_forward_backward_vs_reference_fixture(golden_dir, tag):
    """Mamba.forward (one direction) against the reference's own MambaBlock run (fixture)."""
    g = dict(np.load(os.path.join(golden_dir, f"mamba_block_{tag}.npz")))
    params = {k[len("param."):]: v for k, v in g.items() if k.startswith("param.")}
    d_model = g["x"].shape[-1]
    m = bm.Mamba(d_model, 16).cuda()
    _load_mamba(m, params)
    x = torch.tensor(g["x"], device="cuda", requires_grad=True)
    out = m(x)
    cmp.check("out", out, g["out"], 1e-4, cmp.frames())
    out.backward(torch.tensor(g["cot"], device="cuda"))
    cmp.check("dx", x.grad, g["grad.x"], 1e-4, cmp.frames())
    _check_params(m.named_parameters(), {k[len("grad."):]: v for k, v in g.items() if k.startswith("grad.")}, 1e-4)


def test_encoder_vs_reference_fixture(golden_dir):
    """PN_BiMambas_Encoder (both directions, LN, FFN, residual) against the reference class."""
    g = dict(np.load(os.path.join(golden_dir, "pn_bimamba_encoder_phase6.npz")))
    enc = bm.PN_BiMambas_Encoder(144, 16).cuda()
    sd = {k[len("param."):]: torch.tensor(v).float() for k, v in g.items() if k.startswith("param.")}
    enc.load_state_dict(sd, strict=True)
    x = torch.tensor(g["x"], device="cuda", requires_grad=True)
    out = enc(x)
    cmp.check("out", out, g["out"], 1e-4, cmp.frames())
    out.backward(torch.tensor(g["cot"], device="cuda"))
    cmp.check("dx", x.grad, g["grad.x"], 1e-4, cmp.frames())
    _check_params(enc.named_parameters(), {k[len("grad."):]: v for k, v in g.items() if k.startswith("grad.")}, 1e-4)


@pytest.mark.parametrize("Bsz,L", [(3, 201), (2, 499), (1, 1), (2, 260)])
def test_bidirectional_block_fp32_vs_oracle(Bsz, L):
    p64 = orc.init_mamba_params(144, 16, seed=L, dtype=torch.float64)
    m = bm.Mamba(144, 16).cuda()
    _load_mamba(m, {k: v.numpy() for k, v in p64.items()})
    g = torch.Generator().manual_seed(L)
    x = torch.randn(Bsz, L, 144, generator=g)
    cot = torch.randn(Bsz, L, 144, generator=g)
    pr = {k: v.float().double().requires_grad_(True) for k, v in p64.items()}
    xr = x.double().requires_grad_(True)
    ref = orc.bimamba_ref(pr, xr)
    (ref * cot.double()).sum().backward()
    xd = x.cuda().requires_grad_(True)
    out = m.forward_bidirectional(xd)
    out.backward(cot.cuda())
    cmp.check("out", out, ref, 1e-4, cmp.frames())
    cmp.check("dx", xd.grad, xr.grad, 1e-4, cmp.frames())
    _check_params(m.named_parameters(), {k: v.grad for k, v in pr.items()}, 1e-4)


@pytest.mark.parametrize("Bsz,L", [(3, 201), (2, 13)])
def test_bidirectional_block_conv_tile_variant(Bsz, L):
    """The conv backward's shared-memory tile fallback forced (bimamba_set_tuning) on the fused block (dt projection
    inside the scan kernels, both directions in one launch): fp32, 1e-4 against the oracle."""
    with bm._lib.tuning(bm._lib.TUNE_CONV_BWD, 1):
        test_bidirectional_block_fp32_vs_oracle(Bsz, L)


@pytest.mark.parametrize("Bsz,L,nseg", [(3, 201, 3), (2, 499, 4), (2, 260, 2)])
def test_bidirectional_block_time_split_forward(Bsz, L, nseg):
    """The time-parallel forward scan forced inside the fused block (dt projection in the kernel, both directions, gate,
    checkpoints + ungated y for the backward): outputs and every gradient against the oracle, fp32, 1e-4."""
    with bm._lib.tuning(bm._lib.TUNE_SCAN_SPLIT, nseg):
        test_bidirectional_block_fp32_vs_oracle(Bsz, L)
        if nseg == 3:
            test_block_bf16_autocast_vs_oracle()


def test_block_bf16_autocast_vs_oracle():
    """Config-2 numerics: bf16 activations / fp32 state under autocast; oracle in fp64 on the same
    fp32 master weights.  Tolerance 2e-2 relative."""
    p64 = orc.init_mamba_params(144, 16, seed=2, dtype=torch.float64)
    m = bm.Mamba(144, 16).cuda()
    _load_mamba(m, {k: v.numpy() for k, v in p64.items()})
    g = torch.Generator().manual_seed(2)
    x = torch.randn(4, 201, 144, generator=g)
    cot = torch.randn(4, 201, 144, generator=g)
    pr = {k: v.float().double().requires_grad_(True) for k, v in p64.items()}
    xr = x.double().requires_grad_(True)
    ref = orc.bimamba_ref(pr, xr)
    (ref * cot.double()).sum().backward()
    xd = x.cuda().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = m.forward_bidirectional(xd)
    assert out.dtype == torch.bfloat16
    out.float().backward(cot.cuda())
    cmp.check("out", out, ref, 2e-2, cmp.frames())
    cmp.check("dx", xd.grad, xr.grad, 2e-2, cmp.frames())
    assert all(prm.grad.dtype == torch.float32 for prm in m.parameters())
    _check_params(m.named_parameters(), {k: v.grad for k, v in pr.items()}, 2e-2)


def test_fusion_identities_on_device():
    """Size-independent properties at the Phase-6 training shape (B=64, L=201):
    bidirectional(x) == fwd(x) + flip(fwd(flip(x)))  (DualStreamSEMamba.py:473-481)."""
    torch.manual_seed(0)
    m = bm.Mamba(144, 16).cuda()
    with torch.no_grad():
        m.A_log.add_(0.1 * torch.randn_like(m.A_log))
    x = torch.randn(64, 201, 144, device="cuda")
    with torch.no_grad():
        bi = m.forward_bidirectional(x)
        two = m(x) + torch.flip(m(torch.flip(x, dims=[1])), dims=[1])
    assert cmp.rel(bi, two) < 1e-5


def test_eer_identity_on_synthetic_scoring_set():
    """Identical EER on a fixed synthetic scoring set (fp32): scores = logits[:, 1] of the 4-layer
    backend + head (DualStreamSEMamba.py:755-767, main.py:978-984), EER by evaluation.py:154-160."""
    n_utt, L = 192, 64
    layers = [orc.init_encoder_params(144, 16, seed=10 + i) for i in range(4)]
    head = orc.init_head_params(144, seed=3)
    g = torch.Generator().manual_seed(77)
    feats = torch.randn(n_utt, L, 144, generator=g)
    labels = (torch.rand(n_utt, generator=g) < 0.3).numpy()
    with torch.no_grad():
        _, logits_ref = orc.backend_ref(layers, head, feats)
    net = bm.BiMambaBackend(144, 4, 16).cuda().eval()
    sd = {}
    for i, p in enumerate(layers):
        for k, v in p.items():
            sd[f"backbone_layers.{i}.{k}"] = v
    sd.update(head)
    net.load_state_dict(sd, strict=True)
    with torch.no_grad():
        _, logits = net(feats.cuda())
    s_ref = logits_ref[:, 1].numpy().astype(np.float64)
    s_dev = logits[:, 1].cpu().numpy().astype(np.float64)
    eer_ref, _ = orc.compute_eer_ref(s_ref[labels], s_ref[~labels])
    eer_dev, _ = orc.compute_eer_ref(s_dev[labels], s_dev[~labels])
    assert np.abs(s_ref - s_dev).max() < 1e-4 * max(1.0, np.abs(s_ref).max())
    assert eer_dev == eer_ref


def test_module_surface():
    """deepcopy (EMA AveragedModel, main.py:495), pickle, no_grad / inference_mode
    (filter_dirty_data.py:134-151), frozen params, clip_grad_norm_ (main.py:1104)."""
    m = bm.PN_BiMambas_Encoder(144, 16).cuda()
    m2 = copy.deepcopy(m)
    m3 = pickle.loads(pickle.dumps(m))
    x = torch.randn(2, 33, 144, device="cuda")
    with torch.inference_mode():
        a, b, c = m(x), m2(x), m3(x)
    assert torch.equal(a, b) and torch.equal(a, c)
    for p in m.mamba.parameters():
        p.requires_grad_(False)
    y = m(x.requires_grad_(True))
    y.sum().backward()
    assert x.grad is not None and all(p.grad is None for p in m.mamba.parameters())
    for p in m.mamba.parameters():
        p.requires_grad_(True)
    m(x).sum().backward()
    torch.nn.utils.clip_grad_norm_(m.parameters(), 3.0)
    with torch.autocast("cuda", dtype=torch.float16):
        assert m(x).isfinite().all()


def test_graphed_train_step_pipelined_matches_sequential():
    """GraphedTrainStep.run_pipelined (H2D of batch i+1 overlapping step i) gives the same loss sequence as run()."""
    def make():
        torch.manual_seed(3)
        net = bm.BiMambaBackend(144, 2, 16).cuda()
        params = list(net.backbone_layers.parameters())
        opt = torch.optim.AdamW(params, lr=1e-3, capturable=True, fused=True)

        def zero():
            for p in params:
                p.grad = None

        def loss_fn(x):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return net.forward_features(x).float().square().mean()
        return bm.GraphedTrainStep(loss_fn, torch.zeros(4, 50, 144, device="cuda"), zero, opt, warmup=1)

    g = torch.Generator().manual_seed(0)
    batches = [torch.randn(4, 50, 144, generator=g).pin_memory() for _ in range(5)]
    a = make()
    seq = [float(a.run(b).detach()) for b in batches]
    b_ = make()
    pip = list(b_.run_pipelined(batches))
    assert len(pip) == len(seq)
    for u, v in zip(seq, pip):
        assert abs(u - v) <= 2e-3 * max(1.0, abs(u)), (seq, pip)


@pytest.mark.parametrize("d_model,Bsz,L", [(64, 3, 77), (80, 2, 130), (256, 2, 40)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_block_other_widths(d_model, Bsz, L, dtype):
    """The block is not specialised to d_model 144: other widths (d_inner 128 / 160 / 512, dt_rank 4 / 5 / 16, channel
    counts that do not fill the kernels' 32-channel groups) against the oracle, outputs and every gradient."""
    p64 = orc.init_mamba_params(d_model, 16, seed=d_model, dtype=torch.float64)
    m = bm.Mamba(d_model, 16).cuda()
    _load_mamba(m, {k: v.numpy() for k, v in p64.items()})
    g = torch.Generator().manual_seed(d_model + L)
    x = torch.randn(Bsz, L, d_model, generator=g)
    cot = torch.randn(Bsz, L, d_model, generator=g)
    pr = {k: v.float().double().requires_grad_(True) for k, v in p64.items()}
    xr = x.double().requires_grad_(True)
    ref = orc.bimamba_ref(pr, xr)
    (ref * cot.double()).sum().backward()
    xd = x.cuda().requires_grad_(True)
    if dtype == torch.float32:
        out = m.forward_bidirectional(xd)
        tol = 1e-4
    else:
        with torch.autocast("cuda", dtype=dtype):
            out = m.forward_bidirectional(xd)
        tol = 2e-2
    out.float().backward(cot.cuda())
    cmp.check("out", out, ref, tol, cmp.frames())
    cmp.check("dx", xd.grad, xr.grad, tol, cmp.frames())
    _check_params(m.named_parameters(), {k: v.grad for k, v in pr.items()}, tol)


def test_backward_is_bitwise_deterministic():
    """No atomics anywhere on the path: two runs of the encoder layer's forward + backward at the benchmark shape give
    bit-identical outputs and gradients (also a race detector for the hand-synchronised shared-memory phases)."""
    torch.manual_seed(5)
    enc = bm.PN_BiMambas_Encoder(144, 16).cuda()
    with torch.no_grad():
        enc.mamba.A_log.add_(0.1 * torch.randn_like(enc.mamba.A_log))
    x = torch.randn(64, 201, 144, device="cuda")
    runs = []
    for _ in range(3):
        for p in enc.parameters():
            p.grad = None
        xi = x.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = enc(xi)
        out.float().square().mean().backward()
        torch.cuda.synchronize()
        runs.append([out.detach().clone(), xi.grad.clone()] + [p.grad.clone() for p in enc.parameters()])
    for other in runs[1:]:
        for a, b in zip(runs[0], other):
            assert torch.equal(a, b)


def test_fused_adamw_matches_torch_adamw():
    """One-launch AdamW (optim.py / csrc/optim.cu) against torch.optim.AdamW over several steps with changing
    gradients and a learning-rate change, on tensors of awkward sizes (vector tail, multi-chunk, scalar)."""
    g = torch.Generator().manual_seed(7)
    shapes = [(576, 144), (288, 4), (288,), (9000,), (1,), (37, 3)]
    ref_p = [torch.randn(s, generator=g).cuda().requires_grad_(True) for s in shapes]
    our_p = [p.detach().clone().requires_grad_(True) for p in ref_p]
    ref = torch.optim.AdamW(ref_p, lr=3e-3, betas=(0.9, 0.98), eps=1e-8, weight_decay=0.05)
    ours = bm.FusedAdamW(our_p, lr=3e-3, betas=(0.9, 0.98), eps=1e-8, weight_decay=0.05)
    for it in range(6):
        if it == 3:
            for o in (ref, ours):
                o.param_groups[0]["lr"] = 1e-3
        for a, b in zip(ref_p, our_p):
            gr = torch.randn(a.shape, generator=g).cuda()
            a.grad = gr.clone()
            b.grad = gr.clone()
        ref.step()
        ours.step()
    for a, b in zip(ref_p, our_p):
        assert cmp.rel(b, a) < 1e-6
    st = ours.state[our_p[0]]
    assert cmp.rel(st["exp_avg"], ref.state[ref_p[0]]["exp_avg"]) < 1e-6
    assert cmp.rel(st["exp_avg_sq"], ref.state[ref_p[0]]["exp_avg_sq"]) < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# round 2: reference-generated fixtures of the model tail, the reference's own (unfused) forward, fp16 + GradScaler
# ---------------------------------------------------------------------------------------------------------------------
def _tail_state(g):
    return {k[len("param."):]: torch.tensor(v).float() for k, v in g.items() if k.startswith("param.")}


@pytest.mark.parametrize("tag,dtype", [("linear", torch.float32), ("nearest", torch.float32), ("nearest", torch.bfloat16)])
def test_dual_stream_fusion_vs_reference_fixture(golden_dir, tag, dtype):
    """DualStreamFusion (DualStreamSEMamba.py:537-637, both interpolation branches) against the reference Model run:
    output and every gradient, with the fixture's grad.f_fused as cotangent."""
    g = dict(np.load(os.path.join(golden_dir, f"model_tail_{tag}.npz")))
    fus = bm.DualStreamFusion(1024, 64, 144, reduction=16).cuda().eval()
    sd = {k[len("fusion."):]: v for k, v in _tail_state(g).items() if k.startswith("fusion.")}
    fus.load_state_dict(sd, strict=True)
    fw = torch.tensor(g["f_wavlm"], device="cuda", requires_grad=True)
    fs = torch.tensor(g["f_sinc"], device="cuda", dtype=torch.float32, requires_grad=True)
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        out = fus(fw, fs)
    assert out.dtype == torch.float32
    cmp.check("out", out, g["f_fused"], tol, cmp.frames())
    out.backward(torch.tensor(g["grad.f_fused"], device="cuda", dtype=torch.float32))
    if tag == "linear":
        cmp.check("d f_wavlm", fw.grad, g["grad.f_wavlm"], tol, cmp.frames())
    else:                                      # every 5th element of the flattened gradient: no structure to slice
        cmp.check("d f_wavlm[::5]", fw.grad.reshape(-1)[::5], g["grad5.f_wavlm"], tol)
    cmp.check("d f_sinc", fs.grad, g["grad.f_sinc"], tol, cmp.frames())
    _check_params(fus.named_parameters(), {k[len("grad.fusion."):]: v for k, v in g.items()
                                           if k.startswith("grad.fusion.")}, tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_model_tail_vs_reference_fixture(golden_dir, dtype):
    """Fusion -> 4 x PN_BiMambas_Encoder -> norm_f -> attention pooling -> classifier (DualStreamSEMamba.py:697-710,
    :755-767) against the reference's own Model.forward (fixture; WavLM frontend stubbed): features, logits and every
    gradient, through the TRAINING head (autograd) and, without grad, through the one-launch scoring head."""
    g = dict(np.load(os.path.join(golden_dir, "model_tail_nearest.npz")))
    sd = _tail_state(g)
    fus = bm.DualStreamFusion(1024, 64, 144).cuda().eval()
    fus.load_state_dict({k[len("fusion."):]: v for k, v in sd.items() if k.startswith("fusion.")}, strict=True)
    net = bm.BiMambaBackend(144, 4, 16).cuda().eval()
    net.load_state_dict({k: v for k, v in sd.items() if not k.startswith("fusion.")}, strict=True)
    fw = torch.tensor(g["f_wavlm"], device="cuda", requires_grad=True)
    fs = torch.tensor(g["f_sinc"], device="cuda", dtype=torch.float32, requires_grad=True)
    # fp32: the north_star's 1e-4.  bf16: 2e-2 is the bar of ONE block; this chains fusion + 4 blocks + head in bf16,
    # so outputs keep 2e-2 and the gradients that crossed the whole chain get 5e-2.
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    gtol = 1e-4 if dtype == torch.float32 else 5e-2
    with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        feats, logits = net(fus(fw, fs))
    cmp.check("feats", feats, g["features"], tol, cmp.UTT)
    cmp.check("logits", logits, g["logits"], tol, cmp.UTT)
    cl = torch.tensor(g["cot_logits"], device="cuda", dtype=logits.dtype)
    cf = torch.tensor(g["cot_features"], device="cuda", dtype=feats.dtype)
    ((logits * cl).sum() + (feats * cf).sum()).float().backward()
    cmp.check("d f_wavlm[::5]", fw.grad.reshape(-1)[::5], g["grad5.f_wavlm"], gtol)
    cmp.check("d f_sinc", fs.grad, g["grad.f_sinc"], gtol, cmp.frames())
    for name, p in list(net.named_parameters()) + [("fusion." + n, p) for n, p in fus.named_parameters()]:
        if name == "attention_pool.bias":       # true gradient is 0 (softmax shift invariance)
            assert float(p.grad.abs().max()) < (1e-5 if dtype == torch.float32 else 1e-3)
        elif name.startswith("backbone_layers."):   # every 5th element of the flattened gradient: no structure to slice
            cmp.check(name + "[::5]", p.grad.reshape(-1)[::5], g["grad5." + name], gtol)
        else:
            cmp.check(name, p.grad, g["grad." + name], gtol, cmp.param(name, p.shape))
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        feats2, logits2 = net(fus(fw, fs))                     # scoring path: head in one launch
    cmp.check("scoring feats", feats2, g["features"], tol, cmp.UTT)
    cmp.check("scoring logits", logits2, g["logits"], tol, cmp.UTT)


def test_reference_unfused_forward_through_shim_equals_fused():
    """The reference's own PN_BiMambas_Encoder.forward (DualStreamSEMamba.py:467-486): two single-direction
    `mamba_ssm...Mamba` calls, two flips and an add, with nn.LayerNorm / nn.Sequential from torch - run through
    install_mamba_ssm_shim() - equals this package's fused encoder layer, outputs and every gradient."""
    import sys
    bm.install_mamba_ssm_shim()
    RefMamba = sys.modules["mamba_ssm.modules.mamba_simple"].Mamba
    assert RefMamba is bm.Mamba
    torch.manual_seed(11)
    enc = bm.PN_BiMambas_Encoder(144, 16).cuda()
    with torch.no_grad():
        enc.mamba.A_log.add_(0.1 * torch.randn_like(enc.mamba.A_log))
    x = torch.randn(3, 201, 144, device="cuda")
    cot = torch.randn(3, 201, 144, device="cuda")

    def reference_forward(m, xin):          # DualStreamSEMamba.py:467-486, verbatim dataflow on the module's attributes
        residual = xin
        x_norm = m.norm1(xin)
        x_f = m.mamba(x_norm)
        x_b = torch.flip(m.mamba(torch.flip(x_norm, dims=[1])), dims=[1])
        out = m.norm2(x_f + x_b)
        return m.feed_forward(out) + residual

    res = []
    for fn in (lambda xin: enc(xin), lambda xin: reference_forward(enc, xin)):
        for p in enc.parameters():
            p.grad = None
        xi = x.clone().requires_grad_(True)
        out = fn(xi)
        out.backward(cot)
        res.append([out.detach(), xi.grad] + [p.grad.clone() for p in enc.parameters()])
    for a, b in zip(*res):
        assert cmp.rel(a, b) < 1e-4


def test_block_fp16_autocast_with_grad_scaler_vs_oracle():
    """The reference trains under fp16 autocast + GradScaler (src/main.py:28, :486, :1049, :1077): scaled loss backward,
    unscale_, clip, step.  Unscaled gradients against the fp64 oracle (fp16 I/O, fp32 state): 5e-3 relative."""
    p64 = orc.init_mamba_params(144, 16, seed=4, dtype=torch.float64)
    m = bm.Mamba(144, 16).cuda()
    _load_mamba(m, {k: v.numpy() for k, v in p64.items()})
    g = torch.Generator().manual_seed(4)
    x = torch.randn(4, 201, 144, generator=g)
    cot = torch.randn(4, 201, 144, generator=g) / (4 * 201 * 144)
    pr = {k: v.float().double().requires_grad_(True) for k, v in p64.items()}
    xr = x.double().requires_grad_(True)
    ref = orc.bimamba_ref(pr, xr)
    (ref * cot.double()).sum().backward()
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 14)
    opt = torch.optim.SGD(m.parameters(), lr=0.0)
    xd = x.cuda().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.float16):
        out = m.forward_bidirectional(xd)
        loss = (out.float() * cot.cuda()).sum()
    assert out.dtype == torch.float16
    cmp.check("out", out, ref, 5e-3, cmp.frames())
    scaler.scale(loss).backward()
    scaler.unscale_(opt)
    total = torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=3.0)     # src/main.py:1104
    assert torch.isfinite(total)
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() == 2.0 ** 14                                    # no inf / nan was found
    clip = min(1.0, 3.0 / (float(total) + 1e-6))
    _check_params(m.named_parameters(), {k: v.grad * clip for k, v in pr.items()}, 5e-3)


def test_head_pool_training_vs_oracle():
    """norm_f + attention pooling under autograd (HeadPoolFn: one launch forward, one backward) against the oracle's
    composition (DualStreamSEMamba.py:759-763): features and gradients w.r.t. the frames and all four parameters."""
    head = orc.init_head_params(144, seed=9, dtype=torch.float64)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(5, 201, 144, generator=g)
    cot = torch.randn(5, 144, generator=g)
    hp = {k: v.clone().requires_grad_(True) for k, v in head.items()}
    xr = x.double().requires_grad_(True)
    xn = torch.nn.functional.layer_norm(xr, (144,), hp["norm_f.weight"], hp["norm_f.bias"], 1e-5)
    a = torch.softmax(xn @ hp["attention_pool.weight"].t() + hp["attention_pool.bias"], dim=1)
    f_ref = (a.transpose(1, 2) @ xn).squeeze(1)
    (f_ref * cot.double()).sum().backward()
    dev = {k: v.float().cuda().requires_grad_(True) for k, v in head.items()}
    xd = x.cuda().requires_grad_(True)
    f = bm.ops.head_pool_fn(xd, dev["norm_f.weight"], dev["norm_f.bias"], dev["attention_pool.weight"],
                            dev["attention_pool.bias"])
    cmp.check("feats", f, f_ref, 1e-5, cmp.UTT)
    f.backward(cot.cuda())
    cmp.check("dx", xd.grad, xr.grad, 1e-4, cmp.frames())
    for k in ("norm_f.weight", "norm_f.bias", "attention_pool.weight"):
        cmp.check(k, dev[k].grad, hp[k].grad, 1e-4, cmp.param(k, hp[k].shape))
    assert float(dev["attention_pool.bias"].grad.abs().max()) < 1e-5


def test_eer_identity_full_scoring_set():
    """SURVEY 8c: ~2 000 utterances x (201, 144).  fp32: scores within 1e-4 and the IDENTICAL EER (rank statistic);
    bf16 (config 4's headline precision): score max-abs-diff and EER are reported and bounded (2e-2 of the score range,
    EER within 0.5 % absolute).  The fp64 oracle's python loop runs on the GPU (same code, device-agnostic)."""
    n_utt, L = 2000, 201
    layers = [orc.init_encoder_params(144, 16, seed=20 + i) for i in range(4)]
    head = orc.init_head_params(144, seed=5)
    g = torch.Generator().manual_seed(2021)
    feats = torch.randn(n_utt, L, 144, generator=g)
    labels = (torch.rand(n_utt, generator=g) < 0.1).numpy()
    with torch.no_grad():
        lay_d = [{k: v.double().cuda() for k, v in p.items()} for p in layers]
        head_d = {k: v.double().cuda() for k, v in head.items()}
        s_ref = torch.cat([orc.backend_ref(lay_d, head_d, feats[i:i + 500].double().cuda())[1][:, 1]
                           for i in range(0, n_utt, 500)]).cpu().numpy()
    net = bm.BiMambaBackend(144, 4, 16).cuda().eval()
    sd = {}
    for i, p in enumerate(layers):
        for k, v in p.items():
            sd[f"backbone_layers.{i}.{k}"] = v
    sd.update(head)
    net.load_state_dict(sd, strict=True)
    eer_ref, _ = orc.compute_eer_ref(s_ref[labels], s_ref[~labels])
    out = {}
    for name, dtype in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        with torch.no_grad(), torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
            s = torch.cat([net(feats[i:i + 256].cuda())[1][:, 1].float() for i in range(0, n_utt, 256)])
        s = s.cpu().numpy().astype(np.float64)
        eer, _ = orc.compute_eer_ref(s[labels], s[~labels])
        out[name] = (float(np.abs(s - s_ref).max()), eer)
    print("EER identity set:", {"ref_eer": eer_ref, **out})
    scale = max(1.0, float(np.abs(s_ref).max()))
    assert out["fp32"][0] < 1e-4 * scale and out["fp32"][1] == eer_ref
    assert out["bf16"][0] < 2e-2 * scale and abs(out["bf16"][1] - eer_ref) < 5e-3


def test_fused_adamw_state_dict_round_trip_and_missing_grads():
    """ADVICE r1: the optimizer state must survive state_dict() / load_state_dict() (moments AND the step counter), and
    parameters without a gradient are skipped like torch.optim.AdamW does."""
    g = torch.Generator().manual_seed(3)
    shapes = [(64, 32), (100,), (7, 5)]
    mk = lambda: [torch.randn(s, generator=torch.Generator().manual_seed(1)).cuda().requires_grad_(True) for s in shapes]
    a_p, b_p, r_p = mk(), mk(), mk()
    a = bm.FusedAdamW(a_p, lr=1e-2, weight_decay=0.1)
    ref = torch.optim.AdamW(r_p, lr=1e-2, weight_decay=0.1)
    grads = [[torch.randn(s, generator=g).cuda() for s in shapes] for _ in range(6)]

    def feed(params, gs, skip_last=False):
        for i, (p, gr) in enumerate(zip(params, gs)):
            p.grad = None if (skip_last and i == len(params) - 1) else gr.clone()
    for it in range(3):
        feed(a_p, grads[it]); a.step()
        feed(r_p, grads[it]); ref.step()
    sd = a.state_dict()
    assert float(sd["state"][0]["step"]) == 3.0
    b = bm.FusedAdamW(b_p, lr=1e-2, weight_decay=0.1)
    with torch.no_grad():
        for q, p in zip(b_p, a_p):
            q.copy_(p)
    b.load_state_dict(sd)                       # resume into a fresh optimizer BEFORE its first step
    for it in range(3, 6):
        feed(b_p, grads[it]); b.step()
        feed(r_p, grads[it]); ref.step()
    for q, r in zip(b_p, r_p):
        assert cmp.rel(q, r) < 1e-6
    # a torch.optim.AdamW state_dict loads too
    c_p = mk()
    c = bm.FusedAdamW(c_p, lr=1e-2, weight_decay=0.1)
    with torch.no_grad():
        for q, p in zip(c_p, r_p):
            q.copy_(p)
    c.load_state_dict(ref.state_dict())
    feed(c_p, grads[0]); c.step()
    feed(r_p, grads[0]); ref.step()
    for q, r in zip(c_p, r_p):
        assert cmp.rel(q, r) < 1e-6
    # a parameter without a gradient is left untouched
    before = c_p[-1].detach().clone()
    feed(c_p, grads[1], skip_last=True); c.step()
    assert torch.equal(c_p[-1], before)


def test_graphed_train_step_construction_does_not_train():
    """ADVICE r1: building the runner (3 warm-up steps) must not move the weights, the moments or the step count."""
    torch.manual_seed(2)
    net = bm.BiMambaBackend(144, 1, 16).cuda()
    params = list(net.backbone_layers.parameters())
    opt = bm.FusedAdamW(params, lr=1e-2)
    before = [p.detach().clone() for p in params]

    def zero():
        for p in params:
            p.grad = None

    def loss_fn(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return net.forward_features(x).float().square().mean()
    runner = bm.GraphedTrainStep(loss_fn, torch.randn(2, 40, 144, device="cuda"), zero, opt, warmup=3)
    for p, q in zip(params, before):
        assert torch.equal(p, q)
    assert float(opt.state_dict()["state"][0]["step"]) == 0.0
    runner.run()
    torch.cuda.synchronize()
    assert float(opt.state_dict()["state"][0]["step"]) == 1.0
    assert any(not torch.equal(p, q) for p, q in zip(params, before))


def test_fgm_step_backend_gradients_vs_oracle():
    """One FGM micro-step of the reference loop (src/main.py:1077-1098) on the CUDA backend: clean backward, attack on the
    `feature_projection` parameter upstream of the backend, adversarial forward / backward, restore - both passes
    accumulating into FlatGradBucket(accumulate=True).  The accumulated gradients of every backend parameter equal the
    fp64 oracle's clean + adversarial gradients (fp32, 1e-4)."""
    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(21)
            self.feature_projection = torch.nn.Linear(24, 144)
            self.tail = bm.BiMambaBackend(144, 2, 16)

        def forward(self, x):
            return self.tail(self.feature_projection(x))

    net = Net().cuda().eval()                         # eval: dropout off, the training head is still taken (grad mode on)
    g = torch.Generator().manual_seed(22)
    x = torch.randn(3, 50, 24, generator=g)
    y = torch.randint(0, 2, (3,), generator=g)
    wce = torch.tensor([0.1, 0.9])
    params = [p for p in net.parameters()]
    bucket = bm.FlatGradBucket(params, accumulate=True)
    fgm = bm.FGM(net, "feature_projection", epsilon=0.5)
    bucket.zero()
    loss = torch.nn.functional.cross_entropy(net(x.cuda())[1].float(), y.cuda(), weight=wce.cuda())
    loss.backward()
    fgm.attack()
    adv = torch.nn.functional.cross_entropy(net(x.cuda())[1].float(), y.cuda(), weight=wce.cuda())
    adv.backward()
    fgm.restore()

    # oracle: same two passes in fp64
    sd = {k: v.detach().double().cpu() for k, v in net.state_dict().items()}
    W = sd["feature_projection.weight"].clone().requires_grad_(True)
    b = sd["feature_projection.bias"].clone().requires_grad_(True)
    layers = [{k[len(f"tail.backbone_layers.{i}."):]: v.clone().requires_grad_(True) for k, v in sd.items()
               if k.startswith(f"tail.backbone_layers.{i}.")} for i in range(2)]
    head = {k[len("tail."):]: v.clone().requires_grad_(True) for k, v in sd.items()
            if k.startswith(("tail.norm_f", "tail.attention_pool", "tail.classifier"))}
    leaves = [W, b] + [v for p in layers for v in p.values()] + list(head.values())

    def run(Wv, bv):
        f = x.double() @ Wv.t() + bv
        return torch.nn.functional.cross_entropy(orc.backend_ref(layers, head, f)[1], y, weight=wce.double())
    g1 = torch.autograd.grad(run(W, b), leaves)
    Wa = (W + 0.5 * g1[0] / g1[0].norm()).detach()
    ba = (b + 0.5 * g1[1] / g1[1].norm()).detach()
    W2, b2 = Wa.clone().requires_grad_(True), ba.clone().requires_grad_(True)
    leaves2 = [W2, b2] + leaves[2:]
    g2 = torch.autograd.grad(run(W2, b2), leaves2)
    want = {}
    names = ["feature_projection.weight", "feature_projection.bias"]
    names += [f"tail.backbone_layers.{i}.{k}" for i, p in enumerate(layers) for k in p]
    names += ["tail." + k for k in head]
    for n, a1, a2 in zip(names, g1, g2):
        want[n] = a1 + a2
    assert cmp.rel(adv, run(W2, b2)) < 1e-4
    for n, p in net.named_parameters():
        if n == "tail.attention_pool.bias":
            assert float(p.grad.abs().max()) < 1e-5
        else:
            cmp.check(n, p.grad, want[n], 1e-4, cmp.param(n, p.shape))
    assert torch.equal(net.feature_projection.weight.detach().cpu().double(), sd["feature_projection.weight"])   # restored
