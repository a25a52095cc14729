"""Variable-length DualStreamFusion on the GPU: the interpolation, SE mean and SE scale kernels against torch on every
utterance alone, the module with lengths (scoring and mask_padding=True training) against the fp64 oracle run per
utterance, the model tail (fusion -> 4-layer backend -> head) with lengths from real clip sample counts, full lengths
against the reference fixtures and the fixed-length module, and one captured graph serving every length mix.

Tolerances as elsewhere: 1e-4 fp32, 2e-2 bf16 (5e-2 for bf16 gradients that cross the whole tail), measured per slice
(oracle/compare.py) against the oracle: every utterance and 8-frame chunk, every parameter gradient per its blocks."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bimamba_b200 as bm
from bimamba_b200 import ops
from oracle import compare as cmp
from oracle.varlen_fusion_oracle import (fusion_loss_and_grads_ref, fusion_one_ref, fusion_varlen_ref, tail_fn,
                                         tail_varlen_ref)

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
EPS = {torch.float32: 2.0 ** -23, torch.bfloat16: 2.0 ** -7, torch.float16: 2.0 ** -10}
# (n1, n2) per utterance, padded to (125, 30): n1 == n2 (copy), 1 frame each, n1 == 4 n2 (linear), 4 n2 + 1 (nearest),
# a linear downsample (n1 < n2), the full padded shape (nearest), and (110, 16): a 2.21 s clip, where fp32 and fp64
# nearest rules pick different frames
PAIRS = [(30, 30), (1, 1), (120, 30), (121, 30), (5, 30), (125, 30), (110, 16), (7, 3)]


def wavlm_frames(S):
    return (S - 400) // 320 + 1


def sinc_frames(S):
    n = (S - 128) // 3
    for _ in range(6):
        n //= 3
    return n


def _interp_torch(x, n1):
    """F.interpolate of one utterance x (n2, C) onto n1 frames by the reference's rule, in x's dtype on the GPU."""
    n2 = x.shape[0]
    if n1 == n2:
        return x
    kw = {"mode": "nearest"} if n1 > 4 * n2 else {"mode": "linear", "align_corners": False}
    return F.interpolate(x.t().unsqueeze(0), size=n1, **kw)[0].t()


def _padded(pairs, C, dtype, seed, fill=float("nan")):
    g = torch.Generator().manual_seed(seed)
    T1, T2 = max(p[0] for p in pairs), max(p[1] for p in pairs)
    src = torch.randn(len(pairs), T2, C, generator=g)
    for b, (_, n2) in enumerate(pairs):
        src[b, n2:] = fill
    l1 = torch.tensor([p[0] for p in pairs], dtype=torch.int32, device="cuda")
    l2 = torch.tensor([p[1] for p in pairs], dtype=torch.int32, device="cuda")
    return src.to(dtype).cuda(), l1, l2, T1, T2


# ------------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [144, 13])
def test_interp_forward_matches_f_interpolate_per_utterance(dtype, C):
    """One batch mixing copy, nearest, linear up and linear down: nearest and copy bit for bit, linear within one unit in
    the last place of the output type (measured on |w0 x0| + |w1 x1|, the size of the two terms); padded destination
    frames exactly 0 and NaN in padded source frames reaches nothing.  C = 13 runs the scalar path."""
    src, l1, l2, T1, T2 = _padded(PAIRS, C, dtype, seed=1)
    out = ops.interp_frames(src, l1, l2, T1)
    assert out.shape == (len(PAIRS), T1, C) and out.dtype == dtype
    for b, (n1, n2) in enumerate(PAIRS):
        x = src[b, :n2]
        ref = _interp_torch(x, n1)
        got = out[b, :n1]
        if n1 == n2 or n1 > 4 * n2:
            assert torch.equal(got, ref), (n1, n2)
        else:
            bound = EPS[dtype] * _interp_torch(x.float().abs(), n1)
            assert bool(((got.float() - ref.float()).abs() <= bound).all()), (n1, n2)
        assert bool((out[b, n1:] == 0).all())
    assert torch.isfinite(out).all()


@pytest.mark.parametrize("dtype", DTYPES)
def test_interp_backward_matches_autograd_and_is_repeatable(dtype):
    """Gather-form backward against fp32 autograd of F.interpolate per utterance; frames >= n2 get 0, NaN cotangents
    at padded destination frames are never read, and two runs give the same bits.  The reference runs on the CPU: its
    backward is the adjoint of the forward's index rule, while the CUDA backward of nearest mode finds its destination
    ranges with ceil(j * n1 / n2) and so moves a frame at pairs such as (110, 16), where the forward reads source 7 at
    frame 55 and the CUDA backward credits source 8."""
    C = 144
    src, l1, l2, T1, T2 = _padded(PAIRS, C, dtype, seed=2, fill=0.0)
    g = torch.Generator().manual_seed(3)
    cot = torch.randn(len(PAIRS), T1, C, generator=g)
    for b, (n1, _) in enumerate(PAIRS):
        cot[b, n1:] = float("nan")
    cot = cot.to(dtype).cuda()
    s = src.clone().requires_grad_(True)
    ops.interp_frames(s, l1, l2, T1).backward(cot)
    d1 = s.grad.clone()
    s.grad = None
    ops.interp_frames(s, l1, l2, T1).backward(cot)
    assert torch.equal(d1, s.grad)
    tol = 1e-6 if dtype == torch.float32 else 2 * EPS[dtype]
    for b, (n1, n2) in enumerate(PAIRS):
        x = src[b, :n2].float().cpu().requires_grad_(True)
        _interp_torch(x, n1).backward(cot[b, :n1].float().cpu())
        assert cmp.rel(d1[b, :n2], x.grad) < tol, (n1, n2)
        assert bool((d1[b, n2:] == 0).all())


@pytest.mark.parametrize("dtype", DTYPES)
def test_frame_mean_and_scale_match_torch_per_utterance(dtype):
    lengths = [1, 64, 65, 130, 7, 0]
    Bsz, T, C = len(lengths), 130, 144
    g = torch.Generator().manual_seed(4)
    x = torch.randn(Bsz, T, C, generator=g)
    for b, n in enumerate(lengths):
        x[b, n:] = float("nan")
    x = x.to(dtype).cuda()
    sl = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    gate = torch.rand(Bsz, C, generator=g).cuda()
    dy = torch.randn(Bsz, T, C, generator=g).to(dtype).cuda()
    dmean = torch.randn(Bsz, C, generator=g).cuda()
    xr = x.clone().requires_grad_(True)
    gr = gate.clone().requires_grad_(True)
    mean = ops.frame_mean(xr, sl)
    y = ops.frame_scale(xr, gr, sl)
    tol = 1e-5 if dtype == torch.float32 else 2 * EPS[dtype]
    for b, n in enumerate(lengths):
        xb = x[b, :n].float()
        assert cmp.rel(mean[b], xb.mean(0) if n else torch.zeros(C)) < 1e-5
        assert torch.equal(y[b, :n], (xb * gate[b]).to(dtype))
        assert bool((y[b, n:] == 0).all())
    torch.autograd.backward([mean, y], [dmean, dy])
    for b, n in enumerate(lengths):
        dgr = (dy[b, :n].float() * x[b, :n].float()).sum(0)
        assert (cmp.rel(gr.grad[b], dgr) < 1e-5) if n else bool((gr.grad[b] == 0).all())
        if n:
            dxr = dy[b, :n].float() * gate[b] + dmean[b] / n
            assert cmp.rel(xr.grad[b, :n], dxr) < tol
        assert bool((xr.grad[b, n:] == 0).all())
    g1 = gr.grad.clone()
    gr.grad = None
    ops.frame_scale(xr, gr, sl).backward(dy)
    assert torch.equal(gr.grad, g1)


# -------------------------------------------------------------------------------------------------------------- module
def _module(seed=0):
    torch.manual_seed(seed)
    fus = bm.DualStreamFusion(1024, 64, 144).cuda()
    with torch.no_grad():
        for n in ("ln_wavlm", "ln_sinc", "norm"):
            m = getattr(fus, n)
            m.weight.add_(0.1 * torch.randn_like(m.weight))
            m.bias.add_(0.1 * torch.randn_like(m.bias))
    return fus


def _streams(pairs, seed, fill):
    g = torch.Generator().manual_seed(seed)
    T1, T2 = max(p[0] for p in pairs), max(p[1] for p in pairs)
    fw = torch.randn(len(pairs), T1, 1024, generator=g)
    fs = torch.randn(len(pairs), T2, 64, generator=g)
    for b, (n1, n2) in enumerate(pairs):
        fw[b, n1:] = fill
        fs[b, n2:] = fill
    return fw.cuda(), fs.cuda(), [p[0] for p in pairs], [p[1] for p in pairs]


def _p64(mod, prefix=""):
    return {prefix + k: v.detach().double().cpu() for k, v in mod.state_dict().items()}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_module_scoring_matches_oracle(dtype):
    fus = _module().eval()
    fw, fs, l1, l2 = _streams(PAIRS, seed=5, fill=float("nan"))
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        out = fus(fw, fs, l1, l2)
    assert out.dtype == torch.float32
    ref = fusion_varlen_ref(_p64(fus), fw.double().cpu(), fs.double().cpu(), l1, l2)
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    for b, n1 in enumerate(l1):
        cmp.check(f"out{PAIRS[b]}", out[b, :n1], ref[b, :n1], tol, [{0: cmp.CHUNK}])


@pytest.mark.parametrize("fill", [float("nan"), 1e4])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_module_mask_padding_training_matches_oracle(dtype, fill):
    """Output, grad f_wavlm, grad f_sinc and every parameter gradient against the per-utterance fp64 oracle (summed
    over utterances); padded outputs and padded input gradients exactly 0; NaN / 1e4 padding and NaN cotangents at
    padded output frames reach nothing."""
    fus = _module(1).train()
    fus.dropout.p = 0.0
    fw, fs, l1, l2 = _streams(PAIRS, seed=6, fill=fill)
    g = torch.Generator().manual_seed(7)
    cot = torch.randn(len(PAIRS), fw.shape[1], 144, generator=g, dtype=torch.float64)
    cot_pad = cot.clone()
    for b, n1 in enumerate(l1):
        cot[b, n1:] = 0
        cot_pad[b, n1:] = float("nan")
    fwr, fsr = fw.clone().requires_grad_(True), fs.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        out = fus(fwr, fsr, l1, l2, mask_padding=True)
    out.backward(cot_pad.float().cuda())
    loss_fn = lambda o, idx, n1, n2: (o * cot[idx, :n1]).sum()                       # noqa: E731
    _, grads, dfw, dfs = fusion_loss_and_grads_ref(fusion_one_ref, _p64(fus), fw, fs, l1, l2, loss_fn)
    ref = fusion_varlen_ref(_p64(fus), fw.double().cpu(), fs.double().cpu(), l1, l2)
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    gtol = 1e-4 if dtype == torch.float32 else 5e-2
    for b, (n1, n2) in enumerate(PAIRS):
        assert bool((out[b, n1:] == 0).all()) and bool((fwr.grad[b, n1:] == 0).all()) and bool((fsr.grad[b, n2:] == 0).all())
    cmp.check("out", out, ref, tol, cmp.frames())
    cmp.check("d f_wavlm", fwr.grad, dfw, gtol, cmp.frames())
    cmp.check("d f_sinc", fsr.grad, dfs, gtol, cmp.frames())
    for name, p in fus.named_parameters():
        assert torch.isfinite(p.grad).all(), name
        cmp.check(name, p.grad, grads[name], gtol, cmp.param(name, p.shape))


def test_module_full_lengths_match_fixed_length_path():
    """lengths == T1 and sinc_lengths == T2: the interpolated addend equals the fixed path's F.interpolate bit for bit
    in nearest mode, and the outputs agree to 1e-6 relative in fp32 - not bitwise, because the SE mean sums the frames in
    another order than torch.mean."""
    fus = _module(2).eval()
    for T1, T2 in ((201, 29), (60, 14)):
        fw, fs, l1, l2 = _streams([(T1, T2)] * 3, seed=8, fill=0.0)
        with torch.no_grad():
            a = fus(fw, fs)
            b = fus(fw, fs, l1, l2)
            s2 = torch.randn(3, T2, 144, device="cuda")
            mine = ops.interp_frames(s2, ops.seqlens_tensor(l1, 3, T1, "cuda"), ops.seqlens_tensor(l2, 3, T2, "cuda"), T1)
            mode = "nearest" if T1 / T2 > 4.0 else "linear"
            kw = {} if mode == "nearest" else {"align_corners": False}
            theirs = F.interpolate(s2.transpose(1, 2), size=T1, mode=mode, **kw).transpose(1, 2)
        assert cmp.rel(b, a) < 1e-6
        if mode == "nearest":
            assert torch.equal(mine, theirs)


def _tail_state(g):
    return {k[len("param."):]: torch.tensor(v).float() for k, v in g.items() if k.startswith("param.")}


@pytest.mark.parametrize("tag,dtype", [("linear", torch.float32), ("nearest", torch.float32), ("nearest", torch.bfloat16)])
def test_module_full_lengths_vs_reference_fixture(golden_dir, tag, dtype):
    """The fixtures of test_dual_stream_fusion_vs_reference_fixture through the training form with full lengths."""
    g = dict(np.load(os.path.join(golden_dir, f"model_tail_{tag}.npz")))
    fus = bm.DualStreamFusion(1024, 64, 144, reduction=16).cuda().eval()
    fus.load_state_dict({k[len("fusion."):]: v for k, v in _tail_state(g).items() if k.startswith("fusion.")}, strict=True)
    fw = torch.tensor(g["f_wavlm"], device="cuda", dtype=torch.float32, requires_grad=True)
    fs = torch.tensor(g["f_sinc"], device="cuda", dtype=torch.float32, requires_grad=True)
    B, T1, T2 = fw.shape[0], fw.shape[1], fs.shape[1]
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        out = fus(fw, fs, [T1] * B, [T2] * B, mask_padding=True)
    cmp.check("out", out, g["f_fused"], tol, cmp.frames())
    out.backward(torch.tensor(g["grad.f_fused"], device="cuda", dtype=torch.float32))
    if tag == "linear":
        cmp.check("d f_wavlm", fw.grad, g["grad.f_wavlm"], tol, cmp.frames())
    else:                                      # every 5th element of the flattened gradient: no structure to slice
        cmp.check("d f_wavlm[::5]", fw.grad.reshape(-1)[::5], g["grad5.f_wavlm"], tol)
    cmp.check("d f_sinc", fs.grad, g["grad.f_sinc"], tol, cmp.frames())
    for name, p in fus.named_parameters():
        cmp.check(name, p.grad, g["grad.fusion." + name], tol, cmp.param(name, p.shape))


# ---------------------------------------------------------------------------------------------------------------- tail
def _clips(n, seed, lo_s=1.0, hi_s=10.0):
    g = torch.Generator().manual_seed(seed)
    S = (torch.randint(int(lo_s * 100), int(hi_s * 100) + 1, (n,), generator=g) * 160).tolist()
    return [wavlm_frames(s) for s in S], [sinc_frames(s) for s in S]


@pytest.fixture(scope="module")
def tail_case():
    l1, l2 = _clips(16, seed=9)
    l1[0], l2[0] = 110, 16                                     # a clip where fp32 and fp64 nearest disagree
    fus = _module(3)
    torch.manual_seed(3)
    net = bm.BiMambaBackend(144, 4, 16).cuda()
    fw, fs, _, _ = _streams(list(zip(l1, l2)), seed=10, fill=float("nan"))
    p = _p64(fus, "fusion.")
    p.update(_p64(net))
    g = torch.Generator().manual_seed(11)
    cf, cl = torch.randn(16, 144, generator=g, dtype=torch.float64), torch.randn(16, 2, generator=g, dtype=torch.float64)
    feats, logits = tail_varlen_ref(p, 4, fw.double().cpu(), fs.double().cpu(), l1, l2)
    loss_fn = lambda o, idx, n1, n2: (o[0] * cf[idx]).sum() + (o[1] * cl[idx]).sum()     # noqa: E731
    loss, grads, dfw, dfs = fusion_loss_and_grads_ref(tail_fn(4), p, fw, fs, l1, l2, loss_fn)
    return dict(fus=fus, net=net, fw=fw, fs=fs, l1=l1, l2=l2, cf=cf, cl=cl, feats=feats, logits=logits, loss=loss,
                grads=grads, dfw=dfw, dfs=dfs)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_tail_scoring_matches_oracle(tail_case, dtype):
    c = tail_case
    fus, net = c["fus"].eval(), c["net"].eval()
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        feats, logits = net(fus(c["fw"], c["fs"], c["l1"], c["l2"]), c["l1"])
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    cmp.check("feats", feats, c["feats"], tol, cmp.UTT)
    cmp.check("logits", logits, c["logits"], tol, cmp.UTT)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_tail_training_matches_oracle(tail_case, dtype):
    c = tail_case
    fus, net = c["fus"].train(), c["net"].train()
    fus.dropout.p = 0.0
    for m in net.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    for p in list(fus.parameters()) + list(net.parameters()):
        p.grad = None
    fw, fs = c["fw"].clone().requires_grad_(True), c["fs"].clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        feats, logits = net(fus(fw, fs, c["l1"], c["l2"], mask_padding=True), c["l1"], mask_padding=True)
    loss = (feats.float() * c["cf"].float().cuda()).sum() + (logits.float() * c["cl"].float().cuda()).sum()
    loss.backward()
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    gtol = 1e-4 if dtype == torch.float32 else 5e-2
    assert abs(float(loss.detach()) - float(c["loss"])) <= tol * abs(float(c["loss"])) + tol
    cmp.check("d f_wavlm", fw.grad, c["dfw"], gtol, cmp.frames())
    cmp.check("d f_sinc", fs.grad, c["dfs"], gtol, cmp.frames())
    for b, (n1, n2) in enumerate(zip(c["l1"], c["l2"])):
        assert bool((fw.grad[b, n1:] == 0).all()) and bool((fs.grad[b, n2:] == 0).all())
    named = [("fusion." + n, p) for n, p in fus.named_parameters()] + list(net.named_parameters())
    for name, p in named:
        ref = c["grads"][name]
        if name == "attention_pool.bias":           # exact gradient 0 (softmax shift invariance): on the weight's scale
            assert float(p.grad.abs().max()) <= gtol * float(c["grads"]["attention_pool.weight"].abs().max()), name
        else:
            # bf16: x_proj.weight keeps the whole-tensor rule (rho 1).  On a B200 its column group [:, 256:288] in
            # layer 2, at 0.33 of the tensor's largest element, is 7.4e-2 off, 2.4e-2 of max|ref|: the rounding of its
            # bf16-stored operands (dC and the conv output) after four layers, on a slice too large for a floor
            rho = 1.0 if dtype != torch.float32 and name.endswith("x_proj.weight") else None
            cmp.check(name, p.grad, ref, gtol, cmp.param(name, p.shape), rho=rho)


def test_tail_captured_once_serves_every_length_mix(tail_case):
    """One torch.cuda.graph capture of fusion -> backend -> head over static streams and length buffers; two replays
    with other length mixes equal the eager results bit for bit."""
    c = tail_case
    fus, net = c["fus"].eval(), c["net"].eval()
    fw, fs = c["fw"].nan_to_num(0.0), c["fs"].nan_to_num(0.0)
    l1 = torch.tensor(c["l1"], dtype=torch.int32, device="cuda")
    l2 = torch.tensor(c["l2"], dtype=torch.int32, device="cuda")
    run = lambda: net(fus(fw, fs, l1, l2), l1)                                  # noqa: E731
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static = run()
        mixes = [_clips(16, seed=12), _clips(16, seed=13, lo_s=0.5, hi_s=3.0)]
        for m1, m2 in mixes:
            m1 = [min(v, fw.shape[1]) for v in m1]
            m2 = [min(v, fs.shape[1]) for v in m2]
            l1.copy_(torch.tensor(m1, dtype=torch.int32))
            l2.copy_(torch.tensor(m2, dtype=torch.int32))
            graph.replay()
            got = [t.clone() for t in static]
            eager = net(fus(fw, fs, m1, m2), m1)
            assert all(torch.equal(a, b) for a, b in zip(got, eager))


# -------------------------------------------------------------------------------------------------------------- errors
def test_module_errors():
    fus = _module()
    fw, fs, l1, l2 = _streams([(40, 9), (20, 5)], seed=14, fill=0.0)
    with pytest.raises(ValueError, match="go together"):
        fus(fw, fs, l1)
    with pytest.raises(ValueError, match="go together"):
        fus(fw, fs, sinc_lengths=l2)
    with pytest.raises(ValueError, match="1..40"):
        with torch.no_grad():
            fus(fw, fs, [41, 20], l2)
    with pytest.raises(ValueError, match="1..9"):
        with torch.no_grad():
            fus(fw, fs, l1, [9, 0])
    with pytest.raises(NotImplementedError, match="scoring only"):
        fus(fw, fs, l1, l2)                                  # parameters require grad: autograd is recording
    with pytest.raises(ValueError, match="mask_padding=True needs lengths"):
        fus(fw, fs, mask_padding=True)
