"""Variable-length training on the GPU: the backward of the scan, the conv and the head with per-utterance frame counts,
and the block, encoder layer and backend with mask_padding=True, against the fp64 oracle run on every utterance at its
own length (parameter gradients summed over utterances).  Padding never leaks; lengths == T gives the bits of the
fixed-length path; one captured training step serves every length mix.

Tolerances as elsewhere: 1e-4 fp32, 2e-2 bf16, 5e-3 fp16 at op level; 5e-2 for bf16 end-to-end gradients; measured per
slice (oracle/compare.py), every utterance against its own magnitude."""
import pytest
import torch
import torch.nn.functional as F

import bimamba_b200 as bm
from bimamba_b200 import ops
from oracle import bimamba_oracle as orc
from oracle import compare as cmp
from oracle.varlen_train_oracle import backend_logits_fn, block_fn, layer_fn, varlen_loss_and_grads_ref

pytestmark = pytest.mark.gpu

TOL = cmp.TOL
# shorter than the conv width, around the 8-step checkpoint and 16-step chunk boundaries, and the full padded length
LENGTHS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 40]
LONG = [201, 150, 77, 9, 201, 33]
N, XW = 16, 48


def check_grad(name, got, grads_ref, tol):
    """A parameter gradient per slice; the attention-pool bias gets an exact gradient of zero (the softmax does not
    change when every logit moves by the same amount), so it is measured on the scale of the attention weight's."""
    if "attention_pool.bias" in name or name == "ab":
        w = name.replace("bias", "weight") if name != "ab" else "aw"
        err = float(got.detach().double().abs().max().cpu() / grads_ref[w].abs().max().clamp_min(1e-30).cpu())
        assert err < tol, (name, err)
        return
    cmp.check(name, got, grads_ref[name], tol, cmp.param(name, got.shape))


def _pad_mask(lengths, T, dev="cuda"):
    return torch.arange(T, device=dev).unsqueeze(0) >= torch.tensor(lengths, device=dev).unsqueeze(1)   # (B, T) padded


# ---------------------------------------------------------------------------------------------------------------- scan
def _scan_case(mode, dtype, lengths, D=40, ndir=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    Bsz, L, R, dev = len(lengths), max(lengths), mode, "cuda"
    pad = _pad_mask(lengths, L).cpu()
    nanpad = lambda t: t.masked_fill(pad.view(Bsz, 1, L, 1) if t.dim() == 4 else pad.view(Bsz, L, 1), float("nan"))
    xc = ops.per_dir(Bsz, L, ndir, D, dev, dtype)
    xc.copy_(nanpad(torch.randn(Bsz, ndir, L, D, generator=g)).to(dtype))
    xdbl = torch.zeros((Bsz, L, ndir, XW), dtype=dtype)
    xdbl[..., :2 * N] = torch.randn(Bsz, L, ndir, 2 * N, generator=g).to(dtype)
    if R:
        xdbl[..., 2 * N:2 * N + R] = (torch.randn(Bsz, L, ndir, R, generator=g) * 0.5).to(dtype)
    xdbl = xdbl.masked_fill(pad.view(Bsz, L, 1, 1), float("nan"))
    xd4 = xdbl.to(dev).permute(0, 2, 1, 3)
    bc, dtr = xd4[..., :2 * N], (xd4[..., 2 * N:] if R else None)
    Wdt = (torch.randn(D, R, generator=g) / R ** 0.5).to(dev) if R else None
    delta = None
    if not R:
        delta = ops.per_dir(Bsz, L, ndir, D, dev, dtype)
        delta.copy_(nanpad(0.5 * torch.randn(Bsz, ndir, L, D, generator=g)).to(dtype))
    z = nanpad(torch.randn(Bsz, L, D, generator=g)).to(dtype).to(dev)
    z4 = z.unsqueeze(1).expand(Bsz, ndir, L, D)
    A = (-torch.exp(torch.log(torch.arange(1, N + 1, dtype=torch.float32)).repeat(D, 1)
                    + 0.1 * torch.randn(D, N, generator=g))).to(dev)
    Dp = (1 + 0.1 * torch.randn(D, generator=g)).to(dev)
    dt = torch.exp(torch.rand(D, generator=g) * 4.6 - 6.9)
    bias = (dt + torch.log(-torch.expm1(-dt))).to(dev)
    dout = ops.per_dir(Bsz, L, ndir, D, dev, dtype)
    dout.copy_(nanpad(torch.randn(Bsz, ndir, L, D, generator=g)).to(dtype))
    sl = ops.seqlens_tensor(lengths, Bsz, L, dev)

    out, ckpt, ypre = ops.scan_fwd_raw(xc, z4, delta, bc, dtr, Wdt, A, Dp, bias, True, True, dtr_padded=True,
                                       seqlens=sl)
    run = lambda: ops.scan_bwd_raw(xc, z4, delta, bc, dtr, Wdt, A, Dp, bias, True, dout, ckpt, ypre, dtr_padded=True,
                                   bc_out_dtype=torch.float32, seqlens=sl)
    got = run()
    again = run()
    torch.cuda.synchronize()
    for a, b in zip(got, again):
        assert torch.equal(a, b), "backward is not bitwise repeatable"
    du, ddelta, dz, dbc, dA, dD, dbias = got
    padded = pad.view(Bsz, 1, L, 1).to(dev)
    for name, t in (("out", out), ("ypre", ypre), ("du", du), ("ddelta", ddelta), ("dz", dz), ("dB|dC", dbc)):
        assert bool((t.masked_select(padded) == 0).all()), f"{name} is not zero at padded frames"

    A64 = A.double().cpu().requires_grad_(True)
    D64 = Dp.double().cpu().requires_grad_(True)
    b64 = bias.double().cpu().requires_grad_(True)
    tol, act, state = TOL[dtype], cmp.scan_act(0, 2, 1), cmp.scan_state(0, 2)     # (1, n, D) / (1, n, 2N) pieces
    for b, n in enumerate(lengths):
        for di in range(ndir):
            fl = (lambda t: t.flip(-1)) if di else (lambda t: t)
            cut = lambda t: t[b:b + 1, :n].double().cpu().transpose(1, 2)
            u_d = fl(cut(xc[:, di])).requires_grad_(True)
            draw = (xd4[b:b + 1, di, :n, 2 * N:2 * N + R].double().cpu() @ Wdt.double().cpu().t()) if R else \
                delta[b:b + 1, di, :n].double().cpu()
            dl_d = fl(draw.transpose(1, 2)).detach().requires_grad_(True)
            z_d = fl(cut(z)).requires_grad_(True)
            bc_d = fl(cut(bc[:, di])).requires_grad_(True)
            y = orc.selective_scan_ref(u_d, dl_d, A64, bc_d[:, :N], bc_d[:, N:], D64, z_d, b64, delta_softplus=True)
            k = f"{b}.{di}"
            cmp.check("out" + k, out[b:b + 1, di, :n], fl(y).transpose(1, 2), tol, act)
            (y * fl(cut(dout[:, di]))).sum().backward()
            cmp.check("du" + k, du[b:b + 1, di, :n], fl(u_d.grad).transpose(1, 2), tol, act)
            cmp.check("ddelta" + k, ddelta[b:b + 1, di, :n], fl(dl_d.grad).transpose(1, 2), tol, act)
            cmp.check("dz" + k, dz[b:b + 1, di, :n], fl(z_d.grad).transpose(1, 2), tol, act)
            cmp.check("dB|dC" + k, dbc[b:b + 1, di, :n], fl(bc_d.grad).transpose(1, 2), tol, state)
    cmp.check("dA", dA, A64.grad, tol, cmp.CHANNEL_STATE)
    cmp.check("dD", dD, D64.grad, tol, cmp.CHANNELS)
    cmp.check("dbias", dbias, b64.grad, tol, cmp.CHANNELS)


@pytest.mark.parametrize("variant", [1, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mode", [0, 9, 16])
def test_scan_varlen_forward_and_backward(mode, dtype, variant):
    """Checkpointed forward (both forward kernels, forced) and backward with lengths against the oracle per utterance;
    the padding holds NaN; padded gradients are exactly zero and a second backward gives the same bits."""
    with bm._lib.tuning(bm._lib.TUNE_SCAN_FWD, variant):
        _scan_case(mode, dtype, LENGTHS, seed=10 * mode + variant)


def test_scan_varlen_long_mixed():
    _scan_case(9, torch.bfloat16, LONG, seed=5)


# ---------------------------------------------------------------------------------------------------------------- conv
@pytest.mark.parametrize("kernel,width", [("seg", 4), ("tile", 2), ("tile", 3), ("tile", 4)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_conv_varlen_backward(kernel, width, dtype):
    g = torch.Generator().manual_seed(width)
    lengths, D, ndir = LENGTHS, 64, 2
    Bsz, L = len(lengths), max(lengths)
    pad = _pad_mask(lengths, L).cpu()
    x = torch.randn(Bsz, L, D, generator=g).masked_fill(pad.unsqueeze(-1), float("nan")).to(dtype).cuda()
    w = (0.5 * torch.randn(D, width, generator=g)).cuda()
    b = (0.1 * torch.randn(D, generator=g)).cuda()
    go = torch.randn(Bsz, ndir, L, D, generator=g).masked_fill(pad.view(Bsz, 1, L, 1), float("nan"))
    dout = ops.per_dir(Bsz, L, ndir, D, "cuda", dtype)
    dout.copy_(go.to(dtype))
    dz_in = ops.per_dir(Bsz, L, ndir, D, "cuda", dtype)
    dz_in.copy_(torch.randn(Bsz, ndir, L, D, generator=g).masked_fill(pad.view(Bsz, 1, L, 1), float("nan")).to(dtype))
    sl = ops.seqlens_tensor(lengths, Bsz, L, "cuda")
    out = ops.per_dir(Bsz, L, ndir, D, "cuda", dtype)
    ops.conv_fwd_raw(x, w, b, out, True, sl)
    dxz = torch.empty(Bsz, L, 2 * D, device="cuda", dtype=dtype)
    with bm._lib.tuning(bm._lib.TUNE_CONV_BWD, 1 if kernel == "tile" else 0):
        dwb = ops.conv_bwd_raw(x, w, b, dout, dxz[..., :D], True, dz_in=dz_in, dz_out=dxz[..., D:], seqlens=sl)
    torch.cuda.synchronize()
    dx, dz = dxz[..., :D], dxz[..., D:]
    assert bool((dx[pad.cuda()] == 0).all()) and bool((dz[pad.cuda()] == 0).all())
    w64 = w.double().cpu().requires_grad_(True)
    b64 = b.double().cpu().requires_grad_(True)
    tol, act = TOL[dtype], [{1: 1}, {0: cmp.CHUNK}]               # (n, D) pieces: per channel, per 8-step chunk
    for i, n in enumerate(lengths):
        xi = x[i, :n].double().cpu().t().unsqueeze(0).requires_grad_(True)       # (1, D, n)
        o0 = orc.causal_conv1d_ref(xi, w64, b64, "silu")
        o1 = orc.causal_conv1d_ref(xi.flip(-1), w64, b64, "silu").flip(-1)
        (o0 * dout[i, 0, :n].double().cpu().t() + o1 * dout[i, 1, :n].double().cpu().t()).sum().backward()
        cmp.check(f"dx{i}", dx[i, :n], xi.grad[0].t(), tol, act)
        cmp.check(f"dz{i}", dz[i, :n], dz_in[i, :, :n].double().sum(0), tol, act)
    cmp.check("conv1d.weight", dwb[:, :width], w64.grad, tol, cmp.param("conv1d.weight", w64.shape))
    cmp.check("conv1d.bias", dwb[:, width], b64.grad, tol, cmp.CHANNELS)


# ---------------------------------------------------------------------------------------------------------------- head
def test_head_pool_varlen_backward_and_zero_length():
    g = torch.Generator().manual_seed(3)
    C_, lengths = 144, LENGTHS
    Bsz, T = len(lengths), max(lengths)
    pad = _pad_mask(lengths, T).cpu()
    x = torch.randn(Bsz, T, C_, generator=g).masked_fill(pad.unsqueeze(-1), float("nan")).cuda().requires_grad_(True)
    hp = orc.init_head_params(C_, seed=3)
    nw, nb = hp["norm_f.weight"].cuda().requires_grad_(True), hp["norm_f.bias"].cuda().requires_grad_(True)
    aw, ab = hp["attention_pool.weight"].cuda().requires_grad_(True), hp["attention_pool.bias"].cuda().requires_grad_(True)
    df = torch.randn(Bsz, C_, generator=g).cuda()
    sl = ops.seqlens_tensor(lengths, Bsz, T, "cuda")
    (ops.head_pool_fn(x, nw, nb, aw, ab, 1e-5, sl) * df).sum().backward()
    assert bool((x.grad[pad.cuda()] == 0).all())

    def fn(p, xn):
        y = F.layer_norm(xn, (C_,), p["w"], p["b"], 1e-5)
        a = torch.softmax(y @ p["aw"].t() + p["ab"], dim=1)
        return (a.transpose(1, 2) @ y).squeeze(1)
    params = {"w": nw, "b": nb, "aw": aw, "ab": ab}
    _, gr, dx = varlen_loss_and_grads_ref(fn, params, x.detach(), lengths,
                                          lambda f, idx, n: (f * df[idx].double()).sum())
    cmp.check("dx", x.grad, dx, 1e-4, cmp.frames())
    for k, t in params.items():
        check_grad(k, t.grad, gr, 1e-4)

    # a zero-length utterance (a device vector is trusted and clamped): zero gradient, no NaN, no contribution
    x2 = x.detach().clone().requires_grad_(True)
    for t in params.values():
        t.grad = None
    sl0 = torch.tensor([0] + lengths[1:], device="cuda", dtype=torch.int32)
    feats = ops.head_pool_fn(x2, nw, nb, aw, ab, 1e-5, sl0)
    (feats * df).sum().backward()
    assert bool((feats[0] == 0).all()) and bool((x2.grad[0] == 0).all())
    _, gr0, _ = varlen_loss_and_grads_ref(fn, params, x.detach(), [0] + lengths[1:],
                                          lambda f, idx, n: (f * df[idx].double()).sum())
    for k, t in params.items():
        assert torch.isfinite(t.grad).all(), k
        check_grad(k, t.grad, gr0, 1e-4)


# -------------------------------------------------------------------------------------------------- block / layer / net
def _autocast(dtype):
    return torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32)


def _mamba(d_model=144, seed=1):
    p64 = orc.init_mamba_params(d_model, 16, seed=seed, dtype=torch.float64)
    m = bm.Mamba(d_model, 16).cuda()
    m.load_state_dict({k: v.float() for k, v in p64.items()}, strict=True)
    return m, {k: v.float().double().cuda() for k, v in m.state_dict().items()}


def _block_step(m, x, lengths, wout, dtype, sequenced):
    m.zero_grad(set_to_none=True)
    xg = x.clone().requires_grad_(True)
    seq = ops.sequenced_block() if sequenced else ops._NULL
    with _autocast(dtype), seq:
        out = m.forward_bidirectional(xg, lengths, mask_padding=True)
        loss = (out.float() * wout).sum()
    loss.backward()
    return out.detach(), loss.detach(), xg.grad, {k: p.grad.detach().clone() for k, p in m.named_parameters()}


@pytest.mark.parametrize("dtype,sequenced", [(torch.float32, True), (torch.bfloat16, True), (torch.bfloat16, False)])
def test_block_mask_padding_vs_oracle(dtype, sequenced):
    m, p64 = _mamba()
    lengths = LENGTHS
    Bsz, T = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(11)
    pad = _pad_mask(lengths, T)
    x = torch.randn(Bsz, T, 144, generator=g).cuda().masked_fill(pad.unsqueeze(-1), float("nan"))
    wout = torch.randn(Bsz, T, 144, generator=g).cuda()
    out, loss, dx, grads = _block_step(m, x, lengths, wout, dtype, sequenced)
    assert bool((out[pad] == 0).all()) and bool((dx[pad] == 0).all())
    loss_ref, gr, dx_ref = varlen_loss_and_grads_ref(block_fn, p64, x, lengths,
                                                     lambda o, idx, n: (o * wout[idx, :n].double()).sum())
    tol = TOL[dtype] if dtype == torch.float32 else 5e-2
    assert cmp.rel(loss, loss_ref) < TOL[dtype]
    cmp.check("dx", dx, dx_ref, tol, cmp.frames())
    assert len(grads) == 9
    for k, t in grads.items():
        check_grad(k, t, gr, tol)


def test_block_native_and_sequenced_are_bit_identical_with_lengths():
    m, _ = _mamba()
    lengths = LONG
    Bsz, T = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(12)
    x = torch.randn(Bsz, T, 144, generator=g).cuda()
    wout = torch.randn(Bsz, T, 144, generator=g).cuda()
    a = _block_step(m, x, lengths, wout, torch.bfloat16, False)
    b = _block_step(m, x, lengths, wout, torch.bfloat16, True)
    for u, v in zip(a[:3], b[:3]):
        assert torch.equal(u, v)
    for k in a[3]:
        assert torch.equal(a[3][k], b[3][k]), k


def _backend(n_layers=2, seed=30):
    layers = [orc.init_encoder_params(144, 16, seed=seed + i) for i in range(n_layers)]
    head = orc.init_head_params(144, seed=seed)
    net = bm.BiMambaBackend(144, n_layers, 16).cuda().train()
    net.dropout.p = 0.0
    sd = {f"backbone_layers.{i}.{k}": v for i, p in enumerate(layers) for k, v in p.items()}
    sd.update(head)
    net.load_state_dict(sd, strict=True)
    return net, {k: v.double().cuda() for k, v in net.state_dict().items()}


def _net_step(net, x, lengths, labels, dtype, sequenced=False):
    net.zero_grad(set_to_none=True)
    xg = x.clone().requires_grad_(True)
    seq = ops.sequenced_block() if sequenced else ops._NULL
    with _autocast(dtype), seq:
        _, logits = net(xg, lengths, mask_padding=True)
        loss = F.cross_entropy(logits.float(), labels, reduction="sum")
    loss.backward()
    return loss.detach(), xg.grad, {k: p.grad.detach().clone() for k, p in net.named_parameters()}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layer_mask_padding_vs_oracle(dtype):
    p = orc.init_encoder_params(144, 16, seed=40)
    layer = bm.PN_BiMambas_Encoder(144, 16).cuda()
    layer.load_state_dict(p, strict=True)
    p64 = {k: v.double().cuda() for k, v in layer.state_dict().items()}
    lengths = LENGTHS
    Bsz, T = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(41)
    pad = _pad_mask(lengths, T)
    x = torch.randn(Bsz, T, 144, generator=g).cuda().masked_fill(pad.unsqueeze(-1), float("nan"))
    wout = torch.randn(Bsz, T, 144, generator=g).cuda()       # weights padded output frames too: they are zero
    xg = x.clone().requires_grad_(True)
    with _autocast(dtype):
        out = layer(xg, lengths, mask_padding=True)
        loss = (out.float() * wout).sum()
    loss.backward()
    assert bool((out[pad] == 0).all()) and bool((xg.grad[pad] == 0).all())
    loss_ref, gr, dx_ref = varlen_loss_and_grads_ref(layer_fn, p64, x, lengths,
                                                     lambda o, idx, n: (o * wout[idx, :n].double()).sum())
    tol = 1e-4 if dtype == torch.float32 else 5e-2
    assert cmp.rel(loss, loss_ref) < (1e-4 if dtype == torch.float32 else 2e-2)
    cmp.check("dx", xg.grad, dx_ref, tol, cmp.frames())
    for k, t in layer.named_parameters():
        check_grad(k, t.grad, gr, tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_backend_mask_padding_vs_oracle(dtype):
    net, p64 = _backend()
    lengths = LONG
    Bsz, T = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(31)
    pad = _pad_mask(lengths, T)
    x = torch.randn(Bsz, T, 144, generator=g).cuda().masked_fill(pad.unsqueeze(-1), float("nan"))
    labels = torch.randint(0, 2, (Bsz,), generator=g).cuda()
    loss, dx, grads = _net_step(net, x, lengths, labels, dtype)
    assert torch.isfinite(loss) and bool((dx[pad] == 0).all())
    loss_ref, gr, dx_ref = varlen_loss_and_grads_ref(
        backend_logits_fn(2), p64, x, lengths, lambda lg, idx, n: F.cross_entropy(lg, labels[idx], reduction="sum"))
    tol = 1e-4 if dtype == torch.float32 else 5e-2
    assert cmp.rel(loss, loss_ref) < (1e-4 if dtype == torch.float32 else 2e-2)
    cmp.check("dx", dx, dx_ref, tol, cmp.frames())
    for k, t in grads.items():
        check_grad(k, t, gr, tol)


@pytest.mark.parametrize("dtype,sequenced", [(torch.float32, True), (torch.bfloat16, False), (torch.bfloat16, True)])
def test_padding_never_leaks(dtype, sequenced):
    """Padding of 0, 1e4 and NaN gives the same bits for the loss and every gradient, all finite."""
    net, _ = _backend()
    lengths = LONG
    Bsz, T = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(32)
    x = torch.randn(Bsz, T, 144, generator=g).cuda()
    labels = torch.randint(0, 2, (Bsz,), generator=g).cuda()
    pad = _pad_mask(lengths, T)
    runs = [_net_step(net, x.masked_fill(pad.unsqueeze(-1), v), lengths, labels, dtype, sequenced)
            for v in (0.0, 1e4, float("nan"))]
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1])
        for k in r[2]:
            assert torch.equal(r[2][k], runs[0][2][k]), k
    assert all(torch.isfinite(t).all() for t in runs[0][2].values())


def test_loss_on_padded_output_frames_changes_nothing():
    """A loss that also weights the padded output frames of the encoder gives the bits of one with those weights zero."""
    net, _ = _backend()
    lengths = LONG
    Bsz, T = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(33)
    x = torch.randn(Bsz, T, 144, generator=g).cuda()
    w = torch.randn(Bsz, T, 144, generator=g).cuda()
    pad = _pad_mask(lengths, T)
    res = []
    for ww in (w, w.masked_fill(pad.unsqueeze(-1), 0.0)):
        net.zero_grad(set_to_none=True)
        with _autocast(torch.bfloat16):
            f = net.forward_features(x, lengths, mask_padding=True)
            loss = (f.float() * ww).sum()
        loss.backward()
        res.append((loss.detach(), {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}))
    assert torch.equal(res[0][0], res[1][0])
    for k in res[0][1]:
        assert torch.equal(res[0][1][k], res[1][1][k]), k


@pytest.mark.parametrize("dtype,sequenced", [(torch.float32, True), (torch.bfloat16, False), (torch.bfloat16, True)])
def test_full_lengths_match_fixed_length_bits(dtype, sequenced):
    """lengths == T with mask_padding=True: the loss and every gradient have the bits of the fixed-length step (the
    time-split forward, which has no variable-length form, is held off for both)."""
    net, _ = _backend()
    Bsz, T = 4, 201
    g = torch.Generator().manual_seed(34)
    x = torch.randn(Bsz, T, 144, generator=g).cuda()
    labels = torch.randint(0, 2, (Bsz,), generator=g).cuda()

    def step(lengths):
        net.zero_grad(set_to_none=True)
        xg = x.clone().requires_grad_(True)
        seq = ops.sequenced_block() if sequenced else ops._NULL
        with _autocast(dtype), seq:
            _, logits = net(xg, lengths, mask_padding=lengths is not None)
            loss = F.cross_entropy(logits.float(), labels, reduction="sum")
        loss.backward()
        return loss.detach(), xg.grad, {k: p.grad.clone() for k, p in net.named_parameters()}
    with bm._lib.tuning(bm._lib.TUNE_SCAN_SPLIT, 1):
        a, b = step(None), step([T] * Bsz)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for k in a[2]:
        assert torch.equal(a[2][k], b[2][k]), k


def test_graphed_train_step_with_lengths():
    """One captured step (AdamW in the graph) replayed with a list and a CUDA tensor of lengths: loss and parameters
    equal the eager sequenced step bit for bit, and the gradients match the oracle."""
    Bsz, T = 6, 64
    g = torch.Generator().manual_seed(35)
    xs = [torch.randn(Bsz, T, 144, generator=g).cuda() for _ in range(3)]
    labels = torch.randint(0, 2, (Bsz,), generator=g).cuda()
    lens = [[64, 40, 9, 17, 1, 33], [5, 64, 64, 8, 16, 2], [64, 63, 7, 30, 50, 9]]

    def make():
        net, _ = _backend()
        params = list(net.parameters())
        return net, params, bm.FusedAdamW(params, lr=1e-3, weight_decay=1e-4)

    def step_fn(net):
        def f(x, lengths):
            with _autocast(torch.bfloat16):
                _, logits = net(x, lengths, mask_padding=True)
            return F.cross_entropy(logits.float(), labels, reduction="sum")
        return f

    def zero_grad(params):
        def z():
            for p in params:
                p.grad = None
        return z

    net_g, params_g, opt_g = make()
    gs = bm.GraphedTrainStep(step_fn(net_g), xs[0], zero_grad(params_g), opt_g, lengths=lens[0])
    net_e, params_e, opt_e = make()
    fe = step_fn(net_e)
    _, p64 = _backend()                                    # the parameters before the first update
    for i, lengths in ((1, lens[1]), (2, torch.tensor(lens[2], device="cuda"))):
        loss_g = gs.run(xs[i], lengths).detach().clone()
        grads_g = {k: p.grad.clone() for k, p in net_g.named_parameters()}
        zero_grad(params_e)()
        with ops.sequenced_block():
            loss_e = fe(xs[i], ops.seqlens_tensor(lengths, Bsz, T, "cuda"))
            loss_e.backward()
        opt_e.step()
        torch.cuda.synchronize()
        assert torch.equal(loss_g, loss_e.detach())
        for (k, a), b in zip(net_g.named_parameters(), params_e):
            assert torch.equal(a, b), k
        if i == 1:
            _, gr, _ = varlen_loss_and_grads_ref(
                backend_logits_fn(2), p64, xs[i], lens[1],
                lambda lg, idx, n: F.cross_entropy(lg, labels[idx], reduction="sum"))
            for k, t in grads_g.items():
                check_grad(k, t, gr, 5e-2)


def test_mask_padding_under_no_grad_scores_with_zero_padding():
    net, _ = _backend()
    net.eval()
    lengths = LONG
    Bsz, T = len(lengths), max(lengths)
    x = torch.randn(Bsz, T, 144, generator=torch.Generator().manual_seed(36)).cuda()
    with torch.no_grad():
        f = net.forward_features(x, lengths, mask_padding=True)
        s_mask = net(x, lengths, mask_padding=True)[1]
        s_score = net(x, lengths)[1]
    assert bool((f[_pad_mask(lengths, T)] == 0).all())
    assert cmp.rel(s_mask, s_score) < 1e-5
