"""Mixup on the GPU: bimamba_mixup_frames against torch's expression bit for bit (fixed length) and against the oracle
(variable length); one Phase6TrainStep with Mixup, FGM and lengths on the 4-layer backend against the fp64 oracle run
on every mixed utterance alone; and the captured fp16 recipe with labels, Mixup, lengths, DeviceGradScaler, clipping,
FusedEMA and 4-step accumulation against eager Phase6TrainSteps given the same draws, bit for bit."""
import importlib

import pytest
import torch
import torch.nn.functional as F
from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

import bimamba_b200 as bm
from bimamba_b200 import ops
from oracle import bimamba_oracle as orc
from oracle import compare as cmp
from oracle.mixup_oracle import mixup_ref
from oracle.varlen_train_oracle import backend_logits_fn, varlen_loss_and_grads_ref

pytestmark = pytest.mark.gpu
tr = importlib.import_module("robust-audio-deepfake-evolution_b200.training")

LAMS = [0.0, 1.0, 0.3, 0.5, 0.7311, 1e-7, 2.0 ** -30, 1.0 - 1e-7, 1.0 - 2.0 ** -30]


def _mix(x, perm, lam, seqlens=None, out=None):
    return ops.mixup_frames(x, perm.to(torch.int32), tr.mix_record(lam, x.device), seqlens, out)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,T,C", [(8, 201, 1), (8, 201, 37), (8, 201, 144), (8, 1, 1), (4, 64600, 1)])
def test_fixed_length_is_the_torch_expression_bitwise(dtype, B, T, C):
    g = torch.Generator().manual_seed(B * T + C)
    x = (torch.randn(B, T, C, generator=g) * 3).to(dtype).cuda()
    perm = torch.randperm(B, generator=g).cuda()
    for lam in LAMS:
        got, sl = _mix(x, perm, lam)
        assert sl is None
        assert torch.equal(got, lam * x + (1.0 - lam) * x[perm]), lam
    if C == 144:                                     # an unaligned base takes the scalar path: the same bits
        buf = torch.empty(x.numel() + 1, dtype=dtype, device="cuda")
        xu = buf[1:].view_as(x)
        xu.copy_(x)
        assert torch.equal(_mix(xu, perm, 0.3)[0], 0.3 * x + 0.7 * x[perm])
    # mixup_batch runs on the kernel and keeps today's bits and draws
    y = torch.arange(B, device="cuda")
    mx, ya, yb, lam = bm.mixup_batch(x, y, 1.0, torch.Generator().manual_seed(3), 0.42)
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(3)).cuda()
    assert torch.equal(mx, 0.42 * x + (1.0 - 0.42) * x[idx]) and torch.equal(yb, y[idx]) and lam == 0.42


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("C", [1, 37, 144])
def test_variable_length_against_the_oracle(dtype, C):
    g = torch.Generator().manual_seed(7 + C)
    lengths = [201, 0, 1, 77, 150, 201, 9, 33]
    B, T = len(lengths), 201
    clean = (torch.randn(B, T, C, generator=g) * 2).to(dtype)
    perm = torch.tensor([5, 2, 1, 0, 7, 3, 4, 6])
    lens_dev = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    want_m = [max(lengths[b], lengths[int(perm[b])]) for b in range(B)]
    outs = []
    for pad in (0.0, 1e4, float("nan")):
        x = clean.clone()
        for b, n in enumerate(lengths):
            x[b, n:] = pad
        xd = x.cuda()
        for lam in (0.0, 0.3, 1.0 - 2.0 ** -30, 1.0):
            out = torch.full_like(xd, float("nan"))               # a sentinel: every frame must be written
            got, sl = _mix(xd, perm.cuda(), lam, lens_dev, out)
            assert got is out and sl.tolist() == want_m
            ref, m = mixup_ref(xd, perm, lam, lengths, exact=False)
            assert torch.equal(got, ref), (pad, lam)
            exact, _ = mixup_ref(x, perm, lam, lengths, exact=True)
            assert cmp.rel(got, exact) < (1e-6 if dtype == torch.float32 else 1e-2)
            assert torch.isfinite(got).all()
            for b in range(B):
                assert bool((got[b, want_m[b]:] == 0).all())
            if lam == 0.3:
                outs.append(got)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])     # padding never reaches an output
    # a host list (lengths 1..T) through mixup_batch, and an identity permutation is the masked torch expression
    host = [max(n, 1) for n in lengths]
    xd = clean.cuda()
    y = torch.zeros(B, dtype=torch.long, device="cuda")
    mx, _, _, _, ml = bm.mixup_batch(xd, y, 1.0, None, 0.3, host, index=perm)
    assert torch.equal(mx, mixup_ref(xd, perm, 0.3, host, exact=False)[0])
    assert ml.tolist() == [max(host[b], host[int(perm[b])]) for b in range(B)]
    ident, sl = _mix(xd, torch.arange(B, device="cuda"), 0.5, lens_dev)
    assert sl.tolist() == lengths
    assert torch.equal(ident, ops.mask_frames_raw(0.5 * xd + 0.5 * xd, lens_dev))


# ---- the training contract ------------------------------------------------------------------------------------------
def _backend(n_layers=4, seed=30):
    layers = [orc.init_encoder_params(144, 16, seed=seed + i) for i in range(n_layers)]
    head = orc.init_head_params(144, seed=seed)
    net = bm.BiMambaBackend(144, n_layers, 16).cuda().train()
    net.dropout.p = 0.0
    sd = {f"backbone_layers.{i}.{k}": v for i, p in enumerate(layers) for k, v in p.items()}
    sd.update(head)
    net.load_state_dict(sd, strict=True)
    return net, {k: v.double().cuda() for k, v in net.state_dict().items()}


def check_grad(name, got, grads_ref, tol):
    """As the variable-length training tests: the attention-pool bias has an exact gradient of zero and is measured on
    the scale of the attention weight's."""
    if "attention_pool.bias" in name:
        w = name.replace("bias", "weight")
        err = float(got.detach().double().abs().max().cpu() / grads_ref[w].abs().max().clamp_min(1e-30).cpu())
        assert err < tol, (name, err)
        return
    cmp.check(name, got, grads_ref[name], tol, cmp.param(name, got.shape))


class _Grab(torch.optim.Optimizer):
    """Keeps the gradients the step hands to the optimizer and changes nothing."""

    def __init__(self, named):
        self.named = named
        super().__init__([p for _, p in named], {})

    def step(self, closure=None):
        self.grads = {n: p.grad.detach().clone() for n, p in self.named}


def test_phase6_step_with_mixup_fgm_and_lengths_against_the_oracle():
    """fp32 compute, so the per-slice rule holds at 1e-4; the fp16 recipe is checked bit for bit against eager steps
    below."""
    dtype, tol = None, 1e-4
    net, p64 = _backend()
    lengths = [201, 150, 77, 9, 201, 33, 120, 64]
    B, T = len(lengths), 201
    g = torch.Generator().manual_seed(31)
    x = torch.randn(B, T, 144, generator=g)
    for b, n in enumerate(lengths):
        x[b, n:] = float("nan")
    y = torch.randint(0, 2, (B,), generator=g)
    eps, target = 0.5, "backbone_layers.0.norm1"
    opt = _Grab(list(net.named_parameters()))
    step = bm.Phase6TrainStep(net, opt, lambda lg, f, t: F.cross_entropy(lg.float(), t), autocast_dtype=dtype,
                              fgm=bm.FGM(net, target, eps), mixup_alpha=1.0, max_norm=float("inf"))
    torch.manual_seed(5)
    loss = step([(x.cuda(), y.cuda(), lengths)], generator=torch.Generator().manual_seed(6))
    torch.cuda.synchronize()
    torch.manual_seed(5)
    lam = float(torch.distributions.Beta(1.0, 1.0).sample())
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(6))
    mx, m = mixup_ref(x, perm, lam, lengths)                        # fp64, each mixed clip at its own length
    ya, yb = y.cuda(), y[perm].cuda()

    def lossf(lg, idx, n):
        return (lam * F.cross_entropy(lg, ya[idx], reduction="sum")
                + (1.0 - lam) * F.cross_entropy(lg, yb[idx], reduction="sum")) / B
    fn = backend_logits_fn(4)
    loss_ref, g_clean, _ = varlen_loss_and_grads_ref(fn, p64, mx.cuda(), m.tolist(), lossf)
    adv = dict(p64)
    for k in adv:
        if target in k:
            adv[k] = p64[k] + eps * g_clean[k] / g_clean[k].norm()
    _, g_adv, _ = varlen_loss_and_grads_ref(fn, adv, mx.cuda(), m.tolist(), lossf)
    assert cmp.rel(loss, loss_ref) < tol
    for k, got in opt.grads.items():
        check_grad(k, got, {n: g_clean[n] + g_adv[n] for n in g_clean}, tol)


# ---- the captured recipe --------------------------------------------------------------------------------------------
DECAY = 0.999


def f32(v):
    return float(torch.tensor(v, dtype=torch.float32))


def _setup():
    torch.manual_seed(1234)
    model = bm.BiMambaBackend(144, 4, 16).cuda()
    model.dropout.p = 0.0
    with torch.no_grad():
        for layer in model.backbone_layers:
            layer.mamba.A_log.add_(0.1 * torch.randn_like(layer.mamba.A_log))
    params = [p for p in model.parameters() if p.requires_grad]
    opt = bm.FusedAdamW(params, lr=f32(1e-3), weight_decay=f32(1e-4), betas=(f32(0.9), f32(0.999)), eps=f32(1e-8))
    avg = AveragedModel(model, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    scaler = bm.DeviceGradScaler(init_scale=2.0 ** 10)
    return model, params, opt, avg, bm.FusedEMA(avg, model, DECAY), scaler


def _state(model, opt, avg, scaler):
    out = {"param." + n: p.detach().clone() for n, p in model.named_parameters()}
    out.update({"avg." + n: p.detach().clone() for n, p in avg.module.named_parameters()})
    out["n_averaged"] = avg.n_averaged.detach().clone()
    out["amp"] = scaler._lazy_init().clone()[:2]
    for i, g in enumerate(opt._groups):
        out[f"m{i}"], out[f"v{i}"], out[f"step{i}"] = g["m"].clone(), g["v"].clone(), g["state"].clone()
    return out


def _ce(logits, feats, y):
    return F.cross_entropy(logits.float(), y)


def test_captured_recipe_with_labels_mixup_and_lengths_equals_eager_steps():
    Bsz, T, K, STEPS = 16, 64, 4, 8
    g = torch.Generator().manual_seed(77)
    data = []
    for _ in range(K * STEPS):
        lens = torch.randint(1, T + 1, (Bsz,), generator=g).tolist()
        data.append((torch.randn(Bsz, T, 144, generator=g).cuda(), torch.randint(0, 2, (Bsz,), generator=g).cuda(), lens))

    model, params, opt, avg, ema, scaler = _setup()
    bucket = bm.FlatGradBucket(params, accumulate=True)

    def step_fn(x, y, lengths, mix):
        mx, ya, yb, lam, ml = bm.mixup_batch(x, y, lam=mix.mix, lengths=lengths, index=mix.perm)
        with torch.autocast("cuda", dtype=torch.float16):
            feats, out = model(mx, ml, mask_padding=True)
            return bm.mixup_loss(_ce, out, feats, ya, yb, lam)
    gs = bm.GraphedTrainStep(step_fn, data[0][0], bucket.zero, opt, lengths=data[0][2], scaler=scaler, max_norm=3.0,
                             ema=ema, accumulation_steps=K, labels=data[0][1], mixup_alpha=1.0,
                             generator=torch.Generator().manual_seed(8))
    torch.manual_seed(9)
    gs.generator.manual_seed(8)
    lams, losses, states = [], [], []
    for s in range(STEPS):
        total = None
        for j in range(K):
            x, y, lens = data[K * s + j]
            loss = gs.run(x, lens, y=y).detach().clone() / K
            lams.append(gs.last_lam)
            total = loss if total is None else total + loss
        torch.cuda.synchronize()
        losses.append(total)
        states.append(_state(model, opt, avg, scaler))
    assert len(set(lams)) == len(lams)                        # a fresh lam on every replay: no frozen draw

    model_e, params_e, opt_e, avg_e, ema_e, scaler_e = _setup()
    step = bm.Phase6TrainStep(model_e, opt_e, _ce, scaler=scaler_e, mixup_alpha=1.0, accumulation_steps=K,
                              max_norm=3.0, ema_model=ema_e)
    torch.manual_seed(9)
    gen_e = torch.Generator().manual_seed(8)
    for s in range(STEPS):
        with ops.sequenced_block():
            loss_e = step(data[K * s:K * s + K], generator=gen_e)
        torch.cuda.synchronize()
        assert torch.equal(losses[s], loss_e), s
        want = states[s]
        got = _state(model_e, opt_e, avg_e, scaler_e)
        diff = [k for k in want if not torch.equal(want[k], got[k])]
        assert not diff, (s, diff[:8])
    assert int(avg.n_averaged) == STEPS
