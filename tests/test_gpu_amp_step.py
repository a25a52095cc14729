"""The fp16 recipe's optimizer tail on the device: FusedAdamW.step(scaler=DeviceGradScaler, max_norm=, ema=FusedEMA).

Contract (for the same gradients, against  s.unscale_(opt); clip_grad_norm_(params, max_norm); s.step(opt); s.update();
ema.update_parameters(model)  with torch.optim.AdamW and torch.amp.GradScaler):
  * bitwise: the loss scale, the growth tracker, n_averaged, the step counter, and whether the step was skipped;
  * bitwise on a skipped step: parameters and moments do not move, and the average moves as torch._foreach_lerp_ moves it;
  * 1e-6 relative: parameters, moments and the average on applied steps, and the total norm.
Then the same step captured in GraphedTrainStep: replays equal eager steps bit for bit (fixed length, accumulation over
four micro-batches, variable length), a real fp16 overflow inside the graph is skipped, and building the runner changes
no state.
"""
import pytest
import torch
from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

import bimamba_b200 as bm
from oracle import compare as cmp

pytestmark = pytest.mark.gpu

SHAPES = [(576, 144), (288, 4), (288,), (9000,), (1,), (37, 3)]     # as the FusedAdamW-vs-torch test
DECAY = 0.999


class _Params(torch.nn.Module):
    def __init__(self, shapes, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.randn(s, generator=g).cuda()) for s in shapes])


def _stats(opt, scaler, max_norm):
    """bimamba_amp_grad_stats alone over the optimizer's table of every group -> (found_inf, total_norm) on the host."""
    if opt._groups is None:
        opt._build()
    for g in opt._groups:
        if g["params"]:
            opt._write_table(g, opt._grad_ptrs(g))
    a, rec = opt._all, scaler._lazy_init()
    lib = bm._lib.load()
    bm._lib.check(lib.bimamba_amp_grad_stats(a["table"].data_ptr(), a["bmap"].data_ptr(), a["nblocks"], max_norm,
                                             a["partials"].data_ptr(), rec.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "stats")
    torch.cuda.synchronize()
    f = rec.view(torch.float32)
    return float(f[2]), f[3].clone(), f[4].clone()


def test_gradient_statistics_norm_inf_and_determinism():
    m = _Params(SHAPES, 1)
    ps = list(m.ps)
    opt = bm.FusedAdamW([{"params": ps[:3]}, {"params": ps[3:]}])
    s = bm.DeviceGradScaler(init_scale=1024.0)
    gen = torch.Generator(device="cuda").manual_seed(2)
    for p in ps:
        p.grad = torch.randn(p.shape, device="cuda", generator=gen) * 1024.0
    ref = torch.sqrt(sum(((p.grad.double() * (1.0 / 1024.0)) ** 2).sum() for p in ps))
    found, norm, coef = _stats(opt, s, 3.0)
    assert found == 0.0
    assert cmp.rel(norm, ref) < 1e-6
    assert float(coef) == float((1.0 / (norm + 1e-6)) * 3.0)
    for _ in range(2):                                        # determinism: the same bits on every run
        assert torch.equal(_stats(opt, s, 3.0)[1], norm)
    assert float(_stats(opt, s, 0.0)[2]) == 1.0               # no clipping
    ps[1].grad = None                                         # a tensor without gradient is skipped
    ref_skip = torch.sqrt(sum(((p.grad.double() / 1024.0) ** 2).sum() for p in ps if p.grad is not None))
    assert cmp.rel(_stats(opt, s, 3.0)[1], ref_skip) < 1e-6
    for idx, where, bad in ((0, (5, 7), float("inf")), (3, (8999,), float("nan")), (5, (36, 2), float("-inf"))):
        old = ps[idx].grad[where].item()
        ps[idx].grad[where] = bad                             # (36, 2): element 110 of 111, in the scalar tail
        assert _stats(opt, s, 3.0)[0] == 1.0, (idx, where)
        ps[idx].grad[where] = old
    assert _stats(opt, s, 3.0)[0] == 0.0


def f32(v):
    """The hyper-parameters as the device holds them: torch.optim.AdamW is given the same fp32 values (1 - beta2 of
    fp32(0.999) differs from 1 - 0.999 by 1.3e-5 relative, which the moments would show)."""
    return float(torch.tensor(v, dtype=torch.float32))


HYPER = dict(betas=(f32(0.9), f32(0.999)), eps=f32(1e-8))


def _groups(ps):
    return [{"params": ps[:2], "lr": f32(1e-3), "weight_decay": f32(1e-2)},   # main.py:453: three groups, own lr / wd
            {"params": ps[2:4], "lr": f32(3e-4), "weight_decay": 0.0},
            {"params": ps[4:], "lr": f32(1e-4), "weight_decay": f32(5e-2)}]


def test_ten_steps_against_the_torch_tail():
    m_f, m_t = _Params(SHAPES, 3), _Params(SHAPES, 3)
    ps_f, ps_t = list(m_f.ps), list(m_t.ps)
    avg_f = AveragedModel(m_f, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    avg_t = AveragedModel(m_t, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    ema = bm.FusedEMA(avg_f, m_f, DECAY)
    opt_f, opt_t = bm.FusedAdamW(_groups(ps_f), **HYPER), torch.optim.AdamW(_groups(ps_t), **HYPER)
    s_f = bm.DeviceGradScaler(init_scale=2.0 ** 12, growth_interval=3)
    s_t = torch.amp.GradScaler("cuda", init_scale=2.0 ** 12, growth_interval=3)
    s_t.scale(torch.ones((), device="cuda"))
    gen = torch.Generator(device="cuda").manual_seed(4)
    applied_steps, grown = 0, False
    for k in range(10):
        scale = s_f.get_scale()
        assert scale == s_t.get_scale()
        size = 2.0 if k % 2 else 0.005                       # global norms ~ 600 (clipped) and ~ 1.5 (not clipped)
        for pf, pt in zip(ps_f, ps_t):
            g = torch.randn(pf.shape, device="cuda", generator=gen) * size * scale
            pf.grad, pt.grad = g.clone(), g.clone()
        if k == 4:
            ps_f[3].grad[17] = ps_t[3].grad[17] = float("inf")
        if k == 7:
            ps_f[5].grad[36, 1] = ps_t[5].grad[36, 1] = float("nan")
        before = [p.detach().clone() for p in ps_f]
        mom_before = [(opt_f.state[p]["exp_avg"].clone(), opt_f.state[p]["exp_avg_sq"].clone()) if k else None
                      for p in ps_f]
        ema_before = [a.detach().clone() for _, a in ema.pairs]
        opt_f.step(scaler=s_f, max_norm=3.0, ema=ema)
        s_t.unscale_(opt_t)
        norm_t = torch.nn.utils.clip_grad_norm_(ps_t, 3.0)
        s_t.step(opt_t)
        s_t.update()
        avg_t.update_parameters(m_t)
        torch.cuda.synchronize()
        skipped = k in (4, 7)
        assert float(s_f.found_inf) == (1.0 if skipped else 0.0)
        applied_steps += not skipped
        # bitwise: scale, growth tracker, n_averaged, step counters
        assert torch.equal(s_f._scale, s_t._scale), k
        assert torch.equal(s_f._growth_tracker, s_t._growth_tracker), k
        grown |= s_f.get_scale() > scale
        assert torch.equal(avg_f.n_averaged.cpu(), avg_t.n_averaged.cpu())
        for g in opt_f._groups:
            assert float(g["state"]) == applied_steps
        for p in ps_t:
            assert float(opt_t.state[p]["step"]) == applied_steps
        if skipped:
            for p, b, mb in zip(ps_f, before, mom_before):
                assert torch.equal(p, b)
                assert torch.equal(opt_f.state[p]["exp_avg"], mb[0]) and torch.equal(opt_f.state[p]["exp_avg_sq"], mb[1])
            torch._foreach_lerp_(ema_before, before, 1 - DECAY)
            for (_, a), e in zip(ema.pairs, ema_before):
                assert torch.equal(a, e)
        else:
            assert cmp.rel(opt_f.total_norm, norm_t) < 1e-6, k
            for pf, pt in zip(ps_f, ps_t):
                assert cmp.rel(pf, pt) < 1e-6, k
                assert cmp.rel(opt_f.state[pf]["exp_avg"], opt_t.state[pt]["exp_avg"]) < 1e-6, k
                assert cmp.rel(opt_f.state[pf]["exp_avg_sq"], opt_t.state[pt]["exp_avg_sq"]) < 1e-6, k
        for (_, a), at in zip(ema.pairs, avg_t.module.parameters()):
            assert cmp.rel(a, at) < 1e-6, k
        for pf in ps_f:
            pf.grad = None
    assert grown


def test_scaler_state_dict_round_trip_with_torch():
    def run(scaler, bad, torch_side):
        p = torch.nn.Parameter(torch.ones(8, device="cuda"))
        opt = torch.optim.AdamW([p]) if torch_side else bm.FusedAdamW([p])
        for b in bad:
            p.grad = torch.full((8,), float("inf") if b else 1.0, device="cuda")
            if torch_side:
                scaler.step(opt)
                scaler.update()
            else:
                opt.step(scaler=scaler)
            yield scaler.get_scale(), scaler.state_dict()["_growth_tracker"]

    s = bm.DeviceGradScaler(init_scale=1024.0, growth_interval=2, growth_factor=4.0, backoff_factor=0.25)
    list(run(s, [0, 1, 0], False))
    sd = s.state_dict()
    assert sd == {"scale": 256.0, "growth_factor": 4.0, "backoff_factor": 0.25, "growth_interval": 2,
                  "_growth_tracker": 1}
    t = torch.amp.GradScaler("cuda")
    t.load_state_dict(sd)
    t.scale(torch.ones((), device="cuda"))
    assert t.state_dict() == sd
    pattern = [0, 0, 0, 1, 0, 0]
    assert list(run(t, pattern, True)) == list(run(s, pattern, False))
    s2 = bm.DeviceGradScaler()
    s2.load_state_dict(t.state_dict())
    assert s2.state_dict() == t.state_dict() == s.state_dict()


# ---- the captured backend -------------------------------------------------------------------------------------------
B, L = 16, 201


def _setup():
    torch.manual_seed(1234)
    model = bm.BiMambaBackend(144, 4, 16).cuda()
    with torch.no_grad():
        for layer in model.backbone_layers:
            layer.mamba.A_log.add_(0.1 * torch.randn_like(layer.mamba.A_log))
    params = list(model.backbone_layers.parameters())
    opt = bm.FusedAdamW(params, lr=f32(1e-3), weight_decay=f32(1e-4), **HYPER)
    avg = AveragedModel(model, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    scaler = bm.DeviceGradScaler(init_scale=2.0 ** 10)
    return model, params, opt, avg, bm.FusedEMA(avg, model, DECAY), scaler


def _batch(seed, T=L):
    return torch.randn(B, T, 144, generator=torch.Generator().manual_seed(seed)).cuda()


def _loss_fn(model, lengths=False):
    def f(x, *lens):
        with torch.autocast("cuda", dtype=torch.float16):
            out = model.forward_features(x, *lens, mask_padding=bool(lens))
        return bm.ops.mean_square_loss(out)
    return f


def _zero(params):
    def z():
        for p in params:
            p.grad = None
    return z


def _state(model, opt, avg, scaler):
    """Everything the optimizer tail touches."""
    out = {"param." + n: p.detach().clone() for n, p in model.named_parameters()}
    out.update({"avg." + n: p.detach().clone() for n, p in avg.module.named_parameters()})
    out["n_averaged"] = avg.n_averaged.detach().clone()
    out["amp"] = scaler._lazy_init().clone()[:2]            # scale and growth tracker
    if opt._groups is not None:
        for i, g in enumerate(opt._groups):
            out[f"m{i}"], out[f"v{i}"], out[f"step{i}"] = g["m"].clone(), g["v"].clone(), g["state"].clone()
    return out


def _assert_same(a, b, what):
    diff = [k for k in a if not torch.equal(a[k], b[k])]
    assert not diff, (what, diff[:8])


def test_captured_fp16_recipe_eager_bitwise_torch_tail_and_overflow():
    xs = [_batch(100 + k) for k in range(3)]
    # (a) captured
    model, params, opt, avg, ema, scaler = _setup()
    gs = bm.GraphedTrainStep(_loss_fn(model), xs[0], _zero(params), opt, scaler=scaler, max_norm=3.0, ema=ema)
    # (b) eager, the same arrangement
    model_e, params_e, opt_e, avg_e, ema_e, scaler_e = _setup()
    # (c) torch's tail on the first step
    model_t, params_t, _, avg_t, _, _ = _setup()
    opt_t = torch.optim.AdamW(params_t, lr=f32(1e-3), weight_decay=f32(1e-4), **HYPER)
    scaler_t = torch.amp.GradScaler("cuda", init_scale=2.0 ** 10)
    for k, x in enumerate(xs):
        loss_g = gs.run(x).detach().clone()
        _zero(params_e)()
        loss_e = _loss_fn(model_e)(x)
        scaler_e.scale(loss_e).backward()
        opt_e.step(scaler=scaler_e, max_norm=3.0, ema=ema_e)
        torch.cuda.synchronize()
        assert torch.equal(loss_g, loss_e.detach()), k
        _assert_same(_state(model, opt, avg, scaler), _state(model_e, opt_e, avg_e, scaler_e), f"replay {k}")
        assert torch.equal(opt.total_norm, opt_e.total_norm)
        if k == 0:
            loss_t = _loss_fn(model_t)(x)
            scaler_t.scale(loss_t).backward()
            scaler_t.unscale_(opt_t)
            norm_t = torch.nn.utils.clip_grad_norm_([p for p in params_t if p.grad is not None], 3.0)
            scaler_t.step(opt_t)
            scaler_t.update()
            avg_t.update_parameters(model_t)
            torch.cuda.synchronize()
            assert cmp.rel(opt.total_norm, norm_t) < 1e-6
            assert float(scaler._scale) == float(scaler_t._scale)
            assert int(scaler._growth_tracker) == int(scaler_t._growth_tracker) == 1
            assert int(avg.n_averaged) == int(avg_t.n_averaged) == 1
            for (n, p), pt in zip(model.backbone_layers.named_parameters(), params_t):
                assert cmp.rel(p, pt) < 1e-6, n
                assert cmp.rel(opt.state[p]["exp_avg"], opt_t.state[pt]["exp_avg"]) < 1e-6, n
                assert cmp.rel(opt.state[p]["exp_avg_sq"], opt_t.state[pt]["exp_avg_sq"]) < 1e-6, n
                assert float(opt_t.state[pt]["step"]) == 1.0
            for (n, a), at in zip(avg.module.named_parameters(), avg_t.module.parameters()):
                assert cmp.rel(a, at) < 1e-6, n
    # (d) a real fp16 overflow inside the graph: the scale 2^126 makes the backward's fp16 gradients overflow
    keep = scaler.get_scale()
    scaler._scale.fill_(2.0 ** 126)
    before = _state(model, opt, avg, scaler)
    gs.run(_batch(200))
    torch.cuda.synchronize()
    after = _state(model, opt, avg, scaler)
    assert float(scaler.found_inf) == 1.0
    for key in before:
        if key.startswith("param.") or key[0] in "mv" or key.startswith("step"):
            assert torch.equal(before[key], after[key]), key
    assert float(after["amp"].view(torch.float32)[0]) == 2.0 ** 125 and int(after["amp"][1]) == 0
    assert int(after["n_averaged"]) == int(before["n_averaged"]) + 1
    names = [n for n, _ in model.named_parameters()]
    ema_ref = [before["avg." + n].clone() for n in names]
    torch._foreach_lerp_(ema_ref, [before["param." + n] for n in names], 1 - DECAY)
    for n, e in zip(names, ema_ref):
        assert torch.equal(after["avg." + n], e), n
    assert any(not torch.equal(before["avg." + n], after["avg." + n]) for n in names)
    # the next replay, at a usable scale again, applies
    scaler._scale.fill_(keep)
    gs.run(_batch(201))
    torch.cuda.synchronize()
    assert float(scaler.found_inf) == 0.0
    assert all(float(g["state"]) == 4.0 for g in opt._groups)
    assert not torch.equal(_state(model, opt, avg, scaler)["param.backbone_layers.0.mamba.in_proj.weight"],
                           after["param.backbone_layers.0.mamba.in_proj.weight"])


def test_captured_accumulation_equals_one_eager_step_over_four_micro_batches():
    xs = [_batch(300 + k) for k in range(8)]
    model, params, opt, avg, ema, scaler = _setup()
    bucket = bm.FlatGradBucket(params, accumulate=True)
    gs = bm.GraphedTrainStep(_loss_fn(model), xs[0], bucket.zero, opt, scaler=scaler, max_norm=3.0, ema=ema,
                             accumulation_steps=4)
    model_e, params_e, opt_e, avg_e, ema_e, scaler_e = _setup()
    bucket_e = bm.FlatGradBucket(params_e, accumulate=True)
    start = _state(model, opt, avg, scaler)
    for step in range(2):
        for j in range(4):
            loss_g = gs.run(xs[4 * step + j]).detach().clone()
            loss_e = _loss_fn(model_e)(xs[4 * step + j])
            scaler_e.scale(loss_e / 4).backward()
            torch.cuda.synchronize()
            assert torch.equal(loss_g, loss_e.detach())
            if step == 0 and j < 3:                          # nothing moves before the fourth micro-batch
                _assert_same(_state(model, opt, avg, scaler), start, f"micro {j}")
        opt_e.step(scaler=scaler_e, max_norm=3.0, ema=ema_e)
        bucket_e.zero()
        torch.cuda.synchronize()
        _assert_same(_state(model, opt, avg, scaler), _state(model_e, opt_e, avg_e, scaler_e), f"step {step}")
        assert torch.equal(bucket.flat, torch.zeros_like(bucket.flat))
        assert all(float(g["state"]) == step + 1 for g in opt._groups)


def test_captured_variable_length_step_with_scaler_and_ema():
    T = 64
    xs = [_batch(400 + k, T) for k in range(3)]
    lens = [[64, 40, 9, 17, 1, 33, 64, 2, 50, 64, 12, 8, 30, 61, 5, 64],
            [5, 64, 64, 8, 16, 2, 33, 33, 64, 1, 7, 60, 64, 20, 44, 9],
            [64] * 8 + [32] * 8]
    model, params, opt, avg, ema, scaler = _setup()
    gs = bm.GraphedTrainStep(_loss_fn(model), xs[0], _zero(params), opt, lengths=lens[0], scaler=scaler, max_norm=3.0,
                             ema=ema)
    model_e, params_e, opt_e, avg_e, ema_e, scaler_e = _setup()
    for i, lengths in ((1, lens[1]), (2, torch.tensor(lens[2], device="cuda"))):
        loss_g = gs.run(xs[i], lengths).detach().clone()
        _zero(params_e)()
        with bm.ops.sequenced_block():
            loss_e = _loss_fn(model_e)(xs[i], bm.ops.seqlens_tensor(lengths, B, T, "cuda"))
            scaler_e.scale(loss_e).backward()
        opt_e.step(scaler=scaler_e, max_norm=3.0, ema=ema_e)
        torch.cuda.synchronize()
        assert torch.equal(loss_g, loss_e.detach()), i
        _assert_same(_state(model, opt, avg, scaler), _state(model_e, opt_e, avg_e, scaler_e), f"lengths {i}")


@pytest.mark.parametrize("accumulation_steps", [1, 4])
def test_building_the_runner_changes_no_state(accumulation_steps):
    model, params, opt, avg, ema, scaler = _setup()
    bucket = bm.FlatGradBucket(params, accumulate=True)
    loss = _loss_fn(model)(_batch(500))                     # one eager step first: every piece of state is non-trivial
    scaler.scale(loss).backward()
    opt.step(scaler=scaler, max_norm=3.0, ema=ema)
    bucket.zero()
    torch.cuda.synchronize()
    del loss              # its graph would keep the parameters' gradient accumulators, made on the eager stream
    before = _state(model, opt, avg, scaler)
    assert int(before["n_averaged"]) == 1 and int(before["amp"][1]) == 1 and float(before["step0"]) == 1.0
    bm.GraphedTrainStep(_loss_fn(model), _batch(501), bucket.zero, opt, scaler=scaler, max_norm=3.0, ema=ema,
                        accumulation_steps=accumulation_steps)
    torch.cuda.synchronize()
    _assert_same(before, _state(model, opt, avg, scaler), "construction")


def test_phase6_train_step_fused_tail_matches_fused_step():
    """Phase6TrainStep with a DeviceGradScaler and a FusedAdamW runs its tail as FusedAdamW.step(scaler=, max_norm=,
    ema=): the same bits as calling that step by hand after the same micro-batches."""
    xs = [_batch(600 + k) for k in range(2)]
    labels = torch.zeros(B, dtype=torch.long, device="cuda")

    def loss_fn(logits, feats, y):
        return torch.nn.functional.cross_entropy(logits.float(), y)
    runs = []
    for fused_by_hand in (False, True):
        model, params, opt, avg, ema, scaler = _setup()
        model.dropout.p = 0.0
        if fused_by_hand:
            for x in xs:
                with torch.autocast("cuda", dtype=torch.float16):
                    feats, out = model(x)
                    loss = loss_fn(out, feats, labels)
                scaler.scale(loss / 2).backward()
            opt.step(scaler=scaler, max_norm=3.0, ema=ema)
        else:
            step = bm.Phase6TrainStep(model, opt, loss_fn, scaler=scaler, accumulation_steps=2, ema_model=ema)
            step([(x, labels) for x in xs])
        torch.cuda.synchronize()
        runs.append(_state(model, opt, avg, scaler))
    _assert_same(runs[0], runs[1], "Phase6TrainStep")
