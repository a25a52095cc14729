"""The benchmarked training step at its own shape against the fp64 oracle.

bench.py times one step of the 4-layer backend at batch 64 x 201 frames x 144 channels: forward_features, the
mean-square loss, backward and FusedAdamW, under bf16 autocast, replayed from a GraphedTrainStep.  The block and layer
tests elsewhere run at batch <= 4, where every parameter-gradient sum over partial rows takes the one-lane variant of
bimamba_reduce_partials.  At this shape the scan's A_log / D / dt_proj.bias sums run over B * ndir = 128 partial rows and
the conv's weight / bias sums over 832, so they take the 32-lane variant; a captured step also runs those sums on a side
stream (parallel graph branches) and reads the AdamW hyper-parameters from device memory.

  * fp32, captured: the loss and all 68 backbone gradients against the oracle, 1e-4.
  * bf16: the captured step, the eager sequenced step and the eager native step give the same bits (loss, gradients,
    parameters after AdamW).  Every layer of the native step against the oracle fed that layer's own input and output
    cotangent (output and dx 2e-2, one layer's bar, so it does not widen with depth; parameter gradients 3e-2, see the
    test); the loss (2e-2) and gradients (5e-2) end to end.
  * AdamW inside the graph: three replays on different batches with an lr change through sync_hyper(), against
    torch.optim.AdamW in fp64.
  * bimamba_reduce_partials: each of its three variants, on both sides of the switch points, against an fp64 sum.

Every comparison is per slice (oracle/compare.py): activations per utterance and per 8-frame chunk, each parameter
gradient per its own blocks.  The oracle (oracle/bimamba_oracle.py) runs on the GPU in fp64, one layer at a time: a forward without autograd keeps
each layer's input, then every layer's forward is redone under autograd while the cotangent walks back through it.
"""
import pytest
import torch

import bimamba_b200 as bm
from oracle import bimamba_oracle as orc
from oracle import compare as cmp

pytestmark = pytest.mark.gpu

B, L, D_MODEL, N_LAYERS, D_STATE = 64, 201, 144, 4, 16      # bench.py's workload (BASELINE.json configs[1])
D_INNER, NDIR = 2 * D_MODEL, 2


def _model():
    """The benchmark's model and optimizer (bench.py:run_ours), built from the same seeds every call."""
    torch.manual_seed(1234)
    model = bm.BiMambaBackend(D_MODEL, N_LAYERS, D_STATE).cuda()
    with torch.no_grad():
        for layer in model.backbone_layers:
            layer.mamba.A_log.add_(0.1 * torch.randn_like(layer.mamba.A_log))
    params = list(model.backbone_layers.parameters())
    return model, params, bm.FusedAdamW(params, lr=1e-5, weight_decay=1e-4)


def _batch(seed=1234):
    return torch.randn(B, L, D_MODEL, generator=torch.Generator().manual_seed(seed)).cuda()


def _loss_fn(model, bf16):
    def fwd_loss(x):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            out = model.forward_features(x)
        return bm.ops.mean_square_loss(out)
    return fwd_loss


def _zero_grad(params):
    def zero_grad():
        for p in params:
            p.grad = None
    return zero_grad


def _captured(model, params, opt, x, bf16):
    return bm.GraphedTrainStep(_loss_fn(model, bf16), x, _zero_grad(params), opt, warmup=3)


def _named(model):
    return list(model.backbone_layers.named_parameters(prefix="backbone_layers"))


def _layer_ref(sd, x, cot):
    """One PN_BiMambas_Encoder in fp64: its output and the products of `cot` with the Jacobians w.r.t. x and every
    parameter (sd: the layer's state_dict)."""
    xr = x.detach().double().requires_grad_(True)
    pr = {k: v.detach().double().requires_grad_(True) for k, v in sd.items()}
    out = orc.pn_bimamba_encoder_ref(pr, xr)
    g = torch.autograd.grad(out, [xr, *pr.values()], cot.double())
    return out.detach(), g[0], dict(zip(pr, g[1:]))


@pytest.fixture(scope="module")
def oracle():
    """fp64 loss and gradients of the benchmark's model on the benchmark's batch, at its initial weights."""
    model, _, _ = _model()
    sds = [{k: v.detach().double() for k, v in layer.state_dict().items()} for layer in model.backbone_layers]
    del model
    hs = [_batch().double()]
    with torch.no_grad():
        for sd in sds:
            hs.append(orc.pn_bimamba_encoder_ref(sd, hs[-1]))
    out = hs.pop()
    loss = out.square().mean()
    cot = 2.0 * out / out.numel()
    del out
    grads = {}
    for i in reversed(range(N_LAYERS)):
        _, cot, gp = _layer_ref(sds[i], hs.pop(), cot)
        grads.update({f"backbone_layers.{i}.{k}": v for k, v in gp.items()})
    torch.cuda.empty_cache()
    return loss, grads


def _worst(errs):
    k = max(errs, key=errs.get)
    return k, errs[k]


def test_training_shape_takes_the_wide_reduction_variants():
    """The sizes that make this file's checks differ from the small-batch tests: bimamba_reduce_partials switches from
    one row lane to 8 above 16 partial rows and to 32 above 96.  The scan's dA / dD / dbias partials have one row per
    (utterance, direction); the conv's weight and bias partials have bimamba_conv_bwd_slices rows."""
    lib = bm._lib.load()
    assert lib.bimamba_conv_bwd_slices(B, L, D_INNER) == 832 > 96
    assert B * NDIR == 128 > 96
    assert bm._lib.scan_plan(L, D_INNER, B * NDIR, True)[:2] == (32, 9)     # [dB | dC] partials: 9 channel groups


def test_fp32_captured_step_vs_oracle(oracle):
    """The benchmark's step captured without autocast and replayed once: the loss and the p.grad buffers the replay
    left, against the oracle at the fp32 bar (1e-4).  fp32 takes the same size-based dispatch as bf16 (partial-row
    counts, scan plan, GEMM tiles; the products on split-bf16 operands)."""
    ref_loss, ref_grads = oracle
    model, params, opt = _model()
    runner = _captured(model, params, opt, _batch(), bf16=False)
    loss = runner.run()
    torch.cuda.synchronize()
    named = _named(model)
    assert len(named) == 68
    loss_err = cmp.rel(loss, ref_loss)
    ratios = {n: cmp.check(n, p.grad, ref_grads[n], 1e-4, cmp.param(n, p.shape)) for n, p in named}
    print("fp32 captured step, worst slice ratio vs oracle:", _worst(ratios), "loss rel err", loss_err)
    assert loss_err < 1e-4


class _Recorder:
    """Forward hooks on the encoder layers: each layer's input and output, which autograd Function produced the
    output, and (tensor hook) the gradient that arrives at the output."""

    def __init__(self, model):
        n = len(model.backbone_layers)
        self.x, self.out, self.fn, self.cot = [None] * n, [None] * n, [None] * n, [None] * n
        self.handles = [layer.register_forward_hook(self._hook(i)) for i, layer in enumerate(model.backbone_layers)]

    def _hook(self, i):
        def fwd(mod, args, out):
            f_fused, seqlens = args
            assert seqlens is None
            self.x[i], self.out[i], self.fn[i] = f_fused.detach().clone(), out.detach().clone(), type(out.grad_fn).__name__

            def bwd(g):
                self.cot[i] = g.detach().clone()
            out.register_hook(bwd)
        return fwd

    def remove(self):
        for h in self.handles:
            h.remove()


def _outputs(loss, model):
    """What a caller of the step holds once it returns (bench.py --dump-outputs): the loss, every gradient the AdamW
    update applied and every parameter after it."""
    named = _named(model)
    res = {"loss": loss.detach().clone()}
    res.update({"grad." + n: p.grad.detach().clone() for n, p in named})
    res.update({"param." + n: p.detach().clone() for n, p in named})
    return res


def test_bf16_step_captured_sequenced_native_bitwise_and_vs_oracle(oracle):
    """The benchmark's arrangement exactly (bf16 autocast, FusedAdamW), one step three ways from identical weights:
    (a) the captured GraphedTrainStep, (b) eager inside ops.sequenced_block() (what the capture records), (c) eager on
    the native one-call layer entry points (the default).  All three give the same bits.  (c) layer by layer against the
    oracle on that layer's own input and output cotangent, and end to end (loss 2e-2, gradients 5e-2: the bars of the
    4-layer bf16 chain in test_model_tail_vs_reference_fixture).

    Per layer, the output and dx keep one layer's bf16 bar, 2e-2.  The parameter gradients get 3e-2, per slice.  On a
    B200 the largest of the 68 over the whole tensor is 2.4e-2, layer 2's x_proj.weight, in its C rows: a sum over 25 728 rows whose operands, dC and the
    conv output, are stored in bf16.  The next largest is 1.8e-2 (layer 1's dt_proj.bias), and the same step in fp32 is within 3e-5 of the oracle on every gradient (the fp32 test above), so the
    excess is the rounding of the stored bf16 operands, not the arithmetic."""
    ref_loss, ref_grads = oracle
    x = _batch()
    runs = {}
    model, params, opt = _model()
    runner = _captured(model, params, opt, x, bf16=True)
    runs["captured"] = _outputs(runner.run(), model)
    torch.cuda.synchronize()
    del runner, model, params, opt

    for name in ("sequenced", "native"):
        model, params, opt = _model()
        sds = [{k: v.detach().clone() for k, v in layer.state_dict().items()} for layer in model.backbone_layers]
        rec = _Recorder(model)
        if name == "sequenced":
            with bm.ops.sequenced_block():
                loss = _loss_fn(model, True)(x)
                loss.backward()
        else:
            loss = _loss_fn(model, True)(x)
            loss.backward()
        opt.step()
        torch.cuda.synchronize()
        rec.remove()
        native = ["EncoderLayerNativeFn" in f for f in rec.fn]
        assert native == [name == "native"] * N_LAYERS, rec.fn
        runs[name] = _outputs(loss, model)
    named = _named(model)                  # the native run's model, weights `sds` before its step, hooks `rec`
    grads = {n: p.grad for n, p in named}

    # (a) = (b) = (c), bit for bit
    assert len(runs["captured"]) == 1 + 2 * 68
    for other in ("sequenced", "native"):
        diff = [k for k, v in runs["captured"].items() if not torch.equal(v, runs[other][k])]
        assert not diff, (other, diff)

    # (c) layer by layer: the oracle fed the layer's recorded input and output cotangent
    ratios = {}
    for i in range(N_LAYERS):
        out_ref, dx_ref, gp_ref = _layer_ref(sds[i], rec.x[i], rec.cot[i])
        ratios[f"out.{i}"] = cmp.check(f"out.{i}", rec.out[i], out_ref, 2e-2, cmp.frames())
        if i > 0:                          # the gradient w.r.t. layer i's input arrives at layer i - 1's output
            ratios[f"dx.{i}"] = cmp.check(f"dx.{i}", rec.cot[i - 1], dx_ref, 2e-2, cmp.frames())
        for k, g in gp_ref.items():
            n = f"backbone_layers.{i}.{k}"
            # x_proj.weight keeps the whole-tensor rule (rho 1): on a B200 its column group [:, 128:160] in layer 2,
            # at 0.53 of the tensor's largest element, is 4.3e-2 off, 2.3e-2 of max|ref| - the rounding of its
            # bf16-stored operands described above, on a slice too large for any floor to cover
            rho = 1.0 if k.endswith("x_proj.weight") else None
            ratios[n] = cmp.check(n, grads[n], g, 3e-2, cmp.param(n, g.shape), rho=rho)
        del out_ref, dx_ref, gp_ref
    assert len(ratios) == N_LAYERS * 18 + N_LAYERS - 1
    print("bf16 step, per layer, worst slice ratio vs oracle:", _worst(ratios))

    # end to end against the 4-layer oracle
    e2e = {n: cmp.check("e2e " + n, g, ref_grads[n], 5e-2, cmp.param(n, g.shape)) for n, g in grads.items()}
    loss_err = cmp.rel(runs["native"]["loss"], ref_loss)
    print("bf16 step, end to end: loss rel err", loss_err, "worst gradient slice ratio", _worst(e2e))
    assert loss_err < 2e-2


def test_adamw_inside_the_captured_step_vs_torch_adamw():
    """FusedAdamW replayed from the graph reads lr, betas, eps, weight decay and the step count from device memory.
    Three replays on three batches, the lr changed (param_groups + sync_hyper()) before the third: after each, the
    update every parameter received against torch.optim.AdamW in fp64, fed the gradients the replay produced from the
    same parameters and the same starting state.

    The update (about 1e-5 here) is compared, not the parameter (about 1e-5 of which it is).  The parameter is stored in
    fp32, rounded after the weight decay and again after the step, so each element may differ from the exact update by
    one unit in the last place of the fp32 parameter; beyond that the bar is 1e-6 of the largest update of the tensor.
    The moments are compared directly at 1e-6."""
    model, params, opt = _model()
    runner = _captured(model, params, opt, _batch(), bf16=True)
    # the reference gets the hyper-parameters the device holds: fp32(0.999) is 1 + 1.3e-8 times 0.999, so 1 - beta2,
    # the weight of g^2 in exp_avg_sq, differs by 1.3e-5 between the two roundings
    f32 = lambda v: float(torch.tensor(v, dtype=torch.float32))
    g0 = opt.param_groups[0]
    ref_p = [p.detach().double().clone() for p in params]
    ref = torch.optim.AdamW(ref_p, lr=f32(g0["lr"]), betas=tuple(f32(b) for b in g0["betas"]), eps=f32(g0["eps"]),
                            weight_decay=f32(g0["weight_decay"]))
    names = [n for n, _ in _named(model)]
    worst = {}
    for k, lr in enumerate((1e-5, 1e-5, 3e-5)):
        if lr != opt.param_groups[0]["lr"]:
            opt.param_groups[0]["lr"] = lr
            opt.sync_hyper()
            ref.param_groups[0]["lr"] = f32(lr)
        before = [p.detach().clone() for p in params]
        runner.run(_batch(100 + k))
        torch.cuda.synchronize()
        with torch.no_grad():
            for r, b, p in zip(ref_p, before, params):
                r.copy_(b)
                r.grad = p.grad.detach().double()
        ref.step()
        errs = {}
        for n, r, b, p in zip(names, ref_p, before, params):
            d_ours = (p.detach() - b).double()            # exact: p and b are within a factor of 2 of each other
            d_ref = r.detach() - b.double()
            big = torch.maximum(p.detach().abs(), b.abs())
            ulp = (torch.nextafter(big, torch.full_like(big, float("inf"))) - big).double()
            excess = ((d_ours - d_ref).abs() - ulp).clamp_min(0.0)
            errs[n] = float(excess.max() / d_ref.abs().max())
            worst.setdefault("raw", {})[(k, n)] = cmp.rel(d_ours, d_ref)
        errs_m = {}
        sd = opt.state_dict()["state"]
        for i, (n, r) in enumerate(zip(names, ref_p)):
            errs_m["exp_avg." + n] = cmp.rel(sd[i]["exp_avg"], ref.state[r]["exp_avg"])
            errs_m["exp_avg_sq." + n] = cmp.rel(sd[i]["exp_avg_sq"], ref.state[r]["exp_avg_sq"])
            assert float(sd[i]["step"]) == k + 1
        print(f"AdamW replay {k + 1} (lr {lr:g}): update beyond 1 ulp", _worst(errs), "moments", _worst(errs_m))
        bad = {n: e for n, e in {**errs, **errs_m}.items() if not e < 1e-6}
        assert not bad, (k, bad)
    print("AdamW update, without the 1-ulp allowance:", _worst(worst["raw"]))


# ---------------------------------------------------------------------------------------------------------------------
# bimamba_reduce_partials: out[g*out_gs + j] (+)= sum_i part[g*part_gs + i*row_stride + j] in fixed order, with 1, 8 or 32
# row lanes (rows <= 16, <= 96, more)
# ---------------------------------------------------------------------------------------------------------------------
def _lanes(rows):
    return 1 if rows <= 16 else 8 if rows <= 96 else 32


@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows", [1, 16, 17, 96, 97, 832])
def test_reduce_partials_variants(rows, out_dtype, accumulate):
    """Each variant against an fp64 sum of the same partials, on column counts that are not multiples of 8, 32 or 256,
    several groups with padded group / row / output strides (the padding holds NaN, so a read outside the operand shows),
    and a grid larger than the kernel's cap of 148 x 64 CTAs (the grid-stride loop).  A second call gives the same bits,
    and output padding is left untouched."""
    cpb = 256 // _lanes(rows)                        # columns per CTA
    wide = (148 * 64 * cpb) // 2 + 3                 # 2 groups of `wide` columns: more column tiles than CTAs
    assert 2 * -(-wide // cpb) > 148 * 64
    layouts = [   # groups, cols, row_stride, part_gs, out_gs
        (1, 1, 1, 0, 0),
        (1, 1443, 1443, 0, 0),                                    # 288 x (4 + 1): the conv's [dw | db] rows
        (1, 4611, 4613, 0, 0),
        (3, 37, 41, rows * 41 + 5, 45),
        (2, 1443, 1450, rows * 1450 + 3, 1449),
        (2, wide, wide, rows * wide, wide + 8),
    ]
    gen = torch.Generator(device="cuda").manual_seed(rows * 4 + accumulate)
    for groups, cols, row_stride, part_gs, out_gs in layouts:
        span = (groups - 1) * part_gs + (rows - 1) * row_stride + cols
        part = torch.full((span + 7,), float("nan"), device="cuda")
        P = part.as_strided((groups, rows, cols), (part_gs, row_stride, 1))
        P.copy_(torch.randn(groups, rows, cols, device="cuda", generator=gen))
        out_span = (groups - 1) * out_gs + cols
        init = torch.full((out_span + 5,), -7.0, device="cuda").to(out_dtype)
        O0 = init.as_strided((groups, cols), (max(out_gs, 1), 1))
        O0.copy_(torch.randn(groups, cols, device="cuda", generator=gen).to(out_dtype))
        outs = []
        for _ in range(2):
            out = init.clone()
            bm.ops.reduce_raw(part, out, groups, rows, cols, part_gs, row_stride, out_gs, accumulate=bool(accumulate))
            outs.append(out)
        torch.cuda.synchronize()
        assert torch.equal(outs[0], outs[1])
        O = outs[0].as_strided((groups, cols), (max(out_gs, 1), 1))
        prev = O0.double() if accumulate else torch.zeros_like(O0, dtype=torch.float64)
        ref = P.double().sum(1) + prev
        # fp32 summation in any order: |error| <= (rows + 1) u32 sum|terms|; a 16-bit output adds one rounding
        bound = (rows + 1) * 2.0 ** -24 * (P.double().abs().sum(1) + prev.abs())
        if out_dtype == torch.bfloat16:
            bound = bound + 2.0 ** -8 * ref.abs()
        err = (O.double() - ref).abs()
        assert bool((err <= bound).all()), (groups, cols, float((err - bound).max()))
        mask = torch.ones_like(outs[0], dtype=torch.bool)
        mask.as_strided((groups, cols), (max(out_gs, 1), 1)).fill_(False)
        assert torch.equal(outs[0][mask], init[mask])            # the padding between and after the output rows
