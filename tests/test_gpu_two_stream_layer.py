"""The encoder layer's two-stream native calls (bimamba_layer_fwd_side / bimamba_layer_bwd_side: weight packing and
parameter gradients on a second stream) against the same calls on one stream, bit for bit: the backend's loss, output
gradient and every parameter gradient, eager and captured in a CUDA graph, bf16 and fp16 autocast, fixed length and
with per-utterance frame counts, 1 and 4 layers."""
import pytest
import torch

import bimamba_b200 as bm
from bimamba_b200 import ops

pytestmark = pytest.mark.gpu


def _model(n_layers):
    torch.manual_seed(11)
    model = bm.BiMambaBackend(144, n_layers, 16).cuda()
    with torch.no_grad():
        for layer in model.backbone_layers:
            layer.mamba.A_log.add_(0.1 * torch.randn_like(layer.mamba.A_log))
            layer.norm1.weight.add_(0.1 * torch.randn_like(layer.norm1.weight))
            layer.norm2.bias.add_(0.1 * torch.randn_like(layer.norm2.bias))
    return model


def _step_fn(model, dtype, lengths):
    def step(x, seqlens=None):
        with torch.autocast("cuda", dtype=dtype):
            out = model.forward_features(x, seqlens, mask_padding=seqlens is not None)
        return ops.mean_square_loss(out)
    return step


@pytest.mark.parametrize("n_layers", [1, 4])
@pytest.mark.parametrize("varlen", [False, True])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("captured", [False, True])
def test_two_stream_layer_equals_one_stream_bitwise(n_layers, varlen, dtype, captured, monkeypatch):
    model = _model(n_layers)
    params = list(model.parameters())
    B, L = 6, 201
    x = torch.randn(B, L, 144, generator=torch.Generator().manual_seed(3)).cuda()
    lengths = torch.tensor([201, 150, 7, 201, 90, 1], dtype=torch.int32, device="cuda") if varlen else None
    step = _step_fn(model, dtype, lengths)
    args = (x,) if lengths is None else (x, lengths)

    def zero_grad():
        for p in params:
            p.grad = None

    def grads():
        return [p.grad.clone() if p.grad is not None else None for p in params]

    # reference: the single-stream native calls, eager
    monkeypatch.setattr(ops, "SIDE_STREAM", False)
    zero_grad()
    xr = x.clone().requires_grad_(True)
    loss_ref = step(xr, *args[1:])
    loss_ref.backward()
    torch.cuda.synchronize()
    ref = [loss_ref.detach().clone(), xr.grad.clone()] + grads()
    del loss_ref, xr                   # the eager autograd graph (its AccumulateGrad nodes) must not outlive the run
    monkeypatch.setattr(ops, "SIDE_STREAM", True)

    if captured:
        runner = bm.GraphedTrainStep(step, x, zero_grad, None, warmup=2, lengths=lengths)
        loss = runner.run(x, lengths)
        torch.cuda.synchronize()
        got = [loss.detach().clone(), None] + grads()
    else:
        zero_grad()
        xt = x.clone().requires_grad_(True)
        loss = step(xt, *args[1:])
        loss.backward()
        torch.cuda.synchronize()
        got = [loss.detach().clone(), xt.grad.clone()] + grads()
    names = ["loss", "dx"] + [n for n, _ in model.named_parameters()]
    for n, a, b in zip(names, got, ref):
        if a is None or b is None:
            assert n == "dx" or (a is None and b is None), n
            continue
        assert a.dtype == b.dtype and torch.equal(a, b), n


def test_native_layer_is_what_the_capture_records():
    """Under capture the encoder layer goes through the native two-stream calls, not the sequenced Functions."""
    model = _model(1)
    x = torch.randn(2, 9, 144, device="cuda", requires_grad=True)
    assert ops.SIDE_STREAM
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            model.forward_features(x)          # warm-up: lazy state (side stream, events) made outside the capture
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model.forward_features(x)
    assert "EncoderLayerNativeFn" in type(out.grad_fn).__name__


def test_block_backward_side_stream_equals_one_stream_bitwise():
    """bimamba_block_bwd_side with and without the second stream."""
    torch.manual_seed(5)
    m = bm.Mamba(144, 16).cuda()
    x = torch.randn(4, 201, 144, device="cuda").bfloat16()
    dout = torch.randn(4, 201, 144, device="cuda").bfloat16()
    nb = ops.NativeBlock(x, m.in_proj.weight, m.conv1d.weight, m.conv1d.bias, m.x_proj.weight, m.dt_proj.weight,
                         m.dt_proj.bias, m.A_log, m.D, m.out_proj.weight)
    one = [t.clone() for t in nb.backward(dout, two_stream=False)]
    two = nb.backward(dout, two_stream=True)
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(one, two)):
        assert torch.equal(a, b), i
