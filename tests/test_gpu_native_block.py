"""The one-call native entry points on the GPU (include/bimamba.h; csrc/block.cu):
bimamba_block_fwd / bimamba_block_bwd (SURVEY 8b `conv_scan_bi` + projections) and bimamba_layer_fwd / bimamba_layer_bwd (the
whole PN_BiMambas_Encoder layer) - against the fp64 oracle (outputs and every gradient, bf16 tolerance 2e-2) and, bit for
bit, against the Python autograd Functions that sequence the same kernels (what a captured step replays).  In eager mode
these calls ARE the product path of `bimamba_inner_fn` / `PN_BiMambas_Encoder.forward`."""
import ctypes as C

import pytest
import torch

import bimamba_b200 as bm
from bimamba_b200 import ops
from oracle import bimamba_oracle as orc
from oracle import compare as cmp

pytestmark = pytest.mark.gpu

NAMES = ("in_proj.weight", "conv1d.weight", "conv1d.bias", "x_proj.weight", "dt_proj.weight", "dt_proj.bias", "A_log", "D",
         "out_proj.weight")


def _params(d_model, seed):
    p64 = orc.init_mamba_params(d_model, 16, seed=seed, dtype=torch.float64)
    return p64, [p64[n].float().cuda() for n in NAMES]


@pytest.mark.parametrize("d_model,Bsz,L,bidir,dtype", [
    (144, 3, 201, True, torch.bfloat16),      # the Phase-6 shape
    (144, 2, 5, True, torch.bfloat16),        # a single chunk: no checkpoints
    (64, 2, 260, True, torch.bfloat16),       # another width (d_inner 128, dt_rank 4)
    (144, 2, 77, False, torch.bfloat16),      # one direction: Mamba.forward
    (144, 2, 201, True, torch.float16),       # the reference's training dtype (src/main.py:1049)
])
def test_native_block_equals_autograd_function_bitwise(d_model, Bsz, L, bidir, dtype):
    _, w = _params(d_model, seed=L)
    g = torch.Generator().manual_seed(L)
    x = torch.randn(Bsz, L, d_model, generator=g).cuda().to(dtype)
    cot = torch.randn(Bsz, L, d_model, generator=g).cuda().to(dtype)
    # Python product path, both of its arrangements
    wp = [t.clone().requires_grad_(True) for t in w]
    xp = x.clone().requires_grad_(True)
    with ops.sequenced_block():               # the sequenced autograd Function (what a captured step replays)
        out_p = ops.bimamba_inner_fn(xp, *wp, bidirectional=bidir, compute_dtype=dtype)
        assert "BiMambaInnerFn" in type(out_p.grad_fn).__name__
        out_p.backward(cot)
    # eager default: the same call goes through the native entry points, same bits
    we = [t.clone().requires_grad_(True) for t in w]
    xe = x.clone().requires_grad_(True)
    out_e = ops.bimamba_inner_fn(xe, *we, bidirectional=bidir, compute_dtype=dtype)
    assert "BiMambaNativeFn" in type(out_e.grad_fn).__name__
    out_e.backward(cot)
    assert torch.equal(out_e, out_p) and torch.equal(xe.grad, xp.grad)
    for a, b in zip(we, wp):
        assert torch.equal(a.grad, b.grad)
    # native one-call path
    nb = ops.NativeBlock(x, *w, bidirectional=bidir, save_for_backward=True)
    grads = nb.backward(cot)
    torch.cuda.synchronize()
    assert torch.equal(nb.out, out_p.detach())
    assert torch.equal(grads[0], xp.grad)
    for name, gn, p in zip(NAMES, grads[1:], wp):
        assert gn.shape == p.grad.shape, name
        assert torch.equal(gn, p.grad), name
    # inference call (no checkpoints / ungated y written): same output from a smaller workspace
    nb2 = ops.NativeBlock(x, *w, bidirectional=bidir, save_for_backward=False)
    torch.cuda.synchronize()
    assert nb2.ws.numel() < nb.ws.numel()
    assert torch.equal(nb2.out, nb.out)


def test_native_block_vs_oracle_bf16():
    """Outputs and every gradient of the native calls against the fp64 oracle on bf16-rounded inputs (north_star: 2e-2),
    per slice (oracle/compare.py)."""
    p64, w = _params(144, seed=11)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(4, 201, 144, generator=g).bfloat16()
    cot = torch.randn(4, 201, 144, generator=g).bfloat16()
    pr = {k: v.float().double().requires_grad_(True) for k, v in p64.items()}
    xr = x.double().requires_grad_(True)
    ref = orc.bimamba_ref(pr, xr)
    (ref * cot.double()).sum().backward()
    nb = ops.NativeBlock(x.cuda(), *w)
    grads = nb.backward(cot.cuda())
    cmp.check("out", nb.out, ref, 2e-2, cmp.frames())
    cmp.check("dx", grads[0], xr.grad, 2e-2, cmp.frames())
    for name, gn in zip(NAMES, grads[1:]):
        cmp.check(name, gn, pr[name].grad, 2e-2, cmp.param(name, gn.shape))


def test_native_block_argument_errors_on_device():
    """Workspace too small / missing save_for_backward come back as codes with a message; nothing is launched."""
    _, w = _params(144, seed=3)
    x = torch.randn(2, 40, 144, device="cuda").bfloat16()
    nb = ops.NativeBlock(x, *w, save_for_backward=False)
    lib = bm._lib.load()
    with pytest.raises(RuntimeError, match="save_for_backward"):
        nb.backward(torch.zeros_like(x))
    d = nb.desc
    d.workspace_bytes = 16
    assert lib.bimamba_block_fwd(C.byref(d), None) == -10
    assert b"workspace too small" in lib.bimamba_last_error()


@pytest.mark.parametrize("mode", ["autocast_bf16", "autocast_fp16", "pure_bf16"])
@pytest.mark.parametrize("Bsz,L", [(3, 201), (2, 5)])
def test_native_encoder_layer_equals_sequenced_layer_bitwise(mode, Bsz, L):
    """PN_BiMambas_Encoder.forward in eager mode = bimamba_layer_fwd / bimamba_layer_bwd (one call each way); the
    sequenced Functions (what a captured step replays) give the same bits: output, dx and all 17 parameter gradients."""
    torch.manual_seed(7)
    enc = bm.PN_BiMambas_Encoder(144, 16).cuda()
    with torch.no_grad():
        enc.mamba.A_log.add_(0.1 * torch.randn_like(enc.mamba.A_log))
        enc.norm1.weight.add_(0.1 * torch.randn_like(enc.norm1.weight))
        enc.norm2.bias.add_(0.1 * torch.randn_like(enc.norm2.bias))
    x = torch.randn(Bsz, L, 144, device="cuda")
    cot = torch.randn(Bsz, L, 144, device="cuda")
    if mode == "pure_bf16":
        x, cot = x.bfloat16(), cot.bfloat16()
    ac = dict(device_type="cuda", dtype=torch.float16 if mode == "autocast_fp16" else torch.bfloat16,
              enabled=mode != "pure_bf16")
    runs = []
    for native in (False, True):
        for p in enc.parameters():
            p.grad = None
        xi = x.clone().requires_grad_(True)
        if native:
            with torch.autocast(**ac):
                out = enc(xi)
            assert "EncoderLayerNativeFn" in type(out.grad_fn).__name__
        else:
            with ops.sequenced_block(), torch.autocast(**ac):
                out = enc(xi)
            assert "EncoderLayerNativeFn" not in type(out.grad_fn).__name__
        assert out.dtype == x.dtype
        out.backward(cot)
        torch.cuda.synchronize()
        runs.append([out.detach().clone(), xi.grad.clone()] + [p.grad.clone() for p in enc.parameters()])
    names = ["out", "dx"] + [n for n, _ in enc.named_parameters()]
    for n, a, b in zip(names, *runs):
        assert a.dtype == b.dtype and torch.equal(a, b), n
    # scoring: no_grad forward through the native call (no statistics / checkpoints kept), same bits again
    with torch.no_grad(), torch.autocast(**ac):
        out_ng = enc(x)
    assert torch.equal(out_ng, runs[0][0])


def test_native_encoder_layer_vs_oracle_bf16():
    """The native layer against the fp64 oracle of the reference's PN_BiMambas_Encoder (north_star: 2e-2 in bf16), per
    slice (oracle/compare.py)."""
    torch.manual_seed(3)
    enc = bm.PN_BiMambas_Encoder(144, 16).cuda()
    x = torch.randn(4, 201, 144)
    cot = torch.randn(4, 201, 144)
    pr = {k: v.detach().double().cpu().requires_grad_(True) for k, v in enc.state_dict().items()}
    xr = x.double().requires_grad_(True)
    ref = orc.pn_bimamba_encoder_ref(pr, xr)
    (ref * cot.double()).sum().backward()
    xd = x.cuda().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = enc(xd)
    assert "EncoderLayerNativeFn" in type(out.grad_fn).__name__
    out.backward(cot.cuda())
    cmp.check("out", out, ref, 2e-2, cmp.frames())
    cmp.check("dx", xd.grad, xr.grad, 2e-2, cmp.frames())
    for name, p in enc.named_parameters():
        cmp.check(name, p.grad, pr[name].grad, 2e-2, cmp.param(name, p.shape))
