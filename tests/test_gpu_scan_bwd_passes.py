"""The selective-scan backward kernel (two passes of eight states per 8-step chunk) against the fp64 oracle, called at
the op level in all three delta modes - delta given, and the fused dt projection at rank 9 (the training step's) and
rank 16 - with fp32, bf16 and fp16 I/O, both directions in one launch, 40 channels (a full and a partial 32-channel
group), and sequence lengths that give a single step, a partial chunk, exactly one chunk, and a partial last chunk.
Every case also runs the backward a second time and requires the same bits.  Each output and gradient is measured per
slice (oracle/compare.py): per (utterance, direction, channel), per (utterance, direction, 8-step chunk), per state of
dB | dC, per state and channel of dA, per channel of dD and dbias."""
import pytest
import torch

import bimamba_b200 as bm
from bimamba_b200 import ops
from oracle import bimamba_oracle as orc
from oracle import compare as cmp

pytestmark = pytest.mark.gpu

TOL = cmp.TOL
N, XW = 16, 48
# (B, ndir, L, D) activations and data gradients; (B, ndir, L, 2N) [dB | dC]: one slice per column is one per state
ACT = cmp.scan_act(0, 3, 2, dir=1)
SLICES = {"out": ACT, "du": ACT, "ddelta": ACT, "dz": ACT, "dB|dC": cmp.scan_state(0, 3, dir=1),
          "dA": cmp.CHANNEL_STATE, "dD": cmp.CHANNELS, "dbias": cmp.CHANNELS}


def _case(mode, dtype, L, Bsz=2, D=40, ndir=2, seed=0, dtr_padded=True):
    """mode: 0 = delta given, else the dt_proj rank.  Checks every output and gradient at TOL[dtype]."""
    g = torch.Generator().manual_seed(seed)
    R = mode
    dev = "cuda"
    xc = ops.per_dir(Bsz, L, ndir, D, dev, dtype)                    # u: (B, ndir, L, D) view of (B, L, ndir, D)
    xc.copy_(torch.randn(Bsz, ndir, L, D, generator=g).to(dtype))
    xdbl = torch.zeros((Bsz, L, ndir, XW), dtype=dtype)
    xdbl[..., :2 * N] = torch.randn(Bsz, L, ndir, 2 * N, generator=g).to(dtype)
    if R:
        xdbl[..., 2 * N:2 * N + R] = (torch.randn(Bsz, L, ndir, R, generator=g) * 0.5).to(dtype)
    xd4 = xdbl.to(dev).permute(0, 2, 1, 3)
    bc = xd4[..., :2 * N]
    dtr = (xd4[..., 2 * N:] if dtr_padded else xd4[..., 2 * N:2 * N + R]) if R else None
    Wdt = (torch.randn(D, R, generator=g) / R ** 0.5).to(dev) if R else None
    delta = None
    if not R:
        delta = ops.per_dir(Bsz, L, ndir, D, dev, dtype)
        delta.copy_((0.5 * torch.randn(Bsz, ndir, L, D, generator=g)).to(dtype))
    z = torch.randn(Bsz, L, D, generator=g).to(dtype).to(dev)
    z4 = z.unsqueeze(1).expand(Bsz, ndir, L, D)
    A = (-torch.exp(torch.log(torch.arange(1, N + 1, dtype=torch.float32)).repeat(D, 1)
                    + 0.1 * torch.randn(D, N, generator=g))).to(dev)
    Dp = (1 + 0.1 * torch.randn(D, generator=g)).to(dev)
    dt = torch.exp(torch.rand(D, generator=g) * 4.6 - 6.9)
    bias = (dt + torch.log(-torch.expm1(-dt))).to(dev)
    dout = ops.per_dir(Bsz, L, ndir, D, dev, dtype)
    dout.copy_(torch.randn(Bsz, ndir, L, D, generator=g).to(dtype))

    out, ckpt, ypre = ops.scan_fwd_raw(xc, z4, delta, bc, dtr, Wdt, A, Dp, bias, True, True, dtr_padded=dtr_padded)
    run = lambda: ops.scan_bwd_raw(xc, z4, delta, bc, dtr, Wdt, A, Dp, bias, True, dout, ckpt, ypre,
                                   dtr_padded=dtr_padded, bc_out_dtype=torch.float32)
    got = run()
    again = run()
    torch.cuda.synchronize()
    for a, b in zip(got, again):
        assert torch.equal(a, b), "backward is not bitwise repeatable"
    du, ddelta, dz, dbc, dA, dD, dbias = got

    # fp64 oracle per direction (direction 1 walks time backwards), on the dtype-rounded inputs
    A64 = A.double().cpu().requires_grad_(True)
    D64 = Dp.double().cpu().requires_grad_(True)
    b64 = bias.double().cpu().requires_grad_(True)
    ref = {k: [] for k in ("out", "u", "delta", "z", "bc")}
    for di in range(ndir):
        fl = (lambda t: t.flip(-1)) if di else (lambda t: t)
        u_d = fl(xc[:, di].double().cpu().transpose(1, 2)).requires_grad_(True)
        if R:
            dr = xd4[:, di, :, 2 * N:2 * N + R].double().cpu()
            draw = dr @ Wdt.double().cpu().t()
        else:
            draw = delta[:, di].double().cpu()
        dl_d = fl(draw.transpose(1, 2)).detach().requires_grad_(True)
        z_d = fl(z.double().cpu().transpose(1, 2)).requires_grad_(True)
        bc_d = fl(bc[:, di].double().cpu().transpose(1, 2)).requires_grad_(True)
        y = orc.selective_scan_ref(u_d, dl_d, A64, bc_d[:, :N], bc_d[:, N:], D64, z_d, b64, delta_softplus=True)
        ref["out"].append(fl(y).transpose(1, 2))
        (y * fl(dout[:, di].double().cpu().transpose(1, 2))).sum().backward()
        ref["u"].append(fl(u_d.grad).transpose(1, 2))
        ref["delta"].append(fl(dl_d.grad).transpose(1, 2))
        ref["z"].append(fl(z_d.grad).transpose(1, 2))
        ref["bc"].append(fl(bc_d.grad).transpose(1, 2))
    stack = lambda k: torch.stack(ref[k], 1)
    tol = TOL[dtype]
    for name, got, want in (("out", out, stack("out")), ("du", du, stack("u")), ("ddelta", ddelta, stack("delta")),
                            ("dz", dz, stack("z")), ("dB|dC", dbc, stack("bc")), ("dA", dA, A64.grad),
                            ("dD", dD, D64.grad), ("dbias", dbias, b64.grad)):
        cmp.check(name, got, want, tol, SLICES[name])


@pytest.mark.parametrize("L", [1, 7, 8, 9, 201])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mode", [0, 9, 16])
def test_scan_backward_passes(mode, dtype, L):
    _case(mode, dtype, L, seed=100 * mode + L)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scan_backward_passes_unpadded_dt_rows(dtype):
    """dt_r rows of width 9 (not 16-byte friendly): the element-wise staging path."""
    _case(9, dtype, 37, seed=7, dtr_padded=False)
