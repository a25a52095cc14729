"""The per-slice rule of oracle/compare.py, on fp64 references built with the oracle at the GPU tests' own shapes: the
bidirectional scan at 2 x 40 x 201 (tests/test_gpu_scan_bwd_passes.py's layout), one bidirectional block and one
encoder layer at d_model 144, 3 x 201, and one variable-length block batch (tests/test_gpu_varlen_train.py's lengths).

Two things are pinned.  Correct arithmetic passes with margin: the oracle evaluated in fp32 passes the fp32 rule (1e-4,
rho 1e-3) at a tenth of the tolerance, and the oracle on 16-bit-rounded inputs with its outputs rounded to 16 bits
passes the 16-bit rule (rho 1e-2) at a tenth of fp16's 5e-3 and a fifth of bf16's 2e-2 (rounding to bf16 alone moves
an element by up to 2^-8 of itself, 0.195 of 2e-2).  Named faults fail, and the failure names the slice: each one at
the tolerance and rho the GPU tests use.  A rho too large lets the faults through; one too small fails the fp32 proxy.
"""
import re

import pytest
import torch

from oracle import bimamba_oracle as orc
from oracle import compare as cmp

F32, B16 = cmp.TOL[torch.float32], cmp.TOL[torch.bfloat16]
LENGTHS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 40]
# (B, ndir, D, L) activations, (B, ndir, N, L) dB / dC
ACT = cmp.scan_act(0, 2, 3, dir=1)
SCAN = {"out": ACT, "du": ACT, "ddelta": ACT, "dz": ACT, "dB": cmp.scan_state(0, 2, dir=1),
        "dC": cmp.scan_state(0, 2, dir=1), "dA": cmp.CHANNEL_STATE, "dD": cmp.CHANNELS, "dbias": cmp.CHANNELS}


def _scan(in_dtype, wide):
    """Both directions of the scan on one set of operands (direction 1 walks time backwards), output and every
    gradient, evaluated in `wide`, on operands rounded to `in_dtype`."""
    u, delta, z, Bm, Cm, A, Dp, bias = orc.scan_inputs(2, 40, 201, seed=0, dtype=in_dtype)
    cot = torch.randn(2, 2, 40, 201, generator=torch.Generator().manual_seed(1)).to(in_dtype)
    A_, D_, b_ = (t.to(wide).requires_grad_(True) for t in (A, Dp, bias))
    res = {k: [] for k in ("out", "du", "ddelta", "dz", "dB", "dC")}
    for di in range(2):
        fl = (lambda t: t.flip(-1)) if di else (lambda t: t)
        ins = [fl(t).to(wide, copy=True).requires_grad_(True) for t in (u, delta, z, Bm, Cm)]
        y = orc.selective_scan_ref(ins[0], ins[1], A_, ins[3], ins[4], D_, ins[2], b_, delta_softplus=True)
        (y * fl(cot[:, di]).to(wide)).sum().backward()
        res["out"].append(fl(y.detach()))
        for k, t in zip(("du", "ddelta", "dz", "dB", "dC"), ins):
            res[k].append(fl(t.grad))
    res = {k: torch.stack(v, 1) for k, v in res.items()}
    res.update(dA=A_.grad, dD=D_.grad, dbias=b_.grad)
    return res


def _block(in_dtype, wide, layer):
    """One bidirectional block (or one encoder layer) at d_model 144, 3 x 201: output, dx and every parameter
    gradient, evaluated in `wide` on inputs and parameters rounded to `in_dtype`."""
    if layer:
        p = orc.init_encoder_params(144, 16, seed=3)
        fn = orc.pn_bimamba_encoder_ref
    else:
        p = orc.init_mamba_params(144, 16, seed=201, dtype=torch.float64)
        fn = orc.bimamba_ref
    g = torch.Generator().manual_seed(201)
    x = torch.randn(3, 201, 144, generator=g)
    cot = torch.randn(3, 201, 144, generator=g).to(in_dtype)
    pr = {k: v.float().to(in_dtype).to(wide).requires_grad_(True) for k, v in p.items()}
    xr = x.to(in_dtype).to(wide).requires_grad_(True)
    out = fn(pr, xr)
    (out * cot.to(wide)).sum().backward()
    res = {"out": out.detach(), "dx": xr.grad}
    res.update({k: v.grad for k, v in pr.items()})
    return res


def _varlen(in_dtype, wide):
    """A right-padded block batch at tests/test_gpu_varlen_train.py's lengths, every utterance run alone: output and
    dx (B, T, 144) with zeros at padded frames, and the parameter gradients summed over the utterances."""
    p = orc.init_mamba_params(144, 16, seed=1, dtype=torch.float64)
    g = torch.Generator().manual_seed(11)
    T = max(LENGTHS)
    x = torch.randn(len(LENGTHS), T, 144, generator=g).to(in_dtype)
    w = torch.randn(len(LENGTHS), T, 144, generator=g).to(in_dtype)
    pr = {k: v.float().to(in_dtype).to(wide).requires_grad_(True) for k, v in p.items()}
    out = torch.zeros(x.shape, dtype=wide)
    dx = torch.zeros(x.shape, dtype=wide)
    for b, n in enumerate(LENGTHS):
        xb = x[b:b + 1, :n].to(wide).requires_grad_(True)
        y = orc.bimamba_ref(pr, xb)
        (y * w[b:b + 1, :n].to(wide)).sum().backward()
        out[b, :n], dx[b, :n] = y.detach()[0], xb.grad[0]
    res = {"out": out, "dx": dx}
    res.update({k: v.grad for k, v in pr.items()})
    return res


def _slicings(case, name, t):
    if case == "scan":
        return SCAN[name]
    if name in ("out", "dx"):
        return cmp.frames()
    return cmp.param(name, t.shape)


CASES = {"scan": _scan, "block": lambda i, w: _block(i, w, False), "layer": lambda i, w: _block(i, w, True),
         "varlen": _varlen}


@pytest.fixture(scope="module")
def refs():
    """fp64 references of every case on fp32 and on bf16-rounded inputs, built once."""
    return {(case, dt): fn(dt, torch.float64) for case, fn in CASES.items()
            for dt in (torch.float32, torch.bfloat16, torch.float16)}


@pytest.mark.parametrize("case", list(CASES))
def test_fp32_proxy_passes_with_margin(refs, case):
    """The oracle itself evaluated in fp32 - a plain fp32 implementation - is within a tenth of the fp32 rule on every
    slice of every tensor."""
    got = CASES[case](torch.float32, torch.float32)
    for name, ref in refs[(case, torch.float32)].items():
        assert cmp.check(name, got[name], ref, F32, _slicings(case, name, ref)) < 0.1, name


@pytest.mark.parametrize("dtype,margin", [(torch.float16, 0.1), (torch.bfloat16, 0.2)])
@pytest.mark.parametrize("case", list(CASES))
def test_16bit_proxy_passes_with_margin(refs, case, dtype, margin):
    """Outputs rounded to 16 bits from the fp64 oracle on 16-bit-rounded inputs are within `margin` of the rule.  The
    kernels store activations and data gradients in the 16-bit type and parameter gradients in fp32, and so does this."""
    for name, ref in refs[(case, dtype)].items():
        got = ref.to(dtype if name in ("out", "dx", "du", "ddelta", "dz", "dB", "dC") else torch.float32)
        assert cmp.check(name, got, ref, cmp.TOL[dtype], _slicings(case, name, ref)) < margin, name


def _fault(t, fn):
    t = t.clone()
    fn(t)
    return t


def _swap_rows(a, b):
    def fn(t):
        t[[a, b]] = t[[b, a]]
    return fn


# case, tensor, fault, tolerance, the slice that must report it (regex), whether today's whole-tensor rule catches it
FAULTS = {
    # the second pass of eight states: a state lost, and the pass scaled
    "dA state 13 zero": ("scan", "dA", lambda t: t[:, 13].zero_(), B16, r"dA\[:, 13\]", True),
    "dA states 8-15 x1.3": ("scan", "dA", lambda t: t[:, 8:].mul_(1.3), B16, r"dA\[:, (8|9|1[0-5])\]", False),
    "dB states 8-15 x1.3": ("scan", "dB", lambda t: t[:, :, 8:].mul_(1.3), B16, r"dB\[\d, \d, (8|9|1[0-5])\]", True),
    "dC states 8-15 x1.3": ("scan", "dC", lambda t: t[:, :, 8:].mul_(1.3), B16, r"dC\[\d, \d, (8|9|1[0-5])\]", True),
    # one channel of the data gradients lost
    "ddelta channel 25 zero": ("scan", "ddelta", lambda t: t[:, :, 25].zero_(), B16, r"ddelta\[\d, \d, 25\]", True),
    # a 1 % error on one channel of dA, at the fp32 bar: channel 32, the smallest (6e-3 of the tensor's largest)
    "dA channel 32 x1.01": ("scan", "dA", lambda t: t[32].mul_(1.01), F32, r"dA\[32\]", False),
    # the dt_proj data-gradient columns of [dB | dC | ddt_r], written in place: the dt rows of x_proj.weight.grad
    "x_proj dt rows x1.2": ("block", "x_proj.weight", lambda t: t[:9].mul_(1.2), B16, r"x_proj.weight\[dt\]", False),
    # finalize's [B | C | dt_r] -> [dt_r | B | C] permutation off by one: the last dt_r column and the first B column
    "x_proj rows 8 <-> 9": ("block", "x_proj.weight", _swap_rows(8, 9), B16, r"x_proj.weight\[dt\]", True),
    # the last partial 8-step chunk of direction 1 (which walks time backwards: frame 0 of 201)
    "du dir 1 last chunk zero": ("scan", "du", lambda t: t[:, 1, :, :201 % 8].zero_(), B16, r"du\[\d, 1, :, 0:8\]",
                                 True),
    # the shortest utterance of a variable-length batch, at the bf16 bar of the varlen gradient tests (5e-2)
    "varlen shortest dx x1.1": ("varlen", "dx", lambda t: t[0].mul_(1.1), 5e-2, r"dx\[0(, 0:8)?\]", True),
    # the tail of the second 32-channel group in a 40-channel case
    "dbias channel 39 zero": ("scan", "dbias", lambda t: t[39].zero_(), B16, r"dbias\[39\]", True),
}


@pytest.mark.parametrize("fault", list(FAULTS))
def test_named_fault_fails_and_names_its_slice(refs, fault):
    case, name, fn, tol, where, whole_catches = FAULTS[fault]
    ref = refs[(case, torch.float32)][name]
    got = _fault(ref, fn)
    with pytest.raises(AssertionError) as e:
        cmp.check(name, got, ref, tol, _slicings(case, name, ref))
    label = re.search(r"worst slice (\S+(?:, \S+)*): error", str(e.value)).group(1)
    assert re.fullmatch(where, label), (fault, label)
    assert (cmp.rel(got, ref) >= tol) == whole_catches, (fault, cmp.rel(got, ref))


def test_slicing_labels_and_floor():
    """Groups with a partial tail, named blocks, and the rho floor on a slice that is zero in the reference."""
    ref = torch.arange(1.0, 41.0).double()
    got = ref.clone()
    got[39] += 0.5
    assert cmp.worst(got, ref, cmp.CHANNELS, 1e-3, "v")[:2] == (0.5 / 40, "v[39]")
    ref[5] = 0.0
    got = ref.clone()
    got[5] = 1e-3                       # measured against rho * 40, not against 0
    err, label, _ = cmp.worst(got, ref, cmp.CHANNELS, 1e-3, "v")
    assert label == "v[5]" and abs(err - 1e-3 / (1e-3 * 40)) < 1e-12
    w = torch.ones(41, 64).double()
    g = w.clone()
    g[40, 33] = 2.0
    assert cmp.worst(g, w, cmp.param("x_proj.weight", w.shape), 1e-3, "x")[1] == "x[C]"
    t = torch.ones(2, 2, 40, 201).double()
    g = t.clone()
    g[1, 0, :, 200] = 0.0
    assert cmp.worst(g, t, ACT, 1e-3, "du")[1] == "du[1, 0, 0]"
