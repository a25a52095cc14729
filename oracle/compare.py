"""Per-slice comparison of a CUDA result with its fp64 reference.  TEST INFRASTRUCTURE ONLY.

A single number per tensor, max|got - ref| / max|ref|, lets a slice whose values are small next to the tensor's
largest element be badly wrong: a state of the scan's dA, a channel of dt_proj.bias.grad, the dt rows of
x_proj.weight.grad, a short utterance in a padded batch.  Those slices are where the kernels branch, so the tests
measure each one against its own magnitude:

    err(S) = max_S |got - ref| / max(max_S |ref|, rho * max |ref|)

and a check passes when err(S) < tol for every slice S.  The whole tensor is always one of the slices; with no other
slicing this is the single number above, which is still the right measure for a scalar such as a loss.  rho is a
floor: a slice that is almost zero by cancellation is measured against rho times the tensor's largest element, not
against its own, since no correct kernel has a relative precision below its rounding there.

A slicing is a dict {dim: part}.  part = k cuts that dimension into groups of k indices (1: every index; the last
group may be partial); part = {name: (start, stop)} cuts it into named blocks.  Dimensions not named are taken whole.
The slices of a slicing are the product of its parts.
"""
from __future__ import annotations

import os
from typing import Dict, Iterable, Optional, Union

import torch

Part = Union[int, Dict[str, tuple]]
Slicing = Dict[int, Part]

# north_star tolerances and the starting floor rho of each precision.  A family that needs a larger floor carries it
# (Family below); a single check that needs one passes it, with the measurement beside the call.
TOL = {torch.float32: 1e-4, torch.bfloat16: 2e-2, torch.float16: 5e-3}
RHO_FP32, RHO_16BIT = 1e-3, 1e-2
CHUNK = 8          # time steps per chunk of the scan kernels (and frames per chunk of a layer's activations)
GROUP = 32         # channels per group of the scan, conv and reduction kernels


class Family(list):
    """The slicings of one family of tensors, with the floor rho it takes at the fp32 bar and at the 16-bit bars."""

    def __init__(self, slicings, rho32: float = RHO_FP32, rho16: float = RHO_16BIT):
        super().__init__(slicings)
        self.rho = (rho32, rho16)


def default_rho(tol: float, slicings=()) -> float:
    """fp32 bars (<= 1e-4) take the fp32 floor; the 16-bit bars (5e-3 and up) the 16-bit one."""
    rho32, rho16 = getattr(slicings, "rho", (RHO_FP32, RHO_16BIT))
    return rho32 if tol <= 1e-4 else rho16


# --------------------------------------------------------------------------------------------------- slicings
def scan_act(utt: int, chan: int, time: int, dir: Optional[int] = None):
    """Scan activations and data gradients (out, du, ddelta, dz): per (utterance, direction, channel) and per
    (utterance, direction, 8-step chunk), the partial last chunk included."""
    lead = {utt: 1} if dir is None else {utt: 1, dir: 1}
    return [{**lead, chan: 1}, {**lead, time: CHUNK}]


def scan_state(utt: int, state: int, dir: Optional[int] = None):
    """Scan dB, dC: per (utterance, direction, state)."""
    lead = {utt: 1} if dir is None else {utt: 1, dir: 1}
    return [{**lead, state: 1}]


# dA (the scan op), (channels, states): per channel and per state
CHANNEL_STATE = Family([{0: 1}, {1: 1}])
# per-channel vectors of the ops (dD, dbias, conv1d.bias.grad, LayerNorm gradients, biases): per element (each measured
# against the rho floor at least) and per 32-channel group.  These are sums over every frame that cancel to 1e-4 .. 2e-2
# of the largest channel, and their terms carry the rounding of the whole forward and backward: plain fp32 arithmetic
# (the oracle evaluated in fp32, tests/test_compare_cpu.py) leaves up to 7e-7 of max|ref| in a channel of any size, 0.86
# of the fp32 bar at rho 1e-3 (encoder layer conv1d.bias channel 42, at 2.6e-2 of the largest).  An fp32 floor of 1e-1
# keeps every channel of that proxy below a tenth of the bar; on the B200 the ops' worst is 0.15 of it (dbias, D = 37).
CHANNELS = Family([{0: 1}, {0: GROUP}], rho32=1e-1)
# The same vectors and A_log.grad as parameter gradients of a block, layer or model tail: their terms are GEMM and scan
# outputs stored in the compute type, so the cancellation above meets that type's rounding.  Measured on a B200 at the
# starting floors (1e-3 / 1e-2), as absolute errors over max|ref|, each floor below is 3x the worst:
#   16-bit, per-channel vectors: dt_proj.bias[143] of test_block_other_widths[bf16-80-2-130] is 9.7e-3 of max|ref|
#     (channel at 3.3e-5 of the largest; 0.49 of the 2e-2 bar over the whole tensor): no floor below max|ref| holds, so
#     these vectors are held to the whole-tensor rule (rho 1);
#   16-bit, A_log: A_log[0] of the same test, 4.8e-3 of max|ref| on a channel at 0.16 of the largest: rho 1;
#   fp32, per-channel vectors: fusion.ln_wavlm.weight[623] of test_model_tail_vs_reference_fixture[fp32] (four layers
#     and the fusion block against a reference fixture) is 1.75e-5 of max|ref|: rho 0.6;
#   fp32, A_log: backbone_layers.2.mamba.A_log[98] of test_tail_training_matches_oracle[fp32] is 2e-6 of max|ref|:
#     rho 0.1 (0.2 of the bar).
# The same sums at op level (CHANNELS, CHANNEL_STATE) keep their floors: the scan's dA, dD and dbias stay below 4e-3 of
# the 16-bit bar at rho 1e-2.
PARAM_CHANNELS = Family([{0: 1}, {0: GROUP}], rho32=0.6, rho16=1.0)
PARAM_CHANNEL_STATE = Family([{0: 1}, {1: 1}], rho32=0.1, rho16=1.0)
# per utterance (head features and logits)
UTT = [{0: 1}]


def frames(utt: int = 0, time: int = 1):
    """Layer, backend and head inputs / outputs (B, T, C): per utterance and per (utterance, 8-frame chunk)."""
    return [{utt: 1}, {utt: 1, time: CHUNK}]


def param(name: str, shape, d_state: int = 16):
    """The slicing of a parameter (or its gradient) by the name it has in the module."""
    leaf = name.split("mamba.")[-1]
    if leaf.endswith("x_proj.weight"):          # rows [dt_rank | B | C], and column groups
        r = shape[0] - 2 * d_state
        return [{0: {"dt": (0, r), "B": (r, r + d_state), "C": (r + d_state, r + 2 * d_state)}}, {1: GROUP}]
    if leaf.endswith("in_proj.weight"):         # the x half and the z half
        h = shape[0] // 2
        return [{0: {"x": (0, h), "z": (h, 2 * h)}}]
    if leaf.endswith("conv1d.weight"):          # (D, 1, K): per tap
        return [{len(shape) - 1: 1}]
    if leaf.endswith("dt_proj.weight"):         # (D, rank): per rank column
        return [{1: 1}]
    if leaf.endswith("A_log"):
        return PARAM_CHANNEL_STATE
    if len(shape) == 1:
        return PARAM_CHANNELS
    if len(shape) == 2:                         # out_proj, the feed-forward and the fusion weights: groups of 32 rows
        return [{0: GROUP}]
    return []


# --------------------------------------------------------------------------------------------------- the rule
def _slice_max(x: torch.Tensor, slicing: Slicing):
    """Maximum of x (non-negative) over every slice of `slicing`; returns (maxima, dims, labels per dim)."""
    dims = sorted(slicing)
    other = [d for d in range(x.dim()) if d not in slicing]
    if other:
        x = x.amax(dim=other)
    labels = []
    for i, d in enumerate(dims):
        part, n = slicing[d], x.shape[i]
        if isinstance(part, int):
            k = -(-n // part)
            if k * part != n:
                pad = list(x.shape)
                pad[i] = k * part - n
                x = torch.cat([x, x.new_zeros(pad)], i)
            x = x.unflatten(i, (k, part)).amax(i + 1)
            labels.append([str(j) if part == 1 else f"{j * part}:{min(n, (j + 1) * part)}" for j in range(k)])
        else:
            x = torch.stack([x.narrow(i, a, b - a).amax(i) for a, b in part.values()], i)
            labels.append(list(part))
    return x, dims, labels


def _label(name, ndim, dims, labels, flat):
    idx = [":"] * ndim
    for d, lab in reversed(list(zip(dims, labels))):
        idx[d] = lab[flat % len(lab)]
        flat //= len(lab)
    while idx and idx[-1] == ":":
        idx.pop()
    return f"{name}[{', '.join(idx)}]" if idx else name


def worst(got, ref, slicings: Iterable[Slicing] = (), rho: float = RHO_FP32, name: str = "t"):
    """(error, label, slice max|ref| over tensor max|ref|) of the worst slice; the whole tensor is always a slice."""
    got = torch.as_tensor(got).detach().double().cpu()
    ref = torch.as_tensor(ref).detach().double().cpu()
    assert got.shape == ref.shape, (name, tuple(got.shape), tuple(ref.shape))
    diff, mag = (got - ref).abs(), ref.abs()
    floor = max(rho * float(mag.max()) if mag.numel() else 0.0, 1e-30)
    best = None
    for slicing in [{}] + list(slicings):
        d, dims, labels = _slice_max(diff, slicing)
        m, _, _ = _slice_max(mag, slicing)
        err = torch.nan_to_num(d / m.clamp_min(floor), nan=float("inf")).reshape(-1)
        k = int(err.argmax())
        # a tie with the whole tensor is named by the slice; between slicings, the first listed names it
        if best is None or float(err[k]) > best[0] or (float(err[k]) == best[0] and best[1] == name):
            best = (float(err[k]), _label(name, ref.dim(), dims, labels, k), float(m.reshape(-1)[k]) / floor * rho)
    return best


def check(name: str, got, ref, tol: float, slicings: Iterable[Slicing] = (), rho: Optional[float] = None) -> float:
    """Assert that every slice of `got` is within `tol` of `ref` by the rule above; print and return the worst slice's
    error over tol."""
    rho = default_rho(tol, slicings) if rho is None else rho
    err, label, size = worst(got, ref, slicings, rho, name)
    ratio = err / tol
    test = os.environ.get("PYTEST_CURRENT_TEST", "").split(" ")[0]
    print(f"compare {test} {name}: worst {label} err {err:.3g} tol {tol:g} rho {rho:g} ratio {ratio:.3g} "
          f"size {size:.2g}")
    assert ratio < 1, (f"{name}: worst slice {label}: error {err:.3g} >= tol {tol:g} (slice max|ref| / tensor "
                       f"max|ref| {size:.2g}, rho {rho:g})")
    return ratio


def rel(got, ref) -> float:
    """The whole tensor as the only slice: max|got - ref| / max|ref|."""
    return worst(got, ref)[0]
