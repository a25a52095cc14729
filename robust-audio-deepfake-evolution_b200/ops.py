"""Autograd Functions and functional API of the Bi-Mamba hot path.

Public names mirror what the reference's path binds upstream:
  * ``selective_scan_fn(u, delta, A, B, C, D, z, delta_bias, delta_softplus)``  - mamba_ssm's op;
    reference math at src/models/modules/mamba_block.py:80-120 and :61
  * ``causal_conv1d_fn(x, weight, bias, activation)``                           - causal-conv1d's op;
    reference math at src/models/modules/mamba_block.py:52-55
  * ``bimamba_inner_fn(...)``  - the fused block: in_proj, conv+SiLU, x_proj, dt_proj, scan, gate,
    out_proj in BOTH time directions with shared weights
    (src/models/DualStreamSEMamba.py:473-481 around mamba_block.py:41-63)

All arithmetic runs in the CUDA library (ops on CPU tensors raise: there is no fallback).

Two arrangements of the same kernels, bit-identical in their results: outside CUDA-graph capture the block and the whole
encoder layer go through the library's one-call entry points (``BiMambaNativeFn`` / ``EncoderLayerNativeFn`` ->
bimamba_block_fwd/bwd, bimamba_layer_fwd/bwd: device-bound eager steps); under capture - and inside
``sequenced_block()`` - the Functions below enqueue the kernels one by one and overlap the weight-gradient products on a
second stream.

Layout.  The kernels are channel-last: every activation is (batch, time, channel) with unit channel
stride, the layout the projections produce and consume, so the block has no transposes.  Tensors
that exist once per direction are stored (batch, time, dir, channel) and handed to the kernels as
(batch, dir, time, channel) VIEWS (the C ABI takes element strides), which makes
``y.view(B*L, 2*D)`` the operand of ONE out_proj GEMM over both directions.  The op-level functions
keep the upstream (batch, channel, time) signature and transpose at the boundary.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import ScanDesc

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
D_STATE = 16
MAX_DT_RANK = 16
XW = 48          # row of the padded x_proj output: [B(16) | C(16) | dt_r (<= 16, zero padded)]


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("Bi-Mamba ops run on CUDA tensors only (no CPU fallback)")


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {t.dtype}; use float32, bfloat16 or float16") from None


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _s3(t: torch.Tensor) -> Tuple[int, int, int]:
    """(batch, dir, time) element strides of a (batch, ndir, L, C) tensor with unit channel stride."""
    assert t.dim() == 4
    if t.numel() and t.size(3) > 1 and t.stride(3) != 1:
        raise ValueError("channels must be the contiguous (innermost) axis")
    return t.stride(0), (t.stride(1) if t.size(1) > 1 else 0), t.stride(2)


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


_NULL = _NullCtx()


def _timed(name: str):
    t = _lib.kernel_timer
    return _NULL if t is None else t(name)


# ----------------------------------------------------------------------------------------
# fork / join on a side stream: the weight-gradient GEMMs and bias column sums of a backward are independent of
# the data-gradient chain, and at the Phase-6 sizes every kernel is too small to fill 148 SMs, so they run
# concurrently (under CUDA-graph capture the fork/join becomes parallel graph branches).
# ----------------------------------------------------------------------------------------
_SIDE = {}
SIDE_STREAM = os.environ.get("BIMAMBA_SIDE_STREAM", "1") != "0"


class _Fork:
    """with _Fork() as f: ... work enqueued on the side stream ...;  f.join() makes the current stream wait for it.
    Tensors touched on the side stream must stay referenced until join() (callers join before returning)."""

    def __enter__(self):
        self.cur = torch.cuda.current_stream()
        if not SIDE_STREAM:
            self.side = None
            return self
        dev = self.cur.device_index
        if dev not in _SIDE:
            _SIDE[dev] = torch.cuda.Stream(device=dev)
        self.side = _SIDE[dev]
        self.side.wait_stream(self.cur)
        self.ctx = torch.cuda.stream(self.side)
        self.ctx.__enter__()
        return self

    def __exit__(self, *a):
        if self.side is not None:
            self.ctx.__exit__(*a)
        return False

    def join(self):
        if self.side is not None:
            self.cur.wait_stream(self.side)


def _wants_grad(*ts) -> bool:
    """True when autograd will call backward for these inputs.  Decided in the Python wrappers, not inside
    Function.forward: grad mode is always off there and ctx.needs_input_grad ignores torch.no_grad()."""
    return torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in ts)


def seqlens_tensor(lengths, Bsz: int, T: int, device) -> Optional[torch.Tensor]:
    """Per-utterance frame counts of a right-padded (B, T, ...) batch -> the (B,) int32 vector the kernels read on
    `device` (None stays None: fixed length).  `lengths` may be a list, a CPU tensor or a CUDA tensor.  Host-side lengths
    are checked here without a device sync: shape (B,), integers, 1 <= len <= T, else ValueError.  A CUDA tensor is
    trusted (only its shape is checked): the kernels clamp its values to [0, T], and a zero-length utterance scores as
    zero features."""
    if lengths is None:
        return None
    if isinstance(lengths, torch.Tensor) and lengths.is_cuda:
        if tuple(lengths.shape) != (Bsz,):
            raise ValueError(f"lengths must have shape ({Bsz},), got {tuple(lengths.shape)}")
        return lengths if lengths.dtype == torch.int32 and lengths.is_contiguous() else lengths.to(torch.int32).contiguous()
    t = torch.as_tensor(lengths)
    if tuple(t.shape) != (Bsz,) or t.is_floating_point() or t.is_complex() or t.dtype == torch.bool:
        raise ValueError(f"lengths must be {Bsz} integer frame counts, got {tuple(t.shape)} {t.dtype}")
    if Bsz and (int(t.min()) < 1 or int(t.max()) > T):
        raise ValueError(f"lengths must lie in 1..{T} (the padded frame count), got {int(t.min())}..{int(t.max())}")
    return t.to(torch.int32).to(device)


def _forward_only(seqlens, *ts) -> None:
    if seqlens is not None and _wants_grad(*ts):
        raise NotImplementedError("lengths without mask_padding=True are supported for scoring only: pass "
                                  "mask_padding=True to train on a right-padded batch, or run under torch.no_grad()")


def _check_mask_padding(lengths, mask_padding: bool) -> None:
    if mask_padding and lengths is None:
        raise ValueError("mask_padding=True needs lengths (the per-utterance frame counts of the padded batch)")


def mask_frames_raw(x: torch.Tensor, seqlens: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, T, C) -> a copy (or `out`, which may be x) with the frames t >= seqlens[b] set to zero by selection (padded
    frames are never read: NaN padding cannot pass).  One launch."""
    lib = _lib.load()
    x = x if x.is_contiguous() else x.contiguous()
    out = torch.empty_like(x) if out is None else out
    Bsz, T, C_ = x.shape
    with _timed("mask"):
        _lib.check(lib.bimamba_mask_frames(_ptr(x), _ptr(out), _ptr(seqlens), Bsz, T, C_, _dt(x), _stream()),
                   "bimamba_mask_frames")
    return out


class MaskFramesFn(torch.autograd.Function):
    """The frame mask of variable-length training, forward and backward: padded frames of the value and of its
    gradient are zero."""

    @staticmethod
    def forward(ctx, x, seqlens):
        _require_cuda(x)
        ctx.seqlens = seqlens
        return mask_frames_raw(x.detach(), seqlens)

    @staticmethod
    def backward(ctx, g):
        return mask_frames_raw(g, ctx.seqlens), None


def mask_frames(x: torch.Tensor, seqlens: torch.Tensor) -> torch.Tensor:
    """x (B, T, C) with the frames at or past each utterance's length zeroed, as an autograd op (seqlens_tensor)."""
    return MaskFramesFn.apply(x, seqlens)


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.detach().to(torch.float32).contiguous()


def per_dir(Bsz: int, L: int, ndir: int, C_: int, device, dtype, zero: bool = False) -> torch.Tensor:
    """Allocates (B, L, ndir, C) storage and returns the (B, ndir, L, C) view the kernels take."""
    mk = torch.zeros if zero else torch.empty
    return mk((Bsz, L, ndir, C_), device=device, dtype=dtype).permute(0, 2, 1, 3)


def rows2d(t: torch.Tensor) -> torch.Tensor:
    """(B, ndir, L, C) view of (B, L, ndir, C) storage -> the (B*L*ndir, C) row matrix (no copy)."""
    Bsz, ndir, L, C_ = t.shape
    return t.permute(0, 2, 1, 3).reshape(Bsz * L * ndir, C_)


# ----------------------------------------------------------------------------------------
# raw kernels (no autograd)
# ----------------------------------------------------------------------------------------
def conv_fwd_raw(x, weight, bias, out, silu: bool, seqlens: Optional[torch.Tensor] = None):
    """x (B, L, D) with unit channel stride; weight (D, K) fp32; out (B, ndir, L, D) view.  seqlens: (B,) int32 device
    frame counts (seqlens_tensor) or None; with them the padded frames of out are written as zeros."""
    lib = _lib.load()
    Bsz, L, D = x.shape
    ndir = out.shape[1]
    obs, ods, ots = _s3(out)
    if x.stride(2) != 1 and D > 1:
        raise ValueError("x must have unit channel stride")
    with _timed("conv_fwd"):
        rc = lib.bimamba_causal_conv1d_fwd_varlen(
            _ptr(x), _ptr(weight), _ptr(bias), _ptr(out), _ptr(seqlens), Bsz, ndir, D, L, weight.shape[1],
            x.stride(0), x.stride(1), obs, ods, ots, _dt(x), _lib.FLAG_SILU if silu else 0, _stream())
        _lib.check(rc, "bimamba_causal_conv1d_fwd_varlen")


def conv_bwd_raw(x, weight, bias, dout, dx, silu: bool, dz_in=None, dz_out=None, defer: Optional[list] = None,
                 seqlens: Optional[torch.Tensor] = None):
    """dout (B, ndir, L, D) view; dx (B, L, D) (may be a strided view).  Optionally folds the sum of the
    per-direction gate gradients dz_in (same strides as dout) into dz_out (same strides as dx).
    Returns dwb (D, K+1) fp32 [dw | dbias]; with `defer` (a list) its fixed-order sum over the CTAs' partials runs on
    the side stream and the fork is appended to the list (join() before using dwb).
    seqlens: the backward of conv_fwd_raw with the same frame counts; dx and dz_out are zero at padded frames."""
    lib = _lib.load()
    Bsz, L, D = x.shape
    ndir = dout.shape[1]
    K = weight.shape[1]
    gbs, gds, gts = _s3(dout)
    if dz_in is not None:
        if _s3(dz_in) != (gbs, gds, gts):
            raise ValueError("dz_in must share dout's strides")
        if (dz_out.stride(0), dz_out.stride(1)) != (dx.stride(0), dx.stride(1)):
            raise ValueError("dz_out must share dx's strides")
    nsl = lib.bimamba_conv_bwd_slices(Bsz, L, D)
    part = torch.empty((max(nsl, 1), D, K + 1), device=x.device, dtype=torch.float32)
    with _timed("conv_bwd"):
        rc = lib.bimamba_causal_conv1d_bwd_varlen(
            _ptr(x), _ptr(weight), _ptr(bias), _ptr(dout), _ptr(dx), _ptr(dz_in), _ptr(dz_out), _ptr(part), _ptr(seqlens),
            Bsz, ndir, D, L, K, x.stride(0), x.stride(1), gbs, gds, gts, dx.stride(0), dx.stride(1), _dt(x),
            _lib.FLAG_SILU if silu else 0, _stream())
        _lib.check(rc, "bimamba_causal_conv1d_bwd_varlen")
    dwb = torch.empty((D, K + 1), device=x.device, dtype=torch.float32)
    if Bsz * L == 0:
        return dwb.zero_()
    if defer is None:
        reduce_raw(part, dwb, groups=1, rows=nsl, cols=D * (K + 1), part_gs=0, row_stride=D * (K + 1), out_gs=0)
    else:
        with _Fork() as f:
            reduce_raw(part, dwb, groups=1, rows=nsl, cols=D * (K + 1), part_gs=0, row_stride=D * (K + 1), out_gs=0)
        f.keep = (part,)
        defer.append(f)
    return dwb


def reduce_raw(part, out, groups, rows, cols, part_gs, row_stride, out_gs, accumulate=False):
    lib = _lib.load()
    with _timed("reduce"):
        rc = lib.bimamba_reduce_partials(_ptr(part), _ptr(out), groups, rows, cols, part_gs, row_stride, out_gs,
                                         _dt(out), int(accumulate), _stream())
        _lib.check(rc, "bimamba_reduce_partials")


def _fill_desc(u, z, delta, bc, dtr, Wdt, A, D, delta_bias, softplus, dtr_padded, G) -> ScanDesc:
    d = ScanDesc()
    Bsz, ndir, L, dim = u.shape
    d.u, d.z, d.delta, d.bc, d.dtr = _ptr(u), _ptr(z), _ptr(delta), _ptr(bc), _ptr(dtr)
    d.Wdt, d.A, d.D, d.delta_bias = _ptr(Wdt), _ptr(A), _ptr(D), _ptr(delta_bias)
    d.batch, d.ndir, d.dim, d.seqlen, d.dstate = Bsz, ndir, dim, L, A.shape[1]
    d.dt_rank = 0 if Wdt is None else Wdt.shape[1]
    d.io_dtype = _dt(u)
    d.flags = (_lib.FLAG_SOFTPLUS if softplus else 0) | (_lib.FLAG_DTR_PADDED if dtr_padded else 0)
    d.group_channels = G
    d.u_bs, d.u_ds, d.u_ts = _s3(u)
    for name, t in (("z", z), ("delta", delta), ("bc", bc), ("dtr", dtr)):
        if t is not None:
            if t.dtype != u.dtype:
                raise TypeError(f"{name} must have u's dtype")
            bs, ds, ts = _s3(t)
            setattr(d, name + "_bs", bs), setattr(d, name + "_ds", ds), setattr(d, name + "_ts", ts)
    return d


def scan_fwd_raw(u, z, delta, bc, dtr, Wdt, A, D, delta_bias, softplus: bool, want_ckpt: bool,
                 dtr_padded: bool = False, seqlens: Optional[torch.Tensor] = None):
    """All activations are (B, ndir, L, C) views with unit channel stride (z may be expanded over
    dir).  Returns (out, ckpt, ypre): out / ypre are (B, ndir, L, dim) views of (B, L, ndir, dim).
    seqlens: (B,) int32 device frame counts (seqlens_tensor) or None.  With them each utterance walks its own frames
    (direction 1 from its last valid one), padded frames of out (and ypre) are zeros, and the serial walk is used: the
    time-split forward has no variable-length form.  With want_ckpt the checkpoints keep the padded layout
    (ceil(L / 8) per channel) for scan_bwd_raw with the same seqlens."""
    lib = _lib.load()
    Bsz, ndir, L, dim = u.shape
    G, ngroups, nchunks = _lib.scan_plan(L, dim, Bsz * ndir, False)
    out = per_dir(Bsz, L, ndir, dim, u.device, u.dtype)
    ckpt = ypre = None
    if want_ckpt and nchunks > 1:
        ckpt = torch.empty((Bsz, ndir, nchunks, dim, A.shape[1]), device=u.device, dtype=torch.float32)
    if want_ckpt and z is not None:
        ypre = per_dir(Bsz, L, ndir, dim, u.device, u.dtype)
    d = _fill_desc(u, z, delta, bc, dtr, Wdt, A, D, delta_bias, softplus, dtr_padded, G)
    d.out, d.ypre, d.ckpt = _ptr(out), _ptr(ypre), _ptr(ckpt)
    d.out_bs, d.out_ds, d.out_ts = _s3(out)
    nseg, seg_len = _lib.scan_split_plan(Bsz, ndir, L, dim, _dt(u)) if seqlens is None else (1, L)
    if nseg > 1:
        # long sequence, few channel lanes: time-parallel scan (carry pass + output pass, two launches)
        nbytes = lib.bimamba_scan_fwd_split_workspace_bytes(Bsz, ndir, dim, nseg)
        carry = torch.empty((nbytes // 4,), device=u.device, dtype=torch.float32)
        with _timed("scan_fwd"):
            _lib.check(lib.bimamba_selective_scan_fwd_split(C.byref(d), nseg, seg_len, _ptr(carry), nbytes, _stream()),
                       "bimamba_selective_scan_fwd_split")
        _lib.launch_count += 1   # two kernels per call
        return out, ckpt, ypre
    fwd = lib.bimamba_selective_scan_fwd_varlen_train if want_ckpt else lib.bimamba_selective_scan_fwd_varlen
    with _timed("scan_fwd"):
        _lib.check(fwd(C.byref(d), _ptr(seqlens), _stream()), "bimamba_selective_scan_fwd_varlen")
    return out, ckpt, ypre


def scan_bwd_raw(u, z, delta, bc, dtr, Wdt, A, D, delta_bias, softplus: bool, dout, ckpt, ypre,
                 dtr_padded: bool = False, bc_out_dtype=None, defer: Optional[list] = None,
                 dbc_rows: Optional[torch.Tensor] = None, seqlens: Optional[torch.Tensor] = None):
    """Returns (du, ddelta, dz, dbc, dA, dD, dbias): du / ddelta / dz are (B, ndir, L, dim) views of
    (B, L, ndir, dim) storage; dbc is (B, ndir, L, 32) = [dB | dC] likewise; dA (dim, N), dD, dbias (dim).
    With `defer` (a list) the parameter-gradient sums dA / dD / dbias are enqueued on the side stream and the fork is
    appended to the list: the caller must join() it before using them.
    With `dbc_rows` (a (B*L*ndir, >= 32) row matrix, rows ordered (b, t, dir)) the group sum of [dB | dC] is written
    into its first 32 columns and the returned dbc is None.
    seqlens: the backward of scan_fwd_raw with the same frame counts: du, ddelta, dz and [dB | dC] are zero at padded
    frames, dout there is never read, and dA / dD / dbias sum over valid steps only."""
    lib = _lib.load()
    Bsz, ndir, L, dim = u.shape
    N = A.shape[1]
    dev = u.device
    G, ngroups, _ = _lib.scan_plan(L, dim, Bsz * ndir, True)
    du = per_dir(Bsz, L, ndir, dim, dev, u.dtype)
    ddelta = per_dir(Bsz, L, ndir, dim, dev, u.dtype)
    dz = per_dir(Bsz, L, ndir, dim, dev, u.dtype) if z is not None else None
    dbc_part = torch.empty((Bsz, ngroups, L, ndir, 2 * N), device=dev, dtype=torch.float32)
    dA_part = torch.empty((Bsz * ndir, dim, N), device=dev, dtype=torch.float32)
    dD_part = torch.empty((Bsz * ndir, dim), device=dev, dtype=torch.float32) if D is not None else None
    db_part = torch.empty((Bsz * ndir, dim), device=dev, dtype=torch.float32) if delta_bias is not None else None

    d = _fill_desc(u, z, delta, bc, dtr, Wdt, A, D, delta_bias, softplus, dtr_padded, G)
    if dout.dtype != u.dtype:
        raise TypeError("dout must have u's dtype")
    d.dout = _ptr(dout)
    d.dout_bs, d.dout_ds, d.dout_ts = _s3(dout)
    d.ckpt, d.ypre = _ptr(ckpt), _ptr(ypre)
    d.out_bs, d.out_ds, d.out_ts = _s3(du)
    if ypre is not None and _s3(ypre) != _s3(du):
        raise ValueError("ypre must have the (B, L, ndir, dim) storage the forward wrote")
    d.du, d.ddelta, d.dz = _ptr(du), _ptr(ddelta), _ptr(dz)
    d.dbc_part, d.dA_part, d.dD_part, d.dbias_part = _ptr(dbc_part), _ptr(dA_part), _ptr(dD_part), _ptr(db_part)
    with _timed("scan_bwd"):
        _lib.check(lib.bimamba_selective_scan_bwd_varlen(C.byref(d), _ptr(seqlens), _stream()),
                   "bimamba_selective_scan_bwd_varlen")

    if dbc_rows is not None:
        dbc = None
        if dbc_rows.shape[0] != Bsz * L * ndir or dbc_rows.stride(1) != 1:
            raise ValueError("dbc_rows must be a (B*L*ndir, >= 32) row matrix")
        with _timed("reduce"):
            _lib.check(lib.bimamba_reduce_rows32(_ptr(dbc_part), _ptr(dbc_rows), Bsz, ngroups, L * ndir, dbc_rows.stride(0),
                                                 _dt(dbc_rows), _stream()), "bimamba_reduce_rows32")
    else:
        dbc = per_dir(Bsz, L, ndir, 2 * N, dev, bc_out_dtype or u.dtype)
        cols = L * ndir * 2 * N
        reduce_raw(dbc_part, dbc, groups=Bsz, rows=ngroups, cols=cols, part_gs=ngroups * cols, row_stride=cols,
                   out_gs=cols)
    dA = torch.empty((dim, N), device=dev, dtype=torch.float32)
    dD = torch.empty((dim,), device=dev, dtype=torch.float32) if D is not None else None
    dbias = torch.empty((dim,), device=dev, dtype=torch.float32) if delta_bias is not None else None

    def param_sums():
        reduce_raw(dA_part, dA, 1, Bsz * ndir, dim * N, 0, dim * N, 0)
        if D is not None:
            reduce_raw(dD_part, dD, 1, Bsz * ndir, dim, 0, dim, 0)
        if delta_bias is not None:
            reduce_raw(db_part, dbias, 1, Bsz * ndir, dim, 0, dim, 0)

    if defer is None:
        param_sums()
    else:                                  # off the data-gradient chain
        with _Fork() as f:
            param_sums()
        f.keep = (dA_part, dD_part, db_part)
        defer.append(f)
    return du, ddelta, dz, dbc, dA, dD, dbias


# ----------------------------------------------------------------------------------------
# op-level autograd Functions (single direction, upstream signatures, (B, D, L) operands)
# ----------------------------------------------------------------------------------------
def _cl(t: torch.Tensor) -> torch.Tensor:
    """(B, C, L) -> contiguous channel-last (B, L, C)."""
    return t.transpose(1, 2).contiguous()


class CausalConv1dFn(torch.autograd.Function):
    """causal_conv1d_fn: x (B, D, L), weight (D, K), bias (D) -> (B, D, L).  mamba_block.py:52-55."""

    @staticmethod
    def forward(ctx, x, weight, bias, activation):
        if activation not in (None, "silu", "swish"):
            raise NotImplementedError("activation must be None, silu, or swish")
        _require_cuda(x, weight, bias)
        silu = activation is not None
        xl = _cl(x)
        w32, b32 = _f32c(weight), _f32c(bias)
        Bsz, L, D = xl.shape
        out = torch.empty((Bsz, L, D), device=x.device, dtype=x.dtype)
        conv_fwd_raw(xl, w32, b32, out.unsqueeze(1), silu)
        ctx.save_for_backward(xl, w32, b32 if b32 is not None else torch.empty(0))
        ctx.silu, ctx.has_bias = silu, bias is not None
        ctx.wdtype = weight.dtype
        ctx.bdtype = bias.dtype if bias is not None else None
        return out.transpose(1, 2)

    @staticmethod
    def backward(ctx, dout):
        xl, w32, b32 = ctx.saved_tensors
        b32 = b32 if ctx.has_bias else None
        gl = _cl(dout.to(xl.dtype))
        dx = torch.empty_like(xl)
        dwb = conv_bwd_raw(xl, w32, b32, gl.unsqueeze(1), dx, ctx.silu)
        K = w32.shape[1]
        dw = dwb[:, :K].to(ctx.wdtype)
        db = dwb[:, K].to(ctx.bdtype) if ctx.has_bias else None
        return dx.transpose(1, 2), dw, db, None


def causal_conv1d_fn(x, weight, bias=None, seq_idx=None, initial_states=None, return_final_states=False,
                     final_states_out=None, activation=None):
    if seq_idx is not None or initial_states is not None or return_final_states or final_states_out is not None:
        raise NotImplementedError("seq_idx / initial_states / final_states are not used by the reference path")
    return CausalConv1dFn.apply(x, weight, bias, activation)


def _as_bnl(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.dim() == 4:
        if t.shape[1] != 1:
            raise NotImplementedError(f"{name}: grouped B/C (G > 1) is not used by the reference path")
        t = t[:, 0]
    if t.dim() != 3:
        raise NotImplementedError(f"{name} must be input-dependent: (batch, dstate, L)")
    return t


class SelectiveScanFn(torch.autograd.Function):
    """selective_scan_fn(u, delta, A, B, C, D, z, delta_bias, delta_softplus).
    u, delta, z (B, D, L); A (D, N); B, C (B, N, L).  mamba_block.py:80-120, :61."""

    @staticmethod
    def forward(ctx, u, delta, A, B, C, D, z, delta_bias, delta_softplus, needs_bwd=True):
        _require_cuda(u, delta, A, B, C, D, z, delta_bias)
        Bshape, Cshape = B.shape, C.shape
        Bm, Cm = _as_bnl(B, "B"), _as_bnl(C, "C")
        if A.shape[1] != D_STATE:
            raise NotImplementedError("d_state must be 16 (the Phase-6 configuration)")
        io = u.dtype
        ul = _cl(u).unsqueeze(1)
        dl = _cl(delta.to(io)).unsqueeze(1)
        zl = _cl(z.to(io)).unsqueeze(1) if z is not None else None
        bc = torch.cat([Bm.to(io).transpose(1, 2), Cm.to(io).transpose(1, 2)], dim=2).unsqueeze(1)   # (B, 1, L, 32)
        A32, D32, b32 = _f32c(A), _f32c(D), _f32c(delta_bias)
        out, ckpt, ypre = scan_fwd_raw(ul, zl, dl, bc, None, None, A32, D32, b32, bool(delta_softplus), needs_bwd)
        ctx.save_for_backward(ul, dl, A32, bc, D32 if D32 is not None else torch.empty(0),
                              zl if zl is not None else torch.empty(0), b32 if b32 is not None else torch.empty(0),
                              ckpt if ckpt is not None else torch.empty(0),
                              ypre if ypre is not None else torch.empty(0))
        ctx.meta = (D is not None, z is not None, delta_bias is not None, bool(delta_softplus),
                    A.dtype, None if D is None else D.dtype, None if delta_bias is None else delta_bias.dtype,
                    B.dtype, C.dtype, Bshape, Cshape, None if z is None else z.dtype, delta.dtype)
        return out[:, 0].transpose(1, 2)

    @staticmethod
    def backward(ctx, dout):
        ul, dl, A32, bc, D32, zl, b32, ckpt, ypre = ctx.saved_tensors
        (hasD, hasz, hasb, softplus, Adt, Ddt, bdt, Bdt, Cdt, Bshape, Cshape, zdt, deltadt) = ctx.meta
        D32 = D32 if hasD else None
        zl = zl if hasz else None
        b32 = b32 if hasb else None
        ckpt = ckpt if ckpt.numel() else None
        ypre = ypre if ypre.numel() else None
        gl = _cl(dout.to(ul.dtype)).unsqueeze(1)
        du, ddelta, dz, dbc, dA, dD, dbias = scan_bwd_raw(
            ul, zl, dl, bc, None, None, A32, D32, b32, softplus, gl, ckpt, ypre, bc_out_dtype=torch.float32)
        N = A32.shape[1]
        dB = dbc[:, 0, :, :N].transpose(1, 2).to(Bdt).reshape(Bshape)
        dC = dbc[:, 0, :, N:].transpose(1, 2).to(Cdt).reshape(Cshape)
        return (du[:, 0].transpose(1, 2), ddelta[:, 0].transpose(1, 2).to(deltadt), dA.to(Adt), dB, dC,
                dD.to(Ddt) if hasD else None, dz[:, 0].transpose(1, 2).to(zdt) if hasz else None,
                dbias.to(bdt) if hasb else None, None, None)


def selective_scan_fn(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False,
                      return_last_state=False):
    if return_last_state:
        raise NotImplementedError("return_last_state is not used by the reference path")
    return SelectiveScanFn.apply(u, delta, A, B, C, D, z, delta_bias, delta_softplus,
                                 _wants_grad(u, delta, A, B, C, D, z, delta_bias))


# ----------------------------------------------------------------------------------------
# projections: C = A . B^T on the tcgen05 tensor cores (mamba_block.py:48, :73, :62)
# ----------------------------------------------------------------------------------------
def _tc_ok(A: torch.Tensor, B: torch.Tensor) -> bool:
    return (A.dtype in (torch.bfloat16, torch.float16) and B.dtype == A.dtype and A.dim() == 2
            and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1 and A.stride(0) % 8 == 0
            and B.stride(0) % 8 == 0 and A.data_ptr() % 16 == 0 and B.data_ptr() % 16 == 0 and A.shape[0] > 0)


def _split3(t: torch.Tensor, side: int, stack_rows: bool) -> torch.Tensor:
    """fp32 (rows, cols) -> bf16 six-block split (bimamba_split3_bf16): (rows, 6*cols) for the K-major operands of
    gemm_nt, (6*rows, cols) for the row-contracted operands of gemm_tn."""
    lib = _lib.load()
    rows, cols = t.shape
    if t.stride(1) != 1:
        t = t.contiguous()
    if stack_rows:
        dst = torch.empty((6 * rows, cols), device=t.device, dtype=torch.bfloat16)
        ld_dst, block = cols, rows * cols
    else:
        dst = torch.empty((rows, 6 * cols), device=t.device, dtype=torch.bfloat16)
        ld_dst, block = 6 * cols, cols
    with _timed("split3"):
        _lib.check(lib.bimamba_split3_bf16(_ptr(t), _ptr(dst), rows, cols, t.stride(0), ld_dst, block, side, _stream()),
                   "bimamba_split3_bf16")
    return dst


def _f32_tc_ok(A: torch.Tensor, B: torch.Tensor, k_mult: int) -> bool:
    """fp32 operands that the split path can take: contiguous rows, contraction / row widths that keep the bf16
    blocks 16-byte aligned."""
    return (A.dtype == torch.float32 and B.dtype == torch.float32 and A.dim() == 2 and B.dim() == 2 and A.is_cuda
            and A.shape[0] > 0 and A.shape[1] % k_mult == 0 and B.shape[1] % k_mult == 0 and A.shape[1] > 0)


def gemm_nt(A, B, bias=None, addend=None, out_dtype=None, out=None):
    """A (M, K) . B (N, K)^T (+ bias (N) fp32) (+ addend (M, N)) -> (M, N).  bf16 / fp16 operands run on this
    repository's tcgen05 kernel; fp32 operands (the 1e-4 parity mode, fp32 scoring) are split into three bf16 terms each and
    run on the same kernel with six K blocks (fp32-accurate, bimamba_split3_bf16).  Only shapes whose contraction width is
    not a multiple of 4 fall back to the framework product."""
    out_dtype = out_dtype or (out.dtype if out is not None else A.dtype)
    if _f32_tc_ok(A, B, 4) and A.shape[1] == B.shape[1] and out_dtype == torch.float32:
        # fp32 operands: three-term bf16 split of both, six K blocks, one tcgen05 GEMM with fp32 accumulation
        return gemm_nt(_split3(A, 0, False), _split3(B, 1, False), bias, addend, torch.float32, out)
    if not _tc_ok(A, B):
        C_ = torch.mm(A, B.t()).to(out_dtype)
        if bias is not None:
            C_ = C_ + bias.to(out_dtype)
        if addend is not None:
            C_ = C_ + addend
        if out is not None:
            out.copy_(C_)
            return out
        return C_
    lib = _lib.load()
    M, K = A.shape
    N = B.shape[0]
    if out is None:
        out = torch.empty((M, N), device=A.device, dtype=out_dtype)
    elif out.shape != (M, N) or out.dtype != out_dtype or out.stride(1) != 1:
        raise ValueError("gemm_nt: out must be an (M, N) row matrix of the output dtype with unit column stride")
    if addend is not None:
        if addend.dtype != out_dtype or addend.shape != out.shape or addend.stride() != out.stride():
            addend = addend.to(out_dtype).contiguous()
            if out.stride(0) != N:
                raise ValueError("gemm_nt: addend must share a strided out's layout")
    with _timed("gemm_nt"):
        _lib.check(lib.bimamba_gemm_nt(_ptr(A), A.stride(0), _ptr(B), B.stride(0), _ptr(out), out.stride(0), _ptr(bias),
                                       _ptr(addend), M, N, K, _dt(A), _dt(out), _stream()), "bimamba_gemm_nt")
    return out


def gemm_tn(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """A (M, N1)^T . B (M, N2) -> (N1, N2) fp32: the weight gradient dY^T X on the tcgen05 kernel (MN-major operands,
    deterministic split over the M rows).  fp32 operands are split into three bf16 terms stacked along the contracted rows;
    only misaligned operands use the framework product."""
    if _f32_tc_ok(A, B, 8) and A.shape[0] == B.shape[0]:
        # fp32 operands: the six split blocks are stacked along the contracted rows
        return gemm_tn(_split3(A, 0, True), _split3(B, 1, True))
    if not _tc_ok(A, B):
        return mm_f32(A.t(), B)
    lib = _lib.load()
    M, N1 = A.shape
    N2 = B.shape[1]
    ns = lib.bimamba_gemm_tn_splits(M, N1, N2)
    part = torch.empty((ns, N1 * N2), device=A.device, dtype=torch.float32)
    out = torch.empty((N1, N2), device=A.device, dtype=torch.float32)
    with _timed("gemm_tn"):
        _lib.check(lib.bimamba_gemm_tn(_ptr(A), A.stride(0), _ptr(B), B.stride(0), _ptr(out), _ptr(part), M, N1, N2,
                                       _dt(A), _stream()), "bimamba_gemm_tn")
    _lib.launch_count += 1   # two kernels per call
    return out


def wgrad(dY: torch.Tensor, X: torch.Tensor) -> torch.Tensor:
    """dY (M, N_out)^T . X (M, N_in) -> (N_out, N_in) fp32: the weight gradient of y = x W^T."""
    return gemm_tn(dY, X)


def mm_f32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a @ b with an fp32 result: the weight-gradient products (contraction over B*L) accumulate and leave in fp32
    (library GEMM; 16-bit operands, no separate cast of the result)."""
    if a.dtype in (torch.bfloat16, torch.float16):
        return torch.mm(a, b, out_dtype=torch.float32)
    return torch.mm(a, b)


def colsum(x2: torch.Tensor) -> torch.Tensor:
    """Sum over the rows of a (rows, cols) matrix -> fp32 (cols): bias gradient of a Linear layer."""
    lib = _lib.load()
    rows, cols = x2.shape
    out = torch.empty((cols,), device=x2.device, dtype=torch.float32)
    if rows == 0:
        return out.zero_()
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    nsl = lib.bimamba_colsum_slices(rows)
    part = torch.empty((nsl, cols), device=x2.device, dtype=torch.float32)
    with _timed("colsum"):
        _lib.check(lib.bimamba_colsum(_ptr(x2), _ptr(part), rows, cols, x2.stride(0), _dt(x2), _stream()), "bimamba_colsum")
    reduce_raw(part, out, groups=1, rows=nsl, cols=cols, part_gs=0, row_stride=cols, out_gs=0)
    return out


def cast(t: torch.Tensor, dtype) -> torch.Tensor:
    """t.to(dtype) on this repository's kernel (contiguous result); a no-op when the dtype already matches."""
    if t.dtype == dtype:
        return t
    if t.dtype not in _DT or dtype not in _DT or not t.is_cuda or not t.is_contiguous() or t.data_ptr() % 16:
        return t.to(dtype)
    lib = _lib.load()
    out = torch.empty(t.shape, device=t.device, dtype=dtype)
    with _timed("cast"):
        _lib.check(lib.bimamba_cast(_ptr(t), _ptr(out), t.numel(), _dt(t), _DT[dtype], _stream()), "bimamba_cast")
    return out


class MeanSquareFn(torch.autograd.Function):
    """loss = mean(x^2) in fp32 (the benchmark's synthetic loss on the backend output): one partial-sum launch + the
    fixed-order reduction forward, one launch backward; no host synchronisation."""

    @staticmethod
    def forward(ctx, x):
        _require_cuda(x)
        lib = _lib.load()
        xc = x.detach().contiguous()
        n = xc.numel()
        nsl = lib.bimamba_sumsq_slices(n)
        part = torch.empty((nsl,), device=x.device, dtype=torch.float32)
        with _timed("loss"):
            _lib.check(lib.bimamba_sumsq(_ptr(xc), _ptr(part), n, 1.0 / n, _dt(xc), _stream()), "bimamba_sumsq")
        out = torch.empty((1,), device=x.device, dtype=torch.float32)
        reduce_raw(part, out, groups=1, rows=nsl, cols=1, part_gs=0, row_stride=1, out_gs=0)
        ctx.save_for_backward(xc)
        ctx.xshape = x.shape
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        (xc,) = ctx.saved_tensors
        lib = _lib.load()
        n = xc.numel()
        dx = torch.empty_like(xc)
        g32 = g.detach().to(torch.float32).reshape(1).contiguous()
        with _timed("loss"):
            _lib.check(lib.bimamba_scale_by(_ptr(xc), _ptr(g32), _ptr(dx), n, 2.0 / n, _dt(xc), _stream()), "bimamba_scale_by")
        return dx.view(ctx.xshape)


def mean_square_loss(x: torch.Tensor) -> torch.Tensor:
    return MeanSquareFn.apply(x)


def gelu_fwd(x: torch.Tensor) -> torch.Tensor:
    """Exact (erf) GELU of a contiguous tensor, this repository's kernel (DualStreamSEMamba.py:462)."""
    lib = _lib.load()
    x = x.contiguous()
    y = torch.empty_like(x)
    with _timed("gelu"):
        _lib.check(lib.bimamba_gelu_fwd(_ptr(x), _ptr(y), x.numel(), _dt(x), _stream()), "bimamba_gelu_fwd")
    return y


def gelu_bwd(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """dy * gelu'(x)."""
    lib = _lib.load()
    x, dy = x.contiguous(), dy.contiguous()
    dx = torch.empty_like(x)
    with _timed("gelu"):
        _lib.check(lib.bimamba_gelu_bwd(_ptr(x), _ptr(dy), _ptr(dx), x.numel(), _dt(x), _stream()), "bimamba_gelu_bwd")
    return dx


# ----------------------------------------------------------------------------------------
# feed-forward of the encoder layer: Linear(144, 576) -> GELU -> Linear(576, 144) (+ residual)
# (DualStreamSEMamba.py:460-464, :483-485)
# ----------------------------------------------------------------------------------------
class FeedForwardFn(torch.autograd.Function):
    """y = W2 gelu(W1 x + b1) + b2 (+ residual).  bf16 / fp16: both products and both data gradients run on the
    tcgen05 GEMM with bias / residual in its epilogue; bias gradients are this repository's column-sum kernel."""

    @staticmethod
    def forward(ctx, x, W1, b1, W2, b2, residual, cdtype, needs_bwd=True):
        _require_cuda(x, W1, b1, W2, b2, residual)
        with torch.autocast("cuda", enabled=False):
            shape = x.shape
            x2 = x.detach().to(cdtype).reshape(-1, shape[-1])
            if x2.stride(-1) != 1:
                x2 = x2.contiguous()
            W1c, W1T = cast_transpose(W1.detach(), cdtype)
            W2c, W2T = cast_transpose(W2.detach(), cdtype)
            h = gemm_nt(x2, W1c, bias=_f32c(b1))                               # :461
            a = gelu_fwd(h)                                                    # :462
            res2 = None if residual is None else residual.detach().reshape(-1, W2.shape[0])
            out_dtype = cdtype if residual is None else residual.dtype
            y = gemm_nt(a, W2c, bias=_f32c(b2), addend=res2, out_dtype=out_dtype)   # :463, :485
            if needs_bwd:
                ctx.save_for_backward(x2, h, a, W1T, W2T)
                ctx.meta = (shape, x.dtype, W1.dtype, b1.dtype, W2.dtype, b2.dtype, residual is not None)
            return y.view(*shape[:-1], W2.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, h, a, W1T, W2T = ctx.saved_tensors
        shape, xdt, w1dt, b1dt, w2dt, b2dt, has_res = ctx.meta
        with torch.autocast("cuda", enabled=False):
            cd = x2.dtype
            g = dy.reshape(-1, W2T.shape[1])
            if g.stride(-1) != 1 or g.stride(0) != g.shape[1]:
                g = g.contiguous()
            g = cast(g, cd)
            with _Fork() as f2:                       # second Linear's parameter gradients || its data gradient
                db2 = colsum(g)
                dW2 = wgrad(g, a)
            da = gemm_nt(g, W2T)
            dh = gelu_bwd(da, h)
            f2.join()
            with _Fork() as f1:                       # first Linear's parameter gradients || its data gradient
                db1 = colsum(dh)
                dW1 = wgrad(dh, x2)
            dx = gemm_nt(dh, W1T)
            f1.join()
        return (dx.view(shape).to(xdt), dW1.to(w1dt), db1.to(b1dt), dW2.to(w2dt), db2.to(b2dt),
                dy if has_res else None, None, None)


def feed_forward_fn(x, W1, b1, W2, b2, residual=None, compute_dtype=None):
    if compute_dtype is None:
        compute_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    return FeedForwardFn.apply(x, W1, b1, W2, b2, residual, compute_dtype, _wants_grad(x, W1, b1, W2, b2, residual))


# ----------------------------------------------------------------------------------------
# LayerNorm of the encoder layer (DualStreamSEMamba.py:472, :482, :759)
# ----------------------------------------------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    """y = LayerNorm(x) over the last axis, written directly in `out_dtype` (the dtype the next GEMM
    reads); statistics in fp32.  x (..., C) fp32 / bf16 / fp16."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_dtype, needs_bwd=True, with_residual=False):
        _require_cuda(x, weight, bias)
        lib = _lib.load()
        C_ = x.shape[-1]
        x2 = x.detach().reshape(-1, C_)
        if x2.stride(-1) != 1 or (x2.shape[0] > 1 and x2.stride(0) != C_):
            x2 = x2.contiguous()
        rows = x2.shape[0]
        w32, b32 = _f32c(weight), _f32c(bias)
        y = torch.empty((rows, C_), device=x.device, dtype=out_dtype)
        mean = torch.empty((rows,), device=x.device, dtype=torch.float32) if needs_bwd else None
        rstd = torch.empty((rows,), device=x.device, dtype=torch.float32) if needs_bwd else None
        with _timed("ln_fwd"):
            _lib.check(lib.bimamba_layernorm_fwd(_ptr(x2), _ptr(w32), _ptr(b32), _ptr(y), _ptr(mean), _ptr(rstd),
                                                 rows, C_, float(eps), _dt(x2), _dt(y), _stream()),
                       "bimamba_layernorm_fwd")
        if needs_bwd:
            ctx.save_for_backward(x2, w32, mean, rstd)
            ctx.meta = (x.shape, weight.dtype, bias.dtype)
        if with_residual:
            # second output = x itself (the residual branch): its gradient comes back into backward() and is added to dx
            # inside the LayerNorm backward kernel instead of by a separate autograd add
            return y.view(x.shape), x
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy, dres=None):
        x2, w32, mean, rstd = ctx.saved_tensors
        shape, wdt, bdt = ctx.meta
        lib = _lib.load()
        rows, C_ = x2.shape
        if dy is None:                       # only the residual branch was used
            return (dres, None, None, None, None, None, None)
        add2 = None
        if dres is not None:
            add2 = dres.reshape(rows, C_)
            if add2.dtype != x2.dtype or not add2.is_contiguous():
                add2 = add2.to(x2.dtype).contiguous()
        g2 = dy.reshape(rows, C_)
        if g2.dtype not in _DT or (g2.dtype != x2.dtype and g2.dtype != torch.float32 and x2.dtype != torch.float32):
            g2 = g2.to(x2.dtype)
        g2 = g2.contiguous()
        dx = torch.empty_like(x2)
        nb = lib.bimamba_layernorm_bwd_blocks(rows)
        part = torch.empty((nb, 2, C_), device=x2.device, dtype=torch.float32)
        with _timed("ln_bwd"):
            _lib.check(lib.bimamba_layernorm_bwd(_ptr(x2), _ptr(g2), _ptr(w32), _ptr(mean), _ptr(rstd), _ptr(add2), _ptr(dx),
                                                 _ptr(part), rows, C_, _dt(x2), _dt(g2), _stream()),
                       "bimamba_layernorm_bwd")
        dgb = torch.empty((2, C_), device=x2.device, dtype=torch.float32)
        if rows == 0:
            dgb.zero_()
        else:
            reduce_raw(part, dgb, groups=1, rows=nb, cols=2 * C_, part_gs=0, row_stride=2 * C_, out_gs=0)
        return dx.view(shape), dgb[0].to(wdt), dgb[1].to(bdt), None, None, None, None


def head_fwd(x, norm_w, norm_b, att_w, att_b, cls_w, cls_b, eps=1e-5, lengths=None):
    """Scoring head in one launch (no autograd): LayerNorm -> attention pooling over time -> classifier
    (src/models/DualStreamSEMamba.py:759-767, eval mode).  x (B, T, C) -> features (B, C) fp32, logits (B, n) fp32.
    lengths (B,) (seqlens_tensor): pool utterance b over its first lengths[b] frames only."""
    lib = _lib.load()
    seqlens = seqlens_tensor(lengths, x.shape[0], x.shape[1], x.device)
    _require_cuda(x)
    if x.dtype not in _DT:
        x = x.float()
    x = x.contiguous()
    Bsz, T, C_ = x.shape
    if T < 1:
        raise ValueError("head_fwd needs at least one frame")
    f32 = lambda t: None if t is None else t.detach().to(torch.float32).contiguous()
    gw, gb, aw, ab, cw, cb = (f32(t) for t in (norm_w, norm_b, att_w.reshape(-1), att_b, cls_w, cls_b))
    ncls = cw.shape[0]
    feats = torch.empty((Bsz, C_), device=x.device, dtype=torch.float32)
    logits = torch.empty((Bsz, ncls), device=x.device, dtype=torch.float32)
    with _timed("head_fwd"):
        _lib.check(lib.bimamba_head_fwd_varlen(_ptr(x), _ptr(gw), _ptr(gb), _ptr(aw), _ptr(ab), _ptr(cw), _ptr(cb),
                                               _ptr(feats), _ptr(logits), _ptr(seqlens), Bsz, T, C_, ncls, float(eps),
                                               _dt(x), _stream()), "bimamba_head_fwd_varlen")
    return feats, logits


class HeadPoolFn(torch.autograd.Function):
    """features = sum_t softmax_t(w_att . y_t + b_att) y_t with y = LayerNorm(x): norm_f and the attention pooling of the
    backend head under autograd (DualStreamSEMamba.py:759-763).  x (B, T, C) -> (B, C) fp32; one launch forward, one
    launch backward (+ the fixed-order sum of the per-utterance parameter-gradient rows)."""

    @staticmethod
    def forward(ctx, x, norm_w, norm_b, att_w, att_b, eps, needs_bwd=True, seqlens=None):
        _require_cuda(x, norm_w, norm_b, att_w, att_b)
        lib = _lib.load()
        xc = x.detach()
        if xc.dtype not in _DT:
            xc = xc.float()
        xc = xc.contiguous()
        Bsz, T, C_ = xc.shape
        if T < 1:
            raise ValueError("head pooling needs at least one frame")
        gw, gb, aw, ab = _f32c(norm_w), _f32c(norm_b), _f32c(att_w).reshape(-1), _f32c(att_b)
        feats = torch.empty((Bsz, C_), device=x.device, dtype=torch.float32)
        with _timed("head_fwd"):
            _lib.check(lib.bimamba_head_fwd_varlen(_ptr(xc), _ptr(gw), _ptr(gb), _ptr(aw), _ptr(ab), None, None, _ptr(feats),
                                                   None, _ptr(seqlens), Bsz, T, C_, 0, float(eps), _dt(xc), _stream()),
                       "bimamba_head_fwd_varlen")
        if needs_bwd:
            ctx.save_for_backward(xc, gw, gb, aw, ab if ab is not None else torch.empty(0))
            ctx.seqlens = seqlens
            ctx.meta = (eps, x.dtype, norm_w.dtype, norm_b.dtype, att_w.dtype, tuple(att_w.shape),
                        None if att_b is None else att_b.dtype)
        return feats

    @staticmethod
    def backward(ctx, dfeat):
        xc, gw, gb, aw, ab = ctx.saved_tensors
        eps, xdt, nwdt, nbdt, awdt, awshape, abdt = ctx.meta
        ab = ab if ab.numel() else None
        lib = _lib.load()
        Bsz, T, C_ = xc.shape
        df = dfeat.detach().to(torch.float32).contiguous()
        dx = torch.empty_like(xc)
        part = torch.empty((Bsz, 4, C_), device=xc.device, dtype=torch.float32)
        with _timed("head_bwd"):
            _lib.check(lib.bimamba_head_pool_bwd_varlen(_ptr(xc), _ptr(gw), _ptr(gb), _ptr(aw), _ptr(ab), _ptr(df), _ptr(dx),
                                                        _ptr(part), _ptr(ctx.seqlens), Bsz, T, C_, float(eps), _dt(xc),
                                                        _stream()), "bimamba_head_pool_bwd_varlen")
        sums = torch.empty((4, C_), device=xc.device, dtype=torch.float32)
        reduce_raw(part, sums, groups=1, rows=Bsz, cols=4 * C_, part_gs=0, row_stride=4 * C_, out_gs=0)
        return (dx.to(xdt), sums[0].to(nwdt), sums[1].to(nbdt), sums[2].reshape(awshape).to(awdt),
                None if abdt is None else sums[3, :1].to(abdt), None, None, None)


def head_pool_fn(x, norm_w, norm_b, att_w, att_b, eps=1e-5, seqlens=None):
    """seqlens (seqlens_tensor): pool, and take the gradient of, each utterance's first seqlens[b] frames only; dx is
    zero at padded frames and a zero-length utterance gets zero features and zero gradients."""
    return HeadPoolFn.apply(x, norm_w, norm_b, att_w, att_b, eps, _wants_grad(x, norm_w, norm_b, att_w, att_b), seqlens)


class LinearFn(torch.autograd.Function):
    """y = x W^T (+ b) (+ addend): an nn.Linear on this repository's kernels - gemm_nt forward and data gradient, the
    MN-major weight-gradient GEMM and the column-sum kernel for the bias (DualStreamFusion's projections,
    DualStreamSEMamba.py:565-570).  x (..., K); W (N, K); addend (..., N) in the output's layout."""

    @staticmethod
    def forward(ctx, x, W, b, addend, cdtype, out_dtype, needs_bwd=True):
        _require_cuda(x, W, b, addend)
        with torch.autocast("cuda", enabled=False):
            shape = x.shape
            x2 = x.detach().to(cdtype).reshape(-1, shape[-1])
            if x2.stride(-1) != 1 or (x2.shape[0] > 1 and x2.stride(0) % 8):
                x2 = x2.contiguous()
            Wc, WT = cast_transpose(W.detach(), cdtype)
            add2 = None if addend is None else addend.detach().reshape(-1, W.shape[0])
            y = gemm_nt(x2, Wc, bias=_f32c(b), addend=add2, out_dtype=out_dtype)
            if needs_bwd:
                ctx.save_for_backward(x2, WT)
                ctx.meta = (shape, x.dtype, W.dtype, None if b is None else b.dtype, addend is not None)
            return y.view(*shape[:-1], W.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, WT = ctx.saved_tensors
        shape, xdt, wdt, bdt, has_add = ctx.meta
        with torch.autocast("cuda", enabled=False):
            g = dy.reshape(-1, WT.shape[1]).to(x2.dtype)
            if g.stride(-1) != 1 or g.stride(0) != g.shape[1]:
                g = g.contiguous()
            with _Fork() as f:
                db = colsum(g) if bdt is not None else None
                dW = wgrad(g, x2)
            dx = gemm_nt(g, WT)
            f.join()
        return (dx.view(shape).to(xdt), dW.to(wdt), None if db is None else db.to(bdt), dy if has_add else None,
                None, None, None)


def linear_fn(x, W, b=None, addend=None, compute_dtype=None, out_dtype=None):
    if compute_dtype is None:
        compute_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    out_dtype = out_dtype or (addend.dtype if addend is not None else compute_dtype)
    return LinearFn.apply(x, W, b, addend, compute_dtype, out_dtype, _wants_grad(x, W, b, addend))


def layer_norm_fn(x, weight, bias, eps=1e-5, out_dtype=None, with_residual=False):
    """LayerNorm over the last axis; out_dtype defaults to the autocast dtype when autocast is on, else x.dtype.
    with_residual=True returns (LayerNorm(x), x): use the second output as the residual branch of a pre-norm layer
    (out = f(LN(x)) + x) and its gradient is added inside the LayerNorm backward kernel."""
    if out_dtype is None:
        out_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    return LayerNormFn.apply(x, weight, bias, eps, out_dtype, _wants_grad(x, weight, bias), with_residual)


# ----------------------------------------------------------------------------------------
# the fused block: both directions, shared weights
# ----------------------------------------------------------------------------------------
def pack_weights(W_in, W_x, W_dt, A_log, W_out, ndir: int, dtype):
    """One launch: fp32 master parameters -> (Wi, WiT, Wxp, WxpT, Wo2, WoT, WdT) in `dtype` and A = -exp(A_log) fp32
    (layouts in include/bimamba.h: bimamba_pack_weights)."""
    lib = _lib.load()
    D2, dm = W_in.shape
    D = D2 // 2
    N = A_log.shape[1]
    R = W_dt.shape[1]
    sizes = (D2 * dm, D2 * dm, XW * D, XW * D, dm * ndir * D, D * dm, MAX_DT_RANK * D)
    flat = torch.empty((sum(sizes),), device=W_in.device, dtype=dtype)
    shapes = ((D2, dm), (dm, D2), (XW, D), (D, XW), (dm, ndir * D), (D, dm), (MAX_DT_RANK, D))
    outs, off = [], 0
    for n_, sh in zip(sizes, shapes):       # every size is a multiple of 8 elements -> 16-byte aligned views
        outs.append(flat[off:off + n_].view(sh))
        off += n_
    A32 = torch.empty((D, N), device=W_in.device, dtype=torch.float32)
    srcs = [_f32c(t) for t in (W_in, W_x, W_dt, A_log, W_out)]
    with _timed("pack"):
        _lib.check(lib.bimamba_pack_weights(*[_ptr(t) for t in srcs], *[_ptr(t) for t in outs], _ptr(A32),
                                            dm, D, N, R, ndir, _DT[dtype], _stream()), "bimamba_pack_weights")
    return (*outs, A32)


def cast_transpose(W: torch.Tensor, dtype):
    """fp32 (rows, cols) weight -> (W in dtype, W^T in dtype) with one launch."""
    lib = _lib.load()
    rows, cols = W.shape
    src = _f32c(W)
    dst = torch.empty((rows, cols), device=W.device, dtype=dtype)
    dstT = torch.empty((cols, rows), device=W.device, dtype=dtype)
    with _timed("pack"):
        _lib.check(lib.bimamba_cast_transpose(_ptr(src), _ptr(dst), _ptr(dstT), rows, cols, _DT[dtype], _stream()),
                   "bimamba_cast_transpose")
    return dst, dstT


class BiMambaInnerFn(torch.autograd.Function):
    """out = M(x) [+ flip(M(flip(x)))] for one Mamba block M with shared weights.

    Reference: mamba_block.py:41-63 for M, DualStreamSEMamba.py:473-481 for the two directions.
    Uses (SURVEY 3.3): in_proj(flip x) = flip(in_proj x) so xz is computed once; the reverse
    direction reads the same x, z back to front; out_proj is ONE GEMM over [y_fwd | y_rev] against
    [W_out | W_out].  The dt projection (K = 9) is fused into the scan kernels.
    Every product runs on this repository's tcgen05 kernels: forward and data-gradient GEMMs on gemm_nt, weight
    gradients (contraction over B*L) on gemm_tn, fp32 operands through the three-term bf16 split (_split3).  Conv,
    scan, dt_proj and all reductions are this repository's CUDA kernels too.
    """

    @staticmethod
    def forward(ctx, x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out, bidirectional, cdtype, needs_bwd=True,
                seqlens=None):
        _require_cuda(x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out)
        with torch.autocast("cuda", enabled=False):
            Bsz, L, dm = x.shape
            D = W_in.shape[0] // 2
            N = A_log.shape[1]
            R = W_dt.shape[1]
            if N != D_STATE:
                raise NotImplementedError("d_state must be 16 (the Phase-6 configuration)")
            if R > MAX_DT_RANK:
                raise NotImplementedError("dt_rank must be <= 16")
            ndir = 2 if bidirectional else 1
            M = Bsz * L
            dev = x.device
            Wi, WiT, Wxp, WxpT, Wo2, WoT, WdT, A32 = pack_weights(W_in.detach(), W_x.detach(), W_dt.detach(),
                                                                  A_log.detach(), W_out.detach(), ndir, cdtype)
            Wd32 = _f32c(W_dt)
            cw32 = _f32c(conv_w).reshape(D, -1)
            cb32 = _f32c(conv_b)
            D32, bdt32 = _f32c(Dp), _f32c(b_dt)

            x2 = x.detach().to(cdtype).reshape(M, dm)
            xz = gemm_nt(x2, Wi)                                              # (M, 2D)   mamba_block.py:48
            xz3 = xz.view(Bsz, L, 2 * D)
            xs, z = xz3[:, :, :D], xz3[:, :, D:]                              # :49 (views)
            xc = per_dir(Bsz, L, ndir, D, dev, cdtype)
            conv_fwd_raw(xs, cw32, cb32, xc, True, seqlens)                   # :52-55, both directions
            xdbl = gemm_nt(rows2d(xc), Wxp)                                   # (M*ndir, 48)   :73
            xd4 = xdbl.view(Bsz, L, ndir, XW).permute(0, 2, 1, 3)
            y, ckpt, ypre = scan_fwd_raw(xc, z.unsqueeze(1).expand(Bsz, ndir, L, D), None, xd4[..., :2 * N],
                                         xd4[..., 2 * N:], Wd32, A32, D32, bdt32, True, needs_bwd,
                                         dtr_padded=True, seqlens=seqlens)    # :80-120, :61
            out = gemm_nt(rows2d(y).view(M, ndir * D), Wo2).view(Bsz, L, dm)  # :62 + DualStreamSEMamba.py:481
            if needs_bwd:
                ctx.save_for_backward(x2, xz, xc, xdbl, y, WiT, WxpT, WoT, WdT, Wd32, cw32, cb32, A32, D32, bdt32,
                                      ckpt if ckpt is not None else torch.empty(0), ypre)
                ctx.meta = (Bsz, L, ndir, R, x.dtype,
                            tuple(t.dtype for t in (W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out)),
                            tuple(conv_w.shape))
                ctx.seqlens = seqlens
            return out

    @staticmethod
    def backward(ctx, dout):
        (x2, xz, xc, xdbl, y, WiT, WxpT, WoT, WdT, Wd32, cw32, cb32, A32, D32, bdt32, ckpt, ypre) = ctx.saved_tensors
        Bsz, L, ndir, R, xdt, pdt, cw_shape = ctx.meta
        ckpt = ckpt if ckpt.numel() else None
        with torch.autocast("cuda", enabled=False):
            cd = xz.dtype
            M, dm = x2.shape
            D = xz.shape[1] // 2
            N = A32.shape[1]
            xz3 = xz.view(Bsz, L, 2 * D)
            xs, z = xz3[:, :, :D], xz3[:, :, D:]
            xd4 = xdbl.view(Bsz, L, ndir, XW).permute(0, 2, 1, 3)

            g2 = dout.reshape(M, dm)
            if g2.stride(1) != 1 or g2.stride(0) != dm:
                g2 = g2.contiguous()
            g2 = cast(g2, cd)
            # out_proj
            y2 = rows2d(y).view(M, ndir * D)
            with _Fork() as f_out:                                            # out_proj weight gradient || dy, scan
                dW_out2 = wgrad(g2, y2)                                    # (dm, ndir*D), folded over directions at the end
            dy = gemm_nt(g2, WoT)                                             # (M, D), shared by both directions
            # scan (both directions in one launch); dy and z are broadcast over the direction axis
            dyb = dy.view(Bsz, 1, L, D).expand(Bsz, ndir, L, D)
            forks = []                                                        # dA / dD / dbias sums run beside the chain
            dxdbl = torch.empty((M * ndir, XW), device=xz.device, dtype=cd)   # [dB | dC | ddt_r | 0], rows (b, t, dir)
            du, ddelta, dz, _, dA, dD, dbdt = scan_bwd_raw(
                xc, z.unsqueeze(1).expand(Bsz, ndir, L, D), None, xd4[..., :2 * N], xd4[..., 2 * N:], Wd32,
                A32, D32, bdt32, True, dyb, ckpt, ypre, dtr_padded=True, defer=forks, dbc_rows=dxdbl, seqlens=ctx.seqlens)
            # dt_proj (weight gradient in fp32; the data gradient is written next to dB | dC: no concatenation)
            dd2 = rows2d(ddelta)                                              # (M*ndir, D)
            gemm_nt(dd2, WdT, out=dxdbl[:, 2 * N:])                           # (M*ndir, 16)
            xc2 = rows2d(xc)
            with _Fork() as f_w:                                              # dt_proj / x_proj weight gradients || dxc, conv
                dW_dtf = wgrad(dd2, xdbl)                                   # (D, 48): columns 2N..2N+R are dt_proj.weight's
                dW_xp = wgrad(dxdbl, xc2)                                   # (48, D)
            # x_proj
            dxc = gemm_nt(dxdbl, WxpT, addend=rows2d(du))                     # (M*ndir, D)
            dxc4 = dxc.view(Bsz, L, ndir, D).permute(0, 2, 1, 3)
            # conv (writes dx into the x half and dz_fwd + dz_rev into the z half of dxz)
            dxz = torch.empty_like(xz)
            dxz3 = dxz.view(Bsz, L, 2 * D)
            dwb = conv_bwd_raw(xs, cw32, cb32, dxc4, dxz3[:, :, :D], True, dz_in=dz, dz_out=dxz3[:, :, D:], defer=forks,
                               seqlens=ctx.seqlens)
            K = cw32.shape[1]
            # in_proj
            with _Fork() as f_in:                                             # in_proj weight gradient || its data gradient
                dW_in = wgrad(dxz, x2)                                      # (2D, dm)
            dx = gemm_nt(dxz, WiT).view(Bsz, L, dm)
            for f in (f_out, f_w, f_in, *forks):
                f.join()
            # one launch: dA_log = dA * A, x_proj rows back to [dt_r | B | C], dt_proj slice, out_proj fold, conv split
            dev = xz.device
            f32 = torch.float32
            dA_log = torch.empty((D, N), device=dev, dtype=f32)
            dW_x = torch.empty((R + 2 * N, D), device=dev, dtype=f32)
            dW_dt = torch.empty((D, R), device=dev, dtype=f32)
            dW_out = torch.empty((dm, D), device=dev, dtype=f32)
            dcw = torch.empty(cw_shape, device=dev, dtype=f32)
            dcb = torch.empty((D,), device=dev, dtype=f32)
            with _timed("finalize"):
                _lib.check(_lib.load().bimamba_finalize_param_grads(
                    _ptr(dA), _ptr(A32), _ptr(dW_xp), _ptr(dW_dtf), _ptr(dW_out2), _ptr(dwb), _ptr(dA_log), _ptr(dW_x),
                    _ptr(dW_dt), _ptr(dW_out), _ptr(dcw), _ptr(dcb), dm, D, N, R, ndir, K, _stream()),
                    "bimamba_finalize_param_grads")
        return (dx.to(xdt), dW_in.to(pdt[0]), dcw.to(pdt[1]), dcb.to(pdt[2]),
                dW_x.to(pdt[3]), dW_dt.to(pdt[4]), dbdt.to(pdt[5]), dA_log.to(pdt[6]), dD.to(pdt[7]),
                dW_out.to(pdt[8]), None, None, None, None)


# Eager mode (no CUDA-graph capture): the block runs through the one-call native entry points - the same kernels in the
# same order, bit-identical results (tests/test_gpu_native_block.py), but one ctypes call each way instead of ~30 plus
# their allocations: 0.45 ms against 1.25 ms per block forward + backward at batch 64 x 201 frames, where the Python
# sequencing is host-bound (profiles/r2_native_block_eager.json).  Under capture the sequenced Function stays: it
# overlaps the weight-gradient products with the data-gradient chain on a second stream.
USE_NATIVE_BLOCK = True


class sequenced_block:
    """Context manager: keep the block on the sequenced autograd Function (the warm-up steps of a graph capture run
    exactly what the capture will record; per-kernel timing; A/B tests of the two arrangements)."""

    def __enter__(self):
        global USE_NATIVE_BLOCK
        self.old, USE_NATIVE_BLOCK = USE_NATIVE_BLOCK, False
        return self

    def __exit__(self, *a):
        global USE_NATIVE_BLOCK
        USE_NATIVE_BLOCK = self.old
        return False


def _native_block_ok(x, W_in, cdtype) -> bool:
    return (USE_NATIVE_BLOCK and _lib.kernel_timer is None and cdtype in (torch.bfloat16, torch.float16)
            and x.is_cuda and x.numel() > 0 and W_in.shape[1] % 8 == 0 and (W_in.shape[0] // 2) % 8 == 0
            and not torch.cuda.is_current_stream_capturing())


class BiMambaNativeFn(torch.autograd.Function):
    """BiMambaInnerFn through bimamba_block_fwd / bimamba_block_bwd (csrc/block.cu): eager-mode fast path."""

    @staticmethod
    def forward(ctx, x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out, bidirectional, cdtype, needs_bwd=True,
                seqlens=None):
        with torch.autocast("cuda", enabled=False):
            if A_log.shape[1] != D_STATE:
                raise NotImplementedError("d_state must be 16 (the Phase-6 configuration)")
            if W_dt.shape[1] > MAX_DT_RANK:
                raise NotImplementedError("dt_rank must be <= 16")
            nb = NativeBlock(x.detach().to(cdtype), W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out,
                             bidirectional=bidirectional, save_for_backward=needs_bwd, seqlens=seqlens)
            out, nb.out = nb.out, None          # the output must not be reachable from ctx (reference cycle)
            if needs_bwd:
                ctx.nb = nb
                ctx.meta = (x.dtype, tuple(t.dtype for t in (W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out)))
            return out

    @staticmethod
    def backward(ctx, dout):
        xdt, pdt = ctx.meta
        with torch.autocast("cuda", enabled=False):
            grads = ctx.nb.backward(dout)
        return (grads[0].to(xdt), *[g.to(d) for g, d in zip(grads[1:], pdt)], None, None, None, None)


def bimamba_inner_fn(x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out, bidirectional=True,
                     compute_dtype=None, lengths=None, *, mask_padding=False):
    """x (B, L, d_model) -> (B, L, d_model).  compute_dtype: activation dtype of the kernels and
    GEMMs (default: the autocast dtype when autocast is on, else x.dtype); scan state is fp32.
    lengths (B,): utterance b is frames 0 .. lengths[b]-1 of the right-padded x (seqlens_tensor); each valid output frame
    equals that of the utterance run alone at its own length, output frames at padded positions are unspecified.
    Without mask_padding this is scoring only: with lengths and autograd recording it raises NotImplementedError.
    mask_padding=True (with lengths) is the training form: the padded frames of x are replaced by zeros (selection, so
    NaN padding cannot pass), padded output frames are exactly zero, the gradient at padded input frames is zero, and
    the loss and every gradient are those of each utterance run alone, parameter gradients summed over utterances."""
    if compute_dtype is None:
        compute_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    _check_mask_padding(lengths, mask_padding)
    seqlens = seqlens_tensor(lengths, x.shape[0], x.shape[1], x.device)
    _require_cuda(x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out)
    ps = (x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out)
    if mask_padding:
        ps = (mask_frames(x, seqlens),) + ps[1:]
    else:
        _forward_only(seqlens, *ps)
    fn = BiMambaNativeFn if _native_block_ok(x, W_in, compute_dtype) else BiMambaInnerFn
    return fn.apply(*ps, bool(bidirectional), compute_dtype, _wants_grad(*ps), seqlens)


# ----------------------------------------------------------------------------------------
# the same block through the ONE-CALL native entry points (bimamba_block_fwd / bimamba_block_bwd): what a host without an
# autograd framework binds.  The autograd Function above stays the Python product path (it overlaps the weight-gradient
# products on a side stream); these wrappers exist so that the entry points are exercised against it bit for bit.
# ----------------------------------------------------------------------------------------
class NativeBlock:
    """State of one forward call of the native block: descriptor, saved-activation workspace, packed weights."""

    def __init__(self, x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out, bidirectional=True,
                 save_for_backward=True, seqlens=None):
        _require_cuda(x, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out)
        if x.dtype not in (torch.bfloat16, torch.float16):
            raise TypeError("the native block entry points take bf16 / fp16 activations")
        lib = _lib.load()
        Bsz, L, dm = x.shape
        D = W_in.shape[0] // 2
        R = W_dt.shape[1]
        ndir = 2 if bidirectional else 1
        self.x = x.contiguous()
        self.shape = (Bsz, L, dm, D, R, ndir)
        self.packed = pack_weights(W_in.detach(), W_x.detach(), W_dt.detach(), A_log.detach(), W_out.detach(), ndir, x.dtype)
        Wi, WiT, Wxp, WxpT, Wo2, WoT, WdT, A32 = self.packed
        self.f32 = (_f32c(W_dt.detach()), _f32c(conv_w.detach()).reshape(D, -1), _f32c(conv_b.detach()),
                    _f32c(Dp.detach()), _f32c(b_dt.detach()))
        Wd32, cw32, cb32, D32, bdt32 = self.f32
        K = cw32.shape[1]
        self.K = K
        nbytes = lib.bimamba_block_fwd_workspace_bytes(Bsz, L, dm, D, ndir, _dt(x), int(save_for_backward))
        self.ws = torch.empty((max(nbytes, 1),), device=x.device, dtype=torch.uint8)
        self.out = torch.empty_like(self.x)
        d = _lib.BlockDesc()
        d.x, d.out = _ptr(self.x), _ptr(self.out)
        d.Wi, d.Wxp, d.Wo2 = _ptr(Wi), _ptr(Wxp), _ptr(Wo2)
        d.Wdt, d.A, d.D, d.dt_bias, d.conv_w, d.conv_b = (_ptr(Wd32), _ptr(A32), _ptr(D32), _ptr(bdt32), _ptr(cw32),
                                                          _ptr(cb32))
        d.workspace, d.workspace_bytes = _ptr(self.ws), nbytes
        d.batch, d.seqlen, d.d_model, d.d_inner, d.dt_rank, d.d_conv, d.ndir = Bsz, L, dm, D, R, K, ndir
        d.io_dtype, d.save_for_backward = _dt(x), int(save_for_backward)
        self.desc = d
        self.seqlens = seqlens
        fwd = lib.bimamba_block_fwd_varlen_train if save_for_backward else lib.bimamba_block_fwd_varlen
        _lib.check(fwd(C.byref(d), _ptr(seqlens), _stream()), "bimamba_block_fwd_varlen")
        _lib.launch_count += 4           # the call enqueues 5 kernels (3 GEMMs, conv, scan)

    def backward(self, dout):
        """-> (dx, dW_in, dconv_w, dconv_b, dW_x, dW_dt, db_dt, dA_log, dD, dW_out), fp32 parameter gradients in the
        reference's shapes."""
        lib = _lib.load()
        Bsz, L, dm, D, R, ndir = self.shape
        K, N = self.K, D_STATE
        Wi, WiT, Wxp, WxpT, Wo2, WoT, WdT, A32 = self.packed
        dev, f32 = self.x.device, torch.float32
        dout = dout.to(self.x.dtype).contiguous()
        dx = torch.empty_like(self.x)
        grads = [torch.empty(s, device=dev, dtype=f32) for s in
                 ((2 * D, dm), (D, 1, K), (D,), (R + 2 * N, D), (D, R), (D,), (D, N), (D,), (dm, D))]
        nbytes = lib.bimamba_block_bwd_workspace_bytes(Bsz, L, dm, D, K, ndir, _dt(self.x))
        ws = torch.empty((max(nbytes, 1),), device=dev, dtype=torch.uint8)
        g = _lib.BlockGrads()
        g.dout, g.dx = _ptr(dout), _ptr(dx)
        g.WiT, g.WxpT, g.WoT, g.WdT = _ptr(WiT), _ptr(WxpT), _ptr(WoT), _ptr(WdT)
        (g.dW_in, g.dconv_w, g.dconv_b, g.dW_x, g.dW_dt, g.db_dt, g.dA_log, g.dD, g.dW_out) = [_ptr(t) for t in grads]
        g.workspace, g.workspace_bytes = _ptr(ws), nbytes
        _lib.check(lib.bimamba_block_bwd_varlen(C.byref(self.desc), C.byref(g), _ptr(self.seqlens), _stream()),
                   "bimamba_block_bwd_varlen")
        _lib.launch_count += 19          # 20 kernels: 4 + 4 x 2 GEMMs, scan, conv, row sum, 4 partial sums, layout pass
        self._keep = (dout, ws)
        return (dx, *grads)


# ----------------------------------------------------------------------------------------
# the whole encoder layer through bimamba_layer_fwd / bimamba_layer_bwd (eager-mode fast path of
# PN_BiMambas_Encoder.forward; bit-identical to layer_norm_fn -> bimamba_inner_fn -> layer_norm_fn -> feed_forward_fn)
# ----------------------------------------------------------------------------------------
class NativeLayer:
    """One forward call of the native encoder layer: descriptor, saved-activation workspace, packed Mamba weights."""

    def __init__(self, x, norm1_w, norm1_b, eps1, norm2_w, norm2_b, eps2, W1, b1, W2, b2, W_in, conv_w, conv_b, W_x, W_dt,
                 b_dt, A_log, Dp, W_out, cdtype, save_for_backward=True, seqlens=None):
        _require_cuda(x, norm1_w, W1, W_in)
        lib = _lib.load()
        Bsz, L, dm = x.shape
        D, R, dff = W_in.shape[0] // 2, W_dt.shape[1], W1.shape[0]
        self.x = x.detach().contiguous()
        self.shape = (Bsz, L, dm, D, R, dff)
        self.cdtype = cdtype
        self.packed = pack_weights(W_in.detach(), W_x.detach(), W_dt.detach(), A_log.detach(), W_out.detach(), 2, cdtype)
        Wi, WiT, Wxp, WxpT, Wo2, WoT, WdT, A32 = self.packed
        self.f32 = tuple(_f32c(t) for t in (W_dt, conv_w, conv_b, Dp, b_dt, norm1_w, norm1_b, norm2_w, norm2_b, W1, b1, W2, b2))
        Wd32, cw32, cb32, D32, bdt32, n1w, n1b, n2w, n2b, W1f, b1f, W2f, b2f = self.f32
        cw32 = cw32.reshape(D, -1)
        self.K = K = cw32.shape[1]
        cdt = _DT[cdtype]
        nbytes = lib.bimamba_layer_fwd_workspace_bytes(Bsz, L, dm, D, dff, 2, cdt, int(save_for_backward))
        self.ws = torch.empty((max(nbytes, 1),), device=x.device, dtype=torch.uint8)
        self.out = torch.empty_like(self.x)
        d = _lib.LayerDesc()
        d.x, d.out = _ptr(self.x), _ptr(self.out)
        d.norm1_w, d.norm1_b, d.norm2_w, d.norm2_b = _ptr(n1w), _ptr(n1b), _ptr(n2w), _ptr(n2b)
        d.ff_w1, d.ff_b1, d.ff_w2, d.ff_b2 = _ptr(W1f), _ptr(b1f), _ptr(W2f), _ptr(b2f)
        k = d.block
        k.Wi, k.Wxp, k.Wo2 = _ptr(Wi), _ptr(Wxp), _ptr(Wo2)
        k.Wdt, k.A, k.D, k.dt_bias, k.conv_w, k.conv_b = _ptr(Wd32), _ptr(A32), _ptr(D32), _ptr(bdt32), _ptr(cw32), _ptr(cb32)
        k.batch, k.seqlen, k.d_model, k.d_inner, k.dt_rank, k.d_conv, k.ndir = Bsz, L, dm, D, R, K, 2
        k.io_dtype, k.save_for_backward = cdt, int(save_for_backward)
        d.workspace, d.workspace_bytes = _ptr(self.ws), nbytes
        d.eps1, d.eps2, d.d_ff, d.x_dtype = float(eps1), float(eps2), dff, _dt(self.x)
        self.desc = d
        self._keep_fwd = (cw32,)
        self.seqlens = seqlens
        fwd = lib.bimamba_layer_fwd_varlen_train if save_for_backward else lib.bimamba_layer_fwd_varlen
        _lib.check(fwd(C.byref(d), _ptr(seqlens), _stream()), "bimamba_layer_fwd_varlen")
        _lib.launch_count += 11          # 12 kernels: 2 LayerNorm, 5 of the block, 2 weight casts, 2 GEMMs, GELU

    def backward(self, dout):
        """-> (dx, dnorm1 (2, dm), dnorm2 (2, dm), dW1, db1, dW2, db2, then the nine Mamba gradients in the order
        W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, D, W_out)."""
        lib = _lib.load()
        Bsz, L, dm, D, R, dff = self.shape
        K, N = self.K, D_STATE
        Wi, WiT, Wxp, WxpT, Wo2, WoT, WdT, A32 = self.packed
        dev, f32 = self.x.device, torch.float32
        dout = dout.to(self.x.dtype).contiguous()
        dx = torch.empty_like(self.x)
        lg = [torch.empty(s, device=dev, dtype=f32) for s in ((2, dm), (2, dm), (dff, dm), (dff,), (dm, dff), (dm,))]
        mg = [torch.empty(s, device=dev, dtype=f32) for s in
              ((2 * D, dm), (D, 1, K), (D,), (R + 2 * N, D), (D, R), (D,), (D, N), (D,), (dm, D))]
        nbytes = lib.bimamba_layer_bwd_workspace_bytes(Bsz, L, dm, D, dff, K, 2, _DT[self.cdtype])
        ws = torch.empty((max(nbytes, 1),), device=dev, dtype=torch.uint8)
        g = _lib.LayerGrads()
        g.dout, g.dx = _ptr(dout), _ptr(dx)
        (g.dnorm1, g.dnorm2, g.dff_w1, g.dff_b1, g.dff_w2, g.dff_b2) = [_ptr(t) for t in lg]
        kg = g.block
        kg.WiT, kg.WxpT, kg.WoT, kg.WdT = _ptr(WiT), _ptr(WxpT), _ptr(WoT), _ptr(WdT)
        (kg.dW_in, kg.dconv_w, kg.dconv_b, kg.dW_x, kg.dW_dt, kg.db_dt, kg.dA_log, kg.dD, kg.dW_out) = [_ptr(t) for t in mg]
        g.workspace, g.workspace_bytes = _ptr(ws), nbytes
        _lib.check(lib.bimamba_layer_bwd_varlen(C.byref(self.desc), C.byref(g), _ptr(self.seqlens), _stream()),
                   "bimamba_layer_bwd_varlen")
        _lib.launch_count += 35          # 36 kernels: 20 of the block, 11 of the feed-forward, 2 x 2 of the norms, the cast of dout
        self._keep = (dout, ws)
        return (dx, *lg, *mg)


class EncoderLayerNativeFn(torch.autograd.Function):
    """PN_BiMambas_Encoder.forward (DualStreamSEMamba.py:467-486) as one native call each way."""

    @staticmethod
    def forward(ctx, x, n1w, n1b, n2w, n2b, W1, b1, W2, b2, W_in, conv_w, conv_b, W_x, W_dt, b_dt, A_log, Dp, W_out,
                eps1, eps2, cdtype, needs_bwd=True, seqlens=None):
        with torch.autocast("cuda", enabled=False):
            if A_log.shape[1] != D_STATE:
                raise NotImplementedError("d_state must be 16 (the Phase-6 configuration)")
            if W_dt.shape[1] > MAX_DT_RANK:
                raise NotImplementedError("dt_rank must be <= 16")
            nl = NativeLayer(x, n1w, n1b, eps1, n2w, n2b, eps2, W1, b1, W2, b2, W_in, conv_w, conv_b, W_x, W_dt, b_dt,
                             A_log, Dp, W_out, cdtype, save_for_backward=needs_bwd, seqlens=seqlens)
            out, nl.out = nl.out, None          # the output must not be reachable from ctx (reference cycle)
            if needs_bwd:
                ctx.nl = nl
                ctx.pdt = tuple(t.dtype for t in (n1w, n1b, n2w, n2b, W1, b1, W2, b2, W_in, conv_w, conv_b, W_x, W_dt, b_dt,
                                                  A_log, Dp, W_out))
            return out.view(x.shape)

    @staticmethod
    def backward(ctx, dout):
        with torch.autocast("cuda", enabled=False):
            r = ctx.nl.backward(dout)
        dx, dn1, dn2 = r[0], r[1], r[2]
        grads = [dn1[0], dn1[1], dn2[0], dn2[1], *r[3:]]
        return (dx.view(dout.shape), *[g.to(d) for g, d in zip(grads, ctx.pdt)], None, None, None, None, None)


def native_layer_ok(x, layer) -> bool:
    """Eager-mode fast path of the encoder layer: CUDA, no graph capture, a 16-bit compute dtype (autocast, or 16-bit x),
    x in fp32 or that dtype, exact GELU, widths the kernels take."""
    if not (USE_NATIVE_BLOCK and _lib.kernel_timer is None and x.is_cuda and x.dim() == 3 and x.numel() > 0):
        return False
    cd = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    ff = layer.feed_forward
    if cd not in (torch.bfloat16, torch.float16) or x.dtype not in (torch.float32, cd):
        return False
    if not (len(ff) == 3 and isinstance(ff[0], torch.nn.Linear) and isinstance(ff[1], torch.nn.GELU)
            and ff[1].approximate == "none" and isinstance(ff[2], torch.nn.Linear) and ff[0].bias is not None
            and ff[2].bias is not None):
        return False
    dm = x.shape[-1]
    m = layer.mamba
    return (dm % 8 == 0 and dm <= 1024 and ff[0].out_features % 8 == 0 and m.d_inner % 8 == 0 and m.d_state == D_STATE
            and m.dt_rank <= MAX_DT_RANK and not torch.cuda.is_current_stream_capturing())


def encoder_layer_native(x, layer, seqlens=None, mask_padding=False):
    """seqlens: (B,) int32 device frame counts (seqlens_tensor) or None; scoring only unless mask_padding, which masks
    the layer's input and output (forward and backward, MaskFramesFn) as PN_BiMambas_Encoder.forward does."""
    cd = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    m, ff = layer.mamba, layer.feed_forward
    ps = (layer.norm1.weight, layer.norm1.bias, layer.norm2.weight, layer.norm2.bias, ff[0].weight, ff[0].bias,
          ff[2].weight, ff[2].bias, m.in_proj.weight, m.conv1d.weight, m.conv1d.bias, m.x_proj.weight, m.dt_proj.weight,
          m.dt_proj.bias, m.A_log, m.D, m.out_proj.weight)
    if mask_padding:
        x = mask_frames(x, seqlens)
    else:
        _forward_only(seqlens, x, *ps)
    out = EncoderLayerNativeFn.apply(x, *ps, layer.norm1.eps, layer.norm2.eps, cd, _wants_grad(x, *ps), seqlens)
    return mask_frames(out, seqlens) if mask_padding else out
