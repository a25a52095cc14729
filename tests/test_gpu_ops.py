"""GPU parity of the op-level kernels (through the C ABI) against the CPU oracle.

Tolerances are the ones BASELINE.json's north_star states: <= 1e-4 relative in fp32, <= 2e-2 in bf16 (fp32 state),
measured per slice against the fp64 oracle (oracle/compare.py): every state, channel, 8-step chunk and utterance of a
tensor against its own magnitude.
"""
import pytest
import torch

import bimamba_b200 as bm
from oracle import bimamba_oracle as orc
from oracle import compare as cmp

pytestmark = pytest.mark.gpu

TOL = cmp.TOL
# (B, D, L) scan activations and data gradients, (B, N, L) dB / dC, then the parameter gradients
SLICES = {"out": cmp.scan_act(0, 1, 2), "du": cmp.scan_act(0, 1, 2), "ddelta": cmp.scan_act(0, 1, 2),
          "dz": cmp.scan_act(0, 1, 2), "dB": cmp.scan_state(0, 1), "dC": cmp.scan_state(0, 1),
          "dA": cmp.CHANNEL_STATE, "dD": cmp.CHANNELS, "dbias": cmp.CHANNELS}
_scan_inputs = orc.scan_inputs


def _run_both(Bsz, D, L, dtype, with_z=True, with_D=True, with_bias=True, softplus=True, seed=0):
    """The scan forward and backward on the GPU against the fp64 oracle on the same (dtype-rounded) inputs: the output
    and every gradient, per slice at TOL[dtype]."""
    u, delta, z, Bm, Cm, A, Dp, bias = _scan_inputs(Bsz, D, L, seed=seed, dtype=dtype)
    if not softplus:          # a raw delta must be a positive step size
        delta = (0.2 * delta.float().abs()).to(dtype)
        bias = bias.abs()
    names = ["u", "delta", "A", "B", "C", "D", "z", "bias"]
    cpu = [u, delta, A, Bm, Cm, Dp if with_D else None, z if with_z else None, bias if with_bias else None]
    # oracle in fp64 on the (dtype-rounded) inputs
    ref_in = [None if t is None else t.double().requires_grad_(True) for t in cpu]
    ref = orc.selective_scan_ref(*ref_in, delta_softplus=softplus)
    g = torch.Generator().manual_seed(seed + 1)
    cot = torch.randn(ref.shape, generator=g).to(dtype)
    (ref * cot.double()).sum().backward()
    dev_in = [None if t is None else t.cuda().requires_grad_(True) for t in cpu]
    out = bm.selective_scan_fn(*dev_in, delta_softplus=softplus)
    assert out.dtype == dtype and out.shape == ref.shape
    out.backward(cot.cuda())
    torch.cuda.synchronize()
    tag = f"L={L} D={D} "
    cmp.check(tag + "out", out, ref, TOL[dtype], SLICES["out"])
    for n, a, b in zip(names, dev_in, ref_in):
        if a is not None:
            cmp.check(tag + "d" + n, a.grad, b.grad, TOL[dtype], SLICES["d" + n])


@pytest.mark.parametrize("L", [1, 5, 32, 33, 64, 201, 224, 256])
def test_scan_single_chunk_fp32(L):
    _run_both(2, 40, L, torch.float32)


@pytest.mark.parametrize("L", [257, 300, 499, 777, 1024])
def test_scan_multi_chunk_fp32(L):
    _run_both(2, 24, L, torch.float32, seed=L)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("L", [201, 499])
def test_scan_half_precision_io(dtype, L):
    _run_both(2, 48, L, dtype, seed=3)


@pytest.mark.parametrize("with_z,with_D,with_bias,softplus", [
    (False, True, True, True), (True, False, True, True), (True, True, False, True),
    (True, True, True, False), (False, False, False, False)])
def test_scan_optional_operands(with_z, with_D, with_bias, softplus):
    _run_both(3, 17, 77, torch.float32, with_z, with_D, with_bias, softplus, seed=5)


def test_scan_wide_and_ragged_channels():
    # dim = 288 (Phase 6) and a dim that is not a multiple of the channel group
    for D in (288, 37):
        _run_both(2, D, 201, torch.float32, seed=D)


def test_scan_empty():
    u = torch.zeros(0, 8, 16, device="cuda")
    out = bm.selective_scan_fn(u, u, -torch.ones(8, 16, device="cuda"), torch.zeros(0, 16, 16, device="cuda"),
                               torch.zeros(0, 16, 16, device="cuda"))
    assert out.shape == (0, 8, 16)


def test_scan_long_against_oracle_on_gpu():
    """Config-5 length (L = 8192): the oracle's sequential loop is run on the GPU in fp64
    (same oracle code, device-agnostic) because 8192 python steps on CPU tensors are slow."""
    u, delta, z, Bm, Cm, A, Dp, bias = _scan_inputs(2, 64, 8192, seed=9)
    dev = [t.cuda() for t in (u, delta, A, Bm, Cm, Dp, z, bias)]
    ref = orc.selective_scan_ref(*[t.double() for t in dev], delta_softplus=True)
    out = bm.selective_scan_fn(*dev, delta_softplus=True)
    cmp.check("out", out, ref, TOL[torch.float32], SLICES["out"])


def test_scan_rejects_cpu_and_bad_state():
    u = torch.zeros(1, 8, 16)
    with pytest.raises(RuntimeError):
        bm.selective_scan_fn(u, u, -torch.ones(8, 16), torch.zeros(1, 16, 16), torch.zeros(1, 16, 16))
    uc = u.cuda()
    with pytest.raises(NotImplementedError):
        bm.selective_scan_fn(uc, uc, -torch.ones(8, 8).cuda(), torch.zeros(1, 8, 16).cuda(), torch.zeros(1, 8, 16).cuda())


# ---------------------------------------------------------------- conv
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("L", [1, 3, 8, 201, 300])
@pytest.mark.parametrize("act", [None, "silu"])
def test_causal_conv1d(dtype, L, act):
    g = torch.Generator().manual_seed(L)
    Bsz, D, K = 3, 20, 4
    x = torch.randn(Bsz, D, L, generator=g).to(dtype)
    w = torch.randn(D, K, generator=g) * 0.5
    b = torch.randn(D, generator=g) * 0.5
    cot = torch.randn(Bsz, D, L, generator=g).to(dtype)
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    ref = orc.causal_conv1d_ref(xr, wr, br, act)
    (ref * cot.double()).sum().backward()
    xd, wd, bd = (t.cuda().requires_grad_(True) for t in (x, w, b))
    out = bm.causal_conv1d_fn(xd, wd, bd, activation=act)
    out.backward(cot.cuda())
    tol = TOL[dtype]
    cmp.check("out", out, ref, tol, cmp.scan_act(0, 1, 2))
    cmp.check("dx", xd.grad, xr.grad, tol, cmp.scan_act(0, 1, 2))
    cmp.check("conv1d.weight", wd.grad, wr.grad, tol, cmp.param("conv1d.weight", wr.shape))
    cmp.check("conv1d.bias", bd.grad, br.grad, tol, cmp.CHANNELS)


@pytest.mark.parametrize("D,force_tile", [(20, True), (18, False), (288, True)])
def test_causal_conv1d_backward_tile_kernel(D, force_tile):
    """The shared-memory tile backward (fallback for rows that are not addressable as 4-channel vectors) against the
    oracle: forced through bimamba_set_tuning for vector-friendly widths, taken automatically for D = 18."""
    with bm._lib.tuning(bm._lib.TUNE_CONV_BWD, 1 if force_tile else 0):
        _conv_bwd_case(D)


def _conv_bwd_case(D):
    g = torch.Generator().manual_seed(D)
    Bsz, K, L = 2, 4, 77
    x = torch.randn(Bsz, D, L, generator=g)
    w = torch.randn(D, K, generator=g) * 0.5
    b = torch.randn(D, generator=g) * 0.5
    cot = torch.randn(Bsz, D, L, generator=g)
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    (orc.causal_conv1d_ref(xr, wr, br, "silu") * cot.double()).sum().backward()
    xd, wd, bd = (t.cuda().requires_grad_(True) for t in (x, w, b))
    bm.causal_conv1d_fn(xd, wd, bd, activation="silu").backward(cot.cuda())
    cmp.check("dx", xd.grad, xr.grad, 1e-5, cmp.scan_act(0, 1, 2))
    cmp.check("conv1d.weight", wd.grad, wr.grad, 1e-5, cmp.param("conv1d.weight", wr.shape))
    cmp.check("conv1d.bias", bd.grad, br.grad, 1e-5, cmp.CHANNELS)


@pytest.mark.parametrize("K", [2, 3, 4])
def test_causal_conv1d_widths_no_bias(K):
    g = torch.Generator().manual_seed(K)
    x = torch.randn(2, 9, 50, generator=g)
    w = torch.randn(9, K, generator=g)
    ref = orc.causal_conv1d_ref(x.double(), w.double(), None, "silu")
    out = bm.causal_conv1d_fn(x.cuda(), w.cuda(), None, activation="silu")
    cmp.check("out", out, ref, 1e-5, cmp.scan_act(0, 1, 2))


# ---------------------------------------------------------------- layer norm
@pytest.mark.parametrize("C", [144, 64, 250])
@pytest.mark.parametrize("dtype,out_dtype", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16),
                                             (torch.bfloat16, torch.bfloat16)])
def test_layer_norm(C, dtype, out_dtype):
    """nn.LayerNorm of PN_BiMambas_Encoder (DualStreamSEMamba.py:472, :482) against torch in fp64."""
    g = torch.Generator().manual_seed(C)
    x = (torch.randn(5, 37, C, generator=g) * 2 + 0.5).to(dtype)
    w = 1 + 0.2 * torch.randn(C, generator=g)
    b = 0.3 * torch.randn(C, generator=g)
    cot = torch.randn(5, 37, C, generator=g).to(out_dtype)
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    ref = torch.nn.functional.layer_norm(xr, (C,), wr, br, 1e-5)
    (ref * cot.double()).sum().backward()
    xd, wd, bd = (t.cuda().requires_grad_(True) for t in (x, w, b))
    out = bm.ops.layer_norm_fn(xd, wd, bd, 1e-5, out_dtype=out_dtype)
    assert out.dtype == out_dtype and out.shape == x.shape
    out.backward(cot.cuda())
    tol = 1e-5 if (dtype == torch.float32 and out_dtype == torch.float32) else 2e-2
    cmp.check("out", out, ref, tol, cmp.frames())
    cmp.check("dx", xd.grad, xr.grad, tol, cmp.frames())
    cmp.check("weight", wd.grad, wr.grad, tol, cmp.CHANNELS)
    cmp.check("bias", bd.grad, br.grad, tol, cmp.CHANNELS)


# ---------------------------------------------------------------- tcgen05 GEMM
@pytest.mark.parametrize("M,N,K", [(128, 48, 288), (12864, 576, 144), (25728, 48, 288), (12864, 144, 576),
                                   (201, 288, 48), (1, 16, 8), (300, 41 + 7, 144), (257, 640, 72), (129, 45, 72)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_gemm_nt_tensor_cores(M, N, K, dtype):
    """nn.Linear products of the block (mamba_block.py:48, :73, :62) on the tcgen05 kernel against an fp64 product
    of the same rounded operands; bias, addend, fp32 output, ragged M / N / K."""
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).to(dtype)
    B = (torch.randn(N, K, generator=g) / K ** 0.5).to(dtype)
    bias = torch.randn(N, generator=g)
    add = torch.randn(M, N, generator=g).to(dtype)
    ref = A.double() @ B.double().t()
    Ad, Bd = A.cuda(), B.cuda()
    out = bm.ops.gemm_nt(Ad, Bd)
    assert out.dtype == dtype and out.shape == (M, N)
    assert cmp.rel(out, ref) < (4e-3 if dtype == torch.bfloat16 else 1e-3)
    out32 = bm.ops.gemm_nt(Ad, Bd, bias=bias.cuda(), out_dtype=torch.float32)
    assert cmp.rel(out32, ref + bias.double()) < 1e-5          # fp32 accumulation, exact operands
    out_add = bm.ops.gemm_nt(Ad, Bd, addend=add.cuda())          # product rounded to dtype, then + addend, rounded again
    assert cmp.rel(out_add, ref + add.double()) < (8e-3 if dtype == torch.bfloat16 else 2e-3)


def test_gemm_nt_strided_operand():
    """A as a column slice of a wider matrix (the x half of xz): lda > K."""
    g = torch.Generator().manual_seed(3)
    big = torch.randn(500, 576, generator=g).to(torch.bfloat16).cuda()
    W = (torch.randn(48, 288, generator=g) / 17).to(torch.bfloat16).cuda()
    out = bm.ops.gemm_nt(big[:, :288], W, out_dtype=torch.float32)
    assert cmp.rel(out, big[:, :288].double() @ W.double().t()) < 1e-5


# ---------------------------------------------------------------- feed-forward + column sums
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_feed_forward_fn(dtype):
    """Linear(144,576) -> GELU -> Linear(576,144) + residual (DualStreamSEMamba.py:460-464, :483-485) vs torch fp64."""
    g = torch.Generator().manual_seed(11)
    x = torch.randn(3, 70, 144, generator=g)
    res = torch.randn(3, 70, 144, generator=g)
    W1 = torch.randn(576, 144, generator=g) / 12
    b1 = torch.randn(576, generator=g) * 0.1
    W2 = torch.randn(144, 576, generator=g) / 24
    b2 = torch.randn(144, generator=g) * 0.1
    cot = torch.randn(3, 70, 144, generator=g)
    ref_in = [t.double().requires_grad_(True) for t in (x, W1, b1, W2, b2, res)]
    xr, W1r, b1r, W2r, b2r, rr = ref_in
    ref = torch.nn.functional.linear(torch.nn.functional.gelu(torch.nn.functional.linear(xr, W1r, b1r)), W2r, b2r) + rr
    (ref * cot.double()).sum().backward()
    dev_in = [t.cuda().requires_grad_(True) for t in (x, W1, b1, W2, b2, res)]
    out = bm.ops.feed_forward_fn(dev_in[0], *dev_in[1:5], residual=dev_in[5], compute_dtype=dtype)
    assert out.dtype == torch.float32                      # the residual stream stays fp32
    out.backward(cot.cuda())
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    cmp.check("out", out, ref, tol, cmp.frames())
    names = ["dx", "feed_forward.0.weight", "feed_forward.0.bias", "feed_forward.2.weight", "feed_forward.2.bias",
             "dresidual"]
    for n, a, b in zip(names, dev_in, ref_in):
        # fp32 dx keeps the whole-tensor rule at this test's 1e-5 (rho 1): on a B200, dx[2, 32:40], at 0.71 of the
        # tensor's largest element, is 1.1e-5 off (7.8e-6 of max|ref|), the rounding of the fp32 products on split-bf16
        # operands through both GEMMs
        rho = 1.0 if n == "dx" and dtype == torch.float32 else None
        cmp.check(n, a.grad, b.grad, tol, cmp.frames() if n.startswith("d") else cmp.param(n, b.shape), rho=rho)


@pytest.mark.parametrize("rows,cols", [(12864, 576), (1, 7), (300, 144)])
def test_colsum(rows, cols):
    g = torch.Generator().manual_seed(rows)
    x = torch.randn(rows, cols, generator=g).to(torch.bfloat16)
    out = bm.ops.colsum(x.cuda())
    assert cmp.rel(out, x.double().sum(0)) < 1e-5


@pytest.mark.parametrize("variant", [1, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scan_forward_variants(variant, dtype):
    """The two forward kernels (1: one lane per channel, wide CTAs; 3: one lane per channel, one warp per CTA) are
    forced in turn on the same inputs (bimamba_set_tuning); the size-based dispatch must not change results beyond
    rounding."""
    with bm._lib.tuning(bm._lib.TUNE_SCAN_FWD, variant):
        for L, D in ((201, 288), (37, 40), (499, 17)):
            _run_both(2, D, L, dtype, seed=L + D)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scan_backward_shapes(dtype):
    """The backward kernel on ragged shapes: channel counts that are not multiples of the 32-channel group or of the
    vector width, a single 8-step chunk, and every optional operand absent."""
    for L, D in ((201, 288), (37, 40), (499, 17), (8, 33)):
        _run_both(2, D, L, dtype, seed=L + D)
    _run_both(2, 40, 77, dtype, with_z=False, with_D=False, with_bias=False, softplus=False, seed=5)


@pytest.mark.parametrize("kernel", [1, 2])
def test_gemm_nt_kernel_variants(kernel):
    """Both tcgen05 kernels (1: one tile per CTA; 2: persistent warp-specialised with two TMEM accumulators) forced in
    turn, incl. the 192-column tiles and a tile list several times the SM count."""
    with bm._lib.tuning(bm._lib.TUNE_GEMM_KERNEL, kernel):
        for M, N, K in ((12864, 576, 144), (40000, 288, 48), (300, 144, 576), (70000, 48, 288)):
            g = torch.Generator().manual_seed(M + N)
            A = torch.randn(M, K, generator=g).to(torch.bfloat16).cuda()
            B = (torch.randn(N, K, generator=g) / K ** 0.5).to(torch.bfloat16).cuda()
            bias = torch.randn(N, generator=g).cuda()
            out = bm.ops.gemm_nt(A, B, bias=bias, out_dtype=torch.float32)
            ref = A.double() @ B.double().t() + bias.double()
            assert cmp.rel(out, ref) < 1e-5, (kernel, M, N, K)


@pytest.mark.parametrize("M,N1,N2", [(12864, 576, 144), (25728, 288, 48), (12864, 576, 144), (130, 128, 16), (1000, 144, 576),
                                     (64, 64, 64), (201, 200, 41 + 7)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_gemm_tn_weight_gradient(M, N1, N2, dtype):
    """dW = dY^T X (contraction over the B*L rows, MN-major tcgen05 operands, deterministic split) vs fp64."""
    g = torch.Generator().manual_seed(M + N1 + N2)
    A = torch.randn(M, N1, generator=g).to(dtype).cuda()
    B = torch.randn(M, N2, generator=g).to(dtype).cuda()
    out = bm.ops.gemm_tn(A, B)
    assert out.dtype == torch.float32 and out.shape == (N1, N2)
    ref = A.double().t() @ B.double()
    assert cmp.rel(out, ref) < 1e-5
    assert torch.equal(out, bm.ops.gemm_tn(A, B))


@pytest.mark.parametrize("T", [1, 7, 201, 499])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_head_forward_fused(T, dtype):
    """norm_f -> attention pooling -> classifier in one launch (DualStreamSEMamba.py:759-767, eval) vs fp64."""
    g = torch.Generator().manual_seed(T)
    Bsz, C = 5, 144
    x = (torch.randn(Bsz, T, C, generator=g) * 2 + 0.3).to(dtype)
    gw, gb = 1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    aw, ab = torch.randn(1, C, generator=g) * 0.3, torch.randn(1, generator=g)
    cw, cb = torch.randn(2, C, generator=g) * 0.1, torch.randn(2, generator=g)
    xd = x.double()
    y = torch.nn.functional.layer_norm(xd, (C,), gw.double(), gb.double(), 1e-5)
    a = torch.softmax(y @ aw.double().t() + ab.double(), dim=1)
    feats_ref = (a.transpose(1, 2) @ y).squeeze(1)
    logits_ref = feats_ref @ cw.double().t() + cb.double()
    feats, logits = bm.ops.head_fwd(x.cuda(), gw.cuda(), gb.cuda(), aw.cuda(), ab.cuda(), cw.cuda(), cb.cuda(), 1e-5)
    assert feats.dtype == torch.float32 and logits.shape == (Bsz, 2)
    cmp.check("feats", feats, feats_ref, 1e-5, cmp.UTT)
    cmp.check("logits", logits, logits_ref, 1e-5, cmp.UTT)


def test_scan_long_backward_against_oracle_on_gpu():
    """Config 5 is 'fwd and bwd' up to L = 8192: every gradient of the scan at L = 8192 against the fp64 oracle (its
    python loop under autograd, run on the GPU), fp32 I/O 1e-4 and bf16 I/O 2e-2."""
    for dtype in (torch.float32, torch.bfloat16):
        u, delta, z, Bm, Cm, A, Dp, bias = _scan_inputs(1, 48, 8192, seed=13, dtype=dtype)
        names = ["u", "delta", "A", "B", "C", "D", "z", "bias"]
        cpu = [u, delta, A, Bm, Cm, Dp, z, bias]
        ref_in = [t.double().cuda().requires_grad_(True) for t in cpu]
        ref = orc.selective_scan_ref(*ref_in, delta_softplus=True)
        g = torch.Generator().manual_seed(14)
        cot = torch.randn(ref.shape, generator=g).to(dtype).cuda()
        (ref * cot.double()).sum().backward()
        dev_in = [t.cuda().requires_grad_(True) for t in cpu]
        out = bm.selective_scan_fn(*dev_in, delta_softplus=True)
        out.backward(cot)
        tag = f"{str(dtype)[6:]} "
        cmp.check(tag + "out", out, ref, TOL[dtype], SLICES["out"])
        for n, a, b in zip(names, dev_in, ref_in):
            cmp.check(tag + "d" + n, a.grad, b.grad, TOL[dtype], SLICES["d" + n])


def test_gelu_kernels():
    g = torch.Generator().manual_seed(1)
    for dtype, tol in ((torch.float32, 1e-6), (torch.bfloat16, 1e-2)):
        x = (3 * torch.randn(1000, 577, generator=g)).to(dtype).cuda()
        dy = torch.randn(1000, 577, generator=g).to(dtype).cuda()
        xr = x.double().requires_grad_(True)
        yr = torch.nn.functional.gelu(xr)
        yr.backward(dy.double())
        assert cmp.rel(bm.ops.gelu_fwd(x), yr) < tol
        assert cmp.rel(bm.ops.gelu_bwd(dy, x), xr.grad) < tol


@pytest.mark.parametrize("C_", [1024, 64, 300])
def test_layernorm_wide_rows(C_):
    """LayerNorm forward / backward on the fusion block's widths (1024 = WavLM features, 64 = SincNet features)."""
    g = torch.Generator().manual_seed(C_)
    x = torch.randn(3, 57, C_, generator=g)
    w = 1 + 0.1 * torch.randn(C_, generator=g)
    b = 0.1 * torch.randn(C_, generator=g)
    cot = torch.randn(3, 57, C_, generator=g)
    ref_in = [t.double().requires_grad_(True) for t in (x, w, b)]
    ref = torch.nn.functional.layer_norm(ref_in[0], (C_,), ref_in[1], ref_in[2], 1e-5)
    ref.backward(cot.double())
    dev_in = [t.cuda().requires_grad_(True) for t in (x, w, b)]
    out = bm.ops.layer_norm_fn(*dev_in, 1e-5)
    out.backward(cot.cuda())
    cmp.check("out", out, ref, 1e-5, cmp.frames())
    for n, a, r in zip(("dx", "weight", "bias"), dev_in, ref_in):
        cmp.check(n, a.grad, r.grad, 1e-5, cmp.frames() if n == "dx" else cmp.CHANNELS)


def test_fp32_products_on_the_tensor_cores():
    """fp32 operands take the three-term bf16 split (bimamba_split3_bf16) and the same tcgen05 kernels: fp32-level accuracy
    against fp64 for the forward / data-gradient product (blocks along K) and the weight-gradient product (blocks along
    the contracted rows), with bias, an addend and a strided output."""
    g = torch.Generator().manual_seed(11)
    for M, N, K in ((12864, 576, 144), (515, 48, 288), (300, 144, 1024), (58, 144, 64)):
        A = torch.randn(M, K, generator=g).cuda()
        B = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
        bias = torch.randn(N, generator=g).cuda()
        add = torch.randn(M, N, generator=g).cuda()
        out = bm.ops.gemm_nt(A, B, bias=bias, addend=add)
        assert out.dtype == torch.float32
        assert cmp.rel(out, A.double() @ B.double().t() + bias.double() + add.double()) < 2e-5, (M, N, K)   # fp32 accumulation over 6 K terms
    buf = torch.zeros(515, 48, device="cuda")
    A = torch.randn(515, 288, generator=g).cuda()
    W = (torch.randn(16, 288, generator=g) / 17).cuda()
    bm.ops.gemm_nt(A, W, out=buf[:, 32:])
    assert cmp.rel(buf[:, 32:], A.double() @ W.double().t()) < 2e-5 and float(buf[:, :32].abs().max()) == 0.0
    for M, N1, N2 in ((12864, 576, 144), (25728, 288, 48), (130, 128, 16)):
        A = torch.randn(M, N1, generator=g).cuda()
        B = torch.randn(M, N2, generator=g).cuda()
        assert cmp.rel(bm.ops.gemm_tn(A, B), A.double().t() @ B.double()) < 5e-5, (M, N1, N2)   # up to 154 k fp32-accumulated terms


def test_cast_and_mean_square_loss_kernels():
    g = torch.Generator().manual_seed(2)
    for n in (12864 * 144, 1001, 7):
        x = torch.randn(n, generator=g).cuda()
        xb = bm.ops.cast(x, torch.bfloat16)
        assert xb.dtype == torch.bfloat16 and torch.equal(xb, x.to(torch.bfloat16))
        assert torch.equal(bm.ops.cast(xb, torch.float32), xb.float())
    for dtype, tol in ((torch.float32, 1e-6), (torch.bfloat16, 1e-6)):
        x = torch.randn(64, 201, 144, generator=g).to(dtype).cuda().requires_grad_(True)
        loss = bm.ops.mean_square_loss(x)
        ref_in = x.detach().double().requires_grad_(True)
        ref = ref_in.square().mean()
        assert loss.dtype == torch.float32 and loss.ndim == 0 and cmp.rel(loss, ref) < tol
        (3.0 * loss).backward()
        (3.0 * ref).backward()
        assert cmp.rel(x.grad, ref_in.grad) < (1e-6 if dtype == torch.float32 else 1e-2)


@pytest.mark.parametrize("nseg", [2, 3, 5])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scan_forward_time_split(nseg, dtype):
    """The time-parallel forward (carry pass over the segments, then the output pass from the combined carries;
    bimamba_selective_scan_fwd_split) forced at small sizes through bimamba_set_tuning: the output and - through the
    checkpoints and the ungated y it writes - every gradient against the fp64 oracle, on ragged lengths and channel
    counts and with every optional operand absent."""
    with bm._lib.tuning(bm._lib.TUNE_SCAN_SPLIT, nseg):
        for L, D in ((201, 288), (37, 40), (499, 17), (1024, 24)):
            assert bm._lib.scan_split_plan(2, 1, L, D, bm._lib.F32)[0] >= 2
            _run_both(2, D, L, dtype, seed=L + D)
        _run_both(2, 40, 77, dtype, with_z=False, with_D=False, with_bias=False, softplus=False, seed=5)


def test_scan_time_split_is_automatic_at_long_lengths_and_matches_the_serial_walk():
    """L = 8192 at a small batch with 16-bit I/O (config 5's last point) takes the time-parallel path by itself; the
    Phase-6 training shape and fp32 I/O never do.  Split against the serial walk of the same kernel family (knob = 1):
    rounding only; both against the fp64 oracle."""
    assert bm._lib.scan_split_plan(64, 1, 8192, 288, bm._lib.BF16) == (3, 2736)
    assert bm._lib.scan_split_plan(64, 1, 8192, 288, bm._lib.F32)[0] == 1
    assert bm._lib.scan_split_plan(64, 2, 201, 288, bm._lib.BF16)[0] == 1
    assert bm._lib.scan_split_plan(2048, 1, 256, 288, bm._lib.BF16)[0] == 1
    for dtype, tol_pair in ((torch.bfloat16, 1e-2), (torch.float32, 1e-4)):
        u, delta, z, Bm, Cm, A, Dp, bias = _scan_inputs(3, 72, 8192, seed=21, dtype=dtype)
        dev = [t.cuda() for t in (u, delta, A, Bm, Cm, Dp, z, bias)]
        auto = bm._lib.scan_split_plan(3, 1, 8192, 72, bm._lib.BF16 if dtype == torch.bfloat16 else bm._lib.F32)[0]
        assert auto == (8 if dtype == torch.bfloat16 else 1)
        with torch.no_grad():
            with bm._lib.tuning(bm._lib.TUNE_SCAN_SPLIT, 0 if dtype == torch.bfloat16 else 8):
                out_split = bm.selective_scan_fn(*dev, delta_softplus=True)
            with bm._lib.tuning(bm._lib.TUNE_SCAN_SPLIT, 1):
                out_serial = bm.selective_scan_fn(*dev, delta_softplus=True)
        assert cmp.rel(out_split, out_serial) < tol_pair
        ref = orc.selective_scan_ref(*[t.double() for t in dev], delta_softplus=True)
        cmp.check("split out", out_split, ref, TOL[dtype], SLICES["out"])
        cmp.check("serial out", out_serial, ref, TOL[dtype], SLICES["out"])
