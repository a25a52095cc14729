"""The tcgen05 GEMMs (csrc/gemm.cu) bit for bit, in every configuration the dispatcher can produce.

gemm_nt has two kernels (one tile per CTA; persistent with two TMEM accumulators), two epilogues (staged through
shared memory with 16-byte stores; unstaged, per element, for a ragged N or a misaligned output), a tile-width cost
function, a tuned-shape table and a fallback from the persistent kernel to the one-tile kernel.  gemm_tn has two
operand orientations, 1-4 Q boxes per block and a deterministic split of the contraction.

The oracle is exact integer arithmetic.  Operands are small integers (|a| <= 16 for gemm_nt with K <= 1024, |a| <= 8
for gemm_tn), so every product is exact in fp32 and every partial sum is an integer below 2^24: the tensor core's
accumulation is exact whatever its internal order.  Bias is integer-valued fp32, an addend integer-valued in the
output type.  The expected output is the fp64 product converted to fp32, or for a 16-bit output rounded by torch
(round to nearest even, as __float2bfloat16_rn / __float2half_rn); with an addend the rounded product plus the addend,
rounded again - the Linear output, then `+ residual`.  Outputs are compared with torch.equal on their bits.  Typical
|c| is in the hundreds to thousands, so 16-bit outputs do need rounding and the rounding itself is under test.

Guard bands: operands are windows of NaN-filled buffers (columns past K, rows past M / N), so a read outside them
turns the result NaN; outputs are windows of buffers filled with a sentinel bit pattern, which must survive outside
the window.

The fp32 split path (three bf16 terms per fp32 value, six K blocks) is not exact; it is checked element by element
against |c - ref| <= TAU * 2^-24 * sqrt(6 K) * sum_k |a_ik| |b_jk|.
"""
import math

import pytest
import torch

import bimamba_b200 as bm

pytestmark = pytest.mark.gpu

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
ONE_TILE_WIDTHS = tuple(range(16, 209, 16))    # gemm_nt_kernel: every width the automatic rule or the fallback produces
PERSIST_WIDTHS = tuple(range(16, 193, 16))     # gemm_nt_persist_kernel: two accumulators fit 512 TMEM columns
KS = (8, 56, 64, 72, 144, 288, 576, 1024)
MS = (1, 127, 128, 129, 3 * 128 + 5)
SMS = 148
SENTINEL = {2: 0x7E5B, 4: 0x7FA5A5A5}          # by element size; never a value the products produce
# fp32 split path: the worst ratio the fp32 tests print was 0.74 (gemm_nt, K = 576) on a B200 at its 1000 W limit
TAU = 2.0


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _ints(shape, lim, g):
    return torch.randint(-lim, lim + 1, shape, generator=g, device="cuda", dtype=F32)


def _bits(t):
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16)


def _assert_bits(got, exp, what):
    """Bitwise equality of two same-shaped 2-D tensors, except that -0 equals +0 (a sum of a single -0 product is -0 in
    the fp64 reference, +0 from an accumulator that starts at +0); on failure name how many elements differ and the
    first one."""
    neg0 = -(1 << (8 * got.element_size() - 1))
    gb, eb = _bits(got), _bits(exp)
    gb, eb = gb.masked_fill(gb == neg0, 0), eb.masked_fill(eb == neg0, 0)
    if torch.equal(gb, eb):
        return
    bad = (gb != eb).nonzero()
    r, c = bad[0].tolist()
    mask = (1 << (8 * got.element_size())) - 1
    raise AssertionError(f"{what}: {bad.shape[0]} of {got.numel()} elements differ; first at ({r}, {c}): "
                         f"got {float(got[r, c])} (0x{int(gb[r, c]) & mask:x}), "
                         f"expected {float(exp[r, c])} (0x{int(eb[r, c]) & mask:x})")


def _guarded_operand(rows, cols, dtype, vals):
    """`vals` (rows, cols) as the top-left window of a NaN-filled buffer: row stride cols + 16, three rows below."""
    buf = torch.full((rows + 3, cols + 16), float("nan"), device="cuda", dtype=dtype)
    buf[:rows, :cols] = vals.to(dtype)
    return buf[:rows, :cols]


def _expected_nt(A, B, bias, addend, out_dtype):
    acc = A.double() @ B.double().t()
    if bias is not None:
        acc = acc + bias.double()
    if out_dtype == F32:
        return (acc + addend.double() if addend is not None else acc).float()
    c = acc.float().to(out_dtype)                                  # the Linear output in the output type
    if addend is not None:
        c = (c.float() + addend.float()).to(out_dtype)             # then + addend, rounded again
    return c


def _window(layout, M, N, osz):
    """-> (guard rows, column offset, row stride) of the output window inside its buffer."""
    if layout == "plain":
        return 0, 0, N
    co = 16 // osz if layout == "guarded" else 1                  # "misaligned": breaks 16-byte alignment
    return 2, co, (co + N + 8 + 7) // 8 * 8


def _run_nt(A, B, out_dtype, bias, addend_vals, window):
    """gemm_nt into an output window of a sentinel-filled buffer; -> (buffer, window, addend window)."""
    M, N = A.shape[0], B.shape[0]
    gr, co, ldc = window
    osz = 4 if out_dtype == F32 else 2
    buf = torch.full((M + 2 * gr, ldc), SENTINEL[osz], device="cuda",
                     dtype=torch.int32 if osz == 4 else torch.int16).view(out_dtype)
    C = buf[gr:gr + M, co:co + N]
    add = None
    if addend_vals is not None:                                    # same layout as C; NaN outside the window
        abuf = torch.full_like(buf, float("nan"))
        add = abuf[gr:gr + M, co:co + N]
        add.copy_(addend_vals.to(out_dtype))
    before = bm._lib.launch_count
    bm.ops.gemm_nt(A, B, bias=bias, addend=add, out=C)
    assert bm._lib.launch_count == before + 1                      # one native launch, not the framework product
    return buf, C, add


def _check_nt(g, M, N, K, in_dt, out_dt, use_bias, use_add, layout="guarded", repeat=False):
    osz = 4 if out_dt == F32 else 2
    A = _guarded_operand(M, K, in_dt, _ints((M, K), 16, g))
    B = _guarded_operand(N, K, in_dt, _ints((N, K), 16, g))
    bias = None
    if use_bias:                                                   # NaN past N
        bbuf = torch.full((N + 16,), float("nan"), device="cuda")
        bias = bbuf[:N]
        bias.copy_(_ints((N,), 64, g))
    add_vals = _ints((M, N), 512, g) if use_add else None
    window = _window(layout, M, N, osz)
    buf, C, add = _run_nt(A, B, out_dt, bias, add_vals, window)
    gr, co, _ = window
    exp = torch.full_like(_bits(buf), SENTINEL[osz]).view(out_dt)
    exp[gr:gr + M, co:co + N] = _expected_nt(A, B, bias, add, out_dt)
    what = f"M={M} N={N} K={K} {in_dt}->{out_dt} bias={use_bias} addend={use_add} {layout}"
    _assert_bits(buf, exp, what)
    if repeat:
        buf2, _, _ = _run_nt(A, B, out_dt, bias, add_vals, window)
        _assert_bits(buf2, buf, what + " (repeat)")


def _n_variants(width):
    # a full tile; a ragged last tile (multiple of 8: staged); inside one tile and past one tile with N not a multiple
    # of 4 (unstaged epilogue for every output type)
    return (width, 2 * width - 8, width - 3, width + 5)


# ------------------------------------------------------------------------------------------------ gemm_nt sweep
@pytest.mark.parametrize("kernel,width", [(1, w) for w in ONE_TILE_WIDTHS] + [(2, w) for w in PERSIST_WIDTHS])
def test_gemm_nt_every_tile_width_bit_exact(kernel, width):
    """Both kernels forced (TUNE_GEMM_KERNEL) at every tile width (TUNE_GEMM_BN), stage count left to the code:
    inputs {bf16, fp16} x outputs {same, fp32} x epilogue {none, bias, addend, bias + addend}, each on four N (full
    tile, ragged last tile, N % 4 != 0 inside and past one tile) with M and K cycling through their edge values; the
    combinations with bias and addend on a full tile also write a misaligned output window.  Then a tile list with
    four to five tiles per CTA of the persistent kernel, so that both TMEM accumulators wrap their phase.  (With
    kernel 2 the fp32 outputs of widths above 144 and every unstageable N run on the one-tile kernel: the fallback.)"""
    g = _gen(1000 * kernel + width)
    with bm._lib.tuning(bm._lib.TUNE_GEMM_KERNEL, kernel), bm._lib.tuning(bm._lib.TUNE_GEMM_BN, width):
        i = 0
        for in_dt in (BF16, F16):
            for out_dt in (in_dt, F32):
                for use_bias, use_add in ((False, False), (True, False), (False, True), (True, True)):
                    for nv, N in enumerate(_n_variants(width)):
                        M = MS[i % len(MS)]
                        K = KS[(i + i // 4 + width // 16) % len(KS)]
                        layout = "misaligned" if (nv == 0 and use_bias and use_add) else "guarded"
                        _check_nt(g, M, N, K, in_dt, out_dt, use_bias, use_add, layout)
                        i += 1
        M = 4 * SMS * 128 + 77
        for in_dt, out_dt in ((BF16, BF16), (F16, F32)):
            _check_nt(g, M, width, 144, in_dt, out_dt, True, True, repeat=True)


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("dtype,base", [(BF16, 256), (F16, 2048)])
def test_gemm_nt_addend_rounds_the_product_first_on_both_epilogues(kernel, dtype, base):
    """Every product is base + 1, a tie halfway between base and base + 2 in the output type, and the addend is 1.
    Rounding the product first (the Linear output, then + residual) gives base, and base + 1 rounds to base again;
    adding first would give base + 2.  The staged epilogue (N a multiple of 8, aligned output) and the unstaged one
    (ragged N, or a misaligned output window) must give the same bits."""
    M, K = 129, 64
    s = 16 if dtype == BF16 else 32                                # base = s * (base / s), both exact in dtype
    A = torch.zeros(M, K, device="cuda", dtype=dtype)
    A[:, 0], A[:, 5] = s, 1
    with bm._lib.tuning(bm._lib.TUNE_GEMM_KERNEL, kernel):
        for N, layout in ((16, "guarded"), (13, "guarded"), (16, "misaligned"), (40, "plain"), (45, "plain")):
            B = torch.zeros(N, K, device="cuda", dtype=dtype)
            B[:, 0], B[:, 5] = base // s, 1
            buf, C, _ = _run_nt(A, B, dtype, None, torch.ones(M, N, device="cuda"), _window(layout, M, N, 2))
            exp = torch.full((M, N), base, device="cuda", dtype=dtype)
            assert torch.equal(_bits(C), _bits(exp)), \
                f"N={N} {layout}: got {sorted(set(C.float().flatten().tolist()))}, expected [{float(base)}]"


# Production shapes at the benchmark's row counts (batch 64 x 201 frames, x2 directions for the x_proj rows), with no
# knob set: the tuned table and the automatic choice run as shipped.  (name, M, N, K, bias, addend, fp32 output)
PRODUCTION = [
    ("in_proj", 12864, 576, 144, False, False, False),
    ("ffn_up", 12864, 576, 144, True, False, False),
    ("out_proj_ffn_down", 12864, 144, 576, True, True, True),    # fp32 residual stream: fp32 output and addend
    ("in_proj_data_grad", 12864, 144, 576, False, False, False),
    ("x_proj", 25728, 48, 288, False, False, False),
    ("x_proj_data_grad", 25728, 288, 48, False, True, False),    # + du
]


@pytest.mark.parametrize("dtype", [BF16, F16])
@pytest.mark.parametrize("name,M,N,K,use_bias,use_add,f32_out", PRODUCTION, ids=[p[0] for p in PRODUCTION])
def test_gemm_nt_production_shapes_bit_exact(name, M, N, K, use_bias, use_add, f32_out, dtype):
    """The block's and the feed-forward's products through ops.gemm_nt exactly as the training step calls them."""
    g = _gen(M + N + K)
    assert all(bm._lib.load().bimamba_get_tuning(k) == 0 for k in (bm._lib.TUNE_GEMM_KERNEL, bm._lib.TUNE_GEMM_BN,
                                                                    bm._lib.TUNE_GEMM_STAGES))
    A = _ints((M, K), 16, g).to(dtype)
    B = _ints((N, K), 16, g).to(dtype)
    bias = _ints((N,), 64, g) if use_bias else None
    out_dt = F32 if f32_out else dtype
    add = _ints((M, N), 512, g).to(out_dt) if use_add else None
    out = bm.ops.gemm_nt(A, B, bias=bias, addend=add, out_dtype=out_dt)
    _assert_bits(out, _expected_nt(A, B, bias, add, out_dt), name)
    _assert_bits(bm.ops.gemm_nt(A, B, bias=bias, addend=add, out_dtype=out_dt), out, name + " (repeat)")


@pytest.mark.parametrize("dtype", [BF16, F16])
def test_gemm_nt_dt_slice_into_dxdbl_bit_exact(dtype):
    """The dt_proj data gradient written next to dB | dC: dxdbl[:, 32:] (ldc 48) of the x_proj rows; columns 0..31
    keep their bits."""
    g = _gen(7)
    M, K = 25728, 288
    A = _ints((M, K), 16, g).to(dtype)
    W = _ints((16, K), 16, g).to(dtype)
    buf, C, _ = _run_nt(A, W, dtype, None, None, (0, 32, 48))
    exp = torch.full((M, 48), SENTINEL[2], device="cuda", dtype=torch.int16).view(dtype)
    exp[:, 32:] = _expected_nt(A, W, None, None, dtype)
    _assert_bits(buf, exp, "dt slice")


def test_gemm_nt_automatic_widths_are_all_swept():
    """Every tile width the automatic rule picks for N in 1..1024 is one that test_gemm_nt_every_tile_width_bit_exact
    forces (the tuned table's widths 32, 64, 128 and persistent 144 are among them too); if the cost function
    changes, the sweep must follow."""
    lib = bm._lib.load()
    auto = {lib.bimamba_gemm_nt_block_n_k(n, k) for n in range(1, 1025) for k in KS}
    assert auto <= set(ONE_TILE_WIDTHS), sorted(auto - set(ONE_TILE_WIDTHS))


# ------------------------------------------------------------------------------------------------ gemm_tn sweep
# (M, N1, N2, splits): which operand takes the TMEM lanes, Q boxes per block and P tiles in the comments
TN_CASES = [
    (1, 200, 328, 1),          # B on the lanes (3 P tiles), 4 Q boxes (block 208 for 200 columns), one row
    (63, 328, 200, 1),         # A on the lanes, 4 Q boxes
    (64, 48, 16, 1),           # 1 Q box, exactly one 64-row block
    (65, 576, 144, 2),         # A on the lanes, 3 Q boxes, second split of one row
    (201, 128, 72, 4),         # 2 Q boxes (block 80 for 72 columns)
    (201, 200, 328, 4),        # B on the lanes, ragged P and Q widths
    (1000, 144, 576, 16),      # B on the lanes, 5 P tiles
    (12864, 576, 144, 29),     # A on the lanes; 7 row blocks per split, the last split 5
    (25728, 288, 48, 45),      # 9 row blocks per split, the last 6
    (70001, 576, 576, 9),      # the longest splits: 122 row blocks (7808 rows) each, the last 118
    (70001, 200, 328, 48),
]


@pytest.mark.parametrize("M,N1,N2,splits", TN_CASES)
@pytest.mark.parametrize("dtype", [BF16, F16])
def test_gemm_tn_bit_exact(M, N1, N2, splits, dtype):
    """dW = A^T B against the exact integer product.  A and B are the first M rows and N1 / N2 columns of NaN-filled
    buffers, so a read past M (or past a feature width) poisons the sum."""
    lib = bm._lib.load()
    assert lib.bimamba_gemm_tn_splits(M, N1, N2) == splits
    g = _gen(M + N1 + N2)
    A = _guarded_operand(M, N1, dtype, _ints((M, N1), 8, g))
    B = _guarded_operand(M, N2, dtype, _ints((M, N2), 8, g))
    before = bm._lib.launch_count
    out = bm.ops.gemm_tn(A, B)
    assert bm._lib.launch_count == before + 2                      # partial products + fixed-order split sum
    assert out.dtype == F32 and out.shape == (N1, N2)
    _assert_bits(out, (A.double().t() @ B.double()).float(), f"gemm_tn M={M} N1={N1} N2={N2}")
    _assert_bits(bm.ops.gemm_tn(A, B), out, "gemm_tn repeat")


# ------------------------------------------------------------------------------------------------ fp32 split path
@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("stack_rows", [False, True])
def test_split3_terms_and_block_order(side, stack_rows):
    """bimamba_split3_bf16 as gemm_nt (blocks along the columns) and gemm_tn (blocks along the rows) call it: each
    element of x splits into bf16 terms hi, mid, lo with hi + mid + lo == x exactly, laid out in the six blocks
    [hi|mid|lo|hi|hi|mid] (side 0) or [hi|hi|hi|mid|lo|mid] (side 1)."""
    rows, cols = 301, 40
    g = _gen(17 + side + 2 * stack_rows)
    mant = torch.randint(0, 1 << 23, (rows, cols), generator=g, device="cuda").double()
    expo = torch.randint(-100, 101, (rows, cols), generator=g, device="cuda")
    sign = torch.randint(0, 2, (rows, cols), generator=g, device="cuda").double() * 2 - 1
    x = (sign * torch.ldexp(1 + mant / (1 << 23), expo.double())).float()   # full 24-bit significands, |x| in [2^-100, 2^101)
    x[0, :8] = torch.tensor([1.0, -1.0, 2.0 ** -100, -2.0 ** 100, 257.0, 1 + 2.0 ** -23, -(1 + 2.0 ** -9), 3.0])
    src = torch.full((rows, cols + 24), float("nan"), device="cuda")  # ld_src > cols
    src[:, :cols] = x
    before = bm._lib.launch_count
    dst = bm.ops._split3(src[:, :cols], side, stack_rows)
    assert bm._lib.launch_count == before + 1 and dst.dtype == BF16
    blocks = dst.view(6, rows, cols) if stack_rows else dst.view(rows, 6, cols).transpose(0, 1)
    hi = x.to(BF16)
    r1 = x - hi.float()
    mid = r1.to(BF16)
    lo = (r1 - mid.float()).to(BF16)
    total = hi.double() + mid.double() + lo.double()
    assert torch.equal(total, x.double())
    both = (mid != 0) & (lo != 0)
    assert int(both.sum()) > rows * cols // 2                      # the mid and lo terms are exercised
    order = (hi, mid, lo, hi, hi, mid) if side == 0 else (hi, hi, hi, mid, lo, mid)
    for b, term in enumerate(order):
        _assert_bits(blocks[b], term, f"split3 side {side} block {b}")


def _ratio(out, ref, scale, depth):
    """Largest |out - ref| in units of 2^-24 sqrt(depth) sum |a||b| (element by element)."""
    bound = 2.0 ** -24 * math.sqrt(depth) * scale
    return float(((out.double() - ref).abs() / bound).max())


@pytest.mark.parametrize("M,N,K,co", [(515, 100, 200, 4), (129, 52, 1000, 4), (1, 148, 36, 1), (12864, 144, 576, 4)])
def test_fp32_gemm_nt_elementwise(M, N, K, co):
    """fp32 operands through the three-term bf16 split on the tcgen05 kernel: bias, an fp32 addend and a strided
    output window (16-byte aligned, or misaligned by one element), each element within TAU of the accumulation
    bound; the window's surroundings unchanged; a repeat gives the same bits."""
    g = _gen(M + N + K)
    A = torch.randn(M, K, generator=g, device="cuda")
    B = torch.randn(N, K, generator=g, device="cuda") / K ** 0.5
    bias = torch.randn(N, generator=g, device="cuda")
    ldc = (co + N + 8 + 7) // 8 * 8
    abuf = torch.full((M + 4, ldc), float("nan"), device="cuda")
    add = abuf[2:2 + M, co:co + N]
    add.copy_(torch.randn(M, N, generator=g, device="cuda"))
    ref = A.double() @ B.double().t() + bias.double() + add.double()
    scale = A.double().abs() @ B.double().abs().t() + bias.double().abs() + add.double().abs()
    outs = []
    for _ in range(2):
        buf = torch.full((M + 4, ldc), SENTINEL[4], device="cuda", dtype=torch.int32).view(F32)
        before = bm._lib.launch_count
        bm.ops.gemm_nt(A, B, bias=bias, addend=add, out=buf[2:2 + M, co:co + N])
        assert bm._lib.launch_count == before + 3                  # two splits + one GEMM
        outside = torch.ones_like(buf, dtype=torch.bool)
        outside[2:2 + M, co:co + N] = False
        assert bool((_bits(buf)[outside] == SENTINEL[4]).all())
        outs.append(buf)
    r = _ratio(outs[0][2:2 + M, co:co + N], ref, scale, 6 * K)
    print(f"fp32 gemm_nt M={M} N={N} K={K}: worst error / (2^-24 sqrt(6K) sum|a||b|) = {r:.3f}")
    assert r <= TAU, r
    _assert_bits(outs[1], outs[0], "fp32 gemm_nt repeat")


@pytest.mark.parametrize("M,N1,N2", [(1000, 144, 576), (12864, 576, 144), (201, 200, 328), (65, 48, 16)])
def test_fp32_gemm_tn_elementwise(M, N1, N2):
    """fp32 weight-gradient products through the split (six blocks stacked along the contracted rows)."""
    g = _gen(M + N1 + N2)
    A = torch.randn(M, N1, generator=g, device="cuda")
    B = torch.randn(M, N2, generator=g, device="cuda")
    before = bm._lib.launch_count
    out = bm.ops.gemm_tn(A, B)
    assert bm._lib.launch_count == before + 4                      # two splits + partial products + split sum
    r = _ratio(out, A.double().t() @ B.double(), A.double().abs().t() @ B.double().abs(), 6 * M)
    print(f"fp32 gemm_tn M={M} N1={N1} N2={N2}: worst error / (2^-24 sqrt(6M) sum|a||b|) = {r:.3f}")
    assert r <= TAU, r
    _assert_bits(bm.ops.gemm_tn(A, B), out, "fp32 gemm_tn repeat")
