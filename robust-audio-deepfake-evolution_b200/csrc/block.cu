// The Mamba block of one encoder layer as ONE call each way, for hosts without an autograd framework (SURVEY 8b: the
// `conv_scan_bi` entry together with gemm_{in,x,out}_proj and their dgrad / wgrad).  Host code only: it sequences this
// library's kernels on the caller's stream in the order robust-audio-deepfake-evolution_b200/ops.py: BiMambaInnerFn
// does, carving the activations it keeps for the backward out of a caller-allocated workspace.
//
//   forward  (mamba_block.py:41-63 for both directions of DualStreamSEMamba.py:473-481):
//     xz = x Wi^T -> xc = silu(conv(x half)) for dir 0 / dir 1 -> [B | C | dt_r] = xc Wxp^T -> y = scan(xc, ., z) ->
//     out = [y_fwd | y_rev] [W_out | W_out]^T                                       5 launches
//   backward (autograd of the above): dy -> scan backward -> group sum of dB|dC -> dt_proj / x_proj data gradients ->
//     conv backward -> in_proj data gradient, the four weight-gradient products, the fixed-order parameter sums and the
//     layout pass to the reference's parameter shapes.
// Everything is deterministic (fixed-order reductions), never allocates, never synchronises.
#include "common.cuh"

namespace bimamba {

static inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

struct FwdCarve {
  size_t xz, xc, xdbl, y, ckpt, ypre, total;
  int nck;
};

static FwdCarve carve_fwd(int64_t B, int64_t L, int D, int ndir, int es, bool save) {
  FwdCarve c{};
  const size_t M = (size_t)B * L;
  size_t off = 0;
  c.xz = off;   off += up256(M * 2 * D * es);
  c.xc = off;   off += up256(M * ndir * D * es);
  c.xdbl = off; off += up256(M * ndir * kXW * es);
  c.y = off;    off += up256(M * ndir * D * es);
  c.nck = L > 0 ? (int)((L + BIMAMBA_CKPT - 1) / BIMAMBA_CKPT) : 1;
  c.ckpt = off;
  if (save && c.nck > 1) off += up256((size_t)B * ndir * c.nck * D * kN * 4);
  c.ypre = off;
  if (save) off += up256(M * ndir * D * es);
  c.total = off;
  return c;
}

struct BwdCarve {
  size_t dy, du, ddelta, dz, dxdbl, dxc, dxz, dbc_part, dA_part, dD_part, db_part, dA, conv_part, dwb, tn_part, dWo2,
      dWdtf, dWxp, total;
  int ngroups, conv_slices;
};

static BwdCarve carve_bwd(int64_t B, int64_t L, int dm, int D, int K, int ndir, int es) {
  BwdCarve c{};
  const size_t M = (size_t)B * L;
  int G = 0, ng = 0;
  bimamba_scan_plan((int)L, D, (int)(B * ndir), 1, &G, &ng);
  c.ngroups = ng;
  c.conv_slices = bimamba_conv_bwd_slices((int)B, (int)L, D);
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += up256(bytes); return o; };
  c.dy = take(M * D * es);
  c.du = take(M * ndir * D * es);
  c.ddelta = take(M * ndir * D * es);
  c.dz = take(M * ndir * D * es);
  c.dxdbl = take(M * ndir * kXW * es);
  c.dxc = take(M * ndir * D * es);
  c.dxz = take(M * 2 * D * es);
  c.dbc_part = take((size_t)B * ng * L * ndir * 2 * kN * 4);
  c.dA_part = take((size_t)B * ndir * D * kN * 4);
  c.dD_part = take((size_t)B * ndir * D * 4);
  c.db_part = take((size_t)B * ndir * D * 4);
  c.dA = take((size_t)D * kN * 4);
  c.conv_part = take((size_t)(c.conv_slices > 0 ? c.conv_slices : 1) * D * (K + 1) * 4);
  c.dwb = take((size_t)D * (K + 1) * 4);
  size_t tn = 0;   // the four weight-gradient products run one after the other on the stream: one partial buffer
  auto tn_need = [&](int64_t rows, int n1, int n2) {
    const size_t b = (size_t)bimamba_gemm_tn_splits(rows, n1, n2) * n1 * n2 * 4;
    if (b > tn) tn = b;
  };
  tn_need((int64_t)M, dm, ndir * D);
  tn_need((int64_t)M * ndir, D, kXW);
  tn_need((int64_t)M * ndir, kXW, D);
  tn_need((int64_t)M, 2 * D, dm);
  c.tn_part = take(tn);
  c.dWo2 = take((size_t)dm * ndir * D * 4);
  c.dWdtf = take((size_t)D * kXW * 4);
  c.dWxp = take((size_t)kXW * D * 4);
  c.total = off;
  return c;
}

static int check_block(const bimamba_block_desc* d) {
  if (!d) { set_err("block: null descriptor"); return -1; }
  if (d->batch < 0 || d->seqlen < 0 || d->d_model < 1 || d->d_inner < 1) { set_err("block: bad sizes"); return -3; }
  if (d->ndir < 1 || d->ndir > 2) { set_err("block: ndir must be 1 or 2"); return -3; }
  if (d->dt_rank < 1 || d->dt_rank > BIMAMBA_MAX_DT_RANK) { set_err("block: dt_rank must be 1..16"); return -4; }
  if (d->d_conv < 2 || d->d_conv > 4) { set_err("block: d_conv must be 2..4"); return -4; }
  if (d->io_dtype != BIMAMBA_BF16 && d->io_dtype != BIMAMBA_F16) {
    set_err("block: activations must be bf16 or fp16 (fp32 goes through bimamba_split3_bf16 + the op-level entries)");
    return -6;
  }
  if ((d->d_model & 7) || (d->d_inner & 7)) { set_err("block: d_model and d_inner must be multiples of 8"); return -7; }
  if (!d->x || !d->out || !d->Wi || !d->Wxp || !d->Wo2 || !d->Wdt || !d->A || !d->conv_w) {
    set_err("block: null operand");
    return -7;
  }
  if ((reinterpret_cast<uintptr_t>(d->workspace) & 255) != 0) { set_err("block: workspace must be 256-byte aligned"); return -7; }
  return 0;
}

static void fill_scan(bimamba_scan_desc& s, const bimamba_block_desc* d, const FwdCarve& c, unsigned char* ws, int es) {
  const int64_t L = d->seqlen, D = d->d_inner, nd = d->ndir;
  s = bimamba_scan_desc{};
  unsigned char* xz = ws + c.xz;
  s.u = ws + c.xc;
  s.z = xz + (size_t)D * es;                     // the z half of xz, shared by both directions (dir stride 0)
  s.bc = ws + c.xdbl;
  s.dtr = ws + c.xdbl + (size_t)2 * kN * es;
  s.Wdt = d->Wdt; s.A = d->A; s.D = d->D; s.delta_bias = d->dt_bias;
  s.batch = d->batch; s.ndir = d->ndir; s.dim = d->d_inner; s.seqlen = d->seqlen; s.dstate = kN; s.dt_rank = d->dt_rank;
  s.io_dtype = d->io_dtype;
  s.flags = BIMAMBA_FLAG_SOFTPLUS | BIMAMBA_FLAG_DTR_PADDED;   // x_proj writes all 48 columns of every row
  s.u_bs = L * nd * D; s.u_ds = D; s.u_ts = nd * D;
  s.z_bs = L * 2 * D;  s.z_ds = 0; s.z_ts = 2 * D;
  s.bc_bs = L * nd * kXW; s.bc_ds = kXW; s.bc_ts = nd * kXW;
  s.dtr_bs = s.bc_bs; s.dtr_ds = s.bc_ds; s.dtr_ts = s.bc_ts;
  s.out_bs = L * nd * D; s.out_ds = D; s.out_ts = nd * D;
}

}  // namespace bimamba

using namespace bimamba;

extern "C" size_t bimamba_block_fwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int ndir,
                                                    int io_dtype, int save_for_backward) {
  (void)d_model;
  if (batch <= 0 || seqlen <= 0 || d_inner <= 0 || ndir <= 0) return 0;
  return carve_fwd(batch, seqlen, d_inner, ndir, io_dtype == BIMAMBA_F32 ? 4 : 2, save_for_backward != 0).total;
}

extern "C" size_t bimamba_block_bwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int d_conv,
                                                    int ndir, int io_dtype) {
  if (batch <= 0 || seqlen <= 0 || d_inner <= 0 || d_model <= 0 || ndir <= 0 || d_conv <= 0) return 0;
  return carve_bwd(batch, seqlen, d_model, d_inner, d_conv, ndir, io_dtype == BIMAMBA_F32 ? 4 : 2).total;
}

extern "C" int bimamba_block_fwd(const bimamba_block_desc* d, bimamba_stream_t stream) {
  return bimamba_block_fwd_varlen(d, nullptr, stream);
}

// seqlens != NULL: right-padded utterances of different lengths.  The products run on every row (a row of a product
// depends on that row only); the conv and the scan walk each utterance's own frames and write zeros to the padded ones,
// so valid outputs do not depend on what the padding holds.
extern "C" int bimamba_block_fwd_varlen(const bimamba_block_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  if (d && seqlens && d->save_for_backward) {
    set_err("block_fwd_varlen: variable-length batches are forward-only (save_for_backward must be 0)");
    return -9;
  }
  return bimamba_block_fwd_varlen_train(d, seqlens, stream);
}

// The training forward: with save_for_backward the scan also writes its checkpoints (ceil(seqlen / 8) per channel, the
// padded layout) and the ungated y for bimamba_block_bwd_varlen.
extern "C" int bimamba_block_fwd_varlen_train(const bimamba_block_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  int rc = check_block(d);
  if (rc) return rc;
  if (d->batch == 0 || d->seqlen == 0) return 0;
  const int es = 2, dt = d->io_dtype;
  const int64_t B = d->batch, L = d->seqlen, M = B * L;
  const int dm = d->d_model, D = d->d_inner, nd = d->ndir;
  const bool save = d->save_for_backward != 0;
  const FwdCarve c = carve_fwd(B, L, D, nd, es, save);
  if (!d->workspace || d->workspace_bytes < c.total) { set_err("block_fwd: workspace too small (bimamba_block_fwd_workspace_bytes)"); return -10; }
  unsigned char* ws = static_cast<unsigned char*>(d->workspace);
  void *xz = ws + c.xz, *xc = ws + c.xc, *xdbl = ws + c.xdbl, *y = ws + c.y;
  // in_proj (mamba_block.py:48): once for both directions
  rc = bimamba_gemm_nt(d->x, dm, d->Wi, dm, xz, 2 * D, nullptr, nullptr, M, 2 * D, dm, dt, dt, stream);
  if (rc) return rc;
  // causal conv + SiLU of the x half, direction 0 and the flipped direction from one read (:52-55)
  rc = bimamba_causal_conv1d_fwd_varlen(xz, d->conv_w, d->conv_b, xc, seqlens, (int)B, nd, D, (int)L, d->d_conv, L * 2 * D,
                                        2 * D, L * nd * D, D, (int64_t)nd * D, dt, BIMAMBA_FLAG_SILU, stream);
  if (rc) return rc;
  // x_proj against the repacked (48, D) weight: rows [B | C | dt_r | 0] of both directions in one product (:73)
  rc = bimamba_gemm_nt(xc, D, d->Wxp, D, xdbl, kXW, nullptr, nullptr, M * nd, kXW, D, dt, dt, stream);
  if (rc) return rc;
  // dt_proj + softplus + scan + D skip + z gate, both directions in one launch (:80-120, :61)
  bimamba_scan_desc s;
  fill_scan(s, d, c, ws, es);
  s.out = y;
  s.ypre = save ? ws + c.ypre : nullptr;
  s.ckpt = (save && c.nck > 1) ? reinterpret_cast<float*>(ws + c.ckpt) : nullptr;
  int G = 0, ng = 0;
  bimamba_scan_plan((int)L, D, (int)(B * nd), 0, &G, &ng);
  s.group_channels = G;
  rc = bimamba_selective_scan_fwd_varlen_train(&s, seqlens, stream);
  if (rc) return rc;
  // out_proj of the sum of the directions as one product over [y_fwd | y_rev] (:62, DualStreamSEMamba.py:481)
  return bimamba_gemm_nt(y, (int64_t)nd * D, d->Wo2, (int64_t)nd * D, d->out, dm, nullptr, nullptr, M, dm, nd * D, dt, dt, stream);
}

extern "C" int bimamba_block_bwd(const bimamba_block_desc* d, const bimamba_block_grads* g, bimamba_stream_t stream) {
  return bimamba_block_bwd_varlen(d, g, nullptr, stream);
}

// seqlens != NULL: the backward of bimamba_block_fwd_varlen_train (same seqlens).  The scan and the conv walk each
// utterance's own frames and write zero gradients at padded frames, so every product over the rows sees zeros there.
extern "C" int bimamba_block_bwd_varlen(const bimamba_block_desc* d, const bimamba_block_grads* g, const int32_t* seqlens,
                                        bimamba_stream_t stream) {
  int rc = check_block(d);
  if (rc) return rc;
  if (!g) { set_err("block_bwd: null gradient descriptor"); return -1; }
  if (!g->dout || !g->dx || !g->WiT || !g->WxpT || !g->WoT || !g->WdT || !g->dW_in || !g->dconv_w || !g->dconv_b || !g->dW_x ||
      !g->dW_dt || !g->db_dt || !g->dA_log || !g->dD || !g->dW_out) {
    set_err("block_bwd: null operand");
    return -8;
  }
  if (!d->D || !d->dt_bias || !d->conv_b) { set_err("block_bwd: D, dt_bias and conv_b are required"); return -8; }
  if (!d->save_for_backward) { set_err("block_bwd: the forward must run with save_for_backward"); return -9; }
  if ((reinterpret_cast<uintptr_t>(g->workspace) & 255) != 0) { set_err("block_bwd: workspace must be 256-byte aligned"); return -7; }
  const int es = 2, dt = d->io_dtype;
  const int64_t B = d->batch, L = d->seqlen, M = B * L;
  const int dm = d->d_model, D = d->d_inner, nd = d->ndir, R = d->dt_rank, K = d->d_conv;
  if (M == 0) {   // no rows: every parameter gradient is zero
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaMemsetAsync(g->dW_in, 0, (size_t)2 * D * dm * 4, st);
    cudaMemsetAsync(g->dconv_w, 0, (size_t)D * K * 4, st);
    cudaMemsetAsync(g->dconv_b, 0, (size_t)D * 4, st);
    cudaMemsetAsync(g->dW_x, 0, (size_t)(R + 2 * kN) * D * 4, st);
    cudaMemsetAsync(g->dW_dt, 0, (size_t)D * R * 4, st);
    cudaMemsetAsync(g->db_dt, 0, (size_t)D * 4, st);
    cudaMemsetAsync(g->dA_log, 0, (size_t)D * kN * 4, st);
    cudaMemsetAsync(g->dD, 0, (size_t)D * 4, st);
    cudaMemsetAsync(g->dW_out, 0, (size_t)dm * D * 4, st);
    return 0;
  }
  const FwdCarve c = carve_fwd(B, L, D, nd, es, true);
  const BwdCarve w = carve_bwd(B, L, dm, D, K, nd, es);
  if (!d->workspace || d->workspace_bytes < c.total) { set_err("block_bwd: forward workspace too small"); return -10; }
  if (!g->workspace || g->workspace_bytes < w.total) { set_err("block_bwd: workspace too small (bimamba_block_bwd_workspace_bytes)"); return -10; }
  unsigned char* fs = static_cast<unsigned char*>(d->workspace);
  unsigned char* bs = static_cast<unsigned char*>(g->workspace);
  void *xz = fs + c.xz, *xc = fs + c.xc, *xdbl = fs + c.xdbl, *y = fs + c.y;
  void *dy = bs + w.dy, *du = bs + w.du, *ddelta = bs + w.ddelta, *dz = bs + w.dz, *dxdbl = bs + w.dxdbl, *dxc = bs + w.dxc,
       *dxz = bs + w.dxz;
  float *dbc_part = reinterpret_cast<float*>(bs + w.dbc_part), *dA_part = reinterpret_cast<float*>(bs + w.dA_part),
        *dD_part = reinterpret_cast<float*>(bs + w.dD_part), *db_part = reinterpret_cast<float*>(bs + w.db_part),
        *dA = reinterpret_cast<float*>(bs + w.dA), *conv_part = reinterpret_cast<float*>(bs + w.conv_part),
        *dwb = reinterpret_cast<float*>(bs + w.dwb), *tn_part = reinterpret_cast<float*>(bs + w.tn_part),
        *dWo2 = reinterpret_cast<float*>(bs + w.dWo2), *dWdtf = reinterpret_cast<float*>(bs + w.dWdtf),
        *dWxp = reinterpret_cast<float*>(bs + w.dWxp);
#define BIMAMBA_TRY(call) do { rc = (call); if (rc) return rc; } while (0)
  // out_proj: weight gradient over [y_fwd | y_rev] (folded over the directions by the layout pass) and dy, which both
  // directions share
  BIMAMBA_TRY(bimamba_gemm_tn(g->dout, dm, y, (int64_t)nd * D, dWo2, tn_part, M, dm, nd * D, dt, stream));
  BIMAMBA_TRY(bimamba_gemm_nt(g->dout, dm, g->WoT, dm, dy, D, nullptr, nullptr, M, D, dm, dt, dt, stream));
  // scan backward, both directions in one launch
  bimamba_scan_desc s;
  fill_scan(s, d, c, fs, es);
  s.ypre = fs + c.ypre;
  s.ckpt = c.nck > 1 ? reinterpret_cast<float*>(fs + c.ckpt) : nullptr;
  s.dout = dy; s.dout_bs = L * D; s.dout_ds = 0; s.dout_ts = D;
  s.du = du; s.ddelta = ddelta; s.dz = dz;
  s.dbc_part = dbc_part; s.dA_part = dA_part; s.dD_part = dD_part; s.dbias_part = db_part;
  s.group_channels = 32;
  BIMAMBA_TRY(bimamba_selective_scan_bwd_varlen(&s, seqlens, stream));
  // [dB | dC]: fixed-order sum over the channel groups, written next to where ddt_r goes (no concatenation)
  BIMAMBA_TRY(bimamba_reduce_rows32(dbc_part, dxdbl, B, w.ngroups, L * nd, kXW, dt, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(dA_part, dA, 1, B * nd, (int64_t)D * kN, 0, (int64_t)D * kN, 0, BIMAMBA_F32, 0, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(dD_part, g->dD, 1, B * nd, D, 0, D, 0, BIMAMBA_F32, 0, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(db_part, g->db_dt, 1, B * nd, D, 0, D, 0, BIMAMBA_F32, 0, stream));
  // dt_proj: data gradient into columns 32..47 of the same rows; weight gradient against the saved x_proj rows
  BIMAMBA_TRY(bimamba_gemm_nt(ddelta, D, g->WdT, D, static_cast<unsigned char*>(dxdbl) + (size_t)2 * kN * es, kXW, nullptr, nullptr,
                              M * nd, BIMAMBA_MAX_DT_RANK, D, dt, dt, stream));
  BIMAMBA_TRY(bimamba_gemm_tn(ddelta, D, xdbl, kXW, dWdtf, tn_part, M * nd, D, kXW, dt, stream));
  BIMAMBA_TRY(bimamba_gemm_tn(dxdbl, kXW, xc, D, dWxp, tn_part, M * nd, kXW, D, dt, stream));
  // x_proj data gradient + the scan's du
  BIMAMBA_TRY(bimamba_gemm_nt(dxdbl, kXW, g->WxpT, kXW, dxc, D, nullptr, du, M * nd, D, kXW, dt, dt, stream));
  // conv backward: dx into the x half and dz_fwd + dz_rev into the z half of one [dx | dz] matrix
  BIMAMBA_TRY(bimamba_causal_conv1d_bwd_varlen(xz, d->conv_w, d->conv_b, dxc, dxz, dz,
                                               static_cast<unsigned char*>(dxz) + (size_t)D * es, conv_part, seqlens, (int)B, nd,
                                               D, (int)L, K, L * 2 * D, 2 * D, L * nd * D, D, (int64_t)nd * D, L * 2 * D, 2 * D,
                                               dt, BIMAMBA_FLAG_SILU, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(conv_part, dwb, 1, w.conv_slices, (int64_t)D * (K + 1), 0, (int64_t)D * (K + 1), 0,
                                      BIMAMBA_F32, 0, stream));
  // in_proj
  BIMAMBA_TRY(bimamba_gemm_tn(dxz, 2 * D, d->x, dm, g->dW_in, tn_part, M, 2 * D, dm, dt, stream));
  BIMAMBA_TRY(bimamba_gemm_nt(dxz, 2 * D, g->WiT, 2 * D, g->dx, dm, nullptr, nullptr, M, dm, 2 * D, dt, dt, stream));
  // the reference's parameter layouts (dA_log = dA * A, x_proj row order, dt_proj slice, out_proj fold, conv split)
  BIMAMBA_TRY(bimamba_finalize_param_grads(dA, d->A, dWxp, dWdtf, dWo2, dwb, g->dA_log, g->dW_x, g->dW_dt, g->dW_out,
                                           g->dconv_w, g->dconv_b, dm, D, kN, R, nd, K, stream));
#undef BIMAMBA_TRY
  return 0;
}


// ================================================================================================================
// The whole encoder layer (PN_BiMambas_Encoder.forward, DualStreamSEMamba.py:467-486) in one call each way:
//   out = FFN(LN2(M(LN1 x) + flip(M(flip(LN1 x))))) + x        FFN = Linear(d_model, d_ff) -> GELU (erf) -> Linear(d_ff, d_model)
// Same kernels in the same order as the Python layer (encoder.py: layer_norm_fn -> BiMambaInnerFn -> layer_norm_fn ->
// FeedForwardFn), so results are bit-identical to it; x / out / dout / dx may be fp32 (autocast: fp32 residual stream, the
// 16-bit region between the norms and the feed-forward's second product) or the 16-bit dtype itself.
// ================================================================================================================
namespace bimamba {

struct LayerFwdCarve {
  size_t xn, mo, mn, h, a, stats, w1c, w1t, w2c, w2t, block, total;
};

static LayerFwdCarve carve_layer_fwd(int64_t B, int64_t L, int dm, int D, int dff, int ndir, int es, bool save) {
  LayerFwdCarve c{};
  const size_t M = (size_t)B * L;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += up256(bytes); return o; };
  c.xn = take(M * dm * es);
  c.mo = take(M * dm * es);
  c.mn = take(M * dm * es);
  c.h = take(M * dff * es);
  c.a = take(M * dff * es);
  c.stats = take(M * 4 * 4);               // mean1 | rstd1 | mean2 | rstd2
  c.w1c = take((size_t)dff * dm * es);
  c.w1t = take((size_t)dff * dm * es);
  c.w2c = take((size_t)dff * dm * es);
  c.w2t = take((size_t)dff * dm * es);
  c.block = off;
  off += carve_fwd(B, L, D, ndir, es, save).total;
  c.total = off;
  return c;
}

struct LayerBwdCarve {
  size_t g, da, dh, dmn, dmo, dxn, cs_part, ln_part, tn_part, block, total;
  int cs_slices, ln_blocks;
};

static LayerBwdCarve carve_layer_bwd(int64_t B, int64_t L, int dm, int D, int dff, int K, int ndir, int es) {
  LayerBwdCarve c{};
  const size_t M = (size_t)B * L;
  c.cs_slices = bimamba_colsum_slices((int64_t)M);
  c.ln_blocks = bimamba_layernorm_bwd_blocks((int64_t)M);
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += up256(bytes); return o; };
  c.g = take(M * dm * es);
  c.da = take(M * dff * es);
  c.dh = take(M * dff * es);
  c.dmn = take(M * dm * es);
  c.dmo = take(M * dm * es);
  c.dxn = take(M * dm * es);
  c.cs_part = take((size_t)(c.cs_slices > 0 ? c.cs_slices : 1) * dff * 4);
  c.ln_part = take((size_t)(c.ln_blocks > 0 ? c.ln_blocks : 1) * 2 * dm * 4);
  size_t tn = (size_t)bimamba_gemm_tn_splits((int64_t)M, dm, dff) * dm * dff * 4;
  const size_t tn2 = (size_t)bimamba_gemm_tn_splits((int64_t)M, dff, dm) * dm * dff * 4;
  if (tn2 > tn) tn = tn2;
  c.tn_part = take(tn);
  c.block = off;
  off += carve_bwd(B, L, dm, D, K, ndir, es).total;
  c.total = off;
  return c;
}

static int check_layer(const bimamba_layer_desc* d) {
  if (!d) { set_err("layer: null descriptor"); return -1; }
  const bimamba_block_desc& k = d->block;
  if (k.batch < 0 || k.seqlen < 0 || k.d_model < 1 || k.d_inner < 1 || d->d_ff < 1) { set_err("layer: bad sizes"); return -3; }
  if (k.io_dtype != BIMAMBA_BF16 && k.io_dtype != BIMAMBA_F16) { set_err("layer: the compute dtype must be bf16 or fp16"); return -6; }
  if (d->x_dtype != BIMAMBA_F32 && d->x_dtype != k.io_dtype) { set_err("layer: x must be fp32 or the compute dtype"); return -6; }
  if ((k.d_model & 7) || (k.d_inner & 7) || (d->d_ff & 7) || k.d_model > 1024) {
    set_err("layer: d_model (<= 1024), d_inner and d_ff must be multiples of 8");
    return -7;
  }
  if (!d->x || !d->out || !d->norm1_w || !d->norm1_b || !d->norm2_w || !d->norm2_b || !d->ff_w1 || !d->ff_b1 || !d->ff_w2 || !d->ff_b2) {
    set_err("layer: null operand");
    return -7;
  }
  if (!d->workspace || (reinterpret_cast<uintptr_t>(d->workspace) & 255) != 0) { set_err("layer: workspace missing or not 256-byte aligned"); return -7; }
  return 0;
}

}  // namespace bimamba

extern "C" size_t bimamba_layer_fwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int d_ff, int ndir,
                                                    int io_dtype, int save_for_backward) {
  (void)io_dtype;
  if (batch <= 0 || seqlen <= 0 || d_model <= 0 || d_inner <= 0 || d_ff <= 0 || ndir <= 0) return 0;
  return carve_layer_fwd(batch, seqlen, d_model, d_inner, d_ff, ndir, 2, save_for_backward != 0).total;
}

extern "C" size_t bimamba_layer_bwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int d_ff, int d_conv,
                                                    int ndir, int io_dtype) {
  (void)io_dtype;
  if (batch <= 0 || seqlen <= 0 || d_model <= 0 || d_inner <= 0 || d_ff <= 0 || ndir <= 0 || d_conv <= 0) return 0;
  return carve_layer_bwd(batch, seqlen, d_model, d_inner, d_ff, d_conv, ndir, 2).total;
}

extern "C" int bimamba_layer_fwd(const bimamba_layer_desc* d, bimamba_stream_t stream) {
  return bimamba_layer_fwd_varlen(d, nullptr, stream);
}

// seqlens != NULL: the block walks each utterance's own frames (bimamba_block_fwd_varlen); the norms and the feed-forward
// are per row.
extern "C" int bimamba_layer_fwd_varlen(const bimamba_layer_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  if (d && seqlens && d->block.save_for_backward) {
    set_err("layer_fwd_varlen: variable-length batches are forward-only (save_for_backward must be 0)");
    return -9;
  }
  return bimamba_layer_fwd_varlen_train(d, seqlens, stream);
}

extern "C" int bimamba_layer_fwd_varlen_train(const bimamba_layer_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  int rc = check_layer(d);
  if (rc) return rc;
  bimamba_block_desc k = d->block;
  if (k.batch == 0 || k.seqlen == 0) return 0;
  const int es = 2, cd = k.io_dtype, xd = d->x_dtype;
  const int64_t B = k.batch, L = k.seqlen, M = B * L;
  const int dm = k.d_model, D = k.d_inner, dff = d->d_ff, nd = k.ndir;
  const bool save = k.save_for_backward != 0;
  const LayerFwdCarve c = carve_layer_fwd(B, L, dm, D, dff, nd, es, save);
  if (d->workspace_bytes < c.total) { set_err("layer_fwd: workspace too small (bimamba_layer_fwd_workspace_bytes)"); return -10; }
  unsigned char* ws = static_cast<unsigned char*>(d->workspace);
  void *xn = ws + c.xn, *mo = ws + c.mo, *mn = ws + c.mn, *h = ws + c.h, *a = ws + c.a;
  float* st = reinterpret_cast<float*>(ws + c.stats);
  float *mean1 = save ? st : nullptr, *rstd1 = save ? st + M : nullptr, *mean2 = save ? st + 2 * M : nullptr,
        *rstd2 = save ? st + 3 * M : nullptr;
#define BIMAMBA_TRY(call) do { rc = (call); if (rc) return rc; } while (0)
  // norm1, written in the compute dtype (DualStreamSEMamba.py:472)
  BIMAMBA_TRY(bimamba_layernorm_fwd(d->x, d->norm1_w, d->norm1_b, xn, mean1, rstd1, M, dm, d->eps1, xd, cd, stream));
  // the bidirectional block (:473-481)
  k.x = xn;
  k.out = mo;
  k.workspace = ws + c.block;
  k.workspace_bytes = d->workspace_bytes - c.block;
  BIMAMBA_TRY(bimamba_block_fwd_varlen_train(&k, seqlens, stream));
  // norm2 (:482)
  BIMAMBA_TRY(bimamba_layernorm_fwd(mo, d->norm2_w, d->norm2_b, mn, mean2, rstd2, M, dm, d->eps2, cd, cd, stream));
  // feed-forward + residual (:483-485): weights cast (and transposed for the backward), two products with the bias and
  // the residual in their epilogues, exact GELU in between
  BIMAMBA_TRY(bimamba_cast_transpose(d->ff_w1, ws + c.w1c, ws + c.w1t, dff, dm, cd, stream));
  BIMAMBA_TRY(bimamba_cast_transpose(d->ff_w2, ws + c.w2c, ws + c.w2t, dm, dff, cd, stream));
  BIMAMBA_TRY(bimamba_gemm_nt(mn, dm, ws + c.w1c, dm, h, dff, d->ff_b1, nullptr, M, dff, dm, cd, cd, stream));
  BIMAMBA_TRY(bimamba_gelu_fwd(h, a, M * dff, cd, stream));
  BIMAMBA_TRY(bimamba_gemm_nt(a, dff, ws + c.w2c, dff, d->out, dm, d->ff_b2, d->x, M, dm, dff, cd, xd, stream));
#undef BIMAMBA_TRY
  return 0;
}

extern "C" int bimamba_layer_bwd(const bimamba_layer_desc* d, const bimamba_layer_grads* g, bimamba_stream_t stream) {
  return bimamba_layer_bwd_varlen(d, g, nullptr, stream);
}

// seqlens != NULL: the backward of bimamba_layer_fwd_varlen_train; the block's backward walks each utterance's frames.
// The norms and the feed-forward are per row: for the masked contract dout must be zero at padded frames.
extern "C" int bimamba_layer_bwd_varlen(const bimamba_layer_desc* d, const bimamba_layer_grads* g, const int32_t* seqlens,
                                        bimamba_stream_t stream) {
  int rc = check_layer(d);
  if (rc) return rc;
  if (!g) { set_err("layer_bwd: null gradient descriptor"); return -1; }
  if (!g->dout || !g->dx || !g->dnorm1 || !g->dnorm2 || !g->dff_w1 || !g->dff_b1 || !g->dff_w2 || !g->dff_b2) {
    set_err("layer_bwd: null operand");
    return -8;
  }
  bimamba_block_desc k = d->block;
  if (!k.save_for_backward) { set_err("layer_bwd: the forward must run with save_for_backward"); return -9; }
  if (!g->workspace || (reinterpret_cast<uintptr_t>(g->workspace) & 255) != 0) { set_err("layer_bwd: workspace missing or not 256-byte aligned"); return -7; }
  const int es = 2, cd = k.io_dtype, xd = d->x_dtype;
  const int64_t B = k.batch, L = k.seqlen, M = B * L;
  const int dm = k.d_model, D = k.d_inner, dff = d->d_ff, nd = k.ndir, K = k.d_conv;
  if (M == 0) { set_err("layer_bwd: empty batch"); return -3; }
  const LayerFwdCarve c = carve_layer_fwd(B, L, dm, D, dff, nd, es, true);
  const LayerBwdCarve w = carve_layer_bwd(B, L, dm, D, dff, K, nd, es);
  if (d->workspace_bytes < c.total) { set_err("layer_bwd: forward workspace too small"); return -10; }
  if (g->workspace_bytes < w.total) { set_err("layer_bwd: workspace too small (bimamba_layer_bwd_workspace_bytes)"); return -10; }
  unsigned char* fs = static_cast<unsigned char*>(d->workspace);
  unsigned char* bs = static_cast<unsigned char*>(g->workspace);
  void *xn = fs + c.xn, *mo = fs + c.mo, *mn = fs + c.mn, *h = fs + c.h, *a = fs + c.a;
  const float* st = reinterpret_cast<const float*>(fs + c.stats);
  const float *mean1 = st, *rstd1 = st + M, *mean2 = st + 2 * M, *rstd2 = st + 3 * M;
  void *da = bs + w.da, *dh = bs + w.dh, *dmn = bs + w.dmn, *dmo = bs + w.dmo, *dxn = bs + w.dxn;
  float *cs_part = reinterpret_cast<float*>(bs + w.cs_part), *ln_part = reinterpret_cast<float*>(bs + w.ln_part),
        *tn_part = reinterpret_cast<float*>(bs + w.tn_part);
#define BIMAMBA_TRY(call) do { rc = (call); if (rc) return rc; } while (0)
  // feed-forward backward; its incoming gradient is also the residual branch's (added inside norm1's backward below)
  const void* gy = g->dout;
  if (xd != cd) {
    BIMAMBA_TRY(bimamba_cast(g->dout, bs + w.g, M * dm, xd, cd, stream));
    gy = bs + w.g;
  }
  BIMAMBA_TRY(bimamba_colsum(gy, cs_part, M, dm, dm, cd, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(cs_part, g->dff_b2, 1, w.cs_slices, dm, 0, dm, 0, BIMAMBA_F32, 0, stream));
  BIMAMBA_TRY(bimamba_gemm_tn(gy, dm, a, dff, g->dff_w2, tn_part, M, dm, dff, cd, stream));
  BIMAMBA_TRY(bimamba_gemm_nt(gy, dm, fs + c.w2t, dm, da, dff, nullptr, nullptr, M, dff, dm, cd, cd, stream));
  BIMAMBA_TRY(bimamba_gelu_bwd(h, da, dh, M * dff, cd, stream));
  BIMAMBA_TRY(bimamba_colsum(dh, cs_part, M, dff, dff, cd, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(cs_part, g->dff_b1, 1, w.cs_slices, dff, 0, dff, 0, BIMAMBA_F32, 0, stream));
  BIMAMBA_TRY(bimamba_gemm_tn(dh, dff, mn, dm, g->dff_w1, tn_part, M, dff, dm, cd, stream));
  BIMAMBA_TRY(bimamba_gemm_nt(dh, dff, fs + c.w1t, dff, dmn, dm, nullptr, nullptr, M, dm, dff, cd, cd, stream));
  // norm2 backward
  BIMAMBA_TRY(bimamba_layernorm_bwd(mo, dmn, d->norm2_w, mean2, rstd2, nullptr, dmo, ln_part, M, dm, cd, cd, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(ln_part, g->dnorm2, 1, w.ln_blocks, 2 * dm, 0, 2 * dm, 0, BIMAMBA_F32, 0, stream));
  // the block
  k.x = xn;
  k.out = mo;
  k.workspace = fs + c.block;
  k.workspace_bytes = d->workspace_bytes - c.block;
  bimamba_block_grads kg = g->block;
  kg.dout = dmo;
  kg.dx = dxn;
  kg.workspace = bs + w.block;
  kg.workspace_bytes = g->workspace_bytes - w.block;
  BIMAMBA_TRY(bimamba_block_bwd_varlen(&k, &kg, seqlens, stream));
  // norm1 backward + the residual branch's gradient
  BIMAMBA_TRY(bimamba_layernorm_bwd(d->x, dxn, d->norm1_w, mean1, rstd1, g->dout, g->dx, ln_part, M, dm, xd, cd, stream));
  BIMAMBA_TRY(bimamba_reduce_partials(ln_part, g->dnorm1, 1, w.ln_blocks, 2 * dm, 0, 2 * dm, 0, BIMAMBA_F32, 0, stream));
#undef BIMAMBA_TRY
  return 0;
}
