/* bimamba.h - C ABI of libbimamba_sm100.so (B200 / sm_100a Bi-Mamba hot path).
 *
 * Every entry point is `extern "C"`, takes plain pointers, sizes and element strides
 * and a CUDA stream handle; no torch / C++ types cross this boundary.
 *
 * What each entry point replaces in the reference (lux-liang/Robust-Audio-Deepfake-
 * Evolution).  The reference reaches this arithmetic through the third-party
 * `mamba_ssm` package (import at src/models/DualStreamSEMamba.py:43, constructed at
 * :455, called at :473 and :477); the in-repo statement of the same math is
 * src/models/modules/mamba_block.py.  The FFI the reference's path binds upstream is
 * `selective_scan_cuda.{fwd,bwd}` and `causal_conv1d_cuda.causal_conv1d_{fwd,bwd}`;
 * the functions below are their drop-in equivalents (same operand meaning), with two
 * B200-first changes: (1) activations are CHANNEL-LAST (batch, time, channel) - the
 * layout the in_proj / x_proj / out_proj GEMMs produce and consume - so the path has
 * no transposes, and (2) a direction axis lets the forward scan and the flipped scan
 * of DualStreamSEMamba.py:473-481 share ONE launch with no flipped copies.
 *
 *   bimamba_causal_conv1d_fwd/bwd    <- mamba_block.py:24-31,52-55 (depthwise causal
 *                                       Conv1d k=4, crop to L, SiLU) and its autograd
 *   bimamba_selective_scan_fwd/bwd   <- mamba_block.py:80 (dt_proj + softplus), :82 (A),
 *                                       :92-117 (scan), :120 (D skip), :61 (z gate)
 *                                       and its autograd
 *   bimamba_reduce_partials          <- the sum over batch/time/direction that
 *                                       autograd performs for parameter gradients
 *   bimamba_layernorm_fwd/bwd        <- nn.LayerNorm of the encoder layer (DualStreamSEMamba.py:472,482)
 *   bimamba_gemm_nt                  <- the nn.Linear calls of mamba_block.py:48,73,62
 *                                       (in_proj, x_proj, out_proj) on tcgen05 tensor cores
 *   bimamba_block_fwd/bwd            <- the whole block, both directions, one call each way
 *                                       (mamba_block.py:41-63 + DualStreamSEMamba.py:473-481)
 *
 *   bimamba_*_fwd_varlen              <- scoring of right-padded batches of utterances of different lengths
 *                                       (per-utterance frame counts; see "Variable-length scoring" below)
 *   bimamba_*_varlen_train, *_bwd_varlen, bimamba_mask_frames
 *                                    <- training on such batches (see "Variable-length training" below)
 *   bimamba_mixup_frames             <- Mixup of the training loop (src/main.py:1038-1046), fixed or variable length
 *
 * Ownership: the library never allocates or frees device memory.  All tensors and
 * workspaces are caller-allocated; pointers are borrowed for the duration of the
 * enqueue.  Calls only enqueue work on `stream` (no device sync, CUDA-graph safe).
 * Errors: 0 = success; negative = argument error (see bimamba_last_error());
 * positive = cudaError_t from the launch.  Nothing throws across this boundary.
 */
#ifndef BIMAMBA_H_
#define BIMAMBA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIMAMBA_ABI_VERSION 12

/* element types of activation operands */
#define BIMAMBA_F32 0
#define BIMAMBA_BF16 1
#define BIMAMBA_F16 2

/* flags */
#define BIMAMBA_FLAG_SOFTPLUS 1 /* delta = softplus(delta + delta_bias) (mamba_block.py:80) */
#define BIMAMBA_FLAG_DTR_PADDED 2 /* scan: every dtr row is readable (and finite) up to 16 elements and
                                    16-byte aligned, so it can be staged with vector copies */
#define BIMAMBA_FLAG_SILU 1     /* conv: apply SiLU (mamba_block.py:55) */

#define BIMAMBA_DSTATE 16       /* d_state of the Phase-6 configuration (Phase6_Proposed.conf:26) */
#define BIMAMBA_MAX_DT_RANK 16
#define BIMAMBA_CHUNK 16        /* time steps staged per forward chunk */
#define BIMAMBA_CKPT 8          /* checkpoint interval = steps per backward chunk */

typedef void* bimamba_stream_t; /* a cudaStream_t */

/* Selective scan.  All activations are channel-last and share the element type io_dtype:
 * element (b, dir, t, d) of tensor X lives at X + b*X_bs + dir*X_ds + t*X_ts + d (unit
 * channel stride; strides in ELEMENTS).  "dir" is the direction axis: dir 0 scans
 * t = 0..L-1, dir 1 scans t = L-1..0 over the same storage (natural time order in memory),
 * i.e. dir 1 computes flip(op(flip(.))) of DualStreamSEMamba.py:476-478 with no flipped copy.
 * A stride of 0 on the dir axis shares one tensor between both directions (z, dout).
 *
 * The step size is either given (delta != NULL: the dt_proj output before bias and
 * softplus, as in mamba_ssm's selective_scan_fn) or produced in-kernel from the low-rank
 * projection (delta == NULL:  delta_raw[t,d] = sum_r Wdt[d,r] * dtr[t,r], mamba_block.py:80),
 * which saves writing and re-reading a (B, L, D) tensor. */
typedef struct bimamba_scan_desc {
  const void* u;     /* (batch, ndir, L, dim)   conv output xc                          */
  const void* z;     /* (batch, ndir, L, dim) or NULL (gate input)                       */
  const void* delta; /* (batch, ndir, L, dim) or NULL (then dtr / Wdt are used)          */
  const void* bc;    /* (batch, ndir, L, 32): row t = [B_t(16) | C_t(16)]                */
  const void* dtr;   /* (batch, ndir, L, dt_rank) low-rank step-size features, or NULL   */
  const float* Wdt;  /* (dim, dt_rank) fp32 dt_proj.weight, or NULL                      */
  const float* A;    /* (dim, 16) fp32, = -exp(A_log)                                    */
  const float* D;    /* (dim) fp32 or NULL                                               */
  const float* delta_bias; /* (dim) fp32 or NULL                                         */
  void* out;         /* fwd: (batch, ndir, L, dim) gated output                          */
  void* ypre;        /* (batch, ndir, L, dim) y before the z gate, strides = out's.  Written by
                        fwd when non-NULL; read by bwd to form dz (required there with z) */
  float* ckpt;       /* (batch, ndir, nckpt, dim, 16) fp32 state entering every 8-step chunk,
                        nckpt = ceil(L / 8); written by fwd when non-NULL, read by bwd
                        (required there when nckpt > 1)                                   */
  /* backward only */
  const void* dout;  /* (batch, ndir, L, dim), strides dout_*                             */
  void* du;          /* (batch, ndir, L, dim), strides = out's (out_bs/out_ds/out_ts)     */
  void* ddelta;      /* same layout: gradient w.r.t. the pre-softplus step size           */
  void* dz;          /* same layout or NULL: per-direction gradient of the gate input     */
  float* dbc_part;   /* (batch, ngroups, L, ndir, 32) fp32 partial [dB | dC] of each channel
                        group; reduce over ngroups with bimamba_reduce_partials -> rows
                        ordered (batch, time, dir)                                        */
  float* dA_part;    /* (batch, ndir, dim, 16) fp32                                        */
  float* dD_part;    /* (batch, ndir, dim) fp32 or NULL                                    */
  float* dbias_part; /* (batch, ndir, dim) fp32 or NULL                                    */

  int32_t batch, ndir, dim, seqlen, dstate, dt_rank;
  int32_t io_dtype, flags;
  int32_t group_channels; /* channels per CTA (use bimamba_scan_plan) */
  int32_t reserved0;
  int64_t u_bs, u_ds, u_ts;
  int64_t z_bs, z_ds, z_ts;
  int64_t delta_bs, delta_ds, delta_ts;
  int64_t bc_bs, bc_ds, bc_ts;
  int64_t dtr_bs, dtr_ds, dtr_ts;
  int64_t out_bs, out_ds, out_ts;
  int64_t dout_bs, dout_ds, dout_ts;
} bimamba_scan_desc;

int bimamba_abi_version(void);
const char* bimamba_last_error(void);

/* Tuning knobs: force a kernel variant (parity tests of every shipped variant, tuning experiments).  0 = automatic.
 * Process-wide; not meant to change while launches are in flight on other threads. */
#define BIMAMBA_TUNE_SCAN_FWD 0     /* 1 = wide CTAs sharing the staged rows, 3 = one warp per CTA                 */
#define BIMAMBA_TUNE_CONV_BWD 1     /* 1 = shared-memory tile kernel instead of the register-window kernel         */
#define BIMAMBA_TUNE_GEMM_KERNEL 2  /* 1 = one tile per CTA, 2 = persistent warp-specialised                       */
#define BIMAMBA_TUNE_GEMM_BN 3      /* tile width override                                                         */
#define BIMAMBA_TUNE_GEMM_STAGES 4  /* TMA ring depth override                                                     */
#define BIMAMBA_TUNE_PDL 5          /* 1 = launch without programmatic dependent launch (A/B measurements)         */
#define BIMAMBA_TUNE_SCAN_SPLIT 6   /* forward scan time split: 1 = never, k >= 2 = k segments at any size (parity tests) */
#define BIMAMBA_TUNE_COUNT 7
int bimamba_set_tuning(int knob, int value);
int bimamba_get_tuning(int knob);

/* Bytes of the caller-allocated workspaces of the scan calls (for hosts that do not re-derive the geometry):
 * forward with want_ckpt != 0: ckpt (fp32, (batch, ndir, nckpt, dim, 16), only when nckpt > 1) followed by ypre
 * ((batch, ndir, seqlen, dim) in io_dtype); backward: dbc_part + dA_part + dD_part + dbias_part (all fp32). */
size_t bimamba_scan_fwd_workspace_bytes(int batch, int ndir, int seqlen, int dim, int io_dtype, int want_ckpt);
size_t bimamba_scan_bwd_workspace_bytes(int batch, int ndir, int seqlen, int dim);

/* Chooses the channel-group width for (seqlen, dim, batch*ndir); backward != 0 selects the
 * backward kernel's geometry.  Returns nckpt = ceil(seqlen / 8), the number of checkpoints per
 * (batch, dir, channel); *ngroups = CTAs per (batch, dir) = ceil(dim / *group_channels). */
int bimamba_scan_plan(int seqlen, int dim, int rows, int backward, int* group_channels, int* ngroups);

int bimamba_selective_scan_fwd(const bimamba_scan_desc* d, bimamba_stream_t stream);
int bimamba_selective_scan_bwd(const bimamba_scan_desc* d, bimamba_stream_t stream);

/* ---- Variable-length scoring.  `seqlens` is a DEVICE pointer to `batch` int32 frame counts: utterance b is frames
 * 0 .. seqlens[b]-1 of a right-padded batch of `seqlen` frames, and every valid output equals what the utterance gives
 * when it runs alone at its own length.  Kernels clamp seqlens[b] to [0, seqlen]; frames at or past it are never read
 * by the conv, the scan or the head, so the padding may hold anything (NaN included).  Outputs a call owns per frame
 * (conv out, scan out / ypre) are written as zeros at padded frames; a zero-length utterance yields zeros.  A NULL
 * seqlens is the fixed-length call: bimamba_X(...) is bimamba_X_varlen(..., NULL, ...).  Forward only: the scan rejects
 * checkpoints (d->ckpt != NULL) and the block / layer reject save_for_backward != 0 with a negative code; the
 * _varlen_train entries below are the training forms. */
int bimamba_selective_scan_fwd_varlen(const bimamba_scan_desc* d, const int32_t* seqlens, bimamba_stream_t stream);

/* ---- Variable-length training.  The training forward and the backward of each op walk the same per-utterance frames
 * as the scoring calls above (seqlens: device int32, clamped to [0, seqlen]; NULL = the fixed-length call, so
 * bimamba_X_bwd(...) is bimamba_X_bwd_varlen(..., NULL, ...)).  Each utterance gets the gradients it would get alone at
 * its own length; parameter-gradient partials sum over utterances as a batch does.  Layouts and workspace sizes are
 * those of the padded seqlen (checkpoints: ceil(seqlen / 8) per channel, chunk c = scan steps 8c .. 8c+7 of the
 * utterance).  Gradients a call owns per frame (scan du / ddelta / dz and its [dB | dC] partial rows, conv dx and the
 * folded dz, head dx) are written as zeros at padded frames; dout there is never read by the scan or the conv.
 *
 * The scan forward that also writes checkpoints and ypre (the refusal of bimamba_selective_scan_fwd_varlen lifted): */
int bimamba_selective_scan_fwd_varlen_train(const bimamba_scan_desc* d, const int32_t* seqlens, bimamba_stream_t stream);
int bimamba_selective_scan_bwd_varlen(const bimamba_scan_desc* d, const int32_t* seqlens, bimamba_stream_t stream);

/* out (batch, seqlen, channels) = x where t < seqlens[b], zero elsewhere - by selection: padded frames are never read, so
 * NaN padding cannot pass.  x and out contiguous in `dtype`; out may be x (in place).  One launch.  With the block and
 * layer entries a host gets the masked training contract by masking x before the forward and dout before the backward
 * (and, for the layer, the output after the forward: its feed-forward and residual make padded output rows non-zero). */
int bimamba_mask_frames(const void* x, void* out, const int32_t* seqlens, int batch, int seqlen, int channels, int dtype,
                        bimamba_stream_t stream);

/* Mixup of a right-padded batch (src/main.py:1038-1046), one launch.  x and out (batch, seqlen, channels) contiguous in
 * `dtype`, out not x (rows read other rows); perm: device int32 (batch,) permutation p (values clamped to [0, batch));
 * mix: device fp32 {lam, 1 - lam}, both formed in double on the host and rounded to fp32.  Each product is rounded to
 * `dtype`, then their sum: out[b, t] = rn(rn(lam x[b, t]) + rn((1 - lam) x[p(b), t])), the bits of torch's
 * `lam * x + (1.0 - lam) * x[perm]`.  seqlens_in (device int32, clamped to [0, seqlen]) or NULL = every frame valid: a
 * term is taken only over its own utterance's frames (by selection, so padding is never read), out is exactly zero at
 * t >= max(n_b, n_p(b)), and that mixed length goes to seqlens_out (required with seqlens_in, ignored without it).
 * NULL operand -1, bad sizes / dtype -3, empty batch a no-op 0. */
int bimamba_mixup_frames(const void* x, void* out, const int32_t* perm, const float* mix, const int32_t* seqlens_in,
                         int32_t* seqlens_out, int batch, int seqlen, int channels, int dtype, bimamba_stream_t stream);

/* ---- Variable-length DualStreamFusion (DualStreamSEMamba.py:580-637 run on each utterance alone).  Two streams, two
 * length vectors: seqlens_dst (batch) are the WavLM frame counts n1 of a batch padded to dst_frames, seqlens_src the
 * SincNet frame counts n2 of a batch padded to src_frames (device int32, clamped to [0, frames]).  Activations
 * (batch, frames, channels) contiguous in `dtype`; arithmetic fp32 with one rounding; frames at or past an utterance's
 * length are never read and are written as zeros.  NULL operand -1, bad sizes -3, empty batch a no-op 0.
 *
 * Interpolation of the projected SincNet branch onto the WavLM frames, per utterance (:601-626, F.interpolate):
 * n1 == n2 copies (bit-identical), n1 > 4 n2 is nearest, otherwise linear with align_corners=False, on ATen's fp32
 * index rule (scale = (float)n2 / n1; see DESIGN.md 4.8).  The backward is a gather: each source frame sums the weighted
 * cotangents of the destination frames that read it in increasing frame order (deterministic). */
int bimamba_interp_frames_fwd(const void* src, void* dst, const int32_t* seqlens_dst, const int32_t* seqlens_src,
                              int batch, int dst_frames, int src_frames, int channels, int dtype, bimamba_stream_t stream);
int bimamba_interp_frames_bwd(const void* ddst, void* dsrc, const int32_t* seqlens_dst, const int32_t* seqlens_src,
                              int batch, int dst_frames, int src_frames, int channels, int dtype, bimamba_stream_t stream);
/* SELayer's squeeze (:524-526, AdaptiveAvgPool1d): mean (batch, channels) fp32 = sum_{t < n} x / n in a fixed order;
 * 0 for a zero-length utterance.  Backward: dx = dmean / n at valid frames. */
int bimamba_frame_mean(const void* x, float* mean, const int32_t* seqlens, int batch, int seqlen, int channels,
                       int dtype, bimamba_stream_t stream);
int bimamba_frame_mean_bwd(const float* dmean, void* dx, const int32_t* seqlens, int batch, int seqlen, int channels,
                           int dtype, bimamba_stream_t stream);
/* SELayer's excitation product (:528): y = x * gate[b] (gate (batch, channels) fp32).  Backward in one pass:
 * dx = dy * gate[b] and dgate_part (batch, nslices, channels) fp32, nslices = bimamba_frame_scale_bwd_slices(seqlen),
 * the sums of dy * x over each slice's valid frames: finish with bimamba_reduce_partials(groups = batch, rows = nslices,
 * cols = channels, part_gs = nslices * channels, row_stride = channels, out_gs = channels). */
int bimamba_frame_scale(const void* x, const float* gate, void* y, const int32_t* seqlens, int batch, int seqlen,
                        int channels, int dtype, bimamba_stream_t stream);
int bimamba_frame_scale_bwd_slices(int seqlen);
int bimamba_frame_scale_bwd(const void* x, const float* gate, const void* dy, void* dx, float* dgate_part,
                            const int32_t* seqlens, int batch, int seqlen, int channels, int dtype,
                            bimamba_stream_t stream);

/* Time-parallel forward scan for long sequences at small batches (the scan as an associative operator on pairs,
 * (a2, b2) o (a1, b1) = (a2 a1, a2 b1 + b2); mamba_block.py:92-117 is the serial loop).  Scan time is cut into nseg
 * segments of seg_len steps: a carry pass computes every segment's end state from zero and its decay exponent
 * sum_t delta_t, the output pass starts each segment from the carries combined in order.  Same descriptor, outputs,
 * ypre and checkpoints as bimamba_selective_scan_fwd (the backward is unchanged); results differ from the unsplit call
 * by fp32 rounding only (exp(A sum delta) against the product of per-step decays).
 * bimamba_scan_fwd_split_plan returns *nseg = 1 when splitting does not pay (enough channel lanes to fill the GPU, a
 * short sequence, or fp32 I/O - measured slower): then call bimamba_selective_scan_fwd.  carry: caller-allocated fp32 workspace of
 * bimamba_scan_fwd_split_workspace_bytes(batch, ndir, dim, nseg) bytes, 16-byte aligned. */
int bimamba_scan_fwd_split_plan(int batch, int ndir, int seqlen, int dim, int io_dtype, int* nseg, int* seg_len);
size_t bimamba_scan_fwd_split_workspace_bytes(int batch, int ndir, int dim, int nseg);
int bimamba_selective_scan_fwd_split(const bimamba_scan_desc* d, int nseg, int seg_len, float* carry, size_t carry_bytes,
                                     bimamba_stream_t stream);

/* Depthwise causal conv, channel-last.  x: (batch, L, dim) with strides x_bs, x_ts;
 * out: (batch, ndir, L, dim) with strides out_bs, out_ds, out_ts.  dir 0: taps t-(K-1)..t;
 * dir 1: taps t..t+(K-1), i.e. the causal conv of the time-reversed sequence in natural
 * order.  K in {2,3,4}; weight (dim, K) fp32; bias (dim) fp32 or NULL. */
int bimamba_causal_conv1d_fwd(const void* x, const float* weight, const float* bias, void* out,
                              int batch, int ndir, int dim, int seqlen, int width,
                              int64_t x_bs, int64_t x_ts, int64_t out_bs, int64_t out_ds, int64_t out_ts,
                              int dtype, int flags, bimamba_stream_t stream);
/* Per-utterance frame counts (see bimamba_selective_scan_fwd_varlen): dir 1's taps t + k >= seqlens[b] read as zero. */
int bimamba_causal_conv1d_fwd_varlen(const void* x, const float* weight, const float* bias, void* out,
                                     const int32_t* seqlens, int batch, int ndir, int dim, int seqlen, int width,
                                     int64_t x_bs, int64_t x_ts, int64_t out_bs, int64_t out_ds, int64_t out_ts,
                                     int dtype, int flags, bimamba_stream_t stream);

/* dout: (batch, ndir, L, dim) grads w.r.t. the conv output of each direction.
 * dx: (batch, L, dim), summed over directions.  dz_in (optional, may be NULL): per-direction
 * (batch, ndir, L, dim) gate gradients with dout's strides; when given their sum over
 * directions is written to dz_out (batch, L, dim) with dx's strides, so the in_proj backward
 * reads one [dx | dz] matrix.  dwb_part: (nslices, dim, K+1) fp32 partials
 * [dw_0..dw_{K-1}, dbias] with nslices = bimamba_conv_bwd_slices(batch, seqlen, dim); reduce over
 * slices with bimamba_reduce_partials. */
int bimamba_conv_bwd_slices(int batch, int seqlen, int dim);
int bimamba_causal_conv1d_bwd(const void* x, const float* weight, const float* bias, const void* dout,
                              void* dx, const void* dz_in, void* dz_out, float* dwb_part,
                              int batch, int ndir, int dim, int seqlen, int width,
                              int64_t x_bs, int64_t x_ts, int64_t dout_bs, int64_t dout_ds, int64_t dout_ts,
                              int64_t dx_bs, int64_t dx_ts, int dtype, int flags, bimamba_stream_t stream);
/* Backward of bimamba_causal_conv1d_fwd_varlen: frames t >= seqlens[b] of x and dout are never read; dx and dz_out are
 * zero there. */
int bimamba_causal_conv1d_bwd_varlen(const void* x, const float* weight, const float* bias, const void* dout,
                                     void* dx, const void* dz_in, void* dz_out, float* dwb_part, const int32_t* seqlens,
                                     int batch, int ndir, int dim, int seqlen, int width,
                                     int64_t x_bs, int64_t x_ts, int64_t dout_bs, int64_t dout_ds, int64_t dout_ts,
                                     int64_t dx_bs, int64_t dx_ts, int dtype, int flags, bimamba_stream_t stream);

/* For every g < groups:  out[g*out_gs + j] (+)= sum_{i < rows} part[g*part_gs + i*row_stride + j],
 * j < cols, summed in fixed order (deterministic).  out element type out_dtype;
 * accumulate != 0 adds to the existing contents. */
int bimamba_reduce_partials(const float* part, void* out, int64_t groups, int64_t rows, int64_t cols,
                            int64_t part_gs, int64_t row_stride, int64_t out_gs,
                            int out_dtype, int accumulate, bimamba_stream_t stream);

/* Weight-gradient product C[N1, N2] = A[M, N1]^T . B[M, N2] (bf16 / fp16 row-major activations, contraction over
 * the B*L rows; C fp32 row-major) on the tcgen05 tensor cores with MN-major operands: dW = dY^T X of the nn.Linear
 * layers (autograd of mamba_block.py:48, :73, :62 and DualStreamSEMamba.py:460-464).  The contraction is split over
 * nsplit = bimamba_gemm_tn_splits(M, N1, N2) CTAs (one wave); `part` is a caller-allocated workspace of
 * nsplit * N1 * N2 floats; the splits are summed in fixed order (deterministic) by a second kernel of the same call. */
int bimamba_gemm_tn_splits(int64_t M, int N1, int N2);
int bimamba_gemm_tn(const void* A, int64_t lda, const void* B, int64_t ldb, float* C, float* part, int64_t M, int N1,
                    int N2, int in_dtype, bimamba_stream_t stream);

/* Backend head, forward (scoring path): y = LayerNorm(x) over channels; a = softmax over time of (w_att . y + b_att);
 * features = sum_t a_t y_t; logits = W_cls features + b_cls - src/models/DualStreamSEMamba.py:759-767 in eval mode
 * (dropout = identity), the score of src/main.py:978-984 being logits[:, 1].  x (batch, seqlen, channels) contiguous
 * in `dtype`; parameters fp32; features (batch, channels) and logits (batch, nclasses) fp32.  One launch.
 * nclasses = 0 skips the classifier (w_cls, b_cls, logits may be NULL). */
int bimamba_head_fwd(const void* x, const float* gamma, const float* beta, const float* w_att, const float* b_att,
                     const float* w_cls, const float* b_cls, float* features, float* logits, int batch, int seqlen,
                     int channels, int nclasses, float eps, int dtype, bimamba_stream_t stream);
/* Per-utterance frame counts (see bimamba_selective_scan_fwd_varlen): norm, softmax and pooling over t < seqlens[b];
 * a zero-length utterance gets zero features and logits = b_cls. */
int bimamba_head_fwd_varlen(const void* x, const float* gamma, const float* beta, const float* w_att, const float* b_att,
                            const float* w_cls, const float* b_cls, float* features, float* logits,
                            const int32_t* seqlens, int batch, int seqlen, int channels, int nclasses, float eps,
                            int dtype, bimamba_stream_t stream);

/* Backward of the pooled features of bimamba_head_fwd (the training head: norm_f + attention pooling under autograd,
 * DualStreamSEMamba.py:759-763; call bimamba_head_fwd with nclasses = 0 for the forward - dropout and the classifier
 * act on (batch, channels) outside).  dfeatures (batch, channels) fp32; dx (batch, seqlen, channels) in `dtype`;
 * part (batch, 4, channels) fp32 = per-utterance rows [dgamma | dbeta | dw_att | (db_att, 0, ...)]: sum over the batch
 * with bimamba_reduce_partials.  Two launch-free passes over the frames, fixed summation order (deterministic). */
int bimamba_head_pool_bwd(const void* x, const float* gamma, const float* beta, const float* w_att, const float* b_att,
                          const float* dfeatures, void* dx, float* part, int batch, int seqlen, int channels, float eps,
                          int dtype, bimamba_stream_t stream);
/* Backward of bimamba_head_fwd_varlen (nclasses = 0): both passes over t < seqlens[b]; dx is zero at padded frames and a
 * zero-length utterance gets zero dx and a zero partial row. */
int bimamba_head_pool_bwd_varlen(const void* x, const float* gamma, const float* beta, const float* w_att,
                                 const float* b_att, const float* dfeatures, void* dx, float* part,
                                 const int32_t* seqlens, int batch, int seqlen, int channels, float eps, int dtype,
                                 bimamba_stream_t stream);

/* AdamW (torch.optim.AdamW semantics: decoupled weight decay, no amsgrad - the optimizer of src/main.py:453) over a
 * list of fp32 tensors in one launch.  `table` (device): one entry per tensor; `block_map` (device): nblocks pairs
 * (tensor index, chunk index), one per CTA, chunk = bimamba_adamw_chunk() elements; `hyper` (device) =
 * {lr, beta1, beta2, eps, weight_decay}; `state` (device) = {step}: the call first increments the step on the device
 * (so it can be captured in a CUDA graph and replayed), then updates p, m, v in place. */
struct bimamba_adamw_tensor {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
};
int bimamba_adamw_chunk(void);
int bimamba_adamw_step(const struct bimamba_adamw_tensor* table, const int32_t* block_map, int nblocks,
                       const float* hyper, float* state, bimamba_stream_t stream);

/* The optimizer step of the fp16 recipe (src/main.py:1100-1117) on the device, capturable:
 *   scaler.unscale_ -> clip_grad_norm_(max_norm) -> scaler.step (skipped when a gradient is inf / NaN) -> scaler.update
 *   -> ema.update_parameters
 * over the tables bimamba_adamw_step reads.  Per optimizer step, on one stream:
 *   1. bimamba_amp_grad_stats over ONE table and block map holding every group's tensors;
 *   2. bimamba_adamw_amp_step once per parameter group (and once more, without hyper / state / amp, for parameters the
 *      optimizer does not hold but the average covers);
 *   3. bimamba_amp_update.
 * The gradients stay scaled: the step reads (g * inv_scale) * clip_coef and writes no gradient back.
 *
 * The loss-scaling record (device memory, 4-byte aligned).  scale and growth_tracker are the state of
 * torch.amp.GradScaler (its `_scale` and `_growth_tracker`); the other fields are written by bimamba_amp_grad_stats. */
typedef struct bimamba_amp {
  float scale;            /* loss scale S: the loss is multiplied by S before backward; the step unscales by
                             inv_scale = (float)(1.0 / (double)S), as GradScaler.unscale_ does                       */
  int32_t growth_tracker; /* applied steps since the scale last changed                                              */
  float found_inf;        /* 1 when any gradient element is inf or NaN (the step is then skipped), else 0            */
  float total_norm;       /* 2-norm of the unscaled gradient over every tensor (clip_grad_norm_'s return value),
                             summed in fp64 in a fixed order; NaN or inf when found_inf                              */
  float clip_coef;        /* min(1, max_norm / (total_norm + 1e-6)) in fp32, 1 without clipping                      */
  int32_t reserved[3];    /* unused; pads the record to 32 bytes                                                     */
} bimamba_amp;

/* Averaged copy of one parameter (torch.optim.swa_utils.AveragedModel with get_ema_multi_avg_fn): entry i goes with
 * entry i of the AdamW table.  n = the parameter's element count, also when it has no gradient (table n = 0);
 * n = 0: the parameter has no average. */
struct bimamba_ema_tensor {
  float* avg;
  int64_t n;
};

/* Step 1.  One CTA per block-map entry sums (g * inv_scale)^2 of its chunk into partials[i] (device, nblocks doubles,
 * caller-owned; NaN marks a chunk with a non-finite gradient); one more CTA adds them in a fixed order and writes
 * found_inf, total_norm and clip_coef.  max_norm <= 0: no clipping (clip_coef = 1).  Entries with n = 0 are skipped.
 * Deterministic: the same gradients give the same bits. */
int bimamba_amp_grad_stats(const struct bimamba_adamw_tensor* table, const int32_t* block_map, int nblocks,
                           float max_norm, double* partials, bimamba_amp* amp, bimamba_stream_t stream);
/* Step 2.  bimamba_adamw_step on the gradient (g * amp->inv_scale) * amp->clip_coef (two fp32 roundings in that order,
 * the .grad unscale_ then clip_grad_norm_ leave); when amp->found_inf is set p, m, v and the step counter are left as
 * they are.  hyper, state and amp are given together or all NULL (then only the averages move).
 * ema != NULL (with n_averaged, the AveragedModel's device counter): afterwards every average moves toward its
 * parameter, also on a skipped step - a copy while *n_averaged == 0, else torch's lerp with weight ema_weight
 * (= 1 - decay, in [0, 1]): avg + w (p - avg) for w < 0.5, bit for bit as torch._foreach_lerp_. */
int bimamba_adamw_amp_step(const struct bimamba_adamw_tensor* table, const int32_t* block_map, int nblocks,
                           const float* hyper, float* state, const bimamba_amp* amp,
                           const struct bimamba_ema_tensor* ema, const int64_t* n_averaged, float ema_weight,
                           bimamba_stream_t stream);
/* Step 3.  amp != NULL: torch._amp_update_scale_ - found_inf: scale *= backoff_factor, growth_tracker = 0; else
 * growth_tracker + 1, and at growth_interval scale *= growth_factor (kept if finite) and growth_tracker = 0.
 * n_averaged != NULL: *n_averaged += 1.  At least one of the two. */
int bimamba_amp_update(bimamba_amp* amp, double growth_factor, double backoff_factor, int growth_interval,
                       int64_t* n_averaged, bimamba_stream_t stream);

/* Column sums of a (rows, cols) matrix with row stride ld (elements): the bias gradients of the Linear layers.
 * Writes fp32 partials part (nslices, cols), nslices = bimamba_colsum_slices(rows); finish with
 * bimamba_reduce_partials. */
int bimamba_colsum_slices(int64_t rows);
int bimamba_colsum(const void* x, float* part, int64_t rows, int cols, int64_t ld, int dtype, bimamba_stream_t stream);

/* LayerNorm over the channel axis of a dense (rows, channels) matrix: the nn.LayerNorm(d_model) calls
 * of PN_BiMambas_Encoder (DualStreamSEMamba.py:458-459, :472, :482) and norm_f (:703, :759).
 * y = (x - mean) * rstd * gamma + beta, written in out_dtype (the dtype the following GEMM reads).
 * mean / rstd (rows) fp32 are saved for the backward (may be NULL for inference).  channels <= 1024. */
int bimamba_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean,
                          float* rstd, int64_t rows, int channels, float eps, int in_dtype, int out_dtype,
                          bimamba_stream_t stream);

/* dx (x's dtype) and per-CTA partials dgb_part (nblocks, 2, channels) fp32 = [dgamma | dbeta] with
 * nblocks = bimamba_layernorm_bwd_blocks(rows); reduce with bimamba_reduce_partials.  channels <= 1024.
 * dx_addend (optional, x's dtype, same layout as dx): added to dx - the gradient of a residual branch that bypasses the
 * norm (out = f(LN(x)) + x, DualStreamSEMamba.py:471-485), so autograd needs no separate add. */
int bimamba_layernorm_bwd_blocks(int64_t rows);
int bimamba_layernorm_bwd(const void* x, const void* dy, const float* gamma, const float* mean,
                          const float* rstd, const void* dx_addend, void* dx, float* dgb_part, int64_t rows,
                          int channels, int x_dtype, int dy_dtype, bimamba_stream_t stream);

/* C[M, N] = A[M, K] . B[N, K]^T (+ bias[N]) (+ addend[M, N]) with bf16 / fp16 operands (row-major, K contiguous, row strides
 * lda / ldb in elements, multiples of 8, 16-byte aligned bases) and fp32 accumulation on the tcgen05 tensor
 * cores (TMA-fed, TMEM accumulator).  C has out_dtype (fp32 or the operand dtype) and row stride ldc.  This is
 * nn.Linear: in_proj / x_proj / out_proj (mamba_block.py:48, :73, :62), the feed-forward Linears
 * (DualStreamSEMamba.py:460-464) and, with B = W^T, their data gradients.  Ragged M, N, K are handled by the
 * TMA unit's zero fill.  addend (optional) has C's dtype and row stride (residual / accumulate-into).
 * bimamba_gemm_nt_block_n_k(N, K) is the tile width the kernel will use. */
int bimamba_gemm_nt_block_n(int N);
int bimamba_gemm_nt_block_n_k(int N, int K);
int bimamba_gemm_nt(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
                    const float* bias, const void* addend, int64_t M, int N, int K, int in_dtype, int out_dtype,
                    bimamba_stream_t stream);

/* Per-step weight preparation of one Mamba block in one launch: from the fp32 master parameters
 * (mamba_block.py:22-39) to the arrangements the kernels read, in `dtype`:
 *   Wi (2D, dm) = in_proj.weight; WiT (dm, 2D) its transpose; Wxp (48, D) = x_proj.weight repacked
 *   [B | C | dt_r | 0]; WxpT (D, 48); Wo2 (dm, ndir*D) = [out_proj.weight] x ndir; WoT (D, dm);
 *   WdT (16, D) = dt_proj.weight^T zero padded; A (D, N) fp32 = -exp(A_log) (mamba_block.py:82). */
int bimamba_pack_weights(const float* W_in, const float* W_x, const float* W_dt, const float* A_log,
                         const float* W_out, void* Wi, void* WiT, void* Wxp, void* WxpT, void* Wo2,
                         void* WoT, void* WdT, float* A, int d_model, int d_inner, int d_state,
                         int dt_rank, int ndir, int dtype, bimamba_stream_t stream);

/* dst (rows, cols) = cast(src); dstT (cols, rows) = cast(src)^T: a Linear weight and its data-gradient operand. */
int bimamba_cast_transpose(const float* src, void* dst, void* dstT, int rows, int cols, int dtype,
                           bimamba_stream_t stream);

/* Exact (erf) GELU of the feed-forward (nn.GELU(), DualStreamSEMamba.py:462) and its backward dx = dy * gelu'(x), over n
 * contiguous elements of `dtype` (16-byte aligned bases). */
int bimamba_gelu_fwd(const void* x, void* y, int64_t n, int dtype, bimamba_stream_t stream);
int bimamba_gelu_bwd(const void* x, const void* dy, void* dx, int64_t n, int dtype, bimamba_stream_t stream);

/* fp32-accurate products on the bf16 tensor cores (the 1e-4 parity mode and fp32 scoring, src/main.py:973-976): splits
 * an fp32 (rows, cols) matrix into three bf16 terms x = hi + mid + lo (24 bits) written as six blocks,
 *   side 0: [hi | mid | lo | hi | hi | mid]     side 1: [hi | hi | hi | mid | lo | mid]
 * block b of element (r, c) at dst[b * block_stride + r * ld_dst + c].  With block_stride = cols (ld_dst = 6 * cols) the
 * blocks extend the contraction axis of bimamba_gemm_nt: gemm_nt(split(A, 0), split(B, 1)) = A . B^T to ~2^-24; with
 * block_stride = rows * ld_dst they extend the row axis bimamba_gemm_tn contracts over. */
int bimamba_split3_bf16(const float* src, void* dst, int64_t rows, int cols, int64_t ld_src, int64_t ld_dst,
                        int64_t block_stride, int side, bimamba_stream_t stream);

/* dst = cast(src) over n contiguous elements (16-byte aligned bases): the dtype changes at the edges of a layer's
 * 16-bit region (autocast of src/main.py:1049). */
int bimamba_cast(const void* src, void* dst, int64_t n, int src_dtype, int dst_dtype, bimamba_stream_t stream);

/* Mean-of-squares loss pieces (the benchmark's synthetic loss on the backend output): per-CTA partial sums of x^2
 * (each multiplied by `scale`, e.g. 1/n; nslices = bimamba_sumsq_slices(n) floats; finish with bimamba_reduce_partials) and dx = g[0] * scale * x with g on
 * the device. */
int bimamba_sumsq_slices(int64_t n);
int bimamba_sumsq(const void* x, float* part, int64_t n, float scale, int dtype, bimamba_stream_t stream);
int bimamba_scale_by(const void* x, const float* g, void* dx, int64_t n, float scale, int dtype, bimamba_stream_t stream);

/* Channel-group sum of the backward scan's [dB | dC] partial rows, written into the first 32 columns of a row matrix:
 *   out[(g * nrows + r) * out_ld + c] = sum_{i < nparts} part[((g * nparts + i) * nrows + r) * 32 + c],  c < 32
 * (groups = batch, nparts = ngroups of bimamba_scan_plan, nrows = L * ndir).  `out` is the (batch*L*ndir, 48) operand
 * [dB | dC | ddt_r | 0] of the x_proj backward (autograd of mamba_block.py:73-75) in out_dtype, so no concatenation is
 * needed; fixed summation order (deterministic). */
int bimamba_reduce_rows32(const float* part, void* out, int64_t groups, int nparts, int64_t nrows, int64_t out_ld,
                          int out_dtype, bimamba_stream_t stream);

/* One launch that turns a block's raw fp32 parameter-gradient buffers into the reference's parameter layouts
 * (mamba_block.py:22-39): dA_log = dA * A (A = -exp(A_log), :82); x_proj.weight rows [dt_r | B | C] from the repacked
 * (48, D) [B | C | dt_r | 0]; dt_proj.weight (D, R) = columns 2N..2N+R of dWdt_full (D, 48); out_proj.weight (dm, D) =
 * sum over the ndir column blocks of dWo2 (dm, ndir*D); conv1d.weight (D, 1, K) and conv1d.bias (D) from dwb (D, K+1). */
int bimamba_finalize_param_grads(const float* dA, const float* A, const float* dWxp, const float* dWdt_full,
                                 const float* dWo2, const float* dwb, float* dA_log, float* dWx, float* dWdt,
                                 float* dWo, float* dconv_w, float* dconv_b, int d_model, int d_inner, int d_state,
                                 int dt_rank, int ndir, int d_conv, bimamba_stream_t stream);

/* ---- The whole Mamba block of one encoder layer in ONE call each way (SURVEY 8b: `conv_scan_bi` together with
 * gemm_{in,x,out}_proj and their data / weight gradients), for hosts without an autograd framework.
 *   forward:  out = M(x) [+ flip(M(flip x))]   mamba_block.py:41-63 for M; DualStreamSEMamba.py:473-481 for the directions
 *             in_proj -> conv + SiLU (both directions from one read) -> x_proj -> dt_proj + softplus + scan + D skip +
 *             z gate (both directions, one launch) -> out_proj over [y_fwd | y_rev]:  5 kernels on `stream`
 *   backward: the autograd of the above with every parameter gradient in the reference's layouts (mamba_block.py:22-39).
 * x is the block's input AFTER norm1 (DualStreamSEMamba.py:472); activations are bf16 or fp16, contiguous
 * (batch, seqlen, d_model); d_model and d_inner must be multiples of 8; d_state is 16.  Weights in io_dtype are the
 * arrangements bimamba_pack_weights writes.  The forward keeps xz, xc, the x_proj rows, y (and, with
 * save_for_backward, the scan checkpoints and the ungated y) in `workspace` (256-byte aligned,
 * bimamba_block_fwd_workspace_bytes); the backward reads them from there and needs a scratch workspace of its own.
 * Same kernels, same order of arithmetic as the Python autograd Function (ops.py: BiMambaInnerFn): results are
 * bitwise identical to it. */
typedef struct bimamba_block_desc {
  const void* x;          /* (batch, seqlen, d_model)                                                   */
  void* out;              /* (batch, seqlen, d_model)                                                   */
  const void* Wi;         /* (2*d_inner, d_model)        in_proj.weight                                 */
  const void* Wxp;        /* (48, d_inner)               x_proj.weight repacked [B | C | dt_r | 0]     */
  const void* Wo2;        /* (d_model, ndir*d_inner)     [out_proj.weight] x ndir                       */
  const float* Wdt;       /* (d_inner, dt_rank) fp32     dt_proj.weight                                 */
  const float* A;         /* (d_inner, 16) fp32          -exp(A_log)                                    */
  const float* D;         /* (d_inner) fp32                                                             */
  const float* dt_bias;   /* (d_inner) fp32              dt_proj.bias                                   */
  const float* conv_w;    /* (d_inner, d_conv) fp32      conv1d.weight                                  */
  const float* conv_b;    /* (d_inner) fp32              conv1d.bias                                    */
  void* workspace;        /* saved activations, bimamba_block_fwd_workspace_bytes(...) bytes            */
  size_t workspace_bytes;
  int32_t batch, seqlen, d_model, d_inner, dt_rank, d_conv, ndir, io_dtype;
  int32_t save_for_backward; /* != 0: the forward also writes the scan checkpoints and the ungated y    */
  int32_t reserved0;
} bimamba_block_desc;

typedef struct bimamba_block_grads {
  const void* dout;       /* (batch, seqlen, d_model) io_dtype: gradient of the block output            */
  void* dx;               /* (batch, seqlen, d_model) io_dtype                                          */
  const void* WiT;        /* (d_model, 2*d_inner)  transposed arrangements of bimamba_pack_weights      */
  const void* WxpT;       /* (d_inner, 48)                                                              */
  const void* WoT;        /* (d_inner, d_model)                                                         */
  const void* WdT;        /* (16, d_inner)                                                              */
  float* dW_in;           /* (2*d_inner, d_model)   fp32 parameter gradients, the reference's shapes    */
  float* dconv_w;         /* (d_inner, 1, d_conv)                                                       */
  float* dconv_b;         /* (d_inner)                                                                  */
  float* dW_x;            /* (dt_rank + 32, d_inner)  rows [dt_r | B | C]                               */
  float* dW_dt;           /* (d_inner, dt_rank)                                                         */
  float* db_dt;           /* (d_inner)                                                                  */
  float* dA_log;          /* (d_inner, 16)                                                              */
  float* dD;              /* (d_inner)                                                                  */
  float* dW_out;          /* (d_model, d_inner)                                                         */
  void* workspace;        /* scratch, bimamba_block_bwd_workspace_bytes(...) bytes, 256-byte aligned    */
  size_t workspace_bytes;
} bimamba_block_grads;

size_t bimamba_block_fwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int ndir, int io_dtype,
                                         int save_for_backward);
size_t bimamba_block_bwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int d_conv, int ndir,
                                         int io_dtype);
int bimamba_block_fwd(const bimamba_block_desc* d, bimamba_stream_t stream);
/* Per-utterance frame counts (see bimamba_selective_scan_fwd_varlen); d->save_for_backward must be 0.  Output rows at
 * padded frames are unspecified. */
int bimamba_block_fwd_varlen(const bimamba_block_desc* d, const int32_t* seqlens, bimamba_stream_t stream);
/* `d` is the descriptor the forward ran with (same workspace, save_for_backward != 0). */
int bimamba_block_bwd(const bimamba_block_desc* d, const bimamba_block_grads* g, bimamba_stream_t stream);
/* Variable-length training (see "Variable-length training" above): the forward accepts save_for_backward, and the
 * backward takes the seqlens the forward ran with.  These calls do not mask: padded input rows never reach a valid
 * output or a gradient through the conv and the scan, but the products run over every row, so a host masks x with
 * bimamba_mask_frames before the forward (NaN padding would otherwise reach dW_in) and may mask dout before the backward.
 * Output rows at padded frames are zero (the scan writes zeros there and out_proj has no bias). */
int bimamba_block_fwd_varlen_train(const bimamba_block_desc* d, const int32_t* seqlens, bimamba_stream_t stream);
int bimamba_block_bwd_varlen(const bimamba_block_desc* d, const bimamba_block_grads* g, const int32_t* seqlens,
                             bimamba_stream_t stream);

/* ---- A second stream for the work that depends on the parameters only or produces parameter gradients.  The
 * *_side calls fork it from `stream` with cudaEventRecord / cudaStreamWaitEvent and join it before they return, so
 * they are safe under stream capture and their results are bitwise those of the single-stream calls (same kernels, same
 * inputs).  `stream` NULL, or a NULL pointer to this struct: everything runs on `stream` in the single-stream order.
 * The three events are the caller's (cudaEventCreateWithFlags(.., cudaEventDisableTiming)); calls that share them must
 * not run concurrently from different host threads. */
typedef struct bimamba_side_stream {
  bimamba_stream_t stream; /* a cudaStream_t on the same device, not `stream` itself                     */
  void* events[3];         /* cudaEvent_t                                                                */
} bimamba_side_stream;

/* The block backward with its parameter gradients on the side stream: the four weight-gradient products, the scan's and
 * the conv's parameter sums and the layout pass run beside the data chain (in_proj / x_proj / dt_proj data gradients,
 * scan and conv backward).  The block forward has no such call: its first product needs the packed weights. */
int bimamba_block_bwd_side(const bimamba_block_desc* d, const bimamba_block_grads* g, const int32_t* seqlens,
                           const bimamba_side_stream* side, bimamba_stream_t stream);

/* ---- The whole encoder layer in one call each way: PN_BiMambas_Encoder.forward (DualStreamSEMamba.py:467-486)
 *   out = FFN(LN2(M(LN1 x) + flip(M(flip(LN1 x))))) + x,   FFN = Linear(d_model, d_ff) -> GELU (erf) -> Linear(d_ff, d_model)
 * and its complete backward.  x / out / dout / dx have x_dtype: fp32 (the reference's autocast arrangement: fp32
 * residual stream, 16-bit between the norms and up to the second feed-forward product) or the 16-bit compute dtype
 * (= block.io_dtype).  `block` carries the Mamba weights, sizes, io_dtype and save_for_backward exactly as for
 * bimamba_block_fwd; its x / out / workspace fields are ignored (the layer call sets them).  LayerNorm and feed-forward
 * parameters are the fp32 masters (the call casts / transposes the two Linear weights itself, as the Python layer does
 * every step).  d_model <= 1024; d_model, d_inner, d_ff multiples of 8.  Same kernels in the same order as the Python
 * layer (encoder.py): bit-identical results. */
typedef struct bimamba_layer_desc {
  const void* x;           /* (batch, seqlen, d_model) x_dtype                                           */
  void* out;               /* (batch, seqlen, d_model) x_dtype                                           */
  const float* norm1_w;    /* (d_model) */
  const float* norm1_b;
  const float* norm2_w;
  const float* norm2_b;
  const float* ff_w1;      /* (d_ff, d_model)   feed_forward[0].weight                                   */
  const float* ff_b1;      /* (d_ff)                                                                     */
  const float* ff_w2;      /* (d_model, d_ff)   feed_forward[2].weight                                   */
  const float* ff_b2;      /* (d_model)                                                                  */
  bimamba_block_desc block;
  void* workspace;         /* bimamba_layer_fwd_workspace_bytes(...) bytes, 256-byte aligned             */
  size_t workspace_bytes;
  float eps1, eps2;        /* LayerNorm epsilons                                                         */
  int32_t d_ff, x_dtype;
} bimamba_layer_desc;

typedef struct bimamba_layer_grads {
  const void* dout;        /* (batch, seqlen, d_model) x_dtype                                           */
  void* dx;                /* (batch, seqlen, d_model) x_dtype                                           */
  float* dnorm1;           /* (2, d_model) fp32: [dweight | dbias] of norm1                              */
  float* dnorm2;           /* (2, d_model)                                                               */
  float* dff_w1;           /* (d_ff, d_model)                                                            */
  float* dff_b1;           /* (d_ff)                                                                     */
  float* dff_w2;           /* (d_model, d_ff)                                                            */
  float* dff_b2;           /* (d_model)                                                                  */
  bimamba_block_grads block; /* transposed weight arrangements + the nine Mamba gradients; dout / dx / workspace ignored */
  void* workspace;         /* scratch, bimamba_layer_bwd_workspace_bytes(...) bytes, 256-byte aligned    */
  size_t workspace_bytes;
} bimamba_layer_grads;

size_t bimamba_layer_fwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int d_ff, int ndir, int io_dtype,
                                         int save_for_backward);
size_t bimamba_layer_bwd_workspace_bytes(int batch, int seqlen, int d_model, int d_inner, int d_ff, int d_conv, int ndir,
                                         int io_dtype);
int bimamba_layer_fwd(const bimamba_layer_desc* d, bimamba_stream_t stream);
/* Per-utterance frame counts (see bimamba_selective_scan_fwd_varlen); d->block.save_for_backward must be 0.  Output
 * rows at padded frames are unspecified. */
int bimamba_layer_fwd_varlen(const bimamba_layer_desc* d, const int32_t* seqlens, bimamba_stream_t stream);
int bimamba_layer_bwd(const bimamba_layer_desc* d, const bimamba_layer_grads* g, bimamba_stream_t stream);
/* Variable-length training of the layer.  No masking inside: the masked contract (padded output frames exactly zero,
 * zero gradient at padded input frames, nothing from the padding in any parameter gradient) is
 *   bimamba_mask_frames(x) -> bimamba_layer_fwd_varlen_train -> bimamba_mask_frames(out)
 *   bimamba_mask_frames(dout) -> bimamba_layer_bwd_varlen -> (dx is then zero at padded frames). */
int bimamba_layer_fwd_varlen_train(const bimamba_layer_desc* d, const int32_t* seqlens, bimamba_stream_t stream);
int bimamba_layer_bwd_varlen(const bimamba_layer_desc* d, const bimamba_layer_grads* g, const int32_t* seqlens,
                             bimamba_stream_t stream);

/* The block's per-step weight pack (bimamba_pack_weights): fp32 masters in, the arrangements the kernels read out. */
typedef struct bimamba_block_pack {
  const float* W_in;       /* (2*d_inner, d_model)  in_proj.weight                                       */
  const float* W_x;        /* (dt_rank + 32, d_inner) x_proj.weight                                      */
  const float* W_dt;       /* (d_inner, dt_rank)     dt_proj.weight                                      */
  const float* A_log;      /* (d_inner, 16)                                                              */
  const float* W_out;      /* (d_model, d_inner)     out_proj.weight                                     */
  void* Wi;                /* outputs in block.io_dtype, layouts of bimamba_pack_weights                 */
  void* WiT;
  void* Wxp;
  void* WxpT;
  void* Wo2;
  void* WoT;
  void* WdT;
  float* A;                /* (d_inner, 16) fp32 = -exp(A_log)                                           */
} bimamba_block_pack;

/* bimamba_layer_fwd_varlen_train (seqlens may be NULL) with the weight preparation inside the call.  pack != NULL: the
 * call packs the block's weights first and uses pack->Wi, Wxp, Wo2 and A in place of d->block's (the transposed outputs
 * are the backward's WiT, WxpT, WoT, WdT).  With a side stream the pack and the feed-forward weight casts run there,
 * beside norm1, and the main stream waits for each just before the first product that reads it. */
int bimamba_layer_fwd_side(const bimamba_layer_desc* d, const bimamba_block_pack* pack, const int32_t* seqlens,
                           const bimamba_side_stream* side, bimamba_stream_t stream);
/* bimamba_layer_bwd_varlen with every parameter gradient (bias column sums, weight-gradient products, both norms'
 * dgamma / dbeta sums, the block's, see bimamba_block_bwd_side) on the side stream, joined once at the end. */
int bimamba_layer_bwd_side(const bimamba_layer_desc* d, const bimamba_layer_grads* g, const int32_t* seqlens,
                           const bimamba_side_stream* side, bimamba_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BIMAMBA_H_ */
