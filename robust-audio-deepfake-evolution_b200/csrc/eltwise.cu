// Small element-wise / layout kernels of the encoder layer's backward and feed-forward, so that a training step contains
// no framework (ATen) kernels: exact GELU and its derivative (DualStreamSEMamba.py:462), the group sum of the scan's
// dB|dC partial rows written straight into the x_proj gradient operand, and one "finalize" launch that turns the raw
// parameter-gradient buffers of a Mamba block into the reference's parameter layouts (mamba_block.py:22-39).  sm_100a.
#include "common.cuh"

namespace bimamba {

__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad_f(float x) {
  const float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
  return fmaf(x, pdf, cdf);
}

// y = gelu(x) (kBwd = false) or y = g * gelu'(x) (kBwd = true); 16-byte vectors, grid-stride.
template <typename T, bool kBwd>
__global__ void __launch_bounds__(256) gelu_kernel(const T* __restrict__ x, const T* __restrict__ g, T* __restrict__ y, int64_t n) {
  pdl_prologue();
  constexpr int kV = 16 / sizeof(T);
  const int64_t nv = n / kV;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    T xv[kV], gv[kV], yv[kV];
    *reinterpret_cast<uint4*>(xv) = __ldg(reinterpret_cast<const uint4*>(x) + i);
    if (kBwd) *reinterpret_cast<uint4*>(gv) = __ldg(reinterpret_cast<const uint4*>(g) + i);
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const float xf = to_f(xv[k]);
      yv[k] = from_f<T>(kBwd ? to_f(gv[k]) * gelu_grad_f(xf) : gelu_f(xf));
    }
    *(reinterpret_cast<uint4*>(y) + i) = *reinterpret_cast<const uint4*>(yv);
  }
  // tail (n not a multiple of the vector width)
  for (int64_t i = nv * kV + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float xf = to_f(x[i]);
    y[i] = from_f<T>(kBwd ? to_f(g[i]) * gelu_grad_f(xf) : gelu_f(xf));
  }
}

// out[(g * nrows + r) * out_ld + c] = sum_{i < nparts} part[((g * nparts + i) * nrows + r) * 32 + c],  c < 32:
// the channel-group sum of the backward scan's [dB | dC] partial rows, written into the first 32 columns of the
// (rows, 48) x_proj gradient operand (row stride out_ld) in the GEMM's dtype.  One thread per 4 columns.
template <typename T>
__global__ void __launch_bounds__(256) reduce_rows32_kernel(const float* __restrict__ part, T* __restrict__ out, int64_t groups,
                                                            int nparts, int64_t nrows, int64_t out_ld) {
  pdl_prologue();
  const int64_t total = groups * nrows * 8;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int q = (int)(e & 7);
    const int64_t row = e >> 3, g = row / nrows, r = row - g * nrows;
    const float4* src = reinterpret_cast<const float4*>(part + ((g * nparts) * nrows + r) * 32) + q;
    float4 s = __ldg(src);
    for (int i = 1; i < nparts; ++i) {
      const float4 v = __ldg(src + (int64_t)i * nrows * 8);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    T* dst = out + row * out_ld + 4 * q;
    if constexpr (sizeof(T) == 4) {
      *reinterpret_cast<float4*>(dst) = s;
    } else {
      T v[4] = {from_f<T>(s.x), from_f<T>(s.y), from_f<T>(s.z), from_f<T>(s.w)};
      *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<const uint2*>(v);
    }
  }
}

// fp32 -> three bf16 terms, x = hi + mid + lo to 24 bits (each residual is exact in fp32), laid out as SIX blocks so
// that ONE bf16 tensor-core GEMM with fp32 accumulation over the stacked contraction axis gives an fp32-accurate
// product:   side 0: [hi | mid | lo | hi | hi | mid],  side 1: [hi | hi | hi | mid | lo | mid]
//   sum_blocks a_blk . b_blk = hi.hi + mid.hi + lo.hi + hi.mid + hi.lo + mid.mid     (dropped terms <= 2^-24 relative)
// Block b of element (r, c) goes to dst[b * block_stride + r * ld_dst + c]: block_stride = cols stacks the blocks along
// the columns (K-major operands of gemm_nt), block_stride = rows * ld_dst along the rows (gemm_tn contracts over rows).
__global__ void __launch_bounds__(256) split3_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t rows,
                                                     int cols, int64_t ld_src, int64_t ld_dst, int64_t block_stride, int side) {
  pdl_prologue();
  const int64_t total = rows * cols;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / cols;
    const int c = (int)(e - r * cols);
    const float x = __ldg(src + r * ld_src + c);
    const __nv_bfloat16 hi = __float2bfloat16_rn(x);
    const float r1 = x - __bfloat162float(hi);
    const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
    const __nv_bfloat16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
    __nv_bfloat16* d = dst + r * ld_dst + c;
    if (side == 0) {
      d[0] = hi; d[block_stride] = mid; d[2 * block_stride] = lo; d[3 * block_stride] = hi; d[4 * block_stride] = hi; d[5 * block_stride] = mid;
    } else {
      d[0] = hi; d[block_stride] = hi; d[2 * block_stride] = hi; d[3 * block_stride] = mid; d[4 * block_stride] = lo; d[5 * block_stride] = mid;
    }
  }
}

// dst = cast(src): the dtype changes at the edges of the 16-bit region of a layer (fp32 residual-stream gradient ->
// bf16 GEMM operand), 8 elements per thread.
template <typename TS, typename TD>
__global__ void __launch_bounds__(256) cast_kernel(const TS* __restrict__ src, TD* __restrict__ dst, int64_t n) {
  pdl_prologue();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 8;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += stride) {
    if (i + 8 <= n) {
      TS v[8];
      TD o[8];
      if constexpr (sizeof(TS) == 4) {
        *reinterpret_cast<uint4*>(v) = __ldg(reinterpret_cast<const uint4*>(src + i));
        *reinterpret_cast<uint4*>(v + 4) = __ldg(reinterpret_cast<const uint4*>(src + i + 4));
      } else {
        *reinterpret_cast<uint4*>(v) = __ldg(reinterpret_cast<const uint4*>(src + i));
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = from_f<TD>(to_f(v[k]));
      if constexpr (sizeof(TD) == 4) {
        *reinterpret_cast<uint4*>(dst + i) = *reinterpret_cast<const uint4*>(o);
        *reinterpret_cast<uint4*>(dst + i + 4) = *reinterpret_cast<const uint4*>(o + 4);
      } else {
        *reinterpret_cast<uint4*>(dst + i) = *reinterpret_cast<const uint4*>(o);
      }
    } else {
      for (int64_t j = i; j < n; ++j) dst[j] = from_f<TD>(to_f(src[j]));
    }
  }
}

// Mean of squares (the benchmark's / a regression loss): stage 1 = per-CTA fp32 partial sums in fixed order, finished
// by bimamba_reduce_partials; backward dx = g * 2 x / n with g read from device memory (no host sync).
template <typename T>
__global__ void __launch_bounds__(256) sumsq_kernel(const T* __restrict__ x, float* __restrict__ part, int64_t n, float scale) {
  pdl_prologue();
  __shared__ float sm[8];
  float s = 0.f;
  const int64_t chunk = (n + gridDim.x - 1) / gridDim.x;
  const int64_t lo = (int64_t)blockIdx.x * chunk, hi = lo + chunk < n ? lo + chunk : n;
  for (int64_t i = lo + threadIdx.x; i < hi; i += 256) {
    const float v = to_f(x[i]);
    s = fmaf(v, v, s);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(kFull, s, off);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += sm[w];
    part[blockIdx.x] = t * scale;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) scale_by_kernel(const T* __restrict__ x, const float* __restrict__ g, T* __restrict__ dx,
                                                       int64_t n, float scale) {
  pdl_prologue();
  const float f = __ldg(g) * scale;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dx[i] = from_f<T>(to_f(x[i]) * f);
}

struct FinalizeArgs {
  const float* dA;       // (D, N)       sum_t dh a h delta
  const float* A;        // (D, N)       -exp(A_log)
  const float* dWxp;     // (48, D)      gradient of the repacked x_proj weight [B | C | dt_r | 0]
  const float* dWdtf;    // (D, 48)      ddelta^T . [B | C | dt_r | 0] rows: columns 2N .. 2N+R are dt_proj.weight's gradient
  const float* dWo2;     // (dm, ndir*D) gradient of [W_out | W_out]
  const float* dwb;      // (D, K+1)     [conv dw | conv dbias]
  float* dA_log;         // (D, N)
  float* dWx;            // (R + 2N, D)  rows [dt_r | B | C]
  float* dWdt;           // (D, R)
  float* dWo;            // (dm, D)
  float* dcw;            // (D, K)
  float* dcb;            // (D)
  int D, N, R, dm, ndir, K;
};

__global__ void __launch_bounds__(256) finalize_kernel(const FinalizeArgs a) {
  pdl_prologue();
  const int D = a.D, N = a.N, R = a.R, dm = a.dm, K = a.K;
  const int n0 = D * N, n1 = (R + 2 * N) * D, n2 = D * R, n3 = dm * D, n4 = D * K, n5 = D;
  const int total = n0 + n1 + n2 + n3 + n4 + n5;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    int i = e;
    if (i < n0) { a.dA_log[i] = a.dA[i] * a.A[i]; continue; }                       // A = -exp(A_log): dA_log = dA * A
    i -= n0;
    if (i < n1) {                                                                   // [dt_r | B | C] <- [B | C | dt_r]
      const int r = i / D, c = i - r * D;
      const int src = r < R ? 2 * N + r : r - R;
      a.dWx[i] = a.dWxp[src * D + c];
      continue;
    }
    i -= n1;
    if (i < n2) { const int d = i / R, r = i - d * R; a.dWdt[i] = a.dWdtf[d * kXW + 2 * N + r]; continue; }
    i -= n2;
    if (i < n3) {
      const int r = i / D, c = i - r * D;
      float s = a.dWo2[(int64_t)r * a.ndir * D + c];
      if (a.ndir > 1) s += a.dWo2[(int64_t)r * a.ndir * D + D + c];
      a.dWo[i] = s;
      continue;
    }
    i -= n3;
    if (i < n4) { const int d = i / K, k = i - d * K; a.dcw[i] = a.dwb[d * (K + 1) + k]; continue; }
    i -= n4;
    a.dcb[i] = a.dwb[i * (K + 1) + K];
  }
}


// out[b, t, :] = t < len_b ? x[b, t, :] : 0 with len_b = clamp(seqlens[b], 0, T): the frame mask of variable-length
// training.  Selection, not a product: a padded frame is never loaded, so NaN or huge padding cannot pass.  kVec: rows
// of 16-byte vectors (channels a multiple of the vector width, aligned bases); out may alias x.
template <typename T, bool kVec>
__global__ void __launch_bounds__(256) mask_frames_kernel(const T* x, T* out, const int32_t* __restrict__ seqlens, int T_,
                                                          int64_t C, int64_t n) {
  pdl_prologue();
  constexpr int kV = kVec ? 16 / sizeof(T) : 1;
  const int64_t nv = n / kV, cv = C / kV;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / cv;
    const int b = (int)(row / T_), t = (int)(row - (int64_t)b * T_);
    const bool keep = t < min(max(__ldg(seqlens + b), 0), T_);
    if constexpr (kVec) {
      const uint4 v = keep ? *(reinterpret_cast<const uint4*>(x) + i) : make_uint4(0u, 0u, 0u, 0u);
      *(reinterpret_cast<uint4*>(out) + i) = v;
    } else {
      out[i] = keep ? x[i] : from_f<T>(0.f);
    }
  }
}

}  // namespace bimamba

using namespace bimamba;

static unsigned ew_blocks(int64_t work, int per_block) {
  int64_t n = (work + per_block - 1) / per_block;
  if (n < 1) n = 1;
  return (unsigned)(n > 148 * 16 ? 148 * 16 : n);
}

extern "C" int bimamba_gelu_fwd(const void* x, void* y, int64_t n, int dtype, bimamba_stream_t stream) {
  if (n == 0) return 0;
  if (!x || !y || n < 0 || dtype < 0 || dtype > 2) { set_err("gelu_fwd: bad arguments"); return -1; }
  if (!aligned16(x) || !aligned16(y)) { set_err("gelu_fwd: operands must be 16-byte aligned"); return -10; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == BIMAMBA_F32)
    launch_k(gelu_kernel<float, false>, ew_blocks(n / 4, 256), 256, 0, st, (const float*)x, nullptr, (float*)y, n);
  else if (dtype == BIMAMBA_BF16)
    launch_k(gelu_kernel<__nv_bfloat16, false>, ew_blocks(n / 8, 256), 256, 0, st, (const __nv_bfloat16*)x, nullptr, (__nv_bfloat16*)y, n);
  else
    launch_k(gelu_kernel<__half, false>, ew_blocks(n / 8, 256), 256, 0, st, (const __half*)x, nullptr, (__half*)y, n);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_gelu_bwd(const void* x, const void* dy, void* dx, int64_t n, int dtype, bimamba_stream_t stream) {
  if (n == 0) return 0;
  if (!x || !dy || !dx || n < 0 || dtype < 0 || dtype > 2) { set_err("gelu_bwd: bad arguments"); return -1; }
  if (!aligned16(x) || !aligned16(dy) || !aligned16(dx)) { set_err("gelu_bwd: operands must be 16-byte aligned"); return -10; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == BIMAMBA_F32)
    launch_k(gelu_kernel<float, true>, ew_blocks(n / 4, 256), 256, 0, st, (const float*)x, (const float*)dy, (float*)dx, n);
  else if (dtype == BIMAMBA_BF16)
    launch_k(gelu_kernel<__nv_bfloat16, true>, ew_blocks(n / 8, 256), 256, 0, st, (const __nv_bfloat16*)x, (const __nv_bfloat16*)dy, (__nv_bfloat16*)dx, n);
  else
    launch_k(gelu_kernel<__half, true>, ew_blocks(n / 8, 256), 256, 0, st, (const __half*)x, (const __half*)dy, (__half*)dx, n);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_reduce_rows32(const float* part, void* out, int64_t groups, int nparts, int64_t nrows, int64_t out_ld,
                                     int out_dtype, bimamba_stream_t stream) {
  if (groups == 0 || nrows == 0) return 0;
  if (!part || !out || groups < 0 || nparts < 1 || nrows < 0 || out_ld < 32 || out_dtype < 0 || out_dtype > 2) {
    set_err("reduce_rows32: bad arguments");
    return -1;
  }
  const int es = out_dtype == BIMAMBA_F32 ? 4 : 2;
  if (!aligned16(part) || (reinterpret_cast<uintptr_t>(out) % (4 * es)) || (out_ld % 4)) {
    set_err("reduce_rows32: misaligned operands");
    return -10;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned nb = ew_blocks(groups * nrows * 8, 256);
  if (out_dtype == BIMAMBA_F32) launch_k(reduce_rows32_kernel<float>, nb, 256, 0, st, part, (float*)out, groups, nparts, nrows, out_ld);
  else if (out_dtype == BIMAMBA_BF16) launch_k(reduce_rows32_kernel<__nv_bfloat16>, nb, 256, 0, st, part, (__nv_bfloat16*)out, groups, nparts, nrows, out_ld);
  else launch_k(reduce_rows32_kernel<__half>, nb, 256, 0, st, part, (__half*)out, groups, nparts, nrows, out_ld);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_finalize_param_grads(const float* dA, const float* A, const float* dWxp, const float* dWdt_full,
                                            const float* dWo2, const float* dwb, float* dA_log, float* dWx, float* dWdt,
                                            float* dWo, float* dconv_w, float* dconv_b, int d_model, int d_inner, int d_state,
                                            int dt_rank, int ndir, int d_conv, bimamba_stream_t stream) {
  if (!dA || !A || !dWxp || !dWdt_full || !dWo2 || !dwb || !dA_log || !dWx || !dWdt || !dWo || !dconv_w || !dconv_b) {
    set_err("finalize_param_grads: null operand");
    return -1;
  }
  if (d_model < 1 || d_inner < 1 || d_state != kN || dt_rank < 1 || dt_rank > BIMAMBA_MAX_DT_RANK || ndir < 1 || ndir > 2 || d_conv < 1) {
    set_err("finalize_param_grads: bad sizes");
    return -3;
  }
  FinalizeArgs a{dA, A, dWxp, dWdt_full, dWo2, dwb, dA_log, dWx, dWdt, dWo, dconv_w, dconv_b, d_inner, d_state, dt_rank, d_model, ndir, d_conv};
  const int total = d_inner * d_state + (dt_rank + 2 * d_state) * d_inner + d_inner * dt_rank + d_model * d_inner + d_inner * (d_conv + 1);
  launch_k(finalize_kernel, ew_blocks(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream), a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_split3_bf16(const float* src, void* dst, int64_t rows, int cols, int64_t ld_src, int64_t ld_dst,
                                   int64_t block_stride, int side, bimamba_stream_t stream) {
  if (rows == 0 || cols == 0) return 0;
  if (!src || !dst || rows < 0 || cols < 0 || side < 0 || side > 1 || ld_src < cols || ld_dst < cols || block_stride < 1) {
    set_err("split3_bf16: bad arguments");
    return -1;
  }
  launch_k(split3_kernel, ew_blocks(rows * cols, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream), 
      src, reinterpret_cast<__nv_bfloat16*>(dst), rows, cols, ld_src, ld_dst, block_stride, side);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

#define EW_DISPATCH1(DT, CALL)                                                     \
  do {                                                                             \
    if (DT == BIMAMBA_F32) { using T = float; CALL; }                               \
    else if (DT == BIMAMBA_BF16) { using T = __nv_bfloat16; CALL; }                 \
    else { using T = __half; CALL; }                                               \
  } while (0)

extern "C" int bimamba_cast(const void* src, void* dst, int64_t n, int src_dtype, int dst_dtype, bimamba_stream_t stream) {
  if (n == 0) return 0;
  if (!src || !dst || n < 0 || src_dtype < 0 || src_dtype > 2 || dst_dtype < 0 || dst_dtype > 2) { set_err("cast: bad arguments"); return -1; }
  if (!aligned16(src) || !aligned16(dst)) { set_err("cast: operands must be 16-byte aligned"); return -10; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned nb = ew_blocks((n + 7) / 8, 256);
#define CAST2(TS)                                                                                                    \
  do {                                                                                                               \
    if (dst_dtype == BIMAMBA_F32) launch_k(cast_kernel<TS, float>, nb, 256, 0, st, (const TS*)src, (float*)dst, n);   \
    else if (dst_dtype == BIMAMBA_BF16) launch_k(cast_kernel<TS, __nv_bfloat16>, nb, 256, 0, st, (const TS*)src, (__nv_bfloat16*)dst, n); \
    else launch_k(cast_kernel<TS, __half>, nb, 256, 0, st, (const TS*)src, (__half*)dst, n);                          \
  } while (0)
  if (src_dtype == BIMAMBA_F32) CAST2(float);
  else if (src_dtype == BIMAMBA_BF16) CAST2(__nv_bfloat16);
  else CAST2(__half);
#undef CAST2
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_sumsq_slices(int64_t n) {
  int64_t b = (n + 4095) / 4096;
  return (int)(b < 1 ? 1 : (b > 148 * 4 ? 148 * 4 : b));
}

extern "C" int bimamba_sumsq(const void* x, float* part, int64_t n, float scale, int dtype, bimamba_stream_t stream) {
  if (!x || !part || n < 1 || dtype < 0 || dtype > 2) { set_err("sumsq: bad arguments"); return -1; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned nb = (unsigned)bimamba_sumsq_slices(n);
  EW_DISPATCH1(dtype, (launch_k(sumsq_kernel<T>, nb, 256, 0, st, (const T*)x, part, n, scale)));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_scale_by(const void* x, const float* g, void* dx, int64_t n, float scale, int dtype,
                                bimamba_stream_t stream) {
  if (n == 0) return 0;
  if (!x || !g || !dx || n < 0 || dtype < 0 || dtype > 2) { set_err("scale_by: bad arguments"); return -1; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  EW_DISPATCH1(dtype, (launch_k(scale_by_kernel<T>, ew_blocks(n, 1024), 256, 0, st, (const T*)x, g, (T*)dx, n, scale)));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_mask_frames(const void* x, void* out, const int32_t* seqlens, int batch, int seqlen, int channels,
                                   int dtype, bimamba_stream_t stream) {
  if (batch == 0 || seqlen == 0 || channels == 0) return 0;
  if (!x || !out || !seqlens) { set_err("mask_frames: null operand"); return -1; }
  if (batch < 0 || seqlen < 0 || channels < 0 || dtype < 0 || dtype > 2) { set_err("mask_frames: bad sizes"); return -3; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t n = (int64_t)batch * seqlen * channels;
  const int kV = dtype == BIMAMBA_F32 ? 4 : 8;
  const bool vec = channels % kV == 0 && aligned16(x) && aligned16(out);
  if (vec) EW_DISPATCH1(dtype, (launch_k(mask_frames_kernel<T, true>, ew_blocks(n / kV, 256), 256, 0, st, (const T*)x, (T*)out, seqlens, seqlen, (int64_t)channels, n)));
  else EW_DISPATCH1(dtype, (launch_k(mask_frames_kernel<T, false>, ew_blocks(n, 256), 256, 0, st, (const T*)x, (T*)out, seqlens, seqlen, (int64_t)channels, n)));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}
