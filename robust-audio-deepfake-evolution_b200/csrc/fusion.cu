// Variable-length DualStreamFusion (DualStreamSEMamba.py:580-637 run on each utterance alone): the per-utterance
// interpolation of the projected SincNet branch onto the WavLM frames (:601-626) with its gather-form backward, and the
// masked time mean and channel scaling of SELayer (:524-528) with their backwards.  Utterance b is frames
// 0 .. seqlens[b]-1 of a right-padded batch; kernels clamp seqlens[b] to [0, frames] and never load a frame at or past
// it.  Arithmetic in fp32, one rounding to the storage type.  sm_100a.
#include "common.cuh"

namespace bimamba {

// ---- the interpolation index rule, per utterance (n1 WavLM frames, n2 SincNet frames), as ATen evaluates it for fp32,
// bf16 and fp16 tensors: scale = (float)n2 / n1 in fp32.  n1 == n2: copy; n1 > 4 n2 (the integer form of
// T1 / T2 > 4.0): nearest, min(floor(t * scale), n2 - 1); otherwise linear with align_corners=False,
// src = max(scale * (t + 0.5) - 0.5, 0) with the multiply-subtract fused (one rounding), i0 = floor(src),
// i1 = i0 + (i0 < n2 - 1), lambda = src - i0.  The backward finds its destination ranges with these same functions.
enum { kCopy = 0, kNearest = 1, kLinear = 2 };

__device__ __forceinline__ int interp_mode(int n1, int n2) { return n1 == n2 ? kCopy : (n1 > 4 * n2 ? kNearest : kLinear); }
__device__ __forceinline__ int nearest_src(float scale, int t, int n2) { return min((int)floorf((float)t * scale), n2 - 1); }
__device__ __forceinline__ float linear_src(float scale, int t) { return fmaxf(__fmaf_rn(scale, (float)t + 0.5f, -0.5f), 0.f); }

template <typename T, bool kVec> struct Lanes {
  static constexpr int kV = kVec ? 16 / sizeof(T) : 1;
  T v[kV];
  __device__ __forceinline__ void load(const T* p) {
    if constexpr (kVec) *reinterpret_cast<uint4*>(v) = __ldg(reinterpret_cast<const uint4*>(p));
    else v[0] = p[0];
  }
  __device__ __forceinline__ void store(T* p) const {
    if constexpr (kVec) *reinterpret_cast<uint4*>(p) = *reinterpret_cast<const uint4*>(v);
    else p[0] = v[0];
  }
};

__device__ __forceinline__ int clamp_len(const int32_t* __restrict__ seqlens, int b, int frames) {
  return min(max(__ldg(seqlens + b), 0), frames);
}

// dst[b, t, :] (t < T1) = interpolation of src[b, :n2, :] onto n1 frames at t, zero for t >= n1 (or n2 == 0).
template <typename T, bool kVec>
__global__ void __launch_bounds__(256) interp_fwd_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                         const int32_t* __restrict__ sl1, const int32_t* __restrict__ sl2,
                                                         int B, int T1, int T2, int C) {
  pdl_prologue();
  using L = Lanes<T, kVec>;
  constexpr int kV = L::kV;
  const int cv = C / kV;
  const int64_t total = (int64_t)B * T1 * cv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / cv;
    const int c = (int)(i - row * cv) * kV;
    const int b = (int)(row / T1), t = (int)(row - (int64_t)b * T1);
    const int n1 = clamp_len(sl1, b, T1), n2 = clamp_len(sl2, b, T2);
    L out;
    if (t >= n1 || n2 == 0) {
#pragma unroll
      for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(0.f);
    } else {
      const T* s = src + (int64_t)b * T2 * C + c;
      const int mode = interp_mode(n1, n2);
      const float scale = (float)n2 / (float)n1;
      if (mode == kLinear) {
        const float x = linear_src(scale, t);
        const int i0 = (int)x, i1 = i0 + (i0 < n2 - 1 ? 1 : 0);
        const float w1 = x - (float)i0, w0 = 1.f - w1;
        L a, bb;
        a.load(s + (int64_t)i0 * C);
        bb.load(s + (int64_t)i1 * C);
#pragma unroll
        for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(fmaf(w1, to_f(bb.v[k]), w0 * to_f(a.v[k])));
      } else {
        out.load(s + (int64_t)(mode == kCopy ? t : nearest_src(scale, t, n2)) * C);   // bitwise copy of the source frame
      }
    }
    out.store(dst + row * C + c);
  }
}

// dsrc[b, j, :] = sum over the destination frames t < n1 that read source frame j (increasing t) of weight * ddst[b, t, :];
// zero for j >= n2.  Deterministic (a gather, not atomics); ddst at t >= n1 is never read.
template <typename T, bool kVec>
__global__ void __launch_bounds__(256) interp_bwd_kernel(const T* __restrict__ ddst, T* __restrict__ dsrc,
                                                         const int32_t* __restrict__ sl1, const int32_t* __restrict__ sl2,
                                                         int B, int T1, int T2, int C) {
  pdl_prologue();
  using L = Lanes<T, kVec>;
  constexpr int kV = L::kV;
  const int cv = C / kV;
  const int64_t total = (int64_t)B * T2 * cv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / cv;
    const int c = (int)(i - row * cv) * kV;
    const int b = (int)(row / T2), j = (int)(row - (int64_t)b * T2);
    const int n1 = clamp_len(sl1, b, T1), n2 = clamp_len(sl2, b, T2);
    L out;
    if (j >= n2 || n1 == 0) {
#pragma unroll
      for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(0.f);
    } else if (interp_mode(n1, n2) == kCopy) {
      out.load(ddst + ((int64_t)b * T1 + j) * C + c);
    } else {
      const T* g = ddst + (int64_t)b * T1 * C + c;
      const float scale = (float)n2 / (float)n1;
      float acc[kV];
#pragma unroll
      for (int k = 0; k < kV; ++k) acc[k] = 0.f;
      L gv;
      if (interp_mode(n1, n2) == kNearest) {
        // first t with nearest_src(t) >= j: estimate, then settle on the forward's own index expression
        int t = min(max((int)ceilf((float)j / scale), 0), n1);
        while (t > 0 && nearest_src(scale, t - 1, n2) >= j) --t;
        while (t < n1 && nearest_src(scale, t, n2) < j) ++t;
        for (; t < n1 && nearest_src(scale, t, n2) == j; ++t) {
          gv.load(g + (int64_t)t * C);
#pragma unroll
          for (int k = 0; k < kV; ++k) acc[k] += to_f(gv.v[k]);
        }
      } else {
        // frames read by t have i0(t) in {j - 1, j}: first t with i0(t) >= j - 1, then while i0(t) <= j
        const int lo = j - 1;
        int t = lo <= 0 ? 0 : min(max((int)ceilf(((float)lo + 0.5f) / scale - 0.5f), 0), n1);
        while (t > 0 && (int)linear_src(scale, t - 1) >= lo) --t;
        while (t < n1 && (int)linear_src(scale, t) < lo) ++t;
        for (; t < n1; ++t) {
          const float x = linear_src(scale, t);
          const int i0 = (int)x;
          if (i0 > j) break;
          const int i1 = i0 + (i0 < n2 - 1 ? 1 : 0);
          const float w1 = x - (float)i0, w0 = 1.f - w1;
          gv.load(g + (int64_t)t * C);
#pragma unroll
          for (int k = 0; k < kV; ++k) {
            const float gk = to_f(gv.v[k]);
            if (i0 == j) acc[k] = fmaf(w0, gk, acc[k]);
            if (i1 == j) acc[k] = fmaf(w1, gk, acc[k]);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(acc[k]);
    }
    out.store(dsrc + row * C + c);
  }
}

// mean[b, c] = (sum_{t < n} x[b, t, c]) / n in fp32, 0 for n == 0.  CTA = 32 channels x 8 frame lanes; lane r sums
// frames r, r + 8, ... and the 8 lane sums are added in lane order (fixed order: deterministic).
template <typename T>
__global__ void __launch_bounds__(256) frame_mean_kernel(const T* __restrict__ x, float* __restrict__ mean,
                                                         const int32_t* __restrict__ sl, int T_, int C) {
  pdl_prologue();
  __shared__ float sm[8][33];
  const int b = blockIdx.x, c = blockIdx.y * 32 + threadIdx.x, r = threadIdx.y;
  const int n = clamp_len(sl, b, T_);
  float s = 0.f;
  if (c < C)
    for (int t = r; t < n; t += 8) s += to_f(x[((int64_t)b * T_ + t) * C + c]);
  sm[r][threadIdx.x] = s;
  __syncthreads();
  if (r == 0 && c < C) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += sm[k][threadIdx.x];
    mean[(int64_t)b * C + c] = n > 0 ? tot / (float)n : 0.f;
  }
}

// Element-wise over the padded frames: kMeanBwd = false: y = x * gate[b, c] (the SE scale, :528); kMeanBwd = true:
// y = gate[b, c] / n (the backward of the masked mean, gate = dmean; x unused).  Zero at t >= n.
template <typename T, bool kVec, bool kMeanBwd>
__global__ void __launch_bounds__(256) frame_scale_kernel(const T* __restrict__ x, const float* __restrict__ gate,
                                                          T* __restrict__ y, const int32_t* __restrict__ sl, int B, int T_,
                                                          int C) {
  pdl_prologue();
  using L = Lanes<T, kVec>;
  constexpr int kV = L::kV;
  const int cv = C / kV;
  const int64_t total = (int64_t)B * T_ * cv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / cv;
    const int c = (int)(i - row * cv) * kV;
    const int b = (int)(row / T_), t = (int)(row - (int64_t)b * T_);
    const int n = clamp_len(sl, b, T_);
    const float* g = gate + (int64_t)b * C + c;
    L out;
    if (t >= n) {
#pragma unroll
      for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(0.f);
    } else if constexpr (kMeanBwd) {
#pragma unroll
      for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(__ldg(g + k) / (float)n);
    } else {
      L a;
      a.load(x + row * C + c);
#pragma unroll
      for (int k = 0; k < kV; ++k) out.v[k] = from_f<T>(to_f(a.v[k]) * __ldg(g + k));
    }
    out.store(y + row * C + c);
  }
}

constexpr int kScaleSlice = 64;   // frames per CTA of the scale backward (one partial row of dgate each)

// Backward of frame_scale: dx = dy * gate[b] (zero at t >= n) and the partial rows
// part[b, s, c] = sum_{t in slice s, t < n} dy * x, slice s = frames 64 s .. 64 s + 63.  CTA = (utterance, slice,
// 32 channels) x 8 frame lanes; lane sums are added in lane order, the slices by bimamba_reduce_partials.
template <typename T>
__global__ void __launch_bounds__(256) frame_scale_bwd_kernel(const T* __restrict__ x, const float* __restrict__ gate,
                                                              const T* __restrict__ dy, T* __restrict__ dx,
                                                              float* __restrict__ part, const int32_t* __restrict__ sl,
                                                              int T_, int C, int nslices) {
  pdl_prologue();
  __shared__ float sm[8][33];
  const int b = blockIdx.x, s = blockIdx.y, c = blockIdx.z * 32 + threadIdx.x, r = threadIdx.y;
  const int n = clamp_len(sl, b, T_);
  const int t0 = s * kScaleSlice, t1 = min(t0 + kScaleSlice, T_);
  float acc = 0.f;
  if (c < C) {
    const float g = __ldg(gate + (int64_t)b * C + c);
    for (int t = t0 + r; t < t1; t += 8) {
      const int64_t e = ((int64_t)b * T_ + t) * C + c;
      if (t < n) {
        const float d = to_f(dy[e]);
        dx[e] = from_f<T>(d * g);
        acc = fmaf(d, to_f(x[e]), acc);
      } else {
        dx[e] = from_f<T>(0.f);
      }
    }
  }
  sm[r][threadIdx.x] = acc;
  __syncthreads();
  if (r == 0 && c < C) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += sm[k][threadIdx.x];
    part[((int64_t)b * nslices + s) * C + c] = tot;
  }
}

}  // namespace bimamba

using namespace bimamba;

static unsigned fu_blocks(int64_t work) {
  int64_t n = (work + 255) / 256;
  if (n < 1) n = 1;
  return (unsigned)(n > 148 * 16 ? 148 * 16 : n);
}

static int fu_done(void) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

#define FU_DISPATCH(DT, CALL)                                                      \
  do {                                                                             \
    if (DT == BIMAMBA_F32) { using T = float; CALL; }                               \
    else if (DT == BIMAMBA_BF16) { using T = __nv_bfloat16; CALL; }                 \
    else { using T = __half; CALL; }                                               \
  } while (0)

static bool fu_vec(int channels, int dtype, const void* a, const void* b) {
  return channels % (dtype == BIMAMBA_F32 ? 4 : 8) == 0 && aligned16(a) && aligned16(b);
}

static int fu_interp(bool bwd, const void* in, void* out, const int32_t* seqlens1, const int32_t* seqlens2, int batch,
                     int frames1, int frames2, int channels, int dtype, bimamba_stream_t stream) {
  if (batch == 0 || channels == 0 || (bwd ? frames2 : frames1) == 0) return 0;
  if (!in || !out || !seqlens1 || !seqlens2) { set_err(bwd ? "interp_frames_bwd: null operand" : "interp_frames_fwd: null operand"); return -1; }
  if (batch < 0 || frames1 < 0 || frames2 < 0 || channels < 0 || dtype < 0 || dtype > 2) {
    set_err(bwd ? "interp_frames_bwd: bad sizes" : "interp_frames_fwd: bad sizes");
    return -3;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int kV = dtype == BIMAMBA_F32 ? 4 : 8;
  const bool vec = fu_vec(channels, dtype, in, out);
  const int64_t n = (int64_t)batch * (bwd ? frames2 : frames1) * channels / (vec ? kV : 1);
  if (bwd) {
    if (vec) FU_DISPATCH(dtype, (launch_k(interp_bwd_kernel<T, true>, fu_blocks(n), 256, 0, st, (const T*)in, (T*)out, seqlens1, seqlens2, batch, frames1, frames2, channels)));
    else FU_DISPATCH(dtype, (launch_k(interp_bwd_kernel<T, false>, fu_blocks(n), 256, 0, st, (const T*)in, (T*)out, seqlens1, seqlens2, batch, frames1, frames2, channels)));
  } else {
    if (vec) FU_DISPATCH(dtype, (launch_k(interp_fwd_kernel<T, true>, fu_blocks(n), 256, 0, st, (const T*)in, (T*)out, seqlens1, seqlens2, batch, frames1, frames2, channels)));
    else FU_DISPATCH(dtype, (launch_k(interp_fwd_kernel<T, false>, fu_blocks(n), 256, 0, st, (const T*)in, (T*)out, seqlens1, seqlens2, batch, frames1, frames2, channels)));
  }
  return fu_done();
}

extern "C" int bimamba_interp_frames_fwd(const void* src, void* dst, const int32_t* seqlens_dst, const int32_t* seqlens_src,
                                         int batch, int dst_frames, int src_frames, int channels, int dtype,
                                         bimamba_stream_t stream) {
  return fu_interp(false, src, dst, seqlens_dst, seqlens_src, batch, dst_frames, src_frames, channels, dtype, stream);
}

extern "C" int bimamba_interp_frames_bwd(const void* ddst, void* dsrc, const int32_t* seqlens_dst, const int32_t* seqlens_src,
                                         int batch, int dst_frames, int src_frames, int channels, int dtype,
                                         bimamba_stream_t stream) {
  return fu_interp(true, ddst, dsrc, seqlens_dst, seqlens_src, batch, dst_frames, src_frames, channels, dtype, stream);
}

extern "C" int bimamba_frame_mean(const void* x, float* mean, const int32_t* seqlens, int batch, int seqlen, int channels,
                                  int dtype, bimamba_stream_t stream) {
  if (batch == 0 || channels == 0) return 0;
  if (!x || !mean || !seqlens) { set_err("frame_mean: null operand"); return -1; }
  if (batch < 0 || seqlen < 0 || channels < 0 || dtype < 0 || dtype > 2) { set_err("frame_mean: bad sizes"); return -3; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const dim3 grid(batch, (channels + 31) / 32), block(32, 8);
  FU_DISPATCH(dtype, (launch_k(frame_mean_kernel<T>, grid, block, 0, st, (const T*)x, mean, seqlens, seqlen, channels)));
  return fu_done();
}

extern "C" int bimamba_frame_mean_bwd(const float* dmean, void* dx, const int32_t* seqlens, int batch, int seqlen,
                                      int channels, int dtype, bimamba_stream_t stream) {
  if (batch == 0 || seqlen == 0 || channels == 0) return 0;
  if (!dmean || !dx || !seqlens) { set_err("frame_mean_bwd: null operand"); return -1; }
  if (batch < 0 || seqlen < 0 || channels < 0 || dtype < 0 || dtype > 2) { set_err("frame_mean_bwd: bad sizes"); return -3; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int kV = dtype == BIMAMBA_F32 ? 4 : 8;
  const bool vec = fu_vec(channels, dtype, dx, dx);
  const int64_t n = (int64_t)batch * seqlen * channels / (vec ? kV : 1);
  if (vec) FU_DISPATCH(dtype, (launch_k(frame_scale_kernel<T, true, true>, fu_blocks(n), 256, 0, st, (const T*)nullptr, dmean, (T*)dx, seqlens, batch, seqlen, channels)));
  else FU_DISPATCH(dtype, (launch_k(frame_scale_kernel<T, false, true>, fu_blocks(n), 256, 0, st, (const T*)nullptr, dmean, (T*)dx, seqlens, batch, seqlen, channels)));
  return fu_done();
}

extern "C" int bimamba_frame_scale(const void* x, const float* gate, void* y, const int32_t* seqlens, int batch, int seqlen,
                                   int channels, int dtype, bimamba_stream_t stream) {
  if (batch == 0 || seqlen == 0 || channels == 0) return 0;
  if (!x || !gate || !y || !seqlens) { set_err("frame_scale: null operand"); return -1; }
  if (batch < 0 || seqlen < 0 || channels < 0 || dtype < 0 || dtype > 2) { set_err("frame_scale: bad sizes"); return -3; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int kV = dtype == BIMAMBA_F32 ? 4 : 8;
  const bool vec = fu_vec(channels, dtype, x, y);
  const int64_t n = (int64_t)batch * seqlen * channels / (vec ? kV : 1);
  if (vec) FU_DISPATCH(dtype, (launch_k(frame_scale_kernel<T, true, false>, fu_blocks(n), 256, 0, st, (const T*)x, gate, (T*)y, seqlens, batch, seqlen, channels)));
  else FU_DISPATCH(dtype, (launch_k(frame_scale_kernel<T, false, false>, fu_blocks(n), 256, 0, st, (const T*)x, gate, (T*)y, seqlens, batch, seqlen, channels)));
  return fu_done();
}

extern "C" int bimamba_frame_scale_bwd_slices(int seqlen) {
  const int s = (seqlen + kScaleSlice - 1) / kScaleSlice;
  return s < 1 ? 1 : s;
}

extern "C" int bimamba_frame_scale_bwd(const void* x, const float* gate, const void* dy, void* dx, float* dgate_part,
                                       const int32_t* seqlens, int batch, int seqlen, int channels, int dtype,
                                       bimamba_stream_t stream) {
  if (batch == 0 || channels == 0) return 0;
  if (!x || !gate || !dy || !dx || !dgate_part || !seqlens) { set_err("frame_scale_bwd: null operand"); return -1; }
  if (batch < 0 || seqlen < 0 || channels < 0 || dtype < 0 || dtype > 2) {
    set_err("frame_scale_bwd: bad sizes");
    return -3;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int nsl = bimamba_frame_scale_bwd_slices(seqlen);
  const dim3 grid(batch, nsl, (channels + 31) / 32), block(32, 8);
  FU_DISPATCH(dtype, (launch_k(frame_scale_bwd_kernel<T>, grid, block, 0, st, (const T*)x, gate, (const T*)dy, (T*)dx, dgate_part, seqlens, seqlen, channels, nsl)));
  return fu_done();
}
