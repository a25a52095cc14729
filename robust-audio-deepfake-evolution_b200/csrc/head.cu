// Backend head, forward (scoring): final LayerNorm -> attention pooling over time -> classifier, one kernel.  sm_100a.
//
// Reference: src/models/DualStreamSEMamba.py:759 (norm_f), :762-763 (softmax over T of attention_pool(f), weighted sum
// of the normalised frames), :767 (classifier); dropout (:764) is the identity in eval mode, which is where this
// kernel is used (produce_evaluation_file, src/main.py:958-995: score = logits[:, 1]).
//
// One CTA per utterance.  A warp owns frames t = warp, warp + 8, ...: the frame lives in registers (C <= 256), is
// normalised there (two-pass fp32), and enters a running (max, sum, weighted-frame) triple - the frames are read
// once and the (B, T, C) normalised tensor, the (B, T) logits and the softmax never touch memory.  The eight warps'
// triples are merged in fixed order through shared memory; the classifier is two warp reductions.
#include "common.cuh"

namespace bimamba {

constexpr int kHeadWarps = 8;
constexpr int kHeadThreads = kHeadWarps * 32;

__device__ __forceinline__ float warp_sum_h(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
  return v;
}

// kVar: norm, softmax and pooling over the frames t < clamp(seqlens[b], 0, L) only; a zero-length utterance pools to
// zero features (its logits are the classifier bias).
template <typename T, int NPL, bool kVar>
__global__ void __launch_bounds__(kHeadThreads)
head_fwd_kernel(const T* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                const float* __restrict__ w_att, const float* __restrict__ b_att, const float* __restrict__ w_cls,
                const float* __restrict__ b_cls, float* __restrict__ features, float* __restrict__ logits, int L, int C,
                int ncls, float eps, const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  __shared__ float s_m[kHeadWarps], s_l[kHeadWarps];
  __shared__ float s_acc[kHeadWarps][32 * NPL];
  __shared__ float s_feat[32 * NPL];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x;
  const T* xb = x + (int64_t)b * L * C;
  float g[NPL], be[NPL], wa[NPL], acc[NPL];
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int c = lane + 32 * i;
    g[i] = c < C ? __ldg(gamma + c) : 0.f;
    be[i] = c < C ? __ldg(beta + c) : 0.f;
    wa[i] = c < C ? __ldg(w_att + c) : 0.f;
    acc[i] = 0.f;
  }
  const float ba = b_att ? __ldg(b_att) : 0.f;
  const int Lb = kVar ? min(max(__ldg(seqlens + b), 0), L) : L;
  float m = -INFINITY, l = 0.f;
  for (int t = warp; t < Lb; t += kHeadWarps) {
    const T* xr = xb + (int64_t)t * C;
    float v[NPL];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      v[i] = c < C ? to_f(xr[c]) : 0.f;
      s += v[i];
    }
    const float mu = warp_sum_h(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      const float d = c < C ? v[i] - mu : 0.f;
      q = fmaf(d, d, q);
    }
    const float rs = rsqrtf(warp_sum_h(q) / C + eps);
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      v[i] = c < C ? fmaf((v[i] - mu) * rs, g[i], be[i]) : 0.f;   // norm_f(frame)
      dot = fmaf(wa[i], v[i], dot);
    }
    const float sc = warp_sum_h(dot) + ba;                          // attention logit of this frame
    const float mn = fmaxf(m, sc);
    const float scale = ex2_approx((m - mn) * kLog2e);              // 0 on the first frame (m = -inf)
    const float pw = ex2_approx((sc - mn) * kLog2e);
    l = fmaf(l, scale, pw);
#pragma unroll
    for (int i = 0; i < NPL; ++i) acc[i] = fmaf(acc[i], scale, pw * v[i]);
    m = mn;
  }
  if (lane == 0) {
    s_m[warp] = m;
    s_l[warp] = l;
  }
#pragma unroll
  for (int i = 0; i < NPL; ++i) s_acc[warp][lane + 32 * i] = acc[i];
  __syncthreads();
  // merge the warps in fixed order
  float M = -INFINITY;
#pragma unroll
  for (int w = 0; w < kHeadWarps; ++w) M = fmaxf(M, s_m[w]);
  float den = 0.f;
#pragma unroll
  for (int w = 0; w < kHeadWarps; ++w) den += s_m[w] == -INFINITY ? 0.f : s_l[w] * ex2_approx((s_m[w] - M) * kLog2e);
  for (int c = threadIdx.x; c < C; c += kHeadThreads) {
    float num = 0.f;
#pragma unroll
    for (int w = 0; w < kHeadWarps; ++w)
      num += s_m[w] == -INFINITY ? 0.f : s_acc[w][c] * ex2_approx((s_m[w] - M) * kLog2e);
    const float f = (kVar && !(den > 0.f)) ? 0.f : num / den;
    s_feat[c] = f;
    features[(int64_t)b * C + c] = f;
  }
  __syncthreads();
  for (int j = warp; j < ncls; j += kHeadWarps) {
    float d = 0.f;
    for (int c = lane; c < C; c += 32) d = fmaf(__ldg(w_cls + (int64_t)j * C + c), s_feat[c], d);
    d = warp_sum_h(d);
    if (lane == 0) logits[(int64_t)b * ncls + j] = d + (b_cls ? __ldg(b_cls + j) : 0.f);
  }
}

// Backward of the pooled features f = sum_t softmax_t(w . y_t + b) y_t, y_t = norm_f(x_t), for the TRAINING head
// (DualStreamSEMamba.py:759-763 under autograd; dropout and the classifier (:764-767) stay outside, they act on (B, C)).
// One CTA per utterance, two passes over its frames (both hit L2): pass 1 repeats the forward's running (max, sum,
// weighted frame) merge to get M, the denominator and f; pass 2 recomputes y_t and its softmax weight a_t per frame and
// forms   ds_t = a_t (df . y_t - df . f),   dy_t = a_t df + ds_t w,   dx_t = LayerNorm backward of dy_t,
// accumulating dgamma, dbeta, dw_att (and db_att = sum_t ds_t, which is 0 up to rounding) per warp; the eight warps are
// merged in fixed order into this utterance's partial row; bimamba_reduce_partials sums over the batch.
// kVar: both passes run over t < clamp(seqlens[b], 0, L), the frames the variable-length forward pooled; dx is written as
// zeros at padded frames, and a zero-length utterance gets zero dx and a zero partial row.
template <typename T, int NPL, bool kVar>
__global__ void __launch_bounds__(kHeadThreads)
head_bwd_kernel(const T* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                const float* __restrict__ w_att, const float* __restrict__ b_att, const float* __restrict__ dfeat,
                T* __restrict__ dx, float* __restrict__ part /* (batch, 4, C) */, int L, int C, float eps,
                const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  __shared__ float s_m[kHeadWarps], s_l[kHeadWarps];
  __shared__ float s_acc[kHeadWarps][32 * NPL];
  __shared__ float s_db[kHeadWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x;
  const T* xb = x + (int64_t)b * L * C;
  T* dxb = dx + (int64_t)b * L * C;
  float g[NPL], be[NPL], wa[NPL], df[NPL], acc[NPL];
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int c = lane + 32 * i;
    g[i] = c < C ? __ldg(gamma + c) : 0.f;
    be[i] = c < C ? __ldg(beta + c) : 0.f;
    wa[i] = c < C ? __ldg(w_att + c) : 0.f;
    df[i] = c < C ? __ldg(dfeat + (int64_t)b * C + c) : 0.f;
    acc[i] = 0.f;
  }
  const float ba = b_att ? __ldg(b_att) : 0.f;
  const int Lb = kVar ? min(max(__ldg(seqlens + b), 0), L) : L;
  if (kVar) {
    for (int t = Lb + warp; t < L; t += kHeadWarps) {
      T* dr = dxb + (int64_t)t * C;
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = lane + 32 * i;
        if (c < C) dr[c] = from_f<T>(0.f);
      }
    }
  }
  // normalised frame in registers; returns the attention logit
  auto frame = [&](int t, float (&v)[NPL], float (&xh)[NPL], float& rs) -> float {
    const T* xr = xb + (int64_t)t * C;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      v[i] = c < C ? to_f(xr[c]) : 0.f;
      s += v[i];
    }
    const float mu = warp_sum_h(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      const float d = c < C ? v[i] - mu : 0.f;
      q = fmaf(d, d, q);
    }
    rs = rsqrtf(warp_sum_h(q) / C + eps);
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      xh[i] = c < C ? (v[i] - mu) * rs : 0.f;
      v[i] = c < C ? fmaf(xh[i], g[i], be[i]) : 0.f;
      dot = fmaf(wa[i], v[i], dot);
    }
    return warp_sum_h(dot) + ba;
  };
  // ---- pass 1: M, denominator, f
  float m = -INFINITY, l = 0.f;
  for (int t = warp; t < Lb; t += kHeadWarps) {
    float v[NPL], xh[NPL], rs;
    const float sc = frame(t, v, xh, rs);
    const float mn = fmaxf(m, sc);
    const float scale = ex2_approx((m - mn) * kLog2e);
    const float pw = ex2_approx((sc - mn) * kLog2e);
    l = fmaf(l, scale, pw);
#pragma unroll
    for (int i = 0; i < NPL; ++i) acc[i] = fmaf(acc[i], scale, pw * v[i]);
    m = mn;
  }
  if (lane == 0) {
    s_m[warp] = m;
    s_l[warp] = l;
  }
#pragma unroll
  for (int i = 0; i < NPL; ++i) s_acc[warp][lane + 32 * i] = acc[i];
  __syncthreads();
  float M = -INFINITY;
#pragma unroll
  for (int w = 0; w < kHeadWarps; ++w) M = fmaxf(M, s_m[w]);
  float den = 0.f;
#pragma unroll
  for (int w = 0; w < kHeadWarps; ++w) den += s_m[w] == -INFINITY ? 0.f : s_l[w] * ex2_approx((s_m[w] - M) * kLog2e);
  const float rden = 1.f / den;
  // c0 = df . f (every warp computes it the same way: fixed order)
  float c0 = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    float num = 0.f;
#pragma unroll
    for (int w = 0; w < kHeadWarps; ++w)
      num += s_m[w] == -INFINITY ? 0.f : s_acc[w][lane + 32 * i] * ex2_approx((s_m[w] - M) * kLog2e);
    c0 = fmaf(df[i], num * rden, c0);
  }
  c0 = warp_sum_h(c0);
  __syncthreads();   // s_acc is reused below
  // ---- pass 2
  float dga[NPL], dbe[NPL], dwa[NPL], dba = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i) dga[i] = dbe[i] = dwa[i] = 0.f;
  for (int t = warp; t < Lb; t += kHeadWarps) {
    float v[NPL], xh[NPL], rs;
    const float sc = frame(t, v, xh, rs);
    const float a = ex2_approx((sc - M) * kLog2e) * rden;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) q = fmaf(df[i], v[i], q);
    const float ds = a * (warp_sum_h(q) - c0);
    dba += ds;
    float s1 = 0.f, s2 = 0.f, dxh[NPL];
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const float dy = fmaf(a, df[i], ds * wa[i]);
      dga[i] = fmaf(dy, xh[i], dga[i]);
      dbe[i] += dy;
      dwa[i] = fmaf(ds, v[i], dwa[i]);
      dxh[i] = dy * g[i];
      s1 += dxh[i];
      s2 = fmaf(dxh[i], xh[i], s2);
    }
    s1 = warp_sum_h(s1) / C;
    s2 = warp_sum_h(s2) / C;
    T* dr = dxb + (int64_t)t * C;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < C) dr[c] = from_f<T>(rs * (dxh[i] - s1 - xh[i] * s2));
    }
  }
  // ---- merge the warps in fixed order: three rounds through s_acc
  float* prow = part + (int64_t)b * 4 * C;
  if (lane == 0) s_db[warp] = dba;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int i = 0; i < NPL; ++i) s_acc[warp][lane + 32 * i] = k == 0 ? dga[i] : k == 1 ? dbe[i] : dwa[i];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += kHeadThreads) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kHeadWarps; ++w) s += s_acc[w][c];
      prow[k * C + c] = s;
    }
    __syncthreads();
  }
  for (int c = threadIdx.x; c < C; c += kHeadThreads) {
    float s = 0.f;
    if (c == 0) {
#pragma unroll
      for (int w = 0; w < kHeadWarps; ++w) s += s_db[w];
    }
    prow[3 * C + c] = s;
  }
}

template <typename T>
static void launch_head(const void* x, const float* gamma, const float* beta, const float* w_att, const float* b_att,
                        const float* w_cls, const float* b_cls, float* features, float* logits, const int32_t* seqlens,
                        int batch, int L, int C, int ncls, float eps, cudaStream_t st) {
  const T* xp = reinterpret_cast<const T*>(x);
#define HEAD_FWD(NPL, VAR) launch_k(head_fwd_kernel<T, NPL, VAR>, batch, kHeadThreads, 0, st, xp, gamma, beta, w_att, b_att, w_cls, b_cls, features, logits, L, C, ncls, eps, seqlens)
  if (C <= 160) {
    if (seqlens) HEAD_FWD(5, true);
    else HEAD_FWD(5, false);
  } else {
    if (seqlens) HEAD_FWD(8, true);
    else HEAD_FWD(8, false);
  }
#undef HEAD_FWD
}

}  // namespace bimamba

using namespace bimamba;

extern "C" int bimamba_head_fwd(const void* x, const float* gamma, const float* beta, const float* w_att,
                                const float* b_att, const float* w_cls, const float* b_cls, float* features,
                                float* logits, int batch, int seqlen, int channels, int nclasses, float eps, int dtype,
                                bimamba_stream_t stream) {
  return bimamba_head_fwd_varlen(x, gamma, beta, w_att, b_att, w_cls, b_cls, features, logits, nullptr, batch, seqlen,
                                 channels, nclasses, eps, dtype, stream);
}

extern "C" int bimamba_head_fwd_varlen(const void* x, const float* gamma, const float* beta, const float* w_att,
                                       const float* b_att, const float* w_cls, const float* b_cls, float* features,
                                       float* logits, const int32_t* seqlens, int batch, int seqlen, int channels,
                                       int nclasses, float eps, int dtype, bimamba_stream_t stream) {
  if (batch == 0) return 0;
  if (!x || !gamma || !beta || !w_att || !features || (nclasses > 0 && (!w_cls || !logits))) { set_err("head: null operand"); return -1; }
  if (batch < 0 || seqlen < 1 || channels < 1 || channels > 256 || nclasses < 0) { set_err("head: seqlen >= 1, channels 1..256"); return -3; }
  if (dtype < 0 || dtype > 2) { set_err("head: bad dtype"); return -6; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == BIMAMBA_F32) launch_head<float>(x, gamma, beta, w_att, b_att, w_cls, b_cls, features, logits, seqlens, batch, seqlen, channels, nclasses, eps, st);
  else if (dtype == BIMAMBA_BF16) launch_head<__nv_bfloat16>(x, gamma, beta, w_att, b_att, w_cls, b_cls, features, logits, seqlens, batch, seqlen, channels, nclasses, eps, st);
  else launch_head<__half>(x, gamma, beta, w_att, b_att, w_cls, b_cls, features, logits, seqlens, batch, seqlen, channels, nclasses, eps, st);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_head_pool_bwd(const void* x, const float* gamma, const float* beta, const float* w_att,
                                     const float* b_att, const float* dfeatures, void* dx, float* part, int batch,
                                     int seqlen, int channels, float eps, int dtype, bimamba_stream_t stream) {
  return bimamba_head_pool_bwd_varlen(x, gamma, beta, w_att, b_att, dfeatures, dx, part, nullptr, batch, seqlen, channels,
                                      eps, dtype, stream);
}

extern "C" int bimamba_head_pool_bwd_varlen(const void* x, const float* gamma, const float* beta, const float* w_att,
                                            const float* b_att, const float* dfeatures, void* dx, float* part,
                                            const int32_t* seqlens, int batch, int seqlen, int channels, float eps,
                                            int dtype, bimamba_stream_t stream) {
  if (batch == 0) return 0;
  if (!x || !gamma || !beta || !w_att || !dfeatures || !dx || !part) { set_err("head_pool_bwd: null operand"); return -1; }
  if (batch < 0 || seqlen < 1 || channels < 1 || channels > 256) { set_err("head_pool_bwd: seqlen >= 1, channels 1..256"); return -3; }
  if (dtype < 0 || dtype > 2) { set_err("head_pool_bwd: bad dtype"); return -6; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define HEAD_BWD1(T, NPL, VAR) launch_k(head_bwd_kernel<T, NPL, VAR>, batch, kHeadThreads, 0, st, (const T*)x, gamma, beta, w_att, b_att, dfeatures, (T*)dx, part, seqlen, channels, eps, seqlens)
#define HEAD_BWD(T)                                                                                                         \
  do {                                                                                                                      \
    if (channels <= 160) {                                                                                                  \
      if (seqlens) HEAD_BWD1(T, 5, true);                                                                                   \
      else HEAD_BWD1(T, 5, false);                                                                                          \
    } else {                                                                                                                \
      if (seqlens) HEAD_BWD1(T, 8, true);                                                                                   \
      else HEAD_BWD1(T, 8, false);                                                                                          \
    }                                                                                                                       \
  } while (0)
  if (dtype == BIMAMBA_F32) HEAD_BWD(float);
  else if (dtype == BIMAMBA_BF16) HEAD_BWD(__nv_bfloat16);
  else HEAD_BWD(__half);
#undef HEAD_BWD
#undef HEAD_BWD1
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}
