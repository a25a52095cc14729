// AdamW over a list of fp32 tensors in ONE launch.  sm_100a.
//
// Reference: the optimizer of the training step, torch.optim.AdamW as built in src/main.py:453 (decoupled weight
// decay, no amsgrad).  The framework's multi-tensor kernel walks 64 K-element chunks with a few dozen CTAs, which
// for the Phase-6 backend (52 small tensors, 1.25 M parameters) costs ~0.14 ms of a 2.7 ms step; here every CTA owns
// 4096 elements of one tensor ((tensor, chunk) looked up in a block map built once), so the grid has several
// hundred CTAs and the update runs at memory speed (35 MB moved).
//   p *= 1 - lr wd;  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
// lr, betas, eps, wd and the step counter live in device memory (`hyper`, `state`), so a captured CUDA graph keeps
// stepping and an LR schedule only has to overwrite hyper[0].
#include "common.cuh"

namespace bimamba {

constexpr int kAdamThreads = 256;
constexpr int kAdamChunk = 4096;   // elements per CTA

__global__ void adamw_tick_kernel(float* state) {
  pdl_prologue(); state[0] += 1.f; }

__device__ __forceinline__ void adamw_one(float& p, float g, float& m, float& v, float lr, float b1, float b2, float eps,
                                          float decay, float inv_bc1, float inv_sqrt_bc2) {
  p *= decay;
  m = fmaf(b1, m, (1.f - b1) * g);
  v = fmaf(b2, v, (1.f - b2) * g * g);
  const float denom = fmaf(sqrtf(v), inv_sqrt_bc2, eps);
  p -= lr * inv_bc1 * (m / denom);
}

__global__ void __launch_bounds__(kAdamThreads)
adamw_kernel(const bimamba_adamw_tensor* __restrict__ tab, const int2* __restrict__ blocks,
             const float* __restrict__ hyper, const float* __restrict__ state) {
  pdl_prologue();
  const int2 bm = blocks[blockIdx.x];
  const bimamba_adamw_tensor t = tab[bm.x];
  const float lr = hyper[0], b1 = hyper[1], b2 = hyper[2], eps = hyper[3], wd = hyper[4];
  // bias corrections 1 - beta^t in double: in fp32, 1 - powf(0.999f, t) keeps only about 1e-4 of its value at the first
  // steps (the rounding of beta^t near 1 against a difference of t * 1e-3), a relative error of ~1e-5 in every update
  const double step = state[0];
  const float inv_bc1 = (float)(1.0 / (1.0 - pow((double)b1, step)));
  const float inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)b2, step)));
  const float decay = 1.f - lr * wd;
  const int64_t base = (int64_t)bm.y * kAdamChunk;
  const int64_t end = min(t.n, base + kAdamChunk);
  const bool vec = ((reinterpret_cast<uintptr_t>(t.p) | reinterpret_cast<uintptr_t>(t.g) | reinterpret_cast<uintptr_t>(t.m) |
                     reinterpret_cast<uintptr_t>(t.v)) & 15) == 0;
  if (vec) {
    for (int64_t i = base + 4 * threadIdx.x; i + 3 < end; i += 4 * kAdamThreads) {
      float4 p = *reinterpret_cast<float4*>(t.p + i);
      const float4 g = *reinterpret_cast<const float4*>(t.g + i);
      float4 m = *reinterpret_cast<float4*>(t.m + i), v = *reinterpret_cast<float4*>(t.v + i);
      adamw_one(p.x, g.x, m.x, v.x, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
      adamw_one(p.y, g.y, m.y, v.y, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
      adamw_one(p.z, g.z, m.z, v.z, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
      adamw_one(p.w, g.w, m.w, v.w, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
      *reinterpret_cast<float4*>(t.p + i) = p;
      *reinterpret_cast<float4*>(t.m + i) = m;
      *reinterpret_cast<float4*>(t.v + i) = v;
    }
    const int64_t tail = base + ((end - base) & ~(int64_t)3);
    for (int64_t i = tail + threadIdx.x; i < end; i += kAdamThreads)
      adamw_one(t.p[i], t.g[i], t.m[i], t.v[i], lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
  } else {
    for (int64_t i = base + threadIdx.x; i < end; i += kAdamThreads)
      adamw_one(t.p[i], t.g[i], t.m[i], t.v[i], lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
  }
}

// ---- the fp16 recipe's optimizer step (src/main.py:1100-1117): GradScaler.unscale_ -> clip_grad_norm_ -> scaler.step
// (skipped on inf / NaN) -> scaler.update -> AveragedModel.update_parameters, on the device and capturable.
//   amp_stats_kernel + amp_finish_kernel: found_inf, the 2-norm of the unscaled gradient and the clip coefficient
//   adamw_amp_kernel: AdamW on (g * inv_scale) * coef unless found_inf, then the EMA of every parameter it owns
//   amp_update_kernel: torch._amp_update_scale_ and AveragedModel's n_averaged += 1

// Sum of one double per thread over the CTA in a fixed order (xor butterfly in each warp, then warps 0..7): the same
// bits on every run.  Valid in thread 0.
__device__ __forceinline__ double block_sum_fixed(double v) {
  __shared__ double warp_sums[kAdamThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kAdamThreads / 32; ++w) s += warp_sums[w];
  return s;
}

// torch forms the unscale factor as scale.double().reciprocal().float() (GradScaler.unscale_)
__device__ __forceinline__ float amp_inv_scale(const bimamba_amp* amp) { return (float)(1.0 / (double)amp->scale); }

// One CTA per (tensor, chunk) of the AdamW block map: the partial sum of (g * inv_scale)^2 in fp64 (the square of an
// fp32 value is exact there), or NaN when the chunk holds an inf or NaN gradient (a finite-gradient partial cannot be
// NaN: it sums non-negative terms).  Tensors without a gradient (n = 0) give 0.
__global__ void __launch_bounds__(kAdamThreads)
amp_stats_kernel(const bimamba_adamw_tensor* __restrict__ tab, const int2* __restrict__ blocks,
                 const bimamba_amp* __restrict__ amp, double* __restrict__ partial) {
  pdl_prologue();
  const int2 bm = blocks[blockIdx.x];
  const bimamba_adamw_tensor t = tab[bm.x];
  const float inv = amp_inv_scale(amp);
  const int64_t base = (int64_t)bm.y * kAdamChunk;
  const int64_t end = min(t.n, base + kAdamChunk);
  double acc = 0.0;
  bool bad = false;
  auto one = [&](float g) {
    const float u = g * inv;
    acc = fma((double)u, (double)u, acc);
    bad |= !isfinite(g);
  };
  int64_t i0 = base + threadIdx.x;
  if (aligned16(t.g)) {
    for (int64_t i = base + 4 * threadIdx.x; i + 3 < end; i += 4 * kAdamThreads) {
      const float4 g = *reinterpret_cast<const float4*>(t.g + i);
      one(g.x); one(g.y); one(g.z); one(g.w);
    }
    i0 = base + ((end - base) & ~(int64_t)3) + threadIdx.x;
  }
  for (int64_t i = i0; i < end; i += kAdamThreads) one(t.g[i]);
  bad = __syncthreads_or(bad);
  const double s = block_sum_fixed(acc);
  if (threadIdx.x == 0) partial[blockIdx.x] = bad ? __longlong_as_double(0x7ff8000000000000LL) : s;
}

// One CTA: the partials summed in a fixed order, then the record.  clip_grad_norm_'s coefficient in its own fp32
// arithmetic: max_norm * reciprocal(total_norm + 1e-6), clamped at 1 (NaN stays NaN, as torch.clamp keeps it).
__global__ void __launch_bounds__(kAdamThreads)
amp_finish_kernel(const double* __restrict__ partial, int nblocks, float max_norm, bimamba_amp* __restrict__ amp) {
  pdl_prologue();
  double s = 0.0;
  bool bad = false;
  for (int i = threadIdx.x; i < nblocks; i += kAdamThreads) {
    const double v = partial[i];
    bad |= isnan(v);
    s += v;
  }
  bad = __syncthreads_or(bad);
  s = block_sum_fixed(s);
  if (threadIdx.x == 0) {
    const float norm = (float)sqrt(s);
    float coef = 1.f;
    if (max_norm > 0.f) {
      coef = (1.f / (norm + 1e-6f)) * max_norm;
      coef = coef > 1.f ? 1.f : coef;
    }
    amp->found_inf = bad ? 1.f : 0.f;
    amp->total_norm = norm;
    amp->clip_coef = coef;
  }
}

__global__ void amp_tick_kernel(float* state, const bimamba_amp* amp) {
  pdl_prologue();
  if (amp->found_inf == 0.f) state[0] += 1.f;
}

// torch's lerp (ATen Lerp.h) with the EMA weight w = 1 - decay: ema + w (p - ema) for |w| < 0.5, else
// p - (p - ema)(1 - w); both contracted to one fma, as nvcc builds ATen's kernel
__device__ __forceinline__ float ema_one(float e, float p, float w, bool first) {
  if (first) return p;
  return fabsf(w) < 0.5f ? fmaf(w, p - e, e) : fmaf(-(p - e), 1.f - w, p);
}

// kAdam: AdamW on the gradient (g * inv_scale) * coef (the .grad unscale_ then clip_grad_norm_ leave), nothing when
// amp->found_inf is set.  kEma: then the average of every element the CTA owns moves toward the (new) parameter, also on
// a skipped step; ema[i].n is the parameter's size, which table[i].n equals unless the tensor has no gradient (0);
// ema[i].n = 0: the parameter has no average.
template <bool kAdam, bool kEma>
__global__ void __launch_bounds__(kAdamThreads)
adamw_amp_kernel(const bimamba_adamw_tensor* __restrict__ tab, const int2* __restrict__ blocks,
                 const float* __restrict__ hyper, const float* __restrict__ state, const bimamba_amp* __restrict__ amp,
                 const bimamba_ema_tensor* __restrict__ ema, const int64_t* __restrict__ n_averaged, float ema_w) {
  pdl_prologue();
  const int2 bm = blocks[blockIdx.x];
  const bimamba_adamw_tensor t = tab[bm.x];
  bool adam = false;
  float lr = 0.f, b1 = 0.f, b2 = 0.f, eps = 0.f, decay = 1.f, inv_bc1 = 1.f, inv_sqrt_bc2 = 1.f, inv = 1.f, coef = 1.f;
  if (kAdam) {
    adam = t.n > 0 && amp->found_inf == 0.f;
    lr = hyper[0]; b1 = hyper[1]; b2 = hyper[2]; eps = hyper[3];
    const float wd = hyper[4];
    const double step = state[0];
    inv_bc1 = (float)(1.0 / (1.0 - pow((double)b1, step)));
    inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)b2, step)));
    decay = 1.f - lr * wd;
    inv = amp_inv_scale(amp);
    coef = amp->clip_coef;
  }
  float* e = nullptr;
  int64_t n = adam ? t.n : 0;
  bool avg = false, first = false;
  if (kEma) {
    const bimamba_ema_tensor et = ema[bm.x];
    e = et.avg;
    avg = et.n > 0;
    n = max(n, et.n);
    first = *n_averaged == 0;
  }
  const int64_t base = (int64_t)bm.y * kAdamChunk;
  const int64_t end = min(n, base + kAdamChunk);
  auto one = [&](float& p, const float* g, float* m, float* v, float* ev) {
    if (adam) adamw_one(p, (*g * inv) * coef, *m, *v, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
    if (avg) *ev = ema_one(*ev, p, ema_w, first);
  };
  int64_t i0 = base + threadIdx.x;
  if (aligned16(t.p) && aligned16(t.g) && aligned16(t.m) && aligned16(t.v) && aligned16(e)) {
    for (int64_t i = base + 4 * threadIdx.x; i + 3 < end; i += 4 * kAdamThreads) {
      float4 p = *reinterpret_cast<float4*>(t.p + i);
      if (adam) {
        const float4 g = *reinterpret_cast<const float4*>(t.g + i);
        float4 m = *reinterpret_cast<float4*>(t.m + i), v = *reinterpret_cast<float4*>(t.v + i);
        adamw_one(p.x, (g.x * inv) * coef, m.x, v.x, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
        adamw_one(p.y, (g.y * inv) * coef, m.y, v.y, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
        adamw_one(p.z, (g.z * inv) * coef, m.z, v.z, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
        adamw_one(p.w, (g.w * inv) * coef, m.w, v.w, lr, b1, b2, eps, decay, inv_bc1, inv_sqrt_bc2);
        *reinterpret_cast<float4*>(t.p + i) = p;
        *reinterpret_cast<float4*>(t.m + i) = m;
        *reinterpret_cast<float4*>(t.v + i) = v;
      }
      if (avg) {
        float4 a = *reinterpret_cast<float4*>(e + i);
        a.x = ema_one(a.x, p.x, ema_w, first);
        a.y = ema_one(a.y, p.y, ema_w, first);
        a.z = ema_one(a.z, p.z, ema_w, first);
        a.w = ema_one(a.w, p.w, ema_w, first);
        *reinterpret_cast<float4*>(e + i) = a;
      }
    }
    i0 = base + ((end - base) & ~(int64_t)3) + threadIdx.x;
  }
  for (int64_t i = i0; i < end; i += kAdamThreads) one(t.p[i], t.g + i, t.m + i, t.v + i, e + i);
}

// torch._amp_update_scale_ (ATen AmpKernels.cu: the products in double, stored as fp32), then n_averaged += 1
__global__ void amp_update_kernel(bimamba_amp* amp, double growth_factor, double backoff_factor, int growth_interval,
                                  int64_t* n_averaged) {
  pdl_prologue();
  if (amp) {
    if (amp->found_inf != 0.f) {
      amp->scale = (float)(amp->scale * backoff_factor);
      amp->growth_tracker = 0;
    } else {
      const int successful = amp->growth_tracker + 1;
      if (successful == growth_interval) {
        const float grown = (float)(amp->scale * growth_factor);
        if (isfinite(grown)) amp->scale = grown;
        amp->growth_tracker = 0;
      } else {
        amp->growth_tracker = successful;
      }
    }
  }
  if (n_averaged) *n_averaged += 1;
}

}  // namespace bimamba

using namespace bimamba;

extern "C" int bimamba_adamw_chunk(void) { return kAdamChunk; }

extern "C" int bimamba_adamw_step(const bimamba_adamw_tensor* table, const int32_t* block_map, int nblocks,
                                  const float* hyper, float* state, bimamba_stream_t stream) {
  if (nblocks == 0) return 0;
  if (!table || !block_map || !hyper || !state || nblocks < 0) { set_err("adamw: null operand"); return -1; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  launch_k(adamw_tick_kernel, 1, 1, 0, st, state);
  launch_k(adamw_kernel, nblocks, kAdamThreads, 0, st, table, reinterpret_cast<const int2*>(block_map), hyper, state);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_amp_grad_stats(const bimamba_adamw_tensor* table, const int32_t* block_map, int nblocks,
                                      float max_norm, double* partials, bimamba_amp* amp, bimamba_stream_t stream) {
  if (!amp || nblocks < 0 || (nblocks > 0 && (!table || !block_map || !partials))) {
    set_err("amp_grad_stats: null operand"); return -1;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (nblocks > 0)
    launch_k(amp_stats_kernel, nblocks, kAdamThreads, 0, st, table, reinterpret_cast<const int2*>(block_map),
             (const bimamba_amp*)amp, partials);
  launch_k(amp_finish_kernel, 1, kAdamThreads, 0, st, (const double*)partials, nblocks, max_norm, amp);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_adamw_amp_step(const bimamba_adamw_tensor* table, const int32_t* block_map, int nblocks,
                                      const float* hyper, float* state, const bimamba_amp* amp,
                                      const bimamba_ema_tensor* ema, const int64_t* n_averaged, float ema_weight,
                                      bimamba_stream_t stream) {
  if (nblocks == 0) return 0;
  const bool adam = hyper || state || amp;
  if (!table || !block_map || nblocks < 0 || (adam && (!hyper || !state || !amp)) || (!ema != !n_averaged) ||
      (!adam && !ema)) {
    set_err("adamw_amp_step: null operand"); return -1;
  }
  if (ema && !(ema_weight >= 0.f && ema_weight <= 1.f)) { set_err("adamw_amp_step: ema_weight outside [0, 1]"); return -2; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int2* bmap = reinterpret_cast<const int2*>(block_map);
  if (adam) launch_k(amp_tick_kernel, 1, 1, 0, st, state, amp);
  if (adam && ema)
    launch_k(adamw_amp_kernel<true, true>, nblocks, kAdamThreads, 0, st, table, bmap, hyper, (const float*)state, amp, ema,
             n_averaged, ema_weight);
  else if (adam)
    launch_k(adamw_amp_kernel<true, false>, nblocks, kAdamThreads, 0, st, table, bmap, hyper, (const float*)state, amp, ema,
             n_averaged, ema_weight);
  else
    launch_k(adamw_amp_kernel<false, true>, nblocks, kAdamThreads, 0, st, table, bmap, hyper, (const float*)state, amp, ema,
             n_averaged, ema_weight);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_amp_update(bimamba_amp* amp, double growth_factor, double backoff_factor, int growth_interval,
                                  int64_t* n_averaged, bimamba_stream_t stream) {
  if (!amp && !n_averaged) { set_err("amp_update: null operand"); return -1; }
  launch_k(amp_update_kernel, 1, 1, 0, reinterpret_cast<cudaStream_t>(stream), amp, growth_factor, backoff_factor,
           growth_interval, n_averaged);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}
