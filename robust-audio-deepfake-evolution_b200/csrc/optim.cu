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
