// Depthwise causal conv1d (+ SiLU), channel-last, both time directions from one read of x.  sm_100a.
//
// Reference: src/models/modules/mamba_block.py:24-31 (Conv1d groups=d_inner, k=4, padding=k-1),
// :52-55 (crop to L, SiLU).  Direction 0 is that causal conv; direction 1 is the causal conv of
// the time-reversed sequence written back in natural order (taps t..t+K-1), which is what
// conv(flip(x)) of src/models/DualStreamSEMamba.py:476-478 computes.
//
// A thread owns V consecutive channels (one 8/16-byte vector of a (batch, time) row) and walks
// kSeg consecutive time steps with a register window of 2K-1 rows, producing both directions from
// one read of x.  Consecutive threads own consecutive channel vectors, so every load and store of a
// warp is one contiguous run of the row.
#include <cstdlib>
#include <initializer_list>

#include "common.cuh"

namespace bimamba {

constexpr int kSeg = 16;          // time steps per thread
constexpr int kConvThreads = 128;
constexpr int kMaxK = 4;

template <typename T, int V> struct Vec;
template <> struct Vec<float, 4> { using type = float4; };
template <> struct Vec<float, 1> { using type = float; };
template <> struct Vec<__nv_bfloat16, 4> { using type = uint2; };
template <> struct Vec<__nv_bfloat16, 1> { using type = __nv_bfloat16; };
template <> struct Vec<__half, 4> { using type = uint2; };
template <> struct Vec<__half, 1> { using type = __half; };

template <typename T, int V>
__device__ __forceinline__ void load_row(const T* __restrict__ p, float (&v)[V]) {
  using VT = typename Vec<T, V>::type;
  const VT raw = *reinterpret_cast<const VT*>(p);
  const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
  for (int i = 0; i < V; ++i) v[i] = to_f(e[i]);
}
template <typename T, int V>
__device__ __forceinline__ void store_row(T* __restrict__ p, const float (&v)[V]) {
  using VT = typename Vec<T, V>::type;
  VT raw;
  T* e = reinterpret_cast<T*>(&raw);
#pragma unroll
  for (int i = 0; i < V; ++i) e[i] = from_f<T>(v[i]);
  *reinterpret_cast<VT*>(p) = raw;
}

__device__ __forceinline__ float silu_grad(float pre) {
  const float sg = sigmoid_f(pre);
  return sg * (1.f + pre * (1.f - sg));
}

// kVar: per-utterance frame counts (seqlens, clamped to [0, L]).  Frames t >= len_b read as zero - the window is never
// loaded from them, so whatever the padding holds (NaN included) cannot reach a valid output - and the kernel writes zeros
// to both directions' padded output frames.
template <typename T, int V, int K, bool kVar>
__global__ void __launch_bounds__(kConvThreads)
conv_fwd_kernel(const T* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias, T* __restrict__ out,
                int batch, int ndir, int dim, int L, int64_t x_bs, int64_t x_ts, int64_t o_bs, int64_t o_ds,
                int64_t o_ts, int silu, const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  const int nvec = (dim + V - 1) / V;
  const int nseg = (L + kSeg - 1) / kSeg;
  const int64_t total = (int64_t)batch * nseg * nvec;
  const int64_t gid = (int64_t)blockIdx.x * kConvThreads + threadIdx.x;
  if (gid >= total) return;
  const int v = (int)(gid % nvec);
  const int s = (int)((gid / nvec) % nseg);
  const int b = (int)(gid / ((int64_t)nvec * nseg));
  const int d = v * V, t0 = s * kSeg;
  constexpr int H = K - 1;
  const int Lv = kVar ? min(max(__ldg(seqlens + b), 0), L) : L;   // frames that exist

  float wk[V][K], bs[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
#pragma unroll
    for (int k = 0; k < K; ++k) wk[i][k] = __ldg(w + (int64_t)(d + i) * K + k);
    bs[i] = bias ? __ldg(bias + d + i) : 0.f;
  }
  const T* xb = x + (int64_t)b * x_bs + d;
  // window rows: win[j] = x[t - H + j], j = 0..2H, for the current t
  float win[2 * H + 1][V];
#pragma unroll
  for (int j = 0; j < 2 * H; ++j) {
    const int t = t0 - H + j;
    if (t >= 0 && t < Lv) {
      load_row<T, V>(xb + (int64_t)t * x_ts, win[j + 1]);
    } else {
#pragma unroll
      for (int i = 0; i < V; ++i) win[j + 1][i] = 0.f;
    }
  }
#pragma unroll
  for (int s_ = 0; s_ < kSeg; ++s_) {
    const int t = t0 + s_;
    if (t >= L) break;
#pragma unroll
    for (int j = 0; j < 2 * H; ++j)
#pragma unroll
      for (int i = 0; i < V; ++i) win[j][i] = win[j + 1][i];
    const int tn = t + H;
    if (tn < Lv) {
      load_row<T, V>(xb + (int64_t)tn * x_ts, win[2 * H]);
    } else {
#pragma unroll
      for (int i = 0; i < V; ++i) win[2 * H][i] = 0.f;
    }
    float o0[V], o1[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float a0 = bs[i], a1 = bs[i];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        a0 = fmaf(wk[i][k], win[k][i], a0);           // x[t-H+k]
        a1 = fmaf(wk[i][k], win[2 * H - k][i], a1);   // x[t+H-k]
      }
      if (silu) {
        a0 *= sigmoid_f(a0);
        a1 *= sigmoid_f(a1);
      }
      o0[i] = (kVar && t >= Lv) ? 0.f : a0;
      o1[i] = (kVar && t >= Lv) ? 0.f : a1;
    }
    T* ob = out + (int64_t)b * o_bs + (int64_t)t * o_ts + d;
    store_row<T, V>(ob, o0);
    if (ndir > 1) store_row<T, V>(ob + o_ds, o1);
  }
}

// Backward, tiled through shared memory.  A CTA owns a tile of kBwdT time steps x kBwdC channels of one batch
// row: it stages x (T + 4H rows) and both directions' dout (T + 2H rows) with 16-byte cp.async - every load of
// the tile is in flight at once - converts them in place to
//   g_dir[t] = dout_dir[t] * silu'(bias + sum_k w[k] x[t -/+ (H-k)])
// and then every thread (one channel, half of the tile's steps) forms
//   dx[tau]  = sum_k w[k] ( g_0[tau+H-k] + g_1[tau-H+k] )
//   dw[k]   += sum_t g_0[t] x[t-H+k] + g_1[t] x[t+H-k];   dbias += sum_t g_0[t] + g_1[t]
// from shared memory.  dw / dbias leave as one partial row per CTA (fixed-order reduction afterwards); the sum
// of the two directions' gate gradients dz is folded into the same pass (global -> global, coalesced).
// kVar (both backward kernels): the mirror of the masked forward.  Frames t >= len_b = clamp(seqlens[b], 0, L) of x and
// dout are never loaded (they read as zero), so the padded outputs contribute nothing and the reverse direction's taps
// past len_b add nothing to dw or dbias; dx and the folded dz are written as zeros at padded frames.
constexpr int kBwdT = 16;
constexpr int kBwdC = 64;

template <typename T, int K, bool kVar>
__global__ void __launch_bounds__(kConvThreads)
conv_bwd_tile_kernel(const T* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                     const T* __restrict__ dout, T* __restrict__ dx, const T* __restrict__ dz_in, T* __restrict__ dz_out,
                     float* __restrict__ part, int batch, int ndir, int dim, int L, int64_t x_bs, int64_t x_ts,
                     int64_t g_bs, int64_t g_ds, int64_t g_ts, int64_t dx_bs, int64_t dx_ts, int silu, int vec,
                     const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  constexpr int H = K - 1;
  constexpr int XR = kBwdT + 4 * H, GR = kBwdT + 2 * H;   // rows of the x and g tiles
  constexpr int kV = 16 / sizeof(T);
  __shared__ __align__(16) T s_xraw[XR * kBwdC];
  __shared__ __align__(16) T s_graw[2 * GR * kBwdC];
  __shared__ float s_x[XR * kBwdC];
  __shared__ float s_g[2 * GR * kBwdC];
  __shared__ float s_part[2][kBwdC][K + 1];

  const int tid = threadIdx.x;
  const int nct = (dim + kBwdC - 1) / kBwdC, ntt = (L + kBwdT - 1) / kBwdT;
  const int ct = blockIdx.x % nct, tt = (blockIdx.x / nct) % ntt, b = blockIdx.x / (nct * ntt);
  const int c0 = ct * kBwdC, t0 = tt * kBwdT;
  const T* xb = x + (int64_t)b * x_bs;
  const T* gb = dout + (int64_t)b * g_bs;
  const int Lv = kVar ? min(max(__ldg(seqlens + b), 0), L) : L;   // frames that exist

  // ---- stage: x rows [t0-2H, t0+T+2H), g rows [t0-H, t0+T+H) of both directions (zero outside [0, L) x [0, dim))
  if (vec) {
    constexpr int VPR = kBwdC / kV;
    for (int e = tid; e < XR * VPR; e += kConvThreads) {
      const int r = e / VPR, v = e - r * VPR;
      const int t = t0 - 2 * H + r, c = c0 + v * kV;
      const bool ok = t >= 0 && t < Lv && c < dim;
      cp_async16(s_xraw + r * kBwdC + v * kV, ok ? xb + (int64_t)t * x_ts + c : xb, ok);
    }
    for (int e = tid; e < 2 * GR * VPR; e += kConvThreads) {
      const int dsel = e / (GR * VPR), rr = e - dsel * GR * VPR;
      const int r = rr / VPR, v = rr - r * VPR;
      const int t = t0 - H + r, c = c0 + v * kV;
      const bool ok = t >= 0 && t < Lv && c < dim && dsel < ndir;
      cp_async16(s_graw + (dsel * GR + r) * kBwdC + v * kV, ok ? gb + (int64_t)dsel * g_ds + (int64_t)t * g_ts + c : gb, ok);
    }
    cp_async_commit();
    cp_async_wait<0>();
  } else {
    for (int e = tid; e < XR * kBwdC; e += kConvThreads) {
      const int r = e / kBwdC, cc = e - r * kBwdC;
      const int t = t0 - 2 * H + r, c = c0 + cc;
      s_xraw[e] = (t >= 0 && t < Lv && c < dim) ? xb[(int64_t)t * x_ts + c] : from_f<T>(0.f);
    }
    for (int e = tid; e < 2 * GR * kBwdC; e += kConvThreads) {
      const int dsel = e / (GR * kBwdC), rr = e - dsel * GR * kBwdC;
      const int r = rr / kBwdC, cc = rr - r * kBwdC;
      const int t = t0 - H + r, c = c0 + cc;
      s_graw[e] = (t >= 0 && t < Lv && c < dim && dsel < ndir) ? gb[(int64_t)dsel * g_ds + (int64_t)t * g_ts + c] : from_f<T>(0.f);
    }
  }
  __syncthreads();
  for (int e = tid; e < XR * kBwdC; e += kConvThreads) s_x[e] = to_f(s_xraw[e]);
  __syncthreads();

  // ---- g_dir = dout_dir * silu'(pre_dir) for every staged g row (row r <-> time t0-H+r <-> x row r+H)
  {
    const int cc = tid % kBwdC;
    const int c = c0 + cc;
    float wk[K], bs = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) wk[k] = c < dim ? __ldg(w + (int64_t)c * K + k) : 0.f;
    if (bias && c < dim) bs = __ldg(bias + c);
    for (int r = tid / kBwdC; r < GR; r += kConvThreads / kBwdC) {
      float g0 = to_f(s_graw[r * kBwdC + cc]), g1 = to_f(s_graw[(GR + r) * kBwdC + cc]);
      if (silu) {
        float p0 = bs, p1 = bs;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          p0 = fmaf(wk[k], s_x[(r + H - H + k) * kBwdC + cc], p0);      // x[t-H+k], t = t0-H+r -> x row r+k
          p1 = fmaf(wk[k], s_x[(r + 2 * H - k) * kBwdC + cc], p1);      // x[t+H-k]              -> x row r+2H-k
        }
        g0 *= silu_grad(p0);
        g1 *= silu_grad(p1);
      }
      s_g[r * kBwdC + cc] = g0;
      s_g[(GR + r) * kBwdC + cc] = g1;
    }
    __syncthreads();

    // ---- dx, dw, dbias: thread = (channel cc, half hs of the tile's steps)
    const int hs = tid / kBwdC;
    float dwl[K], dbl = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) dwl[k] = 0.f;
    T* dxb = dx + (int64_t)b * dx_bs;
    constexpr int SPT = kBwdT / (kConvThreads / kBwdC);   // steps per thread
    for (int i = hs * SPT; i < (hs + 1) * SPT; ++i) {
      const int tau = t0 + i;
      if (tau >= L) break;
      // g rows: time tau <-> row i+H;  x rows: time tau <-> row i+2H
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        acc = fmaf(wk[k], s_g[(i + H + H - k) * kBwdC + cc], acc);          // g_0[tau+H-k]
        acc = fmaf(wk[k], s_g[(GR + i + H - H + k) * kBwdC + cc], acc);     // g_1[tau-H+k]
      }
      const float g0 = s_g[(i + H) * kBwdC + cc], g1 = s_g[(GR + i + H) * kBwdC + cc];
      dbl += g0 + g1;
#pragma unroll
      for (int k = 0; k < K; ++k)
        dwl[k] += g0 * s_x[(i + 2 * H - H + k) * kBwdC + cc] + g1 * s_x[(i + 2 * H + H - k) * kBwdC + cc];
      if (c < dim) {
        const bool pad = kVar && tau >= Lv;
        dxb[(int64_t)tau * dx_ts + c] = from_f<T>(pad ? 0.f : acc);
        if (dz_in) {
          float zz = 0.f;
          if (!pad) {
            const T* zi = dz_in + (int64_t)b * g_bs + (int64_t)tau * g_ts + c;
            zz = to_f(zi[0]);
            if (ndir > 1) zz += to_f(zi[g_ds]);
          }
          dz_out[(int64_t)b * dx_bs + (int64_t)tau * dx_ts + c] = from_f<T>(zz);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) s_part[hs][cc][k] = dwl[k];
    s_part[hs][cc][K] = dbl;
    __syncthreads();
    if (hs == 0 && c < dim) {
      float* o = part + ((int64_t)(b * ntt + tt) * dim + c) * (K + 1);
#pragma unroll
      for (int k = 0; k <= K; ++k) o[k] = s_part[0][cc][k] + s_part[1][cc][k];
    }
  }
}

// out[g*out_gs + j] (+)= sum_i part[g*part_gs + i*row_stride + j]
// Block = (256 / RL columns) x (RL row lanes); row lane r sums rows r, r+RL, ... in order and the
// lanes are combined in order through shared memory, so the result does not depend on timing.
template <int RL>
__global__ void __launch_bounds__(256)
reduce_kernel(const float* __restrict__ part, void* __restrict__ out, int64_t groups, int64_t rows, int64_t cols,
              int64_t part_gs, int64_t row_stride, int64_t out_gs, int dt, int accumulate) {
  pdl_prologue();
  constexpr int CPB = 256 / RL;
  __shared__ float sm[RL][CPB + 1];
  const int cx = threadIdx.x % CPB, ry = threadIdx.x / CPB;
  const int64_t tiles = (cols + CPB - 1) / CPB;
  for (int64_t bid = blockIdx.x; bid < groups * tiles; bid += gridDim.x) {
    const int64_t g = bid / tiles, j = (bid - g * tiles) * CPB + cx;
    float s = 0.f;
    if (j < cols) {
      const float* src = part + g * part_gs + j;
      for (int64_t i = ry; i < rows; i += RL) s += __ldg(src + i * row_stride);
    }
    if (RL > 1) {
      sm[ry][cx] = s;
      __syncthreads();
      if (ry == 0) {
#pragma unroll
        for (int r = 1; r < RL; ++r) s += sm[r][cx];
      }
    }
    if (ry == 0 && j < cols) {
      if (accumulate) s += ld_f(out, g * out_gs + j, dt);
      st_f(out, g * out_gs + j, s, dt);
    }
    if (RL > 1) __syncthreads();
  }
}

// Column sums of a (rows, cols) activation matrix (bias gradients of the Linear layers): stage 1 writes one fp32
// partial row per slice of kColRows rows; bimamba_reduce_partials finishes the sum in fixed order.
constexpr int kColRows = 256;
template <typename T>
__global__ void __launch_bounds__(256)
colsum_kernel(const T* __restrict__ x, float* __restrict__ part, int64_t rows, int cols, int64_t ld) {
  pdl_prologue();
  __shared__ float sm[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  const int64_t r0 = (int64_t)blockIdx.y * kColRows;
  float s = 0.f;
  if (col < cols) {
#pragma unroll 4
    for (int i = ry; i < kColRows; i += 8) {
      const int64_t r = r0 + i;
      if (r < rows) s += to_f(x[r * ld + col]);
    }
  }
  sm[ry][cx] = s;
  __syncthreads();
  if (ry == 0 && col < cols) {
#pragma unroll
    for (int k = 1; k < 8; ++k) s += sm[k][cx];
    part[(int64_t)blockIdx.y * cols + col] = s;
  }
}

// Backward, register-window variant (K = 4, channel vectors of 4): a thread owns 4 consecutive channels and walks one
// kBwdT-step segment of one batch row plus a K-1 step warm-up, keeping the x window x[tau..tau+3] and the last four
// g_fwd = dout_fwd silu'(pre_fwd) / g_rev values in registers.  One window serves both directions: it is exactly the
// taps of pre_fwd[tau+3] and of pre_rev[tau].  Everything is read straight from global memory in 8/16-byte row
// vectors (consecutive threads = consecutive channels), nothing goes through shared memory: ~65 instructions per
// (step, channel) against ~230 for the tile kernel above, which stays as the fallback for ragged shapes.
template <typename T, bool kVar>
__global__ void __launch_bounds__(kConvThreads)
conv_bwd_seg_kernel(const T* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                    const T* __restrict__ dout, T* __restrict__ dx, const T* __restrict__ dz_in, T* __restrict__ dz_out,
                    float* __restrict__ part, int batch, int ndir, int dim, int L, int64_t x_bs, int64_t x_ts,
                    int64_t g_bs, int64_t g_ds, int64_t g_ts, int64_t dx_bs, int64_t dx_ts, int silu,
                    const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  constexpr int K = 4, H = 3, V = 4;
  const int nvec = dim / V;
  const int nseg = (L + kBwdT - 1) / kBwdT;
  const int64_t total = (int64_t)batch * nseg * nvec;
  const int64_t gid = (int64_t)blockIdx.x * kConvThreads + threadIdx.x;
  if (gid >= total) return;
  const int cv = (int)(gid % nvec);
  const int seg = (int)((gid / nvec) % nseg);
  const int b = (int)(gid / ((int64_t)nvec * nseg));
  const int c = cv * V, t0 = seg * kBwdT, t1 = min(L, t0 + kBwdT);
  const int Lv = kVar ? min(max(__ldg(seqlens + b), 0), L) : L;   // frames that exist
  const T* xb = x + (int64_t)b * x_bs + c;
  const T* g0b = dout + (int64_t)b * g_bs + c;
  const T* g1b = ndir > 1 ? g0b + g_ds : nullptr;
  const T* z0b = dz_in ? dz_in + (int64_t)b * g_bs + c : nullptr;
  T* dxb = dx + (int64_t)b * dx_bs + c;
  T* zob = dz_out ? dz_out + (int64_t)b * dx_bs + c : nullptr;

  float wk[V][K], bs[V], dw[V][K], db[V];
#pragma unroll
  for (int v = 0; v < V; ++v) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      wk[v][k] = __ldg(w + (int64_t)(c + v) * K + k);
      dw[v][k] = 0.f;
    }
    bs[v] = bias ? __ldg(bias + c + v) : 0.f;
    db[v] = 0.f;
  }
  // windows: xw[j] = x[tau+j]; gf[j] = g_fwd[tau+j]; gr[j] = g_rev[tau-3+j]   (j = 0..3)
  float xw[K][V], gf[K][V], gr[K][V];
#pragma unroll
  for (int j = 0; j < K; ++j)
#pragma unroll
    for (int v = 0; v < V; ++v) {
      xw[j][v] = 0.f;
      gf[j][v] = 0.f;
      gr[j][v] = 0.f;
    }
  auto ldx = [&](int t, float (&o)[V]) {
    if (t >= 0 && t < Lv) load_row<T, V>(xb + (int64_t)t * x_ts, o);
    else {
#pragma unroll
      for (int v = 0; v < V; ++v) o[v] = 0.f;
    }
  };
  // x[t0-3 .. t0-1] (the first window is x[t0-3 .. t0]; its last row is loaded in the loop)
  ldx(t0 - 3, xw[1]);
  ldx(t0 - 2, xw[2]);
  ldx(t0 - 1, xw[3]);

#pragma unroll 4
  for (int tau = t0 - H; tau < t1; ++tau) {
    // slide: window becomes x[tau .. tau+3] (the rotation is free once the loop is unrolled by 4)
#pragma unroll
    for (int j = 0; j < K - 1; ++j)
#pragma unroll
      for (int v = 0; v < V; ++v) {
        xw[j][v] = xw[j + 1][v];
        gf[j][v] = gf[j + 1][v];
        gr[j][v] = gr[j + 1][v];
      }
    ldx(tau + H, xw[K - 1]);
    const int tf = tau + H;                    // time of the forward-direction value made in this iteration
    float d0[V], d1[V];
    const bool f_in = tf < Lv;                 // tf >= t0 - 0 >= 0 always
    const bool r_in = tau >= 0 && (!kVar || tau < Lv);   // tau < t1 <= L always
    if (f_in) load_row<T, V>(g0b + (int64_t)tf * g_ts, d0);
    if (r_in && g1b) load_row<T, V>(g1b + (int64_t)tau * g_ts, d1);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float gfn = f_in ? d0[v] : 0.f, grn = (r_in && g1b) ? d1[v] : 0.f;
      if (silu) {
        float p0 = bs[v], p1 = bs[v];
#pragma unroll
        for (int k = 0; k < K; ++k) {
          p0 = fmaf(wk[v][k], xw[k][v], p0);           // pre_fwd[tf]  = b + sum_k w[k] x[tf-3+k]
          p1 = fmaf(wk[v][k], xw[K - 1 - k][v], p1);   // pre_rev[tau] = b + sum_k w[k] x[tau+3-k]
        }
        gfn *= silu_grad(p0);
        grn *= silu_grad(p1);
      }
      gf[K - 1][v] = gfn;
      gr[K - 1][v] = grn;
      // parameter gradients: each value is counted by the segment that owns its time step
      const float cf = (tf >= t0 && tf < t1) ? gfn : 0.f;
      const float cr = tau >= t0 ? grn : 0.f;
      db[v] += cf + cr;
#pragma unroll
      for (int k = 0; k < K; ++k) dw[v][k] = fmaf(cf, xw[k][v], fmaf(cr, xw[K - 1 - k][v], dw[v][k]));
    }
    if (tau >= t0) {
      float o[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          acc = fmaf(wk[v][k], gf[K - 1 - k][v], acc);   // g_fwd[tau+3-k]
          acc = fmaf(wk[v][k], gr[k][v], acc);           // g_rev[tau-3+k]
        }
        o[v] = (kVar && tau >= Lv) ? 0.f : acc;
      }
      store_row<T, V>(dxb + (int64_t)tau * dx_ts, o);
      if (z0b) {
        float za[V], zb[V];
        if (kVar && tau >= Lv) {
#pragma unroll
          for (int v = 0; v < V; ++v) za[v] = 0.f;
        } else {
          load_row<T, V>(z0b + (int64_t)tau * g_ts, za);
          if (ndir > 1) {
            load_row<T, V>(z0b + g_ds + (int64_t)tau * g_ts, zb);
#pragma unroll
            for (int v = 0; v < V; ++v) za[v] += zb[v];
          }
        }
        store_row<T, V>(zob + (int64_t)tau * dx_ts, za);
      }
    }
  }
  float* o = part + ((int64_t)(b * nseg + seg) * dim + c) * (K + 1);
#pragma unroll
  for (int v = 0; v < V; ++v) {
#pragma unroll
    for (int k = 0; k < K; ++k) o[v * (K + 1) + k] = dw[v][k];
    o[v * (K + 1) + K] = db[v];
  }
}

static int conv_bwd_time_tiles(int seqlen) { return seqlen > 0 ? (seqlen + kBwdT - 1) / kBwdT : 1; }

template <typename T, int V, bool kVar>
static void launch_conv_fwd(const void* x, const float* w, const float* bias, void* out, int batch, int ndir, int dim,
                            int L, int width, int64_t x_bs, int64_t x_ts, int64_t o_bs, int64_t o_ds, int64_t o_ts,
                            int silu, const int32_t* seqlens, cudaStream_t st) {
  const int nvec = (dim + V - 1) / V, nseg = (L + kSeg - 1) / kSeg;
  const int64_t total = (int64_t)batch * nseg * nvec;
  const unsigned blocks = (unsigned)((total + kConvThreads - 1) / kConvThreads);
  const T* xp = reinterpret_cast<const T*>(x);
  T* op = reinterpret_cast<T*>(out);
  switch (width) {
    case 2: launch_k(conv_fwd_kernel<T, V, 2, kVar>, blocks, kConvThreads, 0, st, xp, w, bias, op, batch, ndir, dim, L, x_bs, x_ts, o_bs, o_ds, o_ts, silu, seqlens); break;
    case 3: launch_k(conv_fwd_kernel<T, V, 3, kVar>, blocks, kConvThreads, 0, st, xp, w, bias, op, batch, ndir, dim, L, x_bs, x_ts, o_bs, o_ds, o_ts, silu, seqlens); break;
    default: launch_k(conv_fwd_kernel<T, V, 4, kVar>, blocks, kConvThreads, 0, st, xp, w, bias, op, batch, ndir, dim, L, x_bs, x_ts, o_bs, o_ds, o_ts, silu, seqlens); break;
  }
}

template <typename T, bool kVar>
static void launch_conv_bwd(const void* x, const float* w, const float* bias, const void* dout, void* dx,
                            const void* dz_in, void* dz_out, float* part, int batch, int ndir, int dim, int L, int width,
                            int64_t x_bs, int64_t x_ts, int64_t g_bs, int64_t g_ds, int64_t g_ts, int64_t dx_bs,
                            int64_t dx_ts, int silu, int vec, const int32_t* seqlens, cudaStream_t st) {
  const int nct = (dim + kBwdC - 1) / kBwdC, ntt = conv_bwd_time_tiles(L);
  const unsigned blocks = (unsigned)((int64_t)batch * ntt * nct);
  const T* xp = reinterpret_cast<const T*>(x);
  const T* gp = reinterpret_cast<const T*>(dout);
  const T* zi = reinterpret_cast<const T*>(dz_in);
  T* dxp = reinterpret_cast<T*>(dx);
  T* zo = reinterpret_cast<T*>(dz_out);
  switch (width) {
    case 2: launch_k(conv_bwd_tile_kernel<T, 2, kVar>, blocks, kConvThreads, 0, st, xp, w, bias, gp, dxp, zi, zo, part, batch, ndir, dim, L, x_bs, x_ts, g_bs, g_ds, g_ts, dx_bs, dx_ts, silu, vec, seqlens); break;
    case 3: launch_k(conv_bwd_tile_kernel<T, 3, kVar>, blocks, kConvThreads, 0, st, xp, w, bias, gp, dxp, zi, zo, part, batch, ndir, dim, L, x_bs, x_ts, g_bs, g_ds, g_ts, dx_bs, dx_ts, silu, vec, seqlens); break;
    default: launch_k(conv_bwd_tile_kernel<T, 4, kVar>, blocks, kConvThreads, 0, st, xp, w, bias, gp, dxp, zi, zo, part, batch, ndir, dim, L, x_bs, x_ts, g_bs, g_ds, g_ts, dx_bs, dx_ts, silu, vec, seqlens); break;
  }
}

static bool vec4_ok(int dtype, int dim, std::initializer_list<const void*> ptrs, std::initializer_list<int64_t> strides) {
  const int es = dtype == BIMAMBA_F32 ? 4 : 2;
  if (dim % 4) return false;
  for (const void* p : ptrs)
    if (p && (reinterpret_cast<uintptr_t>(p) % (4 * es))) return false;
  for (int64_t s : strides)
    if (s % 4) return false;
  return true;
}

}  // namespace bimamba

using namespace bimamba;

extern "C" int bimamba_causal_conv1d_fwd(const void* x, const float* weight, const float* bias, void* out, int batch,
                                         int ndir, int dim, int seqlen, int width, int64_t x_bs, int64_t x_ts,
                                         int64_t out_bs, int64_t out_ds, int64_t out_ts, int dtype, int flags,
                                         bimamba_stream_t stream) {
  return bimamba_causal_conv1d_fwd_varlen(x, weight, bias, out, nullptr, batch, ndir, dim, seqlen, width, x_bs, x_ts,
                                          out_bs, out_ds, out_ts, dtype, flags, stream);
}

extern "C" int bimamba_causal_conv1d_fwd_varlen(const void* x, const float* weight, const float* bias, void* out,
                                                const int32_t* seqlens, int batch, int ndir, int dim, int seqlen,
                                                int width, int64_t x_bs, int64_t x_ts, int64_t out_bs, int64_t out_ds,
                                                int64_t out_ts, int dtype, int flags, bimamba_stream_t stream) {
  if (batch == 0 || seqlen == 0) return 0;
  if (!x || !weight || !out) { set_err("conv fwd: null operand"); return -1; }
  if (width < 2 || width > kMaxK) { set_err("conv width must be 2, 3 or 4"); return -2; }
  if (ndir < 1 || ndir > 2 || dtype < 0 || dtype > 2 || batch < 0 || dim < 1 || seqlen < 0) { set_err("conv fwd: bad sizes"); return -3; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int silu = flags & BIMAMBA_FLAG_SILU;
  const bool v4 = vec4_ok(dtype, dim, {x, out}, {x_bs, x_ts, out_bs, out_ds, out_ts});
#define CONV_FWD(T, V)                                                                                                     \
  do {                                                                                                                     \
    if (seqlens) launch_conv_fwd<T, V, true>(x, weight, bias, out, batch, ndir, dim, seqlen, width, x_bs, x_ts, out_bs, out_ds, out_ts, silu, seqlens, st); \
    else launch_conv_fwd<T, V, false>(x, weight, bias, out, batch, ndir, dim, seqlen, width, x_bs, x_ts, out_bs, out_ds, out_ts, silu, nullptr, st); \
  } while (0)
  if (dtype == BIMAMBA_F32) { if (v4) CONV_FWD(float, 4); else CONV_FWD(float, 1); }
  else if (dtype == BIMAMBA_BF16) { if (v4) CONV_FWD(__nv_bfloat16, 4); else CONV_FWD(__nv_bfloat16, 1); }
  else { if (v4) CONV_FWD(__half, 4); else CONV_FWD(__half, 1); }
#undef CONV_FWD
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_conv_bwd_slices(int batch, int seqlen, int dim) {
  (void)dim;
  return batch * conv_bwd_time_tiles(seqlen);
}

extern "C" int bimamba_causal_conv1d_bwd(const void* x, const float* weight, const float* bias, const void* dout, void* dx,
                                         const void* dz_in, void* dz_out, float* dwb_part, int batch, int ndir, int dim,
                                         int seqlen, int width, int64_t x_bs, int64_t x_ts, int64_t dout_bs,
                                         int64_t dout_ds, int64_t dout_ts, int64_t dx_bs, int64_t dx_ts, int dtype,
                                         int flags, bimamba_stream_t stream) {
  return bimamba_causal_conv1d_bwd_varlen(x, weight, bias, dout, dx, dz_in, dz_out, dwb_part, nullptr, batch, ndir, dim,
                                          seqlen, width, x_bs, x_ts, dout_bs, dout_ds, dout_ts, dx_bs, dx_ts, dtype, flags,
                                          stream);
}

extern "C" int bimamba_causal_conv1d_bwd_varlen(const void* x, const float* weight, const float* bias, const void* dout,
                                                void* dx, const void* dz_in, void* dz_out, float* dwb_part,
                                                const int32_t* seqlens, int batch, int ndir, int dim, int seqlen, int width,
                                                int64_t x_bs, int64_t x_ts, int64_t dout_bs, int64_t dout_ds,
                                                int64_t dout_ts, int64_t dx_bs, int64_t dx_ts, int dtype, int flags,
                                                bimamba_stream_t stream) {
  if (batch == 0 || seqlen == 0) return 0;
  if (!x || !weight || !dout || !dx || !dwb_part) { set_err("conv bwd: null operand"); return -1; }
  if ((dz_in == nullptr) != (dz_out == nullptr)) { set_err("conv bwd: dz_in and dz_out go together"); return -1; }
  if (width < 2 || width > kMaxK) { set_err("conv width must be 2, 3 or 4"); return -2; }
  if (ndir < 1 || ndir > 2 || dtype < 0 || dtype > 2 || batch < 0 || dim < 1 || seqlen < 0) { set_err("conv bwd: bad sizes"); return -3; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int silu = flags & BIMAMBA_FLAG_SILU;
  // 16-byte cp.async staging needs 16-byte aligned rows of x and dout (dx / dz are written element-wise)
  const int ev = dtype == BIMAMBA_F32 ? 4 : 8;
  const int vec = (dim % ev == 0) && (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (reinterpret_cast<uintptr_t>(dout) % 16 == 0) &&
                  (x_bs % ev == 0) && (x_ts % ev == 0) && (dout_bs % ev == 0) && (dout_ds % ev == 0) && (dout_ts % ev == 0);
  // register-window kernel: K = 4 and every row addressable as 4-channel vectors
  const bool seg4 = width == 4 && g_tune[BIMAMBA_TUNE_CONV_BWD] != 1 &&
                    vec4_ok(dtype, dim, {x, dout, dx, dz_in, dz_out}, {x_bs, x_ts, dout_bs, dout_ds, dout_ts, dx_bs, dx_ts});
  if (seg4) {
    const int64_t total = (int64_t)batch * conv_bwd_time_tiles(seqlen) * (dim / 4);
    const unsigned blocks = (unsigned)((total + kConvThreads - 1) / kConvThreads);
#define CONV_SEG(T, VAR) launch_k(conv_bwd_seg_kernel<T, VAR>, blocks, kConvThreads, 0, st, reinterpret_cast<const T*>(x), weight, bias, reinterpret_cast<const T*>(dout), reinterpret_cast<T*>(dx), reinterpret_cast<const T*>(dz_in), reinterpret_cast<T*>(dz_out), dwb_part, batch, ndir, dim, seqlen, x_bs, x_ts, dout_bs, dout_ds, dout_ts, dx_bs, dx_ts, silu, seqlens)
#define CONV_SEG2(T) do { if (seqlens) CONV_SEG(T, true); else CONV_SEG(T, false); } while (0)
    if (dtype == BIMAMBA_F32) CONV_SEG2(float);
    else if (dtype == BIMAMBA_BF16) CONV_SEG2(__nv_bfloat16);
    else CONV_SEG2(__half);
#undef CONV_SEG2
#undef CONV_SEG
    cudaError_t e2 = cudaGetLastError();
    if (e2 != cudaSuccess) { set_err(cudaGetErrorString(e2)); return (int)e2; }
    return 0;
  }
#define CONV_BWD(T, VAR) launch_conv_bwd<T, VAR>(x, weight, bias, dout, dx, dz_in, dz_out, dwb_part, batch, ndir, dim, seqlen, width, x_bs, x_ts, dout_bs, dout_ds, dout_ts, dx_bs, dx_ts, silu, vec, seqlens, st)
#define CONV_BWD2(T) do { if (seqlens) CONV_BWD(T, true); else CONV_BWD(T, false); } while (0)
  if (dtype == BIMAMBA_F32) CONV_BWD2(float);
  else if (dtype == BIMAMBA_BF16) CONV_BWD2(__nv_bfloat16);
  else CONV_BWD2(__half);
#undef CONV_BWD2
#undef CONV_BWD
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_reduce_partials(const float* part, void* out, int64_t groups, int64_t rows, int64_t cols,
                                       int64_t part_gs, int64_t row_stride, int64_t out_gs, int out_dtype, int accumulate,
                                       bimamba_stream_t stream) {
  if (groups * cols == 0) return 0;
  if (!part || !out) { set_err("reduce: null operand"); return -1; }
  if (out_dtype < 0 || out_dtype > 2 || groups < 0 || rows < 0 || cols < 0) { set_err("reduce: bad sizes"); return -2; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  auto nblocks = [&](int cpb) {
    int64_t n = groups * ((cols + cpb - 1) / cpb);
    return (unsigned)(n > 148 * 64 ? 148 * 64 : n);
  };
  if (rows <= 16)
    launch_k(reduce_kernel<1>, nblocks(256), 256, 0, st, part, out, groups, rows, cols, part_gs, row_stride, out_gs, out_dtype, accumulate);
  else if (rows <= 96)
    launch_k(reduce_kernel<8>, nblocks(32), 256, 0, st, part, out, groups, rows, cols, part_gs, row_stride, out_gs, out_dtype, accumulate);
  else
    launch_k(reduce_kernel<32>, nblocks(8), 256, 0, st, part, out, groups, rows, cols, part_gs, row_stride, out_gs, out_dtype, accumulate);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_colsum_slices(int64_t rows) { return (int)((rows + kColRows - 1) / kColRows); }

extern "C" int bimamba_colsum(const void* x, float* part, int64_t rows, int cols, int64_t ld, int dtype,
                              bimamba_stream_t stream) {
  if (rows == 0 || cols == 0) return 0;
  if (!x || !part) { set_err("colsum: null operand"); return -1; }
  if (rows < 0 || cols < 0 || dtype < 0 || dtype > 2) { set_err("colsum: bad sizes"); return -3; }
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)bimamba_colsum_slices(rows));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == BIMAMBA_F32) launch_k(colsum_kernel<float>, grid, 256, 0, st, reinterpret_cast<const float*>(x), part, rows, cols, ld);
  else if (dtype == BIMAMBA_BF16) launch_k(colsum_kernel<__nv_bfloat16>, grid, 256, 0, st, reinterpret_cast<const __nv_bfloat16*>(x), part, rows, cols, ld);
  else launch_k(colsum_kernel<__half>, grid, 256, 0, st, reinterpret_cast<const __half*>(x), part, rows, cols, ld);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}
