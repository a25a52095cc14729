// Selective scan, forward, both time directions in one launch.  sm_100a.
//
// Math (reference: src/models/modules/mamba_block.py:80-120 and :61; SURVEY Appendix A):
//   delta = softplus(Wdt . dtr[t] + bias)            (or softplus(delta_raw + bias) when given)
//   a[t,n] = exp(delta[t] * A[n]);  h[t,n] = a[t,n] h[t-1,n] + delta[t] B[t,n] u[t]
//   y[t] = sum_n C[t,n] h[t,n] + D u[t];  out[t] = y[t] * silu(z[t])
//
// Mapping (B200-first; not the upstream block-scan):
//   * activations are channel-last (batch, dir, time, channel).  One THREAD owns one channel of
//     one (batch, direction): its 16 states live in registers (fp32, packed as 8 float2 so the
//     recurrence issues as FMUL2 / FFMA2 - Blackwell's packed fp32 pipe) for the whole
//     sequence, so the n-sum needs no shuffles and the per-element transcendentals (softplus,
//     SiLU) are computed exactly once.  A warp reads 32 consecutive channels of a time row.
//   * time is walked in chunks of 16 steps.  The chunk's tiles - u, z (and delta when given)
//     [16 x G channels] and the per-(batch,time) projection rows [16 x (B|C|dt_r)], which are
//     shared by every channel - are staged by 16-byte cp.async into double-buffered shared
//     memory one chunk ahead of the compute; B/C/dt_r are then broadcast-read as float4.
//   * the dt projection (K = dt_rank = 9: too thin for tensor cores) is 9 FMAs per element
//     against the staged dt_r row, so delta is never written to or read from HBM.
//   * direction 1 walks the same storage back to front (t = L-1-step): flip(M(flip(x))) of
//     src/models/DualStreamSEMamba.py:476-478 with no flipped copy; both directions are
//     blockIdx.y of the same launch.
//   * small problems (fewer than ~16 warps per SM of channel lanes) and fp32 I/O use the one-warp-per-CTA kernel in
//     scan_fwd1.cu: same math, no block barrier.
//   * training forward also writes the fp32 state entering every 8-step chunk ("checkpoints",
//     (B, dir, chunk, D, 16): 64 contiguous bytes per thread) and the pre-gate y; the backward
//     recomputes the states of a chunk from its checkpoint (no (B, L, D, N) tensor).

#include "common.cuh"

namespace bimamba {

constexpr int kFwdMaxThreads = 128;

// kMode: 0 = delta given; 1 = fused dt projection with dt_rank <= 12; 2 = dt_rank <= 16.
// kVar: per-utterance frame counts, as in scan_fwd_warp_kernel (scan_fwd1.cu), checkpoint layout included.
template <typename T, int kMode, bool kGate, bool kVar>
__global__ void __launch_bounds__(kFwdMaxThreads) scan_fwd_kernel(const bimamba_scan_desc p, const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr bool expl = kMode == 0;
  constexpr int R4 = kMode == 1 ? 3 : 4;
  const int G = blockDim.x, tid = threadIdx.x;
  const int b = blockIdx.z, dir = blockIdx.y, d0 = blockIdx.x * G, d = d0 + tid;
  const bool ok = d < p.dim;
  const int L = kVar ? min(max(__ldg(seqlens + b), 0), p.seqlen) : p.seqlen;
  const int nck = (L + kT - 1) / kT, nckpt = ((kVar ? p.seqlen : L) + BIMAMBA_CKPT - 1) / BIMAMBA_CKPT;
  const bool softplus = (p.flags & BIMAMBA_FLAG_SOFTPLUS) != 0;
  const int R = expl ? 0 : p.dt_rank;

  const T* gu = reinterpret_cast<const T*>(p.u) + (int64_t)b * p.u_bs + (int64_t)dir * p.u_ds;
  const T* gz = kGate ? reinterpret_cast<const T*>(p.z) + (int64_t)b * p.z_bs + (int64_t)dir * p.z_ds : nullptr;
  const T* gd = expl ? reinterpret_cast<const T*>(p.delta) + (int64_t)b * p.delta_bs + (int64_t)dir * p.delta_ds : nullptr;
  const T* gbc = reinterpret_cast<const T*>(p.bc) + (int64_t)b * p.bc_bs + (int64_t)dir * p.bc_ds;
  const T* gdtr = expl ? nullptr : reinterpret_cast<const T*>(p.dtr) + (int64_t)b * p.dtr_bs + (int64_t)dir * p.dtr_ds;
  const int64_t obase = (int64_t)b * p.out_bs + (int64_t)dir * p.out_ds;
  if (kVar && ok) {   // padded frames
    for (int t = L; t < p.seqlen; ++t) {
      const int64_t o = obase + (int64_t)t * p.out_ts + d;
      reinterpret_cast<T*>(p.out)[o] = from_f<T>(0.f);
      if (p.ypre) reinterpret_cast<T*>(p.ypre)[o] = from_f<T>(0.f);
    }
  }

  // shared memory: [2][nact][kT*G] T | [2][kT*kXW] T | [kT*kXW] float
  constexpr int nact = 1 + (kGate ? 1 : 0) + (expl ? 1 : 0);
  T* s_act = reinterpret_cast<T*>(smem_raw);
  T* s_xr = s_act + 2 * nact * kT * G;
  float* s_xf = reinterpret_cast<float*>(s_xr + 2 * kT * kXW);

  constexpr int kV = 16 / sizeof(T);
  const bool dim_vec = (p.dim % kV) == 0;
  const bool vec_u = dim_vec && aligned16(gu + d0) && (p.u_ts % kV) == 0;
  const bool vec_z = kGate && dim_vec && aligned16(gz + d0) && (p.z_ts % kV) == 0;
  const bool vec_d = expl && dim_vec && aligned16(gd + d0) && (p.delta_ts % kV) == 0;
  const bool vec_bc = aligned16(gbc) && (p.bc_ts % kV) == 0;
  const bool vec_dtr = !expl && (p.flags & BIMAMBA_FLAG_DTR_PADDED) && aligned16(gdtr) && (p.dtr_ts % kV) == 0;

  auto stage = [&](int c0, int bf) {
    auto row_of = [&](int i) -> int64_t {
      const int tau = c0 * kT + i;
      return tau < L ? (int64_t)(dir ? (L - 1 - tau) : tau) : (int64_t)-1;
    };
    T* sa = s_act + bf * nact * kT * G;
    stage_tile(sa, G, gu, p.u_ts, kT, G, d0, p.dim, vec_u, row_of, tid, G);
    if (kGate) stage_tile(sa + kT * G, G, gz, p.z_ts, kT, G, d0, p.dim, vec_z, row_of, tid, G);
    if (expl) stage_tile(sa + (nact - 1) * kT * G, G, gd, p.delta_ts, kT, G, d0, p.dim, vec_d, row_of, tid, G);
    T* sx = s_xr + bf * kT * kXW;
    stage_tile(sx, kXW, gbc, p.bc_ts, kT, 2 * kN, 0, 2 * kN, vec_bc, row_of, tid, G);
    if (!expl) {
      const int w = vec_dtr ? 16 : R;
      stage_tile(sx + 2 * kN, kXW, gdtr, p.dtr_ts, kT, w, 0, w, vec_dtr, row_of, tid, G);
    }
    cp_async_commit();
  };

  // per-channel constants
  float2 A2[kN / 2], h[kN / 2];
  float2 wdt[2 * R4];
  float bias = 0.f, Dd = 0.f;
#pragma unroll
  for (int j = 0; j < kN / 2; ++j) {
    h[j] = make_float2(0.f, 0.f);
    A2[j] = make_float2(0.f, 0.f);
  }
#pragma unroll
  for (int q = 0; q < 2 * R4; ++q) wdt[q] = make_float2(0.f, 0.f);
  if (ok) {
#pragma unroll
    for (int j = 0; j < kN / 2; ++j) {
      A2[j].x = __ldg(p.A + (int64_t)d * kN + 2 * j) * kLog2e;
      A2[j].y = __ldg(p.A + (int64_t)d * kN + 2 * j + 1) * kLog2e;
    }
    if (p.delta_bias) bias = __ldg(p.delta_bias + d);
    if (p.D) Dd = __ldg(p.D + d);
    if (!expl) {
      float* w = reinterpret_cast<float*>(wdt);
#pragma unroll
      for (int r = 0; r < 4 * R4; ++r)
        if (r < R) w[r] = __ldg(p.Wdt + (int64_t)d * R + r);
    }
  }
  // output walks: element (t, d) with t advancing by +-1 per step
  const int64_t ostep = dir ? -p.out_ts : p.out_ts;
  int64_t opos = obase + (int64_t)(dir ? (L - 1) : 0) * p.out_ts + d;
  T* const gout = reinterpret_cast<T*>(p.out);
  T* const gyp = reinterpret_cast<T*>(p.ypre);

  if (nck > 0) stage(0, 0);
  for (int c0 = 0; c0 < nck; ++c0) {
    const int bf = c0 & 1;
    cp_async_wait<0>();
    __syncthreads();  // chunk c0 is visible; every thread is done with chunk c0-1's buffers
    if (c0 + 1 < nck) stage(c0 + 1, bf ^ 1);
    {
      const T* sx = s_xr + bf * kT * kXW;
      const int valid = 2 * kN + R;
      for (int e = tid; e < kT * kXW; e += G) {
        const int col = e % kXW;
        s_xf[e] = col < valid ? to_f(sx[e]) : 0.f;
      }
    }
    __syncthreads();
    if (ok) {
      const T* su = s_act + bf * nact * kT * G + tid;
      const int nvalid = L - c0 * kT;  // steps of this chunk that exist (>= 1)
#pragma unroll 4
      for (int i = 0; i < kT; ++i) {
        if ((i & (BIMAMBA_CKPT - 1)) == 0 && p.ckpt && i < nvalid) {  // state entering this 8-step chunk
          float4* ck = reinterpret_cast<float4*>(
              p.ckpt + ((((int64_t)b * p.ndir + dir) * nckpt + (c0 * kT + i) / BIMAMBA_CKPT) * p.dim + d) * kN);
#pragma unroll
          for (int q = 0; q < 4; ++q) ck[q] = make_float4(h[2 * q].x, h[2 * q].y, h[2 * q + 1].x, h[2 * q + 1].y);
        }
        const float4* xr = reinterpret_cast<const float4*>(s_xf + i * kXW);
        const float u = to_f(su[i * G]);
        float draw;
        if (expl) {
          draw = bias + to_f(su[((nact - 1) * kT + i) * G]);
        } else {
          float2 acc0 = make_float2(bias, 0.f), acc1 = make_float2(0.f, 0.f);
#pragma unroll
          for (int q = 0; q < R4; ++q) {
            const float4 x = xr[8 + q];
            acc0 = __ffma2_rn(wdt[2 * q], make_float2(x.x, x.y), acc0);
            acc1 = __ffma2_rn(wdt[2 * q + 1], make_float2(x.z, x.w), acc1);
          }
          draw = (acc0.x + acc0.y) + (acc1.x + acc1.y);
        }
        const float delta = softplus ? softplus_f(draw) : draw;
        const float du = delta * u;
        const float2 dd = make_float2(delta, delta), duu = make_float2(du, du);
        float2 ya = make_float2(0.f, 0.f), yb = make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 Bq = xr[q], Cq = xr[4 + q];
          {
            const float2 x = __fmul2_rn(dd, A2[2 * q]);
            const float2 a = make_float2(ex2_approx(x.x), ex2_approx(x.y));
            h[2 * q] = __ffma2_rn(a, h[2 * q], __fmul2_rn(duu, make_float2(Bq.x, Bq.y)));
            ya = __ffma2_rn(make_float2(Cq.x, Cq.y), h[2 * q], ya);
          }
          {
            const float2 x = __fmul2_rn(dd, A2[2 * q + 1]);
            const float2 a = make_float2(ex2_approx(x.x), ex2_approx(x.y));
            h[2 * q + 1] = __ffma2_rn(a, h[2 * q + 1], __fmul2_rn(duu, make_float2(Bq.z, Bq.w)));
            yb = __ffma2_rn(make_float2(Cq.z, Cq.w), h[2 * q + 1], yb);
          }
        }
        float y = fmaf(Dd, u, (ya.x + ya.y) + (yb.x + yb.y));
        if (i < nvalid) {
          if (gyp) gyp[opos] = from_f<T>(y);
          if (kGate) {
            const float z = to_f(su[(kT + i) * G]);
            y *= z * sigmoid_f(z);
          }
          gout[opos] = from_f<T>(y);
        }
        opos += ostep;
      }
    }
  }
}

static size_t fwd_smem_bytes(int G, int esize, bool has_z, bool expl) {
  const int nact = 1 + (has_z ? 1 : 0) + (expl ? 1 : 0);
  return (size_t)2 * nact * kT * G * esize + (size_t)2 * kT * kXW * esize + (size_t)kT * kXW * 4;
}

template <typename T, int kMode, bool kGate, bool kVar>
static void launch_fwd3(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  const int G = d->group_channels;
  const size_t smem = fwd_smem_bytes(G, (int)sizeof(T), kGate, kMode == 0);
  dim3 grid((d->dim + G - 1) / G, d->ndir, d->batch);
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(scan_fwd_kernel<T, kMode, kGate, kVar>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  launch_k(scan_fwd_kernel<T, kMode, kGate, kVar>, grid, G, smem, st, *d, seqlens);
}

template <typename T, int kMode, bool kGate>
static void launch_fwd2(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  if (seqlens) launch_fwd3<T, kMode, kGate, true>(d, seqlens, st);
  else launch_fwd3<T, kMode, kGate, false>(d, seqlens, st);
}

template <typename T>
static void launch_fwd(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  const bool gate = d->z != nullptr;
  const int mode = d->delta ? 0 : (d->dt_rank <= 12 ? 1 : 2);
  if (gate) {
    if (mode == 0) launch_fwd2<T, 0, true>(d, seqlens, st);
    else if (mode == 1) launch_fwd2<T, 1, true>(d, seqlens, st);
    else launch_fwd2<T, 2, true>(d, seqlens, st);
  } else {
    if (mode == 0) launch_fwd2<T, 0, false>(d, seqlens, st);
    else if (mode == 1) launch_fwd2<T, 1, false>(d, seqlens, st);
    else launch_fwd2<T, 2, false>(d, seqlens, st);
  }
}

int check_desc(const bimamba_scan_desc* d, bool bwd);  // api.cu
void launch_fwd_warp(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st);  // scan_fwd1.cu

}  // namespace bimamba

using namespace bimamba;

extern "C" int bimamba_selective_scan_fwd(const bimamba_scan_desc* d, bimamba_stream_t stream) {
  return bimamba_selective_scan_fwd_varlen(d, nullptr, stream);
}

// The kernels after the descriptor check; seqlens may come with checkpoints (the training forward).
static int scan_fwd_run(const bimamba_scan_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  const int G = d->group_channels;
  if (G < 32 || G > kFwdMaxThreads || (G & 31)) { set_err("forward group_channels must be 32, 64, 96 or 128 (use bimamba_scan_plan)"); return -5; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // Two kernels, same math (forced in turn by tests/test_gpu_ops.py::test_scan_forward_variants through
  // bimamba_set_tuning(BIMAMBA_TUNE_SCAN_FWD, .)):
  //   3: one lane per channel, one warp per CTA (scan_fwd1.cu) - the Phase-6 sizes (fewer than ~16 warps per SM of
  //      channel lanes: 0.074 ms per launch at batch 64 x 201 frames vs 0.115 for variant 1) and fp32 I/O (1.04 vs 1.28 ms
  //      at 2048 x 256);
  //   1: one lane per channel, wide CTAs sharing the staged rows - large 16-bit problems (1.06 vs 1.09 ms).
  // (A third, two-lanes-per-channel kernel lost to both at every size and was removed in round 2.)
  const int64_t lanes = (int64_t)d->batch * d->ndir * d->dim;
  const int force = g_tune[BIMAMBA_TUNE_SCAN_FWD];
  const int variant = force ? force : ((lanes < (int64_t)148 * 16 * 32 || d->io_dtype == BIMAMBA_F32) ? 3 : 1);
  if (variant == 3) {
    launch_fwd_warp(d, seqlens, st);
  } else {
    switch (d->io_dtype) {
      case BIMAMBA_F32: launch_fwd<float>(d, seqlens, st); break;
      case BIMAMBA_BF16: launch_fwd<__nv_bfloat16>(d, seqlens, st); break;
      default: launch_fwd<__half>(d, seqlens, st); break;
    }
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

extern "C" int bimamba_selective_scan_fwd_varlen(const bimamba_scan_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  if (d && (d->batch == 0 || d->seqlen == 0)) return 0;  // empty: nothing to do (pointers may be null)
  int rc = check_desc(d, false);
  if (rc) return rc;
  if (seqlens && d->ckpt) { set_err("scan fwd: checkpoints belong to the training forward (bimamba_selective_scan_fwd_varlen_train)"); return -9; }
  return scan_fwd_run(d, seqlens, stream);
}

extern "C" int bimamba_selective_scan_fwd_varlen_train(const bimamba_scan_desc* d, const int32_t* seqlens,
                                                       bimamba_stream_t stream) {
  if (d && (d->batch == 0 || d->seqlen == 0)) return 0;
  int rc = check_desc(d, false);
  if (rc) return rc;
  return scan_fwd_run(d, seqlens, stream);
}
