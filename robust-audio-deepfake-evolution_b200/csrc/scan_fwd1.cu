// Selective scan, forward, one lane per channel with ONE WARP PER CTA (group_channels = 32, compile-time).  sm_100a.
//
// Same math, descriptor and outputs as scan_fwd.cu (reference: src/models/modules/mamba_block.py:80-120, :61); this
// is the forward counterpart of scan_bwd1.cu: a 32-channel CTA needs no block barrier (warp-level sync only), every
// shared-memory access is base + immediate, tiles are staged by a fixed per-lane assignment of 16-byte cp.async one
// 16-step chunk ahead, and the per-element math is branch-free so the unrolled steps interleave.
#include "common.cuh"

namespace bimamba {

constexpr int kF1G = 32;

// kVar: utterance b walks its own len_b = clamp(seqlens[b], 0, seqlen) steps (direction 1 starts at len_b - 1) and the
// padded frames len_b .. seqlen-1 of out (and ypre) are written as zeros.  Checkpoint chunk c holds the state entering
// scan steps 8c .. 8c+7 of the utterance; the checkpoint stride stays ceil(seqlen / 8) of the padded length.
template <typename T, int kMode, bool kGate, bool kVar>
__global__ void __launch_bounds__(kF1G) scan_fwd_warp_kernel(const bimamba_scan_desc p, const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr bool expl = kMode == 0;
  constexpr int R4 = kMode == 1 ? 3 : 4;
  constexpr int kV = 16 / sizeof(T);
  constexpr int G = kF1G;
  constexpr int IZ = 1, IDL = 2, kNAct = 3;
  const int tid = threadIdx.x;
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

  float* s_xf = reinterpret_cast<float*>(smem_raw);                 // [16][kXW] rows as fp32
  T* s_xr = reinterpret_cast<T*>(s_xf + kT * kXW);                  // [2][16][kXW] rows as staged
  T* s_act = s_xr + 2 * kT * kXW;                                   // [2][3][16][G]

  const bool dim_vec = (p.dim % kV) == 0;
  const bool vec_u = dim_vec && aligned16(gu + d0) && (p.u_ts % kV) == 0;
  const bool vec_z = kGate && dim_vec && aligned16(gz + d0) && (p.z_ts % kV) == 0;
  const bool vec_d = expl && dim_vec && aligned16(gd + d0) && (p.delta_ts % kV) == 0;
  const bool vec_bc = aligned16(gbc) && (p.bc_ts % kV) == 0;
  const bool vec_dtr = !expl && (p.flags & BIMAMBA_FLAG_DTR_PADDED) && aligned16(gdtr) && (p.dtr_ts % kV) == 0;
  const bool fast = vec_u && (!kGate || vec_z) && (expl ? vec_d : vec_dtr) && vec_bc;
  constexpr int VPR = G / kV, VT = kT * VPR;
  constexpr int BV = 2 * kN / kV, DV = 16 / kV, RV = BV + (expl ? 0 : DV);

  auto stage = [&](int c0, int bf) {
    auto row_of = [&](int i) -> int64_t {
      const int tau = c0 * kT + i;
      return tau < L ? (int64_t)(dir ? (L - 1 - tau) : tau) : (int64_t)-1;
    };
    T* sa = s_act + bf * kNAct * kT * G;
    T* sx = s_xr + bf * kT * kXW;
    if (fast) {
#pragma unroll
      for (int k = 0; k < VT / G; ++k) {
        const int e = tid + k * G, i = e / VPR, v = e - i * VPR;
        const int64_t t = row_of(i);
        const int c = d0 + v * kV;
        const bool okv = t >= 0 && c < p.dim;
        const int so = i * G + v * kV;
        cp_async16(sa + so, okv ? gu + t * p.u_ts + c : gu, okv);
        if (kGate) cp_async16(sa + IZ * kT * G + so, okv ? gz + t * p.z_ts + c : gz, okv);
        if (expl) cp_async16(sa + IDL * kT * G + so, okv ? gd + t * p.delta_ts + c : gd, okv);
      }
#pragma unroll
      for (int k = 0; k < (kT * RV + G - 1) / G; ++k) {
        const int e = tid + k * G;
        if (e < kT * RV) {
          const int i = e / RV, v = e - i * RV;
          const int64_t t = row_of(i);
          const bool okv = t >= 0;
          const T* src = v < BV ? (gbc + t * p.bc_ts + v * kV) : (gdtr + t * p.dtr_ts + (v - BV) * kV);
          cp_async16(sx + i * kXW + v * kV, okv ? src : gbc, okv);
        }
      }
      cp_async_commit();
      return;
    }
    stage_tile(sa, G, gu, p.u_ts, kT, G, d0, p.dim, vec_u, row_of, tid, G);
    if (kGate) stage_tile(sa + IZ * kT * G, G, gz, p.z_ts, kT, G, d0, p.dim, vec_z, row_of, tid, G);
    if (expl) stage_tile(sa + IDL * kT * G, G, gd, p.delta_ts, kT, G, d0, p.dim, vec_d, row_of, tid, G);
    stage_tile(sx, kXW, gbc, p.bc_ts, kT, 2 * kN, 0, 2 * kN, vec_bc, row_of, tid, G);
    if (!expl) {
      const int w = vec_dtr ? 16 : R;
      stage_tile(sx + 2 * kN, kXW, gdtr, p.dtr_ts, kT, w, 0, w, vec_dtr, row_of, tid, G);
    }
    cp_async_commit();
  };

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
  const int ostep = (int)(dir ? -p.out_ts : p.out_ts);
  T* const gout = reinterpret_cast<T*>(p.out) + obase + d;
  T* const gyp = p.ypre ? reinterpret_cast<T*>(p.ypre) + obase + d : nullptr;
  float* const gck = p.ckpt ? p.ckpt + ((((int64_t)b * p.ndir + dir) * nckpt) * p.dim + d) * kN : nullptr;
  const int valid_cols = 2 * kN + R;

  if (nck > 0) stage(0, 0);
  for (int c0 = 0; c0 < nck; ++c0) {
    const int bf = c0 & 1;
    cp_async_wait<0>();
    __syncwarp();  // chunk c0 is visible; every lane is done with chunk c0-1's buffers
    if (c0 + 1 < nck) stage(c0 + 1, bf ^ 1);
    {
      const T* sx = s_xr + bf * kT * kXW;
#pragma unroll
      for (int k = 0; k < (kT * RV + G - 1) / G; ++k) {
        const int e = tid + k * G;
        if (e < kT * RV) {
          const int i = e / RV, v = e - i * RV;
          const int o = i * kXW + v * kV;
          T raw[kV];
          *reinterpret_cast<uint4*>(raw) = *reinterpret_cast<const uint4*>(sx + o);
          float f[kV];
#pragma unroll
          for (int x = 0; x < kV; ++x) f[x] = (v < BV || v * kV + x < valid_cols) ? to_f(raw[x]) : 0.f;
#pragma unroll
          for (int x = 0; x < kV; x += 4) *reinterpret_cast<float4*>(s_xf + o + x) = make_float4(f[x], f[x + 1], f[x + 2], f[x + 3]);
        }
      }
    }
    __syncwarp();
    const T* su = s_act + bf * kNAct * kT * G + tid;
    const int tau0 = c0 * kT;
    const int nvalid = L - tau0;  // steps of this chunk that exist (>= 1)
    const int64_t off0 = (int64_t)(dir ? (L - 1 - tau0) : tau0) * p.out_ts;
#pragma unroll 8
    for (int i = 0; i < kT; ++i) {
      const bool live = ok && i < nvalid;
      if ((i & (BIMAMBA_CKPT - 1)) == 0 && gck && live) {  // state entering this 8-step chunk
        float4* ck = reinterpret_cast<float4*>(gck + (int64_t)((tau0 + i) / BIMAMBA_CKPT) * p.dim * kN);
#pragma unroll
        for (int q = 0; q < 4; ++q) ck[q] = make_float4(h[2 * q].x, h[2 * q].y, h[2 * q + 1].x, h[2 * q + 1].y);
      }
      const float4* xr = reinterpret_cast<const float4*>(s_xf + i * kXW);
      const float u = to_f(su[i * G]);
      float draw;
      if (expl) {
        draw = bias + to_f(su[(IDL * kT + i) * G]);
      } else {
        float2 acc0 = make_float2(bias, 0.f), acc1 = make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < R4; ++q) {
          const float4 x = xr[8 + q];
          acc0 = __ffma2_rn(wdt[2 * q], make_float2(x.x, x.y), acc0);
          acc1 = __ffma2_rn(wdt[2 * q + 1], make_float2(x.z, x.w), acc1);
        }
        const float2 acc = __fadd2_rn(acc0, acc1);
        draw = acc.x + acc.y;
      }
      const float spl = softplus_f(draw);
      const float delta = softplus ? spl : draw;
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
      const float2 ys = __fadd2_rn(ya, yb);
      float y = fmaf(Dd, u, ys.x + ys.y);
      const int64_t off = off0 + i * ostep;
      if (gyp && live) gyp[off] = from_f<T>(y);
      if (kGate) {
        const float z = to_f(su[(IZ * kT + i) * G]);
        y *= z * sigmoid_f(z);
      }
      if (live) gout[off] = from_f<T>(y);
    }
  }
}

template <typename T, int kMode, bool kGate>
static void launch_warp2(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  const size_t smem = (size_t)kT * kXW * 4 + (size_t)2 * kT * kXW * sizeof(T) + (size_t)2 * 3 * kT * kF1G * sizeof(T);
  dim3 grid((d->dim + kF1G - 1) / kF1G, d->ndir, d->batch);
  if (seqlens) launch_k(scan_fwd_warp_kernel<T, kMode, kGate, true>, grid, kF1G, smem, st, *d, seqlens);
  else launch_k(scan_fwd_warp_kernel<T, kMode, kGate, false>, grid, kF1G, smem, st, *d, seqlens);
}

template <typename T>
static void launch_warp(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  const bool gate = d->z != nullptr;
  const int mode = d->delta ? 0 : (d->dt_rank <= 12 ? 1 : 2);
  if (gate) {
    if (mode == 0) launch_warp2<T, 0, true>(d, seqlens, st);
    else if (mode == 1) launch_warp2<T, 1, true>(d, seqlens, st);
    else launch_warp2<T, 2, true>(d, seqlens, st);
  } else {
    if (mode == 0) launch_warp2<T, 0, false>(d, seqlens, st);
    else if (mode == 1) launch_warp2<T, 1, false>(d, seqlens, st);
    else launch_warp2<T, 2, false>(d, seqlens, st);
  }
}

// group_channels is ignored: this kernel always works on 32-channel groups (the forward has no per-group outputs).
void launch_fwd_warp(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  switch (d->io_dtype) {
    case BIMAMBA_F32: launch_warp<float>(d, seqlens, st); break;
    case BIMAMBA_BF16: launch_warp<__nv_bfloat16>(d, seqlens, st); break;
    default: launch_warp<__half>(d, seqlens, st); break;
  }
}

}  // namespace bimamba
