// Selective scan, backward, ONE LANE PER CHANNEL (both time directions in one launch).  sm_100a.
//
// Gradients (SURVEY Appendix A; autograd of src/models/modules/mamba_block.py:80-120, :61):
//   g = dout * silu(z);  dz = dout * ypre * silu'(z)
//   dh[t] = g[t] C[t] + a[t+1] dh[t+1]                       (reverse-time recurrence)
//   ddelta[t] = sum_n dh a h[t-1] A + u sum_n dh B;  du[t] = g D + delta sum_n dh B
//   dB[t,n] = sum_d dh delta u;  dC[t,n] = sum_d g h;  dA[n] = sum_t dh a h[t-1] delta
//
// Mapping.  A thread owns one channel of one (batch, direction), like the forward: the n-sums are thread-local (no
// shuffles), delta / softplus / SiLU are evaluated once per element by the thread that needs them (no exchange), and
// dA / dD / dbias accumulate in registers over the whole sequence.  One warp (32 channels) per CTA.
//   * time is walked in 8-step chunks (the forward's checkpoint interval) from the last to the first.  Per chunk:
//       1. a prologue computes what does not depend on the state - delta, softplus', g = dout silu(z) - into this
//          lane's shared-memory slots (conflict-free: slot [k][i][lane]) and writes dz;
//       2. TWO PASSES over the chunk, states 0-7 then 8-15.  Each re-runs the chunk forward from its half of the
//          checkpoint, keeping the seven intermediate states (7 x 4 float2) AND the 8 x 8 decays exp2(delta A) in
//          registers, then walks it backwards: m / dA for its 8 states, the 16 dB|dC columns of its states, and its
//          part of the two n-sums, which it adds into the lane's slots;
//       3. an epilogue turns the n-sums into du and ddelta and accumulates dD and dbias.
//     With all 16 states in one walk the history alone was 112 registers: that kernel used all 255, spilled 56-104
//     bytes and recomputed every decay in the reverse walk (33 MUFU exp2 per element).  The half-walks hold 56 + 64
//     registers of history and decays, 236-254 registers in all without spills, 19 MUFU exp2 per element; their loop
//     is not unrolled (the pass's A, m and dA registers are swapped with the other pass's at its end).  Four or two
//     lanes per channel, part of the history in shared memory and a single predicated block were measured slower
//     (profiles/r2_history.md); the two-pass walk is measured in profiles/r3_scan_bwd_passes.md.
//   * dB / dC need a sum over channels.  Each pass exchanges two steps at a time: a lane writes its 16 products of the
//     odd step and then the 16 of the even step to its padded row of shared memory (8 STS.128, conflict-free), the
//     warp transposes-and-adds the 32 x 32 block with 8 LDS.128 + packed adds per lane and two shuffle levels, and
//     every lane writes one column of one of the two steps, summed over the 32 channels in a fixed order.  (One
//     16-column exchange per step doubled the exchanges per chunk and made the kernel 7 % slower than the 16-state
//     walk.)  The partial row goes straight to global; bimamba_reduce_partials sums the groups: deterministic, no
//     atomics.
//   * u, dout, z, ypre (delta) tiles [8 x 32], the chunk's B|C|dt_r rows and the checkpoint are staged by a fixed
//     per-lane assignment of 16-byte cp.async into double buffers one chunk ahead (generic element-wise staging for
//     tensors that are not 16-byte friendly).
//   * all element math is branch-free (the softplus / gate / ypre flags select).
//   * kVar: utterance b walks its own len_b = clamp(seqlens[b], 0, seqlen) steps from its own last chunk (direction 1
//     from frame len_b - 1), the mirror of the variable-length forward.  Every layout keeps the padded seqlen: the
//     checkpoint stride ceil(seqlen / 8) and the (B, ngroups, seqlen, ndir, 32) partial rows.  Padded frames of du,
//     ddelta, dz and of the partial rows are written as zeros (the row sums and the weight-gradient products downstream
//     run over every row); dout there is never read, and dA / dD / dbias see valid steps only.
#include "common.cuh"

namespace bimamba {

constexpr int kLT = BIMAMBA_CKPT;   // steps per chunk == checkpoint interval (8)
static_assert(kLT == 8, "history registers are sized for 8-step chunks");

// kMode: 0 = delta given; 1 = fused dt projection with dt_rank <= 12; 2 = dt_rank <= 16.
// Shared memory per CTA stays <= 28 160 bytes so that 8 CTAs (the 8 warps per SM of the Phase-6 shapes) fit an SM.
template <typename T, int kMode>
struct LaneSmem {
  static constexpr int NT = 32;                                     // threads == channels
  static constexpr int kRow = 36;                                   // floats per channel row of the dB|dC exchange (padded)
  static constexpr int kNAct = kMode == 0 ? 5 : 4;                  // u, dout, z, ypre (, delta)
  static constexpr int kWS = kMode == 0 ? 0 : (kMode == 1 ? 12 : 20);   // floats per lane row of dt_proj.weight
  static constexpr int kNEl = 5;                                    // per-lane slots: delta, softplus', g, rA, rU
  static constexpr int kXF = kMode == 0 ? 2 * kN : kXW;             // floats per fp32 row: B|C (|dt_r)
  static constexpr size_t ck_f4 = (size_t)2 * 4 * NT;               // [2][4][NT] float4
  static constexpr size_t red_f = (size_t)NT * kRow;                // [NT][kRow]
  static constexpr size_t el_f = (size_t)kNEl * kLT * NT;           // [kNEl][8][NT]
  static constexpr size_t xf_f = (size_t)kLT * kXF;
  static constexpr size_t wdt_f = (size_t)NT * kWS;
  static constexpr size_t xr_e = (size_t)2 * kLT * kXW;             // T
  static constexpr size_t act_buf_e = (size_t)kNAct * kLT * NT;     // T, one buffer
  static constexpr size_t total = ck_f4 * 16 + (red_f + el_f + xf_f + wdt_f) * 4 + (xr_e + 2 * act_buf_e) * sizeof(T);
  // (fp32 I/O with dt_rank > 12 takes 1 KB more: 7 CTAs per SM)
  static_assert(total <= 28160 || (kMode == 2 && sizeof(T) == 4), "8 CTAs per SM");
};

template <typename T, int kMode, bool kVar>
__global__ void __launch_bounds__(32, 1) scan_bwd_lane_kernel(const bimamba_scan_desc p, const int32_t* __restrict__ seqlens) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using SM = LaneSmem<T, kMode>;
  constexpr bool expl = kMode == 0;
  constexpr int R4 = kMode == 1 ? 3 : 4;
  constexpr int kV = 16 / sizeof(T);
  constexpr int NT = SM::NT, G = NT, kRow = SM::kRow, kWS = SM::kWS, kXF = SM::kXF;
  constexpr int IZ = 2, IYP = 3, IDL = 4;
  constexpr int EDL = 0, ESP = 1, EG = 2, ERA = 3, ERU = 4;   // slots of s_el
  const int tid = threadIdx.x, lane = tid;
  const int b = blockIdx.z, dir = blockIdx.y, g = blockIdx.x, d0 = g * G, d = d0 + lane;
  const int ngroups = gridDim.x;
  const bool ok = d < p.dim;
  const int L = kVar ? min(max(__ldg(seqlens + b), 0), p.seqlen) : p.seqlen, nsub = (L + kLT - 1) / kLT;
  const int nck = kVar ? (p.seqlen + kLT - 1) / kLT : nsub;   // checkpoint stride (padded length)
  const bool gated = p.z != nullptr, need_yp = gated && p.dz != nullptr;
  const bool softplus = (p.flags & BIMAMBA_FLAG_SOFTPLUS) != 0;
  const int R = expl ? 0 : p.dt_rank;
  const int64_t bd = (int64_t)b * p.ndir + dir;

  const T* gu = reinterpret_cast<const T*>(p.u) + (int64_t)b * p.u_bs + (int64_t)dir * p.u_ds;
  const T* gz = gated ? reinterpret_cast<const T*>(p.z) + (int64_t)b * p.z_bs + (int64_t)dir * p.z_ds : nullptr;
  const T* gdl = expl ? reinterpret_cast<const T*>(p.delta) + (int64_t)b * p.delta_bs + (int64_t)dir * p.delta_ds : nullptr;
  const T* gbc = reinterpret_cast<const T*>(p.bc) + (int64_t)b * p.bc_bs + (int64_t)dir * p.bc_ds;
  const T* gdtr = expl ? nullptr : reinterpret_cast<const T*>(p.dtr) + (int64_t)b * p.dtr_bs + (int64_t)dir * p.dtr_ds;
  const T* gdo = reinterpret_cast<const T*>(p.dout) + (int64_t)b * p.dout_bs + (int64_t)dir * p.dout_ds;
  const int64_t obase = (int64_t)b * p.out_bs + (int64_t)dir * p.out_ds;
  const T* gyp = need_yp ? reinterpret_cast<const T*>(p.ypre) + obase : nullptr;
  T* gdu = reinterpret_cast<T*>(p.du) + obase + d;
  T* gdd = reinterpret_cast<T*>(p.ddelta) + obase + d;
  T* gdz = need_yp ? reinterpret_cast<T*>(p.dz) + obase + d : nullptr;
  // partial layout (batch, ngroups, L, ndir, 32): reducing over ngroups leaves rows ordered (b, t, dir)
  const int pb_ts = p.ndir * 2 * kN;
  float* partB = p.dbc_part + (((int64_t)b * ngroups + g) * (kVar ? p.seqlen : L)) * pb_ts + dir * 2 * kN;
  const float* gck = p.ckpt ? p.ckpt + bd * nck * (int64_t)p.dim * kN : nullptr;
  if (kVar) {   // padded frames: zero gradients and zero partial rows (one column per lane: 32 == 2 * kN)
    for (int t = L; t < p.seqlen; ++t) {
      const int64_t o = (int64_t)t * p.out_ts;
      if (ok) {
        gdu[o] = from_f<T>(0.f);
        gdd[o] = from_f<T>(0.f);
        if (gdz) gdz[o] = from_f<T>(0.f);
      }
      partB[(int64_t)t * pb_ts + lane] = 0.f;
    }
  }

  // ---- shared memory carve
  float4* s_ck = reinterpret_cast<float4*>(smem_raw);               // [2][4][NT]  checkpoint (state entering the chunk)
  float* s_red = reinterpret_cast<float*>(s_ck + SM::ck_f4);        // [NT][kRow]
  float* s_el = s_red + SM::red_f;                                  // [kNEl][8][NT]
  float* s_xf = s_el + SM::el_f;                                    // [8][kXF]    rows as fp32
  float* s_wdt = s_xf + SM::xf_f;                                   // [NT][kWS]   this lane's dt_proj.weight row
  T* s_xr = reinterpret_cast<T*>(s_wdt + SM::wdt_f);                // [2][8][kXW] rows as staged
  T* s_act = s_xr + SM::xr_e;                                       // [2][kNAct][8][G]

  const bool dim_vec = (p.dim % kV) == 0;
  const bool vec_u = dim_vec && aligned16(gu + d0) && (p.u_ts % kV) == 0;
  const bool vec_do = dim_vec && aligned16(gdo + d0) && (p.dout_ts % kV) == 0;
  const bool vec_z = gated && dim_vec && aligned16(gz + d0) && (p.z_ts % kV) == 0;
  const bool vec_yp = need_yp && dim_vec && aligned16(gyp + d0) && (p.out_ts % kV) == 0;
  const bool vec_dl = expl && dim_vec && aligned16(gdl + d0) && (p.delta_ts % kV) == 0;
  const bool vec_bc = aligned16(gbc) && (p.bc_ts % kV) == 0;
  const bool vec_dtr = !expl && (p.flags & BIMAMBA_FLAG_DTR_PADDED) && aligned16(gdtr) && (p.dtr_ts % kV) == 0;
  const bool vec_ck = gck != nullptr && aligned16(gck);
  // Fast staging (every tensor 16-byte friendly): a fixed (row, vector) assignment per thread.
  const bool fast = vec_u && vec_do && (!gated || vec_z) && (!need_yp || vec_yp) && (expl ? vec_dl : vec_dtr) && vec_bc &&
                    (!gck || vec_ck);
  constexpr int VPR = G / kV;          // vectors per activation tile row
  constexpr int VT = kLT * VPR;        // vectors per activation tile
  constexpr int BV = 2 * kN / kV, DV = 16 / kV;   // vectors per row: B|C and padded dt_r
  constexpr int RV = BV + (expl ? 0 : DV);

  auto stage = [&](int c0, int bf) {
    auto row_of = [&](int i) -> int64_t {
      const int tau = c0 * kLT + i;
      return tau < L ? (int64_t)(dir ? (L - 1 - tau) : tau) : (int64_t)-1;
    };
    T* sa = s_act + bf * SM::act_buf_e;
    T* sx = s_xr + bf * kLT * kXW;
    float4* ck = s_ck + bf * 4 * NT + tid;
    if (fast) {
#pragma unroll
      for (int k = 0; k < (VT + NT - 1) / NT; ++k) {
        const int e = tid + k * NT;
        if (VT % NT == 0 || e < VT) {
          const int i = e / VPR, v = e - i * VPR;
          const int64_t t = row_of(i);
          const int c = d0 + v * kV;
          const bool okv = t >= 0 && c < p.dim;
          const int so = i * G + v * kV;
          cp_async16(sa + so, okv ? gu + t * p.u_ts + c : gu, okv);
          cp_async16(sa + kLT * G + so, okv ? gdo + t * p.dout_ts + c : gdo, okv);
          if (gated) cp_async16(sa + IZ * kLT * G + so, okv ? gz + t * p.z_ts + c : gz, okv);
          if (need_yp) cp_async16(sa + IYP * kLT * G + so, okv ? gyp + t * p.out_ts + c : gyp, okv);
          if (expl) cp_async16(sa + IDL * kLT * G + so, okv ? gdl + t * p.delta_ts + c : gdl, okv);
        }
      }
#pragma unroll
      for (int k = 0; k < (kLT * RV + NT - 1) / NT; ++k) {
        const int e = tid + k * NT;
        if (e < kLT * RV) {
          const int i = e / RV, v = e - i * RV;
          const int64_t t = row_of(i);
          const bool okv = t >= 0;
          const T* src = v < BV ? (gbc + t * p.bc_ts + v * kV) : (gdtr + t * p.dtr_ts + (v - BV) * kV);
          cp_async16(sx + i * kXW + v * kV, okv ? src : gbc, okv);
        }
      }
      if (gck) {
        const float* src = gck + ((int64_t)c0 * p.dim + (ok ? d : 0)) * kN;
#pragma unroll
        for (int q = 0; q < 4; ++q) cp_async16(ck + q * NT, src + 4 * q, ok);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) ck[q * NT] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      cp_async_commit();
      return;
    }
    stage_tile(sa, G, gu, p.u_ts, kLT, G, d0, p.dim, vec_u, row_of, tid, NT);
    stage_tile(sa + kLT * G, G, gdo, p.dout_ts, kLT, G, d0, p.dim, vec_do, row_of, tid, NT);
    if (gated) stage_tile(sa + IZ * kLT * G, G, gz, p.z_ts, kLT, G, d0, p.dim, vec_z, row_of, tid, NT);
    if (need_yp) stage_tile(sa + IYP * kLT * G, G, gyp, p.out_ts, kLT, G, d0, p.dim, vec_yp, row_of, tid, NT);
    if (expl) stage_tile(sa + IDL * kLT * G, G, gdl, p.delta_ts, kLT, G, d0, p.dim, vec_dl, row_of, tid, NT);
    stage_tile(sx, kXW, gbc, p.bc_ts, kLT, 2 * kN, 0, 2 * kN, vec_bc, row_of, tid, NT);
    if (!expl) {
      const int w = vec_dtr ? 16 : R;
      stage_tile(sx + 2 * kN, kXW, gdtr, p.dtr_ts, kLT, w, 0, w, vec_dtr, row_of, tid, NT);
    }
    // this lane's checkpoint, into planes [q][NT] (conflict-free float4 reads)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gck && ok) {
        const float* src = gck + ((int64_t)c0 * p.dim + d) * kN + 4 * q;
        v = make_float4(src[0], src[1], src[2], src[3]);
      }
      ck[q * NT] = v;
    }
    cp_async_commit();
  };

  if (nsub > 0) stage(nsub - 1, 0);

  // ---- per-channel constants and accumulators.  Registers [0..3] belong to the pass being walked, [4..7] to the
  // other one; the pass loop swaps the two halves at its end, so the pass code indexes registers at compile time.
  float2 A2[8], m[8], dAa[8];
  float* const my_w = s_wdt + tid * kWS;
  float bias = 0.f, Dd = 0.f, dDacc = 0.f, dbacc = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    A2[j] = make_float2(0.f, 0.f);
    m[j] = make_float2(0.f, 0.f);
    dAa[j] = make_float2(0.f, 0.f);
  }
  if (!expl) {
#pragma unroll
    for (int r = 0; r < 4 * R4; ++r) my_w[r] = 0.f;
  }
  if (ok) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      A2[j].x = __ldg(p.A + (int64_t)d * kN + 2 * j) * kLog2e;
      A2[j].y = __ldg(p.A + (int64_t)d * kN + 2 * j + 1) * kLog2e;
    }
    if (p.delta_bias) bias = __ldg(p.delta_bias + d);
    if (p.D) Dd = __ldg(p.D + d);
    if (!expl) {
#pragma unroll
      for (int r = 0; r < 4 * R4; ++r)
        if (r < R) my_w[r] = __ldg(p.Wdt + (int64_t)d * R + r);   // written and read by this lane only
    }
  }
  // dB|dC exchange of a pass, two steps at a time: row = channel, [16 products of the even step | 16 of the odd step],
  // each [dB of the pass's 8 states | dC of them], in 8 pieces of 4 floats.  Lane (v4 = lane & 7, cq = lane >> 3) adds
  // piece v4 of rows 8 cq .. 8 cq + 7; two shuffle levels finish the sum over the 32 rows and leave element cq of the
  // piece, i.e. row element 4 v4 + cq, in the lane.
  const int v4 = lane & 7, cq = lane >> 3;
  const bool hi = (cq & 2) != 0, odd = (cq & 1) != 0;
  float* const myred = s_red + lane * kRow;
  const float4* const rdred = reinterpret_cast<const float4*>(s_red + 8 * cq * kRow) + v4;
  const int rcol = 4 * v4 + cq, podd = rcol >> 4, pcol = rcol & 15;   // step parity; 0..7: dB, 8..15: dC of the pass
  const int mycol = (pcol & 8) * 2 + (pcol & 7);                      // [dB | dC] column in pass 0; pass 1 adds 8
  float* const myel = s_el + tid;
  const int valid_cols = 2 * kN + R;
  const int ostep = (int)(dir ? -p.out_ts : p.out_ts);    // one step forward in scan time (elements)
  const int pstep = dir ? -pb_ts : pb_ts;

  int bf = 0;
  for (int c0 = nsub - 1; c0 >= 0; --c0, bf ^= 1) {
    cp_async_wait<0>();
    __syncwarp();  // chunk c0's tiles are visible; every lane is done with the previous chunk's buffers
    if (c0 > 0) stage(c0 - 1, bf ^ 1);
    {  // rows -> fp32, columns past B|C|dt_r zeroed
      const T* sx = s_xr + bf * kLT * kXW;
#pragma unroll
      for (int k = 0; k < (kLT * RV + NT - 1) / NT; ++k) {
        const int e = tid + k * NT;
        if (e < kLT * RV) {
          const int i = e / RV, v = e - i * RV;
          const int o = i * kXF + v * kV;
          T raw[kV];
          *reinterpret_cast<uint4*>(raw) = *reinterpret_cast<const uint4*>(sx + i * kXW + v * kV);
          float f[kV];
#pragma unroll
          for (int x = 0; x < kV; ++x) f[x] = (v < BV || v * kV + x < valid_cols) ? to_f(raw[x]) : 0.f;
#pragma unroll
          for (int x = 0; x < kV; x += 4) *reinterpret_cast<float4*>(s_xf + o + x) = make_float4(f[x], f[x + 1], f[x + 2], f[x + 3]);
        }
      }
    }
    __syncwarp();
    const int tau0 = c0 * kLT;
    const int nvalid = min(kLT, L - tau0);
    const T* sa = s_act + bf * SM::act_buf_e + lane;
    const int64_t trow0 = dir ? (L - 1 - tau0) : tau0;
    const int64_t off0 = trow0 * p.out_ts;

    // ---- prologue: the state-independent values of the chunk's 8 steps (eight independent chains, no branches)
#pragma unroll
    for (int i = 0; i < kLT; ++i) {
      const float4* xr = reinterpret_cast<const float4*>(s_xf + i * kXF);
      float draw;
      if (expl) {
        draw = bias + to_f(sa[(IDL * kLT + i) * G]);
      } else {
        float2 acc0 = make_float2(bias, 0.f), acc1 = make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < R4; ++q) {
          const float4 x = xr[8 + q];
          const float4 w = reinterpret_cast<const float4*>(my_w)[q];
          acc0 = __ffma2_rn(make_float2(w.x, w.y), make_float2(x.x, x.y), acc0);
          acc1 = __ffma2_rn(make_float2(w.z, w.w), make_float2(x.z, x.w), acc1);
        }
        const float2 acc = __fadd2_rn(acc0, acc1);
        draw = acc.x + acc.y;
      }
      const float spl = softplus_f(draw);
      const float sgd = draw > 20.f ? 1.f : sigmoid_f(draw);
      float delta = softplus ? spl : draw;
      delta = i < nvalid ? delta : 0.f;   // steps past the end of the sequence are the identity
      const float dov = to_f(sa[(kLT + i) * G]);
      // branch-free: the z / ypre slots are read even when absent (stale but harmless: the flags select)
      const float zz = to_f(sa[(IZ * kLT + i) * G]);
      const float sg = sigmoid_f(zz);
      const float yp = to_f(sa[(IYP * kLT + i) * G]);
      const float dzv = dov * yp * sg * (1.f + zz * (1.f - sg));
      if (need_yp && ok && i < nvalid) gdz[off0 + i * ostep] = from_f<T>(dzv);
      myel[(EDL * kLT + i) * NT] = delta;
      myel[(ESP * kLT + i) * NT] = softplus ? sgd : 1.f;
      myel[(EG * kLT + i) * NT] = gated ? dov * zz * sg : dov;
      myel[(ERA * kLT + i) * NT] = 0.f;
      myel[(ERU * kLT + i) * NT] = 0.f;
    }

    // ---- two passes over the chunk: states 8 ps .. 8 ps + 7
#pragma unroll 1
    for (int ps = 0; ps < 2; ++ps) {
      const float* const xb = s_xf + 8 * ps;          // B of the pass's states at [0..7], C at [16..23]
      const float4* const ckp = s_ck + (bf * 4 + 2 * ps) * NT + tid;
      float* const pB0 = partB + (trow0 + (dir ? -podd : podd)) * pb_ts + mycol + 8 * ps;
      float2 h[4], a[kLT][4], hh[kLT - 1][4];
      auto load_ck = [&](float2 (&dst)[4]) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const float4 v = ckp[q * NT];
          dst[2 * q] = make_float2(v.x, v.y);
          dst[2 * q + 1] = make_float2(v.z, v.w);
        }
      };
      // re-run the chunk forward from the checkpoint, keeping h[0..6] and the decays
      load_ck(h);
#pragma unroll
      for (int i = 0; i < kLT; ++i) {
        const float4* xr = reinterpret_cast<const float4*>(xb + i * kXF);
        const float delta = myel[(EDL * kLT + i) * NT], du = delta * to_f(sa[i * G]);
        const float2 dd = make_float2(delta, delta), duu = make_float2(du, du);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const float4 Bq = xr[q];
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const int j = 2 * q + s;
            const float2 B2 = s ? make_float2(Bq.z, Bq.w) : make_float2(Bq.x, Bq.y);
            const float2 x = __fmul2_rn(dd, A2[j]);
            a[i][j] = make_float2(ex2_approx(x.x), ex2_approx(x.y));
            h[j] = __ffma2_rn(a[i][j], h[j], __fmul2_rn(duu, B2));
          }
        }
        if (i < kLT - 1) {
#pragma unroll
          for (int j = 0; j < 4; ++j) hh[i][j] = h[j];
        }
      }
      // reverse recurrence over the chunk:  dh_i = g_i C_i + m_{i+1},  m_i = a_i dh_i
      auto rev_step = [&](const int i, const float2 (&hc_)[4], const float2 (&hp_)[4]) {
        const float4* xr = reinterpret_cast<const float4*>(xb + i * kXF);
        const float delta = myel[(EDL * kLT + i) * NT], gv = myel[(EG * kLT + i) * NT], du = delta * to_f(sa[i * G]);
        const float2 dd = make_float2(delta, delta), duu = make_float2(du, du), gg = make_float2(gv, gv);
        float2 sAv[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)}, sUv[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const float4 Bq = xr[q], Cq = xr[4 + q];
          float2 dBv[2], dCv[2];
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const int j = 2 * q + s;
            const float2 B2 = s ? make_float2(Bq.z, Bq.w) : make_float2(Bq.x, Bq.y);
            const float2 C2 = s ? make_float2(Cq.z, Cq.w) : make_float2(Cq.x, Cq.y);
            const float2 dh = __ffma2_rn(gg, C2, m[j]);
            m[j] = __fmul2_rn(a[i][j], dh);
            const float2 da = __fmul2_rn(m[j], hp_[j]);
            dAa[j] = __ffma2_rn(da, dd, dAa[j]);
            sAv[s] = __ffma2_rn(da, A2[j], sAv[s]);   // sum_n dh a h[t-1] A (x log2e; scaled back in the epilogue)
            sUv[s] = __ffma2_rn(dh, B2, sUv[s]);      // sum_n dh B
            dBv[s] = __fmul2_rn(dh, duu);
            dCv[s] = __fmul2_rn(gg, hc_[j]);
          }
          *reinterpret_cast<float4*>(myred + 16 * (i & 1) + 4 * q) = make_float4(dBv[0].x, dBv[0].y, dBv[1].x, dBv[1].y);
          *reinterpret_cast<float4*>(myred + 16 * (i & 1) + 8 + 4 * q) = make_float4(dCv[0].x, dCv[0].y, dCv[1].x, dCv[1].y);
        }
        const float2 sA = __fadd2_rn(sAv[0], sAv[1]), sU = __fadd2_rn(sUv[0], sUv[1]);
        myel[(ERA * kLT + i) * NT] += sA.x + sA.y;
        myel[(ERU * kLT + i) * NT] += sU.x + sU.y;
        if (i & 1) return;   // the odd step's products wait in the row for the even step's
        __syncwarp();
        {  // column sums over the warp's channels: lane (v4, cq) adds rows 8 cq .. 8 cq + 7 of piece v4
          float4 t0 = rdred[0], t1 = rdred[kRow / 4];
          float2 lo = __fadd2_rn(make_float2(t0.x, t0.y), make_float2(t1.x, t1.y));
          float2 up = __fadd2_rn(make_float2(t0.z, t0.w), make_float2(t1.z, t1.w));
#pragma unroll
          for (int r = 2; r < 8; ++r) {
            const float4 t = rdred[r * (kRow / 4)];
            lo = __fadd2_rn(lo, make_float2(t.x, t.y));
            up = __fadd2_rn(up, make_float2(t.z, t.w));
          }
          float kx = hi ? up.x : lo.x, ky = hi ? up.y : lo.y;
          const float sx = hi ? lo.x : up.x, sy = hi ? lo.y : up.y;
          kx += __shfl_xor_sync(kFull, sx, 16);
          ky += __shfl_xor_sync(kFull, sy, 16);
          const float keep = odd ? ky : kx, send = odd ? kx : ky;
          const float val = keep + __shfl_xor_sync(kFull, send, 8);
          if (i + podd < nvalid) pB0[i * pstep] = val;
        }
        __syncwarp();   // the rows are rewritten by the next pair of steps
      };
      rev_step(7, h, hh[6]);
#pragma unroll
      for (int i = kLT - 2; i >= 1; --i) rev_step(i, hh[i], hh[i - 1]);
      float2 hck[4];
      load_ck(hck);
      rev_step(0, hh[0], hck);
#pragma unroll
      for (int j = 0; j < 4; ++j) {   // hand the registers to the other pass
        float2 t = A2[j]; A2[j] = A2[4 + j]; A2[4 + j] = t;
        t = m[j]; m[j] = m[4 + j]; m[4 + j] = t;
        t = dAa[j]; dAa[j] = dAa[4 + j]; dAa[4 + j] = t;
      }
    }

    // ---- epilogue: du, ddelta; dD and dbias in the reverse time order of the walk
#pragma unroll
    for (int i = kLT - 1; i >= 0; --i) {
      const float delta = myel[(EDL * kLT + i) * NT], sp = myel[(ESP * kLT + i) * NT], gv = myel[(EG * kLT + i) * NT];
      const float rA = myel[(ERA * kLT + i) * NT], rU = myel[(ERU * kLT + i) * NT];
      const float u = to_f(sa[i * G]);
      const float duv = fmaf(gv, Dd, delta * rU);
      const float dbl = fmaf(u, rU, rA * kLn2) * sp;
      if (ok && i < nvalid) {
        const int64_t off = off0 + i * ostep;
        gdu[off] = from_f<T>(duv);
        gdd[off] = from_f<T>(dbl);
        dDacc = fmaf(gv, u, dDacc);
        dbacc += dbl;
      }
    }
  }

  // ---- per-channel partials of this (batch, direction)
  if (ok) {
    float4* pa = reinterpret_cast<float4*>(p.dA_part + (bd * p.dim + d) * kN);
#pragma unroll
    for (int q = 0; q < 4; ++q) pa[q] = make_float4(dAa[2 * q].x, dAa[2 * q].y, dAa[2 * q + 1].x, dAa[2 * q + 1].y);
    if (p.dD_part) p.dD_part[bd * p.dim + d] = dDacc;
    if (p.dbias_part) p.dbias_part[bd * p.dim + d] = dbacc;
  }
}

// group_channels == 32 (checked by the caller): one warp per CTA, one lane per channel.
template <typename T, int kMode>
static void launch_lane2(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  constexpr size_t smem = LaneSmem<T, kMode>::total;
  dim3 grid((d->dim + 31) / 32, d->ndir, d->batch);
  if (seqlens) launch_k(scan_bwd_lane_kernel<T, kMode, true>, grid, 32, smem, st, *d, seqlens);
  else launch_k(scan_bwd_lane_kernel<T, kMode, false>, grid, 32, smem, st, *d, seqlens);
}

template <typename T>
static void launch_lane(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  const int mode = d->delta ? 0 : (d->dt_rank <= 12 ? 1 : 2);
  if (mode == 0) launch_lane2<T, 0>(d, seqlens, st);
  else if (mode == 1) launch_lane2<T, 1>(d, seqlens, st);
  else launch_lane2<T, 2>(d, seqlens, st);
}

void launch_bwd_lane(const bimamba_scan_desc* d, const int32_t* seqlens, cudaStream_t st) {
  switch (d->io_dtype) {
    case BIMAMBA_F32: launch_lane<float>(d, seqlens, st); break;
    case BIMAMBA_BF16: launch_lane<__nv_bfloat16>(d, seqlens, st); break;
    default: launch_lane<__half>(d, seqlens, st); break;
  }
}

int check_desc(const bimamba_scan_desc* d, bool bwd);  // api.cu

}  // namespace bimamba

using namespace bimamba;

extern "C" int bimamba_selective_scan_bwd(const bimamba_scan_desc* d, bimamba_stream_t stream) {
  return bimamba_selective_scan_bwd_varlen(d, nullptr, stream);
}

extern "C" int bimamba_selective_scan_bwd_varlen(const bimamba_scan_desc* d, const int32_t* seqlens, bimamba_stream_t stream) {
  if (d && (d->batch == 0 || d->seqlen == 0)) return 0;
  int rc = check_desc(d, true);
  if (rc) return rc;
  if (d->group_channels != 32) { set_err("backward group_channels must be 32 (use bimamba_scan_plan)"); return -5; }
  launch_bwd_lane(d, seqlens, reinterpret_cast<cudaStream_t>(stream));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}
