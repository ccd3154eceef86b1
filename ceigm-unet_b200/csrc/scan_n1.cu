// Selective scan for d_state = 1, fp32, contiguous traversals — the lean kernels the live GM-UNet regime runs on
// (4 single-direction SS2Ds with N = 1 per GroupMambaLayer: D in {16, 32, 87, 112} rows per (batch, direction),
// L in {3136, 784, 196, 49}; SURVEY.md §8 table). Replaces selective_scan_{fwd,bwd}_kernel
// (/root/reference/gm-unet/kernels/selective_scan/csrc/selective_scan/cus/selective_scan_fwd_kernel.cuh:61-172,
// selective_scan_bwd_kernel.cuh:66-273) for that regime; every other dtype / layout keeps scan_par.cu.
//
// Same algorithm as scan_par.cu — the scan is parallel ALONG L: a row is owned by seg x wpr threads, each scanning
// P = 8 consecutive positions in registers; the (decay, state) aggregates are combined by a Kogge-Stone shuffle scan inside
// the warp, one shared-memory hop and a second shuffle scan over the warps of the row — but built for calls that move
// 2 ... 60 MB, where scan_par lost to the reference kernel (profiles/r2_time_stages.txt):
//   * ONE code path per launch. ncu on scan_par (profiles/r2_ncu_scan_par_small_shapes.txt) showed its 7 700-instruction
//     bodies (generic dtype / direction / tail handling inlined next to the fast path) stalled on instruction fetch
//     (`no_instruction` 19.7 cycles per issue at the stage-3 shape): every warp runs the code exactly once. Here eligibility
//     is decided on the host and the geometry (lanes per row, warps per row, rows per CTA) is a kernel ARGUMENT.
//   * the whole row in flight at once: up to 16 warps per row, so a 56^2 row is one pass (scan_par: two sequential chunks).
//   * out-of-range positions are loaded as delta = -inf: softplus gives exactly 0 there, the state freezes, and no
//     per-position bound check is left in the arithmetic.
//   * backward (`scan_n1_bwd_rows_kernel`): a CTA walks SEVERAL rows of its group one after the other and keeps dB / dC in
//     registers across them — the sum over the rows of a group costs nothing and is stored once (plain stores when one CTA
//     covers the group, red.global when several share it). The next row's delta / u / dout are in flight meanwhile: one
//     elected thread per row lane streams them through a 2-stage shared-memory ring with 1-D TMA bulk copies
//     (cp.async.bulk + mbarrier); row lanes synchronise on their own named barriers, so they drift apart and overlap.
//     dA / dD / d(delta_bias) go into caller-zeroed accumulators with atomics (`grads_prezeroed`): the call is memset + ONE
//     kernel (scan_par: memset, kernel, finalize). Neither sum is reproducible bit for bit from call to call.
//   * deterministic mode (DET; ss2d_scan_desc.deterministic): every CTA stores dB / dC into its own partial slab (summed in
//     slab order by scan_bwd_fold_kernel) and the per-row sums of dA / dD / d(delta_bias) go to the partial buffer of the
//     fixed-order finalize pass; rows walked in several chunks keep their running sums in shared memory.
#include <algorithm>

#include "common.cuh"
#include "host_util.h"
#include "scan_params.h"

namespace ss2d {

constexpr int N1_P = 8;             // positions per thread
constexpr int N1_MAX_WARPS = 16;    // warps per CTA

struct N1Geom {
  int seg;       // lanes of one row inside a warp: 4, 8, 16 or 32
  int wpr;       // warps per row (1 when seg < 32)
  int rt;        // row lanes per CTA (rows processed concurrently)
  int rseq;      // rows each lane walks one after the other (backward rows kernel; 1 otherwise)
  int lc;        // positions per chunk = seg * wpr * P
  int nchunks;   // ceil(L / lc)
};

template <bool VEC, bool REV>
__device__ __forceinline__ void n1_load(const float* __restrict__ row, int l0, int L, float fill, float (&o)[N1_P]) {
  if constexpr (VEC) {
#pragma unroll
    for (int c = 0; c < N1_P; c += 4) {
      float4 v = make_float4(fill, fill, fill, fill);
      if (l0 + c < L) v = __ldg(reinterpret_cast<const float4*>(row + (REV ? L - 4 - (l0 + c) : l0 + c)));
      o[c] = REV ? v.w : v.x; o[c + 1] = REV ? v.z : v.y; o[c + 2] = REV ? v.y : v.z; o[c + 3] = REV ? v.x : v.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < N1_P; ++i) o[i] = l0 + i < L ? __ldg(row + (REV ? L - 1 - (l0 + i) : l0 + i)) : fill;
  }
}
template <bool VEC, bool REV>
__device__ __forceinline__ void n1_store(float* __restrict__ row, int l0, int L, const float (&v)[N1_P]) {
  if constexpr (VEC) {
#pragma unroll
    for (int c = 0; c < N1_P; c += 4) {
      if (l0 + c < L) {
        const float4 q = REV ? make_float4(v[c + 3], v[c + 2], v[c + 1], v[c]) : make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
        *reinterpret_cast<float4*>(row + (REV ? L - 4 - (l0 + c) : l0 + c)) = q;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < N1_P; ++i)
      if (l0 + i < L) row[REV ? L - 1 - (l0 + i) : l0 + i] = v[i];
  }
}
// dB / dC of 8 positions: plain store when this CTA holds the whole sum, red.global otherwise
template <bool VEC, bool REV>
__device__ __forceinline__ void n1_emit(float* __restrict__ row, int l0, int L, const float (&v)[N1_P], bool plain) {
  if constexpr (VEC) {
#pragma unroll
    for (int c = 0; c < N1_P; c += 4) {
      if (l0 + c < L) {
        float4* q4 = reinterpret_cast<float4*>(row + (REV ? L - 4 - (l0 + c) : l0 + c));
        const float4 x = REV ? make_float4(v[c + 3], v[c + 2], v[c + 1], v[c]) : make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
        if (plain) *q4 = x;
        else asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(q4), "f"(x.x), "f"(x.y), "f"(x.z), "f"(x.w) : "memory");
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < N1_P; ++i) {
      if (l0 + i < L) {
        float* q1 = row + (REV ? L - 1 - (l0 + i) : l0 + i);
        if (plain) *q1 = v[i];
        else atomicAdd(q1, v[i]);
      }
    }
  }
}

__device__ __forceinline__ void n1_bar(int id, int nthreads) {      // named barrier of one row lane (id 1 ... 15)
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Exclusive carry for every thread of a row + the row total, given the thread's own affine map h -> Pm h + Hm.
// UP: composition of the EARLIER threads (prefix); !UP: of the LATER threads (suffix). Rows of wpr > 1 warps synchronise
// on the named barrier `bar_id` (their own: row lanes of one CTA do not wait for each other).
template <bool UP>
__device__ __forceinline__ void n1_row_exclusive(float Pm, float Hm, int lane, int lis, int seg, int wir, int wpr, int bar_id,
                                                 float (*s_agg)[2], float& Pex, float& Hex, float& Ptot, float& Htot) {
  for (int off = 1; off < seg; off <<= 1) {
    const float Pp = UP ? __shfl_up_sync(0xffffffffu, Pm, off) : __shfl_down_sync(0xffffffffu, Pm, off);
    const float Hp = UP ? __shfl_up_sync(0xffffffffu, Hm, off) : __shfl_down_sync(0xffffffffu, Hm, off);
    const bool take = UP ? (lis >= off) : (lis + off < seg);
    if (take) { Hm = fmaf(Pm, Hp, Hm); Pm *= Pp; }
  }
  float Pe = UP ? __shfl_up_sync(0xffffffffu, Pm, 1) : __shfl_down_sync(0xffffffffu, Pm, 1);
  float He = UP ? __shfl_up_sync(0xffffffffu, Hm, 1) : __shfl_down_sync(0xffffffffu, Hm, 1);
  if (UP ? (lis == 0) : (lis == seg - 1)) { Pe = 1.f; He = 0.f; }
  if (wpr == 1) {
    const int src = lane - lis + (UP ? seg - 1 : 0);
    Ptot = __shfl_sync(0xffffffffu, Pm, src);
    Htot = __shfl_sync(0xffffffffu, Hm, src);
    Pex = Pe; Hex = He;
  } else {
    // the warp's aggregate goes to shared memory; afterwards every warp scans the row's <= 16 aggregates with shuffles
    if (UP ? (lis == 31) : (lis == 0)) { s_agg[wir][0] = Pm; s_agg[wir][1] = Hm; }
    n1_bar(bar_id, wpr * 32);
    float Pw = 1.f, Hw = 0.f;
    if (lane < wpr) { Pw = s_agg[lane][0]; Hw = s_agg[lane][1]; }
#pragma unroll
    for (int off = 1; off < N1_MAX_WARPS; off <<= 1) {
      const float Pp = UP ? __shfl_up_sync(0xffffffffu, Pw, off) : __shfl_down_sync(0xffffffffu, Pw, off);
      const float Hp = UP ? __shfl_up_sync(0xffffffffu, Hw, off) : __shfl_down_sync(0xffffffffu, Hw, off);
      const bool take = UP ? (lane >= off) : (lane + off < 32);
      if (take) { Hw = fmaf(Pw, Hp, Hw); Pw *= Pp; }       // lanes >= wpr hold the identity: harmless in either direction
    }
    const int nb = UP ? wir - 1 : wir + 1;                 // neighbour warp whose inclusive value is this warp's carry-in
    float Pq = __shfl_sync(0xffffffffu, Pw, nb & 31), Hq = __shfl_sync(0xffffffffu, Hw, nb & 31);
    if (UP ? (wir == 0) : (wir == wpr - 1)) { Pq = 1.f; Hq = 0.f; }
    Ptot = __shfl_sync(0xffffffffu, Pw, UP ? wpr - 1 : 0);
    Htot = __shfl_sync(0xffffffffu, Hw, UP ? wpr - 1 : 0);
    Hex = fmaf(Pe, Hq, He); Pex = Pe * Pq;
  }
}

struct N1Thread {
  int r, wir, lis, t;     // row lane inside the CTA, warp inside the row, lane inside the row segment, thread index along the row
};
__device__ __forceinline__ N1Thread n1_thread(const N1Geom gm) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  N1Thread q;
  if (gm.seg == 32) { q.r = warp / gm.wpr; q.wir = warp - q.r * gm.wpr; q.lis = lane; }
  else { q.r = warp * (32 / gm.seg) + lane / gm.seg; q.wir = 0; q.lis = lane % gm.seg; }
  q.t = q.wir * 32 + q.lis;
  return q;
}

// activated delta: softplus(raw + bias) with threshold 20, or raw + bias; out-of-range positions (raw = -inf) give 0
template <bool SP>
__device__ __forceinline__ float n1_act(float raw, float bias, bool in_range) {
  if constexpr (SP) return softplus20(raw + bias);
  return in_range ? raw + bias : 0.f;
}

// ------------------------------------------------------------------------------------------------- forward
// STATE: the carry-in of a row's first lane is st.h0 instead of 0
template <bool VEC, bool SP, bool STATE>
__global__ void __launch_bounds__(N1_MAX_WARPS * 32) scan_n1_fwd_kernel(const ScanParams p, const N1Geom gm, const ScanState st) {
  __shared__ float s_agg[2][N1_MAX_WARPS][2];
  const N1Thread q = n1_thread(gm);
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.z, g = blockIdx.y;
  const int row = blockIdx.x * gm.rt + q.r;
  const bool valid = q.r < gm.rt && row < p.dpg;
  const int d = g * p.dpg + (valid ? row : 0);
  const int L = valid ? p.L : 0;                         // invalid rows: every load / store predicated off
  const float A2 = p.A[d] * kLog2e;
  const float bias = p.bias ? p.bias[d] : 0.f;
  const float Dd = p.Dv ? p.Dv[d] : 0.f;
  const float* fu = static_cast<const float*>(p.u) + (int64_t)b * p.u_bs + (int64_t)(p.u_mod > 0 ? d % p.u_mod : d) * p.u_ds;
  const float* fd = static_cast<const float*>(p.delta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  const float* fB = static_cast<const float*>(p.Bm) + (int64_t)b * p.B_bs + (int64_t)g * p.B_gs;
  const float* fC = static_cast<const float*>(p.Cm) + (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;
  float* fo = p.out ? static_cast<float*>(p.out) + (int64_t)b * p.out_bs + (int64_t)d * p.out_ds : nullptr;
  const float dfill = SP ? -INFINITY : 0.f;

  auto body = [&](auto REVT) {
    constexpr bool REV = decltype(REVT)::value;
    float h_carry = (STATE && valid) ? st.h0[state_slot(p, b, d, 0)] : 0.f;
    for (int c = 0; c < gm.nchunks; ++c) {
      const int l0 = c * gm.lc + q.t * N1_P;
      float dl[N1_P], uu[N1_P], bb[N1_P], cc[N1_P];
      n1_load<VEC, REV>(fd, l0, L, dfill, dl);
      n1_load<VEC, REV>(fu, l0, L, 0.f, uu);
      n1_load<VEC, REV>(fB, l0, L, 0.f, bb);
      n1_load<VEC, REV>(fC, l0, L, 0.f, cc);
      // local scan from h = 0: hl = local state, pc = cumulative decay; beyond the end of the row the state is frozen
      float hl[N1_P], pc[N1_P];
      float h = 0.f, pm = 1.f;
#pragma unroll
      for (int i = 0; i < N1_P; ++i) {
        const float x = n1_act<SP>(dl[i], bias, l0 + i < L);
        const float a = ex2f(x * A2);
        h = fmaf(a, h, x * uu[i] * bb[i]);
        pm *= a;
        hl[i] = h; pc[i] = pm;
      }
      float Pex, Hex, Ptot, Htot;
      n1_row_exclusive<true>(pm, h, lane, q.lis, gm.seg, q.wir, gm.wpr, 1 + q.r, s_agg[c & 1] + q.r * gm.wpr, Pex, Hex, Ptot, Htot);
      const float h_in = fmaf(Pex, h_carry, Hex);             // state entering this thread's first position
      if (fo) {
        float y[N1_P];
#pragma unroll
        for (int i = 0; i < N1_P; ++i) y[i] = fmaf(cc[i], fmaf(pc[i], h_in, hl[i]), Dd * uu[i]);
        n1_store<VEC, REV>(fo, l0, L, y);
      }
      // chunk checkpoint every SS2D_CHUNK positions: the thread whose last position closes a chunk owns it
      if (p.ckpt != nullptr && (q.t & 3) == 3 && l0 < L) {
        const int idx = (l0 + N1_P) / SS2D_CHUNK - 1;
        if (idx < p.nck) p.ckpt[((int64_t)b * p.dim + d) * p.nck + idx] = fmaf(pc[N1_P - 1], h_in, hl[N1_P - 1]);
      }
      h_carry = fmaf(Ptot, h_carry, Htot);
    }
    if (p.last_state != nullptr && valid && q.t == 0) {
      const int64_t slot = (int64_t)b * p.dim + d;
      if (p.last_il) { p.last_state[2 * slot] = 0.f; p.last_state[2 * slot + 1] = h_carry; }
      else p.last_state[slot] = h_carry;
    }
  };
  if (p.layout == SS2D_LAYOUT_NATURAL && p.dirs[g] == 3) body(std::true_type{}); else body(std::false_type{});
}

// ------------------------------------------------------------------------------------------------- backward, shared math
// One row segment of 8 positions per thread: forward recompute, row-wide prefix / suffix scans, adjoint. On exit dub / ddl
// hold du / d(delta); dBv / dCv are ADDED to (accumulate over the rows a thread walks); accA / accD / accb likewise.
// STATE: t may be non-zero beyond the end of the row (it starts at dlast), so d(delta) is masked there explicitly.
template <bool SP, bool STATE>
__device__ __forceinline__ void n1_bwd_segment(float (&dl)[N1_P], const float (&uu)[N1_P], const float (&dy)[N1_P],
                                               const float (&bb)[N1_P], const float (&cB)[N1_P], int l0, int L, float A1,
                                               float bias, float Dd, float h_chunk, float& t_carry, int lane, const N1Thread q,
                                               const N1Geom gm, float (*s_agg0)[2], float (*s_agg1)[2], float (&dub)[N1_P],
                                               float (&ddl)[N1_P], float (&dBv)[N1_P], float (&dCv)[N1_P], float& accA,
                                               float& accD, float& accb) {
  const float A2 = A1 * kLog2e;
  float a[N1_P], hh[N1_P], cc[N1_P];
  float h = 0.f, pm = 1.f;
#pragma unroll
  for (int i = 0; i < N1_P; ++i) {
    const float x = n1_act<SP>(dl[i], bias, l0 + i < L);
    dl[i] = x;
    a[i] = ex2f(x * A2);
    h = fmaf(a[i], h, x * uu[i] * bb[i]);
    pm *= a[i];
    hh[i] = h;
    cc[i] = cB[i] * dy[i];                                     // c_l = C_l dy_l
  }
  float Pex, Hex, Ptot, Htot;
  n1_row_exclusive<true>(pm, h, lane, q.lis, gm.seg, q.wir, gm.wpr, 1 + q.r, s_agg0, Pex, Hex, Ptot, Htot);
  const float h_in = fmaf(Pex, h_chunk, Hex);                  // true state before this thread's first position
  {
    float pc = 1.f;
#pragma unroll
    for (int i = 0; i < N1_P; ++i) { pc *= a[i]; hh[i] = fmaf(pc, h_in, hh[i]); }
  }
  // reverse aggregate: t_l = a_l (c_l + t_(l+1)) as an affine map of the t entering from the right
  float tq = 0.f, qm = 1.f;
#pragma unroll
  for (int i = N1_P - 1; i >= 0; --i) { tq = a[i] * (cc[i] + tq); qm *= a[i]; }
  float Qex, Tex, Qtot, Ttot;
  n1_row_exclusive<false>(qm, tq, lane, q.lis, gm.seg, q.wir, gm.wpr, 1 + q.r, s_agg1, Qex, Tex, Qtot, Ttot);
  float t_next = fmaf(Qex, t_carry, Tex);                      // t of the position right after this thread's last one
#pragma unroll
  for (int i = N1_P - 1; i >= 0; --i) {
    const float gi = cc[i] + t_next;                           // g_i = C_i dy_i + a_(i+1) g_(i+1)
    const float ti = a[i] * gi;
    t_next = ti;
    const float hprev = i > 0 ? hh[i - 1] : h_in;
    const float sB = gi * bb[i];
    const float w = ti * hprev;
    float dd = fmaf(uu[i], sB, w * A1);
    if constexpr (SP) {      // sigmoid(raw) = 1 - exp(-softplus(raw)); series for small delta avoids cancellation
      const float de = dl[i];
      dd *= de < 0.015625f ? de * (1.f - de * (0.5f - de * 0.16666667f)) : 1.f - ex2f(-de * kLog2e);
    }
    if (STATE && l0 + i >= L) dd = 0.f;
    dub[i] = fmaf(Dd, dy[i], dl[i] * sB);
    ddl[i] = dd;                                               // 0 beyond the row: u = dout = 0 there and t has not started
    dBv[i] = fmaf(gi * dl[i], uu[i], dBv[i]);
    dCv[i] = fmaf(dy[i], hh[i], dCv[i]);
    accA = fmaf(w, dl[i], accA);
    accD = fmaf(dy[i], uu[i], accD);
    accb += dd;
  }
  t_carry = fmaf(Qtot, t_carry, Ttot);
}

// sum over the seg x wpr threads of a row; result valid in the thread with q.t == 0
__device__ __forceinline__ void n1_row_sum3(float& x, float& y, float& z, int lane, const N1Thread q, const N1Geom gm,
                                            float (*s_red)[3], int bar_id) {
  for (int off = gm.seg >> 1; off >= 1; off >>= 1) {
    x += __shfl_xor_sync(0xffffffffu, x, off);
    y += __shfl_xor_sync(0xffffffffu, y, off);
    z += __shfl_xor_sync(0xffffffffu, z, off);
  }
  if (gm.wpr > 1) {
    if (lane == 0) { s_red[q.wir][0] = x; s_red[q.wir][1] = y; s_red[q.wir][2] = z; }
    n1_bar(bar_id, gm.wpr * 32);
    if (q.t == 0) {
      x = y = z = 0.f;
      for (int w = 0; w < gm.wpr; ++w) { x += s_red[w][0]; y += s_red[w][1]; z += s_red[w][2]; }
    }
    n1_bar(bar_id, gm.wpr * 32);        // s_red is reused by the next row
  }
}

__device__ __forceinline__ void n1_emit_row_grads(const ScanParams& p, int b, int d, float accA, float accD, float accb,
                                                  float* dA, float* dD, float* dbias, int grads_zeroed) {
  if (grads_zeroed) {
    atomicAdd(dA + d, accA);
    if (dD) atomicAdd(dD + d, accD);
    if (dbias) atomicAdd(dbias + d, accb);
  } else {
    float* dst = p.part + ((int64_t)b * p.dim + d) * 3;
    dst[0] = accA; dst[1] = accD; dst[2] = accb;
  }
}

// ------------------------------------------------------------------------------------------------- backward, one row per lane
// Any L (rows longer than 16 warps x 256 positions are walked in chunks, last to first, from the forward's checkpoints), any
// alignment. grads_zeroed != 0: dA / dD / d(delta_bias) are caller-zeroed accumulators; else per-(batch, channel) partials
// go to p.part and scan_bwd_finalize sums them.
// STATE: chunk 0 starts from st.h0, the reverse carry from st.dlast, and st.dh0 receives the adjoint of h0 (each may be null)
template <bool VEC, bool SP, bool STATE, bool DET>
__global__ void __launch_bounds__(N1_MAX_WARPS * 32) scan_n1_bwd_kernel(const ScanParams p, const N1Geom gm, float* __restrict__ dA,
    float* __restrict__ dD, float* __restrict__ dbias, int grads_zeroed, const ScanState st) {
  extern __shared__ __align__(16) float s_slab[];          // [2][rt][lc]: per-row dB / dC of the current chunk (rt > 1)
  __shared__ float s_agg[2][N1_MAX_WARPS][2];
  __shared__ float s_red[N1_MAX_WARPS][3];
  const N1Thread q = n1_thread(gm);
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.z, g = blockIdx.y;
  const int row = blockIdx.x * gm.rt + q.r;
  const bool valid = q.r < gm.rt && row < p.dpg;
  const int d = g * p.dpg + (valid ? row : 0);
  const int L = valid ? p.L : 0;
  const bool plain = DET || gridDim.x == 1;
  const float A1 = p.A[d];
  const float bias = p.bias ? p.bias[d] : 0.f;
  const float Dd = p.Dv ? p.Dv[d] : 0.f;
  const int u_ch = p.u_mod > 0 ? d % p.u_mod : d;
  const float* fu = static_cast<const float*>(p.u) + (int64_t)b * p.u_bs + (int64_t)u_ch * p.u_ds;
  const float* fd = static_cast<const float*>(p.delta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  const float* fy = static_cast<const float*>(p.dout) + (int64_t)b * p.out_bs + (int64_t)u_ch * p.out_ds;
  const float* fB = static_cast<const float*>(p.Bm) + (int64_t)b * p.B_bs + (int64_t)g * p.B_gs;
  const float* fC = static_cast<const float*>(p.Cm) + (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;
  float* fdu = static_cast<float*>(p.du) + (p.u_mod > 0 ? ((int64_t)b * p.dim + d) * (int64_t)p.L : (int64_t)b * p.u_bs + (int64_t)d * p.u_ds);
  float* fdd = static_cast<float*>(p.ddelta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  float* dBrow = (DET ? det_slab(p, 0, blockIdx.x) : p.dB) + (int64_t)(b * p.G + g) * p.L;
  float* dCrow = (DET ? det_slab(p, 1, blockIdx.x) : p.dC) + (int64_t)(b * p.G + g) * p.L;
  const float dfill = SP ? -INFINITY : 0.f;

  auto body = [&](auto REVT) {
    constexpr bool REV = decltype(REVT)::value;
    float t_carry = (STATE && st.dlast && valid) ? st.dlast[state_slot(p, b, d, 0)] : 0.f;   // a_l g_l of the first position of the chunk after this one
    float accA = 0.f, accD = 0.f, accb = 0.f;
    for (int c = gm.nchunks - 1; c >= 0; --c) {
      const int l0 = c * gm.lc + q.t * N1_P;
      float dl[N1_P], uu[N1_P], bb[N1_P], cc[N1_P], dy[N1_P];
      n1_load<VEC, REV>(fd, l0, L, dfill, dl);
      n1_load<VEC, REV>(fu, l0, L, 0.f, uu);
      n1_load<VEC, REV>(fy, l0, L, 0.f, dy);
      n1_load<VEC, REV>(fB, l0, L, 0.f, bb);
      n1_load<VEC, REV>(fC, l0, L, 0.f, cc);
      // state entering the chunk: checkpoint written by the forward at the end of the previous SS2D_CHUNK block
      const float h_chunk = (c > 0 && valid) ? __ldg(p.ckpt_in + ((int64_t)b * p.dim + d) * p.nck + (c * gm.lc) / SS2D_CHUNK - 1)
                            : (STATE && st.h0 && valid) ? __ldg(st.h0 + state_slot(p, b, d, 0)) : 0.f;
      float dub[N1_P], ddl[N1_P], dBv[N1_P], dCv[N1_P];
#pragma unroll
      for (int i = 0; i < N1_P; ++i) { dBv[i] = 0.f; dCv[i] = 0.f; }
      n1_bwd_segment<SP, STATE>(dl, uu, dy, bb, cc, l0, L, A1, bias, Dd, h_chunk, t_carry, lane, q, gm, s_agg[0] + q.r * gm.wpr,
                         s_agg[1] + q.r * gm.wpr, dub, ddl, dBv, dCv, accA, accD, accb);
      n1_store<VEC, REV>(fdu, l0, L, dub);
      n1_store<VEC, REV>(fdd, l0, L, ddl);
      // ---- dB / dC: summed over the rows of this CTA, then one store (CTA = whole group) or reduction per 4 positions ----
      if (gm.rt == 1) {
        n1_emit<VEC, REV>(dBrow, l0, L, dBv, plain);
        n1_emit<VEC, REV>(dCrow, l0, L, dCv, plain);
      } else {
        float* slabB = s_slab + (size_t)q.r * gm.lc + q.t * N1_P;
        float* slabC = slabB + (size_t)gm.rt * gm.lc;
        if (q.r < gm.rt) {
          *reinterpret_cast<float4*>(slabB) = make_float4(dBv[0], dBv[1], dBv[2], dBv[3]);
          *reinterpret_cast<float4*>(slabB + 4) = make_float4(dBv[4], dBv[5], dBv[6], dBv[7]);
          *reinterpret_cast<float4*>(slabC) = make_float4(dCv[0], dCv[1], dCv[2], dCv[3]);
          *reinterpret_cast<float4*>(slabC + 4) = make_float4(dCv[4], dCv[5], dCv[6], dCv[7]);
        }
        __syncthreads();
        const int L0 = p.L, c8 = gm.lc / N1_P;
        for (int i = threadIdx.x; i < 2 * c8; i += blockDim.x) {
          const int which = i / c8, pos = (i - which * c8) * N1_P;
          const int l = c * gm.lc + pos;
          if (l >= L0) continue;
          float acc[N1_P];
#pragma unroll
          for (int e = 0; e < N1_P; ++e) acc[e] = 0.f;
          const float* col = s_slab + (size_t)which * gm.rt * gm.lc + pos;
          for (int rr = 0; rr < gm.rt; ++rr) {
            const float4 v0 = *reinterpret_cast<const float4*>(col + (size_t)rr * gm.lc);
            const float4 v1 = *reinterpret_cast<const float4*>(col + (size_t)rr * gm.lc + 4);
            acc[0] += v0.x; acc[1] += v0.y; acc[2] += v0.z; acc[3] += v0.w;
            acc[4] += v1.x; acc[5] += v1.y; acc[6] += v1.z; acc[7] += v1.w;
          }
          n1_emit<VEC, REV>(which == 0 ? dBrow : dCrow, l, L0, acc, plain);
        }
        __syncthreads();
      }
    }
    if (STATE && st.dh0 && q.t == 0 && valid) st.dh0[state_slot(p, b, d, 0)] = t_carry;      // a_0 g_0
    n1_row_sum3(accA, accD, accb, lane, q, gm, s_red + q.r * gm.wpr, 1 + q.r);
    if (q.t == 0 && valid) n1_emit_row_grads(p, b, d, accA, accD, accb, dA, dD, dbias, !DET && grads_zeroed);
  };
  if (p.layout == SS2D_LAYOUT_NATURAL && p.dirs[g] == 3) body(std::true_type{}); else body(std::false_type{});
}

// ------------------------------------------------------------------------------------------------- backward, rows walked per lane
// 16-byte aligned fp32 rows of at least one warp: see the header comment. Rows longer than 16 warps x 256 positions are
// walked in chunks of 8 warps x 256, last to first (chunk-outer, rows-inner, so dB / dC of a chunk stay in registers across the
// rows; the per-row reverse carry lives in shared memory, the forward state entering a chunk comes from the forward's
// checkpoints). Shared memory: per row lane a 2-stage ring of [delta | u | dout] row pieces (TMA bulk copies), reused after
// each chunk as the slab that sums dB / dC over the row lanes.
constexpr int N1_MAX_RSEQ = 64;

// STATE: as scan_n1_bwd_kernel
template <bool SP, bool STATE, bool DET>
__global__ void __launch_bounds__(N1_MAX_WARPS * 32) scan_n1_bwd_rows_kernel(const ScanParams p, const N1Geom gm, float* __restrict__ dA,
    float* __restrict__ dD, float* __restrict__ dbias, int grads_zeroed, const ScanState st) {
  extern __shared__ __align__(128) float s_ring[];         // [rt][2 stages][3][lr]
  __shared__ float s_agg[2][N1_MAX_WARPS][2];
  __shared__ float s_red[2][N1_MAX_WARPS][3];
  __shared__ float s_tc[N1_MAX_WARPS][N1_MAX_RSEQ];        // reverse carry of each row between chunks (multi-chunk rows)
  __shared__ __align__(8) uint64_t s_full[N1_MAX_WARPS][2];
  __shared__ float s_racc[DET ? N1_MAX_RSEQ : 1][3];       // DET, multi-chunk rows (one row lane): per-row running sums
  N1Geom gq = gm;
  gq.seg = 32;                                             // compile-time constant for the shuffle scans below
  const N1Thread q = n1_thread(gq);
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.z, g = blockIdx.y;
  const int L = p.L;
  const int lr = gm.nchunks == 1 ? ((L + 31) & ~31) : gm.lc;          // ring row length (floats), a multiple of 128 bytes
  const int rows_cta = gm.rt * gm.rseq;
  const int row_base = blockIdx.x * rows_cta + q.r;
  // rows this lane walks: row_base + j rt for j < nj
  const int nj = row_base < p.dpg ? min(gm.rseq, (p.dpg - row_base + gm.rt - 1) / gm.rt) : 0;
  const bool plain = DET || gridDim.x == 1;
  const float* fB = static_cast<const float*>(p.Bm) + (int64_t)b * p.B_bs + (int64_t)g * p.B_gs;
  const float* fC = static_cast<const float*>(p.Cm) + (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;
  float* dBrow = (DET ? det_slab(p, 0, blockIdx.x) : p.dB) + (int64_t)(b * p.G + g) * L;
  float* dCrow = (DET ? det_slab(p, 1, blockIdx.x) : p.dC) + (int64_t)(b * p.G + g) * L;
  float* ring = s_ring + (size_t)q.r * 6 * lr;
  const bool leader = q.t == 0;                            // issues this row lane's TMA copies
  const int total_it = nj * gm.nchunks;

  auto body = [&](auto REVT) {
    constexpr bool REV = decltype(REVT)::value;
    auto issue = [&](int it) {                             // leader only; it = (chunk counted from the end) * nj + j
      if (it >= total_it) return;
      const int ci = it / nj, j = it - ci * nj, c = gm.nchunks - 1 - ci, s = it & 1;
      const int d = g * p.dpg + row_base + j * gm.rt;
      const int u_ch = p.u_mod > 0 ? d % p.u_mod : d;
      const int len = min(gm.lc, L - c * gm.lc);
      const int64_t m0 = REV ? L - c * gm.lc - len : c * gm.lc;       // first memory position of the piece
      const uint32_t bytes = (uint32_t)len * 4u;
      float* stg = ring + (size_t)s * 3 * lr;
      mbar_arrive_expect_tx(&s_full[q.r][s], 3u * bytes);
      tma_load_1d(stg, static_cast<const float*>(p.delta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds + m0, bytes, &s_full[q.r][s]);
      tma_load_1d(stg + lr, static_cast<const float*>(p.u) + (int64_t)b * p.u_bs + (int64_t)u_ch * p.u_ds + m0, bytes, &s_full[q.r][s]);
      tma_load_1d(stg + 2 * lr, static_cast<const float*>(p.dout) + (int64_t)b * p.out_bs + (int64_t)u_ch * p.out_ds + m0, bytes, &s_full[q.r][s]);
    };
    if (leader) { mbar_init(&s_full[q.r][0], 1); mbar_init(&s_full[q.r][1], 1); fence_mbar_init(); }
    __syncthreads();
    if (leader) { issue(0); issue(1); }

    for (int ci = 0; ci < gm.nchunks; ++ci) {
      const int c = gm.nchunks - 1 - ci;
      const int len = min(gm.lc, L - c * gm.lc);           // positions of this chunk
      const int lq = q.t * N1_P;                           // this thread's first position inside the chunk
      const int l0 = c * gm.lc + lq;
      float bb[N1_P], cB[N1_P];
      n1_load<true, REV>(fB, l0, nj > 0 ? L : 0, 0.f, bb);
      n1_load<true, REV>(fC, l0, nj > 0 ? L : 0, 0.f, cB);
      float dBv[N1_P], dCv[N1_P];
#pragma unroll
      for (int i = 0; i < N1_P; ++i) { dBv[i] = 0.f; dCv[i] = 0.f; }
      for (int j = 0; j < nj; ++j) {
        const int it = ci * nj + j, s = it & 1;
        const int d = g * p.dpg + row_base + j * gm.rt;
        const float A1 = p.A[d];
        const float bias = p.bias ? p.bias[d] : 0.f;
        const float Dd = p.Dv ? p.Dv[d] : 0.f;
        const float h_chunk = c > 0 ? __ldg(p.ckpt_in + ((int64_t)b * p.dim + d) * p.nck + (c * gm.lc) / SS2D_CHUNK - 1)
                              : (STATE && st.h0) ? __ldg(st.h0 + state_slot(p, b, d, 0)) : 0.f;
        // written one chunk ago, several row-lane barriers back
        float t_carry = ci > 0 ? s_tc[q.r][j] : (STATE && st.dlast) ? st.dlast[state_slot(p, b, d, 0)] : 0.f;
        mbar_wait(&s_full[q.r][s], (uint32_t)(it >> 1) & 1u);
        const float* stg = ring + (size_t)s * 3 * lr;
        float dl[N1_P], uu[N1_P], dy[N1_P];
#pragma unroll
        for (int cch = 0; cch < N1_P; cch += 4) {
          const bool in = lq + cch < len;
          const int off = REV ? len - 4 - (lq + cch) : lq + cch;
          float4 v0 = make_float4(SP ? -INFINITY : 0.f, SP ? -INFINITY : 0.f, SP ? -INFINITY : 0.f, SP ? -INFINITY : 0.f);
          float4 v1 = make_float4(0.f, 0.f, 0.f, 0.f), v2 = v1;
          if (in) {
            v0 = *reinterpret_cast<const float4*>(stg + off);
            v1 = *reinterpret_cast<const float4*>(stg + lr + off);
            v2 = *reinterpret_cast<const float4*>(stg + 2 * lr + off);
          }
          dl[cch] = REV ? v0.w : v0.x; dl[cch + 1] = REV ? v0.z : v0.y; dl[cch + 2] = REV ? v0.y : v0.z; dl[cch + 3] = REV ? v0.x : v0.w;
          uu[cch] = REV ? v1.w : v1.x; uu[cch + 1] = REV ? v1.z : v1.y; uu[cch + 2] = REV ? v1.y : v1.z; uu[cch + 3] = REV ? v1.x : v1.w;
          dy[cch] = REV ? v2.w : v2.x; dy[cch + 1] = REV ? v2.z : v2.y; dy[cch + 2] = REV ? v2.y : v2.z; dy[cch + 3] = REV ? v2.x : v2.w;
        }
        float dub[N1_P], ddl[N1_P];
        float accA = 0.f, accD = 0.f, accb = 0.f;
        n1_bwd_segment<SP, STATE>(dl, uu, dy, bb, cB, l0, L, A1, bias, Dd, h_chunk, t_carry, lane, q, gq, s_agg[0] + q.r * gm.wpr,
                                  s_agg[1] + q.r * gm.wpr, dub, ddl, dBv, dCv, accA, accD, accb);
        if (STATE && st.dh0 && c == 0 && leader) st.dh0[state_slot(p, b, d, 0)] = t_carry;      // a_0 g_0
        // every thread of the row lane passed the barriers inside the segment after its reads of stage s: refill it
        if (gm.wpr == 1) __syncwarp();
        if (leader) { fence_proxy_async(); issue(it + 2); if (gm.nchunks > 1) s_tc[q.r][j] = t_carry; }
        float* fdu = static_cast<float*>(p.du) + (p.u_mod > 0 ? ((int64_t)b * p.dim + d) * (int64_t)L : (int64_t)b * p.u_bs + (int64_t)d * p.u_ds);
        float* fdd = static_cast<float*>(p.ddelta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
        n1_store<true, REV>(fdu, l0, L, dub);
        n1_store<true, REV>(fdd, l0, L, ddl);
        // per-row sums of dA / dD / d(delta_bias): shuffle tree, one shared-memory hop, warp 0 of the row finishes
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
          accA += __shfl_xor_sync(0xffffffffu, accA, off);
          accD += __shfl_xor_sync(0xffffffffu, accD, off);
          accb += __shfl_xor_sync(0xffffffffu, accb, off);
        }
        if (gm.wpr > 1) {
          float (*red)[3] = s_red[it & 1] + q.r * gm.wpr;
          if (lane == 0) { red[q.wir][0] = accA; red[q.wir][1] = accD; red[q.wir][2] = accb; }
          n1_bar(1 + q.r, gm.wpr * 32);
          if (q.wir == 0) {
            accA = lane < gm.wpr ? red[lane][0] : 0.f;
            accD = lane < gm.wpr ? red[lane][1] : 0.f;
            accb = lane < gm.wpr ? red[lane][2] : 0.f;
#pragma unroll
            for (int off = 8; off >= 1; off >>= 1) {
              accA += __shfl_xor_sync(0xffffffffu, accA, off);
              accD += __shfl_xor_sync(0xffffffffu, accD, off);
              accb += __shfl_xor_sync(0xffffffffu, accb, off);
            }
          }
        }
        if (q.t == 0) {
          if (!DET && grads_zeroed) {
            atomicAdd(dA + d, accA);
            if (dD) atomicAdd(dD + d, accD);
            if (dbias) atomicAdd(dbias + d, accb);
          } else {           // partials for the finalize pass (outside DET the host sends only single-chunk rows here)
            bool last = true;
            if constexpr (DET) {
              if (gm.nchunks > 1) {                        // running sums over the chunks, added in chunk order
                float* acc = s_racc[j];
                if (ci > 0) { accA = acc[0] + accA; accD = acc[1] + accD; accb = acc[2] + accb; }
                last = ci == gm.nchunks - 1;
                if (!last) { acc[0] = accA; acc[1] = accD; acc[2] = accb; }
              }
            }
            if (last) {
              float* dst = p.part + ((int64_t)b * p.dim + d) * 3;
              dst[0] = accA; dst[1] = accD; dst[2] = accb;
            }
          }
        }
      }
      // ---- dB / dC of this chunk over the rows the CTA walked: sum over the row lanes through shared memory ----
      if (gm.rt == 1) {
        if (nj > 0) {
          n1_emit<true, REV>(dBrow, l0, L, dBv, plain);
          n1_emit<true, REV>(dCrow, l0, L, dCv, plain);
        }
      } else {      // single-chunk rows: the ring is idle by now and doubles as the slab; chunked rows have their own slab
        __syncthreads();                                   // also orders this chunk's slab writes after the previous chunk's reads
        float* slab0 = s_ring + (gm.nchunks > 1 ? (size_t)gm.rt * 6 * lr : 0);
        float* slabB = slab0 + (size_t)q.r * gm.lc + lq;
        float* slabC = slabB + (size_t)gm.rt * gm.lc;
        *reinterpret_cast<float4*>(slabB) = make_float4(dBv[0], dBv[1], dBv[2], dBv[3]);
        *reinterpret_cast<float4*>(slabB + 4) = make_float4(dBv[4], dBv[5], dBv[6], dBv[7]);
        *reinterpret_cast<float4*>(slabC) = make_float4(dCv[0], dCv[1], dCv[2], dCv[3]);
        *reinterpret_cast<float4*>(slabC + 4) = make_float4(dCv[4], dCv[5], dCv[6], dCv[7]);
        __syncthreads();
        const int c8 = gm.lc / N1_P;
        for (int i = threadIdx.x; i < 2 * c8; i += blockDim.x) {
          const int which = i / c8, pos = (i - which * c8) * N1_P;
          if (c * gm.lc + pos >= L) continue;
          float acc[N1_P];
#pragma unroll
          for (int e = 0; e < N1_P; ++e) acc[e] = 0.f;
          const float* col = slab0 + (size_t)which * gm.rt * gm.lc + pos;
          for (int rr = 0; rr < gm.rt; ++rr) {
            const float4 v0 = *reinterpret_cast<const float4*>(col + (size_t)rr * gm.lc);
            const float4 v1 = *reinterpret_cast<const float4*>(col + (size_t)rr * gm.lc + 4);
            acc[0] += v0.x; acc[1] += v0.y; acc[2] += v0.z; acc[3] += v0.w;
            acc[4] += v1.x; acc[5] += v1.y; acc[6] += v1.z; acc[7] += v1.w;
          }
          n1_emit<true, REV>(which == 0 ? dBrow : dCrow, c * gm.lc + pos, L, acc, plain);
        }
      }
    }
  };
  if (p.layout == SS2D_LAYOUT_NATURAL && p.dirs[g] == 3) body(std::true_type{}); else body(std::false_type{});
}

// ------------------------------------------------------------------------------------------------- host side
static bool n1_aligned16(const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0; }

// fp32 everywhere, d_state 1 in a single pass, contiguous traversal for every group
static bool n1_eligible(const ScanParams& p, bool backward) {
  if (p.N != 1 || p.A_ld != 1 || p.accum || p.io_dtype != SS2D_F32) return false;
  if ((p.out != nullptr || backward) && p.out_dtype != SS2D_F32) return false;
  if (p.u_mod > 0 && p.dim % p.u_mod != 0) return false;
  for (int g = 0; g < p.G; ++g) {
    const int dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
    if (dir == 2 || dir == 4) return false;
  }
  return true;
}

static bool n1_vec(const ScanParams& p, bool backward) {
  if (p.L & 3) return false;
  const int64_t strides[] = {p.u_bs, p.u_ds, p.dl_bs, p.dl_ds, p.B_bs, p.B_gs, p.C_bs, p.C_gs};
  for (int64_t s : strides) if (s & 3) return false;
  if (!n1_aligned16(p.u) || !n1_aligned16(p.delta) || !n1_aligned16(p.Bm) || !n1_aligned16(p.Cm)) return false;
  if (!backward) return p.out == nullptr || (n1_aligned16(p.out) && !(p.out_bs & 3) && !(p.out_ds & 3));
  return n1_aligned16(p.dout) && !(p.out_bs & 3) && !(p.out_ds & 3) && n1_aligned16(p.du) && n1_aligned16(p.ddelta) &&
         n1_aligned16(p.dB) && n1_aligned16(p.dC);
}

static N1Geom n1_geometry(const ScanParams& p) {
  N1Geom gm;
  const int L = p.L;
  if (L <= 32 * N1_P) {                       // one warp (or a fraction of it) per row
    gm.seg = 4;
    while (gm.seg < 32 && gm.seg * N1_P < L) gm.seg <<= 1;
    gm.wpr = 1;
  } else {                                    // whole warps; a row of up to 16 warps x 256 positions is a single pass
    gm.seg = 32;
    const int need = (L + 32 * N1_P - 1) / (32 * N1_P);
    gm.wpr = need <= N1_MAX_WARPS ? need : 8;
  }
  gm.lc = gm.seg * gm.wpr * N1_P;
  gm.nchunks = (L + gm.lc - 1) / gm.lc;
  gm.rseq = 1;
  // row lanes per CTA: fill about 8 warps, but keep at least ~2 CTAs per SM in the grid when the problem is that small
  const int rows_per_warp = gm.seg == 32 ? 1 : 32 / gm.seg;
  const int warps = gm.wpr > 8 ? gm.wpr : 8;
  int rt = gm.seg == 32 ? warps / gm.wpr : warps * rows_per_warp;
  const int sms = sm_count_current_device();
  while (rt > rows_per_warp && rt > 1 && (long)((p.dpg + rt - 1) / rt) * p.G * p.batch < 2L * sms) rt = (rt + 1) / 2;
  if (gm.seg < 32) rt = (rt + rows_per_warp - 1) / rows_per_warp * rows_per_warp;     // whole warps
  if (rt > p.dpg) rt = gm.seg == 32 ? p.dpg : (p.dpg + rows_per_warp - 1) / rows_per_warp * rows_per_warp;
  gm.rt = rt < 1 ? 1 : rt;
  return gm;
}

static int n1_threads(const N1Geom& gm) {
  return gm.seg == 32 ? gm.rt * gm.wpr * 32 : gm.rt / (32 / gm.seg) * 32;
}

template <bool STATE>
static cudaError_t n1_fwd_launch(const ScanParams& p, const ScanState& st, const N1Geom& gm, dim3 grid, int nt, bool vec,
                                 cudaStream_t stream) {
  const bool sp = p.softplus != 0;
  if (vec && sp) scan_n1_fwd_kernel<true, true, STATE><<<grid, nt, 0, stream>>>(p, gm, st);
  else if (vec) scan_n1_fwd_kernel<true, false, STATE><<<grid, nt, 0, stream>>>(p, gm, st);
  else if (sp) scan_n1_fwd_kernel<false, true, STATE><<<grid, nt, 0, stream>>>(p, gm, st);
  else scan_n1_fwd_kernel<false, false, STATE><<<grid, nt, 0, stream>>>(p, gm, st);
  return cudaGetLastError();
}

// Returns true when the lean path took the call (*err holds the launch status).
bool scan_n1_fwd_try(const ScanParams& p, const ScanState& st, cudaStream_t stream, cudaError_t* err) {
  if (!n1_eligible(p, false)) return false;
  const N1Geom gm = n1_geometry(p);
  dim3 grid((p.dpg + gm.rt - 1) / gm.rt, p.G, p.batch);
  const int nt = n1_threads(gm);
  const bool vec = n1_vec(p, false);
  *err = st.h0 ? n1_fwd_launch<true>(p, st, gm, grid, nt, vec, stream) : n1_fwd_launch<false>(p, st, gm, grid, nt, vec, stream);
  return true;
}

// Geometry of the rows kernel: whole warps per row; single-pass rows up to 16 warps x 256 positions share the CTA between up to
// 8 row lanes (<= 16 warps, <= 15 named barriers, <= 96 KB of ring), longer rows take one lane of 8 warps and are chunked.
// rseq rows per lane such that the grid still has ~1.5 CTAs per SM when the groups are big enough to be split, one CTA per
// group otherwise (then dB / dC are plain stores and the result is deterministic).
static bool n1_rows_geometry(const ScanParams& p, int grads_zeroed, N1Geom* out, size_t* smem) {
  if (p.L <= 32 * N1_P / 2) return false;
  N1Geom gm;
  gm.seg = 32;
  const int need = (p.L + 32 * N1_P - 1) / (32 * N1_P);
  int rt;
  size_t lr;
  if (need <= N1_MAX_WARPS) {
    gm.wpr = need; gm.nchunks = 1;
    lr = (size_t)((p.L + 31) & ~31);
    rt = N1_MAX_WARPS / gm.wpr;
    if (rt > 8) rt = 8;
    if (rt > p.dpg) rt = p.dpg;
    while (rt > 1 && (size_t)rt * 6 * lr * sizeof(float) > 96 * 1024) --rt;
  } else {
    // long rows: one lane of 8 warps x 256 positions per chunk, 2 CTAs per SM. (Measured on the 512^2 batch-64 stage-1 shape:
    // backward 409 us this way, 475 us with 8 row lanes of 2 warps x 256 — the lanes then meet at a CTA-wide barrier for the
    // dB / dC slab after every chunk and B / C are fetched 4x as often.)
    if (!grads_zeroed && !p.det) return false;               // per-chunk row sums: atomics, or shared memory in DET mode
    gm.wpr = 8;
    rt = 1;
    lr = (size_t)gm.wpr * 32 * N1_P;
    gm.nchunks = (int)((p.L + lr - 1) / lr);
  }
  gm.lc = gm.wpr * 32 * N1_P;
  const int sms = sm_count_current_device();
  const long groups = (long)p.G * p.batch;
  long blocks = (3L * sms / 2 + groups - 1) / groups;                   // row blocks per group we would like
  const long max_blocks = (p.dpg + rt - 1) / rt;
  if (blocks > max_blocks) blocks = max_blocks;
  if (blocks < 1) blocks = 1;
  gm.rt = rt;
  gm.rseq = (int)((p.dpg + rt * blocks - 1) / (rt * blocks));
  if (gm.rseq > N1_MAX_RSEQ) return false;
  const size_t ring = (size_t)rt * 6 * lr * sizeof(float), slab = (size_t)2 * rt * gm.lc * sizeof(float);
  *smem = gm.nchunks > 1 ? ring + (rt > 1 ? slab : 0) : (ring > slab ? ring : slab);      // single-chunk rows reuse the idle ring
  *out = gm;
  return true;
}

static int n1_one_row_smem(const N1Geom& gm) { return gm.rt > 1 ? 2 * gm.rt * gm.lc * (int)sizeof(float) : 0; }

// deterministic mode: one slab per CTA along the group, for whichever of the two kernels takes the call
int scan_n1_bwd_det_slabs(const ScanParams& p) {
  if (!n1_eligible(p, true)) return 0;
  int slabs = 0;
  N1Geom gr;
  size_t smem_rows = 0;
  if (n1_rows_geometry(p, 0, &gr, &smem_rows)) slabs = (p.dpg + gr.rt * gr.rseq - 1) / (gr.rt * gr.rseq);
  const N1Geom gm = n1_geometry(p);
  if (n1_one_row_smem(gm) <= 40 * 1024) slabs = std::max(slabs, (p.dpg + gm.rt - 1) / gm.rt);
  return slabs;
}

template <bool DET, bool STATE>
static cudaError_t n1_bwd_rows_launch(const ScanParams& p, const ScanState& st, const N1Geom& gr, size_t smem, float* dA, float* dD,
                                      float* dbias, int grads_zeroed, cudaStream_t stream) {
  const bool sp = p.softplus != 0;
  static PerDeviceOnce once_sp, once_nosp;
  const auto kern = sp ? scan_n1_bwd_rows_kernel<true, STATE, DET> : scan_n1_bwd_rows_kernel<false, STATE, DET>;
  cudaError_t e = func_attr_once(sp ? once_sp : once_nosp, reinterpret_cast<const void*>(kern),
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 136 * 1024);
  if (e != cudaSuccess) return e;
  const int rows_cta = gr.rt * gr.rseq;
  dim3 grid((p.dpg + rows_cta - 1) / rows_cta, p.G, p.batch);
  const int nt = gr.rt * gr.wpr * 32;
  kern<<<grid, nt, smem, stream>>>(p, gr, dA, dD, dbias, grads_zeroed, st);
  return cudaGetLastError();
}

template <bool DET, bool STATE>
static cudaError_t n1_bwd_launch(const ScanParams& p, const ScanState& st, const N1Geom& gm, bool vec, float* dA, float* dD,
                                 float* dbias, int grads_zeroed, cudaStream_t stream) {
  const bool sp = p.softplus != 0;
  dim3 grid((p.dpg + gm.rt - 1) / gm.rt, p.G, p.batch);
  const size_t smem = n1_one_row_smem(gm);
  const int nt = n1_threads(gm);
  auto kern = vec ? (sp ? scan_n1_bwd_kernel<true, true, STATE, DET> : scan_n1_bwd_kernel<true, false, STATE, DET>)
                  : (sp ? scan_n1_bwd_kernel<false, true, STATE, DET> : scan_n1_bwd_kernel<false, false, STATE, DET>);
  kern<<<grid, nt, smem, stream>>>(p, gm, dA, dD, dbias, grads_zeroed, st);
  return cudaGetLastError();
}

bool scan_n1_bwd_try(const ScanParams& p, const ScanState& st, float* dA, float* dD, float* dbias, int grads_zeroed,
                     cudaStream_t stream, cudaError_t* err, int* slabs) {
  if (!n1_eligible(p, true)) return false;
  const bool vec = n1_vec(p, true);
  N1Geom gr;
  size_t smem_rows = 0;
  if (vec && n1_rows_geometry(p, grads_zeroed, &gr, &smem_rows)) {
    *slabs = p.det ? (p.dpg + gr.rt * gr.rseq - 1) / (gr.rt * gr.rseq) : 0;
    if (has_state(st))
      *err = p.det ? n1_bwd_rows_launch<true, true>(p, st, gr, smem_rows, dA, dD, dbias, grads_zeroed, stream)
                   : n1_bwd_rows_launch<false, true>(p, st, gr, smem_rows, dA, dD, dbias, grads_zeroed, stream);
    else
      *err = p.det ? n1_bwd_rows_launch<true, false>(p, st, gr, smem_rows, dA, dD, dbias, grads_zeroed, stream)
                   : n1_bwd_rows_launch<false, false>(p, st, gr, smem_rows, dA, dD, dbias, grads_zeroed, stream);
    return true;
  }
  const N1Geom gm = n1_geometry(p);
  if (n1_one_row_smem(gm) > 40 * 1024) return false;
  *slabs = p.det ? (p.dpg + gm.rt - 1) / gm.rt : 0;
  if (has_state(st))
    *err = p.det ? n1_bwd_launch<true, true>(p, st, gm, vec, dA, dD, dbias, grads_zeroed, stream)
                 : n1_bwd_launch<false, true>(p, st, gm, vec, dA, dD, dbias, grads_zeroed, stream);
  else
    *err = p.det ? n1_bwd_launch<true, false>(p, st, gm, vec, dA, dD, dbias, grads_zeroed, stream)
                 : n1_bwd_launch<false, false>(p, st, gm, vec, dA, dD, dbias, grads_zeroed, stream);
  return true;
}

}  // namespace ss2d
