// Selective-scan backward, fast path for the north-star regime (8 < d_state <= 16, fp32, TMA-stageable operands,
// contiguous traversal: SCAN layout or directions 1 / 3). Everything else runs scan_bwd.cu.
//
// Replaces selective_scan_bwd_kernel (/root/reference/gm-unet/kernels/selective_scan/csrc/selective_scan/cus/
// selective_scan_bwd_kernel.cuh:66-273). Same mathematics as scan_bwd.cu (two-level state recompute from the
// forward's chunk checkpoints, adjoint recurrence g_l = C_l dy_l + a_(l+1) g_(l+1)); different machine mapping:
//   * a warp owns 8 channel rows = 4 ROW PAIRS; lane = (row pair, state lane q): states q and q + 8 of two rows.
//     Everything a lane computes is packed f32x2 with one row per half — both recurrences included; B and C enter
//     as broadcast scalar operands, delta / delta*u / dout as ready-made register pairs.
//   * no producer warp, no polling: each warp streams its own delta / u / dout rows through a private 2-stage TMA
//     ring; the B/C tiles are shared by the CTA and refilled by the last warp that releases them.
//   * per tile the warp rewrites its tiles in place as activated, row-pair-interleaved arrays (scan order, so that
//     reversed traversals cost nothing afterwards); du / d(delta) are written over dout' / delta' and leave as
//     128-bit row-contiguous stores at the end of the tile.
//   * sum over states (du, d delta): shuffle reduce-scatter over the 8 state lanes; sum over rows (dB, dC): x+y of
//     the packed halves, reduce-scatter over the 4 row-pair lanes, then one red.global.add.v2.f32 per lane and state
//     straight from registers: each warp adds the totals of its 8 rows to dB / dC in L2. (A first version folded the
//     four warps' totals through shared-memory slabs with an mbarrier hand-off per group to issue a quarter of the
//     reductions; the hand-off coupled the warps and cost 10 % of the kernel, the extra L2 reductions cost nothing.)
//     Deterministic mode (DET) keeps the warps uncoupled: each warp stores its totals into its own partial slab (index =
//     the warp's position along the group), and scan_bwd_fold_kernel sums the slabs in slab order.
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "scan_params.h"
#include "host_util.h"
#include "common.cuh"
#include "tma_host.h"

namespace ss2d {

constexpr int B2_NW = 4;                    // warps per CTA
constexpr int B2_RPW = 8;                   // rows per warp
constexpr int B2_CH = B2_NW * B2_RPW;       // rows per CTA
constexpr int B2_STAGES = 2;
constexpr int B2_WSTAGE = 3 * 1024;         // delta | u | dout tiles of one warp (8 rows x 128 bytes each)
constexpr int B2_BC_STAGE = 4096;           // B | C tiles, 16 state rows each
constexpr int B2_HS_BYTES = 8 * 512;        // per warp: states at the 7 inner group boundaries of a tile + the tile's entry state
constexpr int B2_OFF_ROWS = B2_STAGES * B2_BC_STAGE;
constexpr int B2_OFF_UP = B2_OFF_ROWS + B2_NW * B2_STAGES * B2_WSTAGE;
constexpr int B2_OFF_HS = B2_OFF_UP + B2_NW * 1024;
constexpr int B2_OFF_BARS = B2_OFF_HS + B2_NW * B2_HS_BYTES;
constexpr size_t B2_SMEM = B2_OFF_BARS + 256 + 1024;

struct Bwd2Maps { TMap u, dl, dy, B, C; };

// Shared-memory accessors on 32-bit shared-window addresses: no generic-pointer arithmetic inside the loops.
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, float2 v) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void mbar_wait32(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive32(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect32(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_4d32(uint32_t dst, const void* tmap, int c0, int c1, int c2, int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void red_add2(float* dst, float a, float c) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(dst), "f"(a), "f"(c) : "memory");
}
__device__ __forceinline__ float2 sel2(bool c, float2 a, float2 b) { return make_float2(c ? a.x : b.x, c ? a.y : b.y); }
__device__ __forceinline__ float2 shfl2(float2 v, int m) {
  return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}
__device__ __forceinline__ int atom_add_acqrel32(uint32_t addr, int v) {
  int old;
  asm volatile("atom.acq_rel.cta.shared::cta.add.s32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(v) : "memory");
  return old;
}

// Row-pair-interleaved array of one warp: 4 row pairs x 32 positions x (row 0, row 1). The 16-byte chunk ch (two
// positions) of row pair rp lives in slot ch ^ rp ^ (ch >> 3) of the pair's 256-byte line: the 4 row pairs read at
// one position hit 4 different bank groups, and so do the 8 chunks {2 c + hh} one quarter-warp writes.
__device__ __forceinline__ int b2_p_off(int rp, int ch) { return rp * 256 + (((ch ^ rp ^ (ch >> 3)) & 15) << 4); }
// TMA SWIZZLE_128B tile of 32-float rows: byte offset of the 16-byte chunk c4 of row r
__device__ __forceinline__ int b2_t_off(int r, int c4) { return r * 128 + (((c4 ^ r) & 7) << 4); }

template <int STRIDE, int CNT, int S>
struct B2ReduceScatter {
  static __device__ __forceinline__ void run(float* v, int lane_id) {
    if constexpr (S >= 1 && CNT > 1) {
      constexpr int HALF = CNT / 2;
      const bool up = (lane_id & S) != 0;
#pragma unroll
      for (int i = 0; i < HALF; ++i) {
        const float send = up ? v[i] : v[i + HALF];
        const float keep = up ? v[i + HALF] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, S * STRIDE);
      }
      B2ReduceScatter<STRIDE, HALF, S / 2>::run(v, lane_id);
    }
  }
};

// STATE: the recompute of tile 0 starts from st.h0, the adjoint from st.dlast, and st.dh0 receives the adjoint of h0 (each
// pointer may be null)
template <bool SOFTPLUS, bool STATE, bool DET>
__global__ void __launch_bounds__(B2_NW * 32, 4) scan_bwd2_kernel(const ScanParams p, const __grid_constant__ Bwd2Maps maps, const ScanState st) {
  extern __shared__ __align__(16) unsigned char smem_rawb2[];
  unsigned char* smem = smem_rawb2 + ((1024 - (smem_u32(smem_rawb2) & 1023)) & 1023);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t sm = smem_u32(smem);
  const uint32_t a_bc = sm;                                                  // [STAGES][B | C]
  const uint32_t a_rows = sm + B2_OFF_ROWS + warp * (B2_STAGES * B2_WSTAGE);  // [STAGES][delta | u | dout]
  const uint32_t a_up = sm + B2_OFF_UP + warp * 1024;                        // u pairs of the current tile
  const uint32_t a_hs = sm + B2_OFF_HS + warp * B2_HS_BYTES + lane * 16;     // this lane's group-boundary states
  const uint32_t a_bars = sm + B2_OFF_BARS;
  const uint32_t a_full_w = a_bars + warp * (B2_STAGES * 8);                 // [NW][STAGES]
  const uint32_t a_full_bc = a_bars + B2_NW * B2_STAGES * 8;                 // [STAGES]
  const uint32_t a_cnt_bc = a_full_bc + B2_STAGES * 8;                      // [STAGES] ints
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + B2_OFF_BARS);

  const int b = blockIdx.z, g = blockIdx.y;
  const int row0 = blockIdx.x * B2_CH + warp * B2_RPW;             // first row of this warp inside the group
  const int rows_valid = p.dpg - row0;                              // <= 0: idle warp (still takes part in the hand-offs)
  const int d0 = g * p.dpg + row0;
  const int L = p.L;
  const int dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
  const bool rev = dir == 3;
  const int ntiles = (L + 31) / 32;
  const int ug = p.u_mod > 0 ? g % (p.u_mod / p.dpg) : g;          // group coordinate of u and dout

  if (threadIdx.x == 0) {
    for (int i = 0; i < B2_NW * B2_STAGES + B2_STAGES; ++i) mbar_init(&bars[i], 1);          // full_w, full_bc
    for (int s = 0; s < B2_STAGES; ++s) reinterpret_cast<int*>(bars + B2_NW * B2_STAGES + B2_STAGES)[s] = 0;
    fence_mbar_init();
  }
  __syncthreads();

  // tiles are visited last to first: iteration `it` handles tile t = ntiles - 1 - it
  auto issue_rows = [&](int it) {     // lane 0 of the warp
    const int s = it % B2_STAGES, t = ntiles - 1 - it;
    const int m0 = rev ? L - t * 32 - 32 : t * 32;
    const uint32_t st = a_rows + s * B2_WSTAGE, bar = a_full_w + s * 8;
    mbar_expect32(bar, B2_WSTAGE);
    tma_load_4d32(st, &maps.dl, m0, row0, g, b, bar);
    tma_load_4d32(st + 1024, &maps.u, m0, row0, ug, b, bar);
    tma_load_4d32(st + 2048, &maps.dy, m0, row0, ug, b, bar);
  };
  auto issue_bc = [&](int it) {
    const int s = it % B2_STAGES, t = ntiles - 1 - it;
    const int m0 = rev ? L - t * 32 - 32 : t * 32;
    const uint32_t bar = a_full_bc + s * 8;
    mbar_expect32(bar, B2_BC_STAGE);
    tma_load_4d32(a_bc + s * B2_BC_STAGE, &maps.B, m0, 0, g, b, bar);
    tma_load_4d32(a_bc + s * B2_BC_STAGE + 2048, &maps.C, m0, 0, g, b, bar);
  };
  if (lane == 0) {
    if (warp == 0) { tma_prefetch_desc(&maps.B); tma_prefetch_desc(&maps.C); }
    tma_prefetch_desc(&maps.dl); tma_prefetch_desc(&maps.u); tma_prefetch_desc(&maps.dy);
    for (int it = 0; it < B2_STAGES && it < ntiles; ++it) {
      if (warp == 0) issue_bc(it);
      issue_rows(it);
    }
  }

  const int q = lane & 7, rp = lane >> 3;
  const int sw = rp >> 1;              // the upper two row pairs hold their two states in swapped order (see the dB / dC sum)
  const bool v0 = 2 * rp < rows_valid, v1 = 2 * rp + 1 < rows_valid;
  // main role: row pair rp, states n_j = q + 8 (j ^ sw)
  float2 A2p[2], carry2[2], dA2[2];      // A2 = A log2(e)
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int n = q + 8 * (j ^ sw);
    const bool okn = n < p.N;
    A2p[j].x = (okn && v0) ? p.A[(int64_t)(d0 + 2 * rp) * p.A_ld + n] * kLog2e : 0.f;
    A2p[j].y = (okn && v1) ? p.A[(int64_t)(d0 + 2 * rp + 1) * p.A_ld + n] * kLog2e : 0.f;
    carry2[j] = make_float2(0.f, 0.f);      // a_(l+1) g_(l+1), zero (STATE: dlast) past the end of the sequence
    if (STATE && st.dlast && okn) {
      if (v0) carry2[j].x = st.dlast[state_slot(p, b, d0 + 2 * rp, n)];
      if (v1) carry2[j].y = st.dlast[state_slot(p, b, d0 + 2 * rp + 1, n)];
    }
    dA2[j] = make_float2(0.f, 0.f);
  }
  // finalising role: row fr = 2 rp + (q >> 2), position fe = q & 3 of every group
  const int rr = q >> 2, fe = q & 3;
  const bool fvalid = 2 * rp + rr < rows_valid;
  const float Dr = (p.Dv && fvalid) ? p.Dv[d0 + 2 * rp + rr] : 0.f;
  float dDacc = 0.f, dbacc = 0.f;
  // activation role: row pair rp, position quad q
  float2 biasp;
  biasp.x = (p.bias && v0) ? p.bias[d0 + 2 * rp] : 0.f;
  biasp.y = (p.bias && v1) ? p.bias[d0 + 2 * rp + 1] : 0.f;
  // shared-memory offsets as (lane constant) ^ (uniform term): one LOP3 per access inside the loops
  const int rowc = (rp * 256) | (rp << 4);                                   // b2_p_off(rp, ch) = rowc ^ (su(ch) << 4)
  const int qc0 = ((q * 128) | (q << 4)) + 1024 * sw, qc1 = qc0 ^ 1024;     // b2_t_off(n_j, c4) = qcj ^ (c4 << 4)
  // The finisher's scalar slot, kept in an opaque register: at the 128-register cap ptxas otherwise re-derives it from
  // %tid in every group.
  uint32_t pk;
  {
    const uint32_t v = (rowc ^ ((fe >> 1) << 4)) | (((fe & 1) * 2 + rr) * 4);
    asm volatile("mov.b32 %0, %1;" : "=r"(pk) : "r"(v));
  }
  // dB / dC destination of this lane after the sum over the row-pair lanes: state n_0 = q + 8 sw, both tensors,
  // positions 2 (rp & 1), + 1 of every group. Lanes of padded states (n_0 >= N: B = C = 0 there, zero-filled by TMA, so
  // their totals are exactly 0) add their zeros to the last real state instead of being predicated off.
  // DET: slab wslab instead, and the padded-state lanes store nothing (a store of their zeros would overwrite state N - 1)
  const int wslab = blockIdx.x * B2_NW + warp;
  float* const red_B = (DET ? det_slab(p, 0, wslab) : p.dB) + ((int64_t)(b * p.G + g) * p.A_ld + min(q + 8 * sw, p.N - 1)) * L;
  const int64_t red_CmB = DET ? det_slab(p, 1, wslab) - det_slab(p, 0, wslab) : p.dC - p.dB;
  const bool red_lane = !DET || q + 8 * sw < p.N;

  auto load_ckpt = [&](int t, float2* h) {     // state before tile t = checkpoint at the end of tile t - 1
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int n = q + 8 * (j ^ sw);
      const bool ok = t > 0 && n < p.N;
      h[j].x = (ok && v0) ? __ldg(p.ckpt_in + (((int64_t)b * p.dim + d0 + 2 * rp) * p.nck + (t - 1)) * p.N + n) : 0.f;
      h[j].y = (ok && v1) ? __ldg(p.ckpt_in + (((int64_t)b * p.dim + d0 + 2 * rp + 1) * p.nck + (t - 1)) * p.N + n) : 0.f;
      if (STATE && t == 0 && st.h0 && n < p.N) {
        if (v0) h[j].x = __ldg(st.h0 + state_slot(p, b, d0 + 2 * rp, n));
        if (v1) h[j].y = __ldg(st.h0 + state_slot(p, b, d0 + 2 * rp + 1, n));
      }
    }
  };

  auto body = [&](auto REV) {
    constexpr bool REVV = decltype(REV)::value;
    for (int it = 0; it < ntiles; ++it) {
      const int t = ntiles - 1 - it;
      const int s = it % B2_STAGES;
      const uint32_t par = (it / B2_STAGES) & 1;
      const int l0 = t * 32, len = min(32, L - l0);
      const uint32_t a_dl = a_rows + s * B2_WSTAGE;       // delta  -> delta' pairs -> d(delta)
      const uint32_t a_du = a_dl + 1024;                  // u      -> (delta' u) pairs
      const uint32_t a_dy = a_dl + 2048;                  // dout   -> dout' pairs  -> du
      float2 h0[2];
      load_ckpt(t, h0);                                   // in flight during the activation pass
      mbar_wait32(a_full_w + s * 8, par);
      // ---- activation + row-pair interleave, in place: this lane handles position quad q of row pair rp ----
      {
        const int tc4 = REVV ? 7 - q : q;
        float4 dv[2], uv[2], yv[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const uint32_t o = b2_t_off(2 * rp + r, tc4);
          dv[r] = lds128(a_dl + o);
          uv[r] = lds128(a_du + o);
          yv[r] = lds128(a_dy + o);
          if (REVV) {
            dv[r] = make_float4(dv[r].w, dv[r].z, dv[r].y, dv[r].x);
            uv[r] = make_float4(uv[r].w, uv[r].z, uv[r].y, uv[r].x);
            yv[r] = make_float4(yv[r].w, yv[r].z, yv[r].y, yv[r].x);
          }
        }
        __syncwarp();
        float dl[2][4], du[2][4];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float x = f4_at(dv[r], e) + (r == 0 ? biasp.x : biasp.y);
            if (SOFTPLUS) x = softplus20(x);
            const bool live = q * 4 + e < len && (r == 0 ? v0 : v1);
            dl[r][e] = live ? x : 0.f;
            du[r][e] = live ? x * f4_at(uv[r], e) : 0.f;
          }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {              // chunk 2 q + hh: positions 4 q + 2 hh, + 1
          const uint32_t off = b2_p_off(rp, 2 * q + hh);
          sts128(a_dl + off, make_float4(dl[0][2 * hh], dl[1][2 * hh], dl[0][2 * hh + 1], dl[1][2 * hh + 1]));
          sts128(a_du + off, make_float4(du[0][2 * hh], du[1][2 * hh], du[0][2 * hh + 1], du[1][2 * hh + 1]));
          sts128(a_dy + off, make_float4(f4_at(yv[0], 2 * hh), f4_at(yv[1], 2 * hh), f4_at(yv[0], 2 * hh + 1), f4_at(yv[1], 2 * hh + 1)));
          sts128(a_up + off, make_float4(f4_at(uv[0], 2 * hh), f4_at(uv[1], 2 * hh), f4_at(uv[0], 2 * hh + 1), f4_at(uv[1], 2 * hh + 1)));
        }
        __syncwarp();
      }
      mbar_wait32(a_full_bc + s * 8, par);
      const uint32_t a_B = a_bc + s * B2_BC_STAGE;

      // ---- (1) forward recompute of h over the tile from the chunk checkpoint; the state after each of the first
      //          7 groups is parked in shared memory. Fully unrolled, with the loads of group gi + 1 requested before the
      //          arithmetic of group gi (the shared-memory accessors are volatile: ptxas keeps their order).
      {
        float2 h[2] = {h0[0], h0[1]};
        sts128(a_hs + 7 * 512, make_float4(h0[0].x, h0[0].y, h0[1].x, h0[1].y));     // read back by the last group (gi = 0)
        struct FwdIn { float4 d01, d23, u01, u23, B0, B1; };
        auto fwd_load = [&](const int gi) {
          FwdIn r;
          const uint32_t pa = a_dl + (rowc ^ (((2 * gi ^ (gi >> 2)) & 15) << 4));
          const int gsh = (REVV ? 7 - gi : gi) << 4;
          r.d01 = lds128(pa); r.d23 = lds128(pa ^ 16);
          r.u01 = lds128(pa + 1024); r.u23 = lds128((pa ^ 16) + 1024);
          r.B0 = lds128(a_B + (qc0 ^ gsh)); r.B1 = lds128(a_B + (qc1 ^ gsh));
          return r;
        };
        FwdIn cur = fwd_load(0);
#pragma unroll
        for (int gi = 0; gi < 7; ++gi) {
          FwdIn nxt = cur;
          if (gi < 6) nxt = fwd_load(gi + 1);
          const float2 dl2[4] = {make_float2(cur.d01.x, cur.d01.y), make_float2(cur.d01.z, cur.d01.w), make_float2(cur.d23.x, cur.d23.y), make_float2(cur.d23.z, cur.d23.w)};
          const float2 du2[4] = {make_float2(cur.u01.x, cur.u01.y), make_float2(cur.u01.z, cur.u01.w), make_float2(cur.u23.x, cur.u23.y), make_float2(cur.u23.z, cur.u23.w)};
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float4 Bq = j == 0 ? cur.B0 : cur.B1;
            if (REVV) Bq = make_float4(Bq.w, Bq.z, Bq.y, Bq.x);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float be = f4_at(Bq, e);
              const float2 arg = __fmul2_rn(dl2[e], A2p[j]);
              const float2 a = make_float2(ex2f(arg.x), ex2f(arg.y));
              h[j] = __ffma2_rn(a, h[j], __fmul2_rn(du2[e], make_float2(be, be)));
            }
          }
          sts128(a_hs + gi * 512, make_float4(h[0].x, h[0].y, h[1].x, h[1].y));
          cur = nxt;
        }
      }

      // ---- (2) groups of 4 positions, last to first: re-expand a and h, run the adjoint recurrence ----
      // unrolled by 4: the swizzle / parity terms of a group become constants and the tail of one group overlaps the
      // head of the next
      float* red_t = red_B + (REVV ? L - 2 - (l0 + 2 * (rp & 1)) : l0 + 2 * (rp & 1));
      asm volatile("mov.b64 %0, %0;" : "+l"(red_t));       // kept as one 64-bit register pair; the groups add immediates
#pragma unroll 4
      for (int gi = 7; gi >= 0; --gi) {
        const int su4 = ((2 * gi ^ (gi >> 2)) & 15) << 4;
        const uint32_t pa = a_dl + (rowc ^ su4);
        const int gsh = (REVV ? 7 - gi : gi) << 4;
        const float4 d01 = lds128(pa), d23 = lds128(pa ^ 16);
        const float4 u01 = lds128(pa + 1024), u23 = lds128((pa ^ 16) + 1024);
        const float4 y01 = lds128(pa + 2048), y23 = lds128((pa ^ 16) + 2048);
        const float4 hin4 = lds128(a_hs + ((gi + 7) & 7) * 512);   // state before the group; slot 7 holds the tile's entry state
        const float4 Bq1 = lds128(a_B + (qc1 ^ gsh)), Cq1 = lds128(a_B + 2048 + (qc1 ^ gsh));
        // the finisher's scalars (row 2 rp + rr, position fe of this group), requested long before their use
        const uint32_t foff = pk ^ su4;
        const float de = lds32(a_dl + foff), dyv = lds32(a_dy + foff), uu = lds32(a_up + foff);
        const float2 dl2[4] = {make_float2(d01.x, d01.y), make_float2(d01.z, d01.w), make_float2(d23.x, d23.y), make_float2(d23.z, d23.w)};
        const float2 du2[4] = {make_float2(u01.x, u01.y), make_float2(u01.z, u01.w), make_float2(u23.x, u23.y), make_float2(u23.z, u23.w)};
        const float2 dy2[4] = {make_float2(y01.x, y01.y), make_float2(y01.z, y01.w), make_float2(y23.x, y23.y), make_float2(y23.z, y23.w)};
        float2 sB2[4], sA2[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) { sB2[e] = make_float2(0.f, 0.f); sA2[e] = make_float2(0.f, 0.f); }
        // one state of the lane: part = [dB (e0, e1) | dB (e2, e3) | dC (e0, e1) | dC (e2, e3)], the two rows of the pair added
        auto state_pass = [&](const int j, float4 Bq, float4 Cq, float2* part) {
          if (REVV) { Bq = make_float4(Bq.w, Bq.z, Bq.y, Bq.x); Cq = make_float4(Cq.w, Cq.z, Cq.y, Cq.x); }
          const float2 hprev = j == 0 ? make_float2(hin4.x, hin4.y) : make_float2(hin4.z, hin4.w);
          float2 a2[4], hh2[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float be = f4_at(Bq, e);
            const float2 arg = __fmul2_rn(dl2[e], A2p[j]);
            a2[e] = make_float2(ex2f(arg.x), ex2f(arg.y));
            hh2[e] = __ffma2_rn(a2[e], e == 0 ? hprev : hh2[e - 1], __fmul2_rn(du2[e], make_float2(be, be)));
          }
          float2 carry = carry2[j];
          float sb[4], sc[4];
#pragma unroll
          for (int e = 3; e >= 0; --e) {
            const float be = f4_at(Bq, e), ce = f4_at(Cq, e);
            const float2 g2 = __ffma2_rn(dy2[e], make_float2(ce, ce), carry);     // g_e = C_e dy_e + a_(e+1) g_(e+1)
            const float2 t2 = __fmul2_rn(g2, a2[e]);                              // a_e g_e
            carry = t2;
            const float2 pb = __fmul2_rn(g2, du2[e]);
            const float2 pc = __fmul2_rn(dy2[e], hh2[e]);
            sb[e] = pb.x + pb.y;
            sc[e] = pc.x + pc.y;
            sB2[e] = __ffma2_rn(g2, make_float2(be, be), sB2[e]);
            const float2 w2 = __fmul2_rn(t2, e == 0 ? hprev : hh2[e - 1]);        // g_e (h_e - delta u B_e)
            sA2[e] = __ffma2_rn(w2, A2p[j], sA2[e]);                           // scaled by log2(e): undone below
            dA2[j] = __ffma2_rn(w2, dl2[e], dA2[j]);
          }
          carry2[j] = carry;
          part[0] = make_float2(sb[0], sb[1]); part[1] = make_float2(sb[2], sb[3]);
          part[2] = make_float2(sc[0], sc[1]); part[3] = make_float2(sc[2], sc[3]);
        };
        // ---- sum over the 4 row-pair lanes (dB, dC). The lanes of row pairs 2, 3 hold their states in swapped order, so the
        //      first exchange (lane ^ 16) needs no selects: every lane sends its local state 1 and keeps its local state 0 —
        //      the same global state n_0 = q + 8 sw on both sides. The second (lane ^ 8) splits the positions. ----
        float2 p0[4], p1[4], r1[4];
        state_pass(1, Bq1, Cq1, p1);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          r1[i] = make_float2(__shfl_xor_sync(0xffffffffu, p1[i].x, 16), __shfl_xor_sync(0xffffffffu, p1[i].y, 16));
        {
          const float4 Bq0 = lds128(a_B + (qc0 ^ gsh)), Cq0 = lds128(a_B + 2048 + (qc0 ^ gsh));
          state_pass(0, Bq0, Cq0, p0);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) p0[i] = __fadd2_rn(p0[i], r1[i]);
        float2 oB, oC;                  // positions 2 (rp & 1), + 1 of the group, state n_0, summed over the warp's 8 rows
        {
          const bool up = (rp & 1) != 0;
          oB = __fadd2_rn(sel2(up, p0[1], p0[0]), shfl2(sel2(up, p0[0], p0[1]), 8));
          oC = __fadd2_rn(sel2(up, p0[3], p0[2]), shfl2(sel2(up, p0[2], p0[3]), 8));
        }
        // this warp's totals go straight to global memory: two red.global.add.v2.f32 per lane (the branch is warp-uniform:
        // idle warps, and the groups past the end of the sequence in its last tile)
        if (rows_valid > 0 && 4 * gi < len && red_lane) {
          float* const dst = red_t + (REVV ? -4 * gi : 4 * gi);
          if constexpr (DET) {
            *reinterpret_cast<float2*>(dst) = make_float2(REVV ? oB.y : oB.x, REVV ? oB.x : oB.y);
            *reinterpret_cast<float2*>(dst + red_CmB) = make_float2(REVV ? oC.y : oC.x, REVV ? oC.x : oC.y);
          } else {
            red_add2(dst, REVV ? oB.y : oB.x, REVV ? oB.x : oB.y);
            red_add2(dst + red_CmB, REVV ? oC.y : oC.x, REVV ? oC.x : oC.y);
          }
        }
        // ---- sum over the 8 state lanes on row-packed pairs: positions first (lane bits 0, 1), the row parity last; lane q ends
        //      up with (sB, sA) of row parity q >> 2, position q & 3 ----
        float sBe, sAe;
        {
          const bool b0 = (q & 1) != 0, b1 = (q & 2) != 0, b2 = (q & 4) != 0;
          float2 RB[2], RA[2];
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            RB[k] = __fadd2_rn(sel2(b0, sB2[2 * k + 1], sB2[2 * k]), shfl2(sel2(b0, sB2[2 * k], sB2[2 * k + 1]), 1));
            RA[k] = __fadd2_rn(sel2(b0, sA2[2 * k + 1], sA2[2 * k]), shfl2(sel2(b0, sA2[2 * k], sA2[2 * k + 1]), 1));
          }
          const float2 SB = __fadd2_rn(sel2(b1, RB[1], RB[0]), shfl2(sel2(b1, RB[0], RB[1]), 2));
          const float2 SA = __fadd2_rn(sel2(b1, RA[1], RA[0]), shfl2(sel2(b1, RA[0], RA[1]), 2));
          sBe = (b2 ? SB.y : SB.x) + __shfl_xor_sync(0xffffffffu, b2 ? SB.x : SB.y, 4);
          sAe = ((b2 ? SA.y : SA.x) + __shfl_xor_sync(0xffffffffu, b2 ? SA.x : SA.y, 4)) * kLn2;
        }
        {
          const float du_out = fmaf(Dr, dyv, de * sBe);
          float ddl = fmaf(uu, sBe, sAe);
          if (SOFTPLUS) {   // sigmoid(raw) = 1 - exp(-softplus(raw)); series for small delta avoids cancellation
            const float sig = de < 0.015625f ? de * (1.f - de * (0.5f - de * 0.16666667f)) : 1.f - ex2f(-de * kLog2e);
            ddl *= sig;
          }
          if (gi * 4 + fe >= len || !fvalid) ddl = 0.f;
          dDacc = fmaf(dyv, uu, dDacc);
          dbacc += ddl;
          // every lane of the row pair has consumed this group's delta' / dout' (the shuffles above ordered them)
          sts32(a_dy + foff, du_out);
          sts32(a_dl + foff, ddl);
        }
      }
      __syncwarp();
      // ---- tile epilogue: du / d(delta) of this warp's rows, 128-bit row-contiguous stores ----
      {
        const uint32_t off0 = b2_p_off(rp, 2 * q), off1 = b2_p_off(rp, 2 * q + 1);
        const float4 ua = lds128(a_dy + off0), ub = lds128(a_dy + off1);
        const float4 da = lds128(a_dl + off0), db = lds128(a_dl + off1);
        const int l = l0 + 4 * q;
        if (l < L) {
          const int64_t mpos = REVV ? L - 4 - l : l;
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            if (r == 0 ? v0 : v1) {
              const int d = d0 + 2 * rp + r;
              float4 uo = r == 0 ? make_float4(ua.x, ua.z, ub.x, ub.z) : make_float4(ua.y, ua.w, ub.y, ub.w);
              float4 dd = r == 0 ? make_float4(da.x, da.z, db.x, db.z) : make_float4(da.y, da.w, db.y, db.w);
              if (REVV) { uo = make_float4(uo.w, uo.z, uo.y, uo.x); dd = make_float4(dd.w, dd.z, dd.y, dd.x); }
              // du has u's strides, except when the groups share u (u_mod > 0): then it is a dense (batch, dim, L) tensor
              const int64_t duo = p.u_mod > 0 ? ((int64_t)b * p.dim + d) * (int64_t)L : (int64_t)b * p.u_bs + (int64_t)d * p.u_ds;
              *reinterpret_cast<float4*>(static_cast<float*>(p.du) + duo + mpos) = uo;
              *reinterpret_cast<float4*>(static_cast<float*>(p.ddelta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds + mpos) = dd;
            }
          }
        }
      }
      // release the stage: generic-proxy accesses are ordered before the async-proxy refill
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        if (it + B2_STAGES < ntiles) issue_rows(it + B2_STAGES);
        if (atom_add_acqrel32(a_cnt_bc + s * 4, 1) == B2_NW - 1) {      // last warp to release the B/C stage refills it
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(a_cnt_bc + s * 4), "r"(0) : "memory");
          if (it + B2_STAGES < ntiles) issue_bc(it + B2_STAGES);
        }
      }
      __syncwarp();
    }
  };
  if (rev) body(std::true_type{}); else body(std::false_type{});

  if (STATE && st.dh0) {      // the carry is now a_0 g_0 = dloss / dh0
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int n = q + 8 * (j ^ sw);
      if (n < p.N) {
        if (v0) st.dh0[state_slot(p, b, d0 + 2 * rp, n)] = carry2[j].x;
        if (v1) st.dh0[state_slot(p, b, d0 + 2 * rp + 1, n)] = carry2[j].y;
      }
    }
  }

  // ---- per-(batch, channel) partials of dA, dD, d(delta_bias) ----
  {
    float dd = dDacc, db = dbacc;
    dd += __shfl_xor_sync(0xffffffffu, dd, 1); db += __shfl_xor_sync(0xffffffffu, db, 1);
    dd += __shfl_xor_sync(0xffffffffu, dd, 2); db += __shfl_xor_sync(0xffffffffu, db, 2);
    if (fvalid && fe == 0) {
      float* dst = p.part + ((int64_t)b * p.dim + d0 + 2 * rp + rr) * (p.N + 2);
      dst[p.N] = dd; dst[p.N + 1] = db;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int n = q + 8 * (j ^ sw);
      if (n < p.N) {
        if (v0) p.part[((int64_t)b * p.dim + d0 + 2 * rp) * (p.N + 2) + n] = dA2[j].x;
        if (v1) p.part[((int64_t)b * p.dim + d0 + 2 * rp + 1) * (p.N + 2) + n] = dA2[j].y;
      }
    }
  }
}

static bool bwd2_maps(const ScanParams& p, Bwd2Maps* m) {
  const long long ugroups = p.u_mod > 0 ? p.u_mod / p.dpg : p.G;
  const long long du[4] = {p.L, p.dpg, ugroups, p.batch}, su[4] = {1, p.u_ds, (long long)p.dpg * p.u_ds, p.u_bs};
  const long long sy[4] = {1, p.out_ds, (long long)p.dpg * p.out_ds, p.out_bs};
  const long long dd[4] = {p.L, p.dpg, p.G, p.batch}, sd[4] = {1, p.dl_ds, (long long)p.dpg * p.dl_ds, p.dl_bs};
  const long long d4[4] = {p.L, p.N, p.G, p.batch};
  const long long s4B[4] = {1, p.B_ns, p.B_gs, p.B_bs}, s4C[4] = {1, p.C_ns, p.C_gs, p.C_bs};
  return make_tmap(&m->u, p.u, 4, du, su, B2_RPW) && make_tmap(&m->dl, p.delta, 4, dd, sd, B2_RPW) &&
         make_tmap(&m->dy, p.dout, 4, du, sy, B2_RPW) && make_tmap(&m->B, p.Bm, 4, d4, s4B, 16) &&
         make_tmap(&m->C, p.Cm, 4, d4, s4C, 16);
}

// the conditions of the fast path that the descriptor alone decides (the rest are pointer alignments)
static bool bwd2_shape_ok(const ScanParams& p) {
  if (p.N <= 8 || p.N > 16 || p.accum || p.io_dtype != SS2D_F32 || p.out_dtype != SS2D_F32) return false;
  if (p.u_mod > 0 && p.u_mod % p.dpg != 0) return false;
  for (int g = 0; g < p.G; ++g) {
    const int dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
    if (dir == 2 || dir == 4) return false;
  }
  return true;
}

// deterministic mode: one slab per warp that owns rows (warp index along the group)
int scan_bwd2_det_slabs(const ScanParams& p) { return bwd2_shape_ok(p) ? (p.dpg + B2_RPW - 1) / B2_RPW : 0; }

template <bool DET, bool STATE>
static cudaError_t bwd2_launch(const ScanParams& p, const Bwd2Maps& maps, const ScanState& st, cudaStream_t stream) {
  static PerDeviceOnce once, once_nosp;
  const auto kern_sp = scan_bwd2_kernel<true, STATE, DET>, kern_nosp = scan_bwd2_kernel<false, STATE, DET>;
  cudaError_t e = func_attr_once(once, reinterpret_cast<const void*>(kern_sp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2_SMEM);
  if (e == cudaSuccess)
    e = func_attr_once(once_nosp, reinterpret_cast<const void*>(kern_nosp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2_SMEM);
  if (e != cudaSuccess) return e;
  dim3 grid((p.dpg + B2_CH - 1) / B2_CH, p.G, p.batch);
  (p.softplus ? kern_sp : kern_nosp)<<<grid, B2_NW * 32, B2_SMEM, stream>>>(p, maps, st);
  return cudaGetLastError();
}

// Returns true when the fast path took the call (*err holds the launch status).
bool scan_bwd2_try(const ScanParams& p, const ScanState& st, cudaStream_t stream, cudaError_t* err, int* slabs) {
  if (!p.tma_ok || !bwd2_shape_ok(p)) return false;
  if ((reinterpret_cast<uintptr_t>(p.du) & 15) || (reinterpret_cast<uintptr_t>(p.ddelta) & 15) ||
      (reinterpret_cast<uintptr_t>(p.dB) & 15) || (reinterpret_cast<uintptr_t>(p.dC) & 15))
    return false;
  Bwd2Maps maps;
  if (!bwd2_maps(p, &maps)) return false;
  *slabs = p.det ? scan_bwd2_det_slabs(p) : 0;
  if (has_state(st)) *err = p.det ? bwd2_launch<true, true>(p, maps, st, stream) : bwd2_launch<false, true>(p, maps, st, stream);
  else *err = p.det ? bwd2_launch<true, false>(p, maps, st, stream) : bwd2_launch<false, false>(p, maps, st, stream);
  return true;
}

}  // namespace ss2d
