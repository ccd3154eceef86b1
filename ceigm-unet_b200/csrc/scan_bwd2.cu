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
template <bool SOFTPLUS, bool DET>
__global__ void __launch_bounds__(B2_NW * 32, 4) scan_bwd2_kernel(const ScanParams p, const __grid_constant__ Bwd2Maps maps) {
  constexpr bool STATE = false;
  const ScanState st{};
#include "scan_bwd2_body.inc"
}
template <bool SOFTPLUS, bool DET>
__global__ void __launch_bounds__(B2_NW * 32, 4) scan_bwd2_state_kernel(const ScanParams p, const __grid_constant__ Bwd2Maps maps, const ScanState st) {
  constexpr bool STATE = true;
#include "scan_bwd2_body.inc"
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
  const void* kern_sp = STATE ? reinterpret_cast<const void*>(scan_bwd2_state_kernel<true, DET>) : reinterpret_cast<const void*>(scan_bwd2_kernel<true, DET>);
  const void* kern_nosp = STATE ? reinterpret_cast<const void*>(scan_bwd2_state_kernel<false, DET>) : reinterpret_cast<const void*>(scan_bwd2_kernel<false, DET>);
  cudaError_t e = func_attr_once(once, kern_sp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2_SMEM);
  if (e == cudaSuccess) e = func_attr_once(once_nosp, kern_nosp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2_SMEM);
  if (e != cudaSuccess) return e;
  dim3 grid((p.dpg + B2_CH - 1) / B2_CH, p.G, p.batch);
  if constexpr (STATE) {
    if (p.softplus) scan_bwd2_state_kernel<true, DET><<<grid, B2_NW * 32, B2_SMEM, stream>>>(p, maps, st);
    else scan_bwd2_state_kernel<false, DET><<<grid, B2_NW * 32, B2_SMEM, stream>>>(p, maps, st);
  } else {
    if (p.softplus) scan_bwd2_kernel<true, DET><<<grid, B2_NW * 32, B2_SMEM, stream>>>(p, maps);
    else scan_bwd2_kernel<false, DET><<<grid, B2_NW * 32, B2_SMEM, stream>>>(p, maps);
  }
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
