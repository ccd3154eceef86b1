// Selective-scan forward for sm_100a.
//
// Replaces selective_scan_fwd_kernel (/root/reference/gm-unet/kernels/selective_scan/csrc/selective_scan/cus/
// selective_scan_fwd_kernel.cuh:61-172) together with CrossScan*/CrossMerge* (model/gm/csms6s.py:11-206) when the
// NATURAL layout is used. Not a port: the reference runs one CTA per (batch, channel) row and a CUB block scan
// per state; here a CTA owns CH channel rows of one (batch, group), every thread owns NS states of one row
// and walks L sequentially (minimum-op recurrence: 1 ex2 + 4 flops per state and element), the R lanes of a
// row combine their partial y with warp shuffles, and B/C tiles are staged once per CTA and broadcast from
// shared memory to all rows. At d_state = 16 the kernel is bound by MUFU.EX2 (16/clk/SM), not by HBM —
// see DESIGN.md.
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "scan_params.h"
#include "host_util.h"
#include "scan_tile.cuh"
#include "tma_host.h"

namespace ss2d {

constexpr int kConsumerWarps = 4;
constexpr int kFwdThreads = 32 * (kConsumerWarps + 1);     // + 1 producer warp
constexpr int LT = kTileL;                                  // scan positions per tile (= SS2D_CHUNK)
static_assert(LT == SS2D_CHUNK, "one checkpoint per tile");

template <int NS, int R, int RPT, int STAGES>
struct FwdShape {
  static constexpr int RL = 32 / R;          // rows per warp per RPT slot
  static constexpr int RPW = RL * RPT;       // rows per warp
  static constexpr int CH = kConsumerWarps * RPW;   // rows per CTA
  static constexpr int NP = NS * R;          // padded states
  static constexpr int NPB = (NP + 7) / 8 * 8;      // B/C tile rows (tiles are multiples of 1024 bytes)
  static constexpr int stage_floats = (2 * CH + 2 * NPB) * LT;     // delta, u, B, C tiles of one pipeline stage
  static constexpr size_t smem_bytes = (size_t)(STAGES * stage_floats + CH * LT + 2 * CH) * 4 + 16 * STAGES + 1024;
};

// Warp-specialised tile pipeline, no CTA-wide barrier inside the loop:
//   warp 4 (producer) fills stage t % STAGES with the delta / u / B / C tiles of scan positions [t LT, (t+1) LT):
//     - fp32 operands whose rows are contiguous along the scan (SCAN layout or direction 1) and 16-byte aligned:
//       four tiled TMA loads through tensor maps (cp.async.bulk.tensor -> UTMALDG, 128-byte swizzle, out-of-bounds
//       rows / tails zero-filled by the hardware), completing on the stage's `full` mbarrier;
//     - anything else (16-bit dtypes, transposed / reversed traversal, unaligned views): index-mapped stage_rows()
//       writing the same swizzled layout.
//   warps 0-3 (consumers) own RPW channel rows each: wait `full`, activate delta for their own rows, run the
//   recurrence over the tile, then release the stage through its `empty` mbarrier. B/C are read-only and shared.
// STATE: the rows start from st.h0 instead of 0
template <int NS, int R, int RPT, int STAGES, bool STATE>
__global__ void __launch_bounds__(kFwdThreads) scan_fwd_kernel(const ScanParams p, const __grid_constant__ TmaMaps maps,
                                                                const ScanState st) {
  using S = FwdShape<NS, R, RPT, STAGES>;
  constexpr int CH = S::CH, NP = S::NP, NPB = S::NPB, RL = S::RL, RPW = S::RPW;
  extern __shared__ __align__(16) float smem_raw[];
  // tiles must be 1024-byte aligned in the shared window for the 128-byte swizzle pattern
  float* smem = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023) / 4;
  float* s_du = smem + STAGES * S::stage_floats;   // delta * u (consumer-written), swizzled   [CH][LT]
  float* s_bias = s_du + CH * LT;                  // [CH]
  float* s_D = s_bias + CH;                        // [CH]
  uint64_t* full = reinterpret_cast<uint64_t*>(s_D + CH);   // [STAGES]
  uint64_t* empty = full + STAGES;                          // [STAGES]
  auto st_dl = [&](int s) { return smem + s * S::stage_floats; };              // delta (raw, then activated) [CH][LT]
  auto st_u = [&](int s) { return smem + s * S::stage_floats + CH * LT; };     // u                            [CH][LT]
  auto st_B = [&](int s) { return smem + s * S::stage_floats + 2 * CH * LT; };             // [NPB][LT]
  auto st_C = [&](int s) { return smem + s * S::stage_floats + (2 * CH + NPB) * LT; };     // [NPB][LT]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.z, g = blockIdx.y;
  const int row0 = blockIdx.x * CH;                        // first channel of this CTA inside the group
  const int rows_valid = min(CH, p.dpg - row0);
  const int d0 = g * p.dpg + row0;                         // global channel of row 0
  const int L = p.L;
  ScanOrder so;
  so.dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
  so.H = p.H; so.W = p.W; so.L = L;
  const bool tma = p.tma_ok && so.contiguous();          // SCAN layout, directions 1 and 3
  const bool rev = tma && so.reversed();                 // TMA-staged tiles of a reversed traversal are mirrored
  const int ntiles = (L + LT - 1) / LT;

  for (int r = tid; r < CH; r += kFwdThreads) {
    const bool ok = r < rows_valid;
    s_bias[r] = (ok && p.bias) ? p.bias[d0 + r] : 0.f;
    s_D[r] = (ok && p.Dv && !p.accum) ? p.Dv[d0 + r] : 0.f;
  }
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumerWarps); }
    fence_mbar_init();
  }
  __syncthreads();

  const int64_t u_boff = (int64_t)b * p.u_bs, dl_boff = (int64_t)b * p.dl_bs, out_boff = (int64_t)b * p.out_bs;
  auto u_off = [&](int r) { const int d = d0 + r; return u_boff + (int64_t)(p.u_mod > 0 ? d % p.u_mod : d) * p.u_ds; };
  auto dl_off = [&](int r) { return dl_boff + (int64_t)(d0 + r) * p.dl_ds; };
  const int64_t B_base = (int64_t)b * p.B_bs + (int64_t)g * p.B_gs;
  const int64_t C_base = (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;
  auto B_off = [&](int n) { return B_base + (int64_t)n * p.B_ns; };
  auto C_off = [&](int n) { return C_base + (int64_t)n * p.C_ns; };

  if (warp == kConsumerWarps) {
    // =============================== producer warp ===============================
    if (tma && lane == 0) {
      tma_prefetch_desc(&maps.u); tma_prefetch_desc(&maps.dl); tma_prefetch_desc(&maps.B); tma_prefetch_desc(&maps.C);
    }
    const int urow0 = p.u_mod > 0 ? d0 % p.u_mod : d0;
    for (int t = 0; t < ntiles; ++t) {
      const int s = t % STAGES, use = t / STAGES;
      const int l0 = t * LT, len = min(LT, L - l0);
      mbar_wait_relaxed(&empty[s], (use & 1) ^ 1);    // passes immediately the first time a stage is used
      if (tma) {
        if (lane == 0) {
          const int m0 = rev ? L - l0 - LT : l0;       // memory offset of the tile (may be < 0: zero-filled by TMA)
          mbar_arrive_expect_tx(&full[s], (uint32_t)S::stage_floats * 4);
          tma_load_3d(st_u(s), &maps.u, m0, urow0, b, &full[s]);
          tma_load_3d(st_dl(s), &maps.dl, m0, d0, b, &full[s]);
          tma_load_4d(st_B(s), &maps.B, m0, 0, g, b, &full[s]);
          tma_load_4d(st_C(s), &maps.C, m0, 0, g, b, &full[s]);
        }
      } else {
        stage_rows<LT, LT>(st_u(s), p.u, p.io_dtype, u_off, CH, rows_valid, l0, len, so, lane, 32);
        stage_rows<LT, LT>(st_dl(s), p.delta, p.io_dtype, dl_off, CH, rows_valid, l0, len, so, lane, 32);
        stage_rows<LT, LT>(st_B(s), p.Bm, p.io_dtype, B_off, NPB, p.N, l0, len, so, lane, 32);
        stage_rows<LT, LT>(st_C(s), p.Cm, p.io_dtype, C_off, NPB, p.N, l0, len, so, lane, 32);
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);         // release: the tile is visible to whoever acquires `full`
      }
    }
    return;
  }

  // =============================== consumer warps ===============================
  const int q = lane % R, rl = lane / R;
  int rk[RPT];
  float A2[RPT][NS], h[RPT][NS];
#pragma unroll
  for (int k = 0; k < RPT; ++k) {
    rk[k] = warp * RPW + k * RL + rl;
#pragma unroll
    for (int j = 0; j < NS; ++j) {
      const int n = j * R + q;
      A2[k][j] = (rk[k] < rows_valid && n < p.N) ? p.A[(int64_t)(d0 + rk[k]) * p.A_ld + n] * kLog2e : 0.f;
      h[k][j] = (STATE && rk[k] < rows_valid && n < p.N) ? st.h0[state_slot(p, b, d0 + rk[k], n)] : 0.f;
    }
  }

  // the tile loop is instantiated twice so that the mirror of reversed traversals costs nothing at run time
  auto consume = [&](auto REV) {
    constexpr bool REVV = decltype(REV)::value;
  for (int t = 0; t < ntiles; ++t) {
    const int s = t % STAGES, use = t / STAGES;
    const int l0 = t * LT, len = min(LT, L - l0);
    float* s_dl = st_dl(s);
    const float* s_u = st_u(s);
    const float* s_B = st_B(s);
    const float* s_C = st_C(s);
    mbar_wait(&full[s], use & 1);
    // activate delta once per element, for this warp's own rows: delta = softplus(raw + bias); du = delta * u
    for (int i = lane; i < RPW * (LT / 4); i += 32) {
      const int r = warp * RPW + i / (LT / 4), c = (i % (LT / 4)) * 4;      // c: scan column of the 4-group
      float4 dv = tile_ld4(s_dl, r, c, REVV);
      float4 uv = tile_ld4(s_u, r, c, REVV);
      const float bias = s_bias[r];
      float4 du;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float x = f4_at(dv, e) + bias;
        if (p.softplus) x = softplus20(x);
        const bool live = c + e < len;       // beyond the end of the sequence the state is frozen (a = 1, b = 0)
        f4_at(dv, e) = live ? x : 0.f;
        f4_at(du, e) = live ? x * f4_at(uv, e) : 0.f;
      }
      tile_st4(s_dl, r, c, REVV, dv);
      tile_st4(s_du, r, c, REVV, du);
    }
    __syncwarp();

    for (int i4 = 0; i4 < LT / 4; i4 += R) {
      float yacc[RPT][R * 4];
#pragma unroll
      for (int gq = 0; gq < R; ++gq) {
        const int c = (i4 + gq) * 4;
        float4 Bv[NS], Cv[NS];
#pragma unroll
        for (int j = 0; j < NS; ++j) {
          Bv[j] = tile_ld4(s_B, j * R + q, c, REVV);
          Cv[j] = tile_ld4(s_C, j * R + q, c, REVV);
        }
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
          const float4 dv = tile_ld4(s_dl, rk[k], c, REVV);
          const float4 du = tile_ld4(s_du, rk[k], c, REVV);
          // two scan positions per packed instruction (FMUL2 / FFMA2 halve the issue slots of the products and of
          // the C.h accumulation); only the recurrence itself is inherently sequential and stays scalar
#pragma unroll
          for (int ep = 0; ep < 2; ++ep) {
            const float2 d2 = ep == 0 ? make_float2(dv.x, dv.y) : make_float2(dv.z, dv.w);
            const float2 u2 = ep == 0 ? make_float2(du.x, du.y) : make_float2(du.z, du.w);
            float2 y2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < NS; ++j) {
              const float2 arg = __fmul2_rn(d2, make_float2(A2[k][j], A2[k][j]));
              const float a0 = ex2f(arg.x), a1 = ex2f(arg.y);
              const float2 b2 = ep == 0 ? make_float2(Bv[j].x, Bv[j].y) : make_float2(Bv[j].z, Bv[j].w);
              const float2 c2 = ep == 0 ? make_float2(Cv[j].x, Cv[j].y) : make_float2(Cv[j].z, Cv[j].w);
              const float2 bu = __fmul2_rn(u2, b2);
              const float h0 = fmaf(a0, h[k][j], bu.x);
              const float h1 = fmaf(a1, h0, bu.y);
              h[k][j] = h1;
              y2 = __ffma2_rn(make_float2(h0, h1), c2, y2);
            }
            yacc[k][gq * 4 + 2 * ep] = y2.x;
            yacc[k][gq * 4 + 2 * ep + 1] = y2.y;
          }
        }
      }
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        reduce_scatter_groups<R>(yacc[k], q);
        const int c = (i4 + q) * 4;                 // this lane owns group q of the R groups just finished
        if (p.out != nullptr && rk[k] < rows_valid && c < len) {
          const float4 uv = tile_ld4(s_u, rk[k], c, REVV);
          const float Dd = s_D[rk[k]];
          const float4 y4 = make_float4(fmaf(Dd, uv.x, yacc[k][0]), fmaf(Dd, uv.y, yacc[k][1]),
                                        fmaf(Dd, uv.z, yacc[k][2]), fmaf(Dd, uv.w, yacc[k][3]));
          store_scan4(p.out, p.out_dtype, out_boff + (int64_t)(d0 + rk[k]) * p.out_ds, l0 + c, l0 + len, y4, so,
                      p.accum != 0);
        }
      }
    }
    // state checkpoint at the end of the tile (= SS2D_CHUNK scan positions), for the backward's recompute:
    // ckpt[b][d][tile][n], states in natural order so that forward and backward may split them over lanes differently
    if (p.ckpt != nullptr) {
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        if (rk[k] < rows_valid) {
          float* dst = p.ckpt + (((int64_t)b * p.dim + d0 + rk[k]) * p.nck + t) * p.N;
#pragma unroll
          for (int j = 0; j < NS; ++j)
            if (j * R + q < p.N) dst[j * R + q] = h[k][j];
        }
      }
    }
    // release the stage: this warp's generic-proxy writes (activated delta) are ordered before the TMA that refills it
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  }
  };
  if (rev) consume(std::true_type{}); else consume(std::false_type{});
  if (p.last_state != nullptr) {
#pragma unroll
    for (int k = 0; k < RPT; ++k)
#pragma unroll
      for (int j = 0; j < NS; ++j) {
        const int n = j * R + q;
        if (rk[k] < rows_valid && n < p.N) {
          const int64_t slot = ((int64_t)b * p.dim + d0 + rk[k]) * p.A_ld + n;
          if (p.last_il) { p.last_state[2 * slot] = 0.f; p.last_state[2 * slot + 1] = h[k][j]; }
          else p.last_state[slot] = h[k][j];
        }
      }
  }
}

template <int NS, int R, int RPT, int STAGES, bool STATE>
static cudaError_t launch_fwd(ScanParams p, const ScanState& st, cudaStream_t stream) {
  using S = FwdShape<NS, R, RPT, STAGES>;
  auto kern = scan_fwd_kernel<NS, R, RPT, STAGES, STATE>;
  static PerDeviceOnce once;     // per instantiation and per device (the attribute is per-function, per-device and sticky)
  cudaError_t ea = func_attr_once(once, reinterpret_cast<const void*>(kern), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::smem_bytes);
  if (ea != cudaSuccess) return ea;
  TmaMaps maps;
  if (p.tma_ok && !(p.u_mod == 0 || p.u_mod % p.dpg == 0)) p.tma_ok = 0;
  if (p.tma_ok && !make_scan_maps(p, S::CH, S::NPB, false, &maps)) p.tma_ok = 0;
  if (!p.tma_ok) memset(&maps, 0, sizeof(maps));
  dim3 grid((p.dpg + S::CH - 1) / S::CH, p.G, p.batch);
  kern<<<grid, kFwdThreads, S::smem_bytes, stream>>>(p, maps, st);
  return cudaGetLastError();
}

template <bool STATE>
static cudaError_t fwd_variant(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  const Variant v = pick_variant(p.N);
  if (v.NS == 1) return launch_fwd<1, 1, 1, 3, STATE>(p, st, stream);
  if (v.NS == 2) return launch_fwd<2, 1, 1, 3, STATE>(p, st, stream);
  if (v.R == 1) return launch_fwd<4, 1, 1, 3, STATE>(p, st, stream);
  if (v.R == 2) return launch_fwd<4, 2, 1, 3, STATE>(p, st, stream);
  if (v.R == 4) return launch_fwd<4, 4, 1, 3, STATE>(p, st, stream);     // measured best of RPT in {1, 2} x STAGES in {2, 3, 4} (DESIGN.md §3.1)
  return launch_fwd<4, 8, 1, 3, STATE>(p, st, stream);
}

cudaError_t scan_fwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  return st.h0 ? fwd_variant<true>(p, st, stream) : fwd_variant<false>(p, st, stream);
}

}  // namespace ss2d
