// Selective-scan forward, fast path of the north-star regime (4 < d_state <= 16, fp32, TMA-stageable operands,
// contiguous traversal: SCAN layout or directions 1 / 3). Everything else runs scan_fwd.cu.
//
// Replaces selective_scan_fwd_kernel (/root/reference/gm-unet/kernels/selective_scan/csrc/selective_scan/cus/
// selective_scan_fwd_kernel.cuh:61-172). Same mathematics as scan_fwd.cu (h = exp(delta A) h + delta u B, y = C.h + D u,
// one state checkpoint per SS2D_CHUNK positions); different machine mapping, driven by what ncu showed for scan_fwd.cu
// (shared-memory pipe 76 % busy with B/C re-reads by every row lane, 15 % of the time in the shuffle reduce-scatter of y,
// 17 % of the stall samples in the producer warp's poll loop, 61 % of the MUFU.EX2 floor):
//   * a ROW belongs to R lanes (R = 1: one lane owns all 16 states of its row; R = 2 for calls that would not fill the
//     machine with 32-row warps). With R = 1 the sum over states never leaves the lane (no shuffles), B and C are
//     warp-uniform broadcast loads (one shared-memory wavefront per LDS.128 instead of four), delta is activated in
//     registers by the lane that owns the row (no activated copy written back to shared memory), and the lane has
//     16 independent recurrences in flight — enough instruction-level parallelism to keep MUFU.EX2 busy with one warp
//     per scheduler.
//   * no producer warp, no polling, no CTA-wide barrier: every warp streams its own 32 / R rows and its own copy of the
//     B / C tiles (L2 hits after the first warp of a group) through a private TMA ring; lane 0 refills a stage the
//     moment its warp is done with it. A CTA is just a container of independent warps; warp blocks are numbered
//     (batch, group, row block) so that a call fills the machine evenly whatever dpg is.
#include <type_traits>

#include "scan_params.h"
#include "host_util.h"
#include "scan_tile.cuh"
#include "tma_host.h"

namespace ss2d {

constexpr int FR_NW = 4;          // independent warps per CTA
constexpr int FR_STAGES = 2;
constexpr int FR_LT = kTileL;     // scan positions per tile = SS2D_CHUNK (one checkpoint per tile)
static_assert(FR_LT == SS2D_CHUNK, "one checkpoint per tile");

struct FwdrMaps { TMap u, dl, B, C; };

template <int R>
struct FwdrShape {
  static constexpr int ROWS = 32 / R;                                  // rows per warp
  static constexpr int stage_bytes = (2 * ROWS + 2 * 16) * FR_LT * 4;  // delta | u | B | C tiles (all multiples of 1024 bytes)
  static constexpr int warp_bytes = FR_STAGES * stage_bytes;
  static constexpr size_t smem_bytes = (size_t)FR_NW * warp_bytes + FR_NW * FR_STAGES * 8 + 1024;
};

// STATE (whole-row mode only): the rows start from st.h0 instead of 0. Segmented mode scans every segment from zero and
// leaves h0 to the carry / fix-up kernels.
// GATE (whole-row mode only, ss2d_scan_fwd_gated): the store step also writes gt.out_z = y * silu(z). z is not staged in the
// ring: a fifth tile would take the 32-row CTA from 97 to 129 KB of shared memory, one CTA per SM instead of two. The lane
// that stores a 4-position group reads its z quad from global memory one group pair ahead instead. The GATE instantiations
// take h0 from st.h0 when it is set (a runtime test once per row), so that their names keep STATE = false.
template <int NS, int R, bool SOFTPLUS, bool SEG, bool GATE, bool STATE>
__global__ void __launch_bounds__(FR_NW * 32) scan_fwdr_kernel(const ScanParams p, const __grid_constant__ FwdrMaps maps,
                                                               const int nrb, const int nwb, const int nseg_arg, const int tps,
                                                               const ScanState st, const ScanGate gt) {
  static_assert(!(GATE && (SEG || STATE)), "the gated instantiations are whole-row and read h0 at run time");
  const int nseg = SEG ? nseg_arg : 1;                     // compile-time 1 in the whole-row instantiation
  using S = FwdrShape<R>;
  constexpr int ROWS = S::ROWS;
  extern __shared__ __align__(16) unsigned char smem_rawfr[];
  unsigned char* smem = smem_rawfr + ((1024 - (smem_u32(smem_rawfr) & 1023)) & 1023);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wb = blockIdx.x * FR_NW + warp;                // warp block: (batch, group, row block), row block fastest
  if (wb >= nwb) return;                                   // warps are independent: no CTA-wide barrier anywhere
  // warp block = (batch, group, segment of the sequence, row block). nseg > 1 (small calls, SEGMENTED mode): every warp scans
  // tps tiles from a ZERO state; scan_fwd_fixup_kernel adds the carried-in states afterwards (see scan_fwdr_try).
  const int rb = wb % nrb, sb = wb / nrb;
  const int seg = SEG ? sb % nseg : 0, bg = SEG ? sb / nseg : sb;
  const int g = bg % p.G, b = bg / p.G;
  const int q = lane % R, rl = lane / R;
  const int row0 = rb * ROWS;                              // first row of this warp inside the group
  const int row = row0 + rl;
  const bool valid = row < p.dpg;
  const int d = g * p.dpg + (valid ? row : 0);             // global channel of this lane's row
  const int L = p.L;
  const int dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
  const bool rev = dir == 3;
  const int ntiles_row = (L + FR_LT - 1) / FR_LT;
  const int tb = SEG ? seg * tps : 0;                      // first tile of this warp's segment
  const int ntiles = SEG ? min(ntiles_row, tb + tps) : ntiles_row;      // one past its last tile

  float* wsm = reinterpret_cast<float*>(smem + warp * S::warp_bytes);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + FR_NW * S::warp_bytes) + warp * FR_STAGES;
  auto st_dl = [&](int s) { return wsm + s * (S::stage_bytes / 4); };
  auto st_u = [&](int s) { return wsm + s * (S::stage_bytes / 4) + ROWS * FR_LT; };
  auto st_B = [&](int s) { return wsm + s * (S::stage_bytes / 4) + 2 * ROWS * FR_LT; };
  auto st_C = [&](int s) { return wsm + s * (S::stage_bytes / 4) + (2 * ROWS + 16) * FR_LT; };

  const int ug = p.u_mod > 0 ? g % (p.u_mod / p.dpg) : g;  // group coordinate of u when the groups share it
  auto issue = [&](int t) {                                // lane 0 only
    const int s = (t - tb) % FR_STAGES;
    const int l0 = t * FR_LT;
    const int m0 = rev ? L - l0 - FR_LT : l0;              // memory offset of the tile (may be < 0: zero-filled by TMA)
    mbar_arrive_expect_tx(&full[s], (uint32_t)S::stage_bytes);
    tma_load_4d(st_dl(s), &maps.dl, m0, row0, g, b, &full[s]);
    tma_load_4d(st_u(s), &maps.u, m0, row0, ug, b, &full[s]);
    tma_load_4d(st_B(s), &maps.B, m0, 0, g, b, &full[s]);
    tma_load_4d(st_C(s), &maps.C, m0, 0, g, b, &full[s]);
  };
  if (lane == 0) {
    for (int s = 0; s < FR_STAGES; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
    for (int t = tb; t < tb + FR_STAGES && t < ntiles; ++t) issue(t);
  }
  __syncwarp();

  float A2[NS], h[NS];
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    const int n = j * R + q;
    A2[j] = (valid && n < p.N) ? p.A[(int64_t)d * p.A_ld + n] * kLog2e : 0.f;
    h[j] = ((STATE || (GATE && st.h0 != nullptr)) && valid && n < p.N) ? st.h0[state_slot(p, b, d, n)] : 0.f;
  }
  const float bias = (valid && p.bias) ? p.bias[d] : 0.f;
  const float Dd = (valid && p.Dv) ? p.Dv[d] : 0.f;
  const int64_t out_ro = (int64_t)b * p.out_bs + (int64_t)d * p.out_ds;
  const bool ck_vec = (p.N & 3) == 0 && R == 1;
  const bool do_out = valid && p.out != nullptr;       // fp32, rows 16-byte aligned (checked by the host)
  float* const outp = static_cast<float*>(p.out) + out_ro;

  // B / C tiles: with R = 1 every load is warp-uniform, so the tiles are staged UNSWIZZLED (plain row * 32 + column:
  // immediate offsets from one base register per group); with R > 1 the row's lanes read different state rows and
  // the TMA 128-byte swizzle keeps them on different banks.
  auto bc_ld4 = [&](const float* tile, int r, int c, bool rv) -> float4 {
    if constexpr (R == 1) {
      const float4 v = *reinterpret_cast<const float4*>(tile + r * FR_LT + (rv ? FR_LT - 4 - c : c));
      return rv ? make_float4(v.w, v.z, v.y, v.x) : v;
    } else {
      return tile_ld4(tile, r, c, rv);
    }
  };

  auto body = [&](auto REV) {
    constexpr bool REVV = decltype(REV)::value;
    // This lane activates the 4-position groups it will also store: delta = softplus(raw + bias), du = delta * u.
    // The activation of the NEXT group — across tile boundaries too — is requested before the recurrences of the current
    // one, so that its shared-memory and MUFU latencies overlap them (one warp per scheduler: nobody else would hide
    // them). Nothing in the group loop branches (softplus is a template parameter, stores are predicated, the source of
    // the next group is chosen by pointer selects), so ptxas interleaves the two in one basic block.
    float4 dm_n, um_n, dum_n;
    auto activate = [&](const float* t_dl, const float* t_u, int i4, int tlen) {
      const int cm = (i4 + q) * 4;
      dm_n = tile_ld4(t_dl, rl, cm, REVV);
      um_n = tile_ld4(t_u, rl, cm, REVV);
      const bool live = cm < tlen;                 // L % 4 == 0 on this path: groups are whole. Beyond the end of the
#pragma unroll                                     // sequence the state is frozen (delta = 0 -> a = 1; u is zero-filled)
      for (int e = 0; e < 4; ++e) {
        float x = f4_at(dm_n, e) + bias;
        if (SOFTPLUS) x = softplus20(x);
        x = live ? x : 0.f;
        f4_at(dm_n, e) = x;
        f4_at(dum_n, e) = x * f4_at(um_n, e);
      }
    };
    // GATE: z quads of the group pair being computed (zc) and of the next one (zn), in memory order like y4
    const float* zrow = GATE ? static_cast<const float*>(gt.z) + out_ro : nullptr;
    float4 zc[2], zn[2];
    auto load_z = [&](int pos) -> float4 {      // scan position of the quad's first element
      return pos < L ? __ldg(reinterpret_cast<const float4*>(zrow + (REVV ? L - 4 - pos : pos))) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    if constexpr (GATE) {
#pragma unroll
      for (int k = 0; k < 2; ++k) zn[k] = load_z((k * R + q) * 4);
    }
    mbar_wait(&full[0], 0);
    activate(st_dl(0), st_u(0), 0, min(FR_LT, L - tb * FR_LT));
    for (int t = tb; t < ntiles; ++t) {
      const int s = (t - tb) % FR_STAGES, sn = (t + 1 - tb) % FR_STAGES;
      const int l0 = t * FR_LT, len = min(FR_LT, L - l0);
      const float* s_dl = st_dl(s);
      const float* s_u = st_u(s);
      const float* s_B = st_B(s);
      const float* s_C = st_C(s);
      const bool more = t + 1 < ntiles;
      const int len_n = more ? min(FR_LT, L - l0 - FR_LT) : 0;
#pragma unroll 1
      for (int i4 = 0; i4 < FR_LT / 4; i4 += 2 * R) {
        const bool last_pair = i4 == FR_LT / 4 - 2 * R;
        if (last_pair && more) mbar_wait(&full[sn], ((t + 1 - tb) / FR_STAGES) & 1);    // requested one tile ago: there by now
        if constexpr (GATE) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            zc[k] = zn[k];
            zn[k] = load_z(l0 + (i4 + k * R + q) * 4 + 8 * R);
          }
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int ii = i4 + k * R;
          const int cm = (ii + q) * 4;
          float4 dm = dm_n, um = um_n, dum = dum_n;
          {
            const bool wrap = k == 1 && last_pair;   // the last group of a tile activates the first group of the next tile
            activate(wrap ? st_dl(sn) : s_dl, wrap ? st_u(sn) : s_u, wrap ? 0 : ii + R, wrap ? len_n : len);
          }
          float yacc[R * 4];
#pragma unroll
          for (int gq = 0; gq < R; ++gq) {
            const int c = (ii + gq) * 4;
            float4 dv = dm, du = dum;
            if constexpr (R > 1) {                 // the group's owner broadcasts its activated values to the row's lanes
              const int src = (lane & ~(R - 1)) | gq;
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                f4_at(dv, e) = __shfl_sync(0xffffffffu, f4_at(dm, e), src);
                f4_at(du, e) = __shfl_sync(0xffffffffu, f4_at(dum, e), src);
              }
            }
            float2 y01 = make_float2(0.f, 0.f), y23 = make_float2(0.f, 0.f);
            const float2 d01 = make_float2(dv.x, dv.y), d23 = make_float2(dv.z, dv.w);
            const float2 u01 = make_float2(du.x, du.y), u23 = make_float2(du.z, du.w);
#pragma unroll
            for (int j = 0; j < NS; ++j) {
              const float4 Bv = bc_ld4(s_B, j * R + q, c, REVV);      // R = 1: warp-uniform address, one wavefront
              const float4 Cv = bc_ld4(s_C, j * R + q, c, REVV);
              const float2 aj = make_float2(A2[j], A2[j]);
              const float2 g01 = __fmul2_rn(d01, aj), g23 = __fmul2_rn(d23, aj);
              const float a0 = ex2f(g01.x), a1 = ex2f(g01.y), a2 = ex2f(g23.x), a3 = ex2f(g23.y);
              const float2 b01 = __fmul2_rn(u01, make_float2(Bv.x, Bv.y)), b23 = __fmul2_rn(u23, make_float2(Bv.z, Bv.w));
              const float h0 = fmaf(a0, h[j], b01.x);
              const float h1 = fmaf(a1, h0, b01.y);
              const float h2 = fmaf(a2, h1, b23.x);
              const float h3 = fmaf(a3, h2, b23.y);
              h[j] = h3;
              y01 = __ffma2_rn(make_float2(h0, h1), make_float2(Cv.x, Cv.y), y01);
              y23 = __ffma2_rn(make_float2(h2, h3), make_float2(Cv.z, Cv.w), y23);
            }
            yacc[gq * 4 + 0] = y01.x; yacc[gq * 4 + 1] = y01.y; yacc[gq * 4 + 2] = y23.x; yacc[gq * 4 + 3] = y23.y;
          }
          reduce_scatter_groups<R>(yacc, q);       // no-op for R = 1; lane q ends up owning group ii + q
          float4 y4 = make_float4(fmaf(Dd, um.x, yacc[0]), fmaf(Dd, um.y, yacc[1]), fmaf(Dd, um.z, yacc[2]),
                                  fmaf(Dd, um.w, yacc[3]));
          if (REVV) y4 = make_float4(y4.w, y4.z, y4.y, y4.x);
          const int mpos = REVV ? L - 4 - (l0 + cm) : l0 + cm;    // memory position of the group's first element
          if (do_out && cm < len) *reinterpret_cast<float4*>(outp + mpos) = y4;
          if constexpr (GATE) {
            const float4 zq = zc[k];
            const float4 g4 = make_float4(y4.x * silu_f(zq.x), y4.y * silu_f(zq.y), y4.z * silu_f(zq.z), y4.w * silu_f(zq.w));
            if (do_out && cm < len) *reinterpret_cast<float4*>(static_cast<float*>(gt.out_z) + out_ro + mpos) = g4;
          }
        }
      }
      // state checkpoint at the end of the tile, for the backward's recompute: ckpt[b][d][tile][n]
      if (p.ckpt != nullptr && valid) {
        float* dst = p.ckpt + (((int64_t)b * p.dim + d) * p.nck + t) * p.N;
        if (ck_vec) {
#pragma unroll
          for (int j = 0; j < NS; j += 4)
            if (j < p.N) *reinterpret_cast<float4*>(dst + j) = make_float4(h[j], h[j + 1], h[j + 2], h[j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < NS; ++j)
            if (j * R + q < p.N) dst[j * R + q] = h[j];
        }
      }
      // refill the stage (only generic-proxy READS touched it; the fence keeps them ahead of the async-proxy writes)
      fence_proxy_async();
      __syncwarp();
      if (lane == 0 && t + FR_STAGES < ntiles) issue(t + FR_STAGES);
    }
  };
  if (rev) body(std::true_type{}); else body(std::false_type{});

  if (p.last_state != nullptr && valid && nseg == 1) {     // segmented mode: written by the fix-up kernel
#pragma unroll
    for (int j = 0; j < NS; ++j) {
      const int n = j * R + q;
      if (n < p.N) {
        const int64_t slot = ((int64_t)b * p.dim + d) * p.A_ld + n;
        if (p.last_il) { p.last_state[2 * slot] = 0.f; p.last_state[2 * slot + 1] = h[j]; }
        else p.last_state[slot] = h[j];
      }
    }
  }
}

template <int R>
static bool fwdr_maps(const ScanParams& p, FwdrMaps* m) {
  constexpr int ROWS = FwdrShape<R>::ROWS;
  const long long ugroups = p.u_mod > 0 ? p.u_mod / p.dpg : p.G;
  const long long du[4] = {p.L, p.dpg, ugroups, p.batch}, su[4] = {1, p.u_ds, (long long)p.dpg * p.u_ds, p.u_bs};
  const long long dd[4] = {p.L, p.dpg, p.G, p.batch}, sd[4] = {1, p.dl_ds, (long long)p.dpg * p.dl_ds, p.dl_bs};
  const long long d4[4] = {p.L, p.N, p.G, p.batch};
  const long long s4B[4] = {1, p.B_ns, p.B_gs, p.B_bs}, s4C[4] = {1, p.C_ns, p.C_gs, p.C_bs};
  return make_tmap(&m->u, p.u, 4, du, su, ROWS) && make_tmap(&m->dl, p.delta, 4, dd, sd, ROWS) &&
         make_tmap(&m->B, p.Bm, 4, d4, s4B, 16, R > 1) && make_tmap(&m->C, p.Cm, 4, d4, s4C, 16, R > 1);
}

template <int NS, int R, bool SOFTPLUS, bool SEG, bool STATE, bool GATE = false>
static cudaError_t launch_fwdr(const ScanParams& p, const FwdrMaps& maps, const ScanState& st, cudaStream_t stream, int nseg = 1,
                               int tps = 0, const ScanGate& gt = ScanGate{nullptr, nullptr}) {
  using S = FwdrShape<R>;
  auto kern = scan_fwdr_kernel<NS, R, SOFTPLUS, SEG, GATE, STATE>;
  static PerDeviceOnce once;
  cudaError_t e = func_attr_once(once, reinterpret_cast<const void*>(kern), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::smem_bytes);
  if (e != cudaSuccess) return e;
  if (!SEG) nseg = 1;
  const int nrb = (p.dpg + S::ROWS - 1) / S::ROWS;
  const long long nwb = (long long)nrb * p.G * p.batch * nseg;
  if (tps <= 0) tps = (p.L + FR_LT - 1) / FR_LT;
  kern<<<(unsigned)((nwb + FR_NW - 1) / FR_NW), FR_NW * 32, S::smem_bytes, stream>>>(p, maps, nrb, (int)nwb, nseg, tps, st, gt);
  return cudaGetLastError();
}

// ---- SEGMENTED mode: the sequence split over several warps (small calls: batch 1 / 2 of the north-star shape give the machine
// 24 / 48 CTAs of sequential work otherwise). The reference chunks L the same way with a running prefix per 2048 positions
// (selective_scan_fwd_kernel.cuh:101-158); here a segment is `tps` 32-position tiles:
//   1. scan_fwdr_kernel with nseg > 1: every (row block, segment) warp scans its tiles from a ZERO state -> local y, local
//      checkpoints (the segment's last checkpoint = its local end state e_s);
//   2. scan_fwd_carry_kernel (warp per row): S_s = sum of the activated delta over segment s (the decay of state n across the
//      whole segment is exp(A_n S_s)), then the true end states h_s = e_s + exp(A S_s) h_(s-1), written over the segments' last
//      checkpoints (and last_state);
//   3. scan_fwd_fixup_kernel (warp per (row, segment >= 1)): with c_l the inclusive running sum of delta inside the segment,
//      y_l += sum_n C_(l,n) exp(A_n c_l) h_in,n and checkpoint_t += exp(A c_(end of t)) h_in.
// Twice the exponentials of the sequential scan for nseg times its parallelism; exact in exact arithmetic (products of
// exponentials = exponential of the sum). Needs the checkpoint buffer (it carries e_s); calls without one take scan_fwd.cu.
constexpr int FX_MAX_SEG = 64;

// 4 consecutive scan positions starting at l of one row (L % 4 == 0, rows 16-byte aligned on this path): one 128-bit access;
// a reversed traversal reads the mirrored quad and swaps it.
__device__ __forceinline__ float4 ldq(const float* __restrict__ row, int l, int L, bool rev) {
  if (!rev) return __ldg(reinterpret_cast<const float4*>(row + l));
  const float4 v = __ldg(reinterpret_cast<const float4*>(row + (L - 4 - l)));
  return make_float4(v.w, v.z, v.y, v.x);
}
template <bool SOFTPLUS>
__device__ __forceinline__ float4 activate4(float4 x, float bias) {
  x.x += bias; x.y += bias; x.z += bias; x.w += bias;
  if (SOFTPLUS) { x.x = softplus20(x.x); x.y = softplus20(x.y); x.z = softplus20(x.z); x.w = softplus20(x.w); }
  return x;
}

// CTA per row: its four warps split the segments for the sums, warp 0 runs the carry chain.
// STATE: the chain starts from h0, so segment 0's end state changes too.
template <bool SOFTPLUS, bool STATE>
__global__ void __launch_bounds__(128) scan_fwd_carry_kernel(const ScanParams p, const int tps, const int nseg, const ScanState st) {
  __shared__ float s_sum[FX_MAX_SEG];
  __shared__ float s_e[FX_MAX_SEG][16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = blockIdx.x;
  const int b = row / p.dim, d = row - b * p.dim, g = d / p.dpg;
  const int L = p.L, N = p.N;
  const bool rev = p.layout == SS2D_LAYOUT_NATURAL && p.dirs[g] == 3;
  const int ntiles = (L + FR_LT - 1) / FR_LT;
  const float* dl = static_cast<const float*>(p.delta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  float* ck = p.ckpt + ((int64_t)b * p.dim + d) * p.nck * N;
  const float bias = p.bias ? p.bias[d] : 0.f;
  // phase 1 (independent iterations): S_s = sum of the activated delta over segment s, and the local end states e_s
#pragma unroll 2
  for (int s = warp; s < nseg; s += 4) {
    const int lb = s * tps * FR_LT, le = min(L, lb + tps * FR_LT);
    float sum = 0.f;
    for (int l = lb + lane * 4; l < le; l += 128) {
      const float4 x = activate4<SOFTPLUS>(ldq(dl, l, L, rev), bias);
      sum += (x.x + x.y) + (x.z + x.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const int tl = min(ntiles, (s + 1) * tps) - 1;           // last tile of the segment
    if (lane == 0) s_sum[s] = sum;
    if (lane < N) s_e[s][lane] = ck[(int64_t)tl * N + lane];
  }
  __syncthreads();
  // phase 2: h_s = e_s + exp(A S_s) h_(s-1), the true end state of segment s
  if (warp == 0 && lane < N) {
    const float A2l = p.A[(int64_t)d * p.A_ld + lane] * kLog2e;
    float h = STATE ? st.h0[state_slot(p, b, d, lane)] : 0.f;
    for (int s = 0; s < nseg; ++s) {
      h = fmaf(ex2f(A2l * s_sum[s]), h, s_e[s][lane]);
      const int tl = min(ntiles, (s + 1) * tps) - 1;
      if (STATE || s > 0) ck[(int64_t)tl * N + lane] = h;
    }
    if (p.last_state != nullptr) {
      const int64_t slot = ((int64_t)b * p.dim + d) * p.A_ld + lane;
      if (p.last_il) { p.last_state[2 * slot] = 0.f; p.last_state[2 * slot + 1] = h; }
      else p.last_state[slot] = h;
    }
  }
}

// warp per (row, segment >= 1; STATE: segment >= 0, whose carried-in state is h0); a lane owns 4 consecutive positions of a
// 128-position step
template <bool SOFTPLUS, bool STATE>
__global__ void __launch_bounds__(128) scan_fwd_fixup_kernel(const ScanParams p, const int tps, const int nseg, const ScanState st) {
  constexpr int S0 = STATE ? 0 : 1;      // first segment fixed up
  const int lane = threadIdx.x & 31;
  const int64_t wid = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (wid >= (int64_t)p.batch * p.dim * (nseg - S0)) return;
  const int row = (int)(wid / (nseg - S0)), seg = S0 + (int)(wid % (nseg - S0));
  const int b = row / p.dim, d = row - b * p.dim, g = d / p.dpg;
  const int L = p.L, N = p.N;
  const bool rev = p.layout == SS2D_LAYOUT_NATURAL && p.dirs[g] == 3;
  const int ntiles = (L + FR_LT - 1) / FR_LT;
  const int tb = seg * tps, te = min(ntiles, tb + tps);
  const int lb = tb * FR_LT, le = min(L, te * FR_LT);
  const float* dl = static_cast<const float*>(p.delta) + (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  const float* Cg = static_cast<const float*>(p.Cm) + (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;
  float* out = p.out ? static_cast<float*>(p.out) + (int64_t)b * p.out_bs + (int64_t)d * p.out_ds : nullptr;
  float* ck = p.ckpt + ((int64_t)b * p.dim + d) * p.nck * N;
  const float bias = p.bias ? p.bias[d] : 0.f;
  const float A2l = lane < N ? p.A[(int64_t)d * p.A_ld + lane] * kLog2e : 0.f;
  // true state entering the segment (carry kernel; h0 for segment 0)
  const float hl = lane >= N ? 0.f : (STATE && seg == 0) ? st.h0[state_slot(p, b, d, lane)] : ck[(int64_t)(tb - 1) * N + lane];
  float A2[16], hin[16];
#pragma unroll
  for (int n = 0; n < 16; ++n) {
    A2[n] = __shfl_sync(0xffffffffu, A2l, n);
    hin[n] = __shfl_sync(0xffffffffu, hl, n);
  }
  // once A_n * (running sum) is below the flush-to-zero range of ex2 for every state, every further term is EXACTLY zero
  float amax = -3.0e38f;
#pragma unroll
  for (int n = 0; n < 16; ++n) amax = n < N ? fmaxf(amax, A2[n]) : amax;
  float base = 0.f;
#pragma unroll 2
  for (int l0 = lb; l0 < le; l0 += 128) {
    if (SOFTPLUS && amax * base < -160.f) break;              // (softplus: delta >= 0, the running sum only grows)
    const int l = l0 + lane * 4;
    const bool live = l < le;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) x = activate4<SOFTPLUS>(ldq(dl, l, L, rev), bias);
    x.y += x.x; x.z += x.y; x.w += x.z;                      // inclusive running sum inside the quad
    float incl = x.w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    const float off = base + (incl - x.w);
    const float4 cum = make_float4(off + x.x, off + x.y, off + x.z, off + x.w);
    if (live && out != nullptr) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      // all C quads first, without a branch per state (states past N re-read row N - 1 and multiply by h_in = 0): 16
      // independent 128-bit loads in flight instead of 16 load -> use round trips
      const float* cp = Cg + (rev ? L - 4 - l : l);          // this lane's quad of state row 0; rows are C_ns apart
      float4 cq[16];
#pragma unroll
      for (int n = 0; n < 16; ++n) cq[n] = __ldg(reinterpret_cast<const float4*>(cp + (int64_t)min(n, N - 1) * p.C_ns));
#pragma unroll
      for (int n = 0; n < 16; ++n) {
        const float4 cv = rev ? make_float4(cq[n].w, cq[n].z, cq[n].y, cq[n].x) : cq[n];
        acc.x = fmaf(cv.x * ex2f(A2[n] * cum.x), hin[n], acc.x);
        acc.y = fmaf(cv.y * ex2f(A2[n] * cum.y), hin[n], acc.y);
        acc.z = fmaf(cv.z * ex2f(A2[n] * cum.z), hin[n], acc.z);
        acc.w = fmaf(cv.w * ex2f(A2[n] * cum.w), hin[n], acc.w);
      }
      float4* op = reinterpret_cast<float4*>(out + (rev ? L - 4 - l : l));
      float4 o4 = *op;
      if (rev) { o4.x += acc.w; o4.y += acc.z; o4.z += acc.y; o4.w += acc.x; }
      else { o4.x += acc.x; o4.y += acc.y; o4.z += acc.z; o4.w += acc.w; }
      *op = o4;
    }
    // the four 32-position tiles of this step end in lanes 7, 15, 23, 31 (flat past the end of the row)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float cend = __shfl_sync(0xffffffffu, cum.w, 8 * j + 7);
      const int t = l0 / FR_LT + j;
      if (t < te - 1 && lane < N) ck[(int64_t)t * N + lane] += ex2f(A2l * cend) * hl;   // the segment's last one is already true
    }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
}

template <bool STATE>
static cudaError_t fwdr_launch_all(const ScanParams& p, const FwdrMaps& maps, const ScanState& st, cudaStream_t stream, bool r1,
                                   int nseg, int tps) {
  if (r1) return p.softplus ? launch_fwdr<16, 1, true, false, STATE>(p, maps, st, stream) : launch_fwdr<16, 1, false, false, STATE>(p, maps, st, stream);
  if (nseg == 1) return p.softplus ? launch_fwdr<8, 2, true, false, STATE>(p, maps, st, stream) : launch_fwdr<8, 2, false, false, STATE>(p, maps, st, stream);
  cudaError_t e = p.softplus ? launch_fwdr<8, 2, true, true, false>(p, maps, st, stream, nseg, tps)
                             : launch_fwdr<8, 2, false, true, false>(p, maps, st, stream, nseg, tps);
  if (e != cudaSuccess) return e;
  const long long rows = (long long)p.batch * p.dim;
  const unsigned gc = (unsigned)rows, gf = (unsigned)((rows * (nseg - (STATE ? 0 : 1)) + 3) / 4);
  if (p.softplus) {
    scan_fwd_carry_kernel<true, STATE><<<gc, 128, 0, stream>>>(p, tps, nseg, st);
    scan_fwd_fixup_kernel<true, STATE><<<gf, 128, 0, stream>>>(p, tps, nseg, st);
  } else {
    scan_fwd_carry_kernel<false, STATE><<<gc, 128, 0, stream>>>(p, tps, nseg, st);
    scan_fwd_fixup_kernel<false, STATE><<<gf, 128, 0, stream>>>(p, tps, nseg, st);
  }
  return cudaGetLastError();
}

// whole-row gated launch: the z / out_z pointers checked by the caller, h0 read at run time
static cudaError_t fwdr_launch_gated(const ScanParams& p, const FwdrMaps& maps, const ScanState& st, const ScanGate& gt,
                                     cudaStream_t stream, bool r1) {
  if (r1) return p.softplus ? launch_fwdr<16, 1, true, false, false, true>(p, maps, st, stream, 1, 0, gt)
                            : launch_fwdr<16, 1, false, false, false, true>(p, maps, st, stream, 1, 0, gt);
  return p.softplus ? launch_fwdr<8, 2, true, false, false, true>(p, maps, st, stream, 1, 0, gt)
                    : launch_fwdr<8, 2, false, false, false, true>(p, maps, st, stream, 1, 0, gt);
}

int scan_path_policy();     // api.cu
bool scan_gate_fusion();    // api.cu: false when the test hook keeps the gate of a gated call in its own pass

// Returns true when the fast path took the call (*err holds the launch status). gt: the output gate of a gated call
// (gt.z == nullptr otherwise); *gated tells whether the launch wrote out_z too (whole-row mode, z / out_z 16-byte aligned).
bool scan_fwdr_try(const ScanParams& p, const ScanState& st, const ScanGate& gt, cudaStream_t stream, cudaError_t* err,
                   bool* gated) {
  *gated = false;
  if (!p.tma_ok || p.N <= 4 || p.N > 16 || p.accum || p.io_dtype != SS2D_F32 || p.out_dtype != SS2D_F32) return false;
  if (p.u_mod > 0 && p.u_mod % p.dpg != 0) return false;
  for (int g = 0; g < p.G; ++g) {
    const int dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
    if (dir == 2 || dir == 4) return false;
  }
  // 128-bit stores of out: rows aligned to 16 bytes
  if (p.out && ((reinterpret_cast<uintptr_t>(p.out) & 15) || (p.out_bs & 3) || (p.out_ds & 3))) return false;
  // Variant by machine fill (measured on B200, DESIGN.md §3.1a): this mapping needs two warps per scheduler to hide its
  // latencies. 32-row warps (R = 1) when there are that many, else 16-row warps (R = 2), else the sequence is split over
  // several 16-row warps (SEGMENTED mode above) when that gives at least eight segments of at least four tiles, else
  // scan_fwd.cu (8-row warps).
  const long long wb1 = (long long)((p.dpg + 31) / 32) * p.G * p.batch;
  const long long wb2 = (long long)((p.dpg + 15) / 16) * p.G * p.batch;
  if (wb2 >= 0x7fffffffLL / 64) return false;
  const long long need = (long long)sm_count_current_device() * 4 * 2 * 9 / 10;
  const int policy = scan_path_policy();      // 0 unless a parity test forces a path (ss2d_test_force_path)
  if (policy == 3) return false;
  const int ntiles = (p.L + FR_LT - 1) / FR_LT;
  int nseg = 1, tps = ntiles;
  if (policy == 4 || (policy == 0 && wb2 < need)) {
    if (p.ckpt == nullptr) return false;
    const int min_tiles = policy == 4 ? 1 : 4;
    long long want = policy == 4 ? 3 : (need + wb2 - 1) / wb2;
    if (want > ntiles / min_tiles) want = ntiles / min_tiles;
    if (want > FX_MAX_SEG) want = FX_MAX_SEG;
    if (want < (policy == 4 ? 2 : 8)) return false;       // measured: the fix-up pass costs about one sequential sweep of the call
                                                             // -> only calls that leave >= 7/8 of the machine idle are split
    tps = (int)((ntiles + want - 1) / want);
    if (policy != 4) tps = tps < 6 ? 4 : (tps + 2) / 4 * 4;  // whole 128-position steps of the fix-up pass (4 tiles each)
    nseg = (ntiles + tps - 1) / tps;
    if (nseg < 2) return false;
  }
  const bool r1 = nseg == 1 && (policy == 0 ? wb1 >= need : policy == 1);
  FwdrMaps maps;
  if (!(r1 ? fwdr_maps<1>(p, &maps) : fwdr_maps<2>(p, &maps))) return false;
  if (gt.z && scan_gate_fusion() && nseg == 1 && !(reinterpret_cast<uintptr_t>(gt.z) & 15) && !(reinterpret_cast<uintptr_t>(gt.out_z) & 15)) {
    *gated = true;              // out's strides (shared by z / out_z) are multiples of 4: checked above
    *err = fwdr_launch_gated(p, maps, st, gt, stream, r1);
    return true;
  }
  *err = st.h0 ? fwdr_launch_all<true>(p, maps, st, stream, r1, nseg, tps) : fwdr_launch_all<false>(p, maps, st, stream, r1, nseg, tps);
  return true;
}

}  // namespace ss2d
