// Selective-scan backward for sm_100a.
//
// Replaces selective_scan_bwd_kernel (/root/reference/gm-unet/kernels/selective_scan/csrc/selective_scan/cus/
// selective_scan_bwd_kernel.cuh:66-273) and, in NATURAL layout, the backward of CrossScan*/CrossMerge*
// (model/gm/csms6s.py). Not a port: the reference runs one CTA per (batch, channel) row, two CUB block scans per
// state and chunk, and one fp32 global atomic per row and element for dB/dC.
//
// Here a CTA owns CH channel rows of one (batch, group) and walks the tiles of 32 scan positions LAST TO FIRST:
//   * warp 4 (producer) streams the u / delta / dout / B / C tiles through a 2-stage shared-memory ring with tiled
//     TMA loads (or the index-mapped generic copy for 16-bit / transposed / reversed operands), and — being idle
//     otherwise — also folds the consumers' per-warp dB/dC slabs together and sends them to global memory;
//   * warps 0-3 (consumers) each own RPW rows, NS states per lane. Per tile: (1) recompute the states h forward from
//     the forward pass' chunk checkpoint, keeping only one state vector per 4 positions in shared memory;
//     (2) for each group of 4 positions, last to first, re-expand h and a = exp(delta A) into registers and run the
//     adjoint recurrence g_l = C_l dy_l + a_(l+1) g_(l+1). Nothing per-element is ever stored in HBM.
//   * dB/dC partials are summed over the thread's rows in registers, over the warp's row lanes with a shuffle
//     reduce-scatter, and over the CTA's warps by the producer: one vector reduction per (state, 4 positions) and
//     CTA reaches global memory (plain stores when the CTA covers the whole group: deterministic). In deterministic mode
//     (DET) every CTA stores into its own partial slab and scan_bwd_fold_kernel sums the slabs in slab order.
//   * dA, dD, d(delta_bias) leave through a per-batch partial buffer and a deterministic second pass.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "scan_params.h"
#include "host_util.h"
#include "scan_tile.cuh"
#include "tma_host.h"

namespace ss2d {

constexpr int kBwdConsumerWarps = 4;
constexpr int kBwdThreads = 32 * (kBwdConsumerWarps + 1);
constexpr int BLT = kTileL;                 // scan positions per tile (= SS2D_CHUNK)
constexpr int kBwdStages = 2;
constexpr int kHalf = BLT / 2;              // slab hand-off granularity (scan positions)

template <int NS, int R, int RPT>
struct BwdShape {
  static constexpr int RL = 32 / R;
  static constexpr int RPW = RL * RPT;
  static constexpr int CH = kBwdConsumerWarps * RPW;
  static constexpr int NP = NS * R;
  static constexpr int NPB = (NP + 7) / 8 * 8;
  static constexpr int CNT = 2 * NS * 4;                      // dB/dC partials per thread and 4-position group
  static constexpr int stage_floats = (3 * CH + 2 * NPB) * BLT;
  static constexpr int kSlabPitch = kHalf + 4;               // 20 floats: consecutive states land in different bank groups
  static constexpr int slab_floats = 2 * NP * kSlabPitch;     // one warp, one half tile: [dB | dC][NP][16 (+4)]
  static constexpr int hs_floats = (BLT / 4) * RPT * 32 * NS; // one warp: state at the end of each group
  static constexpr size_t smem_bytes =
      (size_t)(kBwdStages * stage_floats + kBwdConsumerWarps * (2 * slab_floats + hs_floats) + 2 * CH) * 4 + 128 + 1024;
};

template <int STRIDE, int CNT, int S>
struct LaneReduceScatter {
  static __device__ __forceinline__ void run(float* v, int lane_id) {
    if constexpr (S >= 1) {
      if constexpr (CNT > 1) {
        constexpr int HALF = CNT / 2;
        const bool up = (lane_id & S) != 0;
#pragma unroll
        for (int i = 0; i < HALF; ++i) {
          const float send = up ? v[i] : v[i + HALF];
          const float keep = up ? v[i + HALF] : v[i];
          v[i] = keep + __shfl_xor_sync(0xffffffffu, send, S * STRIDE);
        }
        LaneReduceScatter<STRIDE, HALF, S / 2>::run(v, lane_id);
      } else {
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], S * STRIDE);
        LaneReduceScatter<STRIDE, 1, S / 2>::run(v, lane_id);
      }
    }
  }
};
// Reduce-scatter of CNT per-lane values over LANES lanes spaced STRIDE apart (lane bits consumed MSB first).
// If CNT >= LANES each lane ends with CNT/LANES totals (slice index = its lane id among LANES); otherwise the
// value index is given by the top log2(CNT) lane bits and the remaining lanes hold replicas.
template <int LANES, int STRIDE, int CNT>
__device__ __forceinline__ void lane_reduce_scatter(float* v, int lane_id) {
  LaneReduceScatter<STRIDE, CNT, LANES / 2>::run(v, lane_id);
}

template <int NS>
__device__ __forceinline__ void load_states(const float* __restrict__ src, float* dst) {
  if constexpr (NS == 4) {
    const float4 v = *reinterpret_cast<const float4*>(src);
    dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
  } else if constexpr (NS == 2) {
    const float2 v = *reinterpret_cast<const float2*>(src);
    dst[0] = v.x; dst[1] = v.y;
  } else {
    dst[0] = src[0];
  }
}
template <int NS>
__device__ __forceinline__ void store_states(float* __restrict__ dst, const float* src) {
  if constexpr (NS == 4) *reinterpret_cast<float4*>(dst) = make_float4(src[0], src[1], src[2], src[3]);
  else if constexpr (NS == 2) *reinterpret_cast<float2*>(dst) = make_float2(src[0], src[1]);
  else dst[0] = src[0];
}

// STATE: the recompute of tile 0 starts from st.h0, the adjoint from st.dlast, and st.dh0 receives the adjoint of h0 (each
// pointer may be null)
template <int NS, int R, int RPT, bool DET>
__global__ void __launch_bounds__(kBwdThreads, RPT == 1 ? 4 : 3) scan_bwd_kernel(const ScanParams p, const __grid_constant__ TmaMaps maps) {
  constexpr bool STATE = false;
  const ScanState st{};
#include "scan_bwd_body.inc"
}
template <int NS, int R, int RPT, bool DET>
__global__ void __launch_bounds__(kBwdThreads, RPT == 1 ? 4 : 3) scan_bwd_state_kernel(const ScanParams p, const __grid_constant__ TmaMaps maps, const ScanState st) {
  constexpr bool STATE = true;
#include "scan_bwd_body.inc"
}

// dA[d][n] = sum_b part[b][d][n]; dD[d], dbias[d] likewise. One thread per (d, slot), batch-sequential: deterministic.
__global__ void scan_bwd_finalize_kernel(const float* __restrict__ part, float* __restrict__ dA, float* __restrict__ dD,
                                         float* __restrict__ dbias, int batch, int dim, int N, int A_ld, int accum) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dim * (N + 2)) return;
  const int d = i / (N + 2), s = i - d * (N + 2);
  float acc = 0.f;
  for (int b = 0; b < batch; ++b) acc += part[((int64_t)b * dim + d) * (N + 2) + s];
  if (s < N) dA[(int64_t)d * A_ld + s] = acc;
  else if (s == N) { if (dD && !accum) dD[d] = acc; }
  else if (dbias) dbias[d] = accum ? dbias[d] + acc : acc;
}

// Deterministic mode: dB / dC (slab 0) += slabs 1 ... slabs - 1, in slab order, over this pass' states [n0, n0 + N) of every
// (batch, group): rows of N * L floats, A_ld * L apart. HBM-bound; 128-bit accesses when L % 4 == 0.
template <bool VEC>
__global__ void __launch_bounds__(256) scan_bwd_fold_kernel(const ScanParams p, int slabs) {
  constexpr int V = VEC ? 4 : 1;
  const int which = blockIdx.y;
  float* __restrict__ out = which ? p.dC : p.dB;
  const float* __restrict__ src = which ? p.slabC : p.slabB;
  const int64_t row = (int64_t)p.N * p.L, pitch = (int64_t)p.A_ld * p.L, total = (int64_t)p.batch * p.G * row;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * V; i < total; i += (int64_t)gridDim.x * blockDim.x * V) {
    const int64_t o = i / row, off = o * pitch + (i - o * row);
    if constexpr (VEC) {
      float4 acc = *reinterpret_cast<const float4*>(out + off);
#pragma unroll 4
      for (int s = 1; s < slabs; ++s) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(src + (int64_t)(s - 1) * p.slab_stride + off));
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
      *reinterpret_cast<float4*>(out + off) = acc;
    } else {
      float acc = out[off];
#pragma unroll 4
      for (int s = 1; s < slabs; ++s) acc += __ldg(src + (int64_t)(s - 1) * p.slab_stride + off);
      out[off] = acc;
    }
  }
}

template <int NS, int R, int RPT, bool DET, bool STATE>
static cudaError_t launch_bwd(ScanParams p, const ScanState& st, cudaStream_t stream) {
  using S = BwdShape<NS, R, RPT>;
  const void* kern = STATE ? reinterpret_cast<const void*>(scan_bwd_state_kernel<NS, R, RPT, DET>)
                           : reinterpret_cast<const void*>(scan_bwd_kernel<NS, R, RPT, DET>);
  static PerDeviceOnce once;
  cudaError_t ea = func_attr_once(once, kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::smem_bytes);
  if (ea != cudaSuccess) return ea;
  TmaMaps maps;
  if (p.tma_ok && !(p.u_mod == 0 || p.u_mod % p.dpg == 0)) p.tma_ok = 0;
  if (p.tma_ok && !make_scan_maps(p, S::CH, S::NPB, true, &maps)) p.tma_ok = 0;
  if (!p.tma_ok) memset(&maps, 0, sizeof(maps));
  dim3 grid((p.dpg + S::CH - 1) / S::CH, p.G, p.batch);
  if constexpr (STATE) scan_bwd_state_kernel<NS, R, RPT, DET><<<grid, kBwdThreads, S::smem_bytes, stream>>>(p, maps, st);
  else scan_bwd_kernel<NS, R, RPT, DET><<<grid, kBwdThreads, S::smem_bytes, stream>>>(p, maps);
  return cudaGetLastError();
}

bool scan_bwd2_try(const ScanParams& p, const ScanState& st, cudaStream_t stream, cudaError_t* err, int* slabs);   // scan_bwd2.cu
int scan_bwd2_det_slabs(const ScanParams& p);

// kernel variant of this pass (0 ... 6), shared by the launcher and the slab count of deterministic mode
static int bwd_variant(const ScanParams& p) {
  const int N = p.N;
  if (N <= 1) return 0;
  if (N <= 2) return 1;
  if (N <= 4) return 2;
  if (N <= 8) return 3;
  if (N <= 16) {
    // Two rows per thread amortise the B/C loads and the dB/dC row reduction (best on big grids); one row per thread
    // needs fewer registers / shared memory (4 CTAs per SM instead of 3) and halves the CTA size, which wins when the
    // two-row grid would not fill ~2.5 waves (measured on vm_d96 / vm_d192 / vm_d384, B200).
    const int sms = sm_count_current_device();
    const long ctas2 = (long)((p.dpg + 31) / 32) * p.G * p.batch;
    return ctas2 * 2 < 5L * 3 * sms ? 4 : 5;
  }
  return 6;
}
static int bwd_rows_per_cta(int v) {
  constexpr int ch[7] = {BwdShape<1, 1, 1>::CH, BwdShape<2, 1, 1>::CH, BwdShape<2, 2, 1>::CH, BwdShape<2, 4, 2>::CH,
                         BwdShape<2, 8, 1>::CH, BwdShape<2, 8, 2>::CH, BwdShape<4, 8, 1>::CH};
  return ch[v];
}
template <bool DET, bool STATE>
static cudaError_t launch_variant(int v, const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  switch (v) {
    case 0: return launch_bwd<1, 1, 1, DET, STATE>(p, st, stream);
    case 1: return launch_bwd<2, 1, 1, DET, STATE>(p, st, stream);
    case 2: return launch_bwd<2, 2, 1, DET, STATE>(p, st, stream);
    case 3: return launch_bwd<2, 4, 2, DET, STATE>(p, st, stream);
    case 4: return launch_bwd<2, 8, 1, DET, STATE>(p, st, stream);
    case 5: return launch_bwd<2, 8, 2, DET, STATE>(p, st, stream);
    default: return launch_bwd<4, 8, 1, DET, STATE>(p, st, stream);
  }
}

int scan_bwd_det_slabs(const ScanParams& p) {
  const int ch = bwd_rows_per_cta(bwd_variant(p));
  return std::max(scan_bwd2_det_slabs(p), (p.dpg + ch - 1) / ch);
}

cudaError_t scan_bwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream, int* slabs) {
  cudaError_t e2;
  if (scan_bwd2_try(p, st, stream, &e2, slabs)) return e2;     // fast path: fp32 + TMA, 8 < N <= 16, contiguous traversal
  const int v = bwd_variant(p), ch = bwd_rows_per_cta(v);
  *slabs = p.det ? (p.dpg + ch - 1) / ch : 0;              // = gridDim.x of launch_bwd
  if (has_state(st)) return p.det ? launch_variant<true, true>(v, p, st, stream) : launch_variant<false, true>(v, p, st, stream);
  return p.det ? launch_variant<true, false>(v, p, st, stream) : launch_variant<false, false>(v, p, st, stream);
}

cudaError_t scan_bwd_fold(const ScanParams& p, int slabs, cudaStream_t stream) {
  const bool vec = (p.L & 3) == 0;
  const int64_t units = (int64_t)p.batch * p.G * p.N * p.L / (vec ? 4 : 1);
  const int64_t want = (units + 255) / 256, cap = 8L * sm_count_current_device();
  const dim3 grid((unsigned)(want < cap ? want : cap), 2);
  if (vec) scan_bwd_fold_kernel<true><<<grid, 256, 0, stream>>>(p, slabs);
  else scan_bwd_fold_kernel<false><<<grid, 256, 0, stream>>>(p, slabs);
  return cudaGetLastError();
}

cudaError_t scan_bwd_finalize(const ScanParams& p, float* dA, float* dD, float* dbias, cudaStream_t stream) {
  const int total = p.dim * (p.N + 2);
  scan_bwd_finalize_kernel<<<(total + 255) / 256, 256, 0, stream>>>(p.part, dA, dD, dbias, p.batch, p.dim, p.N, p.A_ld,
                                                                  p.accum);
  return cudaGetLastError();
}

}  // namespace ss2d
