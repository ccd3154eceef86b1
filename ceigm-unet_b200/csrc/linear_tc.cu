// Tensor-core projections of the SS2D module: out = A W^T (+ bias) with the epilogues the module needs.
//
// Replaces, per SS2D call (/root/reference/gm-unet/model/gm/ss2d.py):
//   in_proj  (:504) + chunk (:506) + NHWC -> NCHW copy of the x half (:510)  -> one launch, two output parts
//            (part 0 stored channel-major as (B, D, H, W) planes, part 1 row-major: the gate z, optionally SiLU'ed);
//   out_proj (:518)                                                           -> one launch, one row-major part.
// These are the genuine dense contractions around the scan: tall (M = B H W rows), skinny (K, N <= 256 per part) GEMMs that
// are bound by HBM traffic, not by math. The kernel is a persistent, warp-specialised sm_100a GEMM:
//   * W (one N tile x all of K) is loaded ONCE per CTA by TMA and stays resident in shared memory;
//   * A streams through a ring of 128-row x 128-byte K blocks (tiled TMA loads, 128-byte swizzle, out-of-range rows zero-filled);
//   * one elected thread issues tcgen05.mma (kind::tf32 for fp32 operands, kind::f16 for bf16 operands), accumulating a
//     128 x N fp32 tile in TENSOR MEMORY; two accumulator stages, so the epilogue of tile i overlaps the loads and MMAs of
//     tile i + 1. The tensor core TRUNCATES fp32 containers to TF32 (a bias of ~3e-4 per operand towards zero), so for fp32
//     operands two converter warps round W (once) and every A block (as it lands) to nearest TF32 in place, in shared
//     memory, between the TMA's `full` and the MMA's `ready` barrier: unbiased, <= 2^-12 relative per operand;
//   * eight epilogue warps read the accumulators back with tcgen05.ld (a thread owns one output row, a warp 32 columns at a
//     time) and store them in the part's layout: channel-major planes, where the 32 lanes of a warp write 32 consecutive
//     pixels of one channel (coalesced) — the permuted copy of ss2d.py:510 is just where the stores land — or row-major,
//     through a swizzled 4 KB shared-memory slab per warp so that every store instruction writes whole 128-byte row pieces.
// Handshakes are mbarriers only (TMA -> MMA: full / empty per ring stage; MMA -> epilogue: tmem_full / tmem_empty per
// accumulator stage, signalled by tcgen05.commit); there is no CTA-wide barrier after the prologue.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstring>

#include "tc_common.cuh"

namespace ss2d {

constexpr int TC_BM = 128;              // rows per tile = TMEM lanes
constexpr int TC_EPI_WARPS = 8;         // two per TMEM lane quarter, each taking half of the columns
constexpr int TC_CVT_WARPS = 4;
constexpr int TC_EPI_WARP0 = 2 + TC_CVT_WARPS;
constexpr int TC_THREADS = 32 * (TC_EPI_WARP0 + TC_EPI_WARPS);   // warp 0: TMA, warp 1: MMA, warps 2-5: TF32 rounding (warp 2 also owns TMEM), warps 6-13: epilogue
constexpr int TC_SLAB = 32 * 128;       // per epilogue warp: 32 rows x 128 bytes, staging of row-major stores
constexpr int TC_ABLOCK = TC_BM * 128;  // bytes of one A ring stage (128 rows x 128 bytes)
constexpr int TC_MAX_PARTS = 4;
constexpr int TC_MAX_STAGES = 8;

struct TcPart {
  void* out;
  int64_t ld;         // row-major parts: leading dimension (elements)
  int n0, n;          // columns [n0, n0 + n) of the product
  int planes_L;       // > 0: channel-major planes, out[((m / L) * n + c) * L + m % L]
  int act;            // 1: SiLU
};

struct TcParams {
  int M, N, K, kblocks, stages, esize, m_tiles, n_parts, out_dtype, acc_stride;
  const float* bias;
  TcPart part[TC_MAX_PARTS];
};

struct TcMaps { TMap a, w[TC_MAX_PARTS]; };

template <bool TF32>
__global__ void __launch_bounds__(TC_THREADS, 1) linear_tc_kernel(const TcParams p, const __grid_constant__ TcMaps maps) {
  extern __shared__ __align__(16) unsigned char tc_smem_raw[];
  const uint32_t sm = (smem_u32(tc_smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pi = blockIdx.x % p.n_parts;                 // this CTA's N tile (its W stays resident)
  const int mt0 = blockIdx.x / p.n_parts, mt_step = gridDim.x / p.n_parts;
  const TcPart part = p.part[pi];
  const uint32_t w_bytes = (uint32_t)p.kblocks * part.n * 128u;
  const uint32_t a_w = sm;                                // [kblocks][n rows x 128 bytes]
  const uint32_t a_ring = sm + ((w_bytes + 1023u) & ~1023u);      // [stages][128 rows x 128 bytes]
  const uint32_t a_bars = a_ring + (uint32_t)p.stages * TC_ABLOCK;
  const uint32_t b_full = a_bars, b_empty = a_bars + 8 * TC_MAX_STAGES, b_w = b_empty + 8 * TC_MAX_STAGES;
  const uint32_t b_tfull = b_w + 8, b_tempty = b_tfull + 16, a_tptr = b_tempty + 16;
  const uint32_t a_slabs = a_bars + 512;
  const uint32_t b_ready = a_tptr + 8, b_wready = b_ready + 8 * TC_MAX_STAGES;     // fp32 operands only
  uint32_t tmem_cols = 2u * p.acc_stride;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_full + 8 * s));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_empty + 8 * s));
    }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_w));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_wready), "r"(TC_CVT_WARPS));
    for (int s = 0; s < p.stages; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_ready + 8 * s), "r"(TC_CVT_WARPS));
    for (int a = 0; a < 2; ++a) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_tfull + 8 * a));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_tempty + 8 * a), "r"(TC_EPI_WARPS));      // one arrival per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 2) {     // TMEM: two accumulator stages of acc_stride columns (power of two, >= 32 in total)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(a_tptr), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(a_tptr));

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      tma_prefetch_desc(&maps.a); tma_prefetch_desc(&maps.w[pi]);
      const int kb_elems = 128 / p.esize;
      tc_mbar_expect(b_w, w_bytes);
      for (int kb = 0; kb < p.kblocks; ++kb) tma_load_2d(a_w + (uint32_t)kb * part.n * 128u, &maps.w[pi], kb * kb_elems, 0, b_w);
      int it = 0;
      for (int mt = mt0; mt < p.m_tiles; mt += mt_step) {
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int s = it % p.stages;
          tc_mbar_wait(b_empty + 8 * s, ((it / p.stages) & 1) ^ 1);      // passes immediately the first time round
          tc_mbar_expect(b_full + 8 * s, TC_ABLOCK);
          tma_load_2d(a_ring + (uint32_t)s * TC_ABLOCK, &maps.a, kb * kb_elems, mt * TC_BM, b_full + 8 * s);
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (lane == 0) {
      // instruction descriptor: D fp32; A, B tf32 (or bf16), both K-major; N >> 3 at bit 17, M >> 4 at bit 24
      const uint32_t fmt = TF32 ? 2u : 1u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(part.n >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      tc_mbar_wait(TF32 ? b_wready : b_w, 0);
      int it = 0, tile = 0;
      for (int mt = mt0; mt < p.m_tiles; mt += mt_step, ++tile) {
        const int acc = tile & 1;
        tc_mbar_wait(b_tempty + 8 * acc, ((tile >> 1) & 1) ^ 1);         // the epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * p.acc_stride;
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int s = it % p.stages;
          tc_mbar_wait((TF32 ? b_ready : b_full) + 8 * s, (it / p.stages) & 1);
          tc_fence_after();
          const uint32_t a_blk = a_ring + (uint32_t)s * TC_ABLOCK, w_blk = a_w + (uint32_t)kb * part.n * 128u;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)      // 4 MMAs of 32 bytes of K each per 128-byte block
            tc_mma<TF32>(d_tmem, tc_smem_desc(a_blk + kk * 32), tc_smem_desc(w_blk + kk * 32), idesc, (kb | kk) != 0);
          tc_commit(b_empty + 8 * s);          // the ring stage is free once these MMAs have read it
        }
        tc_commit(b_tfull + 8 * acc);          // accumulator complete
      }
    }
  } else if (warp < TC_EPI_WARP0) {
    // ================================ TF32 rounding (fp32 operands) ================================
    if (TF32) {
      constexpr uint32_t CT = 32u * TC_CVT_WARPS;
      const uint32_t ct = (warp - 2) * 32 + lane;
      // round to nearest TF32 (ties away from zero) on the bit pattern: add half an ulp of the 10-bit mantissa to the
      // magnitude, clear the 13 low bits (cvt.rna.tf32.f32 does the same but ptxas expands it to ~8 instructions per value)
      auto rna1 = [](float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); };
      auto rna = [&](float4 v) { return make_float4(rna1(v.x), rna1(v.y), rna1(v.z), rna1(v.w)); };
      auto round_block = [&](uint32_t base, uint32_t bytes) {      // bytes: multiple of 1024
        for (uint32_t o0 = 0; o0 < bytes; o0 += CT * 16u * 4u) {   // 4 pieces per thread in flight
          float4 v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) { const uint32_t o = o0 + (i * CT + ct) * 16u; if (o < bytes) v[i] = lds128(base + o); }
#pragma unroll
          for (int i = 0; i < 4; ++i) { const uint32_t o = o0 + (i * CT + ct) * 16u; if (o < bytes) sts128(base + o, rna(v[i])); }
        }
        fence_proxy_async();          // generic-proxy writes before the tensor core's async-proxy reads
        __syncwarp();
      };
      tc_mbar_wait(b_w, 0);
      round_block(a_w, w_bytes);
      if (lane == 0) tc_mbar_arrive(b_wready);
      int it = 0;
      for (int mt = mt0; mt < p.m_tiles; mt += mt_step) {
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int s = it % p.stages;
          tc_mbar_wait(b_full + 8 * s, (it / p.stages) & 1);
          round_block(a_ring + (uint32_t)s * TC_ABLOCK, TC_ABLOCK);
          if (lane == 0) tc_mbar_arrive(b_ready + 8 * s);
        }
      }
    }
  } else {
    // ================================ epilogue ================================
    const int ew = warp - TC_EPI_WARP0;
    const int lq = warp & 3;                    // TMEM lanes 32 lq ... 32 lq + 31: the quarter warp (id % 4) may read
    const int c_begin = (ew >> 2) * 32;         // the two warps of a lane quarter alternate over the 32-column chunks
    const uint32_t slab = a_slabs + (uint32_t)ew * TC_SLAB;
    int tile = 0;
    for (int mt = mt0; mt < p.m_tiles; mt += mt_step, ++tile) {
      const int acc = tile & 1;
      tc_mbar_wait(b_tfull + 8 * acc, (tile >> 1) & 1);
      tc_fence_after();
      const int m_warp = mt * TC_BM + lq * 32;
      const int gm = m_warp + lane;
      const bool live = gm < p.M;
      const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)acc * p.acc_stride;
      int64_t pbase = 0;
      if (part.planes_L > 0) {
        const int bb = gm / part.planes_L;
        pbase = (int64_t)bb * part.n * part.planes_L + (gm - bb * part.planes_L);
      }
      for (int c = c_begin; c < part.n; c += 64) {
        const int nc = min(32, part.n - c);       // 16 or 32 columns (n is a multiple of 16)
        float v[32];
        if (nc == 32) tc_ld32(taddr + c, v); else tc_ld16(taddr + c, v);
        if (p.bias) {
#pragma unroll
          for (int i = 0; i < 32; ++i) if (i < nc) v[i] += __ldg(p.bias + part.n0 + c + i);
        }
        if (part.act) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = tc_silu(v[i]);
        }
        if (part.planes_L > 0) {
          if (!live) continue;
          if (p.out_dtype == SS2D_F32) {
            float* o = static_cast<float*>(part.out) + pbase + (int64_t)c * part.planes_L;
#pragma unroll
            for (int i = 0; i < 32; ++i) if (i < nc) o[(int64_t)i * part.planes_L] = v[i];
          } else {
            __nv_bfloat16* o = static_cast<__nv_bfloat16*>(part.out) + pbase + (int64_t)c * part.planes_L;
#pragma unroll
            for (int i = 0; i < 32; ++i) if (i < nc) o[(int64_t)i * part.planes_L] = __float2bfloat16_rn(v[i]);
          }
          continue;
        }
        // row-major part: lane = row -> slab (16-byte pieces XOR-swizzled by the row) -> lane = (row, piece): every store
        // instruction writes whole 128-byte (fp32) / 64-byte (bf16) pieces of 4 / 8 rows
        __syncwarp();
        if (p.out_dtype == SS2D_F32) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            sts128(slab + lane * 128 + ((i ^ (lane & 7)) << 4), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
          __syncwarp();
          const int pieces = nc / 4;              // 16-byte pieces per row: 8 or 4
          const int rows_per = 32 / pieces;
          const int pc = lane % pieces, r0 = lane / pieces;
#pragma unroll 4
          for (int r = r0; r < 32; r += rows_per) {
            const float4 t = lds128(slab + r * 128 + ((pc ^ (r & 7)) << 4));
            if (m_warp + r < p.M)
              *reinterpret_cast<float4*>(static_cast<float*>(part.out) + (int64_t)(m_warp + r) * part.ld + c + pc * 4) = t;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(v[8 * i + 2 * j], v[8 * i + 2 * j + 1]);
            const uint4 u = *reinterpret_cast<uint4*>(h);
            sts128(slab + lane * 128 + ((i ^ (lane & 7)) << 4), make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w)));
          }
          __syncwarp();
          const int pieces = nc / 8;              // 16-byte pieces per row: 4 or 2
          const int rows_per = 32 / pieces;
          const int pc = lane % pieces, r0 = lane / pieces;
#pragma unroll 4
          for (int r = r0; r < 32; r += rows_per) {
            const float4 t = lds128(slab + r * 128 + ((pc ^ (r & 7)) << 4));
            if (m_warp + r < p.M)
              *reinterpret_cast<float4*>(static_cast<__nv_bfloat16*>(part.out) + (int64_t)(m_warp + r) * part.ld + c + pc * 8) = t;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) tc_mbar_arrive(b_tempty + 8 * acc);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

bool linear_tc_supported(int N_part, int K, int dtype) {
  const int esize = dtype == SS2D_F32 ? 4 : 2;
  if (dtype != SS2D_F32 && dtype != SS2D_BF16) return false;
  if (N_part < 16 || N_part > 256 || (N_part & 15) || K <= 0 || ((int64_t)K * esize & 15)) return false;
  const int kblocks = (K * esize + 127) / 128;
  const size_t w_bytes = ((size_t)kblocks * N_part * 128 + 1023) & ~(size_t)1023;
  return w_bytes + 2 * TC_ABLOCK + 2048 + TC_EPI_WARPS * TC_SLAB <= 227 * 1024;
}

// Returns an ss2d_status; *cerr receives the CUDA error behind SS2D_ERR_CUDA.
int linear_tc_launch(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, int M, int N, int K, int dtype,
                     int n_parts, const ss2d_linear_part* parts, cudaStream_t stream, cudaError_t* cerr) {
  *cerr = cudaSuccess;
  if (!A || !W || !parts) return SS2D_ERR_NULL_POINTER;
  if (M <= 0 || N <= 0 || K <= 0 || n_parts <= 0 || n_parts > TC_MAX_PARTS) return SS2D_ERR_BAD_SHAPE;
  if (dtype != SS2D_F32 && dtype != SS2D_BF16) return SS2D_ERR_BAD_DTYPE;
  if (lda < K || ldw < K) return SS2D_ERR_BAD_LAYOUT;            // rows of A / W would overlap
  const int esize = dtype == SS2D_F32 ? 4 : 2;
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K; p.esize = esize; p.out_dtype = dtype; p.bias = bias; p.n_parts = n_parts;
  p.kblocks = (K * esize + 127) / 128;
  p.m_tiles = (M + TC_BM - 1) / TC_BM;
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  int n0 = 0, nmax = 0;
  for (int i = 0; i < n_parts; ++i) {
    const ss2d_linear_part& q = parts[i];
    if (!q.out) return SS2D_ERR_NULL_POINTER;
    if (!linear_tc_supported(q.n_cols, K, dtype)) return SS2D_ERR_UNSUPPORTED;
    if (q.planes_L < 0 || (q.planes_L > 0 && M % q.planes_L != 0)) return SS2D_ERR_BAD_SHAPE;
    if (q.planes_L == 0 && q.ld < q.n_cols) return SS2D_ERR_BAD_LAYOUT;     // output rows would overlap
    if (q.planes_L == 0 && ((q.ld * esize) & 15 || (reinterpret_cast<uintptr_t>(q.out) & 15))) return SS2D_ERR_ALIGNMENT;
    p.part[i].out = q.out; p.part[i].ld = q.ld; p.part[i].n0 = n0; p.part[i].n = q.n_cols;
    p.part[i].planes_L = q.planes_L; p.part[i].act = q.act;
    n0 += q.n_cols;
    nmax = q.n_cols > nmax ? q.n_cols : nmax;
  }
  if (n0 != N) return SS2D_ERR_BAD_SHAPE;
  // tensor maps only once every argument has been validated: their creation is the one check whose outcome depends on the driver
  for (int i = 0; i < n_parts; ++i) {
    const TcPart& q = p.part[i];
    if (!tc_make_map(&maps.w[i], static_cast<const char*>(W) + (size_t)q.n0 * ldw * esize, esize, K, q.n, ldw, q.n))
      return SS2D_ERR_ALIGNMENT;
  }
  if (!tc_make_map(&maps.a, A, esize, K, M, lda, TC_BM)) return SS2D_ERR_ALIGNMENT;
  p.acc_stride = nmax <= 16 ? 16 : nmax <= 32 ? 32 : nmax <= 64 ? 64 : nmax <= 128 ? 128 : 256;
  const size_t w_bytes = ((size_t)p.kblocks * nmax * 128 + 1023) & ~(size_t)1023;
  const size_t avail = 227 * 1024 - 2048 - w_bytes - TC_EPI_WARPS * TC_SLAB;
  int stages = (int)(avail / TC_ABLOCK);
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (stages < 2) return SS2D_ERR_UNSUPPORTED;
  p.stages = stages;
  const size_t smem = w_bytes + (size_t)stages * TC_ABLOCK + 1024 /* alignment slack */ + 512 /* barriers */ + TC_EPI_WARPS * TC_SLAB;
  auto kern = dtype == SS2D_F32 ? linear_tc_kernel<true> : linear_tc_kernel<false>;
  static PerDeviceOnce once32, once16;
  cudaError_t e = func_attr_once(dtype == SS2D_F32 ? once32 : once16, reinterpret_cast<const void*>(kern),
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) { *cerr = e; return SS2D_ERR_CUDA; }
  const int sms = sm_count_current_device();
  int per_part = (sms + n_parts - 1) / n_parts;
  if (per_part > p.m_tiles) per_part = p.m_tiles;
  kern<<<per_part * n_parts, TC_THREADS, smem, stream>>>(p, maps);
  *cerr = cudaGetLastError();
  return *cerr == cudaSuccess ? SS2D_OK : SS2D_ERR_CUDA;
}

}  // namespace ss2d
