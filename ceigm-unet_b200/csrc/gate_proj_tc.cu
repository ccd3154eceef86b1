// The SS2D epilogue with the output projection folded in (north-star property 5): merge over the K directions +
// un-transposition + (B, D, L) -> (B, L, D) + out_norm LayerNorm(D) + SiLU(z) gate + out_proj, ONE kernel.
//
// Replaces CrossMerge, the transpose copy, out_norm, act(z), `y * z` and out_proj of
// /root/reference/gm-unet/model/gm/ss2d.py:486-498, 506-508, 515-518 (the two-kernel version is csrc/epilogue.cu's
// out_gate_fwd followed by linear_tc). The gated tensor never has to reach HBM: the producer warps build it directly in shared
// memory in the layout the tensor core reads (K-major, 128-byte swizzle), a 128-pixel x D tile at a time, and one thread issues
// tcgen05.mma against the resident out_proj weight; the accumulators live in tensor memory and leave through the epilogue warps
// as whole row pieces. For the backward of a training step the gated tensor can be written out as well (g_out != NULL).
//
// Warp roles (512 threads): warp 0 loads W once by TMA; warp 1 issues the MMAs; warp 2 owns the TMEM allocation; warps 4-11
// (256 threads) PRODUCE the A tile; warps 12-15 are the epilogue. A tile is an 8 (h) x 16 (w) pixel patch, so that planes in
// natural pixel order are read in 64-byte runs and planes in transposed order (column-major directions run as row-major scans of
// the transposed image, DESIGN.md §2) in 32-byte runs. Per tile the producers
//   A. sum the K planes: warp 0 streams them as TMA boxes of 16 channels x 8 x 16 pixels (4-D tensor maps over the natural and
//      over the transposed images: both orientations arrive as dense tiles, zero-filled outside the image) through a ring of
//      8 KB slots; a producer thread owns (pixel, 2 channel quads) of a box and accumulates it into the fp32 tile, which
//      already has the tensor core's layout (pixel m = row, channels = K; the pixel numbering m(h, w) = 16 h + ((w + h) & 15)
//      makes the 16-byte stores of a quarter warp hit 8 distinct swizzle slots) — no thread ever waits on a global load;
//   C + D. a warp then owns 16 pixel rows with its lanes along the channels: two-pass LayerNorm statistics by butterflies,
//      normalise, affine, multiply by SiLU(z) (z and the optional G rows are read / written as whole contiguous rows), round
//      (TF32: in place; bf16: into a second, bf16 tile).
// Handshakes: `ready` (producers -> MMA), `afree` (tcgen05.commit -> producers: the tile may be overwritten), tmem_full /
// tmem_empty per accumulator stage (MMA <-> epilogue; the producers also wait for tmem_empty before they reuse the pixel table
// of that stage). The only CTA-wide barrier is in the prologue; the producers synchronise among themselves with a named barrier.
#include <cstring>

#include "tc_common.cuh"

namespace ss2d {

constexpr int GP_THREADS = 512;
constexpr int GP_PROD0 = 4, GP_PROD_WARPS = 8, GP_EPI0 = 12, GP_EPI_WARPS = 4;
constexpr int GP_PT = 32 * GP_PROD_WARPS;     // producer threads
constexpr int GP_TILE = 128, GP_TH = 8, GP_TW = 16;
constexpr int GP_BLOCK = GP_TILE * 128;       // one K block of an operand tile: 128 rows x 128 bytes
constexpr int GP_CB = 16;                     // channels per plane box
constexpr int GP_SLOT = GP_CB * GP_TILE * 4;  // 8 KB
constexpr int GP_MAX_SLOTS = 16;
struct GpMaps { TMap w, nat, tr; };

struct GpParams {
  const float* ys;            // (batch, K, D, L) fp32
  int K;
  unsigned tmask;             // bit k: plane k is in the pixel order of the transposed image
  int64_t ys_bs;
  const float* lnw;
  const float* lnb;
  float eps;
  const void* z;              // rows (batch * L) x D (+ column offset folded into the pointer), dtype of the operands
  int64_t z_rs;
  int z_act;
  void* out;                  // (batch * L, C) rows
  int64_t out_rs;
  void* g_out;                // optional (batch * L, D) rows: the gated tensor, for the backward
  int64_t g_rs;
  float* mean_rstd;           // optional (batch * L, 2)
  const float* bias;          // optional (C)
  int batch, D, L, H, W, C;
  int tiles_w, tiles_per_batch, n_tiles;
  int kb32;                   // D / 32: K blocks of the fp32 tile
  int kblocks;                // K blocks of the MMA operands (D * esize / 128)
  int acc_stride;
  int slots;                  // plane-box ring depth
};

__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void tma_load_4d32(uint32_t dst, const void* tmap, int c0, int c1, int c2, int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// 4-D fp32 tensor map with an explicit box, no swizzle, zero fill: the K direction planes as (inner, outer, channel, batch x K)
static bool gp_make_map4(TMap* out, const void* base, const long long* dims, const long long* strides_elems, const int* box) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  cuuint64_t gdim[4], gstr[3];
  cuuint32_t bx[4], estr[4] = {1, 1, 1, 1};
  for (int i = 0; i < 4; ++i) {
    gdim[i] = (cuuint64_t)dims[i];
    bx[i] = (cuuint32_t)box[i];
    if (i > 0) {
      gstr[i - 1] = (cuuint64_t)strides_elems[i] * 4;
      if (gstr[i - 1] == 0 || (gstr[i - 1] & 15)) return false;
    }
  }
  if (reinterpret_cast<uintptr_t>(base) & 15) return false;
  CUresult r = fn(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), gdim, gstr, bx, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}
__device__ __forceinline__ void gp_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(GP_PT) : "memory"); }
// byte offset of channels [4 cq, 4 cq + 4) of pixel row m in the fp32 tile (K-major, 128-byte swizzle)
__device__ __forceinline__ uint32_t gp_y_off(int m, int cq) { return (uint32_t)(cq >> 3) * GP_BLOCK + m * 128 + (((cq & 7) ^ (m & 7)) << 4); }
__device__ __forceinline__ float gp_silu(float x) { return __fdividef(x, 1.f + ex2f(-x * kLog2e)); }
__device__ __forceinline__ float gp_rna(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }

template <bool TF32, bool HAS_Z, bool HAS_G>
__global__ void __launch_bounds__(GP_THREADS, 1) gate_proj_tc_kernel(const GpParams p, const __grid_constant__ GpMaps maps) {
  extern __shared__ __align__(16) unsigned char gp_smem_raw[];
  const uint32_t sm = (smem_u32(gp_smem_raw) + 1023u) & ~1023u;
  unsigned char* smp = gp_smem_raw + (sm - smem_u32(gp_smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t w_bytes = (uint32_t)p.kblocks * p.C * 128u;
  const uint32_t a_w = sm;
  const uint32_t a_stage = sm;                                        // plane-box ring: ALIASES the weight (see the TMA warp)
  const uint32_t a_y = sm + (uint32_t)p.slots * GP_SLOT;               // fp32 tile: kb32 blocks
  const uint32_t a_a16 = a_y + (uint32_t)p.kb32 * GP_BLOCK;           // bf16 operand tile (bf16 variant only)
  const uint32_t a_slabs = a_a16 + ((TF32 || p.C == 0) ? 0u : (uint32_t)p.kblocks * GP_BLOCK);
  const uint32_t a_misc = a_slabs + GP_EPI_WARPS * 4096u;
  // misc: barriers + tmem pointer (128 B) | pixel tables 2 x 128 ints | statistics partials 2 x 256 floats
  const uint32_t b_w = a_misc, b_ready = a_misc + 8, b_afree = a_misc + 16, b_tfull = a_misc + 24, b_tempty = a_misc + 40, a_tptr = a_misc + 56;
  const uint32_t b_wready = a_misc + 64;                                // TF32: W rounded in place by the producers
  const uint32_t b_full = a_misc + 72, b_empty = b_full + 8 * GP_MAX_SLOTS;    // plane-box ring (ends at + 328)
  int* s_pix = reinterpret_cast<int*>(smp + (a_misc - sm) + 384);       // [2][128]
  const uint32_t tmem_cols = 2u * p.acc_stride;

  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_w));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_ready), "r"(GP_PROD_WARPS));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_afree));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_wready), "r"(GP_PROD_WARPS));
    for (int s2 = 0; s2 < p.slots; ++s2) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_full + 8 * s2));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_empty + 8 * s2), "r"(GP_PROD_WARPS));
    }
    for (int a = 0; a < 2; ++a) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b_tfull + 8 * a));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_tempty + 8 * a), "r"(GP_EPI_WARPS));
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(a_tptr), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(a_tptr));

  const int D = p.D, L = p.L, H = p.H, W = p.W;
  const bool proj = p.C > 0;          // C == 0: epilogue only (merge + LayerNorm + gate -> G rows), no weight, no MMA

  if (warp == 0) {
    // ================================ TMA: per tile the plane boxes, then the weight ================================
    // The ring and the weight share one region of shared memory: the planes of a tile stream through it while the producers
    // accumulate them (13 slots = 104 KB in flight next to a 72 KB weight), and once the last box has been consumed the weight
    // is loaded over it (72 KB from L2, hidden behind the statistics / gate passes) for this tile's MMAs; the next tile's boxes
    // wait for those MMAs (`afree`).
    if (lane == 0) {
      if (proj) tma_prefetch_desc(&maps.w);
      tma_prefetch_desc(&maps.nat); tma_prefetch_desc(&maps.tr);
      const int kb_elems = TF32 ? 32 : 64;
      int rit = 0, it = 0, s2 = 0, ph = 0;
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++it) {
        const int b = t / p.tiles_per_batch, tib = t - b * p.tiles_per_batch;
        const int th = tib / p.tiles_w, tw = tib - th * p.tiles_w;
        const int h0 = th * GP_TH, w0 = tw * GP_TW;
        if (proj) tc_mbar_wait(b_afree, (it & 1) ^ 1);            // MMAs of tile it - 1 have read the weight
        for (int cb = 0; cb < D / GP_CB; ++cb) {
          for (int k = 0; k < p.K; ++k, ++rit) {
            tc_mbar_wait(b_empty + 8 * s2, ph ^ 1);
            tc_mbar_expect(b_full + 8 * s2, GP_SLOT);
            if ((p.tmask >> k) & 1u) tma_load_4d32(a_stage + (uint32_t)s2 * GP_SLOT, &maps.tr, h0, w0, cb * GP_CB, b * p.K + k, b_full + 8 * s2);
            else tma_load_4d32(a_stage + (uint32_t)s2 * GP_SLOT, &maps.nat, w0, h0, cb * GP_CB, b * p.K + k, b_full + 8 * s2);
            if (++s2 == p.slots) { s2 = 0; ph ^= 1; }
          }
        }
        if (!proj) continue;                                      // epilogue only: the boxes of the next tile follow at once
        for (int u = rit > p.slots ? rit - p.slots : 0; u < rit; ++u)       // every box of this tile has been consumed
          tc_mbar_wait(b_empty + 8 * (u % p.slots), (u / p.slots) & 1);
        tc_mbar_expect(b_w, w_bytes);
        for (int kb = 0; kb < p.kblocks; ++kb) tma_load_2d(a_w + (uint32_t)kb * p.C * 128u, &maps.w, kb * kb_elems, 0, b_w);
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (lane == 0 && proj) {
      const uint32_t fmt = TF32 ? 2u : 1u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(p.C >> 3) << 17) | ((uint32_t)(GP_TILE >> 4) << 24);
      const uint32_t a_op = TF32 ? a_y : a_a16;
      int it = 0;
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++it) {
        const int acc = it & 1;
        tc_mbar_wait(b_tempty + 8 * acc, ((it >> 1) & 1) ^ 1);      // the epilogue has drained this accumulator stage
        tc_mbar_wait(b_ready, it & 1);                               // the producers have finished the operand tile
        tc_mbar_wait(TF32 ? b_wready : b_w, it & 1);                 // this tile's copy of the weight is in place (and rounded)
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * p.acc_stride;
        for (int kb = 0; kb < p.kblocks; ++kb) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            tc_mma<TF32>(d_tmem, tc_smem_desc(a_op + (uint32_t)kb * GP_BLOCK + kk * 32), tc_smem_desc(a_w + (uint32_t)kb * p.C * 128u + kk * 32),
                         idesc, (kb | kk) != 0);
        }
        tc_commit(b_afree);              // the operand tile may be overwritten once these MMAs have read it
        tc_commit(b_tfull + 8 * acc);    // accumulator complete
      }
    }
  } else if (warp >= GP_PROD0 && warp < GP_EPI0) {
    // ================================ producers ================================
    const int pt = threadIdx.x - 32 * GP_PROD0, pw = pt >> 5;
    int s2 = 0, ph = 0;          // ring slot and phase, carried across tiles (no division in the box loop)
    int it = 0;
    for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++it) {
      const int b = t / p.tiles_per_batch, tib = t - b * p.tiles_per_batch;
      const int th = tib / p.tiles_w, tw = tib - th * p.tiles_w;
      const int h0 = th * GP_TH, w0 = tw * GP_TW;
      int* pix = s_pix + (it & 1) * GP_TILE;
      if (proj) {
        tc_mbar_wait(b_tempty + 8 * (it & 1), ((it >> 1) & 1) ^ 1);  // epilogue of tile it - 2 done: its pixel table is free
        tc_mbar_wait(b_afree, (it & 1) ^ 1);                         // MMAs of tile it - 1 have read the operand tile
      } else {
        gp_bar_sync();                                               // every producer has left the previous tile
      }
      if (pt < GP_TILE) {
        const int hh = pt >> 4, ww = ((pt & 15) - hh) & 15;
        const int h = h0 + hh, w = w0 + ww;
        pix[pt] = (h < H && w < W) ? h * W + w : -1;
      }
      // ---- A: accumulate the K planes from the TMA ring. natural box [c][hh][ww], transposed box [c][ww][hh] ----
      {
        const int m_hh = (pt & (GP_TILE - 1)) >> 4, m_ww = pt & 15;
        const int mrow = m_hh * 16 + ((m_ww + m_hh) & 15);
        const int qb = (pt >> 7) * 2;                       // this thread's two channel quads of a 16-channel box
        const uint32_t off_n = (uint32_t)(m_hh * 16 + m_ww) * 4u, off_t = (uint32_t)(m_ww * 8 + m_hh) * 4u;
        for (int cb = 0; cb < D / GP_CB; ++cb) {
          for (int k = 0; k < p.K; ++k) {
            tc_mbar_wait(b_full + 8 * s2, ph);
            const uint32_t st = a_stage + (uint32_t)s2 * GP_SLOT + (((p.tmask >> k) & 1u) ? off_t : off_n);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const int q = qb + j;
              float4 v = make_float4(lds32(st + (4 * q) * 512), lds32(st + (4 * q + 1) * 512), lds32(st + (4 * q + 2) * 512), lds32(st + (4 * q + 3) * 512));
              const uint32_t o = a_y + gp_y_off(mrow, cb * 4 + q);
              if (k > 0) { const float4 t4 = lds128(o); v.x += t4.x; v.y += t4.y; v.z += t4.z; v.w += t4.w; }
              sts128(o, v);
            }
            __syncwarp();
            if (lane == 0) tc_mbar_arrive(b_empty + 8 * s2);
            if (++s2 == p.slots) { s2 = 0; ph ^= 1; }
          }
        }
      }
      gp_bar_sync();
      // ---- C + D: a warp owns 16 pixel rows; its lanes run along the channels (quads lane and lane + 32), so the gate z and the
      //      optional G rows are read / written as whole contiguous rows, the LayerNorm statistics are two butterfly sums, and
      //      nothing crosses warps. RU rows in flight per step: their z quads are requested before the statistics are computed.
      constexpr int RU = 4;
      const int nq = D / 4;
      const bool has2 = lane + 32 < nq;                   // D <= 256: at most two quads per lane
      for (int r0 = 0; r0 < 16; r0 += RU) {
        float4 y0[RU], y1[RU], z0[RU], z1[RU];
        int lrow[RU];
#pragma unroll
        for (int u = 0; u < RU; ++u) {
          const int mrow = pw * 16 + r0 + u;
          lrow[u] = pix[mrow];
          y0[u] = lane < nq ? lds128(a_y + gp_y_off(mrow, lane)) : make_float4(0.f, 0.f, 0.f, 0.f);
          y1[u] = has2 ? lds128(a_y + gp_y_off(mrow, lane + 32)) : make_float4(0.f, 0.f, 0.f, 0.f);
          z0[u] = z1[u] = make_float4(1.f, 1.f, 1.f, 1.f);
          if (HAS_Z && lrow[u] >= 0) {
            const int64_t row = (int64_t)b * L + lrow[u];
            if (TF32) {
              const float4* zr = reinterpret_cast<const float4*>(static_cast<const float*>(p.z) + row * p.z_rs);
              if (lane < nq) z0[u] = __ldg(zr + lane);
              if (has2) z1[u] = __ldg(zr + lane + 32);
            } else {
              const uint2* zr = reinterpret_cast<const uint2*>(static_cast<const __nv_bfloat16*>(p.z) + row * p.z_rs);
              // keep the raw 16-bit pairs in the registers (converted where they are used): converting here would wait for
              // each load before the next one is issued
              if (lane < nq) { const uint2 raw = __ldg(zr + lane); z0[u].x = __uint_as_float(raw.x); z0[u].y = __uint_as_float(raw.y); }
              if (has2) { const uint2 raw = __ldg(zr + lane + 32); z1[u].x = __uint_as_float(raw.x); z1[u].y = __uint_as_float(raw.y); }
            }
          }
        }
#pragma unroll
        for (int u = 0; u < RU; ++u) {
          const int mrow = pw * 16 + r0 + u;
          const int l = lrow[u];
          float sm1 = ((y0[u].x + y0[u].y) + (y0[u].z + y0[u].w)) + ((y1[u].x + y1[u].y) + (y1[u].z + y1[u].w));
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) sm1 += __shfl_xor_sync(0xffffffffu, sm1, o);
          const float mean = sm1 / D;
          float q = 0.f;
          if (lane < nq) { const float a0 = y0[u].x - mean, a1 = y0[u].y - mean, a2 = y0[u].z - mean, a3 = y0[u].w - mean; q = fmaf(a0, a0, fmaf(a1, a1, fmaf(a2, a2, a3 * a3))); }
          if (has2) { const float a0 = y1[u].x - mean, a1 = y1[u].y - mean, a2 = y1[u].z - mean, a3 = y1[u].w - mean; q += fmaf(a0, a0, fmaf(a1, a1, fmaf(a2, a2, a3 * a3))); }
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
          const float rstd = rsqrtf(q / D + p.eps);
          const int64_t row = (int64_t)b * L + (l >= 0 ? l : 0);
          if (lane == 0 && l >= 0 && p.mean_rstd) { p.mean_rstd[row * 2] = mean; p.mean_rstd[row * 2 + 1] = rstd; }
#pragma unroll
          for (int hq = 0; hq < 2; ++hq) {
            const int cq = lane + 32 * hq;
            if (hq == 0 ? lane >= nq : !has2) continue;
            const float4 v = hq == 0 ? y0[u] : y1[u];
            float4 zz = hq == 0 ? z0[u] : z1[u];
            if (!TF32 && HAS_Z && l >= 0) {
              const uint32_t r0 = __float_as_uint(zz.x), r1 = __float_as_uint(zz.y);
              const float2 a2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r0));
              const float2 c2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r1));
              zz = make_float4(a2.x, a2.y, c2.x, c2.y);
            }
            float g[4] = {(v.x - mean) * rstd, (v.y - mean) * rstd, (v.z - mean) * rstd, (v.w - mean) * rstd};
            if (p.lnw) {
              const float4 wv = __ldg(reinterpret_cast<const float4*>(p.lnw) + cq);
              const float4 bv = p.lnb ? __ldg(reinterpret_cast<const float4*>(p.lnb) + cq) : make_float4(0.f, 0.f, 0.f, 0.f);
              g[0] = fmaf(g[0], wv.x, bv.x); g[1] = fmaf(g[1], wv.y, bv.y); g[2] = fmaf(g[2], wv.z, bv.z); g[3] = fmaf(g[3], wv.w, bv.w);
            }
            if (l < 0) { g[0] = g[1] = g[2] = g[3] = 0.f; }
            if (HAS_Z && l >= 0) {
              g[0] *= p.z_act ? gp_silu(zz.x) : zz.x; g[1] *= p.z_act ? gp_silu(zz.y) : zz.y;
              g[2] *= p.z_act ? gp_silu(zz.z) : zz.z; g[3] *= p.z_act ? gp_silu(zz.w) : zz.w;
            }
            if (TF32) {
              if (HAS_G && l >= 0)
                *(reinterpret_cast<float4*>(static_cast<float*>(p.g_out) + row * p.g_rs) + cq) = make_float4(g[0], g[1], g[2], g[3]);
              if (proj) sts128(a_y + gp_y_off(mrow, cq), make_float4(gp_rna(g[0]), gp_rna(g[1]), gp_rna(g[2]), gp_rna(g[3])));
            } else {
              const __nv_bfloat162 lo = __floats2bfloat162_rn(g[0], g[1]), hi = __floats2bfloat162_rn(g[2], g[3]);
              uint2 pk;
              pk.x = *reinterpret_cast<const uint32_t*>(&lo);
              pk.y = *reinterpret_cast<const uint32_t*>(&hi);
              if (HAS_G && l >= 0) *(reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(p.g_out) + row * p.g_rs) + cq) = pk;
              // bf16 operand tile: 64 channels per 128-byte row, 16-byte chunk = 8 channels = two quads
              const uint32_t o2 = (uint32_t)(cq >> 4) * GP_BLOCK + mrow * 128 + ((((cq >> 1) & 7) ^ (mrow & 7)) << 4) + ((cq & 1) << 3);
              if (proj) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a_a16 + o2), "r"(pk.x), "r"(pk.y) : "memory");
            }
          }
        }
      }
      if (!proj) continue;
      if (TF32) {      // the tensor core truncates fp32 containers: round this tile's copy of the weight to nearest TF32
        tc_mbar_wait(b_w, it & 1);
        for (uint32_t o = (uint32_t)pt * 16u; o < w_bytes; o += GP_PT * 16u) {
          const float4 v = lds128(a_w + o);
          sts128(a_w + o, make_float4(gp_rna(v.x), gp_rna(v.y), gp_rna(v.z), gp_rna(v.w)));
        }
      }
      fence_proxy_async();           // generic-proxy writes before the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) { tc_mbar_arrive(b_ready); if (TF32) tc_mbar_arrive(b_wready); }
    }
  } else if (warp >= GP_EPI0 && proj) {
    // ================================ epilogue ================================
    const int lq = warp & 3;                    // TMEM lanes 32 lq ... (warp id % 4)
    const uint32_t slab = a_slabs + (uint32_t)(warp - GP_EPI0) * 4096u;
    int it = 0;
    for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      const int b = t / p.tiles_per_batch;
      const int* pix = s_pix + (it & 1) * GP_TILE;
      tc_mbar_wait(b_tfull + 8 * acc, (it >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)acc * p.acc_stride;
      for (int c = 0; c < p.C; c += 32) {
        const int nc = min(32, p.C - c);
        float v[32];
        if (nc == 32) tc_ld32(taddr + c, v); else tc_ld16(taddr + c, v);
        if (p.bias) {
#pragma unroll
          for (int i = 0; i < 32; ++i) if (i < nc) v[i] += __ldg(p.bias + c + i);
        }
        __syncwarp();
        if (TF32) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            sts128(slab + lane * 128 + ((i ^ (lane & 7)) << 4), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
          __syncwarp();
          const int pieces = nc / 4, rows_per = 32 / pieces, pc = lane % pieces;
          for (int r = lane / pieces; r < 32; r += rows_per) {
            const int l = pix[lq * 32 + r];
            if (l < 0) continue;
            const float4 tv = lds128(slab + r * 128 + ((pc ^ (r & 7)) << 4));
            *reinterpret_cast<float4*>(static_cast<float*>(p.out) + ((int64_t)b * L + l) * p.out_rs + c + pc * 4) = tv;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 hv[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) hv[j] = __floats2bfloat162_rn(v[8 * i + 2 * j], v[8 * i + 2 * j + 1]);
            const uint4 u = *reinterpret_cast<uint4*>(hv);
            sts128(slab + lane * 128 + ((i ^ (lane & 7)) << 4), make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w)));
          }
          __syncwarp();
          const int pieces = nc / 8, rows_per = 32 / pieces, pc = lane % pieces;
          for (int r = lane / pieces; r < 32; r += rows_per) {
            const int l = pix[lq * 32 + r];
            if (l < 0) continue;
            const float4 tv = lds128(slab + r * 128 + ((pc ^ (r & 7)) << 4));
            *reinterpret_cast<float4*>(static_cast<__nv_bfloat16*>(p.out) + ((int64_t)b * L + l) * p.out_rs + c + pc * 8) = tv;
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

// ring slots: the weight's region plus 32 KB (fp32) / 16 KB (bf16) of extra staging
static int gp_slots(int D, int C, int esize) {
  if (C == 0) return 12;
  const size_t w = ((size_t)(D * esize / 128) * C * 128 + 1023) & ~(size_t)1023;
  int s = (int)((w + (esize == 4 ? 32768 : 16384)) / GP_SLOT);
  return s > GP_MAX_SLOTS ? GP_MAX_SLOTS : s;
}
static size_t gp_smem_bytes(int D, int C, int esize) {
  const int kblocks = D * esize / 128;
  const size_t w = ((size_t)kblocks * C * 128 + 1023) & ~(size_t)1023;
  const size_t y = (size_t)(D / 32) * GP_BLOCK;
  const size_t a16 = (esize == 2 && C > 0) ? (size_t)kblocks * GP_BLOCK : 0;
  size_t ring = (size_t)gp_slots(D, C, esize) * GP_SLOT;
  if (ring < w) ring = w;
  return ring + y + a16 + GP_EPI_WARPS * 4096 + 384 + 2 * GP_TILE * 4 + 2 * GP_PT * 4 + 1024 /* alignment slack */;
}

bool gate_proj_tc_supported(int D, int C, int K, int dtype) {
  if (dtype != SS2D_F32 && dtype != SS2D_BF16) return false;
  if (D <= 0 || (D % 64) != 0 || D > 256 || K < 1 || K > SS2D_MAX_GROUP_DIRS) return false;
  if (C != 0 && (C < 16 || C > 256 || (C & 15))) return false;        // C == 0: epilogue only
  return gp_smem_bytes(D, C, dtype == SS2D_F32 ? 4 : 2) <= 227 * 1024;
}

// Returns an ss2d_status; *cerr receives the CUDA error behind SS2D_ERR_CUDA.
int gate_proj_tc_launch(const float* ys, int K, unsigned tmask, const float* lnw, const float* lnb, float eps, const void* z,
                        int64_t z_rs, int z_act, const void* W, int64_t ldw, const float* bias, void* out, int64_t out_rs,
                        void* g_out, int64_t g_rs, float* mean_rstd, int batch, int D, int L, int H, int Wd, int C, int dtype,
                        cudaStream_t stream, cudaError_t* cerr) {
  *cerr = cudaSuccess;
  if (!ys || (C > 0 && (!W || !out)) || (C == 0 && !g_out)) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || L <= 0 || H <= 0 || Wd <= 0 || (int64_t)H * Wd != L) return SS2D_ERR_BAD_SHAPE;
  if (!gate_proj_tc_supported(D, C, K, dtype) || (lnb && !lnw)) return SS2D_ERR_UNSUPPORTED;
  if ((H & 3) || (Wd & 3)) return SS2D_ERR_UNSUPPORTED;          // the plane boxes' tensor maps need 16-byte row strides
  if ((C > 0 && out_rs < C) || (z && z_rs < D) || (g_out && g_rs < D)) return SS2D_ERR_BAD_LAYOUT;   // overlapping rows
  const int esize = dtype == SS2D_F32 ? 4 : 2;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if ((C > 0 && (!al16(out) || ((out_rs * esize) & 15))) || (z && (!al16(z) || ((z_rs * esize) & 15))) || (g_out && (!al16(g_out) || ((g_rs * esize) & 15))) ||
      (lnw && !al16(lnw)) || (lnb && !al16(lnb)))
    return SS2D_ERR_ALIGNMENT;
  GpParams p;
  memset(&p, 0, sizeof(p));
  p.ys = ys; p.K = K; p.tmask = tmask; p.ys_bs = (int64_t)K * D * L; p.lnw = lnw; p.lnb = lnb; p.eps = eps;
  p.z = z; p.z_rs = z_rs; p.z_act = z_act; p.out = out; p.out_rs = out_rs; p.g_out = g_out; p.g_rs = g_rs; p.mean_rstd = mean_rstd;
  p.bias = bias; p.batch = batch; p.D = D; p.L = L; p.H = H; p.W = Wd; p.C = C;
  p.tiles_w = (Wd + GP_TW - 1) / GP_TW;
  p.tiles_per_batch = p.tiles_w * ((H + GP_TH - 1) / GP_TH);
  p.n_tiles = batch * p.tiles_per_batch;
  p.kb32 = D / 32;
  p.kblocks = D * esize / 128;
  p.acc_stride = C <= 16 ? 16 : C <= 32 ? 32 : C <= 64 ? 64 : C <= 128 ? 128 : 256;
  p.slots = gp_slots(D, C, esize);
  GpMaps maps;
  memset(&maps, 0, sizeof(maps));
  if (C > 0 && !tc_make_map(&maps.w, W, esize, D, C, ldw, C)) return SS2D_ERR_ALIGNMENT;
  {   // planes as images: natural (W inner) and transposed (H inner); box = 16 x 8 (resp. 8 x 16) pixels x 16 channels
    const long long bk = (long long)batch * K;
    const long long dn[4] = {Wd, H, D, bk}, sn[4] = {1, Wd, L, (long long)D * L};
    const long long dt[4] = {H, Wd, D, bk}, st[4] = {1, H, L, (long long)D * L};
    const int bn[4] = {GP_TW, GP_TH, GP_CB, 1}, bt[4] = {GP_TH, GP_TW, GP_CB, 1};
    if (!gp_make_map4(&maps.nat, ys, dn, sn, bn) || !gp_make_map4(&maps.tr, ys, dt, st, bt)) return SS2D_ERR_UNSUPPORTED;
  }
  const size_t smem = gp_smem_bytes(D, C, esize);
  using KernT = void (*)(const GpParams, const GpMaps);
  static const KernT kerns[8] = {gate_proj_tc_kernel<false, false, false>, gate_proj_tc_kernel<false, false, true>,
                                 gate_proj_tc_kernel<false, true, false>,  gate_proj_tc_kernel<false, true, true>,
                                 gate_proj_tc_kernel<true, false, false>,  gate_proj_tc_kernel<true, false, true>,
                                 gate_proj_tc_kernel<true, true, false>,   gate_proj_tc_kernel<true, true, true>};
  const int ki = (dtype == SS2D_F32 ? 4 : 0) + (z ? 2 : 0) + (g_out ? 1 : 0);
  KernT kern = kerns[ki];
  static PerDeviceOnce once[8];
  cudaError_t e = func_attr_once(once[ki], reinterpret_cast<const void*>(kern), cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) { *cerr = e; return SS2D_ERR_CUDA; }
  int grid = sm_count_current_device();
  if (grid > p.n_tiles) grid = p.n_tiles;
  kern<<<grid, GP_THREADS, smem, stream>>>(p, maps);
  *cerr = cudaGetLastError();
  return *cerr == cudaSuccess ? SS2D_OK : SS2D_ERR_CUDA;
}

}  // namespace ss2d
