// Fused SS2D epilogue: cross-merge sum over the K directions + (B,D,L)->(B,L,D) transpose + LayerNorm(D) +
// SiLU(z) gate, forward and backward. Replaces, per SS2D call, CrossMerge.forward, the transpose copy, out_norm,
// act(z) and `y * z` of /root/reference/gm-unet/model/gm/ss2d.py:486-498, 506-508, 515-517 (5-6 kernels and as
// many round trips through HBM) with one pass: read ys (K planes) and z once, write out once.
// HBM-bound; a CTA owns 32 pixels x all D channels (tile staged in shared memory for the transpose).
#include <cstring>

#include "common.cuh"

namespace ss2d {

constexpr int kEpiTL = 32;         // pixels per tile
constexpr int kEpiThreads = 256;
constexpr int kEpiMaxDPT = 4;     // channels per thread in the backward: D <= 1024 (shared memory caps D near 860)

// Plane k of `ys` is stored either in natural pixel order (offset l = h W + w) or, when bit k of tmask is set, in
// the pixel order of the TRANSPOSED image (offset w H + h): the column-major directions are scanned as row-major
// traversals of a transposed input, and the transposition back happens here, inside the merge.
// A tile is 32 pixels: a 1 x 32 run of the flattened image when every plane is in natural order, a 4 x 8 (h x w) patch
// when some planes are transposed, so that both orders are read in contiguous pieces (32 B and 16 B).
struct PlaneIdx {
  int L, H, W; unsigned tmask; int tiles_w;     // tiles_w: patches per image row (patch mode only; 0 = linear tiles)
  __device__ __forceinline__ int pixel(int tile_in_batch, int px) const {   // -> flattened natural index or -1
    if (!tiles_w) { const int l = tile_in_batch * kEpiTL + px; return l < L ? l : -1; }
    const int th = tile_in_batch / tiles_w, tw = tile_in_batch - th * tiles_w;
    const int h = th * 4 + (px >> 3), w = tw * 8 + (px & 7);
    return (h < H && w < W) ? h * W + w : -1;
  }
};
// Grouped calls (blockIdx.y = group): the G single-direction SS2Ds of a GroupMambaLayer (groupmamba.py:143-149) share one
// launch. Group g reads its K planes at ys + ys_off[g] (per batch: ys_bs), its LayerNorm parameters at lnw + g D, its gate
// at column z_off[g] of a z row, and writes / reads columns io_off[g] ... + D of the out / dout rows (row stride io_rs): the
// concatenation of the G outputs (groupmamba.py:149) is just where the columns land. G = 1 with zero offsets is the plain call.
struct EpiGroups {
  int G;
  int64_t ys_bs, dy_bs, io_rs;
  int dy_two_planes;     // backward, K > 1: dy is (batch, 2, D, L) — plane 0 natural pixel order, plane 1 transposed
  int64_t ys_off[SS2D_MAX_EPI_GROUPS], dy_off[SS2D_MAX_EPI_GROUPS], z_off[SS2D_MAX_EPI_GROUPS];
  int io_off[SS2D_MAX_EPI_GROUPS];
  unsigned tmask[SS2D_MAX_EPI_GROUPS];
};

__device__ __forceinline__ float merge_k(const float* __restrict__ ys, int K, int64_t plane_stride, int64_t row_off, int l,
                                         const PlaneIdx pi) {
  int lt = l;
  if (pi.tmask) { const int h = l / pi.W, w = l - h * pi.W; lt = w * pi.H + h; }
  auto at = [&](int k) { return __ldg(ys + k * plane_stride + row_off + (((pi.tmask >> k) & 1u) ? lt : l)); };
  if (K == 4) {   // association of CrossMerge.forward, csms6s.py:38-39
    const float a = at(0) + at(2);
    const float b = at(1) + at(3);
    return a + b;
  }
  float acc = at(0);
  for (int k = 1; k < K; ++k) acc += at(k);
  return acc;
}

// Loads the merged tile y[d][px] of batch b into s_y[d * 33 + px]. s_pix[px] = natural flattened index of the tile's pixel px
// (or -1). A thread keeps ONE pixel (px = tid % 32: its natural / transposed offsets are computed once per tile, not once per
// element) and walks the channels d = tid / 32, + 8, ...: a warp reads 32 pixels of one channel plane — contiguous runs of 32 /
// 8 / 4 elements depending on the tiling — and the loop body is K loads, K - 1 adds and a shared-memory store (the first
// version recomputed the pixel index, with its integer divisions, per element: 270 instructions per element, 211 us forward
// at B = 24, D = 192, 56^2).
__device__ __forceinline__ void load_merged_tile(float* s_y, const float* __restrict__ ys, int K, int b, int D, int L,
                                                 const int* s_pix, const PlaneIdx pi, int64_t ys_bs) {
  const int64_t plane = (int64_t)D * L;
  const int px = threadIdx.x & 31;
  const int l = s_pix[px];
  int lt = l;
  if (pi.tmask && l >= 0) { const int h = l / pi.W, w = l - h * pi.W; lt = w * pi.H + h; }
  float* dst = s_y + px;
  if (l < 0) {
    for (int d = threadIdx.x >> 5; d < D; d += kEpiThreads / 32) dst[d * (kEpiTL + 1)] = 0.f;
    return;
  }
  const float* base = ys + (int64_t)b * ys_bs;
  if (K == 4) {   // association of CrossMerge.forward, csms6s.py:38-39: (k0 + k2) + (k1 + k3)
    const float* p0 = base + ((pi.tmask & 1u) ? lt : l);
    const float* p1 = base + plane + ((pi.tmask & 2u) ? lt : l);
    const float* p2 = base + 2 * plane + ((pi.tmask & 4u) ? lt : l);
    const float* p3 = base + 3 * plane + ((pi.tmask & 8u) ? lt : l);
#pragma unroll 12
    for (int d = threadIdx.x >> 5; d < D; d += kEpiThreads / 32) {
      const int64_t o = (int64_t)d * L;
      const float a = __ldg(p0 + o) + __ldg(p2 + o);
      const float c = __ldg(p1 + o) + __ldg(p3 + o);
      dst[d * (kEpiTL + 1)] = a + c;
    }
    return;
  }
#pragma unroll 2
  for (int d = threadIdx.x >> 5; d < D; d += kEpiThreads / 32) {
    const int64_t o = (int64_t)d * L;
    float acc = __ldg(base + o + ((pi.tmask & 1u) ? lt : l));
    for (int k = 1; k < K; ++k) acc += __ldg(base + k * plane + o + (((pi.tmask >> k) & 1u) ? lt : l));
    dst[d * (kEpiTL + 1)] = acc;
  }
}

__global__ void __launch_bounds__(kEpiThreads)
out_gate_fwd_kernel(const float* __restrict__ ys, int K, const float* __restrict__ lnw, const float* __restrict__ lnb,
                    const void* __restrict__ z, int64_t z_rs, int z_act, void* __restrict__ out,
                    float* __restrict__ mean_rstd, int batch, int D, int L, float eps, int z_dtype, int out_dtype,
                    int tiles_per_batch, PlaneIdx pi, const EpiGroups eg) {
  extern __shared__ float s_y[];                 // [D][33]
  __shared__ float s_stat[kEpiTL][2];
  __shared__ int s_pixel[2][kEpiTL];             // per-tile pixel table, double-buffered over the tile loop
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gi = blockIdx.y;
  ys += eg.ys_off[gi];
  if (lnw) lnw += gi * D;
  if (lnb) lnb += gi * D;
  if (mean_rstd) mean_rstd += (int64_t)gi * batch * L * 2;
  pi.tmask = eg.tmask[gi];
  const int64_t zo = eg.z_off[gi], oo = eg.io_off[gi];
  int it = 0;
  for (int tile = blockIdx.x; tile < batch * tiles_per_batch; tile += gridDim.x, ++it) {
    const int b = tile / tiles_per_batch, tib = tile - b * tiles_per_batch;
    int* s_pix = s_pixel[it & 1];
    if (threadIdx.x < kEpiTL) s_pix[threadIdx.x] = pi.pixel(tib, threadIdx.x);
    __syncthreads();
    load_merged_tile(s_y, ys, K, b, D, L, s_pix, pi, eg.ys_bs);
    __syncthreads();
    // LayerNorm statistics per pixel (two-pass, fp32): warp w handles pixels w, w+8, ...
    for (int px = warp; px < kEpiTL; px += kEpiThreads / 32) {
      float s = 0.f;
      for (int d = lane; d < D; d += 32) s += s_y[d * (kEpiTL + 1) + px];
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float mean = s / D;
      float v = 0.f;
      for (int d = lane; d < D; d += 32) { const float t = s_y[d * (kEpiTL + 1) + px] - mean; v = fmaf(t, t, v); }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      const float rstd = rsqrtf(v / D + eps);
      if (lane == 0) {
        s_stat[px][0] = mean; s_stat[px][1] = rstd;
        const int l = s_pix[px];
        if (l >= 0 && mean_rstd) {
          mean_rstd[((int64_t)b * L + l) * 2 + 0] = mean;
          mean_rstd[((int64_t)b * L + l) * 2 + 1] = rstd;
        }
      }
    }
    __syncthreads();
    // normalise, gate, write channels-last: a thread keeps its channels (d = tid, + 256, ...: the LayerNorm parameters are
    // loaded once per tile) and walks the tile's pixels; a warp touches 32 consecutive channels of one pixel row (coalesced)
    for (int d = threadIdx.x; d < D; d += kEpiThreads) {
      const float wv = lnw ? __ldg(lnw + d) : 1.f, bv = (lnw && lnb) ? __ldg(lnb + d) : 0.f;
      const float* col = s_y + d * (kEpiTL + 1);
#pragma unroll 16
      for (int px = 0; px < kEpiTL; ++px) {
        const int l = s_pix[px];
        if (l < 0) continue;
        const int64_t row = (int64_t)b * L + l;
        float o = fmaf((col[px] - s_stat[px][0]) * s_stat[px][1], wv, bv);
        if (z) {
          float zz = load1(z, row * z_rs + zo + d, z_dtype);
          if (z_act) zz = silu_f(zz);
          o *= zz;
        }
        store1(out, row * eg.io_rs + oo + d, out_dtype, o);
      }
    }
  }
}

__global__ void __launch_bounds__(kEpiThreads, 4)
out_gate_bwd_kernel(const float* __restrict__ ys, int K, const float* __restrict__ lnw, const float* __restrict__ lnb,
                    const void* __restrict__ z, int64_t z_rs, int z_act, const void* __restrict__ dout,
                    const float* __restrict__ mean_rstd, float* __restrict__ dy, void* __restrict__ dz, int64_t dz_rs,
                    float* __restrict__ dw_part, float* __restrict__ db_part, int batch, int D, int L, int z_dtype,
                    int out_dtype, int tiles_per_batch, PlaneIdx pi, const EpiGroups eg) {
  const int gi = blockIdx.y;
  ys += eg.ys_off[gi];
  dy += eg.dy_off[gi];
  if (lnw) lnw += gi * D;
  if (lnb) lnb += gi * D;
  mean_rstd += (int64_t)gi * batch * L * 2;
  dw_part += (int64_t)gi * gridDim.x * D;
  db_part += (int64_t)gi * gridDim.x * D;
  pi.tmask = eg.tmask[gi];
  const int64_t zo = eg.z_off[gi], oo = eg.io_off[gi];
  extern __shared__ float smem[];
  float* s_y = smem;                               // [D][33] merged y, then dy
  float* s_g = s_y + (size_t)D * (kEpiTL + 1);     // [D][33] d(yn) = dout * gate * w
  __shared__ float s_stat[kEpiTL][4];              // mean, rstd, mean(g), mean(g * yn)
  __shared__ int s_pixel[2][kEpiTL];               // per-tile pixel table, double-buffered over the tile loop
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ float s_red[2][kEpiThreads];          // pixel-lane partials of the LayerNorm weight / bias gradients
  float acc_dw[kEpiMaxDPT], acc_db[kEpiMaxDPT];
#pragma unroll
  for (int m = 0; m < kEpiMaxDPT; ++m) { acc_dw[m] = 0.f; acc_db[m] = 0.f; }
  const int PP = D >= kEpiThreads ? 1 : (kEpiThreads / D < kEpiTL ? kEpiThreads / D : kEpiTL);   // pixel lanes
  const int pl = threadIdx.x / D, dl = threadIdx.x - pl * D;
  int it = 0;
  for (int tile = blockIdx.x; tile < batch * tiles_per_batch; tile += gridDim.x, ++it) {
    const int b = tile / tiles_per_batch, tib = tile - b * tiles_per_batch;
    int* s_pix = s_pixel[it & 1];
    if (threadIdx.x < kEpiTL) s_pix[threadIdx.x] = pi.pixel(tib, threadIdx.x);
    __syncthreads();
    load_merged_tile(s_y, ys, K, b, D, L, s_pix, pi, eg.ys_bs);
    for (int px = threadIdx.x; px < kEpiTL; px += kEpiThreads) {
      const int l = s_pix[px];
      s_stat[px][0] = l >= 0 ? mean_rstd[((int64_t)b * L + l) * 2 + 0] : 0.f;
      s_stat[px][1] = l >= 0 ? mean_rstd[((int64_t)b * L + l) * 2 + 1] : 0.f;
    }
    __syncthreads();
    // pass 1 (threads along D, coalesced): gate grads and d(yn). A thread always meets the same channels, so the
    // LayerNorm weight/bias gradients accumulate in registers, without atomics. For D < 256 (the live GM-UNet regime:
    // D = 16 ... 112) the block is folded into PP = 256 / D pixel lanes x D channels so that every thread has work and
    // a warp still reads whole contiguous pixel rows of dout / z (consecutive pixels are consecutive in memory);
    // the pixel lanes' partials are summed once, at the end of the kernel.
    auto pass1 = [&](int px, int d, int m) {
      const int l = s_pix[px];
      float g = 0.f;
      if (l >= 0) {
        const float yn = (s_y[d * (kEpiTL + 1) + px] - s_stat[px][0]) * s_stat[px][1];
        const float w = lnw ? __ldg(lnw + d) : 1.f;
        const float lin = lnw ? fmaf(yn, w, lnb ? __ldg(lnb + d) : 0.f) : yn;
        float go = load1(dout, ((int64_t)b * L + l) * eg.io_rs + oo + d, out_dtype);
        if (z) {
          const float zr = load1(z, ((int64_t)b * L + l) * z_rs + zo + d, z_dtype);
          const float gate = z_act ? silu_f(zr) : zr;
          if (dz) store1(dz, ((int64_t)b * L + l) * dz_rs + zo + d, z_dtype, go * lin * (z_act ? silu_grad_f(zr) : 1.f));
          go *= gate;
        }
        acc_dw[m] = fmaf(go, yn, acc_dw[m]);
        acc_db[m] += go;
        g = go * w;
      }
      s_g[d * (kEpiTL + 1) + px] = g;
    };
    if (PP == 1) {
#pragma unroll 4
      for (int px = 0; px < kEpiTL; ++px) {
#pragma unroll
        for (int m = 0; m < kEpiMaxDPT; ++m) {
          const int d = threadIdx.x + m * kEpiThreads;
          if (d >= D) break;
          pass1(px, d, m);
        }
      }
    } else if (pl < PP) {
#pragma unroll 4
      for (int px = pl; px < kEpiTL; px += PP) pass1(px, dl, 0);
    }
    __syncthreads();
    for (int px = warp; px < kEpiTL; px += kEpiThreads / 32) {
      float s1 = 0.f, s2 = 0.f;
      const float mean = s_stat[px][0], rstd = s_stat[px][1];
      for (int d = lane; d < D; d += 32) {
        const float g = s_g[d * (kEpiTL + 1) + px];
        s1 += g;
        s2 = fmaf(g, (s_y[d * (kEpiTL + 1) + px] - mean) * rstd, s2);
      }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
      if (lane == 0) { s_stat[px][2] = s1 / D; s_stat[px][3] = s2 / D; }
    }
    __syncthreads();
    // dy[b][d][l] = rstd * (g - mean(g) - yn * mean(g yn)); a thread keeps one pixel (its offsets are computed once per
    // tile) and walks the channels: a warp writes 32 pixels of one channel plane
    {
      const int px = threadIdx.x & 31;
      const int l = s_pix[px];
      if (l >= 0) {
        const float mean = s_stat[px][0], rstd = s_stat[px][1], mg = s_stat[px][2], mgy = s_stat[px][3];
        int lt = l;
        if (pi.H > 0 && pi.W > 0 && (pi.tmask || eg.dy_two_planes)) { const int h = l / pi.W, w = l - h * pi.W; lt = w * pi.H + h; }
        // K == 1: the gradient belongs to the single plane and is written in ITS pixel order (transposed when tmask is set)
        float* o1 = dy + (int64_t)b * eg.dy_bs + ((K == 1 && pi.tmask) ? lt : l);
        float* o2 = dy + (int64_t)b * eg.dy_bs + (int64_t)D * L + lt;      // second plane: the pixel order of the transposed image
#pragma unroll 4
        for (int d = threadIdx.x >> 5; d < D; d += kEpiThreads / 32) {
          const float yn = (s_y[d * (kEpiTL + 1) + px] - mean) * rstd;
          const float gval = rstd * (s_g[d * (kEpiTL + 1) + px] - mg - yn * mgy);
          o1[(int64_t)d * L] = gval;
          if (eg.dy_two_planes) o2[(int64_t)d * L] = gval;
        }
      }
    }
  }
  if (PP == 1) {
#pragma unroll
    for (int m = 0; m < kEpiMaxDPT; ++m) {
      const int d = threadIdx.x + m * kEpiThreads;
      if (d < D) {
        dw_part[(int64_t)blockIdx.x * D + d] = acc_dw[m];
        db_part[(int64_t)blockIdx.x * D + d] = acc_db[m];
      }
    }
  } else {
    s_red[0][threadIdx.x] = acc_dw[0];
    s_red[1][threadIdx.x] = acc_db[0];
    __syncthreads();
    if (threadIdx.x < D) {
      float sw = 0.f, sb = 0.f;
      for (int i = 0; i < PP; ++i) { sw += s_red[0][i * D + threadIdx.x]; sb += s_red[1][i * D + threadIdx.x]; }
      dw_part[(int64_t)blockIdx.x * D + threadIdx.x] = sw;
      db_part[(int64_t)blockIdx.x * D + threadIdx.x] = sb;
    }
  }
}

// ---- live GM-UNet regime: one plane (K = 1), D <= 32 ------------------------------------------------------------
// With 16 or 32 channels a pixel's LayerNorm fits one thread's registers: thread = pixel, visited in the PLANE's own
// order (so the channel-major reads / writes of ys and dy are coalesced across the warp whether or not the plane is
// transposed), while the channels-last rows of z / out / dout are whole 64- or 128-byte rows per thread. No shared
// memory, no barrier in the pixel loop. (The tiled kernels above need three barriers per 32 pixels: 28 us forward and
// 50 us backward at D = 16, B = 24, 56^2 against 15 MB of traffic.)
template <int DP>
__device__ __forceinline__ void row_load(const void* base, int64_t off, int dt, int D, float* v) {
  if (dt == SS2D_F32 && (D & 3) == 0 && ((reinterpret_cast<uintptr_t>(base) + off * 4) & 15) == 0) {
#pragma unroll
    for (int d = 0; d < DP; d += 4)
      if (d < D) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + off + d));
        v[d] = t.x; v[d + 1] = t.y; v[d + 2] = t.z; v[d + 3] = t.w;
      }
  } else {
#pragma unroll
    for (int d = 0; d < DP; ++d)
      if (d < D) v[d] = load1(base, off + d, dt);
  }
}
template <int DP>
__device__ __forceinline__ void row_store(void* base, int64_t off, int dt, int D, const float* v) {
  if (dt == SS2D_F32 && (D & 3) == 0 && ((reinterpret_cast<uintptr_t>(base) + off * 4) & 15) == 0) {
#pragma unroll
    for (int d = 0; d < DP; d += 4)
      if (d < D) *reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + off + d) = make_float4(v[d], v[d + 1], v[d + 2], v[d + 3]);
  } else {
#pragma unroll
    for (int d = 0; d < DP; ++d)
      if (d < D) store1(base, off + d, dt, v[d]);
  }
}

template <int DP>
__global__ void __launch_bounds__(kEpiThreads)
out_gate_fwd_small_kernel(const float* __restrict__ ys, const float* __restrict__ lnw, const float* __restrict__ lnb,
                          const void* __restrict__ z, int64_t z_rs, int z_act, void* __restrict__ out,
                          float* __restrict__ mean_rstd, int batch, int D, int L, float eps, int z_dtype, int out_dtype,
                          int H, int W, const EpiGroups eg) {
  const int gi = blockIdx.y;
  ys += eg.ys_off[gi];
  if (lnw) lnw += gi * D;
  if (lnb) lnb += gi * D;
  if (mean_rstd) mean_rstd += (int64_t)gi * batch * L * 2;
  const int transposed = (int)(eg.tmask[gi] & 1u);
  const int64_t zo = eg.z_off[gi], oo = eg.io_off[gi];
  const int64_t total = (int64_t)batch * L;
  for (int64_t idx = (int64_t)blockIdx.x * kEpiThreads + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * kEpiThreads) {
    const int b = (int)(idx / L), lp = (int)(idx - (int64_t)b * L);          // pixel in plane order
    int l = lp;
    if (transposed) { const int w = lp / H, h = lp - w * H; l = h * W + w; }
    float y[DP];
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < DP; ++d) { y[d] = d < D ? __ldg(ys + (int64_t)b * eg.ys_bs + (int64_t)d * L + lp) : 0.f; s += y[d]; }
    const float mean = s / D;
    float v = 0.f;
#pragma unroll
    for (int d = 0; d < DP; ++d) { const float t = d < D ? y[d] - mean : 0.f; v = fmaf(t, t, v); }
    const float rstd = rsqrtf(v / D + eps);
    const int64_t row = (int64_t)b * L + l;
    if (mean_rstd) { mean_rstd[row * 2] = mean; mean_rstd[row * 2 + 1] = rstd; }
    float zz[DP];
    if (z) row_load<DP>(z, row * z_rs + zo, z_dtype, D, zz);
#pragma unroll
    for (int d = 0; d < DP; ++d) {
      if (d < D) {
        float o = (y[d] - mean) * rstd;
        o = lnw ? fmaf(o, __ldg(lnw + d), lnb ? __ldg(lnb + d) : 0.f) : o;
        if (z) o *= z_act ? silu_f(zz[d]) : zz[d];
        y[d] = o;
      }
    }
    row_store<DP>(out, row * eg.io_rs + oo, out_dtype, D, y);
  }
}

template <int DP>
__global__ void __launch_bounds__(kEpiThreads)
out_gate_bwd_small_kernel(const float* __restrict__ ys, const float* __restrict__ lnw, const float* __restrict__ lnb,
                          const void* __restrict__ z, int64_t z_rs, int z_act, const void* __restrict__ dout,
                          const float* __restrict__ mean_rstd, float* __restrict__ dy, void* __restrict__ dz, int64_t dz_rs,
                          float* __restrict__ dw_part, float* __restrict__ db_part, int batch, int D, int L, int z_dtype,
                          int out_dtype, int H, int W, const EpiGroups eg) {
  const int gi = blockIdx.y;
  ys += eg.ys_off[gi];
  dy += eg.dy_off[gi];
  if (lnw) lnw += gi * D;
  if (lnb) lnb += gi * D;
  mean_rstd += (int64_t)gi * batch * L * 2;
  dw_part += (int64_t)gi * gridDim.x * D;
  db_part += (int64_t)gi * gridDim.x * D;
  const int transposed = (int)(eg.tmask[gi] & 1u);
  const int64_t zo = eg.z_off[gi], oo = eg.io_off[gi];
  __shared__ float s_red[kEpiThreads / 32][2 * DP];
  float acc_dw[DP], acc_db[DP];
#pragma unroll
  for (int d = 0; d < DP; ++d) { acc_dw[d] = 0.f; acc_db[d] = 0.f; }
  const int64_t total = (int64_t)batch * L;
  for (int64_t idx = (int64_t)blockIdx.x * kEpiThreads + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * kEpiThreads) {
    const int b = (int)(idx / L), lp = (int)(idx - (int64_t)b * L);
    int l = lp;
    if (transposed) { const int w = lp / H, h = lp - w * H; l = h * W + w; }
    const int64_t row = (int64_t)b * L + l;
    const float mean = mean_rstd[row * 2], rstd = mean_rstd[row * 2 + 1];
    float g[DP], yn[DP], zz[DP];
    row_load<DP>(dout, row * eg.io_rs + oo, out_dtype, D, g);
    if (z) row_load<DP>(z, row * z_rs + zo, z_dtype, D, zz);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int d = 0; d < DP; ++d) {
      if (d < D) {
        yn[d] = (__ldg(ys + (int64_t)b * eg.ys_bs + (int64_t)d * L + lp) - mean) * rstd;
        const float w = lnw ? __ldg(lnw + d) : 1.f;
        const float lin = lnw ? fmaf(yn[d], w, lnb ? __ldg(lnb + d) : 0.f) : yn[d];
        float go = g[d];
        if (z) {
          const float zr = zz[d];
          zz[d] = go * lin * (z_act ? silu_grad_f(zr) : 1.f);       // d z
          go *= z_act ? silu_f(zr) : zr;
        }
        acc_dw[d] = fmaf(go, yn[d], acc_dw[d]);
        acc_db[d] += go;
        g[d] = go * w;
        s1 += g[d];
        s2 = fmaf(g[d], yn[d], s2);
      } else { g[d] = 0.f; yn[d] = 0.f; }
    }
    if (z && dz) row_store<DP>(dz, row * dz_rs + zo, z_dtype, D, zz);
    s1 /= D; s2 /= D;
    // gradient of the single plane, written in ITS pixel order (coalesced across the warp)
#pragma unroll
    for (int d = 0; d < DP; ++d)
      if (d < D) dy[(int64_t)b * eg.dy_bs + (int64_t)d * L + lp] = rstd * (g[d] - s1 - yn[d] * s2);
  }
  // LayerNorm weight / bias gradients: warp butterflies, then the block's warps through shared memory
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 0; d < DP; ++d) {
    float a = acc_dw[d], c = acc_db[d];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); c += __shfl_xor_sync(0xffffffffu, c, o); }
    if (lane == 0) { s_red[warp][d] = a; s_red[warp][DP + d] = c; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * DP) {
    float t = 0.f;
    for (int w = 0; w < kEpiThreads / 32; ++w) t += s_red[w][threadIdx.x];
    const int d = threadIdx.x < DP ? threadIdx.x : threadIdx.x - DP;
    if (d < D) (threadIdx.x < DP ? dw_part : db_part)[(int64_t)blockIdx.x * D + d] = t;
  }
}

static bool epi_small(int K, int D) { return K == 1 && D <= 32; }

static int epi_tiles_per_batch(int L, int H, int W, bool patch) {
  return patch ? ((H + 3) / 4) * ((W + 7) / 8) : (L + kEpiTL - 1) / kEpiTL;
}
int epi_bwd_partials(int batch, int L) {     // an upper bound that does not depend on the tiling mode
  const int tiles = batch * ((L + kEpiTL - 1) / kEpiTL);
  return tiles < 148 * 4 ? tiles : 148 * 4;      // 4 CTAs per SM fit (2 x D x 33 floats of shared memory each at D = 192)
}
int epi_max_D(bool backward) { return backward ? 832 : 1664; }   // keeps the tile(s) within 227 KB of shared memory

static bool epi_any_transposed(const EpiGroups& eg) {
  for (int g = 0; g < eg.G; ++g) if (eg.tmask[g]) return true;
  return false;
}

static cudaError_t epi_fwd_launch(const float* ys, int K, const float* lnw, const float* lnb, const void* z, int64_t z_rs,
                                  int z_act, void* out, float* mean_rstd, int batch, int D, int L, float eps, int z_dtype,
                                  int out_dtype, int H, int W, const EpiGroups& eg, cudaStream_t stream) {
  if (epi_small(K, D)) {
    const int64_t total = (int64_t)batch * L;
    const int cap = 148 * 8 / eg.G > 0 ? 148 * 8 / eg.G : 1;
    dim3 grid((unsigned)((total + kEpiThreads - 1) / kEpiThreads < cap ? (total + kEpiThreads - 1) / kEpiThreads : cap), eg.G);
    if (D <= 16)
      out_gate_fwd_small_kernel<16><<<grid, kEpiThreads, 0, stream>>>(ys, lnw, lnb, z, z_rs, z_act, out, mean_rstd, batch, D, L,
                                                                       eps, z_dtype, out_dtype, H, W, eg);
    else
      out_gate_fwd_small_kernel<32><<<grid, kEpiThreads, 0, stream>>>(ys, lnw, lnb, z, z_rs, z_act, out, mean_rstd, batch, D, L,
                                                                       eps, z_dtype, out_dtype, H, W, eg);
    return cudaGetLastError();
  }
  const size_t smem = (size_t)D * (kEpiTL + 1) * 4;
  cudaError_t e = cudaFuncSetAttribute(out_gate_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const bool patch = epi_any_transposed(eg);
  const int tpb = epi_tiles_per_batch(L, H, W, patch);
  const int tiles = batch * tpb;
  const int cap = 148 * 8 / eg.G > 0 ? 148 * 8 / eg.G : 1;
  dim3 grid((unsigned)(tiles < cap ? tiles : cap), eg.G);
  const PlaneIdx pi{L, H, W, 0u, patch ? (W + 7) / 8 : 0};
  out_gate_fwd_kernel<<<grid, kEpiThreads, smem, stream>>>(ys, K, lnw, lnb, z, z_rs, z_act, out, mean_rstd, batch, D, L,
                                                          eps, z_dtype, out_dtype, tpb, pi, eg);
  return cudaGetLastError();
}

static cudaError_t epi_bwd_launch(const float* ys, int K, const float* lnw, const float* lnb, const void* z, int64_t z_rs,
                                  int z_act, const void* dout, const float* mean_rstd, float* dy, void* dz, int64_t dz_rs,
                                  float* dw_part, float* db_part, int n_partials, int batch, int D, int L, int z_dtype,
                                  int out_dtype, int H, int W, const EpiGroups& eg, cudaStream_t stream) {
  dim3 grid((unsigned)n_partials, eg.G);
  if (epi_small(K, D)) {
    if (D <= 16)
      out_gate_bwd_small_kernel<16><<<grid, kEpiThreads, 0, stream>>>(ys, lnw, lnb, z, z_rs, z_act, dout, mean_rstd, dy, dz,
                                                                       dz_rs, dw_part, db_part, batch, D, L, z_dtype,
                                                                       out_dtype, H, W, eg);
    else
      out_gate_bwd_small_kernel<32><<<grid, kEpiThreads, 0, stream>>>(ys, lnw, lnb, z, z_rs, z_act, dout, mean_rstd, dy, dz,
                                                                       dz_rs, dw_part, db_part, batch, D, L, z_dtype,
                                                                       out_dtype, H, W, eg);
    return cudaGetLastError();
  }
  const size_t smem = (size_t)2 * D * (kEpiTL + 1) * 4;
  cudaError_t e = cudaFuncSetAttribute(out_gate_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const bool patch = epi_any_transposed(eg);
  const int tpb = epi_tiles_per_batch(L, H, W, patch);
  const PlaneIdx pi{L, H, W, 0u, patch ? (W + 7) / 8 : 0};
  out_gate_bwd_kernel<<<grid, kEpiThreads, smem, stream>>>(ys, K, lnw, lnb, z, z_rs, z_act, dout, mean_rstd, dy, dz,
                                                          dz_rs, dw_part, db_part, batch, D, L, z_dtype, out_dtype,
                                                          tpb, pi, eg);
  return cudaGetLastError();
}

static EpiGroups epi_single(int K, int D, int L, unsigned tmask) {
  EpiGroups eg;
  memset(&eg, 0, sizeof(eg));
  eg.G = 1; eg.ys_bs = (int64_t)K * D * L; eg.dy_bs = (int64_t)D * L; eg.io_rs = D; eg.tmask[0] = tmask;
  return eg;
}

cudaError_t out_gate_fwd_launch(const float* ys, int K, const float* lnw, const float* lnb, const void* z, int64_t z_rs,
                                int z_act, void* out, float* mean_rstd, int batch, int D, int L, float eps, int z_dtype,
                                int out_dtype, int H, int W, unsigned tmask, cudaStream_t stream) {
  return epi_fwd_launch(ys, K, lnw, lnb, z, z_rs, z_act, out, mean_rstd, batch, D, L, eps, z_dtype, out_dtype, H, W,
                        epi_single(K, D, L, tmask), stream);
}

cudaError_t out_gate_bwd_launch(const float* ys, int K, const float* lnw, const float* lnb, const void* z, int64_t z_rs,
                                int z_act, const void* dout, const float* mean_rstd, float* dy, void* dz, int64_t dz_rs,
                                float* dw_part, float* db_part, int n_partials, int batch, int D, int L, int z_dtype,
                                int out_dtype, int H, int W, unsigned tmask, int dy_two_planes, cudaStream_t stream) {
  EpiGroups eg = epi_single(K, D, L, tmask);
  if (dy_two_planes) { eg.dy_two_planes = 1; eg.dy_bs = (int64_t)2 * D * L; }
  return epi_bwd_launch(ys, K, lnw, lnb, z, z_rs, z_act, dout, mean_rstd, dy, dz, dz_rs, dw_part, db_part, n_partials, batch, D,
                        L, z_dtype, out_dtype, H, W, eg, stream);
}

// G single-plane groups in one launch: ys (batch, G, D, L) with group g in plane plane_of[g]; out / dout / z / dz rows hold the
// G groups side by side (columns g D ... of rows of io_rs / z_rs / dz_rs elements; z and dz start at column z_col0 + g z_gs).
static EpiGroups epi_grouped(int G, int D, int L, const int* plane_of, unsigned tmask_bits, int64_t io_rs, int64_t z_col0,
                             int64_t z_gs) {
  EpiGroups eg;
  memset(&eg, 0, sizeof(eg));
  eg.G = G; eg.ys_bs = (int64_t)G * D * L; eg.dy_bs = (int64_t)G * D * L; eg.io_rs = io_rs;
  for (int g = 0; g < G; ++g) {
    eg.ys_off[g] = (int64_t)plane_of[g] * D * L;
    eg.dy_off[g] = eg.ys_off[g];
    eg.z_off[g] = z_col0 + g * z_gs;
    eg.io_off[g] = g * D;
    eg.tmask[g] = (tmask_bits >> plane_of[g]) & 1u;
  }
  return eg;
}

cudaError_t group_gate_fwd_launch(const float* ys, int G, const int* plane_of, unsigned tmask_bits, const float* lnw,
                                  const float* lnb, const void* z, int64_t z_rs, int64_t z_col0, int64_t z_gs, void* out,
                                  int64_t out_rs, float* mean_rstd, int batch, int D, int L, float eps, int z_dtype,
                                  int out_dtype, int H, int W, cudaStream_t stream) {
  return epi_fwd_launch(ys, 1, lnw, lnb, z, z_rs, 1, out, mean_rstd, batch, D, L, eps, z_dtype, out_dtype, H, W,
                        epi_grouped(G, D, L, plane_of, tmask_bits, out_rs, z_col0, z_gs), stream);
}

cudaError_t group_gate_bwd_launch(const float* ys, int G, const int* plane_of, unsigned tmask_bits, const float* lnw,
                                  const float* lnb, const void* z, int64_t z_rs, int64_t z_col0, int64_t z_gs, const void* dout,
                                  int64_t dout_rs, const float* mean_rstd, float* dy, void* dz, int64_t dz_rs, float* dw_part,
                                  float* db_part, int n_partials, int batch, int D, int L, int z_dtype, int out_dtype, int H,
                                  int W, cudaStream_t stream) {
  return epi_bwd_launch(ys, 1, lnw, lnb, z, z_rs, 1, dout, mean_rstd, dy, dz, dz_rs, dw_part, db_part, n_partials, batch, D, L,
                        z_dtype, out_dtype, H, W, epi_grouped(G, D, L, plane_of, tmask_bits, dout_rs, z_col0, z_gs), stream);
}

}  // namespace ss2d
