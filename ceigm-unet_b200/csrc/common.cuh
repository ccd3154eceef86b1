// Shared device helpers for the ss2d_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ss2d_b200.h"

namespace ss2d {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// MUFU.EX2 / MUFU.LG2 (16 lanes/clk/SM measured on B200: tools/ubench/pipes.cu)
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2f(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// softplus with PyTorch's default threshold 20 (reference: selective_scan_fwd_kernel.cuh:117 and
// F.softplus in selective_scan_ref). Small exp(x) uses the log1p series so tiny deltas keep relative accuracy.
__device__ __forceinline__ float softplus20(float x) {
  const float e = ex2f(x * kLog2e);
  const float series = e * (1.f - e * (0.5f - e * 0.33333334f));
  const float full = kLn2 * lg2f(1.f + e);
  const float sp = e < 0.0078125f ? series : full;
  return x > 20.f ? x : sp;
}
// d softplus(x) / dx = sigmoid(x) (1 above the threshold)
__device__ __forceinline__ float softplus20_grad(float x) {
  const float e = ex2f(-x * kLog2e);
  return x > 20.f ? 1.f : __fdividef(1.f, 1.f + e);
}
// silu(x) = x sigmoid(x) and its derivative s (1 + x (1 - s)), s = sigmoid(x)
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.f + ex2f(-x * kLog2e)); }
__device__ __forceinline__ float silu_grad_f(float x) {
  const float s = __fdividef(1.f, 1.f + ex2f(-x * kLog2e));
  return s * (1.f + x * (1.f - s));
}

// ---- dtype-erased 4-element loads/stores (runtime dtype: the math is always fp32 from shared memory) ----
__device__ __forceinline__ size_t dtype_size(int dt) { return dt == SS2D_F32 ? 4 : 2; }

__device__ __forceinline__ float load1(const void* base, int64_t idx, int dt) {
  if (dt == SS2D_F32) return __ldg(reinterpret_cast<const float*>(base) + idx);
  if (dt == SS2D_F16) return __half2float(__ldg(reinterpret_cast<const __half*>(base) + idx));
  return __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(base) + idx));
}
__device__ __forceinline__ void store1(void* base, int64_t idx, int dt, float v) {
  if (dt == SS2D_F32) reinterpret_cast<float*>(base)[idx] = v;
  else if (dt == SS2D_F16) reinterpret_cast<__half*>(base)[idx] = __float2half_rn(v);
  else reinterpret_cast<__nv_bfloat16*>(base)[idx] = __float2bfloat16_rn(v);
}
// true when 4 consecutive elements starting at idx can be moved with one vector access
__device__ __forceinline__ bool vec4_ok(const void* base, int64_t idx, int dt) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(base) + static_cast<uintptr_t>(idx) * dtype_size(dt);
  return (a & (4 * dtype_size(dt) - 1)) == 0;
}
__device__ __forceinline__ float4 load4(const void* base, int64_t idx, int dt) {
  if (dt == SS2D_F32) return __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + idx));
  const uint2 raw = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(base) + idx));
  float4 r;
  if (dt == SS2D_F16) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
    r = make_float4(a.x, a.y, b.x, b.y);
  } else {
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.y));
    r = make_float4(a.x, a.y, b.x, b.y);
  }
  return r;
}
__device__ __forceinline__ void store4(void* base, int64_t idx, int dt, float4 v) {
  if (dt == SS2D_F32) {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + idx) = v;
    return;
  }
  uint2 raw;
  if (dt == SS2D_F16) {
    const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    raw.x = *reinterpret_cast<const uint32_t*>(&a);
    raw.y = *reinterpret_cast<const uint32_t*>(&b);
  } else {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    raw.x = *reinterpret_cast<const uint32_t*>(&a);
    raw.y = *reinterpret_cast<const uint32_t*>(&b);
  }
  *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(base) + idx) = raw;
}

// ---- scan-order addressing: position l of the traversal -> natural offset inside an (H, W) plane ----
// dir 0: tensors already in scan order (identity). 1: row-major, 2: column-major, 3/4: reversed.
// (index maps of CrossScan_1.._4, /root/reference/gm-unet/model/gm/csms6s.py:56-206)
struct ScanOrder {
  int dir, H, W, L;
  __device__ __forceinline__ bool contiguous() const { return dir == 0 || dir == 1 || dir == 3; }
  __device__ __forceinline__ bool reversed() const { return dir == 3 || dir == 4; }
  __device__ __forceinline__ int natural(int l) const {
    if (dir == 0 || dir == 1) return l;
    if (dir == 3) return L - 1 - l;
    const int t = dir == 2 ? l : L - 1 - l;   // column-major position
    const int w = t / H, h = t - w * H;
    return h * W + w;
  }
};

// ---- TMA bulk copies (cp.async.bulk -> SASS UBLKCP) completing on an mbarrier ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// orders this thread's earlier generic-proxy shared-memory accesses before later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// same, for a thread that expects to wait long (the producer): sleep between polls instead of burning issue slots
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (done) break;
    __nanosleep(1000);
  }
}
// global -> shared bulk copy of `bytes` (multiple of 16; both addresses 16-byte aligned)
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// tiled TMA loads through a tensor map (UTMALDG): box lands densely in shared memory, 128-byte swizzled
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* tmap, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const void* tmap, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

// Shared-memory tile layout: rows of 32 floats (128 bytes) with the 16-byte chunks XOR-swizzled by the row index —
// exactly what TMA's SWIZZLE_128B produces for a 1024-byte aligned tile — so that 8 consecutive rows read at the
// same column (the scan's access pattern) hit 8 different bank groups without any padding.
constexpr int kTileL = 32;
__device__ __forceinline__ int swz(int r, int c) { return r * kTileL + ((((c >> 2) ^ r) & 7) << 2) + (c & 3); }

// Tile accessors in SCAN coordinates. When a reversed traversal (direction 3) is staged by TMA the tile holds the 32
// positions in MEMORY order, i.e. mirrored: scan column c lives at tile column 31 - c. rev selects that mirror.
__device__ __forceinline__ int swz1(int r, int c, bool rev) { return swz(r, rev ? kTileL - 1 - c : c); }
__device__ __forceinline__ float4 tile_ld4(const float* tile, int r, int c, bool rev) {   // scan columns c..c+3, c % 4 == 0
  const float4 v = *reinterpret_cast<const float4*>(tile + swz(r, rev ? kTileL - 4 - c : c));
  return rev ? make_float4(v.w, v.z, v.y, v.x) : v;
}
__device__ __forceinline__ void tile_st4(float* tile, int r, int c, bool rev, float4 v) {
  *reinterpret_cast<float4*>(tile + swz(r, rev ? kTileL - 4 - c : c)) = rev ? make_float4(v.w, v.z, v.y, v.x) : v;
}

__device__ __forceinline__ float& f4_at(float4& v, int e) { return reinterpret_cast<float*>(&v)[e]; }

}  // namespace ss2d
