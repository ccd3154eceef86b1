// Output gate of the Mamba selective-scan contract (mamba_ssm's selective_scan_cuda with z), as two elementwise passes:
//   forward:  out_z = y * silu(z)                                   (reads y, z; writes out_z)
//   backward: dy = dout_z * silu(z), dz = dout_z * y * silu'(z)     (reads dout_z, z, y; writes dy fp32 dense and dz)
// y, out_z, dout_z have the out dtype; z, dz the io dtype; all five use the descriptor's out strides. HBM-bound: 12 bytes per
// element forward and 20 backward in fp32. Rows move 8 elements per access (two 128-bit fp32 accesses, one for 16-bit) when
// every row start is 16-byte aligned, else one element at a time.
#include <initializer_list>

#include "common.cuh"
#include "host_util.h"
#include "scan_params.h"

namespace ss2d {

namespace {

constexpr int kGateThreads = 256;

struct GateGeom {
  int dim, L;
  int64_t rows, bs, ds;          // rows = batch * dim; bs, ds: out strides (elements)
};

template <int V>
__device__ __forceinline__ void ld(const float* p, float (&v)[V]) {
  if constexpr (V == 8) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
    v[0] = __ldg(p);
  }
}
__device__ __forceinline__ float2 to_f2(__half2 h) { return __half22float2(h); }
__device__ __forceinline__ float2 to_f2(__nv_bfloat162 h) { return __bfloat1622float2(h); }
__device__ __forceinline__ float to_f(__half h) { return __half2float(h); }
__device__ __forceinline__ float to_f(__nv_bfloat16 h) { return __bfloat162float(h); }
template <typename H> struct Pair;
template <> struct Pair<__half> { using type = __half2; };
template <> struct Pair<__nv_bfloat16> { using type = __nv_bfloat162; };

template <int V, typename H>
__device__ __forceinline__ void ld(const H* p, float (&v)[V]) {
  if constexpr (V == 8) {
    const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = to_f2(*reinterpret_cast<const typename Pair<H>::type*>(&w[i]));
      v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
  } else {
    v[0] = to_f(p[0]);
  }
}

template <int V>
__device__ __forceinline__ void st(float* p, const float (&v)[V]) {
  if constexpr (V == 8) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
  } else {
    p[0] = v[0];
  }
}
template <int V>
__device__ __forceinline__ void st(__half* p, const float (&v)[V]) {
  if constexpr (V == 8) {
    uint4 r;
    uint32_t* w = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = r;
  } else {
    p[0] = __float2half_rn(v[0]);
  }
}
template <int V>
__device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[V]) {
  if constexpr (V == 8) {
    uint4 r;
    uint32_t* w = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = r;
  } else {
    p[0] = __float2bfloat16_rn(v[0]);
  }
}

// element offset of vector i (V elements of one row) under the out strides, and its row / column
template <int V>
__device__ __forceinline__ int64_t gate_off(const GateGeom& g, int64_t i, int64_t* row, int* l) {
  const int per_row = g.L / V;
  *row = i / per_row;
  *l = (int)(i - *row * per_row) * V;
  const int64_t b = *row / g.dim, d = *row - b * g.dim;
  return b * g.bs + d * g.ds + *l;
}

}  // namespace

template <typename TI, typename TO, int V>
__global__ void __launch_bounds__(kGateThreads) scan_gate_fwd_kernel(const TO* __restrict__ y, const TI* __restrict__ z,
                                                                     TO* __restrict__ out_z, const GateGeom g) {
  const int64_t total = g.rows * (g.L / V);
  for (int64_t i = (int64_t)blockIdx.x * kGateThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kGateThreads) {
    int64_t row;
    int l;
    const int64_t o = gate_off<V>(g, i, &row, &l);
    float yv[V], zv[V];
    ld<V>(y + o, yv);
    ld<V>(z + o, zv);
#pragma unroll
    for (int e = 0; e < V; ++e) yv[e] *= silu_f(zv[e]);
    st<V>(out_z + o, yv);
  }
}

template <typename TI, typename TO, int V>
__global__ void __launch_bounds__(kGateThreads) scan_gate_bwd_kernel(const TO* __restrict__ dout_z, const TI* __restrict__ z,
                                                                     const TO* __restrict__ y, float* __restrict__ dy,
                                                                     TI* __restrict__ dz, const GateGeom g) {
  const int64_t total = g.rows * (g.L / V);
  for (int64_t i = (int64_t)blockIdx.x * kGateThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kGateThreads) {
    int64_t row;
    int l;
    const int64_t o = gate_off<V>(g, i, &row, &l);
    float gv[V], zv[V], yv[V], dyv[V];
    ld<V>(dout_z + o, gv);
    ld<V>(z + o, zv);
    ld<V>(y + o, yv);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      dyv[e] = gv[e] * silu_f(zv[e]);
      zv[e] = gv[e] * yv[e] * silu_grad_f(zv[e]);
    }
    st<V>(dy + row * g.L + l, dyv);
    st<V>(dz + o, zv);
  }
}

namespace {

GateGeom geom(const ss2d_scan_desc* d) {
  return GateGeom{d->dim, d->seqlen, (int64_t)d->batch * d->dim, d->out_batch_stride, d->out_dim_stride};
}

// 8-element accesses need every row of every operand to start 16 bytes aligned
bool vec_ok(const ss2d_scan_desc* d, std::initializer_list<const void*> ptrs) {
  if ((d->seqlen | d->out_batch_stride | d->out_dim_stride) & 7) return false;
  for (const void* p : ptrs)
    if (reinterpret_cast<uintptr_t>(p) & 15) return false;
  return true;
}

unsigned grid_for(const GateGeom& g, int V) {
  const int64_t total = g.rows * (g.L / V);
  const int64_t cap = (int64_t)sm_count_current_device() * 8;          // 8 CTAs of 256 threads per SM, grid-stride beyond
  const int64_t n = (total + kGateThreads - 1) / kGateThreads;
  return (unsigned)(n < cap ? n : cap);
}

template <typename TI, typename TO>
cudaError_t fwd_typed(const ss2d_scan_desc* d, const void* y, const void* z, void* out_z, cudaStream_t s) {
  const GateGeom g = geom(d);
  const TO* yp = static_cast<const TO*>(y);
  const TI* zp = static_cast<const TI*>(z);
  TO* op = static_cast<TO*>(out_z);
  if (vec_ok(d, {y, z, out_z})) scan_gate_fwd_kernel<TI, TO, 8><<<grid_for(g, 8), kGateThreads, 0, s>>>(yp, zp, op, g);
  else scan_gate_fwd_kernel<TI, TO, 1><<<grid_for(g, 1), kGateThreads, 0, s>>>(yp, zp, op, g);
  return cudaGetLastError();
}

template <typename TI, typename TO>
cudaError_t bwd_typed(const ss2d_scan_desc* d, const void* dout_z, const void* z, const void* y, float* dy, void* dz,
                      cudaStream_t s) {
  const GateGeom g = geom(d);
  const TO* gp = static_cast<const TO*>(dout_z);
  const TO* yp = static_cast<const TO*>(y);
  const TI* zp = static_cast<const TI*>(z);
  TI* dzp = static_cast<TI*>(dz);
  if (vec_ok(d, {dout_z, z, y, dy, dz})) scan_gate_bwd_kernel<TI, TO, 8><<<grid_for(g, 8), kGateThreads, 0, s>>>(gp, zp, yp, dy, dzp, g);
  else scan_gate_bwd_kernel<TI, TO, 1><<<grid_for(g, 1), kGateThreads, 0, s>>>(gp, zp, yp, dy, dzp, g);
  return cudaGetLastError();
}

}  // namespace

// io / out dtype pairs the descriptor allows: out == io, or out fp32
cudaError_t scan_gate_fwd_launch(const ss2d_scan_desc* d, const void* y, const void* z, void* out_z, cudaStream_t s) {
  const bool o32 = d->out_dtype == SS2D_F32;
  switch (d->io_dtype) {
    case SS2D_F32: return fwd_typed<float, float>(d, y, z, out_z, s);
    case SS2D_F16: return o32 ? fwd_typed<__half, float>(d, y, z, out_z, s) : fwd_typed<__half, __half>(d, y, z, out_z, s);
    default:
      return o32 ? fwd_typed<__nv_bfloat16, float>(d, y, z, out_z, s)
                 : fwd_typed<__nv_bfloat16, __nv_bfloat16>(d, y, z, out_z, s);
  }
}

cudaError_t scan_gate_bwd_launch(const ss2d_scan_desc* d, const void* dout_z, const void* z, const void* y, float* dy, void* dz,
                                 cudaStream_t s) {
  const bool o32 = d->out_dtype == SS2D_F32;
  switch (d->io_dtype) {
    case SS2D_F32: return bwd_typed<float, float>(d, dout_z, z, y, dy, dz, s);
    case SS2D_F16:
      return o32 ? bwd_typed<__half, float>(d, dout_z, z, y, dy, dz, s) : bwd_typed<__half, __half>(d, dout_z, z, y, dy, dz, s);
    default:
      return o32 ? bwd_typed<__nv_bfloat16, float>(d, dout_z, z, y, dy, dz, s)
                 : bwd_typed<__nv_bfloat16, __nv_bfloat16>(d, dout_z, z, y, dy, dz, s);
  }
}

}  // namespace ss2d
