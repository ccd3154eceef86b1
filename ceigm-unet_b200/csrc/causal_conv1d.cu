// Causal depthwise 1-D convolution of Mamba blocks, with the contract of causal-conv1d 1.1.x (channel-first x):
//   forward   out[b,d,l] = act(bias[d] + sum_{k<W} w[d,k] x[b,d,l-(W-1)+k]),  x = 0 at negative positions,
//             act = SiLU or the identity;
//   backward  g = dout act'(pre) with pre recomputed from x,  dx[l] = sum_k w[d,k] g[l+(W-1)-k] (g = 0 past L - 1),
//             dweight[d,k] = sum_{b,l} g[b,d,l] x[b,d,l-(W-1)+k],  dbias[d] = sum_{b,l} g[b,d,l];
//   update    one decode position: the W-value state row shifts left by one, x enters its last slot,
//             out = act(bias + w . state).
// All math in fp32; out / dx are rounded once to the io dtype, dweight / dbias are fp32.
// Lane mapping (forward and backward): a warp owns a segment of kSeg = 256 consecutive positions of one row (b, d), a lane
// kRun = 8 of them. The W - 1 inputs before a lane's run come from the lane below by shuffle; lane 0 reloads them (L1 / L2
// hits: the previous segment's warp read them). In the backward the W - 1 values of g after a run come from the lane above;
// lane 31 recomputes them from x and dout. Weight and bias stay in registers. VEC: x, out / dout / dx 16-byte aligned with
// strides that are multiples of 16 bytes, so a run moves in 128-bit accesses (two for fp32); else element by element. A run
// that crosses the row's end always goes element by element.
// The backward grid is (dim, slabs): the warps of a CTA walk the segments of one channel over the batch, keep the W + 1 sums
// in registers, fold them with warp shuffles and shared memory, and store one partial per slab; a fixed-order finalize pass
// adds the slabs. When one slab covers the channel the CTA stores dweight / dbias itself and the finalize pass is skipped.
// No atomics: the gradients are bit-identical from call to call.
// HBM-bound: the forward reads x and writes out (2 s bytes per element, s = element size), the backward reads x and dout and
// writes dx (3 s).
// Instantiations (52), the SiLU being a uniform runtime flag:
//   conv1d_fwd_kernel<T, W, VEC>, conv1d_bwd_kernel<T, W, VEC>: T in {float, __half, __nv_bfloat16} x W in {2, 3, 4} x
//     VEC in {false, true} (18 each);
//   conv1d_update_kernel<T, W, VEC>: the same T x (W, VEC) in {(2, false), (2, true), (3, false), (4, false), (4, true)} (15;
//     VEC stores the state row in one 32-, 64- or 128-bit access, which a 3-value row cannot have, and loads it in one at
//     width 4; at width 2 only the value that survives the shift is read);
//   conv1d_wgrad_finalize_kernel (1).
#include <cstring>

#include "common.cuh"
#include "conv1d_params.h"

namespace ss2d {

constexpr int kConvThreads = 128;
constexpr int kRun = 8;
constexpr int kSeg = 32 * kRun;

namespace {

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ void from_f(float* p, float v) { *p = v; }
__device__ __forceinline__ void from_f(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void from_f(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// a full run at a 16-byte aligned address
__device__ __forceinline__ void ld_run(const float* p, float (&v)[kRun]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld_run(const __half* p, float (&v)[kRun]) {
  const uint4 raw = __ldg(reinterpret_cast<const uint4*>(p));
  const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void ld_run(const __nv_bfloat16* p, float (&v)[kRun]) {
  const uint4 raw = __ldg(reinterpret_cast<const uint4*>(p));
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void st_run(float* p, const float (&v)[kRun]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void st_run(__half* p, const float (&v)[kRun]) {
  uint4 raw;
  __half2* h = reinterpret_cast<__half2*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = raw;
}
__device__ __forceinline__ void st_run(__nv_bfloat16* p, const float (&v)[kRun]) {
  uint4 raw;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = raw;
}

// positions [l0, l0 + kRun) of a row of length L; zeros past its end
template <typename T, bool VEC>
__device__ __forceinline__ void load_run(const T* row, int64_t l0, int64_t L, float (&v)[kRun]) {
  if (VEC && l0 + kRun <= L) {
    ld_run(row + l0, v);
  } else {
#pragma unroll
    for (int e = 0; e < kRun; ++e) v[e] = l0 + e < L ? to_f(row[l0 + e]) : 0.f;
  }
}
template <typename T, bool VEC>
__device__ __forceinline__ void store_run(T* row, int64_t l0, int64_t L, const float (&v)[kRun]) {
  if (VEC && l0 + kRun <= L) {
    st_run(row + l0, v);
  } else {
#pragma unroll
    for (int e = 0; e < kRun; ++e)
      if (l0 + e < L) from_f(row + l0 + e, v[e]);
  }
}

// v[0 .. W-2]: the W - 1 inputs before the lane's run, v[W-1 ..]: the run
template <typename T, int W>
__device__ __forceinline__ void window(const T* row, int64_t l0, int lane, const float (&own)[kRun], float (&v)[W - 1 + kRun]) {
#pragma unroll
  for (int j = 0; j < W - 1; ++j) {
    float h = __shfl_up_sync(0xffffffffu, own[kRun - (W - 1) + j], 1);
    if (lane == 0) {
      const int64_t l = l0 - (W - 1) + j;
      h = l >= 0 ? to_f(row[l]) : 0.f;
    }
    v[j] = h;
  }
#pragma unroll
  for (int e = 0; e < kRun; ++e) v[W - 1 + e] = own[e];
}

// bias + w . (W consecutive inputs), in the order the forward, the backward and the update all use
template <int W>
__device__ __forceinline__ float pre_act(const float (&w)[W], float bias, const float* v) {
  float acc = bias;
#pragma unroll
  for (int k = 0; k < W; ++k) acc = fmaf(w[k], v[k], acc);
  return acc;
}

template <int W>
__device__ __forceinline__ void load_weights(const Conv1dParams& p, int d, float (&w)[W], float& bias) {
#pragma unroll
  for (int k = 0; k < W; ++k) w[k] = __ldg(p.w + (int64_t)d * W + k);
  bias = p.bias ? __ldg(p.bias + d) : 0.f;
}

}  // namespace

template <typename T, int W, bool VEC>
__global__ void __launch_bounds__(kConvThreads) conv1d_fwd_kernel(const Conv1dParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t spr = (p.L + kSeg - 1) / kSeg;                   // segments per row
  const int64_t gw = (int64_t)blockIdx.x * (kConvThreads / 32) + threadIdx.x / 32;
  const int64_t row = gw / spr;
  if (row >= (int64_t)p.batch * p.dim) return;                   // uniform over the warp
  const int64_t b = row / p.dim;
  const int d = (int)(row - b * p.dim);
  const int64_t l0 = (gw - row * spr) * kSeg + lane * kRun;
  const T* xr = static_cast<const T*>(p.x) + b * p.x_bs + d * p.x_ds;
  float w[W], bias;
  load_weights<W>(p, d, w, bias);
  float own[kRun], v[W - 1 + kRun], o[kRun];
  load_run<T, VEC>(xr, l0, p.L, own);
  window<T, W>(xr, l0, lane, own, v);
#pragma unroll
  for (int e = 0; e < kRun; ++e) {
    const float a = pre_act<W>(w, bias, v + e);
    o[e] = p.silu ? silu_f(a) : a;
  }
  store_run<T, VEC>(static_cast<T*>(p.out) + b * p.o_bs + d * p.o_ds, l0, p.L, o);
}

template <typename T, int W, bool VEC>
__global__ void __launch_bounds__(kConvThreads) conv1d_bwd_kernel(const Conv1dParams p) {
  constexpr int kWarps = kConvThreads / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int d = blockIdx.x;
  const int64_t spr = (p.L + kSeg - 1) / kSeg, total = (int64_t)p.batch * spr;
  const int64_t per = (total + p.slabs - 1) / p.slabs;
  const int64_t s0 = blockIdx.y * per, s1 = s0 + per < total ? s0 + per : total;
  float w[W], bias;
  load_weights<W>(p, d, w, bias);
  float acc[W + 1];
#pragma unroll
  for (int k = 0; k <= W; ++k) acc[k] = 0.f;
  for (int64_t s = s0 + warp; s < s1; s += kWarps) {
    const int64_t b = s / spr;
    const int64_t l0 = (s - b * spr) * kSeg + lane * kRun;
    const T* xr = static_cast<const T*>(p.x) + b * p.x_bs + (int64_t)d * p.x_ds;
    const T* gr = static_cast<const T*>(p.dout) + b * p.o_bs + (int64_t)d * p.o_ds;
    float own[kRun], v[W - 1 + kRun], go[kRun], g[kRun + W - 1], dx[kRun];
    load_run<T, VEC>(xr, l0, p.L, own);
    load_run<T, VEC>(gr, l0, p.L, go);              // dout: zero past the row's end, so g is too
    window<T, W>(xr, l0, lane, own, v);
#pragma unroll
    for (int e = 0; e < kRun; ++e) g[e] = p.silu ? go[e] * silu_grad_f(pre_act<W>(w, bias, v + e)) : go[e];
    // g after the run: the lane above holds it, lane 31 recomputes it
#pragma unroll
    for (int j = 0; j < W - 1; ++j) {
      float gn = __shfl_down_sync(0xffffffffu, g[j], 1);
      if (lane == 31) {
        const int64_t l = l0 + kRun + j;
        gn = 0.f;
        if (l < p.L) {
          gn = to_f(gr[l]);
          if (p.silu) {
            float u[W];
#pragma unroll
            for (int k = 0; k < W; ++k) u[k] = to_f(xr[l - (W - 1) + k]);     // l >= kRun > W - 1
            gn *= silu_grad_f(pre_act<W>(w, bias, u));
          }
        }
      }
      g[kRun + j] = gn;
    }
#pragma unroll
    for (int e = 0; e < kRun; ++e) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < W; ++k) a = fmaf(w[k], g[e + (W - 1) - k], a);
      dx[e] = a;
#pragma unroll
      for (int k = 0; k < W; ++k) acc[k] = fmaf(g[e], v[e + k], acc[k]);
      acc[W] += g[e];
    }
    store_run<T, VEC>(static_cast<T*>(p.out) + b * p.o_bs + (int64_t)d * p.o_ds, l0, p.L, dx);
  }
  __shared__ float s_red[kWarps][W + 1];
#pragma unroll
  for (int k = 0; k <= W; ++k) {
    float a = acc[k];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) s_red[warp][k] = a;
  }
  __syncthreads();
  if (threadIdx.x <= W) {
    const int k = threadIdx.x;
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < kWarps; ++i) a += s_red[i][k];
    if (p.slabs > 1) p.part[((int64_t)d * p.slabs + blockIdx.y) * (W + 1) + k] = a;
    else if (k < W) p.dw[(int64_t)d * W + k] = a;
    else if (p.db) p.db[d] = a;
  }
}

__global__ void conv1d_wgrad_finalize_kernel(const Conv1dParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int W1 = p.width + 1;
  if (i >= (int64_t)p.dim * W1) return;
  const int64_t c = i / W1;
  const int k = (int)(i - c * W1);
  float s = 0.f;
  for (int j = 0; j < p.slabs; ++j) s += p.part[(c * p.slabs + j) * W1 + k];
  if (k < p.width) p.dw[c * p.width + k] = s;
  else if (p.db) p.db[c] = s;
}

namespace {
template <int BYTES> struct RawVec;
template <> struct RawVec<4> { using type = unsigned int; };
template <> struct RawVec<8> { using type = uint2; };
template <> struct RawVec<16> { using type = uint4; };
}  // namespace

// VEC: the state row (W elements) moves in one access; the state base is aligned to W * sizeof(T)
template <typename T, int W, bool VEC>
__global__ void __launch_bounds__(kConvThreads) conv1d_update_kernel(const Conv1dParams p) {
  const int64_t row = (int64_t)blockIdx.x * kConvThreads + threadIdx.x;
  if (row >= (int64_t)p.batch * p.dim) return;
  const int64_t b = row / p.dim;
  const int d = (int)(row - b * p.dim);
  T* sr = static_cast<T*>(p.state) + row * W;
  T s[W];
  if constexpr (VEC) {
    using V = typename RawVec<W * sizeof(T)>::type;
    const V raw = *reinterpret_cast<const V*>(sr);
    memcpy(s, &raw, sizeof(V));
  } else {
#pragma unroll
    for (int k = 0; k < W; ++k) s[k] = sr[k];
  }
#pragma unroll
  for (int k = 0; k < W - 1; ++k) s[k] = s[k + 1];
  s[W - 1] = static_cast<const T*>(p.x)[b * p.x_bs + d * p.x_ds];
  if constexpr (VEC) {
    using V = typename RawVec<W * sizeof(T)>::type;
    V raw;
    memcpy(&raw, s, sizeof(V));
    *reinterpret_cast<V*>(sr) = raw;
  } else {
#pragma unroll
    for (int k = 0; k < W; ++k) sr[k] = s[k];
  }
  float w[W], bias, v[W];
  load_weights<W>(p, d, w, bias);
#pragma unroll
  for (int k = 0; k < W; ++k) v[k] = to_f(s[k]);
  const float a = pre_act<W>(w, bias, v);
  from_f(static_cast<T*>(p.out) + b * p.o_bs + d * p.o_ds, p.silu ? silu_f(a) : a);
}

namespace {

bool vec16(const void* ptr, int64_t s0, int64_t s1, int64_t es) {
  const int64_t n = 16 / es;
  return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && s0 % n == 0 && s1 % n == 0;
}

template <typename T, int W>
cudaError_t fwd_typed(const Conv1dParams& p, cudaStream_t s) {
  const int64_t warps = (int64_t)p.batch * p.dim * ((p.L + kSeg - 1) / kSeg);
  const unsigned grid = (unsigned)((warps + kConvThreads / 32 - 1) / (kConvThreads / 32));
  if (vec16(p.x, p.x_bs, p.x_ds, sizeof(T)) && vec16(p.out, p.o_bs, p.o_ds, sizeof(T)))
    conv1d_fwd_kernel<T, W, true><<<grid, kConvThreads, 0, s>>>(p);
  else
    conv1d_fwd_kernel<T, W, false><<<grid, kConvThreads, 0, s>>>(p);
  return cudaGetLastError();
}

template <typename T, int W>
cudaError_t bwd_typed(const Conv1dParams& p, cudaStream_t s) {
  const dim3 grid(p.dim, p.slabs);
  if (vec16(p.x, p.x_bs, p.x_ds, sizeof(T)) && vec16(p.dout, p.o_bs, p.o_ds, sizeof(T)) &&
      vec16(p.out, p.o_bs, p.o_ds, sizeof(T)))
    conv1d_bwd_kernel<T, W, true><<<grid, kConvThreads, 0, s>>>(p);
  else
    conv1d_bwd_kernel<T, W, false><<<grid, kConvThreads, 0, s>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || p.slabs == 1) return e;
  const int64_t n = (int64_t)p.dim * (W + 1);
  conv1d_wgrad_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(p);
  return cudaGetLastError();
}

template <typename T, int W>
cudaError_t update_typed(const Conv1dParams& p, cudaStream_t s) {
  const unsigned grid = (unsigned)(((int64_t)p.batch * p.dim + kConvThreads - 1) / kConvThreads);
  if constexpr (W != 3) {
    if ((reinterpret_cast<uintptr_t>(p.state) & (W * sizeof(T) - 1)) == 0) {
      conv1d_update_kernel<T, W, true><<<grid, kConvThreads, 0, s>>>(p);
      return cudaGetLastError();
    }
  }
  conv1d_update_kernel<T, W, false><<<grid, kConvThreads, 0, s>>>(p);
  return cudaGetLastError();
}

enum class Op { kFwd, kBwd, kUpdate };

template <Op OP, typename T, int W>
cudaError_t run(const Conv1dParams& p, cudaStream_t s) {
  if constexpr (OP == Op::kFwd) return fwd_typed<T, W>(p, s);
  else if constexpr (OP == Op::kBwd) return bwd_typed<T, W>(p, s);
  else return update_typed<T, W>(p, s);
}

template <Op OP, typename T>
cudaError_t by_width(const Conv1dParams& p, cudaStream_t s) {
  switch (p.width) {
    case 2: return run<OP, T, 2>(p, s);
    case 3: return run<OP, T, 3>(p, s);
    default: return run<OP, T, 4>(p, s);
  }
}

template <Op OP>
cudaError_t by_dtype(const Conv1dParams& p, int io_dtype, cudaStream_t s) {
  switch (io_dtype) {
    case SS2D_F32: return by_width<OP, float>(p, s);
    case SS2D_F16: return by_width<OP, __half>(p, s);
    default: return by_width<OP, __nv_bfloat16>(p, s);
  }
}

}  // namespace

// partial slabs per channel: about 8 CTAs per SM over all channels, at least one segment per warp, at most 65535 (grid y)
int conv1d_bwd_slabs(int batch, int dim, int64_t L) {
  const int64_t total = (int64_t)batch * ((L + kSeg - 1) / kSeg);
  int64_t s = (148 * 8 + dim - 1) / dim;
  const int64_t most = (total + kConvThreads / 32 - 1) / (kConvThreads / 32);
  if (s > most) s = most;
  if (s > 65535) s = 65535;
  return s < 1 ? 1 : (int)s;
}

cudaError_t conv1d_fwd_launch(const Conv1dParams& p, int io_dtype, cudaStream_t s) { return by_dtype<Op::kFwd>(p, io_dtype, s); }
// p.slabs = conv1d_bwd_slabs(...); p.part is read when p.slabs > 1
cudaError_t conv1d_bwd_launch(const Conv1dParams& p, int io_dtype, cudaStream_t s) { return by_dtype<Op::kBwd>(p, io_dtype, s); }
cudaError_t conv1d_update_launch(const Conv1dParams& p, int io_dtype, cudaStream_t s) {
  return by_dtype<Op::kUpdate>(p, io_dtype, s);
}

}  // namespace ss2d
