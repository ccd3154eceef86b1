// One recurrent step of the selective scan (mamba_ssm's selective_state_update), updating the state in place:
//   t = dt[b,d] + dt_bias[d] (softplus20 when asked),  h[b,d,n] = exp(t A[d,n]) h[b,d,n] + t x[b,d] B[b,g,n],
//   out[b,d] = sum_n C[b,g,n] h[b,d,n] + D[d] x[b,d]  (times silu(z[b,d]) with a gate),  g = d / (dim / n_groups).
// A row (b, d) is owned by a segment of P lanes, each holding S consecutive states in registers; the sum over n is a
// shuffle reduction inside the segment. dstate <= 32: S = 4, P = ceil(dstate / 4) rounded up to a power of two, so a warp
// covers 32 / P rows (32 at dstate 1); dstate > 32: P = 32 (one warp per row), S = ceil(dstate / 32) rounded up to a power
// of two. The state moves min(S, 4) floats per access (128-bit at S >= 4) when dstate is a multiple of that width, else one.
// HBM-bound: 8 bytes of state per (b, d, n); A, B and C are re-read by many rows and come from L1 / L2.
#include "common.cuh"
#include "scan_params.h"

namespace ss2d {

constexpr int kStepThreads = 128;

namespace {

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ void from_f(float* p, float v) { *p = v; }
__device__ __forceinline__ void from_f(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void from_f(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

template <int V>
__device__ __forceinline__ void ld_state(const float* p, float (&h)[V]) {
  if constexpr (V == 4) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    h[0] = v.x; h[1] = v.y; h[2] = v.z; h[3] = v.w;
  } else if constexpr (V == 2) {
    const float2 v = *reinterpret_cast<const float2*>(p);
    h[0] = v.x; h[1] = v.y;
  } else {
    h[0] = *p;
  }
}
template <int V>
__device__ __forceinline__ void st_state(float* p, const float (&h)[V]) {
  if constexpr (V == 4) *reinterpret_cast<float4*>(p) = make_float4(h[0], h[1], h[2], h[3]);
  else if constexpr (V == 2) *reinterpret_cast<float2*>(p) = make_float2(h[0], h[1]);
  else *p = h[0];
}

}  // namespace

// T: io dtype; S states per lane, P lanes per row (a power of two), VEC: dstate % min(S, 4) == 0 (vector state accesses)
template <typename T, int S, int P, bool VEC>
__global__ void __launch_bounds__(kStepThreads) ssm_step_kernel(const StepParams p) {
  constexpr int V = VEC ? (S < 4 ? S : 4) : 1;
  const int lane = threadIdx.x & 31, j = lane % P;
  const int64_t row = ((int64_t)blockIdx.x * (kStepThreads / 32) + threadIdx.x / 32) * (32 / P) + lane / P;
  const bool live = row < p.rows;
  const int64_t b = live ? row / p.dim : 0;
  const int d = live ? (int)(row - b * p.dim) : 0;
  const int64_t io = b * p.io_bs + d;
  float xv = 0.f, acc = 0.f;
  if (live) {
    xv = to_f(__ldg(static_cast<const T*>(p.x) + io));
    float t = to_f(__ldg(static_cast<const T*>(p.dt) + io)) + (p.bias ? __ldg(p.bias + d) : 0.f);
    if (p.softplus) t = softplus20(t);
    const float tx = t * xv;
    const int g = d / p.dpg;
    float* h_row = p.state + row * p.dstate;
    const float* A_row = p.A + (int64_t)d * p.dstate;
    const T* B_row = static_cast<const T*>(p.B) + b * p.B_bs + g * p.B_gs;
    const T* C_row = static_cast<const T*>(p.C) + b * p.C_bs + g * p.C_gs;
#pragma unroll
    for (int v = 0; v < S; v += V) {
      const int n = j * S + v;
      if (n < p.dstate) {                 // VEC: dstate % V == 0, so the whole vector is in range
        float h[V];
        ld_state<V>(h_row + n, h);
#pragma unroll
        for (int e = 0; e < V; ++e) {
          const float A2 = __ldg(A_row + n + e) * kLog2e;
          h[e] = fmaf(ex2f(t * A2), h[e], tx * to_f(__ldg(B_row + n + e)));
          acc = fmaf(h[e], to_f(__ldg(C_row + n + e)), acc);
        }
        st_state<V>(h_row + n, h);
      }
    }
  }
#pragma unroll
  for (int o = P / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (live && j == 0) {
    float y = p.D ? fmaf(__ldg(p.D + d), xv, acc) : acc;
    if (p.z) y *= silu_f(to_f(__ldg(static_cast<const T*>(p.z) + io)));
    from_f(static_cast<T*>(p.out) + io, y);
  }
}

namespace {

template <typename T, int S, int P>
cudaError_t launch_regime(const StepParams& p, cudaStream_t s) {
  constexpr int V = S < 4 ? S : 4;
  const int64_t warps = (p.rows + 32 / P - 1) / (32 / P);
  const unsigned grid = (unsigned)((warps + kStepThreads / 32 - 1) / (kStepThreads / 32));
  if (p.dstate % V == 0) ssm_step_kernel<T, S, P, true><<<grid, kStepThreads, 0, s>>>(p);
  else ssm_step_kernel<T, S, P, false><<<grid, kStepThreads, 0, s>>>(p);
  return cudaGetLastError();
}

// the lane mapping follows from dstate alone
template <typename T>
cudaError_t launch_typed(const StepParams& p, cudaStream_t s) {
  const int n = p.dstate;
  if (n <= 4) return launch_regime<T, 4, 1>(p, s);
  if (n <= 8) return launch_regime<T, 4, 2>(p, s);
  if (n <= 16) return launch_regime<T, 4, 4>(p, s);
  if (n <= 32) return launch_regime<T, 4, 8>(p, s);
  if (n <= 64) return launch_regime<T, 2, 32>(p, s);
  if (n <= 128) return launch_regime<T, 4, 32>(p, s);
  return launch_regime<T, 8, 32>(p, s);
}

}  // namespace

cudaError_t ssm_step_launch(const StepParams& p, int io_dtype, cudaStream_t s) {
  switch (io_dtype) {
    case SS2D_F32: return launch_typed<float>(p, s);
    case SS2D_F16: return launch_typed<__half>(p, s);
    default: return launch_typed<__nv_bfloat16>(p, s);
  }
}

}  // namespace ss2d
