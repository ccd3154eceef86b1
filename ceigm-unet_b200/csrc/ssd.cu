// Mamba-2 chunked selective scan (SSD, "state space duality"), forward, with the contract of mamba_ssm 2.x's
// mamba_chunk_scan_combined. Per (batch b, head k) with P = headdim, N = dstate, t_l = clamp(softplus?(dt_l + dt_bias_k)):
//   H_l = exp(t_l A_k) H_{l-1} + t_l x_l (x) B_l   (P x N),   y_l = C_l . H_l + D x_l,   out_l = y_l silu(z_l) (with z).
// Chunks of Q positions, a_l = t_l A_k, cum_l = inclusive cumsum of a within the chunk:
//   ssd_chunk_state_kernel  t, cum (workspace) and S_c = sum_{s in c} exp(cum_last - cum_s) t_s x_s (x) B_s: a P x N product
//                           over Q;
//   ssd_state_pass_kernel   sequential over the chunks of one (b, k): the slot of S_c takes H_c, the state entering chunk c,
//                           then H_{c+1} = exp(cum_last,c) H_c + S_c, with H_0 = h0 (zeros when absent); H_nchunks -> hT;
//   ssd_chunk_out_kernel    per 64-position block of a chunk: y_l = exp(cum_l) C_l . H_c + sum_{s <= l in c} (C_l . B_s)
//                           exp(cum_l - cum_s) t_s x_s + D x_l, then the z gate. The masked (s > l) exponents are replaced by
//                           -inf before the exponential, so they give 0 and never inf * 0.
// The products run on the tensor cores through warp-level mma.sync, from fp32 tiles in shared memory whose fragments are
// converted as they are loaded: 16-bit I/O uses m16n8k16 in the I/O dtype with fp32 accumulation, and computed operands (the
// decayed B rows, the states, the masked scores) are rounded to the I/O dtype first; fp32 I/O uses m16n8k8 TF32 with a 3-term
// hi / lo split (hi*hi + hi*lo + lo*hi), which keeps fp32 accuracy. Cumsums, exponentials (ex2f(v log2 e), as in the scan
// kernels) and state passing are fp32. No atomics: results are bit-identical from call to call.
// Chunk size and dstate are runtime loop bounds (64-position blocks, 64-state slices in steps of 16).
// Backward (nine launches): the forward's first two kernels recompute t, cum and the chunk-entry states (no state is saved),
//   ssd_chunk_state_kernel<BWD> forms R_c = sum_l exp(cum_l) dy_l (x) C_l, ssd_state_pass_bwd_kernel runs the state adjoint
//   backwards over the chunks (dH_c = exp(cum_last,c) dH_{c+1} + R_c, dH_nchunks = dhT, dH_0 -> dh0), ssd_chunk_bwd_kernel
//   forms the chunk-local gradients in its target and source roles, ssd_dt_bwd_kernel turns the per-position terms into
//   d a (a reverse cumsum within the chunk) and ddt, and two finalize kernels add the per-head and per-block partials in a
//   fixed order (dB, dC over the heads of a group; dA, dD, ddt_bias over batch and positions).
// Instantiations (54): ssd_chunk_state_kernel<T, P, BWD>, ssd_chunk_out_kernel<T, P>, ssd_chunk_bwd_kernel<T, P, SRC>, with
// T in {float, __half, __nv_bfloat16} x P in {32, 64, 128} (45); ssd_dt_bwd_kernel<T>, ssd_bc_grad_kernel<T> (6);
// ssd_state_pass_kernel, ssd_state_pass_bwd_kernel, ssd_param_grad_kernel (3).
#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "ssd_params.h"

namespace ss2d {

constexpr int kSsdThreads = 128;   // 4 warps; a warp owns 16 rows of each 64-row product
constexpr int kBlk = 64;           // positions per block, states per slice
constexpr int kPassThreads = 256;

namespace {

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ void from_f(float* p, float v) { *p = v; }
__device__ __forceinline__ void from_f(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void from_f(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
// a computed operand rounded to the I/O dtype (the identity for fp32, whose rounding is the hi / lo split)
template <typename T> __device__ __forceinline__ float round_io(float v) { T r; from_f(&r, v); return to_f(r); }

__device__ __forceinline__ uint32_t pack2(float lo, float hi, __half) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi, __nv_bfloat16) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ void split(float v, uint32_t& hi, uint32_t& lo) {
  hi = tf32(v);
  lo = tf32(v - __uint_as_float(hi));
}

__device__ __forceinline__ void mma16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1, __half) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1, __nv_bfloat16) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// acc[nt] (16 x 8 tile nt, mma C-fragment layout) += A (16 x K) B (K x 8 NT), both fp32 in shared memory:
// A(m, k) = A[m * am + k * ak], B(k, n) = B[k * bk + n * bn]. K is a multiple of 16.
template <typename T, int NT>
__device__ __forceinline__ void warp_gemm(float (&acc)[NT][4], const float* A, int am, int ak, const float* B, int bk, int bn,
                                          int K) {
  const int g = (threadIdx.x & 31) >> 2, t = threadIdx.x & 3;
  if constexpr (std::is_same<T, float>::value) {
    for (int k0 = 0; k0 < K; k0 += 8) {
      const float* a = A + (k0 + t) * ak + g * am;
      uint32_t ah[4], al[4];
      split(a[0], ah[0], al[0]);
      split(a[8 * am], ah[1], al[1]);
      split(a[4 * ak], ah[2], al[2]);
      split(a[8 * am + 4 * ak], ah[3], al[3]);
      const float* b = B + (k0 + t) * bk + g * bn;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        uint32_t bh0, bl0, bh1, bl1;
        split(b[nt * 8 * bn], bh0, bl0);
        split(b[nt * 8 * bn + 4 * bk], bh1, bl1);
        mma_tf32(acc[nt], al, bh0, bh1);
        mma_tf32(acc[nt], ah, bl0, bl1);
        mma_tf32(acc[nt], ah, bh0, bh1);
      }
    }
  } else {
    for (int k0 = 0; k0 < K; k0 += 16) {
      const float* a = A + (k0 + 2 * t) * ak + g * am;
      uint32_t af[4];
      af[0] = pack2(a[0], a[ak], T());
      af[1] = pack2(a[8 * am], a[8 * am + ak], T());
      af[2] = pack2(a[8 * ak], a[9 * ak], T());
      af[3] = pack2(a[8 * am + 8 * ak], a[8 * am + 9 * ak], T());
      const float* b = B + (k0 + 2 * t) * bk + g * bn;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const float* bb = b + nt * 8 * bn;
        mma16(acc[nt], af, pack2(bb[0], bb[bk], T()), pack2(bb[8 * bk], bb[9 * bk], T()), T());
      }
    }
  }
}

__device__ __forceinline__ float proc_dt(const SsdParams& p, float v, int h) {
  if (p.dt_bias) v += p.dt_bias[h];
  if (p.softplus) v = softplus20(v);
  return fminf(fmaxf(v, p.dt_min), p.dt_max);
}

}  // namespace

// grid (nchunks, heads, batch); dynamic shared memory: cum and t [256] each, Xs [64][P + 8], Bw [64][72] (row pitches that
// keep the fragment loads free of bank conflicts).
// BWD: the same product for the backward's state adjoint, R_c = sum_l exp(cum_l) dy_l (x) C_l with dy = dout silu(z); t and
// cum are recomputed with the forward's arithmetic and not stored.
template <typename T, int P, bool BWD>
__global__ void __launch_bounds__(kSsdThreads, 1) ssd_chunk_state_kernel(const SsdParams p) {
  constexpr int NT = P / 8, ldx = P + 8, ldw = kBlk + 8;
  extern __shared__ float smem[];
  float* cum_s = smem;
  float* t_s = cum_s + 256;
  float* Xs = t_s + 256;
  float* Bw = Xs + kBlk * ldx;
  const int c = blockIdx.x, h = blockIdx.y, b = blockIdx.z, tid = threadIdx.x, warp = tid >> 5;
  const int Q = p.Q, N = p.N, grp = h / (p.heads / p.groups);
  const int64_t bh = (int64_t)b * p.heads + h, l_chunk = (int64_t)c * Q;
  const float A = p.A[h];
  for (int i = tid; i < Q; i += kSsdThreads) {
    const int64_t l = l_chunk + i;
    const float t = l < p.L ? proc_dt(p, to_f(static_cast<const T*>(p.dt)[b * p.dt_b + l * p.dt_l + h * p.dt_h]), h) : 0.f;
    t_s[i] = t;
    cum_s[i] = t * A;
  }
  __syncthreads();
  for (int off = 1; off < Q; off <<= 1) {   // Hillis-Steele inclusive scan, a fixed order of additions
    float v[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int i = tid + e * kSsdThreads;
      v[e] = i < Q && i >= off ? cum_s[i - off] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int i = tid + e * kSsdThreads;
      if (i < Q) cum_s[i] += v[e];
    }
    __syncthreads();
  }
  const int64_t ws = bh * p.nchunks * Q + l_chunk;
  if (!BWD)
    for (int i = tid; i < Q; i += kSsdThreads) {
      p.t[ws + i] = t_s[i];
      p.cum[ws + i] = cum_s[i];
    }
  const float cum_last = cum_s[Q - 1];
  const T* x = static_cast<const T*>(BWD ? p.dout : p.x) + b * (BWD ? p.o_b : p.x_b) + h * (BWD ? p.o_h : p.x_h);
  const int64_t x_l = BWD ? p.o_l : p.x_l;
  const T* z = BWD && p.z ? static_cast<const T*>(p.z) + b * p.z_b + h * p.z_h : nullptr;
  const T* Bm = static_cast<const T*>(BWD ? p.C : p.B) + b * p.bc_b + grp * p.bc_g;
  float* S = (BWD ? p.R : p.states) + (bh * p.nchunks + c) * P * N;
  const int g = (tid & 31) >> 2, tq = tid & 3;
  for (int n0 = 0; n0 < N; n0 += kBlk) {
    const int nw = min(kBlk, N - n0);
    float acc[NT][4] = {};
    for (int s0 = 0; s0 < Q && l_chunk + s0 < p.L; s0 += kBlk) {
      for (int e = tid; e < kBlk * P; e += kSsdThreads) {
        const int r = e / P, q = e % P;
        const int64_t l = l_chunk + s0 + r;
        float v = 0.f;
        if (l < p.L) {
          v = to_f(x[l * x_l + q]);
          if (z) v *= silu_f(to_f(z[l * p.z_l + q]));
        }
        Xs[r * ldx + q] = v;
      }
      for (int e = tid; e < kBlk * kBlk; e += kSsdThreads) {
        const int r = e / kBlk, n = e % kBlk;
        const int64_t l = l_chunk + s0 + r;
        float v = 0.f;
        if (l < p.L && n < nw)
          v = round_io<T>((BWD ? ex2f(cum_s[s0 + r] * kLog2e) : ex2f((cum_last - cum_s[s0 + r]) * kLog2e) * t_s[s0 + r]) *
                          to_f(Bm[l * p.bc_l + n0 + n]));
        Bw[r * ldw + n] = v;
      }
      __syncthreads();
      // S^T slice (n x p) += Bw^T (n x s) X (s x p)
      if (warp * 16 < nw) warp_gemm<T, NT>(acc, Bw + warp * 16, 1, ldw, Xs, ldx, 1, kBlk);
      __syncthreads();
    }
    if (warp * 16 < nw) {
      const int n = n0 + warp * 16 + g;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const int q = nt * 8 + 2 * tq;
        S[(int64_t)q * N + n] = acc[nt][0];
        S[(int64_t)(q + 1) * N + n] = acc[nt][1];
        S[(int64_t)q * N + n + 8] = acc[nt][2];
        S[(int64_t)(q + 1) * N + n + 8] = acc[nt][3];
      }
    }
  }
}

// grid (ceil(P N / 256), heads, batch): one thread per state element, sequential over the chunks.
__global__ void __launch_bounds__(kPassThreads) ssd_state_pass_kernel(const SsdParams p) {
  const int64_t PN = (int64_t)p.P * p.N, e = (int64_t)blockIdx.x * kPassThreads + threadIdx.x;
  if (e >= PN) return;
  const int64_t bh = (int64_t)blockIdx.z * p.heads + blockIdx.y;
  float H = p.h0 ? __ldg(p.h0 + bh * PN + e) : 0.f;
  const float* cum = p.cum + bh * p.nchunks * p.Q + p.Q - 1;
  float* st = p.states + bh * p.nchunks * PN + e;
  for (int c = 0; c < p.nchunks; ++c) {
    const float s = st[c * PN];
    st[c * PN] = H;
    H = ex2f(__ldg(cum + (int64_t)c * p.Q) * kLog2e) * H + s;
  }
  if (p.hT) p.hT[bh * PN + e] = H;
}

// grid (nchunks * Q / 64, heads, batch); dynamic shared memory, see ssd_out_smem_floats.
template <typename T, int P>
__global__ void __launch_bounds__(kSsdThreads) ssd_chunk_out_kernel(const SsdParams p) {
  constexpr int NT = P / 8, ldx = P + 8, lds = kBlk + 4;
  extern __shared__ float smem[];
  const int N = p.N, Q = p.Q, ldn = N + 4, nq = Q / kBlk;
  const int c = blockIdx.x / nq, q = blockIdx.x % nq, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid >> 5, g = (tid & 31) >> 2, tq = tid & 3;
  const int64_t l_chunk = (int64_t)c * Q, l0 = l_chunk + q * kBlk;
  if (l0 >= p.L) return;
  const int grp = h / (p.heads / p.groups);
  const int64_t bh = (int64_t)b * p.heads + h;
  float* cum_s = smem;                        // [256]
  float* t_s = cum_s + 256;                   // [256]
  float* Cs = t_s + 256;                      // [64][N + 4]
  float* U = Cs + kBlk * ldn;                 // state slice [P][68], then B rows [64][N + 4]
  float* Xs = U + max(kBlk * ldn, P * lds);   // [64][P + 8]
  float* Ss = Xs + kBlk * ldx;                // [64][68]
  const int span = (q + 1) * kBlk;
  const int64_t ws = bh * p.nchunks * Q + l_chunk;
  for (int i = tid; i < span; i += kSsdThreads) {
    cum_s[i] = __ldg(p.cum + ws + i);
    t_s[i] = __ldg(p.t + ws + i);
  }
  const T* Bm = static_cast<const T*>(p.B) + b * p.bc_b + grp * p.bc_g;
  const T* Cm = static_cast<const T*>(p.C) + b * p.bc_b + grp * p.bc_g;
  const T* x = static_cast<const T*>(p.x) + b * p.x_b + h * p.x_h;
  for (int e = tid; e < kBlk * N; e += kSsdThreads) {
    const int r = e / N, n = e % N;
    Cs[r * ldn + n] = l0 + r < p.L ? to_f(Cm[(l0 + r) * p.bc_l + n]) : 0.f;
  }
  // state term: acc = C_l . H_c over N slices, then scaled by exp(cum_l)
  float acc[NT][4] = {};
  const float* Hc = p.states + (bh * p.nchunks + c) * P * N;
  for (int n0 = 0; n0 < N; n0 += kBlk) {
    const int nw = min(kBlk, N - n0);
    __syncthreads();
    for (int e = tid; e < P * kBlk; e += kSsdThreads) {
      const int r = e / kBlk, n = e % kBlk;
      U[r * lds + n] = n < nw ? round_io<T>(__ldg(Hc + (int64_t)r * N + n0 + n)) : 0.f;
    }
    __syncthreads();
    warp_gemm<T, NT>(acc, Cs + warp * 16 * ldn + n0, ldn, 1, U, 1, lds, nw);
  }
  const int r0 = warp * 16 + g, i0 = q * kBlk + r0;
  {
    const float e0 = ex2f(cum_s[i0] * kLog2e), e1 = ex2f(cum_s[i0 + 8] * kLog2e);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      acc[nt][0] *= e0; acc[nt][1] *= e0; acc[nt][2] *= e1; acc[nt][3] *= e1;
    }
  }
  // intra-chunk term, one 64-position block j <= q of sources at a time
  for (int j = 0; j <= q; ++j) {
    const int64_t s0 = l_chunk + j * kBlk;
    __syncthreads();
    for (int e = tid; e < kBlk * N; e += kSsdThreads) {
      const int r = e / N, n = e % N;
      U[r * ldn + n] = s0 + r < p.L ? to_f(Bm[(s0 + r) * p.bc_l + n]) : 0.f;
    }
    for (int e = tid; e < kBlk * P; e += kSsdThreads) {
      const int r = e / P, k = e % P;
      Xs[r * ldx + k] = s0 + r < p.L ? to_f(x[(s0 + r) * p.x_l + k]) : 0.f;
    }
    __syncthreads();
    float sc[kBlk / 8][4] = {};
    warp_gemm<T, kBlk / 8>(sc, Cs + warp * 16 * ldn, ldn, 1, U, 1, ldn, N);
#pragma unroll
    for (int nt = 0; nt < kBlk / 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = r0 + (e >> 1) * 8, s = nt * 8 + 2 * tq + (e & 1);
        const int li = q * kBlk + r, si = j * kBlk + s;
        const float d = si <= li ? cum_s[li] - cum_s[si] : -INFINITY;
        Ss[r * lds + s] = round_io<T>(sc[nt][e] * ex2f(d * kLog2e) * t_s[si]);
      }
    }
    __syncwarp();
    warp_gemm<T, NT>(acc, Ss + warp * 16 * lds, lds, 1, Xs, ldx, 1, kBlk);
  }
  // epilogue: + D x, z gate, store
  T* out = static_cast<T*>(p.out) + b * p.o_b + h * p.o_h;
  const T* z = p.z ? static_cast<const T*>(p.z) + b * p.z_b + h * p.z_h : nullptr;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t l = l0 + r0 + (e >> 1) * 8;
      const int k = nt * 8 + 2 * tq + (e & 1);
      if (l >= p.L) continue;
      float y = acc[nt][e];
      if (p.d_mode) y += p.D[p.d_mode == 1 ? h : h * P + k] * to_f(x[l * p.x_l + k]);
      if (z) y *= silu_f(to_f(z[l * p.z_l + k]));
      from_f(out + l * p.o_l + k, y);
    }
  }
}

// ---- backward ----------------------------------------------------------------------------------------------------------
// grid (npass, heads, batch): reverse state passing. dH starts at dhT; per chunk c, from the last: the slot of R_c takes
// dH_{c+1}, the block's share of sum dH_{c+1} H_{c+1} goes to dotp (a fixed-order block reduction), then
// dH_c = exp(cum_last,c) dH_{c+1} + R_c; dH_0 -> dh0.
__global__ void __launch_bounds__(kPassThreads) ssd_state_pass_bwd_kernel(const SsdParams p) {
  __shared__ float red[kPassThreads / 32];
  const int64_t PN = (int64_t)p.P * p.N, e = (int64_t)blockIdx.x * kPassThreads + threadIdx.x;
  const bool ok = e < PN;
  const int64_t bh = (int64_t)blockIdx.z * p.heads + blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float dH = ok && p.dhT ? __ldg(p.dhT + bh * PN + e) : 0.f;
  const float* cum = p.cum + bh * p.nchunks * p.Q + p.Q - 1;
  for (int c = p.nchunks - 1; c >= 0; --c) {
    float* rp = p.R + (bh * p.nchunks + c) * PN + e;
    float r = 0.f, v = 0.f;
    if (ok) {
      r = *rp;
      *rp = dH;
      const float Hn = c + 1 < p.nchunks ? p.states[(bh * p.nchunks + c + 1) * PN + e] : p.hfin[bh * PN + e];
      v = dH * Hn;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float sum = 0.f;
      for (int w = 0; w < kPassThreads / 32; ++w) sum += red[w];
      p.dotp[(bh * p.nchunks + c) * p.npass + blockIdx.x] = sum;
    }
    __syncthreads();
    dH = ex2f(__ldg(cum + (int64_t)c * p.Q) * kLog2e) * dH + r;
  }
  if (ok && p.dh0) p.dh0[bh * PN + e] = dH;
}

// grid (nchunks * Q / 64, heads, batch), one 64-position block q of a chunk in one of two roles.
// Target role (SRC = false), rows l of block q, over source blocks j <= q:
//   y_l = exp(cum_l) C_l . H_c + sum_{s <= l} (C_l . B_s) exp(cum_l - cum_s) t_s x_s, recomputed: dz = dout y' silu'(z) with
//   y' = y + D x; dcum1_l = dy_l . exp(cum_l) C_l H_c + sum_s M(l, s) with the pair terms
//   M(l, s) = (dy_l . x_s)(C_l . B_s) exp(cum_l - cum_s) t_s in fp32, whose column sums over the block's rows go to colM (the
//   source side of d cum takes them with the opposite sign, so the diagonal cancels exactly); dC_l = exp(cum_l) dy_l H_c + sum_{s <= l} (dy_l . x_s) exp(cum_l - cum_s) t_s B_s;
//   the per-block column sums of dy x for dD.
// Source role (SRC = true), rows s of block q, over target blocks i >= q of the chunk, with dS = dH_{c+1}:
//   W_s = exp(cum_last - cum_s) B_s dS^T + sum_{l >= s} (C_l . B_s) exp(cum_l - cum_s) dy_l, dx = t_s W_s + D dy_s,
//   ddtd_s = x_s . W_s, ddts_s = x_s . (its state part); dB_s = t_s (exp(cum_last - cum_s) x_s dS + sum_{l >= s} (x_s . dy_l) exp(cum_l - cum_s) C_l).
// The P-wide products accumulate in registers; the N-wide ones run in 64-state slices. Shared memory as in the output kernel
// plus one 64 x (P + 8) tile: own matrix rows M (C or B), own vector rows V (dy or x), the other block's matrix rows or a
// state slice U, its vector rows Wv, and the masked score tile S.
template <typename T, int P, bool SRC>
__global__ void __launch_bounds__(kSsdThreads, 1) ssd_chunk_bwd_kernel(const SsdParams p) {
  constexpr int NT = P / 8, ldx = P + 8, lds = kBlk + 4;
  extern __shared__ float smem[];
  const int N = p.N, Q = p.Q, ldn = N + 4, nq = Q / kBlk;
  const int c = blockIdx.x / nq, q = blockIdx.x % nq, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid >> 5, g = (tid & 31) >> 2, tq = tid & 3;
  const int64_t l_chunk = (int64_t)c * Q, l0 = l_chunk + q * kBlk;
  if (l0 >= p.L) return;
  const int grp = h / (p.heads / p.groups);
  const int64_t bh = (int64_t)b * p.heads + h;
  float* cum_s = smem;
  float* t_s = cum_s + 256;
  float* M = t_s + 256;
  float* V = M + kBlk * ldn;
  float* U = V + kBlk * ldx;
  float* Wv = U + max(kBlk * ldn, max(P, kBlk) * lds);
  float* S = Wv + kBlk * ldx;
  float* colS = S + kBlk * lds;               // [4][64]
  const int64_t ws = bh * p.nchunks * Q + l_chunk;
  for (int i = tid; i < Q; i += kSsdThreads) {
    cum_s[i] = __ldg(p.cum + ws + i);
    t_s[i] = __ldg(p.t + ws + i);
  }
  const T* Bm = static_cast<const T*>(p.B) + b * p.bc_b + grp * p.bc_g;
  const T* Cm = static_cast<const T*>(p.C) + b * p.bc_b + grp * p.bc_g;
  const T* x = static_cast<const T*>(p.x) + b * p.x_b + h * p.x_h;
  const T* dout = static_cast<const T*>(p.dout) + b * p.o_b + h * p.o_h;
  const T* z = p.z ? static_cast<const T*>(p.z) + b * p.z_b + h * p.z_h : nullptr;
  auto dy_at = [&](int64_t l, int k) {
    float v = to_f(dout[l * p.o_l + k]);
    if (z) v *= silu_f(to_f(z[l * p.z_l + k]));
    return v;
  };
  // rows r of block j into a matrix tile (cols n0 .. n0 + nw, pitch ld) and a vector tile
  auto stage_mat = [&](float* dst, int ld, const T* src, int j, int n0, int nw) {
    const int64_t s0 = l_chunk + j * kBlk;
    for (int e = tid; e < kBlk * nw; e += kSsdThreads) {
      const int r = e / nw, n = e % nw;
      dst[r * ld + n] = s0 + r < p.L ? to_f(src[(s0 + r) * p.bc_l + n0 + n]) : 0.f;
    }
  };
  auto stage_vec = [&](float* dst, bool dy, int j) {
    const int64_t s0 = l_chunk + j * kBlk;
    for (int e = tid; e < kBlk * P; e += kSsdThreads) {
      const int r = e / P, k = e % P;
      const int64_t l = s0 + r;
      dst[r * ldx + k] = l < p.L ? (dy ? dy_at(l, k) : to_f(x[l * p.x_l + k])) : 0.f;
    }
  };
  // the state a product reads: H_c (target role) or dS = dH_{c+1} (source role), slice n0 .. n0 + nw, rounded to T
  const float* st = (SRC ? p.R : p.states) + (bh * p.nchunks + c) * P * N;
  auto stage_state = [&](int n0, int nw) {
    for (int e = tid; e < P * kBlk; e += kSsdThreads) {
      const int r = e / kBlk, n = e % kBlk;
      U[r * lds + n] = n < nw ? round_io<T>(__ldg(st + (int64_t)r * N + n0 + n)) : 0.f;
    }
  };
  stage_mat(M, ldn, SRC ? Bm : Cm, q, 0, N);
  stage_vec(V, !SRC, q);
  const int jlo = SRC ? q : 0;
  const int jhi = SRC ? (int)(p.L - 1 - l_chunk < (int64_t)nq * kBlk ? (p.L - 1 - l_chunk) / kBlk : nq - 1) : q;
  const int r0 = warp * 16 + g, i0 = q * kBlk + r0;
  __syncthreads();
  const float cum_last = cum_s[Q - 1];
  // row scale of the state terms
  float sc0, sc1;
  if (SRC) {
    sc0 = ex2f((cum_last - cum_s[i0]) * kLog2e);
    sc1 = ex2f((cum_last - cum_s[i0 + 8]) * kLog2e);
  } else {
    sc0 = ex2f(cum_s[i0] * kLog2e);
    sc1 = ex2f(cum_s[i0 + 8] * kLog2e);
  }
  // masked decayed factor of the pair (row index ri of block q, column index oi of block j)
  auto pair = [&](int ri, int oi) {
    const bool ok = SRC ? oi >= ri : oi <= ri;
    const float d = ok ? (SRC ? cum_s[oi] - cum_s[ri] : cum_s[ri] - cum_s[oi]) : -INFINITY;
    return ex2f(d * kLog2e);
  };

  // ---- P-wide output: y (target) or W (source)
  {
    float acc[NT][4] = {};
    for (int n0 = 0; n0 < N; n0 += kBlk) {
      const int nw = min(kBlk, N - n0);
      __syncthreads();
      stage_state(n0, nw);
      __syncthreads();
      warp_gemm<T, NT>(acc, M + warp * 16 * ldn + n0, ldn, 1, U, 1, lds, nw);
    }
    float rowacc[2] = {0.f, 0.f};   // target: dy . y_off, then + the row sums of M; source: x . W_state
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      acc[nt][0] *= sc0; acc[nt][1] *= sc0; acc[nt][2] *= sc1; acc[nt][3] *= sc1;
#pragma unroll
      for (int e = 0; e < 4; ++e) rowacc[e >> 1] += V[(r0 + (e >> 1) * 8) * ldx + nt * 8 + 2 * tq + (e & 1)] * acc[nt][e];
    }
    for (int j = jlo; j <= jhi; ++j) {
      __syncthreads();
      stage_mat(U, ldn, SRC ? Cm : Bm, j, 0, N);
      stage_vec(Wv, SRC, j);
      __syncthreads();
      float sc[kBlk / 8][4] = {};
      warp_gemm<T, kBlk / 8>(sc, M + warp * 16 * ldn, ldn, 1, U, 1, ldn, N);
      if (!SRC) {
        float xd[kBlk / 8][4] = {};
        warp_gemm<T, kBlk / 8>(xd, V + warp * 16 * ldx, ldx, 1, Wv, 1, ldx, P);
        float col[kBlk / 8][2];
#pragma unroll
        for (int nt = 0; nt < kBlk / 8; ++nt) {
          col[nt][0] = col[nt][1] = 0.f;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int r = r0 + (e >> 1) * 8, oi = j * kBlk + nt * 8 + 2 * tq + (e & 1);
            const float m = sc[nt][e] * xd[nt][e] * pair(q * kBlk + r, oi) * t_s[oi];
            rowacc[e >> 1] += m;
            col[nt][e & 1] += m;
          }
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) {
            col[nt][0] += __shfl_xor_sync(0xffffffffu, col[nt][0], o);
            col[nt][1] += __shfl_xor_sync(0xffffffffu, col[nt][1], o);
          }
          if (g == 0) {
            colS[warp * kBlk + nt * 8 + 2 * tq] = col[nt][0];
            colS[warp * kBlk + nt * 8 + 2 * tq + 1] = col[nt][1];
          }
        }
        __syncthreads();
        if (tid < kBlk)
          p.colM[(((bh * p.nchunks + c) * nq + q) * nq + j) * kBlk + tid] =
              ((colS[tid] + colS[kBlk + tid]) + colS[2 * kBlk + tid]) + colS[3 * kBlk + tid];
      }
#pragma unroll
      for (int nt = 0; nt < kBlk / 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int r = r0 + (e >> 1) * 8, s = nt * 8 + 2 * tq + (e & 1);
          const int oi = j * kBlk + s;
          S[r * lds + s] = round_io<T>(sc[nt][e] * pair(q * kBlk + r, oi) * (SRC ? 1.f : t_s[oi]));
        }
      __syncwarp();
      warp_gemm<T, NT>(acc, S + warp * 16 * lds, lds, 1, Wv, ldx, 1, kBlk);
    }
    float dot[2] = {0.f, 0.f};   // source: x . W
    T* gout = static_cast<T*>(SRC ? p.dx : p.dz) + b * p.o_b + h * p.o_h;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = r0 + (e >> 1) * 8, k = nt * 8 + 2 * tq + (e & 1);
        const int64_t l = l0 + r;
        if (l >= p.L) continue;
        const float a = acc[nt][e], v = V[r * ldx + k];
        const float Dk = p.d_mode ? p.D[p.d_mode == 1 ? h : h * P + k] : 0.f;
        if (SRC) dot[e >> 1] += v * a;
        if (SRC) {
          from_f(gout + l * p.o_l + k, t_s[q * kBlk + r] * a + Dk * dy_at(l, k));
        } else if (p.dz) {
          const float y = a + Dk * to_f(x[l * p.x_l + k]), zz = to_f(z[l * p.z_l + k]);
          from_f(gout + l * p.o_l + k, to_f(dout[l * p.o_l + k]) * y * silu_grad_f(zz));
        }
      }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      dot[e] += __shfl_xor_sync(0xffffffffu, dot[e], 1);
      dot[e] += __shfl_xor_sync(0xffffffffu, dot[e], 2);
      rowacc[e] += __shfl_xor_sync(0xffffffffu, rowacc[e], 1);
      rowacc[e] += __shfl_xor_sync(0xffffffffu, rowacc[e], 2);
    }
    if (tq == 0) {
      float* o = (SRC ? p.ddts : p.dcum1) + ws + q * kBlk;
      o[r0] = rowacc[0];
      o[r0 + 8] = rowacc[1];
      if (SRC) {
        p.ddtd[ws + q * kBlk + r0] = dot[0];
        p.ddtd[ws + q * kBlk + r0 + 8] = dot[1];
      }
    }
  }
  if (!SRC && p.d_mode) {   // column sums of dy x over the block's rows, for dD
    __syncthreads();
    for (int e = tid; e < kBlk * P; e += kSsdThreads) {
      const int r = e / P, k = e % P;
      Wv[r * ldx + k] = l0 + r < p.L ? V[r * ldx + k] * to_f(x[(l0 + r) * p.x_l + k]) : 0.f;
    }
    __syncthreads();
    const int64_t blk = (int64_t)c * nq + q, nblk = (int64_t)p.nchunks * nq;
    for (int k = tid; k < P; k += kSsdThreads) {
      float sum = 0.f;
      for (int r = 0; r < kBlk; ++r) sum += Wv[r * ldx + k];
      p.partD[((b * nblk + blk) * p.heads + h) * P + k] = sum;
    }
  }

  // ---- N-wide output in 64-state slices: dC (target) or dB (source)
  float* gmat = (SRC ? p.dBh : p.dCh) + (bh * p.nchunks * Q) * N;
  const float t0 = t_s[i0], t1 = t_s[i0 + 8];
  for (int n0 = 0; n0 < N; n0 += kBlk) {
    const int nw = min(kBlk, N - n0);
    float acc[kBlk / 8][4] = {};
    __syncthreads();
    stage_state(n0, nw);
    __syncthreads();
    warp_gemm<T, kBlk / 8>(acc, V + warp * 16 * ldx, ldx, 1, U, lds, 1, P);
    const float f0 = SRC ? sc0 * t0 : sc0, f1 = SRC ? sc1 * t1 : sc1;
#pragma unroll
    for (int nt = 0; nt < kBlk / 8; ++nt) {
      acc[nt][0] *= f0; acc[nt][1] *= f0; acc[nt][2] *= f1; acc[nt][3] *= f1;
    }
    for (int j = jlo; j <= jhi; ++j) {
      __syncthreads();
      stage_mat(U, lds, SRC ? Cm : Bm, j, n0, nw);
      for (int e = tid; e < kBlk * kBlk; e += kSsdThreads) {   // columns past nw read as zeros
        const int r = e / kBlk, n = e % kBlk;
        if (n >= nw) U[r * lds + n] = 0.f;
      }
      stage_vec(Wv, SRC, j);
      __syncthreads();
      float xd[kBlk / 8][4] = {};
      warp_gemm<T, kBlk / 8>(xd, V + warp * 16 * ldx, ldx, 1, Wv, 1, ldx, P);
#pragma unroll
      for (int nt = 0; nt < kBlk / 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int r = r0 + (e >> 1) * 8, s = nt * 8 + 2 * tq + (e & 1);
          const int ri = q * kBlk + r, oi = j * kBlk + s;
          S[r * lds + s] = round_io<T>(xd[nt][e] * pair(ri, oi) * t_s[SRC ? ri : oi]);
        }
      __syncwarp();
      warp_gemm<T, kBlk / 8>(acc, S + warp * 16 * lds, lds, 1, U, lds, 1, kBlk);
    }
#pragma unroll
    for (int nt = 0; nt < kBlk / 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = r0 + (e >> 1) * 8, n = nt * 8 + 2 * tq + (e & 1);
        if (l0 + r < p.L && n < nw) gmat[(q * kBlk + r + (int64_t)c * Q) * N + n0 + n] = acc[nt][e];
      }
  }
}

// grid (nchunks, heads, batch), one thread per position of the chunk: dcum_l = dcum1_l - sum_q colM(q, l) - t_l ddts_l
// (+ sum dH_{c+1} H_{c+1} at the chunk's last position), d a_l = its reverse inclusive cumsum within the chunk, d t_l = d a_l A + ddtd_l, then through
// the clamp (zero where it is active), the softplus and dt_bias to ddt. Per-chunk partials of dA = sum d a_l t_l and of
// ddt_bias = sum ddt, by fixed-order block reductions.
template <typename T>
__global__ void __launch_bounds__(256) ssd_dt_bwd_kernel(const SsdParams p) {
  __shared__ float sc[256];
  __shared__ float red[2][8];
  const int c = blockIdx.x, h = blockIdx.y, b = blockIdx.z, i = threadIdx.x, Q = p.Q;
  const int64_t bh = (int64_t)b * p.heads + h, ws = bh * p.nchunks * Q + (int64_t)c * Q, l = (int64_t)c * Q + i;
  const bool live = i < Q && l < p.L;
  float dc = 0.f, dd = 0.f, t = 0.f;
  if (live) {
    t = p.t[ws + i];
    dd = p.ddtd[ws + i];
    const int nq = Q / kBlk, j = i / kBlk;
    const int qhi = (int)min((int64_t)nq - 1, (p.L - 1 - (int64_t)c * Q) / kBlk);
    const float* cm = p.colM + ((bh * p.nchunks + c) * nq * nq + j) * kBlk + i % kBlk;
    float col = 0.f;
    for (int q = j; q <= qhi; ++q) col += cm[(int64_t)q * nq * kBlk];
    dc = (p.dcum1[ws + i] - col) - t * p.ddts[ws + i];
  }
  if (i == Q - 1) {
    const float* dp = p.dotp + (bh * p.nchunks + c) * p.npass;
    float s = 0.f;
    for (int k = 0; k < p.npass; ++k) s += dp[k];
    dc += s;
  }
  sc[i] = dc;
  __syncthreads();
  for (int off = 1; off < Q; off <<= 1) {   // reverse inclusive scan
    const float v = i < Q && i + off < Q ? sc[i + off] : 0.f;
    __syncthreads();
    sc[i] += v;
    __syncthreads();
  }
  float pa = 0.f, pb = 0.f;
  if (live) {
    const float A = p.A[h], da = sc[i];
    pa = da * t;
    float v = to_f(static_cast<const T*>(p.dt)[b * p.dt_b + l * p.dt_l + h * p.dt_h]);
    if (p.dt_bias) v += p.dt_bias[h];
    float gr = da * A + dd;
    if (p.softplus) {
      gr *= softplus20_grad(v);
      v = softplus20(v);
    }
    if (v < p.dt_min || v > p.dt_max) gr = 0.f;
    pb = gr;
    from_f(static_cast<T*>(p.ddt) + (b * p.L + l) * p.heads + h, gr);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    pa += __shfl_xor_sync(0xffffffffu, pa, o);
    pb += __shfl_xor_sync(0xffffffffu, pb, o);
  }
  if ((i & 31) == 0) { red[0][i >> 5] = pa; red[1][i >> 5] = pb; }
  __syncthreads();
  if (i == 0) {
    float a = 0.f, bb = 0.f;
    for (int w = 0; w < 8; ++w) { a += red[0][w]; bb += red[1][w]; }
    p.partA[bh * p.nchunks + c] = a;
    p.partBias[bh * p.nchunks + c] = bb;
  }
}

// one thread per (head, channel): dD, dA and ddt_bias from the partials, summed in a fixed order
__global__ void __launch_bounds__(256) ssd_param_grad_kernel(const SsdParams p) {
  const int e = blockIdx.x * 256 + threadIdx.x;
  if (e >= p.heads * p.P) return;
  const int h = e / p.P, k = e % p.P, nq = p.Q / kBlk;
  const int64_t nblk = (int64_t)p.nchunks * nq, live = (p.L + kBlk - 1) / kBlk;
  if (p.d_mode == 2 || (p.d_mode == 1 && k == 0)) {
    float s = 0.f;
    for (int kk = p.d_mode == 2 ? k : 0; kk < (p.d_mode == 2 ? k + 1 : p.P); ++kk)
      for (int b = 0; b < p.batch; ++b)
        for (int64_t blk = 0; blk < live; ++blk) s += p.partD[((b * nblk + blk) * p.heads + h) * p.P + kk];
    p.dD[p.d_mode == 2 ? e : h] = s;
  }
  if (k == 0) {
    float a = 0.f, bb = 0.f;
    for (int b = 0; b < p.batch; ++b)
      for (int c = 0; c < p.nchunks; ++c) {
        a += p.partA[((int64_t)b * p.heads + h) * p.nchunks + c];
        bb += p.partBias[((int64_t)b * p.heads + h) * p.nchunks + c];
      }
    p.dA[h] = a;
    if (p.ddt_bias) p.ddt_bias[h] = bb;
  }
}

// one thread per element of dB and dC (batch, L, groups, N): the per-head values of the group's heads summed in head order
template <typename T>
__global__ void __launch_bounds__(256) ssd_bc_grad_kernel(const SsdParams p) {
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x, total = (int64_t)p.batch * p.L * p.groups * p.N;
  if (e >= total) return;
  const int n = (int)(e % p.N);
  const int64_t r = e / p.N;
  const int grp = (int)(r % p.groups);
  const int64_t bl = r / p.groups, l = bl % p.L, b = bl / p.L, Lp = (int64_t)p.nchunks * p.Q;
  const int hpg = p.heads / p.groups;
  float sb = 0.f, sc = 0.f;
  for (int k = grp * hpg; k < (grp + 1) * hpg; ++k) {
    const int64_t o = ((b * p.heads + k) * Lp + l) * p.N + n;
    sb += p.dBh[o];
    sc += p.dCh[o];
  }
  from_f(static_cast<T*>(p.dB) + e, sb);
  from_f(static_cast<T*>(p.dC) + e, sc);
}

namespace {

size_t out_smem_bytes(int P, int N) {
  const int ldn = N + 4;
  return sizeof(float) * (512 + (size_t)kBlk * ldn + std::max(kBlk * ldn, P * (kBlk + 4)) + kBlk * (P + 8) + kBlk * (kBlk + 4));
}

template <typename K>
cudaError_t set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

size_t state_smem_bytes(int P) { return sizeof(float) * (512 + kBlk * (P + 8) + kBlk * (kBlk + 8)); }

#define SSD_TRY(...)                     \
  do {                                   \
    const cudaError_t e_ = (__VA_ARGS__); \
    if (e_ != cudaSuccess) return e_;    \
  } while (0)

template <typename T, int P, bool BWD>
cudaError_t chunk_state(const SsdParams& p, cudaStream_t s) {
  SSD_TRY(set_smem(ssd_chunk_state_kernel<T, P, BWD>, state_smem_bytes(P)));
  ssd_chunk_state_kernel<T, P, BWD><<<dim3(p.nchunks, p.heads, p.batch), kSsdThreads, state_smem_bytes(P), s>>>(p);
  return cudaGetLastError();
}

dim3 pass_grid(const SsdParams& p) {
  return dim3((unsigned)(((int64_t)p.P * p.N + kPassThreads - 1) / kPassThreads), p.heads, p.batch);
}

template <typename T, int P>
cudaError_t fwd_typed(const SsdParams& p, cudaStream_t s) {
  SSD_TRY(chunk_state<T, P, false>(p, s));
  ssd_state_pass_kernel<<<pass_grid(p), kPassThreads, 0, s>>>(p);
  SSD_TRY(cudaGetLastError());
  const size_t smem = out_smem_bytes(P, p.N);
  SSD_TRY(set_smem(ssd_chunk_out_kernel<T, P>, smem));
  ssd_chunk_out_kernel<T, P><<<dim3(p.nchunks * (p.Q / kBlk), p.heads, p.batch), kSsdThreads, smem, s>>>(p);
  return cudaGetLastError();
}

template <typename T, int P>
cudaError_t bwd_typed(const SsdParams& p, cudaStream_t s) {
  SSD_TRY(chunk_state<T, P, false>(p, s));   // recompute t, cum and the states entering each chunk
  ssd_state_pass_kernel<<<pass_grid(p), kPassThreads, 0, s>>>(p);
  SSD_TRY(cudaGetLastError());
  SSD_TRY(chunk_state<T, P, true>(p, s));
  ssd_state_pass_bwd_kernel<<<pass_grid(p), kPassThreads, 0, s>>>(p);
  SSD_TRY(cudaGetLastError());
  const size_t smem = sizeof(float) * (512 + (size_t)kBlk * (p.N + 4) + std::max(kBlk * (p.N + 4), std::max(P, kBlk) * (kBlk + 4)) +
                                        2 * kBlk * (P + 8) + kBlk * (kBlk + 4) + 4 * kBlk);
  const dim3 grid(p.nchunks * (p.Q / kBlk), p.heads, p.batch);
  SSD_TRY(set_smem(ssd_chunk_bwd_kernel<T, P, false>, smem));
  ssd_chunk_bwd_kernel<T, P, false><<<grid, kSsdThreads, smem, s>>>(p);
  SSD_TRY(cudaGetLastError());
  SSD_TRY(set_smem(ssd_chunk_bwd_kernel<T, P, true>, smem));
  ssd_chunk_bwd_kernel<T, P, true><<<grid, kSsdThreads, smem, s>>>(p);
  SSD_TRY(cudaGetLastError());
  ssd_dt_bwd_kernel<T><<<dim3(p.nchunks, p.heads, p.batch), 256, 0, s>>>(p);
  SSD_TRY(cudaGetLastError());
  ssd_param_grad_kernel<<<(p.heads * P + 255) / 256, 256, 0, s>>>(p);
  SSD_TRY(cudaGetLastError());
  const int64_t nbc = (int64_t)p.batch * p.L * p.groups * p.N;
  ssd_bc_grad_kernel<T><<<(unsigned)((nbc + 255) / 256), 256, 0, s>>>(p);
  return cudaGetLastError();
}

template <bool BWD, typename T, int P>
cudaError_t run(const SsdParams& p, cudaStream_t s) {
  if constexpr (BWD) return bwd_typed<T, P>(p, s);
  else return fwd_typed<T, P>(p, s);
}

template <bool BWD, typename T>
cudaError_t by_headdim(const SsdParams& p, cudaStream_t s) {
  switch (p.P) {
    case 32: return run<BWD, T, 32>(p, s);
    case 64: return run<BWD, T, 64>(p, s);
    default: return run<BWD, T, 128>(p, s);
  }
}

template <bool BWD>
cudaError_t by_dtype(const SsdParams& p, int io_dtype, cudaStream_t s) {
  switch (io_dtype) {
    case SS2D_F32: return by_headdim<BWD, float>(p, s);
    case SS2D_F16: return by_headdim<BWD, __half>(p, s);
    default: return by_headdim<BWD, __nv_bfloat16>(p, s);
  }
}

}  // namespace

// three launches; p.t, p.cum, p.states point into a workspace of ssd_fwd_workspace_floats(...) floats
cudaError_t ssd_fwd_launch(const SsdParams& p, int io_dtype, cudaStream_t s) { return by_dtype<false>(p, io_dtype, s); }
// nine launches; the backward workspace pointers of p are set (ss2d_ssd_bwd_workspace_bytes)
cudaError_t ssd_bwd_launch(const SsdParams& p, int io_dtype, cudaStream_t s) { return by_dtype<true>(p, io_dtype, s); }

}  // namespace ss2d
