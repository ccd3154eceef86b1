// Host-side parameters of the Mamba-2 chunked selective scan (ss2d_ssd_*, csrc/ssd.cu).
#pragma once
#include <stdint.h>

namespace ss2d {

// Strides in elements; stride 1 along headdim (x, z, out) and along dstate (B, C).
struct SsdParams {
  const void* x;           // (batch, L, heads, P) at b * x_b + l * x_l + h * x_h + p
  const void* dt;          // (batch, L, heads) at b * dt_b + l * dt_l + h * dt_h
  const void* B;           // (batch, L, groups, N) at b * bc_b + l * bc_l + g * bc_g + n
  const void* C;           // like B
  const void* z;           // like x with z_* strides, or null
  const float* A;          // (heads)
  const float* D;          // null, (heads) or (heads, P) by d_mode
  const float* dt_bias;    // (heads) or null
  const float* h0;         // (batch, heads, P, N) contiguous or null
  void* out;               // like x with o_* strides
  float* hT;               // (batch, heads, P, N) contiguous or null
  float *t, *cum;          // workspace: (batch, heads, nchunks * Q) processed dt and its in-chunk inclusive cumsum of t A
  float* states;           // workspace: (batch, heads, nchunks, P, N) chunk states, then the state entering each chunk
  // backward: dout, dx, dz at the o_* strides; ddt (batch, L, heads) and dB, dC (batch, L, groups, N) dense
  const void* dout;
  const float* dhT;        // (batch, heads, P, N) contiguous or null
  void *dx, *dz, *ddt, *dB, *dC;
  float *dA, *dD, *ddt_bias, *dh0;
  // backward workspace: final state (batch, heads, P, N); R: per chunk sum_l exp(cum_l) dy_l (x) C_l, then dH_{c+1};
  // dotp: per (batch, head, chunk, pass block) partial of sum dH_{c+1} H_{c+1}; dcum1 = dy . (y - D x), ddtd = x . W per
  // position (dcum1 with the intra-chunk part as row sums of M); dBh, dCh: per-head dB, dC (batch, heads, nchunks * Q, N); partD, partA, partBias: per-block partials
  // ddts = x . (the state part of W); colM: per (batch, head, chunk, target block q, source block j) column sums over the
  // rows of q of the intra-chunk pair terms M(l, s) = (dy_l . x_s)(C_l . B_s) exp(cum_l - cum_s) t_s
  float *hfin, *R, *dotp, *dcum1, *ddtd, *ddts, *colM, *dBh, *dCh, *partD, *partA, *partBias;
  int npass;               // blocks of the state pass per (batch, head)
  int64_t x_b, x_l, x_h, z_b, z_l, z_h, o_b, o_l, o_h, dt_b, dt_l, dt_h, bc_b, bc_l, bc_g;
  int64_t L;
  int batch, heads, groups, P, N, Q, nchunks, d_mode, softplus;
  float dt_min, dt_max;
};

}  // namespace ss2d
