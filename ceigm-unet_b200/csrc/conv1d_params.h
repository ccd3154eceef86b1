// Host-side parameters of the causal depthwise 1-D convolution (ss2d_conv1d_*, csrc/causal_conv1d.cu).
#pragma once
#include <stdint.h>

namespace ss2d {

// Strides in elements; stride 1 along L.
struct Conv1dParams {
  const void* x;           // (batch, dim, L) at b * x_bs + d * x_ds + l; update: (batch, dim) at b * x_bs + d * x_ds
  const void* dout;        // backward: (batch, dim, L) at b * o_bs + d * o_ds + l
  void* out;               // forward: out; backward: dx (both like dout); update: out (batch, dim) at b * o_bs + d * o_ds
  void* state;             // update: (batch, dim, width) contiguous
  const float* w;          // (dim, width) contiguous
  const float* bias;       // (dim) or null
  float *dw, *db, *part;   // backward: (dim, width), (dim) or null, slab partials (dim, slabs, width + 1)
  int64_t x_bs, x_ds, o_bs, o_ds;
  int64_t L;
  int batch, dim, width, silu, slabs;
};

}  // namespace ss2d
