// Internal kernel parameter block (host fills it from ss2d_scan_desc; passed by value to the kernels).
#pragma once
#include <stdint.h>

#include "ss2d_b200.h"

namespace ss2d {

struct ScanParams {
  int batch, dim, L, N, G, dpg;      // dpg = dim / G channels per group
  int io_dtype, out_dtype, softplus;
  int layout, H, W;
  int dirs[SS2D_MAX_GROUP_DIRS];     // 0 in SCAN layout
  int u_mod;                         // 0 or the channel modulo for u (and for dout in the backward)
  int last_il;                       // last_state interleaved (h in odd slots)
  int tma_ok;                        // fp32 operands, 16-byte aligned rows: TMA bulk staging allowed
  int nck;                           // number of SS2D_CHUNK checkpoints per row
  int NP;                            // padded state count of the kernel variant (ckpt row length)
  int A_ld;                          // row stride of A / dA / last_state (total dstate); N is this pass's count
  int accum;                         // 1: out/du/ddelta += (later state passes when dstate > 32), D-skip already applied
  int64_t u_bs, u_ds, dl_bs, dl_ds, out_bs, out_ds;
  int64_t B_bs, B_gs, B_ns, C_bs, C_gs, C_ns;
  const void* u;
  const void* delta;
  const float* A;
  const void* Bm;
  const void* Cm;
  const float* Dv;
  const float* bias;
  void* out;
  float* ckpt;          // [batch][dim][nck][NP]
  float* last_state;    // [batch][dim][N] or null
  // backward only
  const void* dout;
  const float* ckpt_in;
  void* du;
  void* ddelta;
  float* dB;            // fp32 [batch][G][N][L], pre-zeroed, accumulated with red.global when a group spans several CTAs
  float* dC;
  float* part;          // workspace: [batch][dim][N + 2] per-batch partial sums of dA, dD, dbias
  // deterministic backward: the CTAs (scan_bwd2: warps) that share a group store their dB / dC sums into partial slab s =
  // their index along the group instead of reducing into dB / dC; slab 0 is dB / dC itself, slab s > 0 lives at
  // slabB / slabC + (s - 1) * slab_stride (same indexing as dB / dC), and scan_bwd_fold sums the slabs in slab order
  int det;
  float* slabB;
  float* slabC;
  int64_t slab_stride;
};

// State passing, the last kernel argument of every scan kernel template with a STATE flag (a separate argument, so ScanParams
// keeps its layout and the STATE = false instantiations keep their instructions; they are passed zeros and never read it).
// Rows of A_ld floats like A; this pass's states start at element 0. Forward: the state before a row's first position is h0
// (non-null whenever STATE). Backward: h0 starts the recompute of chunk 0, dlast is the adjoint entering the row's last
// position, dh0 receives the adjoint of h0; each may be null.
struct ScanState {
  const float* h0;
  const float* dlast;
  float* dh0;
};
// Output gate of ss2d_scan_fwd_gated, a separate argument of the scan_fwdr kernels for the same reason: out_z = out * silu(z),
// both fp32 with out's strides. The GATE instantiations read it; the others are passed zeros.
struct ScanGate {
  const void* z;
  void* out_z;
};
// One recurrent step (ss2d_state_update, csrc/state_update.cu); strides in elements, innermost stride 1.
struct StepParams {
  float* state;                      // [batch][dim][dstate]
  const void *x, *dt, *B, *C, *z;    // z may be null
  const float *A, *D, *bias;         // D, bias may be null
  void* out;
  int64_t rows;                      // batch * dim
  int dim, dstate, dpg, softplus;    // dpg = dim / n_groups
  int64_t io_bs, B_bs, B_gs, C_bs, C_gs;
};

// backward: the STATE instantiation runs when any of the three pointers is set
inline bool has_state(const ScanState& st) { return st.h0 || st.dlast || st.dh0; }

// state element n of row (b, d): h0 / dlast / dh0 layout
__host__ __device__ inline int64_t state_slot(const ScanParams& p, int b, int d, int n) {
  return ((int64_t)b * p.dim + d) * p.A_ld + n;
}

// destination of partial slab s of dB (which 0) or dC (which 1)
__host__ __device__ inline float* det_slab(const ScanParams& p, int which, int s) {
  if (s == 0) return which ? p.dC : p.dB;
  return (which ? p.slabC : p.slabB) + (int64_t)(s - 1) * p.slab_stride;
}

// Opaque 128-byte TMA tensor-map descriptors (CUtensorMap), filled on the host by cuTensorMapEncodeTiled and passed
// to the kernels as a __grid_constant__ parameter.
struct alignas(64) TMap { unsigned long long v[16]; };
struct TmaMaps { TMap u, dl, B, C, dy; };

// Kernel variant for a state count: NS states per thread, R lanes per row. NS * R >= N.
struct Variant { int NS, R; };
inline Variant pick_variant(int N) {
  if (N <= 1) return {1, 1};
  if (N <= 2) return {2, 1};
  if (N <= 4) return {4, 1};
  if (N <= 8) return {4, 2};
  if (N <= 16) return {4, 4};
  return {4, 8};      // N <= 32; larger N is processed in passes of 32 states by the host
}

}  // namespace ss2d
