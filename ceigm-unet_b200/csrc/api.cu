// C ABI of libss2d_b200.so: argument validation, parameter packing, variant dispatch. No torch, no allocation.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>

#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "scan_params.h"
#include "ss2d_b200.h"

namespace ss2d {
cudaError_t scan_fwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream);
bool scan_fwdr_try(const ScanParams& p, const ScanState& st, const ScanGate& gt, cudaStream_t stream, cudaError_t* err,
                   bool* gated);
// output gate passes (scan_gate.cu): out_z = y silu(z); dy = dout_z silu(z) (fp32, dense (batch, dim, L)), dz
cudaError_t scan_gate_fwd_launch(const ss2d_scan_desc* d, const void* y, const void* z, void* out_z, cudaStream_t s);
cudaError_t scan_gate_bwd_launch(const ss2d_scan_desc* d, const void* dout_z, const void* z, const void* y, float* dy, void* dz,
                                 cudaStream_t s);
// one recurrent step (state_update.cu)
cudaError_t ssm_step_launch(const StepParams& p, int io_dtype, cudaStream_t stream);
constexpr int kDwnMaxSeg = 4;
struct DwnSegs { int nseg; int cbeg[kDwnMaxSeg + 1]; int k[kDwnMaxSeg]; const float* w[kDwnMaxSeg]; const float* b[kDwnMaxSeg]; };
cudaError_t dwnhwc_stencil_launch(const void* x, const void* aux, void* y, const DwnSegs& sg, int flip, int epi, int B, int H,
                                  int W, int C, int dt, cudaStream_t stream);
int dwnhwc_wgrad_slabs(int B, int H, int W, int nc);
cudaError_t dwnhwc_wgrad_launch(const void* x, const void* g, int c0, int nc, int K, float* dW, float* db, int B, int H, int W,
                                int C, int dt, float* part, cudaStream_t stream);
// backward launchers: *slabs receives the number of dB / dC partial slabs the launch wrote in deterministic mode (0 or 1:
// dB / dC hold the result already)
cudaError_t scan_bwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream, int* slabs);
cudaError_t scan_bwd_finalize(const ScanParams& p, float* dA, float* dD, float* dbias, cudaStream_t stream);
cudaError_t scan_bwd_fold(const ScanParams& p, int slabs, cudaStream_t stream);
cudaError_t scan_par_fwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream);
cudaError_t scan_par_bwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream, int* slabs);
bool scan_n1_fwd_try(const ScanParams& p, const ScanState& st, cudaStream_t stream, cudaError_t* err);
bool scan_n1_bwd_try(const ScanParams& p, const ScanState& st, float* dA, float* dD, float* dbias, int grads_zeroed,
                     cudaStream_t stream, cudaError_t* err, int* slabs);
// most partial slabs any backward kernel the dispatcher may pick for this pass writes in deterministic mode
int scan_bwd_det_slabs(const ScanParams& p);
int scan_n1_bwd_det_slabs(const ScanParams& p);
int scan_par_bwd_det_slabs(const ScanParams& p);

// d_state == 1 (the live GM-UNet regime) runs the parallel-along-L kernels (scan_par.cu)
static bool use_par(const ScanParams& p) { return p.N == 1 && p.A_ld == 1; }
cudaError_t cross_scan_launch(const void* x, void* xs, int batch, int channels, int H, int W, int K, const int* dirs,
                              int dtype, cudaStream_t stream);
cudaError_t cross_merge_launch(const void* ys, void* y, int batch, int channels, int H, int W, int K, const int* dirs,
                               int dtype, cudaStream_t stream);

cudaError_t out_gate_fwd_launch(const float* ys, int K, const float* lnw, const float* lnb, const void* z, int64_t z_rs,
                                int z_act, void* out, float* mean_rstd, int batch, int D, int L, float eps, int z_dtype,
                                int out_dtype, int H, int W, unsigned tmask, cudaStream_t stream);
cudaError_t out_gate_bwd_launch(const float* ys, int K, const float* lnw, const float* lnb, const void* z, int64_t z_rs,
                                int z_act, const void* dout, const float* mean_rstd, float* dy, void* dz, int64_t dz_rs,
                                float* dw_part, float* db_part, int n_partials, int batch, int D, int L, int z_dtype,
                                int out_dtype, int H, int W, unsigned tmask, int dy_two_planes, cudaStream_t stream);
int epi_bwd_partials(int batch, int L);
int layernorm_bwd_partials(int64_t rows);
int layernorm_max_C();
cudaError_t layernorm_fwd_launch(const void* x, const float* w, const float* b, void* y, float* mean_rstd, int64_t rows,
                                 int C, float eps, int dt, cudaStream_t stream);
cudaError_t layernorm_bwd_launch(const void* x, const float* w, const void* dy, const float* mean_rstd, void* dx,
                                 float* dw_part, float* db_part, int n_partials, int64_t rows, int C, int dt,
                                 cudaStream_t stream);
int dwconv3_wgrad_slabs(int batch, int C, int H, int W);
cudaError_t dwconv3_wgrad_launch(const float* x, const float* dy, float* dW, float* db, float* workspace, int batch, int C,
                                 int H, int W, cudaStream_t stream);
bool wgrad_ts_supported(int M, int N);
size_t wgrad_ts_workspace_floats(int64_t total_rows, int M, int N);
cudaError_t wgrad_ts_launch(const void* dY, const void* X, float* dW, int batch, int rows, int M, int N, int64_t y_bs,
                            int64_t y_rs, int64_t y_cs, int64_t x_bs, int64_t x_rs, int64_t x_cs, int y_dt, int x_dt,
                            float* workspace, cudaStream_t stream);
int epi_max_D(bool backward);
cudaError_t group_gate_fwd_launch(const float* ys, int G, const int* plane_of, unsigned tmask_bits, const float* lnw,
                                  const float* lnb, const void* z, int64_t z_rs, int64_t z_col0, int64_t z_gs, void* out,
                                  int64_t out_rs, float* mean_rstd, int batch, int D, int L, float eps, int z_dtype,
                                  int out_dtype, int H, int W, cudaStream_t stream);
cudaError_t group_gate_bwd_launch(const float* ys, int G, const int* plane_of, unsigned tmask_bits, const float* lnw,
                                  const float* lnb, const void* z, int64_t z_rs, int64_t z_col0, int64_t z_gs, const void* dout,
                                  int64_t dout_rs, const float* mean_rstd, float* dy, void* dz, int64_t dz_rs, float* dw_part,
                                  float* db_part, int n_partials, int batch, int D, int L, int z_dtype, int out_dtype, int H,
                                  int W, cudaStream_t stream);

cudaError_t dwconv3_fused_launch(int mode, const void* x, const float* wgt, const float* bias, const void* dy, void* y,
                                 int batch, int C, int H, int W, int dt, cudaStream_t stream);
cudaError_t dwconv3_tiled_launch(int mode, const void* x, const float* wgt, const float* bias, const void* dy, const void* dyT,
                                 void* y, void* yT, int batch, int C, int H, int W, int64_t x_bs, int64_t y_bs, int64_t yT_bs,
                                 int64_t dy_bs, int64_t dyT_bs, int dt, cudaStream_t stream);
bool gate_proj_tc_supported(int D, int C, int K, int dtype);
int gate_proj_tc_launch(const float* ys, int K, unsigned tmask, const float* lnw, const float* lnb, float eps, const void* z,
                        int64_t z_rs, int z_act, const void* W, int64_t ldw, const float* bias, void* out, int64_t out_rs,
                        void* g_out, int64_t g_rs, float* mean_rstd, int batch, int D, int L, int H, int Wd, int C, int dtype,
                        cudaStream_t stream, cudaError_t* cerr);
bool linear_tc_supported(int N_part, int K, int dtype);
int linear_tc_launch(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, int M, int N, int K, int dtype,
                     int n_parts, const ss2d_linear_part* parts, cudaStream_t stream, cudaError_t* cerr);

thread_local char g_cuda_err[256] = "";
// process-wide: the autograd engine launches the backward kernels from its own per-device threads
static std::atomic<int64_t> g_launches{0};
static std::atomic<int> g_path_policy{0};
int scan_path_policy() { return g_path_policy.load(std::memory_order_relaxed) & 7; }
bool scan_gate_fusion() { return !(g_path_policy.load(std::memory_order_relaxed) & 8); }

static int cuda_fail(cudaError_t e) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
  return SS2D_ERR_CUDA;
}

static bool dtype_ok(int d) { return d == SS2D_F32 || d == SS2D_F16 || d == SS2D_BF16; }
static size_t esize(int d) { return d == SS2D_F32 ? 4 : 2; }
static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

constexpr int kStatesPerPass = 32;

static int validate(const ss2d_scan_desc* d) {
  if (!d) return SS2D_ERR_NULL_POINTER;
  if (d->batch <= 0 || d->dim <= 0 || d->seqlen <= 0 || d->dstate <= 0 || d->n_groups <= 0) return SS2D_ERR_BAD_SHAPE;
  if (d->dim % d->n_groups != 0) return SS2D_ERR_BAD_SHAPE;      // reference: selective_scan.cpp:190
  if (d->dstate > SS2D_MAX_DSTATE) return SS2D_ERR_DSTATE;       // reference: selective_scan.cpp:191
  if (!dtype_ok(d->io_dtype) || !dtype_ok(d->out_dtype)) return SS2D_ERR_BAD_DTYPE;
  if (d->out_dtype != d->io_dtype && d->out_dtype != SS2D_F32) return SS2D_ERR_BAD_DTYPE;
  if (d->layout == SS2D_LAYOUT_NATURAL) {
    if (d->H <= 0 || d->W <= 0 || (int64_t)d->H * d->W != d->seqlen) return SS2D_ERR_BAD_SHAPE;
    if (d->n_groups > SS2D_MAX_GROUP_DIRS) return SS2D_ERR_BAD_LAYOUT;
    for (int g = 0; g < d->n_groups; ++g)
      if (d->dirs[g] < 1 || d->dirs[g] > 4) return SS2D_ERR_BAD_LAYOUT;
  } else if (d->layout != SS2D_LAYOUT_SCAN) {
    return SS2D_ERR_BAD_LAYOUT;
  }
  if (d->u_dim_modulo < 0) return SS2D_ERR_BAD_SHAPE;
  if (d->deterministic != 0 && d->deterministic != 1) return SS2D_ERR_BAD_SHAPE;
  return SS2D_OK;
}

static void pack(const ss2d_scan_desc* d, ScanParams& p) {
  memset(&p, 0, sizeof(p));
  p.batch = d->batch; p.dim = d->dim; p.L = d->seqlen; p.N = d->dstate; p.G = d->n_groups;
  p.dpg = d->dim / d->n_groups;
  p.io_dtype = d->io_dtype; p.out_dtype = d->out_dtype; p.softplus = d->delta_softplus;
  p.layout = d->layout; p.H = d->H; p.W = d->W;
  for (int g = 0; g < SS2D_MAX_GROUP_DIRS; ++g) p.dirs[g] = d->layout == SS2D_LAYOUT_NATURAL ? d->dirs[g] : 0;
  p.u_mod = d->u_dim_modulo;
  p.last_il = d->last_state_interleaved;
  p.nck = (d->seqlen + SS2D_CHUNK - 1) / SS2D_CHUNK;
  p.A_ld = d->dstate;
  p.u_bs = d->u_batch_stride; p.u_ds = d->u_dim_stride;
  p.dl_bs = d->delta_batch_stride; p.dl_ds = d->delta_dim_stride;
  p.out_bs = d->out_batch_stride; p.out_ds = d->out_dim_stride;
  p.B_bs = d->B_batch_stride; p.B_gs = d->B_group_stride; p.B_ns = d->B_state_stride;
  p.C_bs = d->C_batch_stride; p.C_gs = d->C_group_stride; p.C_ns = d->C_state_stride;
  p.det = d->deterministic;
}

// TMA bulk copies need 16-byte aligned fp32 rows: every stride a multiple of 4 elements, bases 16-byte aligned
static bool tma_eligible(const ss2d_scan_desc* d, const void* u, const void* delta, const void* B, const void* C,
                         const void* extra) {
  if (d->io_dtype != SS2D_F32 || (d->seqlen & 3)) return false;
  const int64_t strides[] = {d->u_batch_stride, d->u_dim_stride, d->delta_batch_stride, d->delta_dim_stride,
                             d->B_batch_stride, d->B_group_stride, d->B_state_stride,
                             d->C_batch_stride, d->C_group_stride, d->C_state_stride};
  for (int64_t s : strides) if (s & 3) return false;
  return aligned(u, 16) && aligned(delta, 16) && aligned(B, 16) && aligned(C, 16) && (!extra || aligned(extra, 16));
}

// states are processed in passes of <= 32; pass i covers states [n0, n0 + n) = [32 i, 32 i + n)
static int n_passes(int N) { return (N + kStatesPerPass - 1) / kStatesPerPass; }
struct Pass { int n0, n; };
static Pass pass_states(int dstate, int i) {
  const int n0 = i * kStatesPerPass;
  return {n0, std::min(dstate - n0, kStatesPerPass)};
}
static size_t ckpt_floats_pass(const ss2d_scan_desc* d, int n) {
  const size_t nck = (d->seqlen + SS2D_CHUNK - 1) / SS2D_CHUNK;
  return (size_t)d->batch * d->dim * nck * (size_t)n;
}
static size_t round4(size_t x) { return (x + 3) & ~(size_t)3; }

// pass i: state count, kernel variant, whether later passes accumulate; returns the pass' states
static Pass set_pass(ScanParams& p, const ss2d_scan_desc* d, int i) {
  const Pass ps = pass_states(d->dstate, i);
  const Variant v = pick_variant(ps.n);
  p.N = ps.n; p.NP = v.NS * v.R; p.accum = i > 0;
  return ps;
}

// Deterministic mode: one partial slab (batch, G, dstate, L) of dB and one of dC per extra CTA a group is split over, for the
// widest split of any pass. The dispatcher launches with geometries derived from the same per-kernel functions.
static int det_slabs(const ss2d_scan_desc* d) {
  if (!d->deterministic) return 0;
  ScanParams p;
  pack(d, p);
  int smax = 0;
  for (int i = 0; i < n_passes(d->dstate); ++i) {
    set_pass(p, d, i);
    const int s = use_par(p) ? std::max(scan_n1_bwd_det_slabs(p), scan_par_bwd_det_slabs(p)) : scan_bwd_det_slabs(p);
    smax = std::max(s, smax);
  }
  return smax;
}
static size_t slab_stride(const ss2d_scan_desc* d) { return round4((size_t)d->batch * d->n_groups * d->dstate * d->seqlen); }

}  // namespace ss2d

using namespace ss2d;

extern "C" {

size_t ss2d_scan_ckpt_floats(const ss2d_scan_desc* d) {
  if (validate(d) != SS2D_OK) return 0;
  size_t total = 0;
  for (int i = 0; i < n_passes(d->dstate); ++i) total += round4(ckpt_floats_pass(d, pass_states(d->dstate, i).n));
  return total;
}

size_t ss2d_scan_bwd_workspace_bytes(const ss2d_scan_desc* d, int have_ckpt) {
  if (validate(d) != SS2D_OK) return 0;
  const int nmax = d->dstate < kStatesPerPass ? d->dstate : kStatesPerPass;
  size_t floats = round4((size_t)d->batch * d->dim * (nmax + 2));
  if (!have_ckpt) floats += ss2d_scan_ckpt_floats(d);
  const int slabs = det_slabs(d);
  if (slabs > 1) floats += (size_t)2 * (slabs - 1) * slab_stride(d);
  return floats * sizeof(float);
}

int ss2d_scan_fwd(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                  const void* Cmat, const float* Dvec, const float* delta_bias, void* out, float* ckpt,
                  float* last_state, ss2d_stream_t stream) {
  return ss2d_scan_fwd_state(d, u, delta, A, Bmat, Cmat, Dvec, delta_bias, nullptr, out, ckpt, last_state, stream);
}

}  // extern "C"

static int bwd_check(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                     const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, const void* dout,
                     const float* dlast, const float* ckpt, void* du, void* ddelta, float* dA, float* dB, float* dC,
                     float* dD, float* ddelta_bias, float* dh0, void* workspace, size_t workspace_bytes);

// The forward of ss2d_scan_fwd_state; gt.z != nullptr offers the output gate to scan_fwdr when the call is one state pass,
// and *gated reports whether the scan kernel wrote out_z.
static int scan_fwd_impl(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                         const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, void* out, float* ckpt,
                         float* last_state, const ScanGate& gt, ss2d_stream_t stream, bool* gated) {
  *gated = false;
  int rc = validate(d);
  if (rc != SS2D_OK) return rc;
  if (!u || !delta || !A || !Bmat || !Cmat || (!out && !ckpt && !last_state)) return SS2D_ERR_NULL_POINTER;
  if (!aligned(u, esize(d->io_dtype)) || !aligned(delta, esize(d->io_dtype)) || !aligned(Bmat, esize(d->io_dtype)) ||
      !aligned(Cmat, esize(d->io_dtype)) || !aligned(A, 4) || (out && !aligned(out, esize(d->out_dtype))) ||
      (ckpt && !aligned(ckpt, 16)) || !aligned(h0, 16))
    return SS2D_ERR_ALIGNMENT;
  ScanParams p;
  pack(d, p);
  p.u = u; p.delta = delta; p.Dv = Dvec; p.bias = delta_bias; p.out = out; p.last_state = last_state;
  p.tma_ok = tma_eligible(d, u, delta, Bmat, Cmat, nullptr);
  size_t ck_off = 0;
  for (int i = 0; i < n_passes(d->dstate); ++i) {
    const auto [n0, n] = set_pass(p, d, i);
    p.A = A + n0;
    p.Bm = static_cast<const char*>(Bmat) + (size_t)n0 * d->B_state_stride * esize(d->io_dtype);
    p.Cm = static_cast<const char*>(Cmat) + (size_t)n0 * d->C_state_stride * esize(d->io_dtype);
    p.ckpt = ckpt ? ckpt + ck_off : nullptr;
    p.last_state = last_state ? last_state + (d->last_state_interleaved ? 2 : 1) * n0 : nullptr;
    const ScanState st = {h0 ? h0 + n0 : nullptr, nullptr, nullptr};
    ck_off += round4(ckpt_floats_pass(d, n));
    cudaError_t e;
    if (use_par(p)) {      // d_state = 1: lean fp32 kernels (scan_n1.cu) when eligible, else the generic parallel-along-L ones
      if (!scan_n1_fwd_try(p, st, static_cast<cudaStream_t>(stream), &e)) e = scan_par_fwd_dispatch(p, st, static_cast<cudaStream_t>(stream));
    } else if (!scan_fwdr_try(p, st, n_passes(d->dstate) == 1 ? gt : ScanGate{nullptr, nullptr},
                              static_cast<cudaStream_t>(stream), &e, gated)) {     // lane-owns-row fast path (scan_fwdr.cu)
      e = scan_fwd_dispatch(p, st, static_cast<cudaStream_t>(stream));
    }
    if (e != cudaSuccess) return cuda_fail(e);
    ++g_launches;
  }
  return SS2D_OK;
}

extern "C" {

int ss2d_scan_fwd_state(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                        const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, void* out,
                        float* ckpt, float* last_state, ss2d_stream_t stream) {
  bool gated;
  return scan_fwd_impl(d, u, delta, A, Bmat, Cmat, Dvec, delta_bias, h0, out, ckpt, last_state, ScanGate{nullptr, nullptr},
                       stream, &gated);
}

// NULL / alignment / layout checks shared by the gated calls
static int gate_check(const ss2d_scan_desc* d, const void* z, const void* y, const void* g) {
  int rc = validate(d);
  if (rc != SS2D_OK) return rc;
  if (!z || !y || !g) return SS2D_ERR_NULL_POINTER;
  if (d->u_dim_modulo > 0) return SS2D_ERR_UNSUPPORTED;
  if (!aligned(z, esize(d->io_dtype)) || !aligned(y, esize(d->out_dtype)) || !aligned(g, esize(d->out_dtype)))
    return SS2D_ERR_ALIGNMENT;
  return SS2D_OK;
}

int ss2d_scan_fwd_gated(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                        const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, const void* z, void* out,
                        void* out_z, float* ckpt, float* last_state, ss2d_stream_t stream) {
  int rc = gate_check(d, z, out, out_z);
  if (rc != SS2D_OK) return rc;
  bool gated = false;
  rc = scan_fwd_impl(d, u, delta, A, Bmat, Cmat, Dvec, delta_bias, h0, out, ckpt, last_state, ScanGate{z, out_z}, stream, &gated);
  if (rc != SS2D_OK || gated) return rc;
  // every other forward path: y is final only after the call's last kernel (segmented fix-up, last state pass)
  const cudaError_t e = scan_gate_fwd_launch(d, out, z, out_z, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

size_t ss2d_scan_bwd_gated_workspace_bytes(const ss2d_scan_desc* d, int have_ckpt) {
  if (validate(d) != SS2D_OK) return 0;
  return ss2d_scan_bwd_workspace_bytes(d, have_ckpt) + (size_t)d->batch * d->dim * d->seqlen * sizeof(float);
}

int ss2d_scan_bwd_gated(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                        const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, const void* z,
                        const void* out, const void* dout_z, const float* dlast, const float* ckpt, void* du, void* ddelta,
                        float* dA, float* dB, float* dC, float* dD, float* ddelta_bias, void* dz, float* dh0, void* workspace,
                        size_t workspace_bytes, ss2d_stream_t stream) {
  int rc = gate_check(d, z, out, dout_z);
  if (rc != SS2D_OK) return rc;
  if (!dz) return SS2D_ERR_NULL_POINTER;
  if (!aligned(dz, esize(d->io_dtype))) return SS2D_ERR_ALIGNMENT;
  const size_t inner_bytes = ss2d_scan_bwd_workspace_bytes(d, ckpt != nullptr);
  if (!workspace || workspace_bytes < ss2d_scan_bwd_gated_workspace_bytes(d, ckpt != nullptr) || !aligned(workspace, 16))
    return SS2D_ERR_WORKSPACE;
  // dy lives behind the ungated workspace (whose size is a multiple of 16 bytes); the ungated backward reads it as an fp32
  // dout with dense strides, which the workspace query does not depend on
  float* dy = reinterpret_cast<float*>(static_cast<char*>(workspace) + inner_bytes);
  ss2d_scan_desc di = *d;
  di.out_dtype = SS2D_F32;
  di.out_batch_stride = (int64_t)d->dim * d->seqlen;
  di.out_dim_stride = d->seqlen;
  rc = bwd_check(&di, u, delta, A, Bmat, Cmat, Dvec, delta_bias, h0, dy, dlast, ckpt, du, ddelta, dA, dB, dC, dD, ddelta_bias, dh0,
                 workspace, inner_bytes);
  if (rc != SS2D_OK) return rc;
  cudaError_t e = scan_gate_bwd_launch(d, dout_z, z, out, dy, dz, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return ss2d_scan_bwd_state(&di, u, delta, A, Bmat, Cmat, Dvec, delta_bias, h0, dy, dlast, ckpt, du, ddelta, dA, dB, dC, dD,
                             ddelta_bias, dh0, workspace, inner_bytes, stream);
}

int ss2d_scan_bwd(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                  const void* Cmat, const float* Dvec, const float* delta_bias, const void* dout, const float* ckpt,
                  void* du, void* ddelta, float* dA, float* dB, float* dC, float* dD, float* ddelta_bias,
                  void* workspace, size_t workspace_bytes, ss2d_stream_t stream) {
  return ss2d_scan_bwd_state(d, u, delta, A, Bmat, Cmat, Dvec, delta_bias, nullptr, dout, nullptr, ckpt, du, ddelta, dA, dB,
                             dC, dD, ddelta_bias, nullptr, workspace, workspace_bytes, stream);
}

}  // extern "C"

// argument checks of ss2d_scan_bwd_state, also run by ss2d_scan_bwd_gated before it launches anything
static int bwd_check(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                     const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, const void* dout,
                     const float* dlast, const float* ckpt, void* du, void* ddelta, float* dA, float* dB, float* dC,
                     float* dD, float* ddelta_bias, float* dh0, void* workspace, size_t workspace_bytes) {
  int rc = validate(d);
  if (rc != SS2D_OK) return rc;
  if (!u || !delta || !A || !Bmat || !Cmat || !dout || !du || !ddelta || !dA || !dB || !dC) return SS2D_ERR_NULL_POINTER;
  if ((Dvec && !dD) || (delta_bias && !ddelta_bias)) return SS2D_ERR_NULL_POINTER;
  if (!workspace || workspace_bytes < ss2d_scan_bwd_workspace_bytes(d, ckpt != nullptr) || !aligned(workspace, 16))
    return SS2D_ERR_WORKSPACE;
  if (ckpt && !aligned(ckpt, 16)) return SS2D_ERR_ALIGNMENT;
  // element alignment as in the forward; dB / dC are accumulated with 128-bit red.global / vector stores when L % 4 == 0
  const size_t bc_al = (d->seqlen & 3) ? 4 : 16;
  if (!aligned(u, esize(d->io_dtype)) || !aligned(delta, esize(d->io_dtype)) || !aligned(Bmat, esize(d->io_dtype)) ||
      !aligned(Cmat, esize(d->io_dtype)) || !aligned(A, 4) || !aligned(dout, esize(d->out_dtype)) ||
      !aligned(du, esize(d->io_dtype)) || !aligned(ddelta, esize(d->io_dtype)) || !aligned(dA, 4) ||
      !aligned(dB, bc_al) || !aligned(dC, bc_al) || !aligned(h0, 16) || !aligned(dlast, 16) || !aligned(dh0, 16))
    return SS2D_ERR_ALIGNMENT;
  return SS2D_OK;
}

extern "C" {

int ss2d_scan_bwd_state(const ss2d_scan_desc* d, const void* u, const void* delta, const float* A, const void* Bmat,
                        const void* Cmat, const float* Dvec, const float* delta_bias, const float* h0, const void* dout,
                        const float* dlast, const float* ckpt, void* du, void* ddelta, float* dA, float* dB, float* dC,
                        float* dD, float* ddelta_bias, float* dh0, void* workspace, size_t workspace_bytes,
                        ss2d_stream_t stream) {
  int rc = bwd_check(d, u, delta, A, Bmat, Cmat, Dvec, delta_bias, h0, dout, dlast, ckpt, du, ddelta, dA, dB, dC, dD, ddelta_bias,
                     dh0, workspace, workspace_bytes);
  if (rc != SS2D_OK) return rc;
  cudaStream_t cst = static_cast<cudaStream_t>(stream);
  float* ws = static_cast<float*>(workspace);
  const int nmax = d->dstate < kStatesPerPass ? d->dstate : kStatesPerPass;
  float* part = ws;
  float* own_ckpt = ws + round4((size_t)d->batch * d->dim * (nmax + 2));
  float* slab_base = own_ckpt + (ckpt ? 0 : ss2d_scan_ckpt_floats(d));
  const int smax = det_slabs(d);
  if (!ckpt) {   // recompute the chunk states with a forward sweep that writes nothing else
    rc = ss2d_scan_fwd_state(d, u, delta, A, Bmat, Cmat, Dvec, delta_bias, h0, nullptr, own_ckpt, nullptr, stream);
    if (rc != SS2D_OK) return rc;
    ckpt = own_ckpt;
  }
  ScanParams p;
  pack(d, p);
  p.u = u; p.delta = delta; p.Dv = Dvec; p.bias = delta_bias; p.dout = dout; p.du = du; p.ddelta = ddelta;
  p.tma_ok = tma_eligible(d, u, delta, Bmat, Cmat, dout) && d->out_dtype == SS2D_F32 && !(d->out_batch_stride & 3) &&
             !(d->out_dim_stride & 3);
  p.part = part;
  p.slab_stride = (int64_t)slab_stride(d);
  // dA / dD / d(delta_bias) accumulated in place only outside deterministic mode (the N = 1 kernels add per-row sums atomically)
  const int zeroed = d->grads_prezeroed && !d->deterministic;
  size_t ck_off = 0;
  for (int i = 0; i < n_passes(d->dstate); ++i) {
    const auto [n0, n] = set_pass(p, d, i);
    p.A = A + n0;
    p.Bm = static_cast<const char*>(Bmat) + (size_t)n0 * d->B_state_stride * esize(d->io_dtype);
    p.Cm = static_cast<const char*>(Cmat) + (size_t)n0 * d->C_state_stride * esize(d->io_dtype);
    p.ckpt_in = ckpt + ck_off;
    p.dB = dB + (size_t)n0 * d->seqlen;
    p.dC = dC + (size_t)n0 * d->seqlen;
    p.slabB = slab_base + (size_t)n0 * d->seqlen;
    p.slabC = slab_base + (size_t)(smax > 1 ? smax - 1 : 0) * p.slab_stride + (size_t)n0 * d->seqlen;
    const ScanState st = {h0 ? h0 + n0 : nullptr, dlast ? dlast + n0 : nullptr, dh0 ? dh0 + n0 : nullptr};
    ck_off += round4(ckpt_floats_pass(d, n));
    cudaError_t e;
    bool finalize = true;
    int slabs = 0;
    if (use_par(p)) {
      if (scan_n1_bwd_try(p, st, dA, dD, ddelta_bias, zeroed, cst, &e, &slabs)) finalize = !zeroed;
      else e = scan_par_bwd_dispatch(p, st, cst, &slabs);
    } else {
      e = scan_bwd_dispatch(p, st, cst, &slabs);
    }
    if (e != cudaSuccess) return cuda_fail(e);
    ++g_launches;
    if (slabs > 1) {
      e = scan_bwd_fold(p, slabs, cst);
      if (e != cudaSuccess) return cuda_fail(e);
      ++g_launches;
    }
    if (finalize) {
      e = scan_bwd_finalize(p, dA + n0, dD, ddelta_bias, cst);
      if (e != cudaSuccess) return cuda_fail(e);
      ++g_launches;
    }
  }
  return SS2D_OK;
}

int ss2d_state_update(const ss2d_step_desc* d, float* state, const void* x, const void* dt, const float* A, const void* Bmat,
                      const void* Cmat, const float* Dvec, const float* dt_bias, const void* z, void* out, ss2d_stream_t stream) {
  if (!d) return SS2D_ERR_NULL_POINTER;
  if (d->batch <= 0 || d->dim <= 0 || d->dstate <= 0 || d->n_groups <= 0 || d->dim % d->n_groups != 0) return SS2D_ERR_BAD_SHAPE;
  if (d->dstate > SS2D_MAX_DSTATE) return SS2D_ERR_DSTATE;
  if (!dtype_ok(d->io_dtype) || (d->dt_softplus != 0 && d->dt_softplus != 1)) return SS2D_ERR_BAD_DTYPE;
  if (!state || !x || !dt || !A || !Bmat || !Cmat || !out) return SS2D_ERR_NULL_POINTER;
  const size_t es = esize(d->io_dtype);
  if (!aligned(state, 16) || !aligned(x, es) || !aligned(dt, es) || !aligned(Bmat, es) || !aligned(Cmat, es) || !aligned(z, es) ||
      !aligned(out, es) || !aligned(A, 4) || !aligned(Dvec, 4) || !aligned(dt_bias, 4))
    return SS2D_ERR_ALIGNMENT;
  StepParams p;
  p.state = state; p.x = x; p.dt = dt; p.B = Bmat; p.C = Cmat; p.z = z;
  p.A = A; p.D = Dvec; p.bias = dt_bias; p.out = out;
  p.rows = (int64_t)d->batch * d->dim;
  p.dim = d->dim; p.dstate = d->dstate; p.dpg = d->dim / d->n_groups; p.softplus = d->dt_softplus;
  p.io_bs = d->io_batch_stride;
  p.B_bs = d->B_batch_stride; p.B_gs = d->B_group_stride;
  p.C_bs = d->C_batch_stride; p.C_gs = d->C_group_stride;
  const cudaError_t e = ssm_step_launch(p, d->io_dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int ss2d_cross_scan(const void* x, void* xs, int32_t batch, int32_t channels, int32_t H, int32_t W, int32_t K,
                    const int32_t* dirs, int32_t dtype, ss2d_stream_t stream) {
  if (!x || !xs || !dirs) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || channels <= 0 || H <= 0 || W <= 0 || K <= 0 || K > SS2D_MAX_GROUP_DIRS) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  for (int k = 0; k < K; ++k) if (dirs[k] < 1 || dirs[k] > 4) return SS2D_ERR_BAD_LAYOUT;
  cudaError_t e = cross_scan_launch(x, xs, batch, channels, H, W, K, dirs, dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int ss2d_cross_merge(const void* ys, void* y, int32_t batch, int32_t channels, int32_t H, int32_t W, int32_t K,
                     const int32_t* dirs, int32_t dtype, ss2d_stream_t stream) {
  if (!ys || !y || !dirs) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || channels <= 0 || H <= 0 || W <= 0 || K <= 0 || K > SS2D_MAX_GROUP_DIRS) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  for (int k = 0; k < K; ++k) if (dirs[k] < 1 || dirs[k] > 4) return SS2D_ERR_BAD_LAYOUT;
  cudaError_t e = cross_merge_launch(ys, y, batch, channels, H, W, K, dirs, dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int32_t ss2d_out_gate_max_width(int32_t backward) { return epi_max_D(backward != 0); }

int32_t ss2d_out_gate_bwd_partials(int32_t batch, int32_t L) {
  if (batch <= 0 || L <= 0) return 0;
  return epi_bwd_partials(batch, L);
}

int ss2d_out_gate_fwd(const float* ys, int32_t K, const float* ln_weight, const float* ln_bias, const void* z,
                      int64_t z_row_stride, int32_t z_act, void* out, float* mean_rstd, int32_t batch, int32_t D,
                      int32_t L, float eps, int32_t z_dtype, int32_t out_dtype, int32_t H, int32_t W,
                      uint32_t transposed_mask, ss2d_stream_t stream) {
  if (!ys || !out) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || D <= 0 || L <= 0 || K <= 0 || K > SS2D_MAX_GROUP_DIRS) return SS2D_ERR_BAD_SHAPE;
  if (transposed_mask && (H <= 0 || W <= 0 || (int64_t)H * W != L)) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(z_dtype) || !dtype_ok(out_dtype)) return SS2D_ERR_BAD_DTYPE;
  if (D > epi_max_D(false) || (ln_bias && !ln_weight)) return SS2D_ERR_UNSUPPORTED;
  cudaError_t e = out_gate_fwd_launch(ys, K, ln_weight, ln_bias, z, z_row_stride, z_act, out, mean_rstd, batch, D, L, eps,
                                      z_dtype, out_dtype, H, W, transposed_mask, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int ss2d_out_gate_bwd(const float* ys, int32_t K, const float* ln_weight, const float* ln_bias, const void* z,
                      int64_t z_row_stride, int32_t z_act, const void* dout, const float* mean_rstd, float* dy,
                      void* dz, int64_t dz_row_stride, float* dln_weight_partial, float* dln_bias_partial,
                      int32_t n_partials, int32_t batch, int32_t D, int32_t L, int32_t z_dtype, int32_t out_dtype,
                      int32_t H, int32_t W, uint32_t transposed_mask, int32_t dy_two_planes, ss2d_stream_t stream) {
  if (!ys || !dout || !mean_rstd || !dy || !dln_weight_partial || !dln_bias_partial) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || D <= 0 || L <= 0 || K <= 0 || K > SS2D_MAX_GROUP_DIRS) return SS2D_ERR_BAD_SHAPE;
  if ((transposed_mask || dy_two_planes) && (H <= 0 || W <= 0 || (int64_t)H * W != L)) return SS2D_ERR_BAD_SHAPE;
  if (dy_two_planes && (K < 2 || !transposed_mask)) return SS2D_ERR_UNSUPPORTED;      // patch tiles are what makes the second store cheap
  if (n_partials != epi_bwd_partials(batch, L)) return SS2D_ERR_WORKSPACE;
  if (!dtype_ok(z_dtype) || !dtype_ok(out_dtype)) return SS2D_ERR_BAD_DTYPE;
  if (D > epi_max_D(true) || (ln_bias && !ln_weight)) return SS2D_ERR_UNSUPPORTED;
  cudaError_t e = out_gate_bwd_launch(ys, K, ln_weight, ln_bias, z, z_row_stride, z_act, dout, mean_rstd, dy, dz,
                                      dz_row_stride, dln_weight_partial, dln_bias_partial, n_partials, batch, D, L,
                                      z_dtype, out_dtype, H, W, transposed_mask, dy_two_planes, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

static int group_gate_check(int32_t G, const int32_t* plane_of, const float* ln_weight, const float* ln_bias, int32_t batch,
                            int32_t D, int32_t L, int32_t H, int32_t W, int32_t z_dtype, int32_t out_dtype, bool backward) {
  if (!plane_of) return SS2D_ERR_NULL_POINTER;
  if (G <= 0 || G > SS2D_MAX_EPI_GROUPS || batch <= 0 || D <= 0 || L <= 0 || H <= 0 || W <= 0 || (int64_t)H * W != L)
    return SS2D_ERR_BAD_SHAPE;
  // a permutation: the backward writes group g's dy into plane plane_of[g], so two groups on one plane would race
  unsigned seen = 0;
  for (int g = 0; g < G; ++g) {
    if (plane_of[g] < 0 || plane_of[g] >= G || ((seen >> plane_of[g]) & 1u)) return SS2D_ERR_BAD_LAYOUT;
    seen |= 1u << plane_of[g];
  }
  if (!dtype_ok(z_dtype) || !dtype_ok(out_dtype)) return SS2D_ERR_BAD_DTYPE;
  if (D > epi_max_D(backward) || (ln_bias && !ln_weight)) return SS2D_ERR_UNSUPPORTED;
  return SS2D_OK;
}

int ss2d_group_gate_fwd(const float* ys, int32_t G, const int32_t* plane_of, uint32_t transposed_planes,
                        const float* ln_weight, const float* ln_bias, const void* z, int64_t z_row_stride,
                        int64_t z_col0, int64_t z_group_stride, void* out, int64_t out_row_stride, float* mean_rstd,
                        int32_t batch, int32_t D, int32_t L, float eps, int32_t z_dtype, int32_t out_dtype, int32_t H,
                        int32_t W, ss2d_stream_t stream) {
  if (!ys || !z || !out) return SS2D_ERR_NULL_POINTER;
  int rc = group_gate_check(G, plane_of, ln_weight, ln_bias, batch, D, L, H, W, z_dtype, out_dtype, false);
  if (rc != SS2D_OK) return rc;
  cudaError_t e = group_gate_fwd_launch(ys, G, plane_of, transposed_planes, ln_weight, ln_bias, z, z_row_stride, z_col0,
                                        z_group_stride, out, out_row_stride, mean_rstd, batch, D, L, eps, z_dtype, out_dtype,
                                        H, W, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int ss2d_group_gate_bwd(const float* ys, int32_t G, const int32_t* plane_of, uint32_t transposed_planes,
                        const float* ln_weight, const float* ln_bias, const void* z, int64_t z_row_stride,
                        int64_t z_col0, int64_t z_group_stride, const void* dout, int64_t dout_row_stride,
                        const float* mean_rstd, float* dy, void* dz, int64_t dz_row_stride,
                        float* dln_weight_partial, float* dln_bias_partial, int32_t n_partials, int32_t batch,
                        int32_t D, int32_t L, int32_t z_dtype, int32_t out_dtype, int32_t H, int32_t W,
                        ss2d_stream_t stream) {
  if (!ys || !z || !dout || !mean_rstd || !dy || !dz || !dln_weight_partial || !dln_bias_partial) return SS2D_ERR_NULL_POINTER;
  int rc = group_gate_check(G, plane_of, ln_weight, ln_bias, batch, D, L, H, W, z_dtype, out_dtype, true);
  if (rc != SS2D_OK) return rc;
  if (n_partials != epi_bwd_partials(batch, L)) return SS2D_ERR_WORKSPACE;
  cudaError_t e = group_gate_bwd_launch(ys, G, plane_of, transposed_planes, ln_weight, ln_bias, z, z_row_stride, z_col0,
                                        z_group_stride, dout, dout_row_stride, mean_rstd, dy, dz, dz_row_stride,
                                        dln_weight_partial, dln_bias_partial, n_partials, batch, D, L, z_dtype, out_dtype, H, W,
                                        static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

size_t ss2d_dwconv3_wgrad_workspace_bytes(int32_t batch, int32_t C, int32_t H, int32_t W) {
  if (batch <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
  return (size_t)C * dwconv3_wgrad_slabs(batch, C, H, W) * 10 * sizeof(float);
}

int ss2d_dwconv3_wgrad(const float* x, const float* dy, float* dweight, float* dbias, int32_t batch, int32_t C, int32_t H,
                       int32_t W, void* workspace, size_t workspace_bytes, ss2d_stream_t stream) {
  if (!x || !dy || !dweight) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || C <= 0 || H <= 0 || W <= 0 || C > 65535) return SS2D_ERR_BAD_SHAPE;
  const size_t va = (W & 3) == 0 ? 16 : 4;      // W % 4 == 0: the kernel reads x and dy as float4 pixel quads
  if (!aligned(x, va) || !aligned(dy, va) || !aligned(dweight, 4) || !aligned(dbias, 4)) return SS2D_ERR_ALIGNMENT;
  if (!workspace || workspace_bytes < ss2d_dwconv3_wgrad_workspace_bytes(batch, C, H, W) || !aligned(workspace, 4))
    return SS2D_ERR_WORKSPACE;
  cudaError_t e = dwconv3_wgrad_launch(x, dy, dweight, dbias, static_cast<float*>(workspace), batch, C, H, W,
                                       static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  g_launches += 2;
  return SS2D_OK;
}

int32_t ss2d_layernorm_bwd_partials(int64_t rows) { return rows > 0 ? layernorm_bwd_partials(rows) : 0; }

int ss2d_layernorm_fwd(const void* x, const float* weight, const float* bias, void* y, float* mean_rstd, int64_t rows,
                       int32_t C, float eps, int32_t dtype, ss2d_stream_t stream) {
  if (!x || !y) return SS2D_ERR_NULL_POINTER;
  if (rows <= 0 || C <= 0) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  if (C > layernorm_max_C()) return SS2D_ERR_UNSUPPORTED;
  cudaError_t e = layernorm_fwd_launch(x, weight, bias, y, mean_rstd, rows, C, eps, dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int ss2d_layernorm_bwd(const void* x, const float* weight, const void* dy, const float* mean_rstd, void* dx,
                       float* dweight_partial, float* dbias_partial, int32_t n_partials, int64_t rows, int32_t C,
                       int32_t dtype, ss2d_stream_t stream) {
  if (!x || !dy || !mean_rstd || !dx || !dweight_partial || !dbias_partial) return SS2D_ERR_NULL_POINTER;
  if (rows <= 0 || C <= 0) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  if (C > layernorm_max_C()) return SS2D_ERR_UNSUPPORTED;
  if (n_partials != layernorm_bwd_partials(rows)) return SS2D_ERR_WORKSPACE;
  cudaError_t e = layernorm_bwd_launch(x, weight, dy, mean_rstd, dx, dweight_partial, dbias_partial, n_partials, rows, C,
                                       dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

size_t ss2d_wgrad_ts_workspace_bytes(int32_t batch, int32_t rows, int32_t M, int32_t N) {
  if (batch <= 0 || rows <= 0 || !wgrad_ts_supported(M, N)) return 0;
  return wgrad_ts_workspace_floats((int64_t)batch * rows, M, N) * sizeof(float);
}

int ss2d_wgrad_ts(const void* dY, const void* X, float* dW, int32_t batch, int32_t rows, int32_t M, int32_t N,
                  int64_t dy_batch_stride, int64_t dy_row_stride, int64_t dy_col_stride, int64_t x_batch_stride,
                  int64_t x_row_stride, int64_t x_col_stride, int32_t dy_dtype, int32_t x_dtype, void* workspace,
                  size_t workspace_bytes, ss2d_stream_t stream) {
  if (!dY || !X || !dW) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || rows <= 0 || M <= 0 || N <= 0) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dy_dtype) || !dtype_ok(x_dtype)) return SS2D_ERR_BAD_DTYPE;
  if (!wgrad_ts_supported(M, N)) return SS2D_ERR_UNSUPPORTED;
  if (!workspace || workspace_bytes < ss2d_wgrad_ts_workspace_bytes(batch, rows, M, N) || !aligned(workspace, 16))
    return SS2D_ERR_WORKSPACE;
  cudaError_t e = wgrad_ts_launch(dY, X, dW, batch, rows, M, N, dy_batch_stride, dy_row_stride, dy_col_stride,
                                  x_batch_stride, x_row_stride, x_col_stride, dy_dtype, x_dtype,
                                  static_cast<float*>(workspace), static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  g_launches += 2;
  return SS2D_OK;
}

int ss2d_dwconv3_act(int32_t mode, const void* x, const float* weight, const float* bias, const void* dy, void* y,
                     int32_t batch, int32_t C, int32_t H, int32_t W, int32_t dtype, ss2d_stream_t stream) {
  if (!x || !weight || !y || (mode == 1 && !dy)) return SS2D_ERR_NULL_POINTER;
  if (mode < 0 || mode > 2) return SS2D_ERR_UNSUPPORTED;
  if (batch <= 0 || C <= 0 || H <= 0 || W <= 0) return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  const size_t va = (W & 3) == 0 ? 4 * esize(dtype) : esize(dtype);
  if (!aligned(x, va) || !aligned(y, va) || (dy && !aligned(dy, va)) || !aligned(weight, 4)) return SS2D_ERR_ALIGNMENT;
  cudaError_t e = dwconv3_fused_launch(mode, x, weight, bias, dy, y, batch, C, H, W, dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int ss2d_dwnhwc_stencil(const void* x, const void* aux, void* y, int32_t nseg, const int32_t* cbeg, const int32_t* ksize,
                        const float* const* weight, const float* const* bias, int32_t flip, int32_t epi, int32_t batch,
                        int32_t H, int32_t W, int32_t C, int32_t dtype, ss2d_stream_t stream) {
  if (!x || !y || !cbeg || !ksize || !weight || (epi == 3 && !aux)) return SS2D_ERR_NULL_POINTER;
  if (epi < 0 || epi > 3) return SS2D_ERR_UNSUPPORTED;
  if (batch <= 0 || H <= 0 || W <= 0 || C <= 0 || nseg < 1 || nseg > kDwnMaxSeg || (int64_t)batch * H * W >= (1ll << 31))
    return SS2D_ERR_BAD_SHAPE;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  DwnSegs sg;
  memset(&sg, 0, sizeof(sg));
  sg.nseg = nseg;
  if (cbeg[0] != 0 || cbeg[nseg] != C) return SS2D_ERR_BAD_SHAPE;
  for (int s = 0; s < nseg; ++s) {
    if (cbeg[s + 1] <= cbeg[s]) return SS2D_ERR_BAD_SHAPE;
    if (ksize[s] != 0 && ksize[s] != 1 && ksize[s] != 3 && ksize[s] != 5 && ksize[s] != 7) return SS2D_ERR_UNSUPPORTED;
    if (ksize[s] > 1 && !weight[s]) return SS2D_ERR_NULL_POINTER;
    sg.cbeg[s] = cbeg[s]; sg.k[s] = ksize[s]; sg.w[s] = weight[s]; sg.b[s] = bias ? bias[s] : nullptr;
    if (!aligned(sg.w[s], 4) || !aligned(sg.b[s], 4)) return SS2D_ERR_ALIGNMENT;
  }
  sg.cbeg[nseg] = C;
  const size_t va = 2 * esize(dtype);      // channel pairs move as one access when every segment starts on an even channel
  if (!aligned(x, va) || !aligned(y, va) || (aux && !aligned(aux, va))) return SS2D_ERR_ALIGNMENT;
  cudaError_t e = dwnhwc_stencil_launch(x, aux, y, sg, flip != 0, epi, batch, H, W, C, dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

size_t ss2d_dwnhwc_wgrad_workspace_bytes(int32_t batch, int32_t H, int32_t W, int32_t channels, int32_t ksize) {
  if (batch <= 0 || H <= 0 || W <= 0 || channels <= 0 || (ksize != 3 && ksize != 5 && ksize != 7)) return 0;
  return (size_t)dwnhwc_wgrad_slabs(batch, H, W, channels) * channels * (ksize * ksize + 1) * sizeof(float);
}

int ss2d_dwnhwc_wgrad(const void* x, const void* g, int32_t c0, int32_t c1, int32_t ksize, float* dweight, float* dbias,
                      int32_t batch, int32_t H, int32_t W, int32_t C, int32_t dtype, void* workspace, size_t workspace_bytes,
                      ss2d_stream_t stream) {
  if (!x || !g || !dweight) return SS2D_ERR_NULL_POINTER;
  if (batch <= 0 || H <= 0 || W <= 0 || C <= 0 || c0 < 0 || c1 <= c0 || c1 > C || (int64_t)batch * H * W >= (1ll << 31))
    return SS2D_ERR_BAD_SHAPE;
  if (ksize != 3 && ksize != 5 && ksize != 7) return SS2D_ERR_UNSUPPORTED;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  if (!aligned(x, esize(dtype)) || !aligned(g, esize(dtype)) || !aligned(dweight, 4) || !aligned(dbias, 4)) return SS2D_ERR_ALIGNMENT;
  if (!workspace || workspace_bytes < ss2d_dwnhwc_wgrad_workspace_bytes(batch, H, W, c1 - c0, ksize) || !aligned(workspace, 4))
    return SS2D_ERR_WORKSPACE;
  cudaError_t e = dwnhwc_wgrad_launch(x, g, c0, c1 - c0, ksize, dweight, dbias, batch, H, W, C, dtype,
                                      static_cast<float*>(workspace), static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  g_launches += 2;
  return SS2D_OK;
}

int ss2d_dwconv3_act_planes(int32_t mode, const void* x, int64_t x_batch_stride, const float* weight, const float* bias,
                            const void* dy, int64_t dy_batch_stride, const void* dyT, int64_t dyT_batch_stride, void* y,
                            int64_t y_batch_stride, void* yT, int64_t yT_batch_stride, int32_t batch, int32_t C, int32_t H,
                            int32_t W, int32_t dtype, ss2d_stream_t stream) {
  if (!x || !weight || !y || (mode == 1 && !dy)) return SS2D_ERR_NULL_POINTER;
  if (mode < 0 || mode > 1) return SS2D_ERR_UNSUPPORTED;
  if (batch <= 0 || C <= 0 || H <= 0 || W <= 0 || C > 65535 || batch > 65535) return SS2D_ERR_BAD_SHAPE;
  if ((H & 3) || (W & 3)) return SS2D_ERR_UNSUPPORTED;
  if (!dtype_ok(dtype)) return SS2D_ERR_BAD_DTYPE;
  const size_t va = 4 * esize(dtype);
  auto ok = [&](const void* p, int64_t bs) { return !p || (aligned(p, va) && (bs * (int64_t)esize(dtype)) % (int64_t)va == 0); };
  if (!ok(x, x_batch_stride) || !ok(y, y_batch_stride) || !ok(yT, yT_batch_stride) || !ok(dy, dy_batch_stride) ||
      !ok(dyT, dyT_batch_stride) || !aligned(weight, 4))
    return SS2D_ERR_ALIGNMENT;
  cudaError_t e = dwconv3_tiled_launch(mode, x, weight, bias, dy, dyT, y, yT, batch, C, H, W, x_batch_stride, y_batch_stride,
                                       yT_batch_stride, dy_batch_stride, dyT_batch_stride, dtype, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e);
  ++g_launches;
  return SS2D_OK;
}

int32_t ss2d_gate_proj_supported(int32_t D, int32_t C, int32_t K, int32_t dtype) { return gate_proj_tc_supported(D, C, K, dtype) ? 1 : 0; }

int ss2d_gate_proj_fwd(const float* ys, int32_t K, uint32_t transposed_mask, const float* ln_weight, const float* ln_bias, float eps,
                       const void* z, int64_t z_row_stride, int32_t z_act, const void* W, int64_t ldw, const float* bias, void* out,
                       int64_t out_row_stride, void* g_out, int64_t g_row_stride, float* mean_rstd, int32_t batch, int32_t D,
                       int32_t L, int32_t H, int32_t Wd, int32_t C, int32_t dtype, ss2d_stream_t stream) {
  cudaError_t e = cudaSuccess;
  const int rc = gate_proj_tc_launch(ys, K, transposed_mask, ln_weight, ln_bias, eps, z, z_row_stride, z_act, W, ldw, bias, out,
                                     out_row_stride, g_out, g_row_stride, mean_rstd, batch, D, L, H, Wd, C, dtype,
                                     static_cast<cudaStream_t>(stream), &e);
  if (rc == SS2D_ERR_CUDA) return cuda_fail(e);
  if (rc == SS2D_OK) ++g_launches;
  return rc;
}

int32_t ss2d_linear_tc_supported(int32_t n_cols, int32_t K, int32_t dtype) { return linear_tc_supported(n_cols, K, dtype) ? 1 : 0; }

int ss2d_linear_tc(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, int32_t M, int32_t N, int32_t K,
                   int32_t dtype, int32_t n_parts, const ss2d_linear_part* parts, ss2d_stream_t stream) {
  cudaError_t e = cudaSuccess;
  const int rc = linear_tc_launch(A, lda, W, ldw, bias, M, N, K, dtype, n_parts, parts, static_cast<cudaStream_t>(stream), &e);
  if (rc == SS2D_ERR_CUDA) return cuda_fail(e);
  if (rc == SS2D_OK) ++g_launches;
  return rc;
}

const char* ss2d_strerror(int status) {
  switch (status) {
    case SS2D_OK: return "ok";
    case SS2D_ERR_NULL_POINTER: return "a required pointer is NULL";
    case SS2D_ERR_BAD_SHAPE: return "bad shape (sizes must be positive, dim % n_groups == 0, H*W == seqlen)";
    case SS2D_ERR_BAD_DTYPE: return "bad dtype (fp32/fp16/bf16; out dtype must equal io dtype or be fp32)";
    case SS2D_ERR_DSTATE: return "selective_scan only supports state dimension <= 256";
    case SS2D_ERR_BAD_LAYOUT: return "bad layout or scan direction";
    case SS2D_ERR_WORKSPACE: return "workspace missing, misaligned or too small";
    case SS2D_ERR_CUDA: return "CUDA runtime error (see ss2d_last_cuda_error)";
    case SS2D_ERR_UNSUPPORTED: return "unsupported combination";
    case SS2D_ERR_ALIGNMENT: return "pointer not aligned to its element size (checkpoints, and dB / dC when L % 4 == 0: 16 bytes)";
    default: return "unknown status";
  }
}

const char* ss2d_last_cuda_error(void) { return g_cuda_err; }
const char* ss2d_version(void) { return "ss2d_b200 0.2.0 sm_100a"; }
int64_t ss2d_launch_count(int reset) {
  return reset ? g_launches.exchange(0) : g_launches.load();
}
int32_t ss2d_test_force_path(int32_t policy) {
  if (policy < 0 || (policy & 7) > 4 || policy > 12) return SS2D_ERR_BAD_SHAPE;
  g_path_policy.store(policy, std::memory_order_relaxed);
  return SS2D_OK;
}

}  // extern "C"
