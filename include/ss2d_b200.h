/* ss2d_b200.h — C ABI of the B200-native SS2D selective-scan library (libss2d_b200.so).
 *
 * This is the drop-in boundary for GM-UNet's 2D selective-scan hot path. Every entry point takes
 * plain device pointers, sizes, element strides and a CUDA stream; nothing here depends on PyTorch.
 * The library never allocates, never synchronises and keeps no global state: the caller owns all
 * buffers (the reference's host code allocates its outputs with torch the same way,
 * kernels/selective_scan/csrc/selective_scan/cus/selective_scan.cpp:217-220, 307-323).
 *
 * Reference interfaces replaced (paths under /root/reference/gm-unet/):
 *   ss2d_scan_fwd        <- selective_scan_cuda_core.fwd / selective_scan_cuda_oflex.fwd
 *                           kernels/selective_scan/csrc/selective_scan/cus/selective_scan.cpp:157-239
 *                           kernels/selective_scan/csrc/selective_scan/cusoflex/selective_scan_oflex.cpp (out_float)
 *   ss2d_scan_bwd        <- selective_scan_cuda_core.bwd / _oflex.bwd       cus/selective_scan.cpp:241-349
 *   layout NATURAL + dirs <- CrossScan[_1.._4] / CrossMerge[_1.._4] folded into the scan's addressing
 *                           model/gm/csms6s.py:11-206
 *   ss2d_cross_scan / ss2d_cross_merge  <- the same classes as stand-alone permutation kernels (b2 API)
 *   ss2d_out_gate_fwd/bwd <- out_norm LayerNorm + y*SiLU(z) gate   model/gm/ss2d.py:498, 515-517
 *
 * All functions return SS2D_OK (0) or a negative ss2d_status; ss2d_strerror() names it. Kernel
 * launches are asynchronous on `stream`.
 */
#ifndef SS2D_B200_H_
#define SS2D_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* ss2d_stream_t; /* cudaStream_t */

typedef enum {
  SS2D_OK = 0,
  SS2D_ERR_NULL_POINTER = -1,   /* a required pointer is NULL */
  SS2D_ERR_BAD_SHAPE = -2,      /* non-positive size, dim % n_groups != 0, H*W != seqlen ... */
  SS2D_ERR_BAD_DTYPE = -3,      /* dtype enum out of range */
  SS2D_ERR_DSTATE = -4,         /* dstate > SS2D_MAX_DSTATE (reference: MAX_DSTATE 256) */
  SS2D_ERR_BAD_LAYOUT = -5,     /* layout / direction code invalid */
  SS2D_ERR_WORKSPACE = -6,      /* workspace missing or too small */
  SS2D_ERR_CUDA = -7,           /* a CUDA runtime call failed: see ss2d_last_cuda_error() */
  SS2D_ERR_UNSUPPORTED = -8,    /* combination not implemented */
  SS2D_ERR_ALIGNMENT = -9       /* a pointer is not aligned to its element size */
} ss2d_status;

typedef enum { SS2D_F32 = 0, SS2D_F16 = 1, SS2D_BF16 = 2 } ss2d_dtype;

/* SCAN: tensors are already in scan order, (batch, dim, L) — the reference extension's layout.
 * NATURAL: u/delta/out are (batch, dim, H, W) images and B/C are (batch, group, dstate, H, W); each
 * group g is traversed in direction dirs[g] (1 row-major, 2 column-major, 3 reversed row-major,
 * 4 reversed column-major — the CrossScan_1.._4 numbering). No permuted copy is materialised. */
typedef enum { SS2D_LAYOUT_SCAN = 0, SS2D_LAYOUT_NATURAL = 1 } ss2d_layout;

#define SS2D_MAX_DSTATE 256
#define SS2D_MAX_GROUP_DIRS 8
/* groups of one grouped epilogue call (the four SS2Ds of a GroupMambaLayer) */
#define SS2D_MAX_EPI_GROUPS 4
/* checkpoint interval of the chunked scan (elements of L between saved states) */
#define SS2D_CHUNK 32

/* Problem descriptor shared by forward and backward. Strides are in ELEMENTS; the innermost (L or W)
 * stride is 1 for every tensor (the reference requires the same: selective_scan.cpp:180-181,197,199). */
typedef struct ss2d_scan_desc {
  int32_t batch;          /* B */
  int32_t dim;            /* Dt = K * D channels (all groups) */
  int32_t seqlen;         /* L = H * W */
  int32_t dstate;         /* N */
  int32_t n_groups;       /* G: B/C are shared by dim / n_groups consecutive channels */
  int32_t io_dtype;       /* ss2d_dtype of u, delta, B, C, du, ddelta */
  int32_t out_dtype;      /* ss2d_dtype of out and dout (== io_dtype for "core"; SS2D_F32 allowed for "oflex") */
  int32_t delta_softplus; /* 1: delta = softplus(delta + delta_bias), threshold 20 */
  int32_t layout;         /* ss2d_layout */
  int32_t H, W;           /* NATURAL layout only (H * W == seqlen) */
  int32_t dirs[SS2D_MAX_GROUP_DIRS]; /* NATURAL layout only: direction (1..4) of group g */
  /* element strides */
  int64_t u_batch_stride, u_dim_stride;         /* u_group wrap: see u_dim_modulo */
  int64_t delta_batch_stride, delta_dim_stride;
  int64_t out_batch_stride, out_dim_stride;
  int64_t B_batch_stride, B_group_stride, B_state_stride;
  int64_t C_batch_stride, C_group_stride, C_state_stride;
  /* If > 0, channel d reads u at channel (d % u_dim_modulo): lets the K directions of one SS2D share a
   * single (B, D, H, W) input instead of K copies (CrossScan's 4x duplication, csms6s.py:15-19).
   * In the backward, dout is then ALSO shared: (batch, u_dim_modulo, L) with out's strides (every direction
   * receives the merged gradient, csms6s.py:42-53), and du is a dense (batch, dim, L) tensor holding one
   * gradient plane per direction (the caller sums the K planes: CrossScan.backward, csms6s.py:23-29). */
  int32_t u_dim_modulo;
  /* 1: last_state is (batch, dim, 2*dstate) with h in the ODD slots and 0 in the even ones — the layout of
   * the last chunk row of the reference's `x` output (read as x[:, :, -1, 1::2]). */
  int32_t last_state_interleaved;
  /* Backward only. 1: dA, dD and ddelta_bias were ZEROED by the caller (together with dB / dC, e.g. one memset over one
   * buffer) and may be accumulated into; the d_state = 1 path then adds its per-batch sums straight into them and the call is
   * a single kernel. 0: they are fully overwritten (per-batch partials in `workspace` + a fixed-order finalize pass). */
  int32_t grads_prezeroed;
  /* Backward only. 1: every output of ss2d_scan_bwd is a function of its inputs alone — no floating-point sum depends on
   * the order in which CTAs finish, so the results are bit-identical across calls, streams and CUDA-graph replays on the
   * same GPU model with the same library build. The launch geometry depends on the SM count, so results are NOT promised
   * to match across GPU models. dA, dD and ddelta_bias are then fully overwritten whatever grads_prezeroed says; dB / dC
   * are fully written (zeroing them first is harmless). The CTAs that share a group write partial slabs (in `workspace`,
   * see ss2d_scan_bwd_workspace_bytes) that a second pass sums in slab order. 0: the default; values other than 0 / 1
   * are rejected (SS2D_ERR_BAD_SHAPE). */
  int32_t deterministic;
} ss2d_scan_desc;

/* ---- forward -------------------------------------------------------------------------------
 * out[b,d,l] = sum_n C[b,g,n,l] * h[l,n] + D[d] * u[b,d,l],  h[l,n] = exp(dt*A[d,n]) h[l-1,n] + dt*u*B[b,g,n,l]
 * A: (dim, dstate) fp32 contiguous. Dvec, delta_bias: (dim) fp32 or NULL.
 * ckpt: fp32 buffer of ss2d_scan_ckpt_floats(desc) elements, or NULL when no backward will follow.
 *       It receives the state at the end of every SS2D_CHUNK-element chunk (the reference's `x`,
 *       selective_scan.cpp:217-220, at a finer interval) in an internal channel-major order.
 * last_state: (batch, dim, dstate) fp32 or NULL — h after the last element (reference: x[:, :, -1, 1::2]). */
int ss2d_scan_fwd(const ss2d_scan_desc* desc, const void* u, const void* delta, const float* A,
                  const void* Bmat, const void* Cmat, const float* Dvec, const float* delta_bias,
                  void* out, float* ckpt, float* last_state, ss2d_stream_t stream);

size_t ss2d_scan_ckpt_floats(const ss2d_scan_desc* desc);

/* ---- backward ------------------------------------------------------------------------------
 * dout has out's dtype/strides; du, ddelta have u's / delta's dtype and strides.
 * dA (dim, dstate), dD (dim) or NULL, ddelta_bias (dim) or NULL: fp32, fully overwritten (see desc->grads_prezeroed).
 * dB, dC: fp32 (batch, group, dstate, L | H, W) contiguous accumulators that the caller has ZEROED
 *         (the reference does the same: torch::zeros_like(B, fp32), selective_scan.cpp:322-323); 16-byte aligned
 *         when L % 4 == 0 (they are then updated with 128-bit accesses), else SS2D_ERR_ALIGNMENT.
 * ckpt: the buffer written by ss2d_scan_fwd for the same inputs, or NULL: the states are then
 *       recomputed by an extra forward sweep into `workspace`.
 * workspace: ss2d_scan_bwd_workspace_bytes(desc, ckpt != NULL) bytes, 16-byte aligned. */
int ss2d_scan_bwd(const ss2d_scan_desc* desc, const void* u, const void* delta, const float* A,
                  const void* Bmat, const void* Cmat, const float* Dvec, const float* delta_bias,
                  const void* dout, const float* ckpt, void* du, void* ddelta, float* dA, float* dB,
                  float* dC, float* dD, float* ddelta_bias, void* workspace, size_t workspace_bytes,
                  ss2d_stream_t stream);

/* Includes the partial dB / dC slabs when desc->deterministic is 1 (about (S - 1) x 2 x batch x groups x dstate x L floats,
 * S = the most CTAs or warps one group is split over); with it at 0 the size does not depend on the field. */
size_t ss2d_scan_bwd_workspace_bytes(const ss2d_scan_desc* desc, int have_ckpt);

/* ---- state passing: a scan that starts from a given state, and its adjoint ----------------------
 * The same calls as ss2d_scan_fwd / ss2d_scan_bwd (which are these with NULL state pointers), with
 *   h_(-1) = h0 instead of 0:  h_l = exp(dt_l A) h_(l-1) + dt_l u_l B_l, l counted in traversal order (in NATURAL
 *   layout h0 is the state before the first element the direction visits: the last pixel for directions 3 / 4);
 *   backward: the adjoint entering position L - 1 from the right is dlast instead of 0, and dh0 = dloss / dh0 =
 *   exp(dt_0 A) g_0 with g_0 the adjoint of h_0. The terms of h0 in dA and d(delta) at position 0 are included.
 * h0, dlast, dh0: fp32 (batch, dim, dstate) contiguous (last_state's non-interleaved layout), 16-byte aligned, else
 *   SS2D_ERR_ALIGNMENT. h0 / dlast NULL: zeros. dh0 NULL: not computed; else fully overwritten, each element by one thread
 *   (deterministic whatever desc->deterministic says).
 * Chaining: the forward of [0, m) hands its last_state to the forward of [m, L) as h0; the backward of [m, L) hands its
 *   dh0 to the backward of [0, m) as dlast. dA, dD and d(delta_bias) of the two calls add up to those of one call over [0, L).
 * ckpt from a forward given h0 must go to a backward given the same h0; with ckpt == NULL the recompute starts from h0.
 * ss2d_scan_bwd_workspace_bytes applies unchanged. */
int ss2d_scan_fwd_state(const ss2d_scan_desc* desc, const void* u, const void* delta, const float* A,
                        const void* Bmat, const void* Cmat, const float* Dvec, const float* delta_bias,
                        const float* h0, void* out, float* ckpt, float* last_state, ss2d_stream_t stream);
int ss2d_scan_bwd_state(const ss2d_scan_desc* desc, const void* u, const void* delta, const float* A,
                        const void* Bmat, const void* Cmat, const float* Dvec, const float* delta_bias,
                        const float* h0, const void* dout, const float* dlast, const float* ckpt,
                        void* du, void* ddelta, float* dA, float* dB, float* dC, float* dD, float* ddelta_bias,
                        float* dh0, void* workspace, size_t workspace_bytes, ss2d_stream_t stream);

/* ---- output gate: the z argument of mamba_ssm's selective_scan_cuda --------------------------------------------
 * The state calls above with the gate of the Mamba selective-scan contract applied to y = out:
 *   out_z = y * silu(z),  silu(z) = z / (1 + exp(-z));
 *   backward, given dout_z:  dy = dout_z * silu(z) (the ungated backward runs on dy),
 *                            dz = dout_z * y * s * (1 + z (1 - s)),  s = sigmoid(z).
 * z, dz: io dtype; out, out_z, dout_z: out dtype. All five use out's strides (desc->out_*_stride, innermost stride 1).
 * out is still written: the backward reads y from it. NULL z / out / out_z / dout_z / dz: SS2D_ERR_NULL_POINTER; a pointer not
 * aligned to its element size: SS2D_ERR_ALIGNMENT; u_dim_modulo > 0 (a shared dout plane cannot carry per-direction gates):
 * SS2D_ERR_UNSUPPORTED. The gate terms are elementwise, so the gradients are deterministic exactly when the ungated ones are.
 * workspace: ss2d_scan_bwd_gated_workspace_bytes(desc, ckpt != NULL) bytes, 16-byte aligned: the ungated size plus an fp32
 * (batch, dim, L) buffer for dy. */
int ss2d_scan_fwd_gated(const ss2d_scan_desc* desc, const void* u, const void* delta, const float* A,
                        const void* Bmat, const void* Cmat, const float* Dvec, const float* delta_bias,
                        const float* h0, const void* z, void* out, void* out_z, float* ckpt, float* last_state,
                        ss2d_stream_t stream);
size_t ss2d_scan_bwd_gated_workspace_bytes(const ss2d_scan_desc* desc, int have_ckpt);
int ss2d_scan_bwd_gated(const ss2d_scan_desc* desc, const void* u, const void* delta, const float* A,
                        const void* Bmat, const void* Cmat, const float* Dvec, const float* delta_bias,
                        const float* h0, const void* z, const void* out, const void* dout_z, const float* dlast,
                        const float* ckpt, void* du, void* ddelta, float* dA, float* dB, float* dC, float* dD,
                        float* ddelta_bias, void* dz, float* dh0, void* workspace, size_t workspace_bytes,
                        ss2d_stream_t stream);

/* ---- recurrent step: advance a saved state by one position (mamba_ssm's selective_state_update) ------------------
 * Per (b, d, n), g = d / (dim / n_groups), all in fp32:
 *   t = dt[b,d] + dt_bias[d], then t = softplus(t) (threshold 20) when dt_softplus;
 *   state[b,d,n] = exp(t A[d,n]) state[b,d,n] + t x[b,d] B[b,g,n]      (in place);
 *   out[b,d] = sum_n C[b,g,n] state[b,d,n] + D[d] x[b,d], times silu(z[b,d]) when z != NULL; rounded once to the io dtype.
 * state: fp32 (batch, dim, dstate), contiguous, 16-byte aligned: the layout of last_state / h0 / dh0 above, so a scan's final
 *   state is a step's input and the other way round. A: fp32 (dim, dstate) contiguous. Dvec, dt_bias: fp32 (dim) or NULL.
 * x, dt, z, out: (batch, dim) of io_dtype, element (b, d) at b * io_batch_stride + d. B, C: (batch, n_groups, dstate) of
 *   io_dtype, element (b, g, n) at b * X_batch_stride + g * X_group_stride + n. z may be NULL.
 * Errors, returned before any launch: SS2D_ERR_NULL_POINTER (desc, state, x, dt, A, B, C or out NULL), SS2D_ERR_BAD_SHAPE
 * (a size <= 0, dim % n_groups != 0), SS2D_ERR_DSTATE (dstate > SS2D_MAX_DSTATE), SS2D_ERR_BAD_DTYPE (io_dtype, or
 * dt_softplus not 0 / 1), SS2D_ERR_ALIGNMENT (state not 16-byte aligned, an io pointer not aligned to its element size, A / D /
 * dt_bias not 4-byte aligned). One kernel, no atomics: the results are bit-identical across calls and CUDA-graph replays. */
typedef struct ss2d_step_desc {
  int32_t batch;
  int32_t dim;
  int32_t dstate;
  int32_t n_groups;
  int32_t io_dtype;        /* ss2d_dtype of x, dt, B, C, z, out */
  int32_t dt_softplus;     /* 1: t = softplus(dt + dt_bias), threshold 20 */
  /* element strides */
  int64_t io_batch_stride; /* x, dt, z, out */
  int64_t B_batch_stride, B_group_stride;
  int64_t C_batch_stride, C_group_stride;
} ss2d_step_desc;
int ss2d_state_update(const ss2d_step_desc* desc, float* state, const void* x, const void* dt, const float* A,
                      const void* Bmat, const void* Cmat, const float* Dvec, const float* dt_bias, const void* z,
                      void* out, ss2d_stream_t stream);

/* ---- stand-alone cross-scan / cross-merge (exact permutations; model/gm/csms6s.py:11-206) ----
 * cross_scan : x (batch, channels, H, W) -> xs (batch, K, channels, L), xs[:,k] in direction dirs[k].
 * cross_merge: ys (batch, K, channels, L) in scan order -> y (batch, channels, L) natural order,
 *              summed over k in the reference's association ((k0 + k2) + (k1 + k3)) when K == 4.
 * The two are each other's adjoints: the backward of merge is scan and the backward of scan is merge. */
int ss2d_cross_scan(const void* x, void* xs, int32_t batch, int32_t channels, int32_t H, int32_t W,
                    int32_t K, const int32_t* dirs, int32_t dtype, ss2d_stream_t stream);
int ss2d_cross_merge(const void* ys, void* y, int32_t batch, int32_t channels, int32_t H, int32_t W,
                     int32_t K, const int32_t* dirs, int32_t dtype, ss2d_stream_t stream);

/* Largest D the fused epilogue handles (its tiles live in shared memory): forward 1664, backward 832. Wider rows return
 * SS2D_ERR_UNSUPPORTED; the caller composes merge + LayerNorm + gate from separate passes instead (modules.SS2D does). */
int32_t ss2d_out_gate_max_width(int32_t backward);

/* ---- fused epilogue: merge over K + (B,D,L)->(B,L,D) + LayerNorm(D) + SiLU gate ------------------
 * Replaces CrossMerge + the transpose copy + out_norm + act(z) + `y * z` of model/gm/ss2d.py:486-498,
 * 506-508, 515-517 with one pass over HBM.
 * ys: (batch, K, D, L) fp32 per-direction scan outputs in NATURAL pixel order (what ss2d_scan_fwd writes
 *     in NATURAL layout); the K planes are summed on the fly ((k0+k2)+(k1+k3) when K == 4).
 * z:  gate rows, element (b, l, d) at z[(b*L + l) * z_row_stride + d] (a strided view of in_proj's output),
 *     or NULL for no gate; z_act != 0 applies SiLU to z inside the kernel.
 * out: (batch, L, D) channels-last. mean_rstd: (batch, L, 2) fp32 saved for the backward (may be NULL).
 * ln_weight / ln_bias: (D) fp32 or NULL (no affine); a bias without a weight (which nn.LayerNorm cannot produce) is
 *     SS2D_ERR_UNSUPPORTED. D <= 1664 forward, <= 832 backward.
 * transposed_mask: bit k set = plane k of ys is in the pixel order of the TRANSPOSED (W, H) image — how the
 *     column-major directions 2 and 4 are run (as directions 1 and 3 of a transposed input); the kernel undoes
 *     the transposition while merging. H, W are the natural image sizes (only read when the mask is non-zero). */
int ss2d_out_gate_fwd(const float* ys, int32_t K, const float* ln_weight, const float* ln_bias,
                      const void* z, int64_t z_row_stride, int32_t z_act, void* out, float* mean_rstd,
                      int32_t batch, int32_t D, int32_t L, float eps, int32_t z_dtype, int32_t out_dtype,
                      int32_t H, int32_t W, uint32_t transposed_mask, ss2d_stream_t stream);
/* dy: (batch, D, L) fp32 gradient of the MERGED y in natural pixel order — except for K == 1, where it is the
 *     gradient of the single plane and is written in THAT plane's pixel order (transposed when bit 0 of
 *     transposed_mask is set) — (every direction receives the same gradient: pass it to
 *     ss2d_scan_bwd as a shared dout through u_dim_modulo). dz: gradient of the RAW z when z_act != 0, rows
 *     strided by dz_row_stride, or NULL. dy_two_planes != 0 (K > 1, some plane transposed): dy is (batch, 2, D, L) and receives
 *     the merged gradient TWICE, plane 0 in natural and plane 1 in transposed pixel order — the two shared dout planes of
 *     the K = 4 scan backward, written by the kernel that computes them instead of by a transpose-copy + stack.
 *     dln_*_partial: (n_partials, D) fp32, n_partials =
 *     ss2d_out_gate_bwd_partials(batch, L); the caller sums over the first axis. */
int ss2d_out_gate_bwd(const float* ys, int32_t K, const float* ln_weight, const float* ln_bias,
                      const void* z, int64_t z_row_stride, int32_t z_act, const void* dout,
                      const float* mean_rstd, float* dy, void* dz, int64_t dz_row_stride,
                      float* dln_weight_partial, float* dln_bias_partial, int32_t n_partials, int32_t batch,
                      int32_t D, int32_t L, int32_t z_dtype, int32_t out_dtype, int32_t H, int32_t W,
                      uint32_t transposed_mask, int32_t dy_two_planes, ss2d_stream_t stream);
int32_t ss2d_out_gate_bwd_partials(int32_t batch, int32_t L);

/* ---- grouped epilogue: the G single-direction SS2Ds of one GroupMambaLayer in one launch ---------------------
 * (model/gm/groupmamba.py:143-149: four SS2D modules on channel quarters, outputs concatenated along C.)
 * ys: fp32 (batch, G, D, L) scan outputs, one plane per group; group g's plane is plane_of[g], a permutation of 0 ... G - 1
 *     (an index out of range or repeated: SS2D_ERR_BAD_LAYOUT); bit p of transposed_planes: plane p is stored in the pixel
 *     order of the TRANSPOSED image (column-major directions run as row-major scans of it).
 * ln_weight / ln_bias: fp32 (G, D) — each group's own out_norm (ss2d.py:498); as for ss2d_out_gate_fwd, either may be NULL,
 * but a bias without a weight is SS2D_ERR_UNSUPPORTED. z: rows of z_row_stride elements; group g's
 * D gate values start at column z_col0 + g * z_group_stride of a row (raw, SiLU applied here: ss2d.py:506-508, 517).
 * out: (batch, L, ...) rows of out_row_stride elements; group g writes columns g*D ... g*D + D - 1 — the concatenation.
 * mean_rstd: fp32 (G, batch, L, 2), kept for the backward.
 * backward: dy fp32 (batch, G, D, L), plane p in plane p's own pixel order; dz has z's column layout and its own row stride;
 * dln_*_partial: fp32 (G, n_partials, D) with n_partials = ss2d_out_gate_bwd_partials(batch, L), summed by the caller. */
int ss2d_group_gate_fwd(const float* ys, int32_t G, const int32_t* plane_of, uint32_t transposed_planes,
                        const float* ln_weight, const float* ln_bias, const void* z, int64_t z_row_stride,
                        int64_t z_col0, int64_t z_group_stride, void* out, int64_t out_row_stride, float* mean_rstd,
                        int32_t batch, int32_t D, int32_t L, float eps, int32_t z_dtype, int32_t out_dtype, int32_t H,
                        int32_t W, ss2d_stream_t stream);
int ss2d_group_gate_bwd(const float* ys, int32_t G, const int32_t* plane_of, uint32_t transposed_planes,
                        const float* ln_weight, const float* ln_bias, const void* z, int64_t z_row_stride,
                        int64_t z_col0, int64_t z_group_stride, const void* dout, int64_t dout_row_stride,
                        const float* mean_rstd, float* dy, void* dz, int64_t dz_row_stride,
                        float* dln_weight_partial, float* dln_bias_partial, int32_t n_partials, int32_t batch,
                        int32_t D, int32_t L, int32_t z_dtype, int32_t out_dtype, int32_t H, int32_t W,
                        ss2d_stream_t stream);

/* ---- weight / bias gradient of SS2D's depthwise 3 x 3 convolution -----------------------------------
 * dweight[c][ky][kx] = sum_(b,h,w) dy[b,c,h,w] * x[b,c,h+ky-1,w+kx-1] (zero padding 1), dbias[c] = sum dy[b,c,h,w]:
 * the backward of nn.Conv2d(D, D, groups=D, kernel_size=3, padding=1, bias=True) w.r.t. its parameters
 * (model/gm/ss2d.py:316-325, 512). x, dy: fp32 (batch, C, H, W) contiguous; dweight: (C, 1, 3, 3) fp32; dbias: (C) fp32
 * or NULL. Fully overwritten, deterministic. workspace: ss2d_dwconv3_wgrad_workspace_bytes(batch, C, H, W) bytes.
 * x and dy 16-byte aligned when W % 4 == 0 (else 4), dweight / dbias 4-byte aligned, else SS2D_ERR_ALIGNMENT. */
int ss2d_dwconv3_wgrad(const float* x, const float* dy, float* dweight, float* dbias, int32_t batch, int32_t C, int32_t H,
                       int32_t W, void* workspace, size_t workspace_bytes, ss2d_stream_t stream);
size_t ss2d_dwconv3_wgrad_workspace_bytes(int32_t batch, int32_t C, int32_t H, int32_t W);

/* ---- the depthwise stack of the GroupMamba FFNs on channels-last tensors (SURVEY.md §8-f3) -----------------
 * PVT2FFN (model/gm/groupmamba.py:54-83: fc1 -> DWConv 3x3 -> GELU -> fc2; DWConv = :446-455) and custom_ffn
 * (model/gm/custom_mlp.py:338-368: ... -> GELU -> InceptionDWConv2d_MultiScale (:313-336) -> fc2) between the two
 * linear layers. The (B, L, C) token tensor is read as the (batch, H, W, C) channels-last image it is: no NCHW copies.
 *   y = epi(bias[c] + sum_(i,j) weight[c][i][j] * x[b, h+i-P, w+j-P, c]),  zero padding P = k / 2,
 * with the kernel size chosen per channel SEGMENT: channels [cbeg[s], cbeg[s+1]) use ksize[s] in {0, 1, 3, 5, 7}
 * (0: no taps, acc = 0; 1: identity, acc = x, no weight — the untouched channels of the multi-scale block), weight[s] = (channels, 1, k, k) fp32 as nn.Conv2d(groups=channels).weight, bias[s] (fp32) or NULL.
 * nseg <= 4, cbeg[0] = 0, cbeg[nseg] = C. flip = 1 correlates with the flipped kernel (the transposed convolution:
 * data gradient). epi 0: y = acc; 1: y = GELU(acc) (exact erf, nn.GELU()); 2: y = x + acc (the multi-scale residual);
 * 3: y = aux * GELU'(acc) (gradient of the pre-activation, recomputed from x). x, aux, y: `dtype`, contiguous. */
int ss2d_dwnhwc_stencil(const void* x, const void* aux, void* y, int32_t nseg, const int32_t* cbeg, const int32_t* ksize,
                        const float* const* weight, const float* const* bias, int32_t flip, int32_t epi, int32_t batch,
                        int32_t H, int32_t W, int32_t C, int32_t dtype, ss2d_stream_t stream);
/* Weight / bias gradient of one segment [c0, c1) with kernel size ksize in {3, 5, 7}:
 * dweight[c][i][j] = sum_(b,h,w) g[b,h,w,c] x[b,h+i-P,w+j-P,c] ((c1 - c0, 1, k, k) fp32), dbias[c] = sum g (fp32 or NULL).
 * x, g: (batch, H, W, C) of `dtype`. Fully overwritten, deterministic. workspace: ss2d_dwnhwc_wgrad_workspace_bytes. */
int ss2d_dwnhwc_wgrad(const void* x, const void* g, int32_t c0, int32_t c1, int32_t ksize, float* dweight, float* dbias,
                      int32_t batch, int32_t H, int32_t W, int32_t C, int32_t dtype, void* workspace, size_t workspace_bytes,
                      ss2d_stream_t stream);
size_t ss2d_dwnhwc_wgrad_workspace_bytes(int32_t batch, int32_t H, int32_t W, int32_t channels, int32_t ksize);

/* ---- depthwise 3 x 3 convolution fused with SiLU: forward and input gradient -------------------------------
 * nn.Conv2d(D, D, groups=D, kernel_size=3, padding=1) followed by SiLU (model/gm/ss2d.py:512-513) as one pass.
 * x, dy, y: (batch, C, H, W) contiguous tensors of `dtype`; weight: (C, 1, 3, 3) fp32; bias: (C) fp32 or NULL.
 *   mode 0: y = SiLU(bias + conv(x))                       (forward)
 *   mode 1: y = dy * SiLU'(bias + conv(x))                 (gradient of the pre-activation, recomputed from x)
 *   mode 2: y = conv of x with the flipped kernel, no bias (input gradient: pass mode 1's output as x)
 * The parameter gradients come from ss2d_dwconv3_wgrad(x, <mode 1 output>). */
int ss2d_dwconv3_act(int32_t mode, const void* x, const float* weight, const float* bias, const void* dy, void* y,
                     int32_t batch, int32_t C, int32_t H, int32_t W, int32_t dtype, ss2d_stream_t stream);

/* Same convolution + SiLU on (batch, C, H, W) planes addressed by explicit BATCH strides (elements; channel planes are
 * contiguous), H % 4 == 0 and W % 4 == 0, with the cross-scan layout change folded in:
 *   mode 0: y = SiLU(bias + conv(x)); when yT != NULL the result is ALSO stored in transposed pixel order (offset w * H + h)
 *           — the image the column-major scan directions traverse as row-major (model/gm/csms6s.py:95-129, 172-206). y and yT
 *           may be the two halves of one (batch, 2 C, H * W) buffer (batch stride 2 C H W): the scan's input planes, written
 *           by the kernel that produces them, with no permuted copy and no concatenation pass;
 *   mode 1: y = (dy + dyT^T) * SiLU'(bias + conv(x)): dyT (optional) is a second upstream gradient in transposed pixel order. */
int ss2d_dwconv3_act_planes(int32_t mode, const void* x, int64_t x_batch_stride, const float* weight, const float* bias,
                            const void* dy, int64_t dy_batch_stride, const void* dyT, int64_t dyT_batch_stride, void* y,
                            int64_t y_batch_stride, void* yT, int64_t yT_batch_stride, int32_t batch, int32_t C, int32_t H,
                            int32_t W, int32_t dtype, ss2d_stream_t stream);

/* ---- row-wise LayerNorm over C <= 512 channels of channels-last rows --------------------------------
 * Replaces nn.LayerNorm as used by GroupMambaLayer.norm (model/gm/groupmamba.py:131, 156; two applications per layer
 * call with shared weights). x, y, dy, dx: (rows, C) contiguous, dtype = ss2d_dtype; weight / bias: (C) fp32 or NULL.
 * mean_rstd: (rows, 2) fp32, written by the forward (may be NULL there), read by the backward.
 * dweight_partial / dbias_partial: (n_partials, C) fp32 with n_partials = ss2d_layernorm_bwd_partials(rows); the caller
 * sums over the first axis (deterministic). C > 512: SS2D_ERR_UNSUPPORTED. */
int ss2d_layernorm_fwd(const void* x, const float* weight, const float* bias, void* y, float* mean_rstd, int64_t rows,
                       int32_t C, float eps, int32_t dtype, ss2d_stream_t stream);
int ss2d_layernorm_bwd(const void* x, const float* weight, const void* dy, const float* mean_rstd, void* dx,
                       float* dweight_partial, float* dbias_partial, int32_t n_partials, int64_t rows, int32_t C,
                       int32_t dtype, ss2d_stream_t stream);
int32_t ss2d_layernorm_bwd_partials(int64_t rows);

/* ---- weight gradient of the small projections around the scan ("tall-skinny" reduction) -----------------
 * dW[m][n] = sum over (b, r) of dY(b, r, m) * X(b, r, n), fp32 (M, N) contiguous, fully overwritten, deterministic.
 * Replaces the weight-gradient GEMMs autograd/cuBLAS run for in_proj / out_proj (nn.Linear, model/gm/ss2d.py:294,
 * 335, 504, 518), x_proj / dt_proj (the einsums of ss2d.py:465-477) and GroupMambaLayer.proj (groupmamba.py:157)
 * when M x N is tiny and batch * rows huge. Element (b, r, m) of dY lives at
 * dY[b * dy_batch_stride + r * dy_row_stride + m * dy_col_stride] (element strides; either the row or the column
 * stride should be 1 for coalesced reads), likewise X. dtypes: ss2d_dtype of dY / X (fp32 accumulation).
 * Supported: M, N <= 256 and ceil(M/4) * ceil(N/4) <= 256, else SS2D_ERR_UNSUPPORTED (use a library GEMM).
 * workspace: ss2d_wgrad_ts_workspace_bytes(batch, rows, M, N) bytes, 16-byte aligned (0 = unsupported shape). */
int ss2d_wgrad_ts(const void* dY, const void* X, float* dW, int32_t batch, int32_t rows, int32_t M, int32_t N,
                  int64_t dy_batch_stride, int64_t dy_row_stride, int64_t dy_col_stride, int64_t x_batch_stride,
                  int64_t x_row_stride, int64_t x_col_stride, int32_t dy_dtype, int32_t x_dtype, void* workspace,
                  size_t workspace_bytes, ss2d_stream_t stream);
size_t ss2d_wgrad_ts_workspace_bytes(int32_t batch, int32_t rows, int32_t M, int32_t N);

/* ---- tensor-core projections: out = A W^T (+ bias), split into column parts with their own layouts -------------
 * Replaces nn.Linear in_proj + chunk + the NHWC -> NCHW copy of the x half (model/gm/ss2d.py:504-510) and out_proj
 * (ss2d.py:518): tall, skinny GEMMs on tcgen05 tensor cores (TF32 math for fp32 operands, bf16 for bf16; fp32
 * accumulation in tensor memory), A streamed once by TMA, W resident in shared memory.
 * A: (M, K) rows lda elements apart; W: (N, K) rows ldw elements apart (nn.Linear's weight layout); bias: (N) fp32 or NULL.
 * dtype: SS2D_F32 or SS2D_BF16, the type of A, W and every output. A, W and row-major outputs 16-byte aligned with
 * row strides that are multiples of 16 bytes, else SS2D_ERR_ALIGNMENT.
 * The N columns are cut into n_parts <= 4 consecutive parts of n_cols columns each (16 <= n_cols <= 256, multiple of 16;
 * ss2d_linear_tc_supported(n_cols, K, dtype) tells whether W's part fits next to the A ring in shared memory):
 *   planes_L == 0: row-major part, out[m * ld + c];
 *   planes_L  > 0: channel-major planes of planes_L pixels, out[((m / planes_L) * n_cols + c) * planes_L + m % planes_L]
 *                  (M % planes_L == 0): (B, H, W, C) rows in, (B, n_cols, H, W) planes out;
 *   act != 0: SiLU applied to the part. */
typedef struct ss2d_linear_part {
  void* out;
  int64_t ld;
  int32_t n_cols;
  int32_t planes_L;
  int32_t act;
} ss2d_linear_part;
int ss2d_linear_tc(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, int32_t M, int32_t N, int32_t K,
                   int32_t dtype, int32_t n_parts, const ss2d_linear_part* parts, ss2d_stream_t stream);
int32_t ss2d_linear_tc_supported(int32_t n_cols, int32_t K, int32_t dtype);

/* ---- fused epilogue WITH the output projection (north-star property 5) -----------------------------------
 * out = out_proj( LayerNorm_D( merge_K(ys) ) * SiLU(z) ) in one kernel: ss2d_out_gate_fwd followed by nn.Linear(D, C)
 * (model/gm/ss2d.py:486-498, 506-508, 515-518) without the gated tensor's round trip through HBM. The producer warps build
 * the 128-pixel x D operand tile in shared memory in the tensor core's layout, tcgen05.mma multiplies it with the resident
 * weight (TF32 math for SS2D_F32, bf16 for SS2D_BF16; fp32 accumulation in tensor memory).
 * ys: fp32 (batch, K, D, L); bit k of transposed_mask: plane k is in the pixel order of the transposed image.
 * z: rows of z_row_stride elements (batch * L rows, D columns), dtype `dtype`, or NULL; z_act != 0: SiLU(z).
 * W: (C, D) rows ldw elements apart, `dtype`; bias: (C) fp32 or NULL. out: (batch * L, C) rows out_row_stride apart, `dtype`.
 * g_out: optional (batch * L, D) rows: the gated tensor (what out_proj's weight gradient needs); mean_rstd: optional
 * (batch * L, 2) fp32 for ss2d_out_gate_bwd. ln_weight / ln_bias as for ss2d_out_gate_fwd (a bias without a weight:
 * SS2D_ERR_UNSUPPORTED). D % 64 == 0, C % 16 == 0, C <= 256, operand tile + weight within shared memory
 * (ss2d_gate_proj_supported); H % 4 == 0 and Wd % 4 == 0 (the planes are read as TMA boxes); all row pointers / strides
 * 16-byte aligned.
 * C == 0 (W = NULL, out = NULL): epilogue only — the kernel stops after the gate and g_out (required) receives what
 * ss2d_out_gate_fwd would write; the TMA-fed alternative to that kernel for 4-aligned images. */
int ss2d_gate_proj_fwd(const float* ys, int32_t K, uint32_t transposed_mask, const float* ln_weight, const float* ln_bias, float eps,
                       const void* z, int64_t z_row_stride, int32_t z_act, const void* W, int64_t ldw, const float* bias, void* out,
                       int64_t out_row_stride, void* g_out, int64_t g_row_stride, float* mean_rstd, int32_t batch, int32_t D,
                       int32_t L, int32_t H, int32_t Wd, int32_t C, int32_t dtype, ss2d_stream_t stream);
int32_t ss2d_gate_proj_supported(int32_t D, int32_t C, int32_t K, int32_t dtype);

/* ---- misc ------------------------------------------------------------------------------------ */
const char* ss2d_strerror(int status);
const char* ss2d_last_cuda_error(void);   /* thread-local text of the last SS2D_ERR_CUDA */
const char* ss2d_version(void);           /* "ss2d_b200 <semver> sm_100a" */
/* number of this library's kernel launches issued by the calling thread since the last reset */
int64_t ss2d_launch_count(int reset);
/* TEST HOOK, not part of the operator interface. The forward kernel of a d_state 5..16 call is picked by how many warps
 * the call gives the machine (csrc/scan_fwdr.cu); parity tests use this to run a small case through a kernel that only
 * large calls would select. policy 0: automatic (the default, the only value a product caller ever needs); 1: lane-owns-row
 * forward with 32-row warps; 2: the same with 16-row warps; 3: the 8-row-warp forward (scan_fwd.cu) — and, for
 * ss2d_dwnhwc_stencil, the tiled kernel where the single-segment 3 x 3 case would take the column walker (csrc/ffn_dw.cu);
 * 4: the segmented forward of small calls (sequence split over several warps + carry + fix-up kernels, csrc/scan_fwdr.cu).
 * policy + 8: the same path, and ss2d_scan_fwd_gated never applies the gate inside scan_fwdr (its separate pass always runs).
 * Process-wide; returns SS2D_OK or SS2D_ERR_BAD_SHAPE. */
int32_t ss2d_test_force_path(int32_t policy);

#ifdef __cplusplus
}
#endif
#endif /* SS2D_B200_H_ */
