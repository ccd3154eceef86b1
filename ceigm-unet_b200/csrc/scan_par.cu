// Selective scan for d_state = 1 — the regime GM-UNet actually runs (4 single-direction SS2Ds with N = 1 per
// GroupMambaLayer, D in {16, 32, 87, 112}, L in {3136, 784, 196, 49}; SURVEY.md §8 table).
//
// With one state there is almost no arithmetic per byte (3 MUFU + ~20 flops per 12 bytes): the path is HBM-bound and
// has far too few (batch, channel) rows to fill 148 SMs with one thread per row. So here the scan is parallel ALONG L:
// a row is owned by T threads, each thread scans P consecutive positions in registers, the T (decay, state) aggregates
// are combined with warp shuffles (Kogge-Stone, plus one shared-memory hop between the warps of a row), and every
// thread fixes its positions up with the carried-in state. Loads and stores are 128-bit, each thread moving its own
// 32/64 contiguous bytes. Longer rows are walked in chunks of T*P positions with the carry kept on chip.
// Replaces the same reference code as scan_fwd.cu / scan_bwd.cu (selective_scan_{fwd,bwd}_kernel.cuh) for N = 1.
#include "scan_params.h"
#include "host_util.h"
#include "scan_tile.cuh"

namespace ss2d {

constexpr int kParThreads = 256;

// P consecutive scan positions [l, l+P) of one row -> registers (zero beyond l_end). Vector path for contiguous
// traversals (SCAN layout, directions 1 and 3), index-mapped scalar path otherwise.
template <int P>
__device__ __forceinline__ void load_seg(const void* __restrict__ src, int dt, int64_t ro, int l, int l_end,
                                         const ScanOrder so, float* out) {
#pragma unroll
  for (int c = 0; c < P; c += 4) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    bool done = false;
    if (l + c + 3 < l_end && so.contiguous()) {
      if (!so.reversed()) {
        if (vec4_ok(src, ro + l + c, dt)) { v = load4(src, ro + l + c, dt); done = true; }
      } else if ((so.L & 3) == 0) {
        const int64_t idx = ro + (so.L - 4 - (l + c));
        if (vec4_ok(src, idx, dt)) { const float4 t = load4(src, idx, dt); v = make_float4(t.w, t.z, t.y, t.x); done = true; }
      }
    }
    if (!done) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (l + c + e < l_end) f4_at(v, e) = load1(src, ro + so.natural(l + c + e), dt);
    }
    out[c] = v.x; out[c + 1] = v.y; out[c + 2] = v.z; out[c + 3] = v.w;
  }
}

// Fast path: fp32, contiguous traversal (forward or reversed), 16-byte aligned row, segment fully inside the row.
// `base` points at the row's first element in memory; rev = traversal runs against memory order.
template <int P>
__device__ __forceinline__ void load_seg_fast(const float* __restrict__ base, int l, int L, bool rev, float* out) {
  if (!rev) {
#pragma unroll
    for (int c = 0; c < P; c += 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + l + c));
      out[c] = v.x; out[c + 1] = v.y; out[c + 2] = v.z; out[c + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int c = 0; c < P; c += 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + (L - 4 - (l + c))));
      out[c] = v.w; out[c + 1] = v.z; out[c + 2] = v.y; out[c + 3] = v.x;
    }
  }
}
template <int P>
__device__ __forceinline__ void store_seg_fast(float* __restrict__ base, int l, int L, bool rev, const float* v) {
  if (!rev) {
#pragma unroll
    for (int c = 0; c < P; c += 4) *reinterpret_cast<float4*>(base + l + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
  } else {
#pragma unroll
    for (int c = 0; c < P; c += 4)
      *reinterpret_cast<float4*>(base + (L - 4 - (l + c))) = make_float4(v[c + 3], v[c + 2], v[c + 1], v[c]);
  }
}
// true when a row starting at element offset `ro` of an fp32 tensor can use the fast path
__device__ __forceinline__ bool row_fast(const void* p, int64_t ro) {
  return ((reinterpret_cast<uintptr_t>(p) + static_cast<uintptr_t>(ro) * 4) & 15) == 0;
}

template <int P>
__device__ __forceinline__ void store_seg(void* __restrict__ dst, int dt, int64_t ro, int l, int l_end, const ScanOrder so,
                                          const float* v, bool accum) {
#pragma unroll
  for (int c = 0; c < P; c += 4)
    store_scan4(dst, dt, ro, l + c, l_end, make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]), so, accum);
}

// Inclusive scan of the affine maps h -> Pm*h + Hm over the SEG lanes of a row segment (composition order: earlier
// lane first). up = true scans towards higher lanes (prefix), false towards lower lanes (suffix).
template <int SEG, bool UP>
__device__ __forceinline__ void seg_scan(float& Pm, float& Hm, int lane_in_seg) {
#pragma unroll
  for (int off = 1; off < SEG; off <<= 1) {
    const float Pp = UP ? __shfl_up_sync(0xffffffffu, Pm, off) : __shfl_down_sync(0xffffffffu, Pm, off);
    const float Hp = UP ? __shfl_up_sync(0xffffffffu, Hm, off) : __shfl_down_sync(0xffffffffu, Hm, off);
    const bool take = UP ? (lane_in_seg >= off) : (lane_in_seg + off < SEG);
    if (take) { Hm = fmaf(Pm, Hp, Hm); Pm *= Pp; }
  }
}

template <int T>
struct ParShape {
  static constexpr int RT = kParThreads / T;            // rows per CTA
  static constexpr int SEG = T < 32 ? T : 32;           // lanes of one row inside a warp
  static constexpr int WPR = T < 32 ? 1 : T / 32;       // warps per row
};

// Exclusive carry for every thread of a row + the row total, given each thread's own map (Pm, Hm).
// Returns (Pex, Hex) = composition of all EARLIER (UP) / LATER (!UP) threads' maps; (Ptot, Htot) = whole row.
template <int T, bool UP>
__device__ __forceinline__ void row_exclusive(float Pm, float Hm, int t, int r, float (*s_agg)[2], float& Pex, float& Hex,
                                              float& Ptot, float& Htot) {
  using S = ParShape<T>;
  const int lis = t % S::SEG, wir = t / 32;
  seg_scan<S::SEG, UP>(Pm, Hm, lis);                    // inclusive within the warp segment
  float Pe = UP ? __shfl_up_sync(0xffffffffu, Pm, 1) : __shfl_down_sync(0xffffffffu, Pm, 1);
  float He = UP ? __shfl_up_sync(0xffffffffu, Hm, 1) : __shfl_down_sync(0xffffffffu, Hm, 1);
  if (UP ? (lis == 0) : (lis == S::SEG - 1)) { Pe = 1.f; He = 0.f; }
  if constexpr (S::WPR == 1) {
    const int src = (threadIdx.x & 31) - lis + (UP ? S::SEG - 1 : 0);
    Ptot = __shfl_sync(0xffffffffu, Pm, src);
    Htot = __shfl_sync(0xffffffffu, Hm, src);
    Pex = Pe; Hex = He;
  } else {
    if (UP ? (lis == 31) : (lis == 0)) { s_agg[r * S::WPR + wir][0] = Pm; s_agg[r * S::WPR + wir][1] = Hm; }
    __syncthreads();
    float Pq = 1.f, Hq = 0.f;                           // composition of the warps before (UP) / after (!UP) this one
    Ptot = 1.f; Htot = 0.f;
#pragma unroll
    for (int i = 0; i < S::WPR; ++i) {
      const int w = UP ? i : S::WPR - 1 - i;            // visit in composition order
      const float Pw = s_agg[r * S::WPR + w][0], Hw = s_agg[r * S::WPR + w][1];
      if (UP ? (w < wir) : (w > wir)) { Hq = fmaf(Pw, Hq, Hw); Pq *= Pw; }
      Htot = fmaf(Pw, Htot, Hw); Ptot *= Pw;
    }
    Hex = fmaf(Pe, Hq, He); Pex = Pe * Pq;
  }
}

// ------------------------------------------------------------------------------------------------- forward
// STATE: the carry-in of a row's first thread is st.h0 instead of 0
template <int T, bool STATE>
__global__ void __launch_bounds__(kParThreads) scan_par_fwd_kernel(const ScanParams p, const ScanState st) {
  using S = ParShape<T>;
  constexpr int P = 16, LC = T * P;
  __shared__ float s_agg[2][S::RT * S::WPR][2];
  const int tid = threadIdx.x, r = tid / T, t = tid % T;
  const int b = blockIdx.z, g = blockIdx.y;
  const int row = blockIdx.x * S::RT + r;                  // channel inside the group
  const bool valid = row < p.dpg;
  const int d = g * p.dpg + (valid ? row : 0);
  const int L = p.L;
  ScanOrder so;
  so.dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
  so.H = p.H; so.W = p.W; so.L = L;
  const int l_end = valid ? L : 0;

  const float A2 = valid ? p.A[(int64_t)d * p.A_ld] * kLog2e : 0.f;
  const float bias = (valid && p.bias) ? p.bias[d] : 0.f;
  const float Dd = (valid && p.Dv && !p.accum) ? p.Dv[d] : 0.f;
  const int64_t u_ro = (int64_t)b * p.u_bs + (int64_t)(p.u_mod > 0 ? d % p.u_mod : d) * p.u_ds;
  const int64_t dl_ro = (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  const int64_t out_ro = (int64_t)b * p.out_bs + (int64_t)d * p.out_ds;
  const int64_t B_ro = (int64_t)b * p.B_bs + (int64_t)g * p.B_gs;
  const int64_t C_ro = (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;

  // one decision per thread: 128-bit unchecked accesses are possible for its rows (fp32, contiguous traversal, aligned)
  const bool rev = so.reversed();
  const bool fast_in = valid && p.io_dtype == SS2D_F32 && so.contiguous() && (L & 3) == 0 && row_fast(p.u, u_ro) &&
                       row_fast(p.delta, dl_ro) && row_fast(p.Bm, B_ro) && row_fast(p.Cm, C_ro);
  const bool fast_out = valid && p.out_dtype == SS2D_F32 && so.contiguous() && (L & 3) == 0 && !p.accum && p.out != nullptr &&
                        row_fast(p.out, out_ro);
  const float* fu = reinterpret_cast<const float*>(p.u) + u_ro;
  const float* fd = reinterpret_cast<const float*>(p.delta) + dl_ro;
  const float* fB = reinterpret_cast<const float*>(p.Bm) + B_ro;
  const float* fC = reinterpret_cast<const float*>(p.Cm) + C_ro;

  float h_carry = (STATE && valid) ? st.h0[state_slot(p, b, d, 0)] : 0.f;
  const int nchunks = (L + LC - 1) / LC;
  for (int c = 0; c < nchunks; ++c) {
    const int l0 = c * LC + t * P;
    const bool full = l0 + P <= l_end;
    float dl[P], uu[P], bb[P];
    if (fast_in && full) {
      load_seg_fast<P>(fd, l0, L, rev, dl);
      load_seg_fast<P>(fu, l0, L, rev, uu);
      load_seg_fast<P>(fB, l0, L, rev, bb);
    } else {
      load_seg<P>(p.delta, p.io_dtype, dl_ro, l0, l_end, so, dl);
      load_seg<P>(p.u, p.io_dtype, u_ro, l0, l_end, so, uu);
      load_seg<P>(p.Bm, p.io_dtype, B_ro, l0, l_end, so, bb);
    }
    // local scan from h = 0: hl = local state, pc = cumulative decay; beyond the end of the row the state is frozen
    float hl[P], pc[P];
    float h = 0.f, pm = 1.f;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      float x = dl[i] + bias;
      if (p.softplus) x = softplus20(x);
      if (l0 + i >= l_end) x = 0.f;
      const float a = ex2f(x * A2);
      h = fmaf(a, h, x * uu[i] * bb[i]);
      pm *= a;
      hl[i] = h; pc[i] = pm;
    }
    // C is not needed before the fix-up: its loads are issued now so that their latency overlaps the row-wide scan
    // (delta and B are dead by here, so the 16 registers are free): 0.237 -> 0.211 ms on the 512^2 batch-64 stage-1 shape.
    // (Staging the next chunk with cp.async into shared memory on top of this was measured slower: 0.254 ms.)
    float cc[P], y[P];
    if (fast_in && full) load_seg_fast<P>(fC, l0, L, rev, cc);
    else load_seg<P>(p.Cm, p.io_dtype, C_ro, l0, l_end, so, cc);
    float Pex, Hex, Ptot, Htot;
    row_exclusive<T, true>(pm, h, t, r, s_agg[c & 1], Pex, Hex, Ptot, Htot);
    const float h_in = fmaf(Pex, h_carry, Hex);             // state entering this thread's first position
#pragma unroll
    for (int i = 0; i < P; ++i) y[i] = fmaf(cc[i], fmaf(pc[i], h_in, hl[i]), Dd * uu[i]);
    if (fast_out && full) store_seg_fast<P>(reinterpret_cast<float*>(p.out) + out_ro, l0, L, rev, y);
    else if (p.out != nullptr) store_seg<P>(p.out, p.out_dtype, out_ro, l0, l_end, so, y, p.accum != 0);
    // chunk checkpoint every SS2D_CHUNK positions: the thread whose last position closes a chunk owns it
    if (p.ckpt != nullptr && valid && ((l0 + P) % SS2D_CHUNK) == 0) {
      const int idx = (l0 + P) / SS2D_CHUNK - 1;
      if (idx < p.nck) p.ckpt[(((int64_t)b * p.dim + d) * p.nck + idx) * p.N] = fmaf(pc[P - 1], h_in, hl[P - 1]);
    }
    h_carry = fmaf(Ptot, h_carry, Htot);
  }
  if (p.last_state != nullptr && valid && t == 0) {
    const int64_t slot = ((int64_t)b * p.dim + d) * p.A_ld;
    if (p.last_il) { p.last_state[2 * slot] = 0.f; p.last_state[2 * slot + 1] = h_carry; }
    else p.last_state[slot] = h_carry;
  }
}

// ------------------------------------------------------------------------------------------------- backward
// DET: dB / dC go to partial slab blockIdx.x with plain stores (summed in slab order by scan_bwd_fold_kernel)
// STATE: chunk 0 starts from st.h0, the reverse carry from st.dlast, and st.dh0 receives the adjoint of h0 (each may be null)
template <int T, bool STATE, bool DET>
__global__ void __launch_bounds__(kParThreads, 2) scan_par_bwd_kernel(const ScanParams p, const ScanState st) {
  using S = ParShape<T>;
  constexpr int P = 8, LC = T * P;
  __shared__ float s_agg[2][S::RT * S::WPR][2];
  __shared__ __align__(16) float s_slab[2][S::RT][LC];     // per-row dB / dC of the current chunk
  __shared__ float s_red[S::RT * S::WPR][3];
  const int tid = threadIdx.x, r = tid / T, t = tid % T;
  const int b = blockIdx.z, g = blockIdx.y;
  const int row = blockIdx.x * S::RT + r;
  const bool valid = row < p.dpg;
  const int d = g * p.dpg + (valid ? row : 0);
  const int L = p.L;
  ScanOrder so;
  so.dir = p.layout == SS2D_LAYOUT_NATURAL ? p.dirs[g] : 0;
  so.H = p.H; so.W = p.W; so.L = L;
  const int l_end = valid ? L : 0;
  const bool single_cta_group = DET || gridDim.x == 1;

  const float A1 = valid ? p.A[(int64_t)d * p.A_ld] : 0.f;
  const float A2 = A1 * kLog2e;
  const float bias = (valid && p.bias) ? p.bias[d] : 0.f;
  const float Dd = (valid && p.Dv && !p.accum) ? p.Dv[d] : 0.f;
  const int du_ch = d, u_ch = p.u_mod > 0 ? d % p.u_mod : d;
  const int64_t u_ro = (int64_t)b * p.u_bs + (int64_t)u_ch * p.u_ds;
  const int64_t du_ro = p.u_mod > 0 ? ((int64_t)b * p.dim + du_ch) * (int64_t)L : (int64_t)b * p.u_bs + (int64_t)d * p.u_ds;
  const int64_t dl_ro = (int64_t)b * p.dl_bs + (int64_t)d * p.dl_ds;
  const int64_t dy_ro = (int64_t)b * p.out_bs + (int64_t)u_ch * p.out_ds;
  const int64_t B_ro = (int64_t)b * p.B_bs + (int64_t)g * p.B_gs;
  const int64_t C_ro = (int64_t)b * p.C_bs + (int64_t)g * p.C_gs;
  float* dBrow = (DET ? det_slab(p, 0, blockIdx.x) : p.dB) + (int64_t)(b * p.G + g) * p.A_ld * L;
  float* dCrow = (DET ? det_slab(p, 1, blockIdx.x) : p.dC) + (int64_t)(b * p.G + g) * p.A_ld * L;

  const bool rev = so.reversed();
  const bool fast_io = valid && p.io_dtype == SS2D_F32 && p.out_dtype == SS2D_F32 && so.contiguous() && (L & 3) == 0 &&
                       !p.accum && row_fast(p.u, u_ro) && row_fast(p.delta, dl_ro) && row_fast(p.dout, dy_ro) &&
                       row_fast(p.Bm, B_ro) && row_fast(p.Cm, C_ro) && row_fast(p.du, du_ro) && row_fast(p.ddelta, dl_ro);
  const float* fu = reinterpret_cast<const float*>(p.u) + u_ro;
  const float* fd = reinterpret_cast<const float*>(p.delta) + dl_ro;
  const float* fy = reinterpret_cast<const float*>(p.dout) + dy_ro;
  const float* fB = reinterpret_cast<const float*>(p.Bm) + B_ro;
  const float* fC = reinterpret_cast<const float*>(p.Cm) + C_ro;

  float t_carry = (STATE && st.dlast && valid) ? st.dlast[state_slot(p, b, d, 0)] : 0.f;   // a_l g_l of the first position of the chunk after this one
  float accA = 0.f, accD = 0.f, accb = 0.f;
  const int nchunks = (L + LC - 1) / LC;
  for (int c = nchunks - 1; c >= 0; --c) {
    const int l0 = c * LC + t * P;
    const bool full = l0 + P <= l_end;
    float dl[P], uu[P], bb[P], cc[P], dy[P];
    if (fast_io && full) {
      load_seg_fast<P>(fd, l0, L, rev, dl);
      load_seg_fast<P>(fu, l0, L, rev, uu);
      load_seg_fast<P>(fy, l0, L, rev, dy);
      load_seg_fast<P>(fB, l0, L, rev, bb);
      load_seg_fast<P>(fC, l0, L, rev, cc);
    } else {
      load_seg<P>(p.delta, p.io_dtype, dl_ro, l0, l_end, so, dl);
      load_seg<P>(p.u, p.io_dtype, u_ro, l0, l_end, so, uu);
      load_seg<P>(p.dout, p.out_dtype, dy_ro, l0, l_end, so, dy);
      load_seg<P>(p.Bm, p.io_dtype, B_ro, l0, l_end, so, bb);
      load_seg<P>(p.Cm, p.io_dtype, C_ro, l0, l_end, so, cc);
    }
    // state entering the chunk: checkpoint written by the forward at the end of the previous SS2D_CHUNK block
    const float h_chunk = (c > 0 && valid)
                              ? __ldg(p.ckpt_in + (((int64_t)b * p.dim + d) * p.nck + (c * LC) / SS2D_CHUNK - 1) * p.N)
                              : (STATE && st.h0 && valid) ? __ldg(st.h0 + state_slot(p, b, d, 0)) : 0.f;
    // ---- forward recompute: a, local h, decay products ----
    float a[P], hh[P];
    float h = 0.f, pm = 1.f;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      float x = dl[i] + bias;
      if (p.softplus) x = softplus20(x);
      if (l0 + i >= l_end) x = 0.f;
      dl[i] = x;
      a[i] = ex2f(x * A2);
      h = fmaf(a[i], h, x * uu[i] * bb[i]);
      pm *= a[i];
      hh[i] = h;
      cc[i] *= dy[i];                                        // c_l = C_l dy_l
    }
    float Pex, Hex, Ptot, Htot;
    row_exclusive<T, true>(pm, h, t, r, s_agg[0], Pex, Hex, Ptot, Htot);
    const float h_in = fmaf(Pex, h_chunk, Hex);              // true state before this thread's first position
    {                                                        // true states: h_i = local_i + (prod a_0..i) h_in
      float pc = 1.f;
#pragma unroll
      for (int i = 0; i < P; ++i) { pc *= a[i]; hh[i] = fmaf(pc, h_in, hh[i]); }
    }
    // ---- reverse: t_l = a_l (c_l + t_(l+1)); g_l = c_l + t_(l+1) ----
    float tl[P];
    float tq = 0.f, qm = 1.f;
#pragma unroll
    for (int i = P - 1; i >= 0; --i) { tq = a[i] * (cc[i] + tq); qm *= a[i]; tl[i] = tq; }
    float Qex, Tex, Qtot, Ttot;
    row_exclusive<T, false>(qm, tq, t, r, s_agg[1], Qex, Tex, Qtot, Ttot);
    const float t_in = fmaf(Qex, t_carry, Tex);              // t of the position right after this thread's last one
    float dub[P], ddl[P], dBv[P], dCv[P];
    {
      float qc = 1.f, t_next = t_in;
#pragma unroll
      for (int i = P - 1; i >= 0; --i) {
        qc *= a[i];
        const float ti = fmaf(qc, t_in, tl[i]);              // true t_i
        const float gi = cc[i] + t_next;                     // true g_i
        t_next = ti;
        const float hprev = i > 0 ? hh[i - 1] : h_in;
        const float sB = gi * bb[i];
        const float w = ti * hprev;
        float dd = fmaf(uu[i], sB, w * A1);
        if (p.softplus) {
          const float de = dl[i];
          dd *= de < 0.015625f ? de * (1.f - de * (0.5f - de * 0.16666667f)) : 1.f - ex2f(-de * kLog2e);
        }
        if (l0 + i >= l_end) dd = 0.f;
        dub[i] = fmaf(Dd, dy[i], dl[i] * sB);
        ddl[i] = dd;
        dBv[i] = gi * dl[i] * uu[i];
        dCv[i] = dy[i] * hh[i];
        accA = fmaf(w, dl[i], accA);
        accD = fmaf(dy[i], uu[i], accD);
        accb += dd;
      }
    }
    if (fast_io && full) {
      store_seg_fast<P>(reinterpret_cast<float*>(p.du) + du_ro, l0, L, rev, dub);
      store_seg_fast<P>(reinterpret_cast<float*>(p.ddelta) + dl_ro, l0, L, rev, ddl);
    } else {
      store_seg<P>(p.du, p.io_dtype, du_ro, l0, l_end, so, dub, p.accum != 0);
      store_seg<P>(p.ddelta, p.io_dtype, dl_ro, l0, l_end, so, ddl, p.accum != 0);
    }
    t_carry = fmaf(Qtot, t_carry, Ttot);
    // ---- dB / dC: sum over the rows of this CTA, then one (vector) reduction per 4 positions to global memory ----
#pragma unroll
    for (int i = 0; i < P; i += 4) {
      *reinterpret_cast<float4*>(&s_slab[0][r][t * P + i]) = make_float4(dBv[i], dBv[i + 1], dBv[i + 2], dBv[i + 3]);
      *reinterpret_cast<float4*>(&s_slab[1][r][t * P + i]) = make_float4(dCv[i], dCv[i + 1], dCv[i + 2], dCv[i + 3]);
    }
    __syncthreads();
    for (int i = tid; i < 2 * (LC / 4); i += kParThreads) {
      const int which = i / (LC / 4), pos = (i - which * (LC / 4)) * 4;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
      for (int rr = 0; rr < S::RT; ++rr) {
        const float4 v = *reinterpret_cast<const float4*>(&s_slab[which][rr][pos]);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
      const int l = c * LC + pos;
      if (l < L) {
        float* dst = which == 0 ? dBrow : dCrow;
        if (so.dir <= 1 && l + 3 < L && (L & 3) == 0) {
          float4* q4 = reinterpret_cast<float4*>(dst + l);
          if (single_cta_group) *q4 = acc;
          else asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(q4), "f"(acc.x), "f"(acc.y), "f"(acc.z), "f"(acc.w) : "memory");
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (l + e < L) {
              float* q1 = dst + so.natural(l + e);
              if (single_cta_group) *q1 = f4_at(acc, e);
              else atomicAdd(q1, f4_at(acc, e));
            }
          }
        }
      }
    }
    __syncthreads();
  }
  if (STATE && st.dh0 && t == 0 && valid) st.dh0[state_slot(p, b, d, 0)] = t_carry;      // a_0 g_0
  // ---- dA, dD, d(delta_bias): sum over the T threads of the row -> per-(batch, channel) partials ----
#pragma unroll
  for (int off = S::SEG / 2; off >= 1; off >>= 1) {
    accA += __shfl_xor_sync(0xffffffffu, accA, off);
    accD += __shfl_xor_sync(0xffffffffu, accD, off);
    accb += __shfl_xor_sync(0xffffffffu, accb, off);
  }
  if constexpr (S::WPR > 1) {
    if ((t & 31) == 0) { s_red[r * S::WPR + t / 32][0] = accA; s_red[r * S::WPR + t / 32][1] = accD; s_red[r * S::WPR + t / 32][2] = accb; }
    __syncthreads();
    if (t == 0) {
      accA = accD = accb = 0.f;
      for (int w = 0; w < S::WPR; ++w) { accA += s_red[r * S::WPR + w][0]; accD += s_red[r * S::WPR + w][1]; accb += s_red[r * S::WPR + w][2]; }
    }
  }
  if (t == 0 && valid) {
    float* dst = p.part + ((int64_t)b * p.dim + d) * (p.N + 2);
    dst[0] = accA; dst[1] = accD; dst[2] = accb;
  }
}

// threads per row: the smallest power of two whose T*P positions cover the row, at most 128 (longer rows are chunked)
static int pick_T(int L, int P) {
  int T = 4;
  while (T < 128 && T * P < L) T <<= 1;
  return T;
}

template <int T, bool STATE>
static cudaError_t launch_par_fwd(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  dim3 grid((p.dpg + ParShape<T>::RT - 1) / ParShape<T>::RT, p.G, p.batch);
  scan_par_fwd_kernel<T, STATE><<<grid, kParThreads, 0, stream>>>(p, st);
  return cudaGetLastError();
}
template <int T, bool DET, bool STATE>
static cudaError_t launch_par_bwd(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  dim3 grid((p.dpg + ParShape<T>::RT - 1) / ParShape<T>::RT, p.G, p.batch);
  static PerDeviceOnce once;   // 16.6 KB of static shared memory per CTA: ask for a carve-out that fits several CTAs per SM
  func_attr_once(once, reinterpret_cast<const void*>(scan_par_bwd_kernel<T, STATE, DET>), cudaFuncAttributePreferredSharedMemoryCarveout, 50);
  scan_par_bwd_kernel<T, STATE, DET><<<grid, kParThreads, 0, stream>>>(p, st);
  return cudaGetLastError();
}
template <bool DET, bool STATE>
static cudaError_t par_bwd_launch(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  switch (pick_T(p.L, 8)) {
    case 4: return launch_par_bwd<4, DET, STATE>(p, st, stream);
    case 8: return launch_par_bwd<8, DET, STATE>(p, st, stream);
    case 16: return launch_par_bwd<16, DET, STATE>(p, st, stream);
    case 32: return launch_par_bwd<32, DET, STATE>(p, st, stream);
    case 64: return launch_par_bwd<64, DET, STATE>(p, st, stream);
    default: return launch_par_bwd<128, DET, STATE>(p, st, stream);
  }
}

template <bool STATE>
static cudaError_t par_fwd_launch(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  switch (pick_T(p.L, 16)) {
    case 4: return launch_par_fwd<4, STATE>(p, st, stream);
    case 8: return launch_par_fwd<8, STATE>(p, st, stream);
    case 16: return launch_par_fwd<16, STATE>(p, st, stream);
    case 32: return launch_par_fwd<32, STATE>(p, st, stream);
    case 64: return launch_par_fwd<64, STATE>(p, st, stream);
    default: return launch_par_fwd<128, STATE>(p, st, stream);
  }
}

cudaError_t scan_par_fwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream) {
  return st.h0 ? par_fwd_launch<true>(p, st, stream) : par_fwd_launch<false>(p, st, stream);
}

// deterministic mode: one slab per CTA along the group (= gridDim.x of launch_par_bwd)
int scan_par_bwd_det_slabs(const ScanParams& p) {
  const int rt = kParThreads / pick_T(p.L, 8);
  return (p.dpg + rt - 1) / rt;
}

cudaError_t scan_par_bwd_dispatch(const ScanParams& p, const ScanState& st, cudaStream_t stream, int* slabs) {
  *slabs = p.det ? scan_par_bwd_det_slabs(p) : 0;
  if (has_state(st)) return p.det ? par_bwd_launch<true, true>(p, st, stream) : par_bwd_launch<false, true>(p, st, stream);
  return p.det ? par_bwd_launch<true, false>(p, st, stream) : par_bwd_launch<false, false>(p, st, stream);
}

}  // namespace ss2d
