// "v2" transform of the NUFFT Lomb-Scargle path (included by ls_nufft.cu; also compiled for the CPU through
// tests/native/cuda_emu.h).  Every light curve is ONE REAL series on the fine grid of M = 2^p cells, transformed as a
// complex series of Mh = M / 2 points  z[n] = g[2n] + i g[2n + 1]:
//     G[k] = E[k] + exp(2 pi i k / M) O[k],   E = (Z[k] + conj Z[Mh - k]) / 2,   O = (Z[k] - conj Z[Mh - k]) / 2i.
// (Round 2, hardware finding: packing TWO light curves into one complex transform leaks the partner's spectral peak
// into a quiet light curve with relative weight ~1e-7 - fp32 rounding of Z at the partner's peak bin - which is
// 2-3x the parity tolerance when the partner is >~ 300x louder; tools/worst_bins_detail.py.  A light curve's own
// transform has no such cross-talk, batches of odd size need no padding, and the result of a light curve no longer
// depends on its neighbour.)
//
// Mh = A * Bc, Bc = 2^V2_PB = 512 fixed, A = 2^pa;  n = n1 Bc + n2,  k = k1 + A k2  (four-step transform):
//   spread : G[lc][c][n1][j]   (c = n2 / TC, j = n2 % TC, TC = 8192 / A columns per CTA), rows n1 < n1max only -
//            the cadences reach just the first df * baseline (20 % at lightkurve's default oversampling) of the grid;
//            kernel weights come from a per-cadence table (built once per call), one thread = one z cell = two fine
//            grid cells of LCS light curves;
//   cols   : one CTA = TC columns of one light curve: length-A transforms over n1 in shared memory (in place, one
//            radix-16 butterfly per thread and pass, twiddles from tables), times exp(2 pi i n2 k1 / Mh), written as
//            T[lc][c][k1][j] - one contiguous 64 KB block per CTA;
//   rows   : one tile = rows k1 = 1 + 8 g .. 8 (g + 1) and their mirror rows A - k1 of one light curve: length-Bc
//            transforms over n2 (persistent CTAs, two tiles in flight and the next one arriving: v2_ring), then the finish (unpack E / O, deconvolve + tau rotation through one folded table,
//            epilogue) -> power, written in 32-byte runs (8 consecutive k1 at one k2 are 8 consecutive frequency
//            bins); the transform itself never goes back to global memory.  The tile that would hold row A / 2 twice
//            takes row 0 (which mirrors onto itself) instead.
// All tile geometry is compile-time (template parameter PA): every shared-memory offset inside the passes is
// `runtime base + constant`.
#pragma once
#include "nufft_core.h"
#include "ptx.cuh"

namespace lkb {
namespace {

using nufft::V2_PB;
using nufft::V2_THREADS;
using nufft::V2_TILE;
constexpr int V2_LOG_TILE = 13;
static_assert((1 << V2_LOG_TILE) == V2_TILE, "tile size");
constexpr int V2_BC = 1 << V2_PB;
constexpr int V2_R = V2_TILE / (2 * V2_BC);                     // rows per block of the row kernel (8)
constexpr int V2_LSB = V2_BC + V2_BC / 16 + 1;                  // skewed line of Bc points
// real-mode limits: Mh = 2^(p - 1) = A * Bc with 16 <= A <= 8192
constexpr int V2R_P_MIN = V2_PB + 4 + 1, V2R_P_MAX = V2_PB + 13 + 1;

__host__ __device__ constexpr int v2_radix(int plog, int idx) {
  return (idx < plog / 4) ? 16 : ((idx == plog / 4 && (plog % 4)) ? (1 << (plog % 4)) : 0);
}
__host__ __device__ constexpr int v2_log2i(int r) { return r == 16 ? 4 : r == 8 ? 3 : r == 4 ? 2 : r == 2 ? 1 : 0; }
__device__ __forceinline__ int v2_skew(int a) { return a + (a >> 4); }
// offset of input r of a butterfly (r * nb points further) in a skewed line; exact because the butterfly index is
// either a multiple-of-16 aligned case (nb % 16 == 0) or smaller than nb <= 8
template <int nb>
__host__ __device__ constexpr int v2_in_off(int r) {
  return (nb % 16 == 0) ? r * (nb + nb / 16) : r * nb + ((r * nb) >> 4);
}

// ---- tables -------------------------------------------------------------------------------------------------------
// pass tables of the length-A and the length-Bc transforms, the two-level inter-step table of exp(2 pi i q / Mh)
template <class CT>
__global__ void nufft2_tables_kernel(int pa, int pb, int ph, CT* __restrict__ tw_a, CT* __restrict__ tw_b,
                                     CT* __restrict__ t_hi, CT* __restrict__ t_lo) {
  const int la = nufft::v2_pass_table_len(pa), lb = nufft::v2_pass_table_len(pb), pl = nufft::v2_log2_lo(ph);
  const int nlo = 1 << pl, nhi = 1 << (ph - pl);
  int e = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  int64_t num = 0, den = 1;
  CT* dst = nullptr;
  if (e < la) { nufft::v2_pass_table_entry(pa, e, &num, &den); dst = tw_a + e; }
  else if ((e -= la) < lb) { nufft::v2_pass_table_entry(pb, e, &num, &den); dst = tw_b + e; }
  else if ((e -= lb) < nhi) { num = e; den = nhi; dst = t_hi + e; }
  else if ((e -= nhi) < nlo) { num = e; den = (int64_t)1 << ph; dst = t_lo + e; }
  else return;
  double sn, cs;
  sincospi(2.0 * (double)num / (double)den, &sn, &cs);
  typedef typename nufft::CplxOf<CT>::real RT;
  *dst = nufft::CplxOf<CT>::mk((RT)cs, (RT)sn);
}

// kernel weights of every cadence: Wt[n w + q] = phi((i0_n + q - x_n) / (w / 2)), q = 0 .. w - 1, evaluated in FP64
// from the time stamp itself and rounded once.  (Round 2, hardware finding: with fp32 offsets and expf the weights
// carry ~1e-6 relative errors - a perturbation of the kernel SHAPE that the deconvolution does not undo; it leaked
// strong lines from above the frequency band into the band at 2e-8 of their amplitude, 1.5x the tolerance on light
// curves whose in-band spectrum is 1000x below their variability, and a WIDER kernel made it worse, not better.)
template <class RT>
__global__ void nufft2_weights_kernel(const double* __restrict__ t, int64_t N, double df, int64_t M, int w, double beta,
                                      RT* __restrict__ Wt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N * w) return;
  const int64_t n = e / w;
  const int q = (int)(e - n * w);
  const double x = df * t[n] * (double)M + (double)nufft::grid_shift(w);       // as nufft::cad_entry
  const double i0 = ceil(x - 0.5 * (double)w);
  const double z = (i0 + (double)q - x) * (2.0 / (double)w);
  const double s2 = 1.0 - z * z;
  Wt[e] = (s2 > 0.0) ? (RT)exp(beta * (sqrt(s2) - 1.0)) : (RT)0.0;
}

// z index (n = n1 Bc + n2) of position e of the G layout [c][n1][j]
__device__ __forceinline__ int64_t v2_zcell_of(int64_t e, int ptc, int n1max) {
  const int64_t j = e & (((int64_t)1 << ptc) - 1), rest = e >> ptc;
  const int64_t n1 = rest % n1max, c = rest / n1max;
  return (n1 << V2_PB) + (c << ptc) + j;
}

// ---- spread -------------------------------------------------------------------------------------------------------
// G[lc][e] = (cell 2n, cell 2n + 1) of light curves lc0 .. lc0 + LCS - 1; grid (ceil(cells / 256), ceil(B / LCS)).
// y rows [B, ystride] (centred flux); no scaling: a light curve's transform is its own.
template <int LCS>
__global__ void __launch_bounds__(256)
nufft2_spread_kernel(const int32_t* __restrict__ first_ge, const nufft::Cad* __restrict__ cad,
                     const float* __restrict__ Wt, const float* __restrict__ y, int64_t ystride, int B, int w, int p,
                     int ptc, int n1max, float2* __restrict__ G) {
  const int64_t cells = (int64_t)n1max << V2_PB;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= cells) return;
  const int64_t M = (int64_t)1 << p, m = 2 * v2_zcell_of(e, ptc, n1max);
  const int lc0 = (int)blockIdx.y * LCS;
  const float* yr[LCS];
#pragma unroll
  for (int q = 0; q < LCS; ++q) {
    int b = lc0 + q;
    if (b > B - 1) b = B - 1;                      // clamped rows are computed and dropped
    yr[q] = y + (int64_t)b * ystride;
  }
  float a0[LCS], a1[LCS];
#pragma unroll
  for (int q = 0; q < LCS; ++q) { a0[q] = 0.0f; a1[q] = 0.0f; }
  const int64_t L = nufft::table_len(M, w);
  for (int wrap = 0; wrap < 2; ++wrap) {           // wrap = 1: cadences whose support runs past cell M - 1
    const int64_t mm = m + (int64_t)wrap * M;
    if (mm + 1 >= L) break;
    int64_t lo_c = mm - w + 1, hi_c = mm + 2;
    if (lo_c < 0) lo_c = 0;
    if (hi_c > L - 1) hi_c = L - 1;
    const int32_t na = first_ge[lo_c], nb = first_ge[hi_c];          // cadences with mm - w + 1 <= i0 <= mm + 1
    for (int32_t n = na; n < nb; ++n) {
      const int tap = (int)(mm - (int64_t)cad[n].i0);                // in [-1, w - 1]
      const float* wr = Wt + (int64_t)n * w;
      const float w0 = (tap >= 0) ? wr[tap] : 0.0f;                  // weight on cell mm
      const float w1 = (tap + 1 < w) ? wr[tap + 1] : 0.0f;           // weight on cell mm + 1
#pragma unroll
      for (int q = 0; q < LCS; ++q) {
        const float v = yr[q][n];
        a0[q] = fmaf(w0, v, a0[q]);
        a1[q] = fmaf(w1, v, a1[q]);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < LCS; ++q)
    if (lc0 + q < B) G[(int64_t)(lc0 + q) * cells + e] = make_float2(a0[q], a1[q]);
}

// ---- who works on a tile -----------------------------------------------------------------------------------------
// V2Cta: all V2_THREADS threads of a CTA (the double-precision list kernels): __syncthreads, tile loads through
// registers.  V2Half: group g of the two V2_THREADS-thread groups of a ring CTA (v2_ring): named barrier 1 + g, tile
// loads as cp.async copies that land while the group computes another tile.
struct V2Cta {
  __device__ __forceinline__ int tid() const { return (int)threadIdx.x; }
  __device__ __forceinline__ void sync() const { __syncthreads(); }
  template <class CT>
  __device__ __forceinline__ void put(CT* dst, const CT* src, bool ok) const {
    *dst = ok ? *src : nufft::CplxOf<CT>::mk(0, 0);
  }
};
struct V2Half {                     // (stateless: the group and the thread index are read afresh, see ptx::tid_x)
  __device__ __forceinline__ static int group() { return ptx::tid_x() / V2_THREADS; }
  __device__ __forceinline__ int tid() const { return ptx::tid_x() & (V2_THREADS - 1); }
  __device__ __forceinline__ void sync() const { ptx::bar_sync_named(1 + group(), V2_THREADS); }
  __device__ __forceinline__ void put(float2* dst, const float2* src, bool ok) const {
    ptx::cp_async_8(dst, src, ok ? 8u : 0u);
  }
};

// ---- in-place passes over the lines of a tile (compile-time geometry) ---------------------------------------------
// PLOG: log2 of the line length, LS: skewed line stride, IDX / NS: pass number and the product of earlier radices.
// nz (first pass only): line positions >= nz hold zeros that were never stored - they are not read either
template <int PLOG, int LS, int IDX, int NS, class CT, class Grp>
__device__ __forceinline__ void v2_pass_t(CT* buf, const CT* __restrict__ tw, const Grp gp, int nz = 1 << 30) {
  constexpr int R = v2_radix(PLOG, IDX);
  if constexpr (R != 0) {
    constexpr int LR = v2_log2i(R), NB = 16 / R, PNB = PLOG - LR, nb = 1 << PNB;      // nb butterflies per line
    constexpr bool WIDE = nb > V2_THREADS;           // one line, several butterflies of it per thread
    static_assert(WIDE || (V2_THREADS % nb) == 0, "geometry");
    // per-input offset r * nb in the skewed line: v2_in_off<nb>(r)
    const int t = gp.tid();
    CT u[NB][R];
    int base_in[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      int line, i;
      if constexpr (WIDE) { line = 0; i = t + V2_THREADS * q; }
      else { line = (t >> PNB) + ((V2_THREADS * q) >> PNB); i = t & (nb - 1); }
      base_in[q] = line * LS + ((nb % 16 == 0) ? v2_skew(i) : i);
#pragma unroll
      for (int r = 0; r < R; ++r)
        u[q][r] = (IDX > 0 || r * nb < nz) ? buf[base_in[q] + v2_in_off<nb>(r)] : nufft::CplxOf<CT>::mk(0, 0);
    }
    gp.sync();
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      int line, i;
      if constexpr (WIDE) { line = 0; i = t + V2_THREADS * q; }
      else { line = (t >> PNB) + ((V2_THREADS * q) >> PNB); i = t & (nb - 1); }
      const int k = i & (NS - 1);
      if constexpr (NS > 1) {
#pragma unroll
        for (int r = 1; r < R; ++r) u[q][r] = nufft::cmul(u[q][r], tw[r * NS + k]);
      }
      nufft::SmallDft<R, CT>::run(u[q]);
      const int j = ((i - k) << LR) + k;
      // NS = 1 (then R = 16): skew(16 i + r) = 17 i + r;  NS >= 16: skew(j + r NS) = skew(j) + r NS 17 / 16
      const int base_out = line * LS + ((NS == 1) ? (j + i) : v2_skew(j));
#pragma unroll
      for (int r = 0; r < R; ++r) buf[base_out + ((NS == 1) ? r : r * (NS + NS / 16))] = u[q][r];
    }
    gp.sync();
    v2_pass_t<PLOG, LS, IDX + 1, NS * R, CT>(buf, tw + ((IDX > 0) ? R * NS : 0), gp);
  }
}

// Number of transforms a launch works on: the grid's y extent, or (escalation pass, sized before the host knows how many
// light curves were listed) the device-side count minus `base`, at most `cap`; blocks stride over them by gridDim.y.
struct V2Count {
  const int* count;     // NULL: gridDim.y transforms
  int base, cap;
};
__device__ __forceinline__ int v2_count(const V2Count nc, int grid_y) {
  if (!nc.count) return grid_y;
  const int n = *nc.count - nc.base;
  return n < 0 ? 0 : (n > nc.cap ? nc.cap : n);
}

// ---- cols ---------------------------------------------------------------------------------------------------------
// G: pruned fine grids [B][c][n1 < n1max][j]; T: [B][c][k1][j].  Tile (lc, c): the TC columns c TC .. of light curve
// slot lc, one length-A transform per column.
template <int PA>
struct V2Cols {
  static constexpr int A = 1 << PA, PTC = V2_LOG_TILE - PA, TC = 1 << PTC, LS = A + A / 16 + 1, C = V2_BC / TC;
  static constexpr int ELEMS = TC * LS;                           // points of one tile in shared memory
  // one sweep of the 512 threads covers JW columns x RW rows (RW is a multiple of 16: constant skew increments)
  static constexpr int JW = TC < 32 ? TC : 32, RW = V2_THREADS / JW, CG = TC / JW;
  static constexpr int LJW = JW == 32 ? 5 : JW == 16 ? 4 : JW == 8 ? 3 : JW == 4 ? 2 : JW == 2 ? 1 : 0;
  static_assert((1 << LJW) == JW && RW % 16 == 0, "geometry");
  // rows the first pass reads: whole input blocks (of A / R1 rows) that contain a row < n1max
  static constexpr int NB1 = A / v2_radix(PA, 0);
  __device__ __forceinline__ static int nz(int n1max) { return ((n1max + NB1 - 1) / NB1) * NB1; }
};
// tile (lc, c) of G -> buf (rows < nz; rows >= n1max as zeros)
template <int PA, class CT, class Grp>
__device__ __forceinline__ void v2_cols_load(CT* buf, const CT* __restrict__ G, int n1max, const int64_t lc, const int c,
                                             const Grp gp) {
  using Q = V2Cols<PA>;
  const int t = gp.tid();
  const int jl = t & (Q::JW - 1), nl = t >> Q::LJW;
  const int nvalid = n1max << Q::PTC, nz = Q::nz(n1max);
  const CT* Gp = G + (lc * Q::C + c) * (int64_t)nvalid;
  const int s_base = jl * Q::LS + v2_skew(nl), g_base = nl * Q::TC + jl;
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int cg = u % Q::CG, nbk = u / Q::CG;                     // column group, row block of this sweep
    if (nbk * Q::RW < nz) {
      const int idx = g_base + nbk * Q::RW * Q::TC + cg * Q::JW;
      gp.put(buf + s_base + cg * Q::JW * Q::LS + nbk * (Q::RW + Q::RW / 16), Gp + (idx < nvalid ? idx : 0), idx < nvalid);
    }
  }
}
// the loaded tile: length-A transforms in shared memory (in place), times exp(2 pi i n2 k1 / Mh) -> T
template <int PA, class CT, class Grp>
__device__ __forceinline__ void v2_cols_one(CT* buf, CT* __restrict__ T, int n1max, const CT* __restrict__ tw_a,
                                            const CT* __restrict__ t_hi, const CT* __restrict__ t_lo, const int64_t lc,
                                            const int c, const Grp gp) {
  using Q = V2Cols<PA>;
  const int t = gp.tid();
  const int jl = t & (Q::JW - 1), nl = t >> Q::LJW;
  const int s_base = jl * Q::LS + v2_skew(nl), g_base = nl * Q::TC + jl;
  v2_pass_t<PA, Q::LS, 0, 1, CT>(buf, tw_a, gp, Q::nz(n1max));
  CT* Tp = T + (lc * Q::C + c) * (int64_t)V2_TILE;
  const int ph = PA + V2_PB, pl = nufft::v2_log2_lo(ph);
  const unsigned Mmask = (1u << ph) - 1u, lmask = (1u << pl) - 1u;
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int cg = u % Q::CG, nbk = u / Q::CG;
    const int k1 = nl + nbk * Q::RW, n2 = c * Q::TC + jl + cg * Q::JW;
    const unsigned q = ((unsigned)n2 * (unsigned)k1) & Mmask;       // n2 k1 < 2^22
    const CT wq = nufft::cmul(t_hi[q >> pl], t_lo[q & lmask]);
    Tp[g_base + nbk * Q::RW * Q::TC + cg * Q::JW] =
        nufft::cmul(buf[s_base + cg * Q::JW * Q::LS + nbk * (Q::RW + Q::RW / 16)], wq);
  }
}
// grid (Bc / TC, B): one tile per CTA, 2 CTAs/SM.  (Kept free of any extra kernel parameter: it sits exactly at the
// 64-register cap, and a 16-byte parameter more made ptxas spill 184 bytes - 1.12 -> 1.66 ms,
// profiles/launches_r02_c2_escalation_v2_spill.csv.  The persistent ring form of v2_ring measured slower here: 1.25
// instead of 1.13 ms at config 2 on a B200 - the 16 loads a thread has in flight already cover most of the gather.)
template <int PA>
__global__ void __launch_bounds__(V2_THREADS, 2)
nufft2_cols_kernel(const float2* __restrict__ G, float2* __restrict__ T, int n1max, const float2* __restrict__ tw_a,
                   const float2* __restrict__ t_hi, const float2* __restrict__ t_lo) {
  LKB_DYN_SMEM(float2, buf);
  v2_cols_load<PA>(buf, G, n1max, (int64_t)blockIdx.y, (int)blockIdx.x, V2Cta());
  __syncthreads();
  v2_cols_one<PA>(buf, T, n1max, tw_a, t_hi, t_lo, (int64_t)blockIdx.y, (int)blockIdx.x, V2Cta());
}
// escalation pass (double precision): grid (Bc / TC, gy); blocks stride over a device-side count of transforms
template <int PA>
__global__ void __launch_bounds__(V2_THREADS, 1)
nufft2_cols_list_kernel(const double2* __restrict__ G, double2* __restrict__ T, int n1max,
                        const double2* __restrict__ tw_a, const double2* __restrict__ t_hi,
                        const double2* __restrict__ t_lo, V2Count nc) {
  LKB_DYN_SMEM(double2, buf);
  const int64_t ntr = v2_count(nc, (int)gridDim.y);
  for (int64_t lc = blockIdx.y; lc < ntr; lc += gridDim.y) {
    __syncthreads();
    v2_cols_load<PA>(buf, G, n1max, lc, (int)blockIdx.x, V2Cta());
    __syncthreads();
    v2_cols_one<PA>(buf, T, n1max, tw_a, t_hi, t_lo, lc, (int)blockIdx.x, V2Cta());
  }
}

// ---- persistent ring of tiles (fp32 rows) ----------------------------------------------------------------
// One CTA of 2 x V2_THREADS threads per SM: two compute groups and three tile buffers in shared memory.  CTA b takes
// tiles b, b + gridDim.x, ... (local index j = 0, 1, ...); tile j lands in buffer j % 3 and group j % 2 computes it.
// The group that has finished tile j - past the group barrier after its last read of buffer j % 3 - fetches tile
// j + 3, the other group's next tile, into that buffer, and goes on to its own tile j + 2, which the other group
// fetched one step earlier: a tile's global loads overlap the other group's passes.  A fetch is one cp.async per
// point; its 512 issuing threads arrive (.noinc) on mbarrier j % 6 once their copies have landed, and the computing
// group waits there.  One mbarrier per (buffer, computing group) and not per buffer: each group then waits on
// consecutive phases of its own barriers.  (A group sees only every other phase of buffer j % 3, so a parity wait for
// tile j + 3 made before tile j had landed would pass on the phase before it.)  Epilogue stores stay plain stores.
// smem: 3 tiles of `elems` points, then the 6 mbarriers.
template <class Load, class Body>
__device__ __forceinline__ void v2_ring(float2* smem, const int elems, const int ntiles, Load load, Body body) {
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 3 * elems);
  const V2Half gp{};
  if (threadIdx.x < 6) ptx::mbar_init(bar + threadIdx.x, V2_THREADS);
  __syncthreads();
  const int b = (int)blockIdx.x, nb = (int)gridDim.x;
  auto fetch = [&](int j) {
    if (b + j * nb < ntiles) {
      load(smem + (j % 3) * elems, b + j * nb, gp);
      ptx::cp_async_mbar_arrive_noinc(bar + j % 6);
    }
  };
  for (int j = V2Half::group(); j < 3; j += 2) fetch(j);          // group 0: tiles 0 and 2, group 1: tile 1
  for (int j = V2Half::group(); b + j * nb < ntiles; j += 2) {
    ptx::mbar_wait(bar + j % 6, (uint32_t)(j / 6) & 1u);
    body(smem + (j % 3) * elems, b + j * nb, gp);
    gp.sync();
    fetch(j + 3);
  }
  ptx::cp_async_wait_all();                                        // no copy of this thread outlives it
}
// ---- rows + finish -----------------------------------------------------------------------------------------------
// Folded per-frequency table (built once per call, y-independent): with G d = (C + i S) of a light curve at bin j,
//   yc + i ys = E d1 + O d2 - ysum c2,   power = yc^2 wz + ys^2 ww
//   d1 = dec conj(tau),  d2 = exp(2 pi i kk / M) d1,  c2 = (Ctau, Stau),  (wz, ww) = 1 / (2 N CC'), 1 / (2 N SS')
struct V2FTab {
  float4 d;       // d1.x, d1.y, d2.x, d2.y
  float4 c;       // c2.x, c2.y, wz, ww
};
struct V2Finish {
  const V2FTab* ftab;      // [F]
  int64_t k0, F, k_lo;
  const float* ysum;       // [B]
  float Nf;
  int normalization;
  float scale;
  float* power;            // [B, F]
  unsigned* peak;          // [B] or NULL: running maximum of the psd-scaled power of a light curve (float bits)
  const int* lcmap;        // NULL: blockIdx.y is the light curve; else the light curve of transform blockIdx.y
  int log2M;               // (double-precision finish: exp(2 pi i kk / M) is evaluated, not tabulated)
};

__device__ __forceinline__ float v2_normalise(float pw, float Nf, int normalization, float scale) {
  if (normalization == LKB_LS_NORM_PSD_SCALE) return pw * scale;
  if (normalization == LKB_LS_NORM_AMPLITUDE) return sqrtf(pw * (4.0f / Nf));
  return pw;
}
// psd-scaled power (before the normalisation) of one bin from the modes k (g1) and Mh - k (g2) of the packed transform
__device__ __forceinline__ float v2_finish_pw(float2 g1, float2 g2, const V2FTab tb, float ysum, int64_t, int) {
  const float ex = 0.5f * (g1.x + g2.x), ey = 0.5f * (g1.y - g2.y);        // E = (g1 + conj g2) / 2
  const float ox = 0.5f * (g1.y + g2.y), oy = 0.5f * (g2.x - g1.x);        // O = (g1 - conj g2) / 2i
  const float yc = ex * tb.d.x - ey * tb.d.y + ox * tb.d.z - oy * tb.d.w - ysum * tb.c.x;
  const float ys = ex * tb.d.y + ey * tb.d.x + ox * tb.d.w + oy * tb.d.z - ysum * tb.c.y;
  return yc * yc * tb.c.z + ys * ys * tb.c.w;
}
// the same in double precision: G = E + exp(2 pi i kk / M) O first (E and O can be orders of magnitude above G - the
// mirror image of a strong line), then the fp32 table's d1 and window terms
__device__ __forceinline__ float v2_finish_pw(double2 g1, double2 g2, const V2FTab tb, float ysum, int64_t kk, int log2M) {
  const double ex = 0.5 * (g1.x + g2.x), ey = 0.5 * (g1.y - g2.y);
  const double ox = 0.5 * (g1.y + g2.y), oy = 0.5 * (g2.x - g1.x);
  double sw, cw;
  sincospi(ldexp((double)kk, 1 - log2M), &sw, &cw);
  const double gx = ex + cw * ox - sw * oy, gy = ey + cw * oy + sw * ox;
  const double yc = gx * (double)tb.d.x - gy * (double)tb.d.y - (double)ysum * (double)tb.c.x;
  const double ys = gx * (double)tb.d.y + gy * (double)tb.d.x - (double)ysum * (double)tb.c.y;
  return (float)(yc * yc * (double)tb.c.z + ys * ys * (double)tb.c.w);
}

// row k1 of slot s (0 .. 15) of row group g: rows 1 + 8 g + r (s = r < 8), then their mirrors A - k1
template <int PA>
__device__ __forceinline__ int v2_slot_k1(int s, int g) {
  constexpr int A = 1 << PA, R = V2_R;
  const int h = s >> 3, r = s & (R - 1);
  if (h == 0) return 1 + g * R + r;
  if (g == (A / (2 * R)) - 1 && r == 0) return 0;    // instead of a second copy of row A / 2
  return A - (g + 1) * R + r;
}
// tile (lc, g) of T -> buf: the 16 rows of row group g of light curve slot lc, one skewed line of Bc points each
template <int PA, class CT, class Grp>
__device__ __forceinline__ void v2_rows_load(CT* buf, const CT* __restrict__ T, const int64_t lc, const int g,
                                             const Grp gp) {
  constexpr int PTC = V2_LOG_TILE - PA, TC = 1 << PTC, R = V2_R, LS = V2_LSB;
  const int t = gp.tid();
  const CT* Tp = T + (lc << (PA + V2_PB));
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int e = t + V2_THREADS * u;
    const int j = e & (TC - 1), r = (e >> PTC) & (R - 1), h = (e >> (PTC + 3)) & 1, c = e >> (PTC + 4);
    const int s = h * R + r;
    gp.put(buf + s * LS + v2_skew((c << PTC) + j), Tp + ((((c << PA) + v2_slot_k1<PA>(s, g)) << PTC) + j), true);
  }
}
// MODE 1: finish -> power.  MODE 2: the modes k < nk2_keep * A and their mirrors Mh - k go to Zout [B][Mh] in natural
// order (the ragged finish kernel reads them there).  The loaded tile (lc, g) (lc_base + lc indexes fa.lcmap).
template <int PA, int MODE, class CT, class Grp>
__device__ __forceinline__ void v2_rows_one(CT* buf, const CT* __restrict__ tw_b, const V2Finish& fa,
                                            CT* __restrict__ Zout, int nk2_keep, const int64_t lc, const int lc_base,
                                            const int g, const Grp gp) {
  constexpr int A = 1 << PA, R = V2_R, LS = V2_LSB, Bc = V2_BC;
  const int t = gp.tid();
  const bool last = g == (A / (2 * R)) - 1;
  const int64_t Mh = (int64_t)1 << (PA + V2_PB);
  v2_pass_t<V2_PB, LS, 0, 1, CT>(buf, tw_b, gp);
  // one slot per thread for all its items: s = t % 16, k2 = t / 16 + 32 u
  const int s = t & (2 * R - 1), h = s >> 3, r = s & (R - 1), k1 = v2_slot_k1<PA>(s, g);
  if (MODE == 2) {
    const int keep = nk2_keep < Bc / 2 ? nk2_keep : Bc / 2;
    for (int q = t >> 4; q < 2 * keep; q += V2_THREADS / 16) {
      const int k2 = q < keep ? q : Bc - 2 * keep + q;          // [0, keep) and [Bc - keep, Bc)
      Zout[lc * Mh + k1 + ((int64_t)k2 << PA)] = buf[s * LS + v2_skew(k2)];
    }
  } else {
  int ps = (1 - h) * R + (R - 1 - r);                              // mode Mh - k: row A - k1, column Bc - 1 - k2
  bool row0 = false;
  if (last && h == 0 && r == R - 1) ps = s;                        // row A / 2 mirrors onto itself
  if (last && h == 1 && r == 0) { ps = s; row0 = true; }           // row 0: column (Bc - k2) mod Bc
  int64_t nK2 = ((fa.k0 + fa.F - 1) >> PA) + 1;
  if (nK2 > Bc) nK2 = Bc;
  const int64_t lcd = fa.lcmap ? (int64_t)fa.lcmap[lc_base + lc] : lc;   // the light curve whose flux this transform holds
  const float ys0 = fa.ysum[lcd];
  float* prow = fa.power + lcd * fa.F;
  const int64_t jbase = (int64_t)k1 - fa.k0;
  float pmax = 0.0f;
  // items of a thread: k2 = t / 16 + 32 u, table loads in batches of UB (4 made ptxas spill 124 bytes in the persistent
  // kernel at its 64-register cap; the ring's other group hides the rest of the latency)
  constexpr int KSTEP = V2_THREADS / 16, UB = 2;
  for (int k2b = t >> 4; k2b < (int)nK2; k2b += KSTEP * UB) {
    V2FTab tb[UB];
    int64_t jj[UB];
    bool valid[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) {                                 // all table loads of the batch in flight together
      const int k2 = k2b + KSTEP * u;
      jj[u] = jbase + ((int64_t)k2 << PA);
      valid[u] = k2 < (int)nK2 && jj[u] >= fa.k_lo && jj[u] < fa.F;
      if (valid[u]) tb[u] = fa.ftab[jj[u]];
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      if (!valid[u]) continue;
      const int k2 = k2b + KSTEP * u;
      const int pi = row0 ? ((Bc - k2) & (Bc - 1)) : (Bc - 1 - k2);
      const CT g1 = buf[s * LS + v2_skew(k2)], g2 = buf[ps * LS + v2_skew(pi)];
      const float pw = v2_finish_pw(g1, g2, tb[u], ys0, fa.k0 + jj[u], fa.log2M);
      pmax = fmaxf(pmax, pw);
      prow[jj[u]] = v2_normalise(pw, fa.Nf, fa.normalization, fa.scale);
    }
  }
  if (fa.peak) {                                                   // (power >= 0: float bits order as unsigned)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
    if ((t & 31) == 0 && pmax > 0.0f) atomicMax(fa.peak + lcd, __float_as_uint(pmax));
  }
  }
}

// escalation pass (double precision, finish mode): grid (A / 16, gy); blocks stride over a device-side count of
// transforms; transform slot lc holds light curve fa.lcmap[nc.base + lc]
template <int PA>
__global__ void __launch_bounds__(V2_THREADS, 1)
nufft2_rows_list_kernel(const double2* __restrict__ T, const double2* __restrict__ tw_b, V2Finish fa, V2Count nc) {
  LKB_DYN_SMEM(double2, buf);
  const int64_t ntr = v2_count(nc, (int)gridDim.y);
  for (int64_t lc = blockIdx.y; lc < ntr; lc += gridDim.y) {
    __syncthreads();
    v2_rows_load<PA>(buf, T, lc, (int)blockIdx.x, V2Cta());
    __syncthreads();
    v2_rows_one<PA, 1>(buf, tw_b, fa, (double2*)nullptr, 0, lc, nc.base, (int)blockIdx.x, V2Cta());
  }
}
// grid (min(SMs, B A / 16)), 1024 threads: tile = lc (A / 16) + g (row group fastest).  (Tried in the one-tile-per-CTA
// form: the light curve as the fast index, so that the CTAs in flight share one 100 KB slice of the finish table -
// 1.84 ms instead of 1.76 ms: the tile reads of 296 different light curves scatter over DRAM pages, which costs more
// than the table locality gains.)
template <int PA, int MODE>
__global__ void __launch_bounds__(2 * V2_THREADS, 1)
nufft2_rows_ring_kernel(const float2* __restrict__ T, const float2* __restrict__ tw_b, V2Finish fa,
                        float2* __restrict__ Zout, int nk2_keep, int B) {
  constexpr int NG = (1 << PA) / (2 * V2_R);
  LKB_DYN_SMEM(float2, smem);
  v2_ring(smem, 2 * V2_R * V2_LSB, B * NG,
          [&](float2* buf, int tile, const V2Half gp) { v2_rows_load<PA>(buf, T, tile / NG, tile % NG, gp); },
          [&](float2* buf, int tile, const V2Half gp) {
            v2_rows_one<PA, MODE>(buf, tw_b, fa, Zout, nk2_keep, tile / NG, 0, tile % NG, gp);
          });
}

// ---- precision escalation -------------------------------------------------------------------------------------
// The fp32 transform's rounding noise is proportional to the LARGEST component of a light curve, wherever it lies - for
// instance a strong line above the frequency grid's upper end - while the parity tolerance is relative to the highest
// peak INSIDE the grid.  Measured on config C2 (tools/worst_bins.py): worst bin at 1.09x the tolerance, on light
// curves whose flux excursion is > 1000x their in-band peak amplitude; a generic fp32 NUFFT (pocketfft single precision)
// shows the same noise floor.  So the finish records every light curve's in-band peak, light curves with
//     max |y - mean| > ratio * (in-band peak amplitude)
// are listed, and the listed ones are transformed again in double precision (same kernels, double2 instantiation).
__global__ void nufft2_flag_kernel(const unsigned* __restrict__ peak, const float* __restrict__ absmax, int B, float Nf,
                                   float ratio, int* __restrict__ count, int* __restrict__ list, int* __restrict__ total) {
  const int b = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  bool f = false;
  if (b < B) {
    const float amp = sqrtf(__uint_as_float(peak[b]) * (4.0f / Nf));
    f = absmax[b] > ratio * amp;
  }
  const unsigned bal = __ballot_sync(0xffffffffu, f);
  if (bal) {
    int base = 0;
    if ((threadIdx.x & 31) == 0) {
      base = atomicAdd(count, __popc(bal));
      if (total) atomicAdd(total, __popc(bal));
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (f) list[base + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u))] = b;
  }
}

// double-precision fine grids of the listed light curves: G[i][e] for light curve list[i0 + i]; grid (cells / 256, n)
__global__ void __launch_bounds__(256)
nufft2_spread_list_kernel(const int32_t* __restrict__ first_ge, const nufft::Cad* __restrict__ cad,
                          const double* __restrict__ Wt, const float* __restrict__ y, int64_t ystride,
                          const int* __restrict__ list, int w, int p, int ptc, int n1max, double2* __restrict__ G,
                          V2Count nc) {
  const int64_t cells = (int64_t)n1max << V2_PB;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= cells) return;
  const int64_t M = (int64_t)1 << p, m = 2 * v2_zcell_of(e, ptc, n1max);
  const int ntr = v2_count(nc, (int)gridDim.y);
  for (int i = (int)blockIdx.y; i < ntr; i += (int)gridDim.y) {
  const float* yr = y + (int64_t)list[nc.base + i] * ystride;
  double a0 = 0.0, a1 = 0.0;
  const int64_t L = nufft::table_len(M, w);
  for (int wrap = 0; wrap < 2; ++wrap) {
    const int64_t mm = m + (int64_t)wrap * M;
    if (mm + 1 >= L) break;
    int64_t lo_c = mm - w + 1, hi_c = mm + 2;
    if (lo_c < 0) lo_c = 0;
    if (hi_c > L - 1) hi_c = L - 1;
    const int32_t na = first_ge[lo_c], nb = first_ge[hi_c];
    for (int32_t n = na; n < nb; ++n) {
      const int tap = (int)(mm - (int64_t)cad[n].i0);
      const double* wr = Wt + (int64_t)n * w;
      const double w0 = (tap >= 0) ? wr[tap] : 0.0, w1 = (tap + 1 < w) ? wr[tap + 1] : 0.0;
      const double v = (double)yr[n];
      a0 = fma(w0, v, a0);
      a1 = fma(w1, v, a1);
    }
  }
  G[(int64_t)i * cells + e] = make_double2(a0, a1);
  }
}

// ---- launch helpers ------------------------------------------------------------------------------------------------
inline unsigned v2_blocks_for(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

template <class CT>
struct V2TablesT {
  const CT *tw_a, *tw_b, *t_hi, *t_lo;
};
typedef V2TablesT<float2> V2Tables;
typedef V2TablesT<double2> V2TablesD;
// twiddle tables of the transform of 2^p real cells in workspace slot `slot`
template <class CT>
inline int v2_tables(int p, int slot, cudaStream_t st, V2TablesT<CT>* out) {
  const int ph = p - 1, pa = ph - V2_PB, pl = nufft::v2_log2_lo(ph);
  const int la = nufft::v2_pass_table_len(pa), lb = nufft::v2_pass_table_len(V2_PB), nhi = 1 << (ph - pl), nlo = 1 << pl;
  CT* base = nullptr;
  LKB_TRY(ws_get_t<CT>(slot, (size_t)(la + lb + nhi + nlo + 4), &base));
  CT *tw_a = base, *tw_b = base + la, *t_hi = tw_b + lb, *t_lo = t_hi + nhi;
  LKB_LAUNCH(v2_blocks_for(la + lb + nhi + nlo, 256), 256, st, nufft2_tables_kernel<CT>)(pa, V2_PB, ph, tw_a, tw_b, t_hi, t_lo);
  LKB_LAUNCH_CHECK();
  out->tw_a = tw_a; out->tw_b = tw_b; out->t_hi = t_hi; out->t_lo = t_lo;
  return LKB_OK;
}
// rows n1 of the [A][Bc] grid of z cells that cadences can reach when the last one's support starts at cell i0_last
inline int v2_n1max(int p, int64_t i0_last, int w) {
  const int64_t M = (int64_t)1 << p, A = (M / 2) >> V2_PB;
  const int64_t reach = i0_last + w + 1;                   // fine-grid cells [0, reach) (a support past M wraps to 0)
  if (reach >= M) return (int)A;
  const int64_t n = ((reach + 1) / 2 + V2_BC - 1) >> V2_PB;
  return (int)(n < 1 ? 1 : (n > A ? A : n));
}
inline bool v2_supported(int p) { return p >= V2R_P_MIN && p <= V2R_P_MAX; }

// shared memory of a ring CTA: three tiles of `elems` points and the six mbarriers
inline size_t v2_ring_smem(int elems) { return 3 * (size_t)elems * sizeof(float2) + 6 * sizeof(uint64_t); }
// CTAs of a ring launch: one per SM (2 on the CPU emulator), at most one per tile; LKB_NUFFT_RING_CTAS overrides the
// per-SM count (tests: a forced split of the tiles over CTAs and groups)
inline unsigned v2_ring_ctas(int64_t ntiles) {
#if defined(LKB_CUDA_EMU)
  int64_t n = 2;
#else
  int64_t n = sm_count();
#endif
  if (const char* e = getenv("LKB_NUFFT_RING_CTAS")) n = std::max(1, atoi(e));
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(n, ntiles));
}

template <int PA, class CT>
int v2_cols_pa(const CT* G, CT* T, int n1max, int B, const V2TablesT<CT>& tb, cudaStream_t st, V2Count nc) {
  using Q = V2Cols<PA>;
  const size_t smem = (size_t)Q::ELEMS * sizeof(CT);
  const dim3 grid((unsigned)Q::C, (unsigned)B);
  if constexpr (sizeof(CT) == 16) {                  // the escalation pass
    LKB_CUDA_CHECK(cudaFuncSetAttribute(nufft2_cols_list_kernel<PA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LKB_LAUNCH_SMEM(grid, V2_THREADS, smem, st, nufft2_cols_list_kernel<PA>)(G, T, n1max, tb.tw_a, tb.t_hi, tb.t_lo, nc);
  } else {
    LKB_CUDA_CHECK(cudaFuncSetAttribute(nufft2_cols_kernel<PA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LKB_LAUNCH_SMEM(grid, V2_THREADS, smem, st, nufft2_cols_kernel<PA>)(G, T, n1max, tb.tw_a, tb.t_hi, tb.t_lo);
  }
  LKB_LAUNCH_CHECK();
  return LKB_OK;
}
template <int PA, class CT>
int v2_rows_pa(const CT* T, int B, const V2TablesT<CT>& tb, const V2Finish* fa, CT* Zout, int nk2_keep, cudaStream_t st,
               V2Count nc) {
  constexpr int NG = (1 << PA) / (2 * V2_R);
  if constexpr (sizeof(CT) == 16) {                  // the escalation pass: always the finish
    const size_t smem = (size_t)(2 * V2_R) * V2_LSB * sizeof(CT);
    LKB_CUDA_CHECK(cudaFuncSetAttribute(nufft2_rows_list_kernel<PA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LKB_LAUNCH_SMEM(dim3((unsigned)NG, (unsigned)B), V2_THREADS, smem, st, nufft2_rows_list_kernel<PA>)(T, tb.tw_b, *fa, nc);
  } else {
    const size_t smem = v2_ring_smem(2 * V2_R * V2_LSB);
    const unsigned grid = v2_ring_ctas((int64_t)B * NG);
    LKB_CUDA_CHECK(cudaFuncSetAttribute(nufft2_rows_ring_kernel<PA, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LKB_CUDA_CHECK(cudaFuncSetAttribute(nufft2_rows_ring_kernel<PA, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (fa) LKB_LAUNCH_SMEM(grid, 2 * V2_THREADS, smem, st, nufft2_rows_ring_kernel<PA, 1>)(T, tb.tw_b, *fa, nullptr, 0, B);
    else LKB_LAUNCH_SMEM(grid, 2 * V2_THREADS, smem, st, nufft2_rows_ring_kernel<PA, 2>)(T, tb.tw_b, V2Finish(), Zout, nk2_keep, B);
  }
  LKB_LAUNCH_CHECK();
  return LKB_OK;
}
#define V2_DISPATCH_PA(pa, CALL)                                                                       \
  switch (pa) {                                                                                         \
    case 4: return CALL(4); case 5: return CALL(5); case 6: return CALL(6); case 7: return CALL(7);      \
    case 8: return CALL(8); case 9: return CALL(9); case 10: return CALL(10); case 11: return CALL(11);  \
    case 12: return CALL(12); case 13: return CALL(13);                                                  \
    default: set_error("NUFFT v2: fine grid of 2^%d cells out of range", (pa) + V2_PB + 1); return LKB_E_UNSUPPORTED; \
  }
// G -> T for B transforms of 2^p real cells
template <class CT>
inline int v2_cols(const CT* G, CT* T, int p, int n1max, int B, const V2TablesT<CT>& tb, cudaStream_t st,
                   V2Count nc = V2Count{nullptr, 0, 0}) {
#define V2_CALL(PA) v2_cols_pa<PA, CT>(G, T, n1max, B, tb, st, nc)
  V2_DISPATCH_PA(p - 1 - V2_PB, V2_CALL)
#undef V2_CALL
}
// T -> power (fa != NULL) or -> Zout in natural order, modes k < nk2_keep * A and their mirrors
template <class CT>
inline int v2_rows(const CT* T, int p, int B, const V2TablesT<CT>& tb, const V2Finish* fa, CT* Zout, int nk2_keep,
                   cudaStream_t st, V2Count nc = V2Count{nullptr, 0, 0}) {
#define V2_CALL(PA) v2_rows_pa<PA, CT>(T, B, tb, fa, Zout, nk2_keep, st, nc)
  V2_DISPATCH_PA(p - 1 - V2_PB, V2_CALL)
#undef V2_CALL
}

}  // namespace
}  // namespace lkb
