// K3: Box Least Squares, the search lightkurve obtains from astropy at
//   /root/reference/src/lightkurve/periodogram.py:1161-1169
//   (BoxLeastSquares(t, y, dy).power(period, duration, objective, method="fast", oversample)).
// Algorithm = astropy bls.c (restated in oracle/bls_c.c): per trial period, fold the samples
// into bins of width min(duration)/oversample, wrap-pad, inclusive prefix sum, then scan every
// (duration, start bin) box and keep the FIRST strict maximum of the objective with y_out >= y_in.
//
// B200 mapping: one WARP per (light curve, period).  A CTA = BLS_WARPS warps working on
// consecutive periods of the SAME light curve, so the (t, w*y, w) sample tiles are staged into
// shared memory once per CTA and re-used by every warp.  Each warp owns a private
// shared-memory histogram (plain `+=`, no atomics): 32 consecutive samples have non-decreasing
// bin indices except at a period wrap, so a warp-segmented reduction leaves exactly one
// writer per bin (wrap blocks are split into monotone pieces).
//
// Densely sampled light curves (more cadences than bin boundaries over the baseline, e.g. TESS 2-min
// data with 7-min bins) take the BOUNDARY path instead: the exact (cycle, bin) index is monotone in
// time, so each bin of each cycle is a contiguous run of cadences; a lane finds the first cadence of
// its run with a table lookup + a short exact walk and adds the run's sum as a difference of a
// per-light-curve prefix sum - work per period ~ baseline / bin_duration instead of N, no scan.
//
// Bit-exactness: the bin index (int)(fabs(fmod(t - min_t, P)) / bin_duration) + 1 is evaluated
// with an exact fmod (fma remainder + fix-up) and an IEEE fp64 division, so it equals the C
// result bit for bit.  This file is compiled with -fmad=false so that no a*b+c is contracted
// where the C code (built with -ffp-contract=off) has two roundings.  The binned sums are
// accumulated in a different order than the sequential C loop => equal to ~1e-13 relative,
// not bitwise; exact ties between boxes that cover the same samples are preserved by the
// scan construction (see bls_cumsum).
#include "bls_common.cuh"
#include <float.h>
#include <algorithm>
#include <vector>

namespace lkb {

constexpr int BLS_WARPS = 8;
constexpr int BLS_TILE = 1024;

// (int)(r / bd) with the IEEE division replaced, on the fast path, by a reciprocal multiply whose
// result is PROVEN equal: k = trunc(r * (1/bd)); rem = fma(-k, bd, r) is the (once rounded) remainder;
// if 0 <= rem < bd_safe = bd * (1 - (kmax + 2) 2^-51) with kmax >= k, the real quotient lies in
// [k, k + 1 - margin) and RN(r / bd) cannot reach k + 1, so trunc(RN(r/bd)) = k.  Anything else (a
// sample within ~1e-13 of a bin edge) takes the true division - a warp-uniform, out-of-line branch so
// that the ~25-instruction IEEE division is not if-converted into every iteration.
__device__ __noinline__ double bls_div_slow(double r, double bd) { return r / bd; }

__device__ __forceinline__ double bls_safe_width(double bd, int kmax) {
  return bd - bd * (((double)kmax + 2.0) * 4.440892098500626e-16);
}

// bin index of a sample at x >= 0 (time since the first cadence); `valid` lanes only.  Warp-collective.
__device__ __forceinline__ int bls_bin_warp(double x, bool valid, double period, double inv_period, double bd,
                                            double inv_bd, double bd_safe) {
  double q = trunc(x * inv_period);
  double r = fma(-q, period, x);
  if (r < 0.0) { q -= 1.0; r = fma(-q, period, x); }
  else if (r >= period) { q += 1.0; r = fma(-q, period, x); }
  double k = trunc(r * inv_bd);
  const double rem = fma(-k, bd, r);
  const bool slow = valid && !(rem >= 0.0 && rem < bd_safe);
  if (__any_sync(0xffffffffu, slow)) {
    if (slow) k = trunc(bls_div_slow(r, bd));
  }
  return valid ? (int)k + 1 : -1;
}

// exact (cycle q, bin k) of a sample at x >= 0; callable from divergent code
__device__ __forceinline__ void bls_cycle_bin(double x, double period, double inv_period, double bd, double inv_bd,
                                              double bd_safe, int& qi, int& ki) {
  double q = trunc(x * inv_period);
  double r = fma(-q, period, x);
  if (r < 0.0) { q -= 1.0; r = fma(-q, period, x); }
  else if (r >= period) { q += 1.0; r = fma(-q, period, x); }
  double k = trunc(r * inv_bd);
  const double rem = fma(-k, bd, r);
  if (!(rem >= 0.0 && rem < bd_safe)) k = trunc(bls_div_slow(r, bd));
  qi = (int)q;
  ki = (int)k;
}

__device__ __forceinline__ int bls_bin(double t, double min_t, double period, double inv_period, double bin_duration,
                                       double inv_bin) {
  const double r = fabs(bls_fmod(t - min_t, period, inv_period));
  const double k = trunc(r * inv_bin);
  const double rem = fma(-k, bin_duration, r);
  const double margin = bin_duration * ((k + 2.0) * 4.440892098500626e-16);
  if (rem >= 0.0 && rem < bin_duration - margin && k < 1073741824.0) return (int)k + 1;
  return (int)(r / bin_duration) + 1;
}

__global__ void bls_bin_index_kernel(const double* __restrict__ t, int64_t N, double min_t, double period,
                                     double bin_duration, int32_t* __restrict__ ind) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) ind[i] = bls_bin(t[i], min_t, period, 1.0 / fabs(period), bin_duration, 1.0 / bin_duration);
}

// ---- per-warp pieces ------------------------------------------------------------------------
// Add the 32 samples held one per lane into the warp's histogram h[bin] = {sum w*y, sum w}.
// key < 0 => lane inactive.  Equal keys are contiguous (bins are monotone between period wraps), so each
// run's sum is a difference of the light curve's exclusive prefix sums: c_i = prefix before this lane's
// sample, c_next = prefix after it; the run's last lane adds  c_next - c_(run head)  - one writer per bin.
__device__ __forceinline__ void bls_warp_bin(int key, double2 c_i, double2 c_next, double2* h, int lane) {
  const unsigned full = 0xffffffffu;
  const int prev = __shfl_up_sync(full, key, 1);
  const bool head = (lane == 0) || (key != prev);
  const bool wrap = (lane != 0) && (key < prev) && (key >= 0);
  const unsigned headmask = __ballot_sync(full, head);
  const unsigned wrapmask = __ballot_sync(full, wrap);
  const unsigned le = (lane == 31) ? 0xffffffffu : ((2u << lane) - 1u);
  const int start = 31 - __clz(headmask & le);          // lane of this run's head
  const double hy = __shfl_sync(full, c_i.x, start), hi = __shfl_sync(full, c_i.y, start);
  const bool tail = (((headmask >> 1) | 0x80000000u) >> lane & 1u) && key >= 0;
  const double vy = c_next.x - hy, vi = c_next.y - hi;
  if (wrapmask == 0) {
    if (tail) { double2 c = h[key]; c.x += vy; c.y += vi; h[key] = c; }
  } else {
    // split into monotone pieces so that equal keys are contiguous within a piece
    const int piece = __popc(wrapmask & le);
    const int npieces = __popc(wrapmask) + 1;
    for (int q = 0; q < npieces; ++q) {
      if (tail && piece == q) { double2 c = h[key]; c.x += vy; c.y += vi; h[key] = c; }
      __syncwarp();
    }
  }
  __syncwarp();
}

// Inclusive prefix sum over h[0..n] (n+1 entries, both components), in place.  Each lane scans a
// contiguous chunk sequentially; chunk offsets are a SEQUENTIAL prefix (lane 0) so that an empty bin
// leaves the running sum bitwise unchanged also across chunk boundaries (tie preservation).
__device__ __forceinline__ void bls_cumsum(double2* h, int n_entries, double2* scratch, int lane) {
  const int L = (n_entries + 31) / 32;
  const int lo = min(lane * L, n_entries), hi = min(lo + L, n_entries);
  double rx = 0.0, ry = 0.0;
  for (int i = lo; i < hi; ++i) {
    double2 c = h[i];
    rx += c.x; ry += c.y;
    h[i] = make_double2(rx, ry);
  }
  scratch[lane] = make_double2(rx, ry);
  __syncwarp();
  if (lane == 0) {
    double ox = 0.0, oy = 0.0;
    for (int l = 0; l < 32; ++l) {
      const double2 tot = scratch[l];
      scratch[l] = make_double2(ox, oy);
      ox += tot.x; oy += tot.y;
    }
  }
  __syncwarp();
  const double2 off = scratch[lane];
  if (lane > 0)
    for (int i = lo; i < hi; ++i) {
      double2 c = h[i];
      h[i] = make_double2(off.x + c.x, off.y + c.y);
    }
  __syncwarp();
}

// Everything after the histogram is filled: wrap-pad, prefix sums, box scan, first-max, outputs.
__device__ __forceinline__ void bls_finish_warp(double2* h, int n_bins, int oversample, double2* scr, int lane,
                                                const BlsLcInfo& li, const int* __restrict__ dur_bins, int D,
                                                double bin_duration, int objective, double per, double inv_per,
                                                int64_t oi, double* __restrict__ o_power,
                                                double* __restrict__ o_depth, double* __restrict__ o_depth_err,
                                                double* __restrict__ o_duration, double* __restrict__ o_ttime,
                                                double* __restrict__ o_snr, double* __restrict__ o_ll,
                                                int32_t* __restrict__ o_bins) {
  // wrap-pad: mean[n_bins - oversample + (n-1)] = mean[n], n = 1..oversample (no overlap, see DESIGN.md)
  for (int i = lane + 1; i <= oversample; i += 32) h[n_bins - oversample + (i - 1)] = h[i];
  __syncwarp();
  bls_cumsum(h, n_bins + 1, scr, lane);

  // search: only the objective is evaluated per box; the statistics of the winner are recomputed below
  double best_obj = -INFINITY;
  int best_k = 0x7fffffff, best_n = 0x7fffffff;
  for (int k = 0; k < D; ++k) {
    const int dur = dur_bins[k];
    const int n_max = n_bins - dur;
    for (int nn = lane; nn <= n_max; nn += 32) {
      const double2 hb = h[nn + dur], ha = h[nn];
      double y_in = hb.x - ha.x;
      const double ivar_in = hb.y - ha.y;
      double y_out = li.sum_y - y_in;
      const double ivar_out = li.sum_ivar - ivar_in;
      if ((ivar_in < DBL_EPSILON) || (ivar_out < DBL_EPSILON)) continue;
      y_in /= ivar_in;
      y_out /= ivar_out;
      if (!(y_out >= y_in)) continue;
      double obj;
      if (objective) obj = (y_out - y_in) / sqrt(1.0 / ivar_in + 1.0 / ivar_out);
      else obj = 0.5 * ivar_in * (y_out - y_in) * (y_out - y_in);
      if (obj > best_obj) { best_obj = obj; best_k = k; best_n = nn; }
    }
  }
  // first maximum in (duration-major, start-bin-minor) order across lanes
  double wobj = best_obj;
  int wk = best_k, wn = best_n;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    const double oo = __shfl_xor_sync(0xffffffffu, wobj, s);
    const int ok = __shfl_xor_sync(0xffffffffu, wk, s);
    const int on = __shfl_xor_sync(0xffffffffu, wn, s);
    const bool take = (oo > wobj) || (oo == wobj && (ok < wk || (ok == wk && on < wn)));
    if (take) { wobj = oo; wk = ok; wn = on; }
  }
  if (lane == 0) {
    double depth = 0.0, depth_err = 0.0, snr = 0.0, ll = 0.0, bd = 0.0, ph = 0.0;
    int dur = -1;
    if (wk != 0x7fffffff) {
      dur = dur_bins[wk];
      const double2 hb = h[wn + dur], ha = h[wn];
      double y_in = hb.x - ha.x;
      const double ivar_in = hb.y - ha.y;
      double y_out = li.sum_y - y_in;
      const double ivar_out = li.sum_ivar - ivar_in;
      y_in /= ivar_in;
      y_out /= ivar_out;
      depth = y_out - y_in;
      depth_err = sqrt(1.0 / ivar_in + 1.0 / ivar_out);
      snr = depth / depth_err;
      ll = 0.5 * ivar_in * (y_out - y_in) * (y_out - y_in);
      bd = dur * bin_duration;
      ph = bls_fmod(wn * bin_duration + 0.5 * bd + li.min_t, per, inv_per);
    }
    o_power[oi] = wobj;
    o_depth[oi] = depth;
    o_depth_err[oi] = depth_err;
    o_snr[oi] = snr;
    o_ll[oi] = ll;
    o_duration[oi] = bd;
    o_ttime[oi] = ph + li.t_ref;
    if (o_bins) {
      o_bins[2 * oi] = dur >= 0 ? wn : -1;
      o_bins[2 * oi + 1] = dur;
    }
  }
}

struct BlsFast {            // boundary-path inputs (null tab => cadence path only)
  const double2* cpre;      // [total + B] exclusive prefix sums
  const int32_t* tab;       // lookup tables
  const int64_t* tab_offsets;
  double delta, inv_delta;
  double min_density;       // use the boundary path when N >= min_density * (x_max / bin_duration)
};

// GHIST = false: per-warp histograms in shared memory; true: in an (L2-resident) global workspace.
template <bool GHIST>
__global__ void __launch_bounds__(BLS_WARPS * 32)
bls_search_kernel(const double* __restrict__ trel, const double* __restrict__ wy, const double* __restrict__ iv,
                  const int64_t* __restrict__ offsets, const BlsLcInfo* __restrict__ info,
                  const double* __restrict__ period, int64_t p_begin, int64_t p_end, int64_t P,
                  const int* __restrict__ dur_bins, int D, double bin_duration,
                  int oversample, int objective, int hist_stride, double2* __restrict__ g_hist, BlsFast fast, int b_base,
                  double* __restrict__ o_power, double* __restrict__ o_depth, double* __restrict__ o_depth_err,
                  double* __restrict__ o_duration, double* __restrict__ o_ttime, double* __restrict__ o_snr,
                  double* __restrict__ o_ll, int32_t* __restrict__ o_bins) {
  extern __shared__ __align__(16) unsigned char bls_smem[];
  double* s_t = reinterpret_cast<double*>(bls_smem);              // sample times of the tile
  double2* s_c = reinterpret_cast<double2*>(s_t + BLS_TILE);      // BLS_TILE + 1 exclusive prefix sums
  double2* s_scr = s_c + BLS_TILE + 1;                            // BLS_WARPS * 32
  double2* s_hist = s_scr + BLS_WARPS * 32;                       // BLS_WARPS * hist_stride (unless GHIST)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = b_base + blockIdx.y;            // the launch covers light curves [b_base, b_base + gridDim.y)
  const int64_t o = offsets[b], n = offsets[b + 1] - o;
  const int nwarps = blockDim.x >> 5;
  const int64_t p = p_begin + (int64_t)blockIdx.x * nwarps + warp;
  if (n <= 0) {      // empty light curve: every output NaN
    if (p < p_end && lane == 0) {
      const double qn = __longlong_as_double(0x7ff8000000000000ll);
      const int64_t oi = (int64_t)b * P + p;
      o_power[oi] = qn; o_depth[oi] = qn; o_depth_err[oi] = qn; o_duration[oi] = qn; o_ttime[oi] = qn;
      o_snr[oi] = qn; o_ll[oi] = qn;
      if (o_bins) { o_bins[2 * oi] = -1; o_bins[2 * oi + 1] = -1; }
    }
    return;
  }
  const bool active = p < p_end;
  const double per = active ? period[p] : 1.0;
  const double inv_per = 1.0 / per;
  const double inv_bin = 1.0 / bin_duration;
  const int K1 = (int)ceil(per / bin_duration);
  const int n_bins = K1 + oversample;
  const double bd_safe = bls_safe_width(bin_duration, n_bins);
  const BlsLcInfo li = info[b];      // min(t - t_ref) = 0: the samples below are times since the first cadence

  double2* h;
  if constexpr (GHIST) {
    const size_t slot = ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * nwarps + warp;
    h = g_hist + slot * (size_t)hist_stride;
  } else {
    h = s_hist + (size_t)warp * hist_stride;
  }
  if (active)
    for (int i = lane; i <= n_bins; i += 32) h[i] = make_double2(0.0, 0.0);

  // boundary path?  CTA-uniform: sorted times, >= 33 bin slots per cycle (so that the 32 runs a warp
  // adds per step hit 32 different bins) and dense enough sampling for it to be the cheaper one.
  bool use_fast = false;
  if (fast.tab != nullptr && li.sorted) {
    const bool mine = !active || (K1 + 1 >= 33 && per < 1.0e9 * bin_duration &&
                                  (double)n >= fast.min_density * (li.x_max * inv_bin));
    use_fast = __syncthreads_and(mine ? 1 : 0) != 0;
  }

  if (use_fast) {
    if (!active) return;
    __syncwarp();
    const double* x = trel + o;
    const double2* c = fast.cpre + o + b;
    const int32_t* tab = fast.tab + fast.tab_offsets[b];
    const int nT = (int)(fast.tab_offsets[b + 1] - fast.tab_offsets[b]);
    const int kc = K1 + 1;                       // bin slots per cycle: k = 0 .. K1 (the last one normally empty)
    int q_last, k_last;
    bls_cycle_bin(x[n - 1], per, inv_per, bin_duration, inv_bin, bd_safe, q_last, k_last);
    const long long m_end = (long long)q_last * kc + k_last + 1;     // first boundary after the last cadence
    int q = 0, k = lane;                         // boundary m = it * 32 + lane  <->  (q, k); kc >= 33 > lane
    int carry_e = 0;
    double2 carry_c = make_double2(0.0, 0.0);
    for (long long m0 = 0; m0 <= m_end; m0 += 32) {
      int e = (int)n;
      if (m0 + lane <= m_end) {
        // (slot K1 starts at or after the end of the cycle: cap at the cycle end so that the walk starts before it)
        const double xb = fma((double)q, per, fmin((double)k * bin_duration, per));
        int j = (int)(xb * fast.inv_delta) - 1;
        j = max(0, min(j, nT - 1));
        const int e0 = tab[j];                   // every cadence before e0 is more than delta/2 before the boundary
        // Common case: the run starts at the first cadence with x >= xb (plain comparisons on three
        // speculatively loaded candidates).  Only when a cadence sits within ~1e-13 of the boundary can the
        // rounded fmod/division of bls.c disagree with real arithmetic: then walk with the exact function.
        const int nm1 = (int)n - 1;
        const double x0 = x[min(e0, nm1)], x1 = x[min(e0 + 1, nm1)], x2 = x[min(e0 + 2, nm1)];
        double xlo = -1.0e300, xhi = 1.0e300;
        if (x0 >= xb) { e = e0; xhi = x0; }
        else if (x1 >= xb) { e = e0 + 1; xlo = x0; xhi = x1; }
        else if (x2 >= xb) { e = e0 + 2; xlo = x1; xhi = x2; }
        else {
          e = e0 + 3;
          xlo = x2;
          while (e < n) {
            const double xv = x[e];
            if (xv >= xb) { xhi = xv; break; }
            xlo = xv;
            ++e;
          }
        }
        if (e > n) e = (int)n;                   // (the clamped candidates repeat the last cadence)
        const double tol = 1.0e-13 * (xb + per);
        if ((e < n && xhi - xb <= tol) || xb - xlo <= tol) {
          e = e0;
          while (e < n) {
            int qi, ki;
            bls_cycle_bin(x[e], per, inv_per, bin_duration, inv_bin, bd_safe, qi, ki);
            if (qi > q || (qi == q && ki >= k)) break;
            ++e;
          }
        }
      }
      const double2 ce = c[e];
      int e_prev = __shfl_up_sync(0xffffffffu, e, 1);
      double2 c_prev;
      c_prev.x = __shfl_up_sync(0xffffffffu, ce.x, 1);
      c_prev.y = __shfl_up_sync(0xffffffffu, ce.y, 1);
      if (lane == 0) { e_prev = carry_e; c_prev = carry_c; }
      if (e > e_prev) {                          // the run that ends at this boundary: bin slot k - 1 (cyclic)
        const int key = (k == 0 ? kc - 1 : k - 1) + 1;
        double2 cur = h[key];
        cur.x += ce.x - c_prev.x;
        cur.y += ce.y - c_prev.y;
        h[key] = cur;
      }
      carry_e = __shfl_sync(0xffffffffu, e, 31);
      carry_c.x = __shfl_sync(0xffffffffu, ce.x, 31);
      carry_c.y = __shfl_sync(0xffffffffu, ce.y, 31);
      k += 32;
      if (k >= kc) { k -= kc; ++q; }
      __syncwarp();
    }
  } else {
    const double2* cg = fast.cpre + o + b;
    for (int64_t c0 = 0; c0 < n; c0 += BLS_TILE) {
      const int cnt = (int)min((int64_t)BLS_TILE, n - c0);
      __syncthreads();
      for (int i = threadIdx.x; i <= cnt; i += blockDim.x) {
        if (i < cnt) s_t[i] = trel[o + c0 + i];
        s_c[i] = cg[c0 + i];
      }
      __syncthreads();
      if (active) {
        for (int i0 = 0; i0 < cnt; i0 += 32) {
          const int i = i0 + lane;
          const bool valid = i < cnt;
          const int ic = valid ? i : cnt - 1;
          const int key = bls_bin_warp(s_t[ic], valid, per, inv_per, bin_duration, inv_bin, bd_safe);
          bls_warp_bin(key, s_c[ic], s_c[ic + 1], h, lane);
        }
      }
    }
    if (!active) return;
  }
  __syncwarp();
  bls_finish_warp(h, n_bins, oversample, s_scr + warp * 32, lane, li, dur_bins, D, bin_duration, objective, per,
                  inv_per, (int64_t)b * P + p, o_power, o_depth, o_depth_err, o_duration, o_ttime, o_snr, o_ll, o_bins);
}

// ---- host ------------------------------------------------------------------------------------
int bls_bin_index(const double* t_rel, int64_t N, double min_t, double period, double bin_duration, int32_t* ind,
                  int mem, cudaStream_t st) {
  LKB_REQUIRE(t_rel && ind && N > 0, "lkb_bls_bin_index: null/empty argument");
  LKB_REQUIRE(period > 0 && bin_duration > 0, "lkb_bls_bin_index: period and bin_duration must be positive");
  LKB_TRY(ensure_device());
  const double* d_t = nullptr;
  int32_t* d_i = nullptr;
  LKB_TRY(stage_in<double>(mem, WS_IN0, t_rel, N, &d_t, st));
  LKB_TRY(stage_out_alloc<int32_t>(mem, WS_OUT0, ind, N, &d_i));
  bls_bin_index_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d_t, N, min_t, period, bin_duration, d_i);
  LKB_LAUNCH_CHECK();
  LKB_TRY(stage_out_copy<int32_t>(mem, ind, d_i, N, st));
  if (mem == LKB_MEM_HOST) LKB_CUDA_CHECK(cudaStreamSynchronize(st));
  return LKB_OK;
}

int bls_power(const double* t, const double* y, const double* dy, const int64_t* h_offsets, int B,
              const double* period, int64_t P, const double* duration, int D, int oversample, int objective,
              double* power, double* depth, double* depth_err, double* duration_out, double* transit_time,
              double* depth_snr, double* log_like, int32_t* best_bins, int mem, cudaStream_t st) {
  LKB_REQUIRE(t && y && h_offsets && period && duration, "lkb_bls_power: null input");
  LKB_REQUIRE(power && depth && depth_err && duration_out && transit_time && depth_snr && log_like,
              "lkb_bls_power: null output");
  LKB_REQUIRE(B > 0 && B <= 65535 && P > 0 && D > 0 && oversample > 0, "lkb_bls_power: bad sizes");
  LKB_REQUIRE(objective == 0 || objective == 1, "lkb_bls_power: bad objective");
  LKB_TRY(ensure_device());
  const int64_t total = h_offsets[B];

  // the period / duration grids are needed on the host for validation and launch shaping
  std::vector<double> h_per(P), h_dur(D);
  if (mem == LKB_MEM_HOST) {
    memcpy(h_per.data(), period, sizeof(double) * P);
    memcpy(h_dur.data(), duration, sizeof(double) * D);
  } else {
    LKB_CUDA_CHECK(cudaMemcpyAsync(h_per.data(), period, sizeof(double) * P, cudaMemcpyDeviceToHost, st));
    LKB_CUDA_CHECK(cudaMemcpyAsync(h_dur.data(), duration, sizeof(double) * D, cudaMemcpyDeviceToHost, st));
    LKB_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  double min_period = h_per[0], max_period = h_per[0], min_dur = h_dur[0], max_dur = h_dur[0];
  for (int64_t i = 0; i < P; ++i) {
    if (!(h_per[i] == h_per[i]) || isinf(h_per[i])) { set_error("lkb_bls_power: period contains nan/inf"); return LKB_E_ARG; }
    min_period = fmin(min_period, h_per[i]);
    max_period = fmax(max_period, h_per[i]);
  }
  for (int i = 0; i < D; ++i) {
    if (!(h_dur[i] == h_dur[i]) || isinf(h_dur[i])) { set_error("lkb_bls_power: duration contains nan/inf"); return LKB_E_ARG; }
    min_dur = fmin(min_dur, h_dur[i]);
    max_dur = fmax(max_dur, h_dur[i]);
  }
  if (min_period < DBL_EPSILON) { set_error("lkb_bls_power: periods must be positive"); return LKB_E_ARG; }
  if (max_dur >= min_period || min_dur < DBL_EPSILON) {
    set_error("The maximum transit duration must be shorter than the minimum period");
    return LKB_E_ARG;
  }
  const double bin_duration = min_dur / (double)oversample;
  std::vector<int> h_durbins(D);
  for (int i = 0; i < D; ++i) h_durbins[i] = (int)round(h_dur[i] / bin_duration);

  const double *d_t = nullptr, *d_y = nullptr, *d_dy = nullptr, *d_per = nullptr, *d_dur = nullptr;
  LKB_TRY(stage_in<double>(mem, WS_IN0, t, total, &d_t, st));
  LKB_TRY(stage_in<double>(mem, WS_IN1, y, total, &d_y, st));
  LKB_TRY(stage_in<double>(mem, WS_IN2, dy, total, &d_dy, st));
  LKB_TRY(stage_in<double>(mem, WS_IN3, period, P, &d_per, st));
  LKB_TRY(stage_in<double>(mem, WS_IN4, duration, D, &d_dur, st));
  int64_t* d_off = nullptr;
  int* d_durbins = nullptr;
  LKB_TRY(ws_get_t<int64_t>(WS_A, B + 1, &d_off));
  LKB_TRY(ws_get_t<int>(WS_B, D, &d_durbins));
  LKB_CUDA_CHECK(cudaMemcpyAsync(d_off, h_offsets, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, st));
  LKB_CUDA_CHECK(cudaMemcpyAsync(d_durbins, h_durbins.data(), sizeof(int) * D, cudaMemcpyHostToDevice, st));
  LKB_CUDA_CHECK(cudaStreamSynchronize(st));   // h_durbins is a local

  double *d_trel = nullptr, *d_wy = nullptr, *d_iv = nullptr;
  BlsLcInfo* d_info = nullptr;
  LKB_TRY(ws_get_t<double>(WS_C, total, &d_trel));
  LKB_TRY(ws_get_t<double>(WS_D, total, &d_wy));
  LKB_TRY(ws_get_t<double>(WS_E, total, &d_iv));
  LKB_TRY(ws_get_t<BlsLcInfo>(WS_F, B, &d_info));

  const size_t outn = (size_t)B * P;
  double *o0, *o1, *o2, *o3, *o4, *o5, *o6;
  int32_t* ob = nullptr;
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT0, power, outn, &o0));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT1, depth, outn, &o1));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT2, depth_err, outn, &o2));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT3, duration_out, outn, &o3));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT4, transit_time, outn, &o4));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT5, depth_snr, outn, &o5));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT6, log_like, outn, &o6));
  LKB_TRY(stage_out_alloc<int32_t>(mem, WS_OUT7, best_bins, 2 * outn, &ob));

  double2* d_cpre = nullptr;
  LKB_TRY(ws_get_t<double2>(WS_H, total + B, &d_cpre));
  bls_prep_kernel<<<B, 256, 0, st>>>(d_t, d_y, d_dy, d_off, d_trel, d_wy, d_iv, d_cpre, d_info);
  LKB_LAUNCH_CHECK();

  // boundary path set-up: per-light-curve lookup tables "first cadence at or after j * delta"
  BlsFast fast;
  fast.cpre = d_cpre;
  fast.tab = nullptr;
  fast.tab_offsets = nullptr;
  fast.delta = bin_duration / 8.0;
  fast.inv_delta = 1.0 / fast.delta;
  fast.min_density = 0.8;
  if (const char* e = getenv("LKB_BLS_MIN_DENSITY")) fast.min_density = atof(e);
  {
    std::vector<BlsLcInfo> h_info(B);
    LKB_CUDA_CHECK(cudaMemcpyAsync(h_info.data(), d_info, sizeof(BlsLcInfo) * B, cudaMemcpyDeviceToHost, st));
    LKB_CUDA_CHECK(cudaStreamSynchronize(st));
    std::vector<int64_t> h_to(B + 1, 0);
    bool ok = fast.min_density < 1e30;
    int64_t nT_max = 0;
    for (int b = 0; b < B && ok; ++b) {
      const int64_t nb = h_offsets[b + 1] - h_offsets[b];
      int64_t nT = 0;
      if (nb > 0) {
        const double cells = h_info[b].x_max * fast.inv_delta;
        if (!(cells >= 0.0) || cells > 6.0e7) { ok = false; break; }
        nT = (int64_t)cells + 3;
      }
      h_to[b + 1] = h_to[b] + nT;
      nT_max = nT > nT_max ? nT : nT_max;
    }
    if (ok && h_to[B] > 0 && h_to[B] <= ((int64_t)1 << 28)) {
      int64_t* d_to = nullptr;
      int32_t* d_tab = nullptr;
      LKB_TRY(ws_get_t<int64_t>(WS_I, B + 1, &d_to));
      LKB_TRY(ws_get_t<int32_t>(WS_J, h_to[B], &d_tab));
      LKB_CUDA_CHECK(cudaMemcpyAsync(d_to, h_to.data(), sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, st));
      LKB_CUDA_CHECK(cudaStreamSynchronize(st));   // h_to is a local
      const unsigned gxT = (unsigned)min((int64_t)64, (nT_max + 255) / 256);
      bls_table_kernel<<<dim3(gxT ? gxT : 1, (unsigned)B), 256, 0, st>>>(d_trel, d_off, d_to, fast.delta, d_tab);
      LKB_LAUNCH_CHECK();
      fast.tab = d_tab;
      fast.tab_offsets = d_to;
    }
  }

  // chunk the period list so that one launch's per-warp histograms have a common size
  const size_t fixed_smem = (size_t)(3 * BLS_TILE + 2 + 2 * BLS_WARPS * 32) * sizeof(double);
  const size_t smem_cap = 200 * 1024;
  static bool attr_set = false;
  if (!attr_set) {
    LKB_CUDA_CHECK(cudaFuncSetAttribute(bls_search_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    LKB_CUDA_CHECK(cudaFuncSetAttribute(bls_search_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  int64_t p0 = 0;
  prof_begin(st);
  while (p0 < P) {
    int nb_min = (int)ceil(h_per[p0] / bin_duration) + oversample, nb_max = nb_min;
    int64_t p1 = p0 + 1;
    while (p1 < P) {
      const int nb = (int)ceil(h_per[p1] / bin_duration) + oversample;
      const int lo = nb < nb_min ? nb : nb_min, hi = nb > nb_max ? nb : nb_max;
      if (hi > lo + lo / 4 + 64) break;
      nb_min = lo; nb_max = hi;
      ++p1;
    }
    const int stride = ((nb_max + 1 + 3) / 4) * 4;
    // warps (= periods) per CTA: as many as fit with their private histograms in shared memory
    int W = BLS_WARPS;
    while (W > 1 && fixed_smem + (size_t)W * 2 * stride * sizeof(double) > smem_cap) W >>= 1;
    size_t hist_bytes = (size_t)W * 2 * stride * sizeof(double);
    double2* g_hist = nullptr;
    size_t smem = fixed_smem + hist_bytes;
    // Occupancy beats locality here (measured: 108 -> 84 ms on the config-3 probe): once the shared-memory
    // histograms would leave fewer than 4 CTAs (32 warps) per SM, keep them in the L2-resident workspace.
    static const int ghist_bins = getenv("LKB_BLS_GHIST_BINS") ? atoi(getenv("LKB_BLS_GHIST_BINS")) : -1;
    if (ghist_bins >= 0 ? stride > ghist_bins : 4 * (smem + 1024) > 227 * 1024) smem = smem_cap + 1;
    if (smem > smem_cap) { W = BLS_WARPS; hist_bytes = (size_t)W * 2 * stride * sizeof(double); }
    const unsigned gx = (unsigned)((p1 - p0 + W - 1) / W);
    int b_group = B;
    if (smem > smem_cap) {
      // histograms do not fit in shared memory: keep them in (L2-resident) global workspace
      smem = fixed_smem;
      // one histogram slot per warp of the launch: bound the workspace by launching the light curves in groups
      const size_t per_lc = (size_t)gx * hist_bytes;
      const size_t cap = getenv("LKB_BLS_HIST_CAP_MB") ? (size_t)atoll(getenv("LKB_BLS_HIST_CAP_MB")) << 20 : (size_t)12 << 30;
      if (per_lc > cap) {
        set_error("lkb_bls_power: %d bins per period needs %zu bytes of histogram workspace per light curve", nb_max,
                  per_lc);
        return LKB_E_UNSUPPORTED;
      }
      b_group = (int)std::min<size_t>((size_t)B, std::max<size_t>(1, cap / per_lc));
      LKB_TRY(ws_get_t<double2>(WS_G, per_lc * b_group / sizeof(double2), &g_hist));
    }
    for (int bb = 0; bb < B; bb += b_group) {
      dim3 grid(gx, (unsigned)std::min(b_group, B - bb));
      if (g_hist)
        bls_search_kernel<true><<<grid, W * 32, smem, st>>>(d_trel, d_wy, d_iv, d_off, d_info, d_per, p0, p1, P,
                                                            d_durbins, D, bin_duration, oversample, objective, stride,
                                                            g_hist, fast, bb, o0, o1, o2, o3, o4, o5, o6, ob);
      else
        bls_search_kernel<false><<<grid, W * 32, smem, st>>>(d_trel, d_wy, d_iv, d_off, d_info, d_per, p0, p1, P,
                                                             d_durbins, D, bin_duration, oversample, objective, stride,
                                                             nullptr, fast, bb, o0, o1, o2, o3, o4, o5, o6, ob);
    }
    LKB_LAUNCH_CHECK();
    p0 = p1;
  }
  prof_end(st);

  LKB_TRY(stage_out_copy<double>(mem, power, o0, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, depth, o1, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, depth_err, o2, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, duration_out, o3, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, transit_time, o4, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, depth_snr, o5, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, log_like, o6, outn, st));
  LKB_TRY(stage_out_copy<int32_t>(mem, best_bins, ob, 2 * outn, st));
  if (mem == LKB_MEM_HOST) LKB_CUDA_CHECK(cudaStreamSynchronize(st));
  return LKB_OK;
}

}  // namespace lkb
