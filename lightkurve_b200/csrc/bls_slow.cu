// K3s: exact (unbinned) Box Least Squares, astropy's BoxLeastSquares.power(..., method="slow"), which lightkurve
// reaches by passing `method=` through to_periodogram("bls", ...) (periodogram.py:1169 in lightkurve).
// The numerical contract (astropy timeseries/periodograms/bls/methods.py::_bls_slow_one, restated in
// oracle/bls.py::bls_power_slow_numpy): for every period P and every trial duration d (in the given order), the
// transit epochs t0_i = i * (d / oversample), i = 0 .. ceil((P + d/oversample) / (d/oversample)) - 1, and the box
//     in(x) = |((x - t0 + P/2) % P) - P/2| < d/2          (x = t - min(t); numpy %: fmod, + P if negative)
// the statistics of the in-box and out-of-box weighted means, kept for the FIRST strict maximum of the objective with
// depth > 0.  The reported duration is d itself and the transit time (t0 % P) + min(t).
//
// B200 mapping: one WARP per (light curve, period), CTA = BLS_SLOW_WARPS consecutive periods of one light curve (its
// time stamps, prefix sums and lookup table are shared through L1/L2); lanes take consecutive t0 of one duration.
// For one t0, the cadences of cycle c (centre xc = t0 + c P) that pass the predicate form ONE contiguous run of the
// ascending times: every rounded operation of the predicate is monotone in x within the half-open cycle domain
// (xc - P/2, xc + P/2], and d/2 < P/2 (the duration/period validation).  So a lane
//   - lands a few cadences before each end of the window through the table "first cadence at or after j * delta",
//   - moves each end with the EXACT predicate on the neighbouring cadences (never with arithmetic on the bounds),
//   - adds the run's {w*y, w} as a difference of the exclusive prefix sums cpre,
// which costs O(number of cycles) per box instead of O(N).  The out-of-box sums are the totals minus the in-box sums.
//
// Bit-exactness of the membership: (x - t0) + P/2 is rounded twice like numpy, the fmod is exact (bls_fmod) and the
// file is compiled with -fmad=false (no contraction of a*b+c anywhere).  Sums are formed in a different order than
// numpy's => values agree to ~1e-13 relative; boxes with the same member cadences have bitwise equal sums (the same
// runs), so exact ties are broken like astropy's loop: the first (duration index, t0 index) wins.
#include "bls_common.cuh"
#include <float.h>
#include <algorithm>
#include <vector>

namespace lkb {

constexpr int BLS_SLOW_WARPS = 8;

struct BlsSlowTab {
  const double2* cpre;        // [total + B] exclusive prefix sums of {w*y, w}
  const int32_t* tab;         // per light curve: first cadence with x >= j * delta
  const int64_t* tab_offsets; // [B + 1]
  double inv_delta;
};

// astropy's membership test for one cadence (x = time since the first cadence, min(x) = 0)
__device__ __forceinline__ bool bls_slow_in(double x, double t0, double hp, double per, double inv_per,
                                            double half_dur) {
  double r = bls_fmod((x - t0) + hp, per, inv_per);
  if (r < 0.0) r = r + per;
  return fabs(r - hp) < half_dur;
}

// first cadence at or after the table cell below v - delta (every cadence before it lies below v - delta)
__device__ __forceinline__ int bls_slow_land(const int32_t* tab, int nT, double v, double inv_delta) {
  double j = floor(v * inv_delta) - 1.0;
  j = fmin(fmax(j, 0.0), (double)(nT - 1));
  return tab[(int)j];
}

struct BlsSlowStats {
  double depth, depth_err, snr, ll, obj;
};

// astropy's statistics of one box from its in-box sums {sy = sum w*y, si = sum w} and member count
__device__ __forceinline__ BlsSlowStats bls_slow_stats(double sy, double si, int cnt, int n, double sum_y,
                                                      double sum_ivar, int objective) {
  double yw_out = sum_y - sy, ivar_out = sum_ivar - si;
  if (cnt == n) { yw_out = 0.0; ivar_out = 0.0; }      // no cadence out of the box: 0/0 like numpy's empty sums
  BlsSlowStats s;
  s.depth = yw_out / ivar_out - sy / si;                // y_out - y_in; an empty box gives 0/0 = NaN
  s.depth_err = sqrt(1.0 / si + 1.0 / ivar_out);
  s.snr = s.depth / s.depth_err;
  s.ll = 0.5 * si * s.depth * s.depth;                  // = the likelihood difference of astropy's two sums
  s.obj = objective ? s.snr : s.ll;
  return s;
}

__global__ void __launch_bounds__(BLS_SLOW_WARPS * 32)
bls_slow_kernel(const double* __restrict__ trel, const int64_t* __restrict__ offsets,
                const BlsLcInfo* __restrict__ info, const double* __restrict__ period, int64_t P,
                const double* __restrict__ duration, int D, int oversample, int objective, BlsSlowTab tb,
                double* __restrict__ o_power, double* __restrict__ o_depth, double* __restrict__ o_depth_err,
                double* __restrict__ o_duration, double* __restrict__ o_ttime, double* __restrict__ o_snr,
                double* __restrict__ o_ll, int32_t* __restrict__ o_index) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (p >= P) return;                                   // warp-uniform
  const int64_t o = offsets[b], n64 = offsets[b + 1] - o;
  const int64_t oi = (int64_t)b * P + p;
  if (n64 <= 0) {                                       // empty light curve: every output NaN
    if (lane == 0) {
      const double qn = __longlong_as_double(0x7ff8000000000000ll);
      o_power[oi] = qn; o_depth[oi] = qn; o_depth_err[oi] = qn; o_duration[oi] = qn; o_ttime[oi] = qn;
      o_snr[oi] = qn; o_ll[oi] = qn;
      if (o_index) { o_index[3 * oi] = -1; o_index[3 * oi + 1] = -1; o_index[3 * oi + 2] = 0; }
    }
    return;
  }
  const int n = (int)n64;
  const double sum_y = info[b].sum_y, sum_ivar = info[b].sum_ivar, x_max = info[b].x_max;
  const double* x = trel + o;
  const double2* cp = tb.cpre + o + b;
  const int32_t* tab = tb.tab + tb.tab_offsets[b];
  const int nT = (int)(tb.tab_offsets[b + 1] - tb.tab_offsets[b]);
  const double per = period[p], inv_per = 1.0 / per, hp = 0.5 * per;

  // this lane's first strict maximum, in its own (duration, t0) order; its statistics are re-derived at the end from
  // the in-box sums
  double best_obj = -INFINITY, b_sy = 0.0, b_si = 0.0;
  int best_k = 0x7fffffff, best_i = 0x7fffffff, b_cnt = 0;
  for (int k = 0; k < D; ++k) {
    const double dur = duration[k];
    const double d_phase = dur / (double)oversample;
    const double half = 0.5 * dur;
    const int n_t0 = (int)ceil((per + d_phase) / d_phase);     // len(np.arange(0, P + d_phase, d_phase))
    for (int i = lane; i < n_t0; i += 32) {
      const double t0 = (double)i * d_phase;
      // cycles whose domain (xc - P/2, xc + P/2] can hold a cadence of [0, x_max]
      const int c_lo = (int)floor((-hp - t0) * inv_per), c_hi = (int)ceil((x_max + hp - t0) * inv_per);
      double sy = 0.0, si = 0.0;
      int cnt = 0;
      for (int c = c_lo; c <= c_hi; ++c) {
        const double xc = t0 + (double)c * per;
        // lower end: first cadence of the run (or, if the window is empty, the first at or after the centre)
        int e = bls_slow_land(tab, nT, xc - half, tb.inv_delta);
        while (e < n) {
          const double xv = x[e];
          if (xv >= xc || (xv > xc - hp && bls_slow_in(xv, t0, hp, per, inv_per, half))) break;
          ++e;
        }
        const int lo = e;
        // upper end: every cadence between lo and the landing point is inside the window by ~delta
        e = max(lo, bls_slow_land(tab, nT, xc + half, tb.inv_delta));
        while (e < n) {
          const double xv = x[e];
          if (xv > xc + hp || !bls_slow_in(xv, t0, hp, per, inv_per, half)) break;
          ++e;
        }
        if (e > lo) {
          const double2 ca = cp[lo], cb = cp[e];
          sy += cb.x - ca.x;
          si += cb.y - ca.y;
          cnt += e - lo;
        }
      }
      const BlsSlowStats st = bls_slow_stats(sy, si, cnt, n, sum_y, sum_ivar, objective);
      if (st.depth > 0.0 && st.obj > best_obj) {        // (NaN depth of an empty box fails the test)
        best_obj = st.obj; best_k = k; best_i = i; b_cnt = cnt; b_sy = sy; b_si = si;
      }
    }
  }
  // first maximum in (duration index, t0 index) order across lanes
  double wobj = best_obj;
  int wk = best_k, wi = best_i;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    const double oo = __shfl_xor_sync(0xffffffffu, wobj, s);
    const int ok = __shfl_xor_sync(0xffffffffu, wk, s);
    const int on = __shfl_xor_sync(0xffffffffu, wi, s);
    const bool take = (oo > wobj) || (oo == wobj && (ok < wk || (ok == wk && on < wi)));
    if (take) { wobj = oo; wk = ok; wi = on; }
  }
  if (wk == 0x7fffffff) {
    // no box with depth > 0 (astropy itself fails here): power -inf, the rest as K3 leaves a period without a box
    if (lane == 0) {
      o_power[oi] = -INFINITY; o_depth[oi] = 0.0; o_depth_err[oi] = 0.0; o_snr[oi] = 0.0; o_ll[oi] = 0.0;
      o_duration[oi] = 0.0; o_ttime[oi] = info[b].t_ref;
      if (o_index) { o_index[3 * oi] = -1; o_index[3 * oi + 1] = -1; o_index[3 * oi + 2] = 0; }
    }
    return;
  }
  if (best_k == wk && best_i == wi) {                   // the lane that holds the winner writes it
    const BlsSlowStats st = bls_slow_stats(b_sy, b_si, b_cnt, n, sum_y, sum_ivar, objective);
    const double dur = duration[wk];
    o_power[oi] = best_obj;
    o_depth[oi] = st.depth;
    o_depth_err[oi] = st.depth_err;
    o_snr[oi] = st.snr;
    o_ll[oi] = st.ll;
    o_duration[oi] = dur;
    o_ttime[oi] = bls_fmod((double)wi * (dur / (double)oversample), per, inv_per) + info[b].t_ref;
    if (o_index) { o_index[3 * oi] = wk; o_index[3 * oi + 1] = wi; o_index[3 * oi + 2] = b_cnt; }
  }
}

// ---- host ------------------------------------------------------------------------------------
int bls_power_slow(const double* t, const double* y, const double* dy, const int64_t* h_offsets, int B,
                   const double* period, int64_t P, const double* duration, int D, int oversample, int objective,
                   double* power, double* depth, double* depth_err, double* duration_out, double* transit_time,
                   double* depth_snr, double* log_like, int32_t* best_index, int mem, cudaStream_t st) {
  LKB_REQUIRE(t && y && h_offsets && period && duration, "lkb_bls_power_slow: null input");
  LKB_REQUIRE(power && depth && depth_err && duration_out && transit_time && depth_snr && log_like,
              "lkb_bls_power_slow: null output");
  LKB_REQUIRE(B > 0 && B <= 65535 && P > 0 && D > 0 && oversample > 0, "lkb_bls_power_slow: bad sizes");
  LKB_REQUIRE(objective == 0 || objective == 1, "lkb_bls_power_slow: bad objective");
  LKB_TRY(ensure_device());
  const int64_t total = h_offsets[B];
  for (int b = 0; b < B; ++b)
    LKB_REQUIRE(h_offsets[b + 1] - h_offsets[b] < ((int64_t)1 << 31), "lkb_bls_power_slow: light curve too long");

  // the grids are needed on the host for validation and for the table resolution
  std::vector<double> h_per(P), h_dur(D);
  if (mem == LKB_MEM_HOST) {
    memcpy(h_per.data(), period, sizeof(double) * P);
    memcpy(h_dur.data(), duration, sizeof(double) * D);
  } else {
    LKB_CUDA_CHECK(cudaMemcpyAsync(h_per.data(), period, sizeof(double) * P, cudaMemcpyDeviceToHost, st));
    LKB_CUDA_CHECK(cudaMemcpyAsync(h_dur.data(), duration, sizeof(double) * D, cudaMemcpyDeviceToHost, st));
    LKB_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  double min_period = h_per[0], max_period = h_per[0], max_dur = h_dur[0], min_dur = h_dur[0];
  for (int64_t i = 0; i < P; ++i) {
    if (!(h_per[i] == h_per[i]) || isinf(h_per[i])) { set_error("lkb_bls_power_slow: period contains nan/inf"); return LKB_E_ARG; }
    min_period = fmin(min_period, h_per[i]);
    max_period = fmax(max_period, h_per[i]);
  }
  for (int i = 0; i < D; ++i) {
    if (!(h_dur[i] == h_dur[i]) || isinf(h_dur[i])) { set_error("lkb_bls_power_slow: duration contains nan/inf"); return LKB_E_ARG; }
    min_dur = fmin(min_dur, h_dur[i]);
    max_dur = fmax(max_dur, h_dur[i]);
  }
  if (min_period < DBL_EPSILON) { set_error("lkb_bls_power_slow: periods must be positive"); return LKB_E_ARG; }
  if (max_dur >= min_period || min_dur < DBL_EPSILON) {
    set_error("The maximum transit duration must be shorter than the minimum period");
    return LKB_E_ARG;
  }
  if (max_period / (min_dur / (double)oversample) > 1.0e9) {
    set_error("lkb_bls_power_slow: more than 1e9 transit epochs per (period, duration)");
    return LKB_E_UNSUPPORTED;
  }
  // table resolution: K3's boundary-path cell, a few cadences of walking per window end at TESS cadences
  const double delta = min_dur / (double)oversample / 8.0;

  const double *d_t = nullptr, *d_y = nullptr, *d_dy = nullptr, *d_per = nullptr, *d_dur = nullptr;
  LKB_TRY(stage_in<double>(mem, WS_IN0, t, total, &d_t, st));
  LKB_TRY(stage_in<double>(mem, WS_IN1, y, total, &d_y, st));
  LKB_TRY(stage_in<double>(mem, WS_IN2, dy, total, &d_dy, st));
  LKB_TRY(stage_in<double>(mem, WS_IN3, period, P, &d_per, st));
  LKB_TRY(stage_in<double>(mem, WS_IN4, duration, D, &d_dur, st));
  int64_t* d_off = nullptr;
  LKB_TRY(ws_get_t<int64_t>(WS_A, B + 1, &d_off));
  LKB_CUDA_CHECK(cudaMemcpyAsync(d_off, h_offsets, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, st));

  double *d_trel = nullptr, *d_wy = nullptr, *d_iv = nullptr;
  BlsLcInfo* d_info = nullptr;
  double2* d_cpre = nullptr;
  LKB_TRY(ws_get_t<double>(WS_C, total, &d_trel));
  LKB_TRY(ws_get_t<double>(WS_D, total, &d_wy));
  LKB_TRY(ws_get_t<double>(WS_E, total, &d_iv));
  LKB_TRY(ws_get_t<BlsLcInfo>(WS_F, B, &d_info));
  LKB_TRY(ws_get_t<double2>(WS_H, total + B, &d_cpre));
  LKB_LAUNCH(B, 256, st, bls_prep_kernel)(d_t, d_y, d_dy, d_off, d_trel, d_wy, d_iv, d_cpre, d_info);
  LKB_LAUNCH_CHECK();

  // per-light-curve tables "first cadence at or after j * delta"; the search needs ascending times
  std::vector<BlsLcInfo> h_info(B);
  LKB_CUDA_CHECK(cudaMemcpyAsync(h_info.data(), d_info, sizeof(BlsLcInfo) * B, cudaMemcpyDeviceToHost, st));
  LKB_CUDA_CHECK(cudaStreamSynchronize(st));
  std::vector<int64_t> h_to(B + 1, 0);
  int64_t nT_max = 0;
  for (int b = 0; b < B; ++b) {
    const int64_t nb = h_offsets[b + 1] - h_offsets[b];
    int64_t nT = 0;
    if (nb > 0) {
      if (!h_info[b].sorted) {
        set_error("lkb_bls_power_slow: light curve %d: times are not ascending (sort them first)", b);
        return LKB_E_UNSUPPORTED;
      }
      const double cells = h_info[b].x_max / delta;
      if (!(cells >= 0.0) || cells > 1.0e9) {
        set_error("lkb_bls_power_slow: light curve %d: baseline / (min(duration) / oversample / 8) = %g cells is too "
                  "many for the lookup table", b, cells);
        return LKB_E_UNSUPPORTED;
      }
      nT = (int64_t)cells + 3;
    }
    h_to[b + 1] = h_to[b] + nT;
    nT_max = nT > nT_max ? nT : nT_max;
  }
  int64_t* d_to = nullptr;
  int32_t* d_tab = nullptr;
  LKB_TRY(ws_get_t<int64_t>(WS_I, B + 1, &d_to));
  LKB_TRY(ws_get_t<int32_t>(WS_J, h_to[B] > 0 ? h_to[B] : 1, &d_tab));
  LKB_CUDA_CHECK(cudaMemcpyAsync(d_to, h_to.data(), sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, st));
  LKB_CUDA_CHECK(cudaStreamSynchronize(st));   // h_to is a local
  if (nT_max > 0) {
    const unsigned gxT = (unsigned)std::min((int64_t)64, (nT_max + 255) / 256);
    LKB_LAUNCH(dim3(gxT, (unsigned)B), 256, st, bls_table_kernel)(d_trel, d_off, d_to, delta, d_tab);
    LKB_LAUNCH_CHECK();
  }

  const size_t outn = (size_t)B * P;
  double *o0, *o1, *o2, *o3, *o4, *o5, *o6;
  int32_t* oidx = nullptr;
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT0, power, outn, &o0));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT1, depth, outn, &o1));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT2, depth_err, outn, &o2));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT3, duration_out, outn, &o3));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT4, transit_time, outn, &o4));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT5, depth_snr, outn, &o5));
  LKB_TRY(stage_out_alloc<double>(mem, WS_OUT6, log_like, outn, &o6));
  LKB_TRY(stage_out_alloc<int32_t>(mem, WS_OUT7, best_index, 3 * outn, &oidx));

  BlsSlowTab tb;
  tb.cpre = d_cpre;
  tb.tab = d_tab;
  tb.tab_offsets = d_to;
  tb.inv_delta = 1.0 / delta;
  const dim3 grid((unsigned)((P + BLS_SLOW_WARPS - 1) / BLS_SLOW_WARPS), (unsigned)B);
  prof_begin(st);
  LKB_LAUNCH(grid, BLS_SLOW_WARPS * 32, st, bls_slow_kernel)(d_trel, d_off, d_info, d_per, P, d_dur, D, oversample,
                                                             objective, tb, o0, o1, o2, o3, o4, o5, o6, oidx);
  LKB_LAUNCH_CHECK();
  prof_end(st);

  LKB_TRY(stage_out_copy<double>(mem, power, o0, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, depth, o1, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, depth_err, o2, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, duration_out, o3, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, transit_time, o4, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, depth_snr, o5, outn, st));
  LKB_TRY(stage_out_copy<double>(mem, log_like, o6, outn, st));
  LKB_TRY(stage_out_copy<int32_t>(mem, best_index, oidx, 3 * outn, st));
  if (mem == LKB_MEM_HOST) LKB_CUDA_CHECK(cudaStreamSynchronize(st));
  return LKB_OK;
}

}  // namespace lkb
