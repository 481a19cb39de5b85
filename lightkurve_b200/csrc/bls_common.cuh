// Pieces shared by the two BLS searches: K3 (bls.cu, astropy method="fast") and K3s (bls_slow.cu, method="slow").
// Both translation units are compiled with -fmad=false; the kernels here are `static` so that each unit keeps its own
// copy.
#pragma once
#include "common.cuh"
#include "select.cuh"

namespace lkb {

// exact fmod for finite x, p != 0, |x/p| < 2^50 (true for any real light curve)
__device__ __forceinline__ double bls_fmod(double x, double p, double inv_p) {
  const double a = fabs(x), b = fabs(p);
  if (a < b) return x;
  double q = trunc(a * inv_p);
  double r = fma(-q, b, a);
  if (r < 0.0) { q -= 1.0; r = fma(-q, b, a); }
  else if (r >= b) { q += 1.0; r = fma(-q, b, a); }
  return copysign(r, x);
}

// ---- prologue: astropy core.py power(): t - min(t), y - median(y), ivar = 1/dy^2 ----------
struct BlsLcInfo {
  double t_ref, sum_y, sum_ivar, min_t, x_max;
  int sorted, pad;
};

// Also produces what the boundary path needs: sortedness, the baseline, and the exclusive prefix sums
// cpre[i] = sum_{i' < i} {w*y, w} (N + 1 entries per light curve, at offset o + b).
static __global__ void __launch_bounds__(256)
bls_prep_kernel(const double* __restrict__ t, const double* __restrict__ y, const double* __restrict__ dy,
                const int64_t* __restrict__ offsets, double* __restrict__ trel, double* __restrict__ wy,
                double* __restrict__ iv, double2* __restrict__ cpre, BlsLcInfo* __restrict__ info) {
  __shared__ SelSmem sm;
  __shared__ double2 s_part[256];
  __shared__ int s_unsorted;
  const int b = blockIdx.x;
  const int64_t o = offsets[b], n = offsets[b + 1] - o;
  if (n <= 0) return;
  if (threadIdx.x == 0) s_unsorted = 0;
  // t_ref = min(t)
  double mn = __longlong_as_double(0x7ff0000000000000ll), mx = -mn;
  int unsorted = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = t[o + i];
    mn = fmin(mn, v);
    mx = fmax(mx, v);
    if (i + 1 < n && !(t[o + i + 1] >= v)) unsorted = 1;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, s));
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  }
  if ((threadIdx.x & 31) == 0) { sm.red[threadIdx.x >> 5] = mn; s_part[threadIdx.x >> 5].x = mx; }
  __syncthreads();
  if (unsorted) s_unsorted = 1;
  if (threadIdx.x == 0) {
    double x = sm.red[0], z = s_part[0].x;
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { x = fmin(x, sm.red[w]); z = fmax(z, s_part[w].x); }
    sm.red[32] = x;
    sm.red[31] = z;
  }
  __syncthreads();
  const double t_ref = sm.red[32], t_max = sm.red[31];
  __syncthreads();
  const double* yy = y + o;
  const double med = block_nanmedian([&](int64_t i) { return yy[i]; }, n, sm);
  // each thread owns a contiguous chunk so that the prefix sums can be formed in two passes
  const int64_t L = (n + blockDim.x - 1) / blockDim.x;
  const int64_t lo = min((int64_t)threadIdx.x * L, n), hi = min(lo + L, n);
  double sy = 0.0, si = 0.0;
  for (int64_t i = lo; i < hi; ++i) {
    const double w = dy ? 1.0 / (dy[o + i] * dy[o + i]) : 1.0;
    const double v = (yy[i] - med) * w;
    trel[o + i] = t[o + i] - t_ref;
    wy[o + i] = v;
    iv[o + i] = w;
    sy += v;
    si += w;
  }
  s_part[threadIdx.x] = make_double2(sy, si);
  __syncthreads();
  if (threadIdx.x == 0) {
    double ax = 0.0, ay = 0.0;
    for (int k = 0; k < (int)blockDim.x; ++k) {
      const double2 p = s_part[k];
      s_part[k] = make_double2(ax, ay);
      ax += p.x; ay += p.y;
    }
    info[b].t_ref = t_ref;
    info[b].sum_y = ax;
    info[b].sum_ivar = ay;
    info[b].min_t = 0.0;   // min(t - t_ref)
    info[b].x_max = t_max - t_ref;
    info[b].sorted = s_unsorted ? 0 : 1;
    info[b].pad = 0;
  }
  __syncthreads();
  if (cpre) {
    double2* c = cpre + o + b;
    double ax = s_part[threadIdx.x].x, ay = s_part[threadIdx.x].y;
    for (int64_t i = lo; i < hi; ++i) {
      c[i] = make_double2(ax, ay);
      ax += wy[o + i]; ay += iv[o + i];
    }
    if (hi == n && lo <= n) c[n] = make_double2(ax, ay);   // (every thread with hi == n holds the full sum)
  }
}

// T[j] = first cadence with x >= j * delta (lower bound), j = 0 .. nT - 1, per light curve.
static __global__ void __launch_bounds__(256)
bls_table_kernel(const double* __restrict__ trel, const int64_t* __restrict__ offsets,
                 const int64_t* __restrict__ tab_offsets, double delta, int32_t* __restrict__ tab) {
  const int b = blockIdx.y;
  const int64_t o = offsets[b], n = offsets[b + 1] - o;
  const int64_t to = tab_offsets[b], nT = tab_offsets[b + 1] - to;
  const double* x = trel + o;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nT; j += (int64_t)gridDim.x * blockDim.x) {
    const double target = (double)j * delta;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (x[mid] < target) lo = mid + 1; else hi = mid;
    }
    tab[to + j] = (int32_t)lo;
  }
}

}  // namespace lkb
