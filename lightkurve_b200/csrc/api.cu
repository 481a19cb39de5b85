// extern "C" surface of liblkb200.so (declared in include/lkb200.h) + context/workspace.
#include <stdarg.h>
#include <mutex>
#include <thread>
#include <algorithm>
#include <cstring>
#include "common.cuh"

namespace lkb {

static thread_local char t_err[512] = "";
int64_t g_launches = 0;
int g_last_ls_algo = -1;      // kernel family the last Lomb-Scargle call ran (LKB_LS_ALGO_*; -1: none yet)

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

struct Ctx {
  bool inited = false;
  int device = -1;
  int sms = 0;
  void* ptr[WS_NSLOTS] = {nullptr};
  size_t cap[WS_NSLOTS] = {0};
};
static Ctx g_ctx;
static std::mutex g_mu;

// every compute entry point passes through ensure_device() exactly once: the epoch tells a cached plan (the shared-grid
// Lomb-Scargle keeps its y-independent tables in workspace slots) whether another entry point ran in between
int64_t g_epoch = 0;
int ensure_device() {
  g_epoch++;
  if (g_ctx.inited) {
    cudaError_t e = cudaSetDevice(g_ctx.device);
    if (e != cudaSuccess) { set_error("cudaSetDevice(%d): %s", g_ctx.device, cudaGetErrorString(e)); return LKB_E_CUDA; }
    return LKB_OK;
  }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    set_error("no CUDA device available (%s); liblkb200 has no CPU fallback",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    cudaGetLastError();
    return LKB_E_CUDA;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) { set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e)); return LKB_E_CUDA; }
  if (prop.major != 10) {
    set_error("liblkb200 is built for sm_100a only; device %d is sm_%d%d", dev, prop.major, prop.minor);
    return LKB_E_CUDA;
  }
  g_ctx.device = dev;
  g_ctx.sms = prop.multiProcessorCount;
  g_ctx.inited = true;
  return LKB_OK;
}

int sm_count() { return g_ctx.sms; }

static cudaStream_t g_aux = nullptr;
static cudaEvent_t g_ev_fork = nullptr, g_ev_join = nullptr;
int aux_stream_get(cudaStream_t* aux, cudaEvent_t* ev_fork, cudaEvent_t* ev_join) {
  if (!g_aux) {
    LKB_CUDA_CHECK(cudaStreamCreateWithFlags(&g_aux, cudaStreamNonBlocking));
    LKB_CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_fork, cudaEventDisableTiming));
    LKB_CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_join, cudaEventDisableTiming));
  }
  *aux = g_aux; *ev_fork = g_ev_fork; *ev_join = g_ev_join;
  return LKB_OK;
}

// two copy streams + a few events for the chunk-pipelined host-mode paths
static cudaStream_t g_h2d = nullptr, g_d2h = nullptr;
static cudaEvent_t g_pipe_ev[16];
int pipe_streams_get(cudaStream_t* h2d, cudaStream_t* d2h, cudaEvent_t** events, int* n_events) {
  if (!g_h2d) {
    LKB_CUDA_CHECK(cudaStreamCreateWithFlags(&g_h2d, cudaStreamNonBlocking));
    LKB_CUDA_CHECK(cudaStreamCreateWithFlags(&g_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 16; ++i) LKB_CUDA_CHECK(cudaEventCreateWithFlags(&g_pipe_ev[i], cudaEventDisableTiming));
  }
  *h2d = g_h2d; *d2h = g_d2h; *events = g_pipe_ev; *n_events = 16;
  return LKB_OK;
}

// ---- bounce-buffered copies of pageable host memory ----
constexpr size_t BOUNCE_BYTES = (size_t)32 << 20;
constexpr size_t BOUNCE_MIN = (size_t)16 << 20;           // smaller copies: plain cudaMemcpyAsync
static void* g_bounce[2] = {nullptr, nullptr};
static cudaEvent_t g_bounce_ev[2];
static int bounce_init() {
  if (g_bounce[0]) return LKB_OK;
  for (int i = 0; i < 2; ++i) {
    LKB_CUDA_CHECK(cudaHostAlloc(&g_bounce[i], BOUNCE_BYTES, cudaHostAllocDefault));
    LKB_CUDA_CHECK(cudaEventCreateWithFlags(&g_bounce_ev[i], cudaEventDisableTiming));
  }
  return LKB_OK;
}
static bool host_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}
static void par_memcpy(void* dst, const void* src, size_t n) {
  constexpr int NT = 4;
  std::thread th[NT - 1];
  const size_t part = ((n / NT) + 63) & ~(size_t)63;
  for (int i = 1; i < NT; ++i) {
    const size_t lo = std::min(n, part * i), hi = std::min(n, part * (i + 1));
    th[i - 1] = std::thread([=] { if (hi > lo) memcpy((char*)dst + lo, (const char*)src + lo, hi - lo); });
  }
  memcpy(dst, src, std::min(n, part));
  for (int i = 1; i < NT; ++i) th[i - 1].join();
}
int big_copy_h2d(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st) {
  if (bytes < BOUNCE_MIN || host_is_pinned(src_host) || getenv("LKB_NO_BOUNCE")) {
    LKB_CUDA_CHECK(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
    return LKB_OK;
  }
  LKB_TRY(bounce_init());
  int k = 0;
  for (size_t off = 0; off < bytes; off += BOUNCE_BYTES, k ^= 1) {
    const size_t n = std::min(BOUNCE_BYTES, bytes - off);
    LKB_CUDA_CHECK(cudaEventSynchronize(g_bounce_ev[k]));          // the DMA that last read this buffer is done
    par_memcpy(g_bounce[k], (const char*)src_host + off, n);
    LKB_CUDA_CHECK(cudaMemcpyAsync((char*)dst_dev + off, g_bounce[k], n, cudaMemcpyHostToDevice, st));
    LKB_CUDA_CHECK(cudaEventRecord(g_bounce_ev[k], st));
  }
  return LKB_OK;
}
int big_copy_d2h(void* dst_host, const void* src_dev, size_t bytes, cudaStream_t st) {
  if (bytes < BOUNCE_MIN || host_is_pinned(dst_host) || getenv("LKB_NO_BOUNCE")) {
    LKB_CUDA_CHECK(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, st));
    return LKB_OK;
  }
  LKB_TRY(bounce_init());
  // both buffers may still be the source of an earlier host->device DMA
  LKB_CUDA_CHECK(cudaEventSynchronize(g_bounce_ev[0]));
  LKB_CUDA_CHECK(cudaEventSynchronize(g_bounce_ev[1]));
  size_t prev_off = 0, prev_n = 0;
  int k = 0;
  for (size_t off = 0; off < bytes; off += BOUNCE_BYTES, k ^= 1) {
    const size_t n = std::min(BOUNCE_BYTES, bytes - off);
    LKB_CUDA_CHECK(cudaMemcpyAsync(g_bounce[k], (const char*)src_dev + off, n, cudaMemcpyDeviceToHost, st));
    LKB_CUDA_CHECK(cudaEventRecord(g_bounce_ev[k], st));
    if (prev_n) {                                                   // drain the previous chunk while this one flies
      LKB_CUDA_CHECK(cudaEventSynchronize(g_bounce_ev[k ^ 1]));
      par_memcpy((char*)dst_host + prev_off, g_bounce[k ^ 1], prev_n);
    }
    prev_off = off; prev_n = n;
  }
  if (prev_n) {
    LKB_CUDA_CHECK(cudaEventSynchronize(g_bounce_ev[k ^ 1]));
    par_memcpy((char*)dst_host + prev_off, g_bounce[k ^ 1], prev_n);
  }
  return LKB_OK;
}

// ---- dominant-kernel profiling ring ----
constexpr int PROF_MAX = 512;
static bool g_prof_on = false;
static int g_prof_n = 0;
static cudaEvent_t g_prof_ev[PROF_MAX][2];
static bool g_prof_created = false;
void prof_begin(cudaStream_t st) {
  if (!g_prof_on || g_prof_n >= PROF_MAX) return;
  if (!g_prof_created) {
    for (int i = 0; i < PROF_MAX; ++i) { cudaEventCreate(&g_prof_ev[i][0]); cudaEventCreate(&g_prof_ev[i][1]); }
    g_prof_created = true;
  }
  cudaEventRecord(g_prof_ev[g_prof_n][0], st);
}
void prof_end(cudaStream_t st) {
  if (!g_prof_on || g_prof_n >= PROF_MAX) return;
  cudaEventRecord(g_prof_ev[g_prof_n][1], st);
  g_prof_n++;
}

int ws_get(int slot, size_t bytes, void** out) {
  if (slot < 0 || slot >= WS_NSLOTS) { set_error("bad workspace slot"); return LKB_E_ARG; }
  if (bytes == 0) bytes = 16;
  if (g_ctx.cap[slot] < bytes) {
    if (g_ctx.ptr[slot]) {
      cudaDeviceSynchronize();   // buffer may still be in use by an earlier async call
      cudaFree(g_ctx.ptr[slot]);
      g_ctx.ptr[slot] = nullptr;
      g_ctx.cap[slot] = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&g_ctx.ptr[slot], want);
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
      return LKB_E_OOM;
    }
    g_ctx.cap[slot] = want;
  }
  *out = g_ctx.ptr[slot];
  return LKB_OK;
}

// implemented in the kernel translation units
int ls_power_ragged(const double*, const void*, int, const int64_t*, int, const double*, const int64_t*, int64_t,
                    int, const double*, float*, int, cudaStream_t, int);
int ls_power_shared(const double*, const void*, int, int, int64_t, const double*, int64_t, int, const double*,
                    float*, int, cudaStream_t, int);
int ls_power_chi2(const double*, const void*, int, const int64_t*, int, const double*, const int64_t*, int64_t, int,
                  int, const double*, float*, double*, int, cudaStream_t);
int bls_power(const double*, const double*, const double*, const int64_t*, int, const double*, int64_t,
              const double*, int, int, int, double*, double*, double*, double*, double*, double*, double*, int32_t*,
              int, cudaStream_t);
int bls_bin_index(const double*, int64_t, double, double, double, int32_t*, int, cudaStream_t);
int bls_power_slow(const double*, const double*, const double*, const int64_t*, int, const double*, int64_t,
                   const double*, int, int, int, double*, double*, double*, double*, double*, double*, double*,
                   int32_t*, int, cudaStream_t);
int flatten(const double*, const double*, const double*, const uint8_t*, const int64_t*, int, int, int, double, int,
            double, double*, double*, double*, int, cudaStream_t);
int regress(const double*, int, const double*, const double*, const uint8_t*, const double*, const double*, int,
            int64_t, int, double, int, double*, double*, uint8_t*, int32_t*, double*, int, cudaStream_t);
int nanmedian_std(const double*, const int64_t*, int, double*, double*, int, cudaStream_t);
int pg_logmedian(const double*, int, int64_t, const int32_t*, const int32_t*, int, double, double*, int, cudaStream_t);
int savgol_tables_host(int, int, double*, double*);

}  // namespace lkb

using namespace lkb;

extern "C" {

const char* lkb_last_error(void) { return t_err; }
int lkb_version(void) { return 1000 * 0 + 2; }

int lkb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int lkb_init(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  int n = lkb_device_count();
  if (n <= 0) { set_error("lkb_init: no CUDA device; liblkb200 has no CPU fallback"); return LKB_E_CUDA; }
  if (device < 0 || device >= n) { set_error("lkb_init: device %d out of range [0,%d)", device, n); return LKB_E_ARG; }
  if (g_ctx.inited && g_ctx.device != device) {
    set_error("lkb_init: already bound to device %d (one device per process)", g_ctx.device);
    return LKB_E_ARG;
  }
  LKB_CUDA_CHECK(cudaSetDevice(device));
  return ensure_device();
}

int lkb_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx.inited) return LKB_OK;
  cudaSetDevice(g_ctx.device);
  cudaDeviceSynchronize();
  for (int i = 0; i < WS_NSLOTS; ++i) {
    if (g_ctx.ptr[i]) cudaFree(g_ctx.ptr[i]);
    g_ctx.ptr[i] = nullptr;
    g_ctx.cap[i] = 0;
  }
  if (g_aux) { cudaStreamDestroy(g_aux); cudaEventDestroy(g_ev_fork); cudaEventDestroy(g_ev_join); g_aux = nullptr; }
  if (g_h2d) {
    cudaStreamDestroy(g_h2d); cudaStreamDestroy(g_d2h);
    for (int i = 0; i < 16; ++i) cudaEventDestroy(g_pipe_ev[i]);
    g_h2d = g_d2h = nullptr;
  }
  for (int i = 0; i < 2; ++i)
    if (g_bounce[i]) { cudaFreeHost(g_bounce[i]); cudaEventDestroy(g_bounce_ev[i]); g_bounce[i] = nullptr; }
  g_ctx.inited = false;
  g_epoch += 2;              // (nothing cached survives a shutdown)
  return LKB_OK;
}

int lkb_sm_count(void) { return g_ctx.inited ? g_ctx.sms : 0; }

int lkb_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_prof_on = on != 0;
  g_prof_n = 0;
  return LKB_OK;
}

int lkb_profile_read(double* ms_out, int max_n) {
  std::lock_guard<std::mutex> lk(g_mu);
  int n = g_prof_n < max_n ? g_prof_n : max_n;
  for (int i = 0; i < n; ++i) {
    if (cudaEventSynchronize(g_prof_ev[i][1]) != cudaSuccess) { set_error("profile event sync failed"); return LKB_E_CUDA; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, g_prof_ev[i][0], g_prof_ev[i][1]);
    ms_out[i] = (double)ms;
  }
  g_prof_n = 0;
  return n;
}
int64_t lkb_launch_count(void) { return g_launches; }
int lkb_ls_last_algo(void) { return g_last_ls_algo; }
int lkb_ls_last_escalated(void) { return g_last_ls_algo == LKB_LS_ALGO_NUFFT ? ls_nufft_last_escalated() : 0; }

// Diagnostic: copy `bytes` bytes at `offset` of workspace slot `slot` to the host buffer `out` (after a device
// synchronise).  Lets a test or tools/nufft_gpu_check.py look at the intermediate buffers of the last call.
int lkb_ws_read(int slot, int64_t offset, int64_t bytes, void* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  LKB_REQUIRE(g_ctx.inited, "lkb_ws_read: engine not initialised");
  LKB_REQUIRE(slot >= 0 && slot < WS_NSLOTS && out != nullptr && offset >= 0 && bytes >= 0, "lkb_ws_read: bad argument");
  LKB_REQUIRE(g_ctx.ptr[slot] != nullptr && (size_t)(offset + bytes) <= g_ctx.cap[slot],
              "lkb_ws_read: range outside the slot's current buffer");
  LKB_CUDA_CHECK(cudaDeviceSynchronize());
  LKB_CUDA_CHECK(cudaMemcpy(out, (const char*)g_ctx.ptr[slot] + offset, (size_t)bytes, cudaMemcpyDeviceToHost));
  return LKB_OK;
}

int lkb_ls_power(const double* t, const void* y, int y_dtype, const int64_t* offsets, int B, const double* freq,
                 const int64_t* freq_offsets, int64_t F, int normalization, const double* norm_scale, float* power,
                 int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return ls_power_ragged(t, y, y_dtype, offsets, B, freq, freq_offsets, F, normalization, norm_scale, power, mem,
                         (cudaStream_t)stream, LKB_LS_ALGO_AUTO);
}

int lkb_ls_power_ex(const double* t, const void* y, int y_dtype, const int64_t* offsets, int B, const double* freq,
                    const int64_t* freq_offsets, int64_t F, int normalization, const double* norm_scale, float* power,
                    int mem, void* stream, int algo) {
  std::lock_guard<std::mutex> lk(g_mu);
  return ls_power_ragged(t, y, y_dtype, offsets, B, freq, freq_offsets, F, normalization, norm_scale, power, mem,
                         (cudaStream_t)stream, algo);
}

int lkb_ls_power_shared(const double* t, const void* y, int y_dtype, int B, int64_t N, const double* freq, int64_t F,
                        int normalization, const double* norm_scale, float* power, int mem, void* stream, int algo) {
  std::lock_guard<std::mutex> lk(g_mu);
  return ls_power_shared(t, y, y_dtype, B, N, freq, F, normalization, norm_scale, power, mem, (cudaStream_t)stream,
                         algo);
}

int lkb_ls_power_chi2(const double* t, const void* y, int y_dtype, const int64_t* offsets, int B, const double* freq,
                      const int64_t* freq_offsets, int64_t F, int nterms, int normalization, const double* norm_scale,
                      float* power, double* theta, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return ls_power_chi2(t, y, y_dtype, offsets, B, freq, freq_offsets, F, nterms, normalization, norm_scale, power,
                       theta, mem, (cudaStream_t)stream);
}

int lkb_bls_power(const double* t, const double* y, const double* dy, const int64_t* offsets, int B,
                  const double* period, int64_t P, const double* duration, int D, int oversample, int objective,
                  double* power, double* depth, double* depth_err, double* duration_out, double* transit_time,
                  double* depth_snr, double* log_likelihood, int32_t* best_bins, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return bls_power(t, y, dy, offsets, B, period, P, duration, D, oversample, objective, power, depth, depth_err,
                   duration_out, transit_time, depth_snr, log_likelihood, best_bins, mem, (cudaStream_t)stream);
}

int lkb_bls_power_slow(const double* t, const double* y, const double* dy, const int64_t* offsets, int B,
                       const double* period, int64_t P, const double* duration, int D, int oversample, int objective,
                       double* power, double* depth, double* depth_err, double* duration_out, double* transit_time,
                       double* depth_snr, double* log_likelihood, int32_t* best_index, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return bls_power_slow(t, y, dy, offsets, B, period, P, duration, D, oversample, objective, power, depth, depth_err,
                        duration_out, transit_time, depth_snr, log_likelihood, best_index, mem, (cudaStream_t)stream);
}

int lkb_bls_bin_index(const double* t_rel, int64_t N, double min_t, double period, double bin_duration,
                      int32_t* ind, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return bls_bin_index(t_rel, N, min_t, period, bin_duration, ind, mem, (cudaStream_t)stream);
}

int lkb_flatten(const double* time, const double* flux, const double* flux_err, const uint8_t* exclude_mask,
                const int64_t* offsets, int B, int window_length, int polyorder, double break_tolerance, int niters,
                double sigma, double* flat, double* flat_err, double* trend, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return flatten(time, flux, flux_err, exclude_mask, offsets, B, window_length, polyorder, break_tolerance, niters,
                 sigma, flat, flat_err, trend, mem, (cudaStream_t)stream);
}

int lkb_regress(const double* X, int x_batched, const double* y, const double* flux_err, const uint8_t* cadence_mask,
                const double* prior_mu, const double* prior_sigma, int B, int64_t N, int K, double clip_sigma,
                int niters, double* coeff, double* model, uint8_t* outlier_mask, int32_t* status_out,
                double* coeff_cov, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return regress(X, x_batched, y, flux_err, cadence_mask, prior_mu, prior_sigma, B, N, K, clip_sigma, niters, coeff,
                 model, outlier_mask, status_out, coeff_cov, mem, (cudaStream_t)stream);
}

int lkb_savgol_tables(int window_length, int polyorder, double* coeffs, double* edge) {
  return savgol_tables_host(window_length, polyorder, coeffs, edge);
}

int lkb_nanmedian_std(const double* x, const int64_t* offsets, int B, double* out_median, double* out_std, int mem,
                      void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return nanmedian_std(x, offsets, B, out_median, out_std, mem, (cudaStream_t)stream);
}

int lkb_pg_logmedian(const double* power, int B, int64_t F, const int32_t* win_lo, const int32_t* win_hi, int W,
                     double corr_factor, double* background, int mem, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  return pg_logmedian(power, B, F, win_lo, win_hi, W, corr_factor, background, mem, (cudaStream_t)stream);
}

}  // extern "C"
