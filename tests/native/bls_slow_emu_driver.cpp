// Runs lightkurve_b200/csrc/bls_slow.cu - the WHOLE translation unit: the prologue and table kernels it shares with
// K3, the K3s search kernel, launch shapes and the host orchestration - on the CPU through tests/native/cuda_emu.h
// (TEST INFRASTRUCTURE).  Built by tests/test_bls_slow_emulated.py.
#include "cuda_emu.h"

#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <map>

#include "../../lightkurve_b200/csrc/bls_slow.cu"

// ---- the pieces of api.cu the translation unit links against ----
namespace lkb {
int64_t g_launches = 0;
static char g_err[512];
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
static std::map<int, std::pair<void*, size_t>> g_ws;
int ws_get(int slot, size_t bytes, void** out) {
  auto& e = g_ws[slot];
  if (e.second != bytes) {             // exact size, no slack: an out-of-bounds access is visible to ASan
    free(e.first);
    e.first = calloc(bytes ? bytes : 1, 1);
    e.second = bytes;
  }
  *out = e.first;
  return LKB_OK;
}
int ensure_device() { return LKB_OK; }
void prof_begin(cudaStream_t) {}
void prof_end(cudaStream_t) {}
int big_copy_h2d(void* dst, const void* src, size_t bytes, cudaStream_t) { memcpy(dst, src, bytes); return LKB_OK; }
int big_copy_d2h(void* dst, const void* src, size_t bytes, cudaStream_t) { memcpy(dst, src, bytes); return LKB_OK; }
}  // namespace lkb

extern "C" {

const char* emu_last_error() { return lkb::g_err; }
int64_t emu_launches() { return lkb::g_launches; }

// lkb_bls_power_slow with host buffers (mem = LKB_MEM_HOST: the staging path) or, with mem = LKB_MEM_DEVICE, the
// caller's buffers used in place
int emu_bls_power_slow(const double* t, const double* y, const double* dy, const int64_t* offsets, int B,
                       const double* period, int64_t P, const double* duration, int D, int oversample, int objective,
                       double* power, double* depth, double* depth_err, double* duration_out, double* transit_time,
                       double* depth_snr, double* log_likelihood, int32_t* best_index, int mem) {
  return lkb::bls_power_slow(t, y, dy, offsets, B, period, P, duration, D, oversample, objective, power, depth,
                             depth_err, duration_out, transit_time, depth_snr, log_likelihood, best_index, mem, nullptr);
}

}  // extern "C"
