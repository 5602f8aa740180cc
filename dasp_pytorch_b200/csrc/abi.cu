// Library-level entry points of the C ABI: versioning, thread-local error string, device info.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"
#include "../../include/dasp_b200.h"

namespace dasp {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static thread_local int cached_dev = -1;
  static thread_local int cached_sms = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached_dev = dev;
    cached_sms = n;
  }
  return cached_sms;
}

static int g_forced_warps = 0;
int debug_forced_warps() { return g_forced_warps; }
static int g_flat_fb = 0;
int debug_flat_filterbank() { return g_flat_fb; }

void reverb_shutdown();  // reverb.cu

// (0,1) -> physical range of every element of a (rows, cols) parameter tensor, with the reference's range check
// (modules.py:83-84) done on the device: an element outside [0, 1] becomes NaN (its item can no longer produce a
// silently wrong result) and raises bit 0 of *flag; nothing is read back by the host here.
__global__ void denormalize_kernel(const float* __restrict__ p01, const float* __restrict__ lo,
                                   const float* __restrict__ span, float* __restrict__ out, int* __restrict__ flag,
                                   int64_t total, int cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % cols);
  const float v = p01[i];
  const bool ok = (v >= 0.0f) && (v <= 1.0f);          // NaN input fails both comparisons
  out[i] = ok ? fmaf(v, span[c], lo[c]) : __int_as_float(0x7fc00000);
  if (!ok && flag) atomicOr(flag, 1);
}

}  // namespace dasp

extern "C" {

int dasp_abi_version(void) { return DASP_ABI_VERSION; }
const char* dasp_last_error(void) { return dasp::g_err; }
int dasp_compiled_arch(void) { return 1000; }
void dasp_shutdown(void) { dasp::reverb_shutdown(); }
void dasp_debug_force_warps(int warps) { dasp::g_forced_warps = (warps == 1 || warps == 2 || warps == 4 || warps == 8 || warps == 16) ? warps : 0; }

int dasp_denormalize(const float* p01, const float* lo, const float* span, float* out, int* flag, int64_t rows,
                     int64_t cols, void* stream) {
  DASP_REQUIRE(rows >= 0 && cols >= 1 && cols < (1 << 20), "denormalize: bad shape rows=%lld cols=%lld", (long long)rows,
               (long long)cols);
  if (rows == 0) return DASP_OK;
  DASP_REQUIRE(p01 && lo && span && out, "denormalize: null pointer");
  const int64_t total = rows * cols;
  dasp::denormalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p01, lo, span, out, flag,
                                                                                               total, (int)cols);
  DASP_LAUNCH_OK("denormalize_kernel");
  return DASP_OK;
}

void dasp_debug_reverb_flat_filterbank(int on) { dasp::g_flat_fb = on ? 1 : 0; }

}  // extern "C"
