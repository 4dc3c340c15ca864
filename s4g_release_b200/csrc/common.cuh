// Shared helpers for the sm_100a kernels behind include/s4g_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/s4g_b200.h"

namespace s4g {

// thread-local error text, returned by s4g_last_error()
char* error_buffer();
int set_error(int code, const char* fmt, ...);

#define S4G_CHECK_ARG(cond, ...)                               \
  do {                                                         \
    if (!(cond)) return s4g::set_error(S4G_E_ARG, __VA_ARGS__); \
  } while (0)

#define S4G_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) return s4g::set_error((int)_e, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

// every kernel launch of the library passes here: s4g_launch_count() lets a caller report how many of OUR kernels ran
void count_launch();

#define S4G_LAUNCH_CHECK(name)                                                                 \
  do {                                                                                         \
    s4g::count_launch();                                                                       \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) return s4g::set_error((int)_e, "%s launch: %s", name, cudaGetErrorString(_e)); \
  } while (0)

// Squared distance with exactly the rounding sequence nvcc emits for the reference expression
// (x2-x1)*(x2-x1)+(y2-y1)*(y2-y1)+(z2-z1)*(z2-z1) under -fmad=true (checked in the SASS of the
// reference objects, oracle/_ref):  FMUL dy*dy ; FFMA dx*dx + . ; FFMA dz*dz + .
// The _rn intrinsics are never re-contracted by the compiler.
__device__ __forceinline__ float sqdist(float dx, float dy, float dz) {
  return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

// The reference's 3-NN starts from distances {1e40, 0, 0} and indices {-1, 0, 0} (interpolate_kernel.cu:53-54; 1e40 is
// +inf in fp32) and inserts a key only when its distance is below a slot's.  The searches here start all three slots at
// `big` (1e40 in the dtype), which reaches the same state once two keys are below `big`.  With fewer (NaN points,
// distances that overflow), this rewrites the slots to the reference's leftovers: with c keys below `big`, slot c is
// (big, -1) and the slots after it (0, index 0).  Slots are ascending, so the filled ones come first; a slot at `big` or
// above counts as unfilled, which also drops keys a search kept on a tie at +inf.  No-op when c = 3.
template <typename T>
__device__ __forceinline__ void three_nn_reference_tail(T& d0, T& d1, T& d2, int& i0, int& i1, int& i2, T big) {
  if (!(d2 < big)) { d2 = big; i2 = -1; }
  if (!(d1 < big)) { d1 = big; i1 = -1; d2 = T(0); i2 = 0; }
  if (!(d0 < big)) { d0 = big; i0 = -1; d1 = T(0); i1 = 0; }
}

// SM count of the CURRENT device (cached per device: a process may drive several GPUs)
inline int num_sms() {
  static int cache[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (cache[dev] == 0) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    cache[dev] = n > 0 ? n : 148;
  }
  return cache[dev];
}

// true the first time it is called for (flags, CURRENT device): per-device one-time set-up such as
// cudaFuncSetAttribute (function attributes are per device; a process may drive several GPUs)
inline bool first_use_on_device(bool (&flags)[64]) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (flags[dev]) return false;
  flags[dev] = true;
  return true;
}

}  // namespace s4g
