// Shared helpers for libsc_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/scb.h"

namespace scb {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define SCB_CHECK_ARG(cond, msg)                       \
  do {                                                 \
    if (!(cond)) {                                     \
      scb::set_error("%s: %s", __func__, msg);         \
      return SCB_ERR_INVALID;                          \
    }                                                  \
  } while (0)

#define SCB_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t _e = (call);                                                        \
    if (_e != cudaSuccess) {                                                        \
      scb::set_error("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
      return SCB_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

#define SCB_LAUNCH_CHECK()                                                          \
  do {                                                                              \
    scb::count_launch();                                                            \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess) {                                                        \
      scb::set_error("%s:%d kernel launch: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return SCB_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

// delaunay.cu: exclusive scan of count[0 .. ncells) in place with the total in count[ncells] (one CTA), and the
// sort of every cell's list order[start[c] .. start[c + 1]) by value
int launch_cell_scan(int32_t* count, int64_t ncells, cudaStream_t s);
int launch_cell_sort(int64_t ncells, const int32_t* start, int32_t* order, cudaStream_t s);

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

constexpr double kOneOver4Pi = 0.07957747154594767;  // 1/(4*pi)

// r2^(-3/2) in fp64 from the MUFU.RSQ64H seed y0 (relative error d <= 2^-22.9): with
// e = 1 - r2 y0^2 (|e| ~ 2 d, computed with one rounding of r2 y0 and an exact fma),
//   r2^(-3/2) = y0^3 (1 - e)^(-3/2) = y0^3 (1 + e (3/2 + 15/8 e) + O(e^3)),   35/16 e^3 < 2^-64,
// i.e. 7 DFMA-class operations (two Newton steps + cube: 9).  No denormal / special-case fix-ups:
// r2 is a squared distance between distinct mesh points; r2 == 0 yields NaN and callers mask it
// (q_ii = 0).
__device__ __forceinline__ double inv_r3(double r2) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(r2));
  const double e = fma(-(r2 * y), y, 1.0);
  const double ec = e * fma(1.875, e, 1.5);
  const double y3 = (y * y) * y;
  return fma(y3, ec, y3);
}
// r2^(-1/2) the same way: y0 (1 + e (1/2 + 3/8 e))
__device__ __forceinline__ double inv_r1(double r2) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(r2));
  const double e = fma(-(r2 * y), y, 1.0);
  return fma(y, e * fma(0.375, e, 0.5), y);
}

}  // namespace scb
