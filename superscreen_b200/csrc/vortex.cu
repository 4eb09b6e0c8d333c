// Vortices of a film solve (solver/solve_film.py:541-554).  The vortex term is linear in the
// right-hand side: with K = -(-A)^-1,  g += flux nPhi0 K[:, j_film] / w[j_device]  is the solution of
// (-A) x = h - flux nPhi0 / w[j_device] e_{j_film}.  So a vortex costs no extra solve: it is a sparse
// correction to its column's right-hand side before the triangular solves.
#include <math.h>

#include "scb_common.cuh"

namespace scb {

constexpr int kLocateThreads = 128;

// numpy's argmin order on (value, index) pairs: NaN first, then the smaller value, ties to the lower index.
// A total order, so the reduction result does not depend on the order in which pairs are combined.
__device__ __forceinline__ bool argmin_before(double da, int64_t ia, double db, int64_t ib) {
  const bool na = isnan(da), nb = isnan(db);
  if (na || nb) return na && (!nb || ia < ib);
  return da < db || (da == db && ia < ib);
}

// np.linalg.norm(p - q) of one 2-vector, rounded exactly as numpy rounds it: sqrt((px-qx)^2 + (py-qy)^2)
// with every operation rounded on its own (no FMA contraction).
__device__ __forceinline__ double norm2_rn(double px, double py, double qx, double qy) {
  const double dx = __dsub_rn(px, qx), dy = __dsub_rn(py, qy);
  return __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

__device__ __forceinline__ void block_argmin(double& d, int64_t& i, double* sd, int64_t* si) {
  for (int off = 16; off > 0; off >>= 1) {
    const double d2 = __shfl_down_sync(0xffffffffu, d, off);
    const int64_t i2 = __shfl_down_sync(0xffffffffu, i, off);
    if (argmin_before(d2, i2, d, i)) d = d2, i = i2;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();  // (sd / si are reused by the second reduction)
  if (lane == 0) sd[warp] = d, si[warp] = i;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kLocateThreads / 32; w++)
      if (argmin_before(sd[w], si[w], d, i)) d = sd[w], i = si[w];
  }
}

// One block per query point: the nearest of the n_sub sites sites[sub[k]] (-> k) and of all n sites (-> i).
__global__ void __launch_bounds__(kLocateThreads) locate_vortices_kernel(
    const double* __restrict__ xy, int64_t n, const double* __restrict__ sites, int64_t n_sub,
    const int64_t* __restrict__ sub, int64_t* __restrict__ j_sub, int64_t* __restrict__ j_all) {
  __shared__ double sd[kLocateThreads / 32];
  __shared__ int64_t si[kLocateThreads / 32];
  const int64_t v = blockIdx.x;
  const double qx = xy[2 * v], qy = xy[2 * v + 1];
  double d_all = INFINITY, d_sub = INFINITY;
  int64_t i_all = INT64_MAX, i_sub = INT64_MAX;
  for (int64_t i = threadIdx.x; i < n; i += kLocateThreads) {
    const double d = norm2_rn(sites[2 * i], sites[2 * i + 1], qx, qy);
    if (argmin_before(d, i, d_all, i_all)) d_all = d, i_all = i;
  }
  for (int64_t k = threadIdx.x; k < n_sub; k += kLocateThreads) {
    const int64_t i = sub[k];
    const double d = norm2_rn(sites[2 * i], sites[2 * i + 1], qx, qy);
    if (argmin_before(d, k, d_sub, i_sub)) d_sub = d, i_sub = k;
  }
  block_argmin(d_all, i_all, sd, si);
  block_argmin(d_sub, i_sub, sd, si);
  if (threadIdx.x == 0) {
    j_all[v] = i_all;
    j_sub[v] = i_sub;
  }
}

// One thread per column c: B[row[v], c] -= flux nphi0[v] / weights[j_all[v]] * scale[row[v]] for the
// vortices v of that column, in order (no atomics; two vortices at one vertex simply add).  Evaluated left
// to right with one rounding per operation (no FMA contraction): the result is fixed by IEEE arithmetic.
__global__ void vortex_rhs_kernel(int64_t nrhs, const int64_t* __restrict__ col_ptr, const int64_t* __restrict__ row,
                                  const int64_t* __restrict__ j_all, const double* __restrict__ nphi0,
                                  const double* __restrict__ weights, double flux, const double* __restrict__ scale,
                                  double* __restrict__ B) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= nrhs) return;
  for (int64_t v = col_ptr[c]; v < col_ptr[c + 1]; v++) {
    const int64_t r = row[v];
    double t = __ddiv_rn(__dmul_rn(flux, nphi0[v]), weights[j_all[v]]);
    if (scale) t = __dmul_rn(t, scale[r]);
    B[r * nrhs + c] = __dsub_rn(B[r * nrhs + c], t);
  }
}
}  // namespace scb

using namespace scb;

extern "C" int scb_locate_vortices(int64_t nv, const double* xy, int64_t n, const double* sites, int64_t n_sub,
                                   const int64_t* sub, int64_t* j_sub, int64_t* j_all, scb_stream_t stream) {
  SCB_CHECK_ARG(nv >= 0 && n >= 0 && n_sub >= 0, "bad sizes");
  if (nv == 0) return SCB_OK;
  SCB_CHECK_ARG(n > 0 && n_sub > 0, "bad sizes: no sites to search");
  SCB_CHECK_ARG(nv <= 0x7fffffff, "bad sizes: too many query points");
  locate_vortices_kernel<<<(unsigned)nv, kLocateThreads, 0, (cudaStream_t)stream>>>(xy, n, sites, n_sub, sub,
                                                                                      j_sub, j_all);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

extern "C" int scb_vortex_rhs(int64_t nrhs, const int64_t* col_ptr, const int64_t* row, const int64_t* j_all,
                              const double* nphi0, const double* weights, double flux, const double* scale, double* B,
                              scb_stream_t stream) {
  SCB_CHECK_ARG(nrhs >= 0, "bad sizes");
  if (nrhs == 0) return SCB_OK;
  vortex_rhs_kernel<<<(unsigned)ceil_div(nrhs, 128), 128, 0, (cudaStream_t)stream>>>(nrhs, col_ptr, row, j_all, nphi0,
                                                                                    weights, flux, scale, B);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}
