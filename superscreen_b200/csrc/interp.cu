// Point location, linear interpolation and polygon masks on a triangulation: the device stage between a batch of
// solutions and the images drawn from it (Solution.interp_current_density / interp_field, reference
// solution.py:272-276,310-312, matplotlib's LinearTriInterpolator; the film mask of geometry.points_in_polygon).
//
//   scb_tri_grid_count / _fill  uniform cell grid over the triangles: every triangle is registered in every cell
//                               that its padded bounding box overlaps (count -> scan -> scatter -> per-cell sort,
//                               the sequence and the scan / sort kernels of delaunay.cu's point grid);
//   scb_tri_locate              one thread per query point: the best triangle among those of the point's cell;
//   scb_tri_interpolate         one thread per (point, group of value sets);
//   scb_points_in_polygon       one thread per point, polygon edges staged through shared memory.
//
// Every comparison that decides a result is made on values rounded exactly as the host's numpy code rounds them
// (explicit __d*_rn operations: no FMA contraction), so the results are functions of the inputs alone.
#include <math.h>

#include "scb_common.cuh"

namespace scb {

constexpr int kPolyTile = 256;  // polygon vertices staged per shared-memory tile (= threads per block)
constexpr int kInterpSets = 8;  // value sets per thread of the interpolation kernel

__device__ __forceinline__ int grid_coord(double v, double v0, double inv_cell, int nc) {
  const int c = (int)floor(__dmul_rn(__dsub_rn(v, v0), inv_cell));
  return c < 0 ? 0 : (c >= nc ? nc - 1 : c);
}

// Cell range [cx0, cx1] x [cy0, cy1] of every triangle, and the number of triangles of every cell.
//
// Padding.  A point p outside a triangle by a distance R has an exact barycentric coordinate <= -R / L (L: the
// longest edge, which bounds every height).  The rounded coordinates of _barycentric differ from the exact ones
// by at most c eps (kappa (1 + R / L) + 1), kappa = L^2 / |det|, c a small constant.  So a point whose rounded
// coordinates are all >= -1e-12 lies within R <= 2 L (1e-12 + c eps kappa) of the triangle as long as
// c eps kappa < 1/2.  The box is padded by twice that bound with c = 32 (plus the rounding of the coordinates
// themselves); a triangle with c eps kappa >= 1/8 -- all but degenerate -- is registered in every cell.  A
// triangle with det == 0 has no finite coordinates and never wins: it is registered nowhere.
__global__ void tri_grid_count_kernel(int64_t ntri, const double* __restrict__ sites, const int64_t* __restrict__ el,
                                      double x0, double y0, double inv_cell, int ncx, int ncy,
                                      int4* __restrict__ range, int32_t* __restrict__ count) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= ntri) return;
  const int64_t ia = el[3 * t], ib = el[3 * t + 1], ic = el[3 * t + 2];
  const double ax = sites[2 * ia], ay = sites[2 * ia + 1], bx = sites[2 * ib], by = sites[2 * ib + 1];
  const double cx = sites[2 * ic], cy = sites[2 * ic + 1];
  const double det = __dadd_rn(__dmul_rn(__dsub_rn(by, cy), __dsub_rn(ax, cx)),
                               __dmul_rn(__dsub_rn(cx, bx), __dsub_rn(ay, cy)));
  int4 r = make_int4(0, -1, 0, -1);  // (empty)
  if (det != 0.0) {
    const double lab = hypot(ax - bx, ay - by), lbc = hypot(bx - cx, by - cy), lca = hypot(cx - ax, cy - ay);
    const double L = fmax(lab, fmax(lbc, lca));
    const double ce_kappa = 32.0 * 2.220446049250313e-16 * (L * L / fabs(det));
    if (ce_kappa < 0.125) {  // (false for NaN / inf as well)
      const double xmin = fmin(ax, fmin(bx, cx)), xmax = fmax(ax, fmax(bx, cx));
      const double ymin = fmin(ay, fmin(by, cy)), ymax = fmax(ay, fmax(by, cy));
      const double absmax = fmax(fmax(fabs(xmin), fabs(xmax)), fmax(fabs(ymin), fabs(ymax)));
      const double pad = 4.0 * L * (1e-12 + ce_kappa) + 16.0 * 2.220446049250313e-16 * absmax;
      r = make_int4(grid_coord(xmin - pad, x0, inv_cell, ncx), grid_coord(xmax + pad, x0, inv_cell, ncx),
                    grid_coord(ymin - pad, y0, inv_cell, ncy), grid_coord(ymax + pad, y0, inv_cell, ncy));
    } else {
      r = make_int4(0, ncx - 1, 0, ncy - 1);
    }
  }
  range[t] = r;
  for (int j = r.z; j <= r.w; j++)
    for (int i = r.x; i <= r.y; i++) atomicAdd(&count[(int64_t)j * ncx + i], 1);
}

__global__ void tri_grid_scatter_kernel(int64_t ntri, int ncx, const int4* __restrict__ range,
                                        const int32_t* __restrict__ start, int32_t* __restrict__ fill,
                                        int32_t* __restrict__ cell_tris) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= ntri) return;
  const int4 r = range[t];
  for (int j = r.z; j <= r.w; j++)
    for (int i = r.x; i <= r.y; i++) {
      const int64_t c = (int64_t)j * ncx + i;
      cell_tris[start[c] + atomicAdd(&fill[c], 1)] = (int32_t)t;
    }
}

// _barycentric (solution.py:122-130) operation by operation; l3 = (1.0 - l1) - l2
__device__ __forceinline__ void barycentric_rn(double ax, double ay, double bx, double by, double cx, double cy,
                                               double x, double y, double& l1, double& l2, double& l3) {
  const double det = __dadd_rn(__dmul_rn(__dsub_rn(by, cy), __dsub_rn(ax, cx)),
                               __dmul_rn(__dsub_rn(cx, bx), __dsub_rn(ay, cy)));
  const double dx = __dsub_rn(x, cx), dy = __dsub_rn(y, cy);
  l1 = __ddiv_rn(__dadd_rn(__dmul_rn(__dsub_rn(by, cy), dx), __dmul_rn(__dsub_rn(cx, bx), dy)), det);
  l2 = __ddiv_rn(__dadd_rn(__dmul_rn(__dsub_rn(cy, ay), dx), __dmul_rn(__dsub_rn(ax, cx), dy)), det);
  l3 = __dsub_rn(__dsub_rn(1.0, l1), l2);
}

__global__ void tri_locate_kernel(int64_t q, const double* __restrict__ xy, const double* __restrict__ sites,
                                  const int64_t* __restrict__ el, double x0, double y0, double x1, double y1,
                                  double inv_cell, int ncx, int ncy, const int32_t* __restrict__ start,
                                  const int32_t* __restrict__ cell_tris, int64_t* __restrict__ tri,
                                  double* __restrict__ bary) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= q) return;
  const double x = xy[2 * p], y = xy[2 * p + 1];
  int64_t best = -1;
  double bmin = 0.0, b1 = 0.0, b2 = 0.0, b3 = 0.0;
  if (x >= x0 && x <= x1 && y >= y0 && y <= y1) {  // (false for NaN)
    const int64_t c = (int64_t)grid_coord(y, y0, inv_cell, ncy) * ncx + grid_coord(x, x0, inv_cell, ncx);
    for (int32_t k = start[c], kend = start[c + 1]; k < kend; k++) {
      const int64_t t = cell_tris[k];
      const int64_t ia = el[3 * t], ib = el[3 * t + 1], ic = el[3 * t + 2];
      double l1, l2, l3;
      barycentric_rn(sites[2 * ia], sites[2 * ia + 1], sites[2 * ib], sites[2 * ib + 1], sites[2 * ic],
                     sites[2 * ic + 1], x, y, l1, l2, l3);
      if (!(isfinite(l1) && isfinite(l2) && isfinite(l3))) continue;
      const double mn = fmin(l1, fmin(l2, l3));
      // total order: larger minimum first, then the lower triangle index (independent of the list order)
      if (best < 0 || mn > bmin || (mn == bmin && t < best)) {
        best = t;
        bmin = mn;
        b1 = l1;
        b2 = l2;
        b3 = l3;
      }
    }
  }
  if (best < 0 || !(bmin >= -1e-12)) {
    best = -1;
    b1 = b2 = b3 = 0.0;
  }
  tri[p] = best;
  bary[3 * p] = b1;
  bary[3 * p + 1] = b2;
  bary[3 * p + 2] = b3;
}

// out[s, p, :] = (sum of the three weighted corner values in np.einsum's order) * scale, zero where the point is
// outside, masked out, or any component is not finite.
template <int NCOMP>
__global__ void tri_interpolate_kernel(int64_t q, const int64_t* __restrict__ tri, const double* __restrict__ bary,
                                       const int64_t* __restrict__ el, int64_t nsets, int64_t n,
                                       const double* __restrict__ values, const uint8_t* __restrict__ mask,
                                       double scale, double* __restrict__ out) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= q) return;
  const int64_t s0 = (int64_t)blockIdx.y * kInterpSets;
  const int64_t s1 = s0 + kInterpSets < nsets ? s0 + kInterpSets : nsets;
  const int64_t t = tri[p];
  const bool live = t >= 0 && (mask == nullptr || mask[p] != 0);
  int64_t v0 = 0, v1 = 0, v2 = 0;
  double w0 = 0.0, w1 = 0.0, w2 = 0.0;
  if (live) {
    v0 = el[3 * t];
    v1 = el[3 * t + 1];
    v2 = el[3 * t + 2];
    w0 = bary[3 * p];
    w1 = bary[3 * p + 1];
    w2 = bary[3 * p + 2];
  }
  for (int64_t s = s0; s < s1; s++) {
    double r[NCOMP];
    bool finite = true;
    const double* vs = values + s * n * NCOMP;
#pragma unroll
    for (int k = 0; k < NCOMP; k++) {
      r[k] = 0.0;
      if (live) {
        const double t0 = __dmul_rn(w0, vs[v0 * NCOMP + k]);
        const double t1 = __dmul_rn(w1, vs[v1 * NCOMP + k]);
        const double t2 = __dmul_rn(w2, vs[v2 * NCOMP + k]);
        // np.einsum("qk,qk...->q...") adds (t0 + t2) + t1 for scalar values and (t0 + t1) + t2 per component
        // for 2-vectors; its accumulator starts at +0.0, which turns a -0.0 sum into +0.0
        const double sum = NCOMP == 1 ? __dadd_rn(__dadd_rn(t0, t2), t1) : __dadd_rn(__dadd_rn(t0, t1), t2);
        r[k] = __dadd_rn(0.0, sum);
        finite = finite && isfinite(r[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < NCOMP; k++) out[(s * q + p) * NCOMP + k] = finite ? __dmul_rn(r[k], scale) : 0.0;
  }
}

// geometry.points_in_polygon (geometry.py:77-103): even-odd rule, edges half-open in y, crossing abscissa
// dx * (y - y1) / dy + x1 rounded in that order.  op 0: inside = test; 1: inside |= test; 2: inside &= !test.
__global__ void __launch_bounds__(kPolyTile) points_in_polygon_kernel(int64_t m, const double* __restrict__ pts,
                                                                      int64_t nv, const double* __restrict__ poly,
                                                                      int op, uint8_t* __restrict__ inside) {
  __shared__ double sx[kPolyTile + 1], sy[kPolyTile + 1];
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double x = 0.0, y = 0.0;
  if (i < m) {
    x = pts[2 * i];
    y = pts[2 * i + 1];
  }
  int crossings = 0;
  for (int64_t base = 0; base < nv; base += kPolyTile) {
    const int64_t cnt = nv - base < kPolyTile ? nv - base : kPolyTile;
    __syncthreads();
    for (int64_t k = threadIdx.x; k <= cnt; k += blockDim.x) {  // cnt + 1 vertices: the tile's edges
      const int64_t v = base + k == nv ? 0 : base + k;
      sx[k] = poly[2 * v];
      sy[k] = poly[2 * v + 1];
    }
    __syncthreads();
    for (int k = 0; k < cnt; k++) {
      const double x1 = sx[k], y1 = sy[k], x2 = sx[k + 1], y2 = sy[k + 1];
      if ((y1 > y) != (y2 > y)) {
        const double xint =
            __dadd_rn(__ddiv_rn(__dmul_rn(__dsub_rn(x2, x1), __dsub_rn(y, y1)), __dsub_rn(y2, y1)), x1);
        crossings += x < xint ? 1 : 0;
      }
    }
  }
  if (i >= m) return;
  const bool in = crossings & 1;
  if (op == 0) inside[i] = in ? 1 : 0;
  else if (op == 1) inside[i] = (inside[i] || in) ? 1 : 0;
  else inside[i] = (inside[i] && !in) ? 1 : 0;
}

}  // namespace scb

using namespace scb;

// workspace layout (int32): range[4 ntri] (int4 per triangle) | start[ncells + 1] | fill[ncells]
extern "C" int64_t scb_tri_grid_workspace_elems(int64_t ntri, int64_t ncells) {
  return 4 * ntri + (ncells + 1) + ncells;
}

extern "C" int scb_tri_grid_count(int64_t ntri, const double* sites, const int64_t* elements, double x0, double y0,
                                  double cell, int32_t ncx, int32_t ncy, int32_t* workspace, scb_stream_t stream) {
  SCB_CHECK_ARG(ntri >= 0 && ntri < ((int64_t)1 << 31), "bad number of triangles");
  SCB_CHECK_ARG(cell > 0.0 && ncx > 0 && ncy > 0 && (int64_t)ncx * ncy < ((int64_t)1 << 30), "bad cell grid");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t ncells = (int64_t)ncx * ncy;
  int4* range = (int4*)workspace;
  int32_t* start = workspace + 4 * ntri;
  SCB_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "workspace must be 16-byte aligned");
  SCB_CUDA(cudaMemsetAsync(start, 0, (2 * ncells + 1) * sizeof(int32_t), s));  // start + fill
  if (ntri > 0) {
    tri_grid_count_kernel<<<(unsigned)ceil_div(ntri, 256), 256, 0, s>>>(ntri, sites, elements, x0, y0, 1.0 / cell,
                                                                       ncx, ncy, range, start);
      SCB_LAUNCH_CHECK();
  }
  return launch_cell_scan(start, ncells, s);
  return SCB_OK;
}

extern "C" int scb_tri_grid_fill(int64_t ntri, int32_t ncx, int32_t ncy, int32_t* workspace, int32_t* cell_tris,
                                 scb_stream_t stream) {
  SCB_CHECK_ARG(ntri >= 0 && ncx > 0 && ncy > 0, "bad sizes");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t ncells = (int64_t)ncx * ncy;
  const int4* range = (const int4*)workspace;
  int32_t* start = workspace + 4 * ntri;
  int32_t* fill = start + ncells + 1;
  if (ntri > 0) {
    tri_grid_scatter_kernel<<<(unsigned)ceil_div(ntri, 256), 256, 0, s>>>(ntri, ncx, range, start, fill, cell_tris);
    SCB_LAUNCH_CHECK();
  }
  return launch_cell_sort(ncells, start, cell_tris, s);
}

extern "C" int scb_tri_locate(int64_t q, const double* xy, const double* sites, const int64_t* elements, double x0,
                              double y0, double x1, double y1, double cell, int32_t ncx, int32_t ncy,
                              const int32_t* start, const int32_t* cell_tris, int64_t* tri, double* bary,
                              scb_stream_t stream) {
  SCB_CHECK_ARG(q >= 0, "negative size");
  SCB_CHECK_ARG(cell > 0.0 && ncx > 0 && ncy > 0, "bad cell grid");
  if (q == 0) return SCB_OK;
  tri_locate_kernel<<<(unsigned)ceil_div(q, 128), 128, 0, (cudaStream_t)stream>>>(
      q, xy, sites, elements, x0, y0, x1, y1, 1.0 / cell, ncx, ncy, start, cell_tris, tri, bary);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

extern "C" int scb_tri_interpolate(int64_t q, const int64_t* tri, const double* bary, const int64_t* elements,
                                   int64_t nsets, int ncomp, int64_t n, const double* values, const uint8_t* mask,
                                   double scale, double* out, scb_stream_t stream) {
  SCB_CHECK_ARG(q >= 0 && nsets >= 0 && n >= 0, "negative size");
  SCB_CHECK_ARG(ncomp == 1 || ncomp == 2, "ncomp must be 1 or 2");
  if (q == 0 || nsets == 0) return SCB_OK;
  SCB_CHECK_ARG(ceil_div(nsets, kInterpSets) <= 65535, "too many value sets");
  const dim3 grid((unsigned)ceil_div(q, 128), (unsigned)ceil_div(nsets, kInterpSets));
  cudaStream_t s = (cudaStream_t)stream;
  if (ncomp == 1)
    tri_interpolate_kernel<1><<<grid, 128, 0, s>>>(q, tri, bary, elements, nsets, n, values, mask, scale, out);
  else
    tri_interpolate_kernel<2><<<grid, 128, 0, s>>>(q, tri, bary, elements, nsets, n, values, mask, scale, out);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

extern "C" int scb_points_in_polygon(int64_t m, const double* points, int64_t nv, const double* vertices, int op,
                                     uint8_t* inside, scb_stream_t stream) {
  SCB_CHECK_ARG(m >= 0 && nv >= 0, "negative size");
  SCB_CHECK_ARG(op >= 0 && op <= 2, "op must be 0 (set), 1 (or) or 2 (and not)");
  if (m == 0) return SCB_OK;
  points_in_polygon_kernel<<<(unsigned)ceil_div(m, kPolyTile), kPolyTile, 0, (cudaStream_t)stream>>>(
      m, points, nv, vertices, op, inside);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}
