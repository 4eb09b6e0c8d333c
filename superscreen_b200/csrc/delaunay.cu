// Mesh generation on the device (SURVEY.md section 8f.4): the replacement of the reference's
// meshpy / Triangle call in device/utils.py:17-136 (generate_mesh) for the quasi-uniform point sets
// this path meshes with.
//
//   scb_lattice_points   jittered hexagonal point lattice clipped to a polygonal region (even-odd
//                        rule over any number of rings) and kept clear of the fixed (polygon) points;
//   scb_points_in_rings  even-odd point-in-region test (triangle centroids: cut the triangulation of
//                        the convex hull down to the region);
//   scb_delaunay         Delaunay triangulation of a point set: ONE THREAD PER POINT clips that point's
//                        Voronoi cell against its neighbours, which it finds ring by ring in a uniform
//                        cell grid (security-radius termination: the cell is final once every
//                        unvisited point is farther away than twice the farthest cell vertex).  The
//                        Delaunay triangles are the triples (p, a, b) of consecutive Voronoi
//                        neighbours; each triangle is emitted by its smallest vertex, counter-clockwise,
//                        starting the walk around p at p's smallest neighbour, and the per-point lists
//                        are compacted in point order -- the triangle array is a deterministic
//                        function of the point array (no atomics decide any index).
//
// Points in general position (no four co-circular points) are assumed; the generated lattices are
// jittered and the caller validates the result (manifold check of scb_mesh_analyze + Euler count)
// and re-seeds on failure.  All arithmetic is done relative to the point that owns the cell.
#include "scb_common.cuh"

namespace scb {

constexpr int kMaxCellVerts = 48;  // Voronoi cell vertices kept per point (degree + bounding box)
constexpr int kMaxEmit = 24;       // triangles a point can emit as their smallest vertex

__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double u01(uint64_t z) { return (double)(z >> 11) * (1.0 / 9007199254740992.0); }

// even-odd rule over all rings; ring r = vertices ring_ptr[r] .. ring_ptr[r + 1] - 1 (closed implicitly)
__device__ __forceinline__ bool in_rings(double x, double y, int nrings, const int64_t* __restrict__ ring_ptr,
                                         const double* __restrict__ rv) {
  bool inside = false;
  for (int r = 0; r < nrings; r++) {
    const int64_t lo = ring_ptr[r], hi = ring_ptr[r + 1];
    double x0 = rv[2 * (hi - 1)], y0 = rv[2 * (hi - 1) + 1];
    for (int64_t k = lo; k < hi; k++) {
      const double x1 = rv[2 * k], y1 = rv[2 * k + 1];
      if ((y0 > y) != (y1 > y)) {
        const double xc = x0 + (y - y0) * (x1 - x0) / (y1 - y0);
        if (x < xc) inside = !inside;
      }
      x0 = x1;
      y0 = y1;
    }
  }
  return inside;
}

__global__ void points_in_rings_kernel(int64_t m, const double* __restrict__ pts, int nrings,
                                       const int64_t* __restrict__ ring_ptr, const double* __restrict__ rv,
                                       uint8_t* __restrict__ inside) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < m) inside[i] = in_rings(pts[2 * i], pts[2 * i + 1], nrings, ring_ptr, rv) ? 1 : 0;
}

// lattice point (ix, iy): rows are h sqrt(3)/2 apart, odd rows shifted by h/2, jitter uniform in
// [-jitter h, jitter h]^2 from a counter-based generator (seed, point index): reproducible anywhere
__global__ void lattice_kernel(int64_t nx, int64_t ny, double x0, double y0, double h, double jitter, uint64_t seed,
                               int nrings, const int64_t* __restrict__ ring_ptr, const double* __restrict__ rv,
                               int64_t nfixed, const double* __restrict__ fixed, double min_dist,
                               double* __restrict__ pts, uint8_t* __restrict__ keep) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nx * ny) return;
  const int64_t iy = i / nx, ix = i - iy * nx;
  const uint64_t r0 = splitmix64(seed * 0x632BE59BD9B4E019ull + 2 * (uint64_t)i);
  const uint64_t r1 = splitmix64(seed * 0x632BE59BD9B4E019ull + 2 * (uint64_t)i + 1);
  const double x = x0 + ((double)ix + 0.5 * (double)(iy & 1)) * h + jitter * h * (2.0 * u01(r0) - 1.0);
  const double y = y0 + (double)iy * (h * 0.8660254037844386) + jitter * h * (2.0 * u01(r1) - 1.0);
  pts[2 * i] = x;
  pts[2 * i + 1] = y;
  bool ok = in_rings(x, y, nrings, ring_ptr, rv);
  if (ok) {
    const double d2min = min_dist * min_dist;
    for (int64_t k = 0; k < nfixed && ok; k++) {
      const double dx = fixed[2 * k] - x, dy = fixed[2 * k + 1] - y;
      ok = fma(dx, dx, dy * dy) > d2min;
    }
  }
  keep[i] = ok ? 1 : 0;
}

// ---- uniform grid ----
__device__ __forceinline__ int cell_coord(double v, double v0, double inv_cell, int nc) {
  int c = (int)floor((v - v0) * inv_cell);
  return c < 0 ? 0 : (c >= nc ? nc - 1 : c);
}
__global__ void cell_count_kernel(int64_t n, const double* __restrict__ pts, double x0, double y0, double inv_cell,
                                  int ncx, int ncy, int32_t* __restrict__ cell_of, int32_t* __restrict__ count) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = cell_coord(pts[2 * i + 1], y0, inv_cell, ncy) * ncx + cell_coord(pts[2 * i], x0, inv_cell, ncx);
  cell_of[i] = c;
  atomicAdd(&count[c], 1);
}
// exclusive scan of `count` (length m) by ONE CTA of 1024 threads; data[m] receives the total
__global__ void scan_kernel(int32_t* __restrict__ data, int64_t m) {
  __shared__ int32_t wsum[32];
  __shared__ int32_t carry_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int64_t base = 0; base < m; base += 1024) {
    const int64_t i = base + tid;
    const int32_t v = i < m ? data[i] : 0;
    int32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int32_t w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int32_t y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      wsum[lane] = w;
    }
    __syncthreads();
    const int32_t carry = carry_s;
    const int32_t excl = carry + (warp ? wsum[warp - 1] : 0) + x - v;
    if (i < m) data[i] = excl;
    __syncthreads();
    if (tid == 1023) carry_s = carry + wsum[31];
    __syncthreads();
  }
  if (tid == 0) data[m] = carry_s;
}
__global__ void cell_scatter_kernel(int64_t n, const int32_t* __restrict__ cell_of, const int32_t* __restrict__ start,
                                    int32_t* __restrict__ fill, int32_t* __restrict__ order) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = cell_of[i];
  order[start[c] + atomicAdd(&fill[c], 1)] = (int32_t)i;
}
// the scatter above is not ordered inside a cell: sort every cell's (few) points by index, so that the
// clipping order -- and with it every rounding -- is the same in every run
__global__ void cell_sort_kernel(int64_t ncells, const int32_t* __restrict__ start, int32_t* __restrict__ order) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= ncells) return;
  const int lo = start[c], hi = start[c + 1];
  for (int a = lo + 1; a < hi; a++) {
    const int32_t v = order[a];
    int b = a - 1;
    while (b >= lo && order[b] > v) {
      order[b + 1] = order[b];
      b--;
    }
    order[b + 1] = v;
  }
}

// ---- Voronoi cell of one point by half-plane clipping ----
struct Cell {
  double vx[kMaxCellVerts], vy[kMaxCellVerts];  // vertices relative to the owner, counter-clockwise
  int32_t nb[kMaxCellVerts];                    // neighbour whose bisector carries edge k -> k + 1 (-1: box)
  int nv;
  double r2max;  // largest squared vertex distance from the owner
};

// clips the cell by the bisector of the owner (origin) and q = (qx, qy): keeps {x : x.q <= |q|^2 / 2}
__device__ __forceinline__ bool clip_cell(Cell& c, double qx, double qy, int32_t qid) {
  const double half = 0.5 * fma(qx, qx, qy * qy);
  // A vertex counts as cut off only if it lies beyond the bisector by more than 1e-12 |q| (relative to
  // the distance of q): bisectors that merely graze a vertex within rounding -- many co-circular points
  // around an empty circle, e.g. the polygon points of a circular hole -- must not shave slivers off it.
  const double tol = 2e-12 * half;
  double s[kMaxCellVerts];
  bool any_out = false;
  for (int k = 0; k < c.nv; k++) {
    s[k] = fma(c.vx[k], qx, c.vy[k] * qy) - half - tol;
    any_out |= s[k] > 0.0;
  }
  if (!any_out) return true;
  // first vertex that is outside while its predecessor is inside
  int first_out = -1;
  for (int k = 0; k < c.nv; k++) {
    const int prev = k == 0 ? c.nv - 1 : k - 1;
    if (s[k] > 0.0 && s[prev] <= 0.0) {
      first_out = k;
      break;
    }
  }
  if (first_out < 0) return true;  // every vertex outside: cannot happen for a cell that contains its owner
  // run of outside vertices first_out .. last_out (cyclic)
  int nout = 0;
  while (nout < c.nv && s[(first_out + nout) % c.nv] > 0.0) nout++;
  const int last_out = (first_out + nout - 1) % c.nv;
  const int before = first_out == 0 ? c.nv - 1 : first_out - 1;  // inside
  const int after = (last_out + 1) % c.nv;                       // inside
  // entry point on edge before -> first_out (keeps that edge's label), exit point on edge last_out -> after
  const double ta = s[before] / (s[before] - s[first_out]);
  const double ax = fma(ta, c.vx[first_out] - c.vx[before], c.vx[before]);
  const double ay = fma(ta, c.vy[first_out] - c.vy[before], c.vy[before]);
  const double tb = s[last_out] / (s[last_out] - s[after]);
  const double bx = fma(tb, c.vx[after] - c.vx[last_out], c.vx[last_out]);
  const double by = fma(tb, c.vy[after] - c.vy[last_out], c.vy[last_out]);
  const int32_t exit_label = c.nb[last_out];  // the edge last_out -> after survives from b on
  const int new_nv = c.nv - nout + 2;
  if (new_nv > kMaxCellVerts) return false;
  // rebuild: [a (label q), b (label of the exit edge)] followed by after .. before
  double tx[kMaxCellVerts], ty[kMaxCellVerts];
  int32_t tn[kMaxCellVerts];
  int m = 0;
  tx[m] = ax; ty[m] = ay; tn[m] = qid; m++;
  tx[m] = bx; ty[m] = by; tn[m] = exit_label; m++;
  for (int k = after; k != first_out; k = (k + 1) % c.nv) {
    tx[m] = c.vx[k]; ty[m] = c.vy[k]; tn[m] = c.nb[k]; m++;
  }
  // (the label of vertex `before` is the label of edge before -> first_out, which now ends at a: unchanged)
  c.nv = m;
  double r2 = 0.0;
  for (int k = 0; k < m; k++) {
    c.vx[k] = tx[k]; c.vy[k] = ty[k]; c.nb[k] = tn[k];
    const double d2 = fma(tx[k], tx[k], ty[k] * ty[k]);
    r2 = d2 > r2 ? d2 : r2;
  }
  c.r2max = r2;
  return true;
}

// status bits per point
enum : int32_t { DT_CELL_OVERFLOW = 1, DT_EMIT_OVERFLOW = 2 };

__global__ void __launch_bounds__(128)
voronoi_kernel(int64_t n, const double* __restrict__ pts, double x0, double y0, double cell, int ncx, int ncy,
               const int32_t* __restrict__ start, const int32_t* __restrict__ order, double big,
               int32_t* __restrict__ emit /*[n][kMaxEmit][2]*/, int32_t* __restrict__ nemit /*[n + 1]*/,
               int32_t* __restrict__ status) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double px = pts[2 * i], py = pts[2 * i + 1];
  const double inv_cell = 1.0 / cell;
  const int cx = cell_coord(px, x0, inv_cell, ncx), cy = cell_coord(py, y0, inv_cell, ncy);
  Cell c;
  c.nv = 4;
  c.vx[0] = -big; c.vy[0] = -big; c.nb[0] = -1;
  c.vx[1] = big;  c.vy[1] = -big; c.nb[1] = -1;
  c.vx[2] = big;  c.vy[2] = big;  c.nb[2] = -1;
  c.vx[3] = -big; c.vy[3] = big;  c.nb[3] = -1;
  c.r2max = 2.0 * big * big;
  int32_t st = 0;
  // clips the cell against every point of grid cell (cx + dx, cy + dy) that can still reach it
  auto visit = [&](int dx, int dy) {
    const int xx = cx + dx, yy = cy + dy;
    if (xx < 0 || xx >= ncx || yy < 0 || yy >= ncy) return;
    // distance from the owner to the grid cell's rectangle; a point q clips only if |q| < 2 max |v|
    const double gx = dx == 0 ? 0.0 : (dx > 0 ? x0 + xx * cell - px : px - (x0 + (xx + 1) * cell));
    const double gy = dy == 0 ? 0.0 : (dy > 0 ? y0 + yy * cell - py : py - (y0 + (yy + 1) * cell));
    const double gxx = gx > 0.0 ? gx : 0.0, gyy = gy > 0.0 ? gy : 0.0;
    if (fma(gxx, gxx, gyy * gyy) >= 4.0 * c.r2max) return;
    const int cc = yy * ncx + xx;
    for (int a = start[cc]; a < start[cc + 1]; a++) {
      const int32_t j = order[a];
      if (j == i) continue;
      const double qx = pts[2 * j] - px, qy = pts[2 * j + 1] - py;
      if (fma(qx, qx, qy * qy) >= 4.0 * c.r2max) continue;
      if (!clip_cell(c, qx, qy, j)) st |= DT_CELL_OVERFLOW;
    }
  };
  const int max_ring = ncx > ncy ? ncx : ncy;
  for (int ring = 0; ring <= max_ring; ring++) {
    // every unvisited point is at least (ring - 1) cell widths away: stop at the security radius
    if (ring >= 2) {
      const double reach = (double)(ring - 1) * cell;
      if (reach * reach >= 4.0 * c.r2max) break;
    }
    if (ring == 0) {
      visit(0, 0);
      continue;
    }
    for (int dx = -ring; dx <= ring; dx++) {  // bottom and top rows of the ring
      visit(dx, -ring);
      visit(dx, ring);
    }
    for (int dy = -ring + 1; dy <= ring - 1; dy++) {  // left and right columns
      visit(-ring, dy);
      visit(ring, dy);
    }
  }
  // Delaunay triangles (i, a, b): consecutive Voronoi neighbours a = nb[k], b = nb[k + 1] around the
  // shared Voronoi vertex k + 1; emitted by the smallest vertex, walk started at the smallest neighbour
  int kstart = 0;
  int32_t best = 0x7fffffff;
  for (int k = 0; k < c.nv; k++)
    if (c.nb[k] >= 0 && c.nb[k] < best) {
      best = c.nb[k];
      kstart = k;
    }
  int cnt = 0;
  for (int t = 0; t < c.nv; t++) {
    const int k = (kstart + t) % c.nv, k1 = (k + 1) % c.nv;
    const int32_t a = c.nb[k], b = c.nb[k1];
    if (a < 0 || b < 0 || a == b) continue;
    if (i < a && i < b) {
      if (cnt < kMaxEmit) {
        emit[(i * kMaxEmit + cnt) * 2] = a;
        emit[(i * kMaxEmit + cnt) * 2 + 1] = b;
        cnt++;
      } else {
        st |= DT_EMIT_OVERFLOW;
      }
    }
  }
  nemit[i] = cnt;
  status[i] = st;
}

__global__ void emit_compact_kernel(int64_t n, const int32_t* __restrict__ emit, const int32_t* __restrict__ offset,
                                    int64_t max_tri, int64_t* __restrict__ tri) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int lo = offset[i], hi = offset[i + 1];
  for (int t = lo; t < hi; t++) {
    if (t >= max_tri) break;
    tri[3 * (int64_t)t] = i;
    tri[3 * (int64_t)t + 1] = emit[(i * kMaxEmit + (t - lo)) * 2];
    tri[3 * (int64_t)t + 2] = emit[(i * kMaxEmit + (t - lo)) * 2 + 1];
  }
}

__global__ void delaunay_info_kernel(int64_t n, const int32_t* __restrict__ offset, const int32_t* __restrict__ status,
                                     int64_t* __restrict__ info) {
  // info[0] = triangles, info[1] = points whose cell overflowed, info[2] = points whose emit list overflowed
  __shared__ int s1, s2;
  if (threadIdx.x == 0) s1 = s2 = 0;
  __syncthreads();
  int a = 0, b = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    a += (status[i] & DT_CELL_OVERFLOW) ? 1 : 0;
    b += (status[i] & DT_EMIT_OVERFLOW) ? 1 : 0;
  }
  atomicAdd(&s1, a);
  atomicAdd(&s2, b);
  __syncthreads();
  if (threadIdx.x == 0) {
    info[0] = offset[n];
    info[1] = s1;
    info[2] = s2;
    info[3] = 0;
  }
}

// the scan and the per-cell sort for other cell grids (interp.cu's triangle grid)
int launch_cell_scan(int32_t* count, int64_t ncells, cudaStream_t s) {
  scan_kernel<<<1, 1024, 0, s>>>(count, ncells);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}
int launch_cell_sort(int64_t ncells, const int32_t* start, int32_t* order, cudaStream_t s) {
  cell_sort_kernel<<<(unsigned)ceil_div(ncells, 256), 256, 0, s>>>(ncells, start, order);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

}  // namespace scb

using namespace scb;

extern "C" int scb_points_in_rings(int64_t m, const double* points, int nrings, const int64_t* ring_ptr,
                                   const double* ring_vertices, uint8_t* inside, scb_stream_t stream) {
  SCB_CHECK_ARG(m >= 0 && nrings >= 0, "negative size");
  if (m == 0) return SCB_OK;
  cudaStream_t s = (cudaStream_t)stream;
  points_in_rings_kernel<<<(unsigned)ceil_div(m, 256), 256, 0, s>>>(m, points, nrings, ring_ptr, ring_vertices, inside);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

extern "C" int scb_lattice_points(int64_t nx, int64_t ny, double x0, double y0, double h, double jitter,
                                  uint64_t seed, int nrings, const int64_t* ring_ptr, const double* ring_vertices,
                                  int64_t nfixed, const double* fixed, double min_dist, double* points,
                                  uint8_t* keep, scb_stream_t stream) {
  SCB_CHECK_ARG(nx > 0 && ny > 0 && h > 0.0, "empty lattice");
  SCB_CHECK_ARG(jitter >= 0.0 && jitter < 0.5, "jitter must be in [0, 0.5)");
  cudaStream_t s = (cudaStream_t)stream;
  lattice_kernel<<<(unsigned)ceil_div(nx * ny, 256), 256, 0, s>>>(nx, ny, x0, y0, h, jitter, seed, nrings, ring_ptr,
                                                                   ring_vertices, nfixed, fixed, min_dist, points, keep);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

extern "C" int scb_delaunay(int64_t n, const double* points, double x0, double y0, double cell, int32_t ncx,
                            int32_t ncy, int64_t max_triangles, int64_t* triangles, int64_t* info,
                            scb_stream_t stream) {
  SCB_CHECK_ARG(n >= 3, "at least three points are needed");
  SCB_CHECK_ARG(n < (int64_t)1 << 30, "too many points");
  SCB_CHECK_ARG(cell > 0.0 && ncx > 0 && ncy > 0 && (int64_t)ncx * ncy < (int64_t)1 << 30, "bad cell grid");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t ncells = (int64_t)ncx * ncy;
  // scratch: cell_of[n] start[ncells + 1] fill[ncells] order[n] nemit[n + 1] status[n] emit[n][kMaxEmit][2]
  const size_t words = (size_t)n + (ncells + 1) + ncells + n + (n + 1) + n + (size_t)n * kMaxEmit * 2;
  int32_t* scratch = nullptr;
  SCB_CUDA(cudaMallocAsync(&scratch, words * sizeof(int32_t), s));
  int32_t* cell_of = scratch;
  int32_t* start = cell_of + n;
  int32_t* fill = start + (ncells + 1);
  int32_t* order = fill + ncells;
  int32_t* nemit = order + n;
  int32_t* status = nemit + (n + 1);
  int32_t* emit = status + n;
  SCB_CUDA(cudaMemsetAsync(start, 0, (2 * ncells + 1) * sizeof(int32_t), s));  // start + fill
  const unsigned gn = (unsigned)ceil_div(n, 256);
  cell_count_kernel<<<gn, 256, 0, s>>>(n, points, x0, y0, 1.0 / cell, ncx, ncy, cell_of, start);
  SCB_LAUNCH_CHECK();
  scan_kernel<<<1, 1024, 0, s>>>(start, ncells);
  SCB_LAUNCH_CHECK();
  cell_scatter_kernel<<<gn, 256, 0, s>>>(n, cell_of, start, fill, order);
  SCB_LAUNCH_CHECK();
  cell_sort_kernel<<<(unsigned)ceil_div(ncells, 256), 256, 0, s>>>(ncells, start, order);
  SCB_LAUNCH_CHECK();
  // bounding box of the (unbounded) hull cells: 1e4 domain extents.  A Delaunay triangle whose circumradius
  // exceeds it -- three all but collinear hull points -- is not produced; such slivers are useless to the
  // FEM operators and the host drops near-degenerate triangles anyway.
  const double big = 1.0e4 * cell * (double)((ncx > ncy ? ncx : ncy) + 2);
  voronoi_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, s>>>(n, points, x0, y0, cell, ncx, ncy, start, order, big, emit,
                                                            nemit, status);
  SCB_LAUNCH_CHECK();
  scan_kernel<<<1, 1024, 0, s>>>(nemit, n);
  SCB_LAUNCH_CHECK();
  emit_compact_kernel<<<gn, 256, 0, s>>>(n, emit, nemit, max_triangles, triangles);
  SCB_LAUNCH_CHECK();
  delaunay_info_kernel<<<1, 256, 0, s>>>(n, nemit, status, info);
  SCB_LAUNCH_CHECK();
  SCB_CUDA(cudaFreeAsync(scratch, s));
  return SCB_OK;
}
