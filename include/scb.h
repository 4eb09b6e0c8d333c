/*
 * scb.h -- C ABI of libsc_b200.so: the B200 (sm_100a) implementation of SuperScreen's
 * solve hot path.
 *
 * The reference (loganbvh/superscreen 0.13.0) is pure Python and has no FFI of its own;
 * its seam for this path is the set of module-level callables listed in SURVEY.md 8(a).
 * Each entry point below names the reference callable (file:line under
 * /root/reference/superscreen/) whose arithmetic it replaces.  INTEGRATION.md shows the
 * ctypes binding a SuperScreen maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *  - matrices are row-major (C order), fp64; index arrays are int64 where the reference
 *    exposes int64 (elements, index sets, edges) and int32 for CSR indptr/indices
 *    (scipy's native index dtype);
 *  - one call == stream-ordered work on `stream` (a cudaStream_t passed as void*); no call
 *    synchronises the device unless documented;
 *  - return value 0 on success, negative on error (scb_last_error() gives the message);
 *    no exceptions cross the boundary;
 *  - there is no CPU fallback anywhere in this library.
 */
#ifndef SCB_H
#define SCB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* scb_stream_t;

#define SCB_OK 0
#define SCB_ERR_INVALID (-1)
#define SCB_ERR_CUDA (-2)
#define SCB_ERR_SINGULAR (-3)

#define SCB_LU_BLOCK 128 /* LU panel width; LU workspaces are padded to a multiple of it */

int scb_version(void);
const char* scb_last_error(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
int64_t scb_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Mesh topology + FEM operators  (K4-K7, rows a4-a8)
 *   device/utils.py:139-152 get_edges, :230-273 triangle_areas/vertex_areas
 *   device/mesh.py:157-170 find_boundary_indices, :400-432 C_vector
 *   device/edge_mesh.py:38-63, fem.py:70-121 adjacency / directed-edge map
 *   fem.py:124-296 weights + laplace_operator, :299-402 gradient_triangles/_vertices
 * ------------------------------------------------------------------------------------ */

/* int32 workspace elements needed by scb_mesh_analyze/scb_mesh_build for n vertices, m triangles */
int64_t scb_mesh_workspace_elems(int64_t n, int64_t m);

/* Phase 1: vertex stars, neighbour sets, edge / boundary counts.
 * counts (device, int64[4]) <- { nnz of adjacency (=2E), E, #boundary vertices, #boundary edges }.
 * flags  (device, int32[1]) <- nonzero if the mesh is not a consistently oriented manifold
 *                              (an undirected edge shared by >2 triangles or a duplicated
 *                              directed edge). */
int scb_mesh_analyze(int64_t n, int64_t m, const int64_t* elements, int32_t* workspace,
                     int64_t* counts, int32_t* flags, scb_stream_t stream);

typedef struct scb_mesh_out {
  /* per triangle / vertex floats */
  double* triangle_areas;   /* [m]   device/utils.py:230-248 */
  double* vertex_areas;     /* [n]   device/utils.py:251-273 (sum over the star in triangle order) */
  double* centroids;        /* [m,2] device/mesh.py:144 */
  double* C;                /* [n]   device/mesh.py:400-432 */
  /* integer structures (bit-exact contract) */
  int32_t* adj_indptr;      /* [n+1] fem.py:70-98 (symmetric 0/1 adjacency, sorted rows) */
  int32_t* adj_indices;     /* [2E] */
  int64_t* edges;           /* [E,2] device/utils.py:149-151, i<j, lexicographic */
  uint8_t* edge_is_boundary;/* [E]   device/utils.py:152 */
  int64_t* boundary_indices;/* [nb]  device/mesh.py:167-170 ascending */
  int32_t* star_indptr;     /* [n+1] fem.py:101-121 in LIL (row) form: */
  int32_t* star_heads;      /* [3m]  head vertex j of directed edge i->j, ascending per row */
  int32_t* star_tris;       /* [3m]  triangle owning that edge */
  /* edge mesh floats, device/edge_mesh.py:49-56 */
  double* edge_centers;     /* [E,2] */
  double* edge_directions;  /* [E,2] */
  double* edge_lengths;     /* [E] */
  /* operators; laplacian / gradient_x / gradient_y share the pattern adjacency + I */
  int32_t* op_indptr;       /* [n+1] */
  int32_t* op_indices;      /* [2E+n] sorted per row */
  double* laplacian;        /* [2E+n] fem.py:259-296 */
  double* gradient_x;       /* [2E+n] fem.py:350-402 */
  double* gradient_y;       /* [2E+n] */
  int32_t* gtri_indices;    /* [3m]  fem.py:299-347, 3 sorted columns per row */
  double* gtri_x;           /* [3m] */
  double* gtri_y;           /* [3m] */
} scb_mesh_out;

/* weight_method: 0 = half_cotangent, 1 = uniform, 2 = inv_euclidean (fem.py:225-256).
 * Needs the workspace filled by scb_mesh_analyze for the same (n, m, elements). */
int scb_mesh_build(int64_t n, int64_t m, const double* sites, const int64_t* elements,
                   const int32_t* workspace, int weight_method, const scb_mesh_out* out,
                   scb_stream_t stream);

/* One Laplacian-smoothing sweep (Mesh.smooth, device/mesh.py:172-211): out_sites[i] = mean of the
 * neighbours of i (summed in the reference's order: neighbours > i ascending, then neighbours < i
 * ascending), boundary vertices copied unchanged.  adj_* and boundary_indices are the arrays
 * produced by scb_mesh_build for the same triangulation.  Not in place. */
int scb_mesh_smooth(int64_t n, const double* sites, const int32_t* adj_indptr, const int32_t* adj_indices,
                    int64_t n_boundary, const int64_t* boundary_indices, double* out_sites,
                    scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Mesh generation (row f4): the reference calls meshpy / Triangle in device/utils.py:17-136
 * (generate_mesh: points + boundary facets -> refined Delaunay mesh, refined until `min_points` /
 * `max_edge_length` hold).  Here: quasi-uniform point cloud + Delaunay triangulation on the device.
 * ------------------------------------------------------------------------------------ */

/* inside[i] (uint8) <- even-odd rule of points[i] = (x, y) against `nrings` closed rings (ring r =
 * ring_vertices[ring_ptr[r] .. ring_ptr[r + 1]), implicitly closed); outer boundary + holes of a region. */
int scb_points_in_rings(int64_t m, const double* points, int nrings, const int64_t* ring_ptr,
                        const double* ring_vertices, uint8_t* inside, scb_stream_t stream);

/* Jittered hexagonal lattice: point (ix, iy), ix < nx, iy < ny, at
 *   (x0 + (ix + (iy & 1) / 2) h, y0 + iy h sqrt(3) / 2) + jitter * h * U(-1, 1)^2
 * (counter-based generator of (seed, point index): the same on every device and launch geometry).
 * points <- f64[nx * ny, 2]; keep[i] (uint8) <- 1 iff the point lies in the region (even-odd over the
 * rings) and farther than min_dist from every one of the `nfixed` fixed (polygon) points. */
int scb_lattice_points(int64_t nx, int64_t ny, double x0, double y0, double h, double jitter, uint64_t seed,
                       int nrings, const int64_t* ring_ptr, const double* ring_vertices, int64_t nfixed,
                       const double* fixed, double min_dist, double* points, uint8_t* keep,
                       scb_stream_t stream);

/* Delaunay triangulation of n points in general position (what scipy.spatial.Delaunay / Triangle
 * compute for the same points).  (x0, y0, cell, ncx, ncy): a uniform grid that covers the points
 * (cell width of the order of the point spacing).  triangles <- int64[<= max_triangles, 3],
 * counter-clockwise, smallest vertex first, ordered by that vertex and then counter-clockwise around
 * it starting at its smallest neighbour: a deterministic function of the point array.
 * info (device, int64[4]) <- { number of triangles found (may exceed max_triangles: call again),
 *   points whose Voronoi cell overflowed, points whose triangle list overflowed, 0 }. */
int scb_delaunay(int64_t n, const double* points, double x0, double y0, double cell, int32_t ncx, int32_t ncy,
                 int64_t max_triangles, int64_t* triangles, int64_t* info, scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Point location and linear interpolation on a triangulation, polygon masks: the device stage of
 * Solution.interp_current_density / interp_field for a batch of solutions (solution.py:272-276,310-312,
 * which stand in for matplotlib's LinearTriInterpolator; geometry.points_in_polygon, geometry.py:77-103).
 * ------------------------------------------------------------------------------------ */

/* int32 workspace elements of scb_tri_grid_count / _fill for ntri triangles and ncells = ncx * ncy cells.
 * Layout: per-triangle cell ranges [4 ntri] | start [ncells + 1] | fill [ncells]; 16-byte aligned. */
int64_t scb_tri_grid_workspace_elems(int64_t ntri, int64_t ncells);

/* Uniform cell grid over the triangles of a mesh: cell (i, j) = [x0 + i cell, x0 + (i + 1) cell) x [y0 + j cell,
 * ...), i < ncx, j < ncy.  Every triangle is registered in every cell that its bounding box overlaps, the box
 * padded so that no point whose rounded barycentric coordinates (scb_tri_locate) are all >= -1e-12 falls outside
 * it; an all but degenerate triangle (longest edge^2 / |det| >= 2^-8 / eps) is registered in every cell, one with
 * det == 0 in none.  Two calls with a host read in between:
 *   scb_tri_grid_count  cell ranges and counts, exclusive scan: workspace[4 ntri + ncells] <- number of entries;
 *   scb_tri_grid_fill   cell_tris (int32 [entries]) <- the triangles of every cell, cell after cell (cell c:
 *                       cell_tris[start[c] .. start[c + 1]), start = workspace + 4 ntri), ascending per cell. */
int scb_tri_grid_count(int64_t ntri, const double* sites, const int64_t* elements, double x0, double y0, double cell,
                       int32_t ncx, int32_t ncy, int32_t* workspace, scb_stream_t stream);
int scb_tri_grid_fill(int64_t ntri, int32_t ncx, int32_t ncy, int32_t* workspace, int32_t* cell_tris,
                      scb_stream_t stream);

/* Containing triangle of q points xy [q, 2]: tri (int64 [q], -1 outside) and bary (f64 [q, 3]; 0 outside).  The
 * result is a function of the mesh and the grid bounds alone; the grid only prunes the candidates:
 *  - the barycentric coordinates are _barycentric's (solution.py:122-130) operation by operation, one rounding
 *    per operation, no FMA contraction, l3 = (1.0 - l1) - l2;
 *  - the point's triangle is the one, among all triangles, with the largest min(l1, l2, l3), ties to the lowest
 *    index; a triangle with a non-finite coordinate never wins;
 *  - the point is inside iff that maximum is >= -1e-12;
 *  - a point with a non-finite coordinate, or outside [x0, x1] x [y0, y1] (x1 = x0 + ncx cell and y1 = y0 +
 *    ncy cell as the caller computed them), is outside.
 * The order of the cell lists does not matter.  start / cell_tris are those of scb_tri_grid_fill. */
int scb_tri_locate(int64_t q, const double* xy, const double* sites, const int64_t* elements, double x0, double y0,
                   double x1, double y1, double cell, int32_t ncx, int32_t ncy, const int32_t* start,
                   const int32_t* cell_tris, int64_t* tri, double* bary, scb_stream_t stream);

/* Linear interpolation of nsets value sets at q located points: values [nsets, n, ncomp] (set-major, as a batch
 * is staged: one contiguous copy of the B arrays; the output is set-major too, so the writes of a warp are
 * contiguous), ncomp 1 or 2, out [nsets, q, ncomp]:
 *   out[s, p, c] = (0.0 + sum) * scale,  sum over the corners k of w_k v_k (one rounding per operation) in the
 *   order of np.einsum("qk,qk...->q...") (measured on the host): ncomp = 1: (w0 v0 + w2 v2) + w1 v1;
 *   ncomp = 2: (w0 v0 + w1 v1) + w2 v2; the 0.0 + of einsum's accumulator turns -0.0 into +0.0.
 * out is 0 where tri < 0, where mask (uint8 [q], may be NULL) is 0, and for every component of a point whose
 * components are not all finite. */
int scb_tri_interpolate(int64_t q, const int64_t* tri, const double* bary, const int64_t* elements, int64_t nsets,
                        int ncomp, int64_t n, const double* values, const uint8_t* mask, double scale, double* out,
                        scb_stream_t stream);

/* Even-odd test of m points against ONE ring of nv vertices (open: the closing edge is implicit), bit for bit
 * geometry.points_in_polygon: edges half-open in y, crossing abscissa dx * (y - y1) / dy + x1 rounded in that
 * order.  op 0: inside = test; 1: inside |= test; 2: inside &= !test (the rings of a CompositePolygon,
 * device.py:286-293).  Not scb_points_in_rings, which rounds in another order. */
int scb_points_in_polygon(int64_t m, const double* points, int64_t nv, const double* vertices, int op,
                          uint8_t* inside, scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Kernel matrix pieces and system assembly  (K1-K3, K8-K10, K19, rows a1-a3, a9-a11)
 *   distance.py:87-115 q_matrix, device/mesh.py:434-458 Q_matrix,
 *   solver/utils.py:290-297 (dense casts, never materialised here),
 *   solver/solve_film.py:181-185 grad_Lambda_term, :285-305 _build_system_1d/_2d
 * ------------------------------------------------------------------------------------ */

/* Edge-correction vector C for arbitrary points (MeshOperators.C_vector, device/mesh.py:400-432).
 * scratch: device double[8]. */
int scb_c_vector(int64_t n, const double* points, double* scratch, double* C, scb_stream_t stream);

/* qdw[i] = C[i] + sum_{j != i} q_ij w_j  ( == Q_ii * w_i, device/mesh.py:456 ) */
int scb_kernel_diagonal(int64_t n, const double* sites, const double* weights, const double* C,
                        double* qdw, scb_stream_t stream);

/* grad-Lambda term on the operator pattern (solve_film.py:181-185):
 * T[k] = gLx[row] * gradient_x[k] + gLy[row] * gradient_y[k],  gL = gradient @ Lambda */
int scb_grad_lambda_term(int64_t n, const int32_t* op_indptr, const int32_t* op_indices,
                         const double* gradient_x, const double* gradient_y,
                         const double* Lambda, double* T, scb_stream_t stream);

/* Writes M = -A  (A of solve_film.py:296-305 restricted to rows/cols `ix`) into the padded
 * row-major LU workspace negA[n_pad, n_pad] (n_pad = multiple of SCB_LU_BLOCK >= n_int;
 * the padding block is the identity).  pos_scratch is int32[n].
 *   M[r,c] = q(ix_r, ix_c) w[ix_c] + Lambda[ix_c] lap[ix_r, ix_c] + T[ix_r, ix_c]   (r != c)
 *   M[r,r] = -qdw[ix_r]           + Lambda[ix_r] lap[ix_r, ix_r] + T[ix_r, ix_r]
 * T may be NULL (homogeneous Lambda).  margin (may be NULL; needs C) receives a lower bound
 * of the row-dominance margin |M_rr| - sum_{c != r} |M_rc| (exact when ix covers every vertex)
 * used to validate the unpivoted LU (SURVEY.md Q11).
 * sym_scale (NULL, or sqrt(w) per mesh vertex; needs T == NULL and a constant Lambda): writes the
 * diagonally similar SYMMETRIC matrix S = D M D^-1, D = diag(sqrt(w[ix])), instead of M, for
 * scb_getrf_sym_nopiv:  S[r,c] = q sqrt(w_r w_c) + Lambda lap[r,c] sqrt(w_r / w_c),  S[r,r] = M[r,r];
 * M x = h  <=>  S (D x) = D h. */
int scb_system_assemble(int64_t n, const double* sites, const double* weights, const double* qdw,
                        const double* C, const double* Lambda, const int32_t* op_indptr,
                        const int32_t* op_indices,
                        const double* laplacian, const double* T, int64_t n_int, const int64_t* ix,
                        int32_t* pos_scratch, int64_t n_pad, double* negA, double* margin,
                        const double* sym_scale, scb_stream_t stream);

/* Matrix-free action of the FULL (n x n) operator A on nrhs vectors, sources restricted
 * to `src_idx` (NULL = all vertices; n_src = 0 with a non-NULL src_idx: no source):
 *   out[i,:] (+)= sum_{j in src} A_ij v[j,:],  A_ij = Q_ij w_j - Lambda_j lap_ij - T_ij
 * with Q_ij w_j = -q_ij w_j (i != j), Q_ii w_i = qdw_i.  v, out are [n, nrhs] row-major.
 * Only the dense part -q_ij w_j reads src_idx; the diagonal and sparse parts act on all of v, so the
 * sum is over src when v vanishes outside src (as every caller's v does).
 * Replaces the hole slabs `_build_system_1d` @ g[hole] (solve_film.py:285-293,498-503),
 * `Q @ (weights * g)` (solve_film.py:565, with Lambda == NULL: kernel part only) and the
 * check_inversion product (solve_film.py:533-540).  The dense part runs as tiled N-body sums on the
 * fp64 CUDA cores, or for nrhs >= 16 as a DMMA GEMM whose kernel-matrix operand is evaluated on the
 * fly in the mma fragment layout. */
int scb_apply_operator(int64_t n, const double* sites, const double* weights, const double* qdw,
                       const double* Lambda, const int32_t* op_indptr, const int32_t* op_indices,
                       const double* laplacian, const double* T, int64_t n_src,
                       const int64_t* src_idx, int64_t nrhs, const double* v, double* out,
                       int accumulate, scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Dense LU  (K11, K12, row a12/a13): scipy.linalg.lu_factor / lu_solve at
 *   solver/solve_film.py:232,253,279 and :367,388,530,545
 * ------------------------------------------------------------------------------------ */

/* bytes of the factorization side buffer `dinv` for an n_pad x n_pad system: inverses of the
 * 128x128 diagonal blocks (kept, used by scb_getrs_nopiv), two sets of fragment-major packed
 * panels (scratch of the look-ahead LU) and the ready flags / work counter of scb_getrs_nopiv */
int64_t scb_getrf_dinv_bytes(int64_t n_pad);

/* In-place two-level blocked right-looking LU of the row-major matrix M[n_pad, n_pad] WITHOUT
 * pivoting (valid for the row-diagonally-dominant systems of this path, SURVEY.md Q11; the caller
 * checks `margin` from scb_system_assemble).  Inner panels of 128 columns, outer panels of 1024
 * columns whose trailing update runs on DMMA tensor cores with TMA-staged packed panels; the
 * factorization of the next outer panel runs on an internal high-priority stream concurrently
 * with the trailing update (look-ahead) and is joined back into `stream` before returning.
 * On return M holds L (unit lower) and U; dinv holds inv(L_kk), inv(U_kk) of every 128x128
 * diagonal block.  info (device int32[1]) <- 0, or 1 + index of the first zero/non-finite pivot.
 * Repeated calls with the same (n_pad, M, dinv, info) -- a steady-state loop over a device whose buffers
 * come from a caching allocator -- are captured into a CUDA graph at the second call (on a stream of the
 * library) and replayed with one cudaGraphLaunch into `stream` from then on: small films are latency-bound and
 * enqueueing their few hundred launches costs the host as long as the GPU needs to run them.  Identical
 * kernels and arguments, bit-identical factors.  n_pad <= SCB_LU_GRAPH_MAX_N (12288) only; SCB_LU_GRAPH=0
 * disables it.  A call made while `stream` is itself being captured simply takes part in that capture. */
int scb_getrf_nopiv(int64_t n_pad, double* M, double* dinv, int32_t* info, scb_stream_t stream);

/* Same for a SYMMETRIC matrix (the symmetrised system of scb_system_assemble): only the lower
 * triangle is read and updated, the row panels are obtained from the column panels
 * (U12 = diag(U11) L21^T), and the trailing update touches only tiles on or below the diagonal --
 * 1/3 n^3 flop instead of 2/3 n^3.  On return M holds L (unit lower) and U (upper) of the LU
 * factorization of the symmetric matrix, exactly as scb_getrf_nopiv would produce. */
int scb_getrf_sym_nopiv(int64_t n_pad, double* M, double* dinv, int32_t* info, scb_stream_t stream);

/* The same factorization WITH partial (row) pivoting, P M = L U -- what the reference's
 * scipy.linalg.lu_factor (LAPACK dgetrf) computes -- for systems that are not provably safe without it
 * (general systems whose `margin` from scb_system_assemble is not positive).  Per 128-column panel the
 * pivot rows are found on a scratch copy (maximum magnitude over all rows below the diagonal, ties to the
 * lower row index), the interchanges are applied to the full rows, and the panel is then factored and
 * applied by the unpivoted kernels (K = 128 trailing updates on DMMA).  piv (device int32[n_pad]):
 * LAPACK-style, row k was interchanged with row piv[k] (0-based).  perm (device int32[n_pad]): row r of
 * P M is row perm[r] of M, i.e. solve M x = h as scb_getrs_nopiv on B[r] = h[perm[r]].  The identity
 * padding block is never interchanged with real rows.  info as for scb_getrf_nopiv. */
int scb_getrf_piv(int64_t n_pad, double* M, double* dinv, int32_t* piv, int32_t* perm, int32_t* info,
                  scb_stream_t stream);

/* Solves M X = B in place for nrhs right-hand sides, B[n_pad, nrhs] row-major, with the factors
 * and the `dinv` buffer produced by scb_getrf_nopiv / scb_getrf_sym_nopiv / scb_getrf_piv (for the
 * latter, B holds the permuted right-hand side).  Two persistent flag-driven sweep kernels (forward,
 * backward) over column chains: one right-hand side: one scalar chain; 2..8: one chain of 8 columns with
 * DMMA block products; more: chains of 16 columns, at most 8 chains (128 columns) per launch -- beyond
 * that a further launch pair per 128 columns. */
int scb_getrs_nopiv(int64_t n_pad, const double* LU, const double* dinv, int64_t nrhs, double* B,
                    scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Sparse mat-vec (K14): grad_y @ g, grad_x @ g  (solver/solve_film.py:556-559)
 *   y[nrows, nrhs] = alpha * CSR @ x[ncols, nrhs] + beta * y
 * ------------------------------------------------------------------------------------ */
int scb_spmv(int64_t nrows, const int32_t* indptr, const int32_t* indices, const double* data,
             int64_t nrhs, const double* x, double alpha, double beta, double* y,
             scb_stream_t stream);

/* Fused steps of one film solve (solver/solve_film.py:526-531,556); all arrays are [rows, nrhs]
 * row-major.
 *   scb_solve_rhs:  B[r, c] = (applied[ix[r], c] + other[ix[r], c] - ha_eff[ix[r], c]) * scale[r] for
 *       r < n_int and 0 for the padding rows n_int <= r < n_pad  (h = Hz_applied[ix] - Ha_eff[ix], in the
 *       symmetrised system scaled by D).  other, ha_eff, scale may be NULL.
 *   scb_solve_stream:  g[i, c] = g0[i, c] + (pos[i] >= 0 ? X[pos[i], c] / scale[pos[i]] : 0)  (g[ix] += gf on
 *       top of the hole / transport boundary values g0; pos = the vertex -> system-row map that
 *       scb_system_assemble leaves in pos_scratch, -1 outside the system).  scale, g0 may be NULL.
 *   scb_current_density:  J[i, c, :] = ((gradient_y g)[i, c], -(gradient_x g)[i, c])  in one pass. */
int scb_solve_rhs(int64_t n_int, int64_t n_pad, const int64_t* ix, int64_t nrhs, const double* applied,
                  const double* other, const double* ha_eff, const double* scale, double* B, scb_stream_t stream);
int scb_solve_stream(int64_t n, int64_t nrhs, const int32_t* pos, const double* X, const double* scale,
                     const double* g0, double* g, scb_stream_t stream);
int scb_current_density(int64_t n, const int32_t* op_indptr, const int32_t* op_indices, const double* gradient_x,
                        const double* gradient_y, int64_t nrhs, const double* g, double* J, scb_stream_t stream);
/* The whole device-side body of one film solve in a single call (solver/solve_film.py:526-531,545,556-559):
 * scb_solve_rhs -> scb_getrs_nopiv -> scb_solve_stream -> scb_current_density with the arguments of those
 * entry points (B is the [n_pad, nrhs] workspace of the triangular solves).  A Jacobi step of a small film is
 * latency-bound; one foreign call instead of four shortens the host side of it. */
int scb_solve_step(int64_t n, int64_t n_int, int64_t n_pad, int64_t nrhs, const int64_t* rhs_ix,
                   const double* applied, const double* other, const double* ha_eff, const double* scale,
                   const double* LU, const double* dinv, double* B, const int32_t* pos, const double* g0, double* g,
                   const int32_t* op_indptr, const int32_t* op_indices, const double* gradient_x,
                   const double* gradient_y, double* J, scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Vortices (solver/solve_film.py:541-554).  The vortex term of the reference,
 *   g[ix] += flux nPhi0 K[:, j_film] / w[j_device],   K = -(-A)^-1,
 * is the solution of (-A) x = h - c e_{j_film} with c = flux nPhi0 / w[j_device]: a sparse correction to
 * the right-hand side, applied between scb_solve_rhs and scb_getrs_nopiv (or to h itself before a
 * solve), with no solve of its own.  A film with vortices runs
 *   scb_solve_rhs -> scb_vortex_rhs -> scb_getrs_nopiv -> scb_solve_stream -> scb_current_density.
 * ------------------------------------------------------------------------------------ */

/* Nearest vertex of each of the nv query points xy [nv, 2] among the n_sub sites sites[sub[k]]
 * (j_sub [nv] <- k: the system row j_film for sub = the system's index set) and among all n sites
 * (j_all [nv] <- i: j_device), in one pass.  Bit for bit np.argmin(np.linalg.norm(P - xy, axis=1)): the
 * distances are rounded as numpy rounds them (sqrt(dx*dx + dy*dy), no FMA contraction), the ROUNDED
 * distances are compared (distinct squared distances can round to one norm), ties and NaN resolve as in
 * numpy (lowest index).  The reduction runs on (distance, index) pairs under that total order: the result
 * does not depend on its order.  sub, j_sub, j_all are int64.  nv = 0 does nothing; otherwise n, n_sub >= 1. */
int scb_locate_vortices(int64_t nv, const double* xy, int64_t n, const double* sites, int64_t n_sub,
                        const int64_t* sub, int64_t* j_sub, int64_t* j_all, scb_stream_t stream);

/* Vortex right-hand-side terms of nrhs columns.  The vortices are sorted by column in a CSR layout:
 * column c holds vortices col_ptr[c] .. col_ptr[c+1] (int64 [nrhs+1]).  For each of them, in order,
 *   B[row[v], c] -= flux * nphi0[v] / weights[j_all[v]] * scale[row[v]]
 * (one rounding per operation, left to right; B [rows, nrhs] row-major).  `row` is the row of B, not the
 * vertex: j_sub of scb_locate_vortices, or for a pivoted system (B[r] = h[perm[r]]) invperm[j_sub].
 * scale (NULL: not symmetrised) is the D of the symmetrised system.  One thread per column, no atomics:
 * deterministic, and two vortices at one vertex simply add.  row, j_all are int64 [nv]. */
int scb_vortex_rhs(int64_t nrhs, const int64_t* col_ptr, const int64_t* row, const int64_t* j_all,
                   const double* nphi0, const double* weights, double flux, const double* scale, double* B,
                   scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Biot-Savart family (K15-K18, rows a14, a15, a17, a18)
 * ------------------------------------------------------------------------------------ */
enum scb_bs_kind {
  /* solver/solve.py:28-73 biot_savart_film_to_film; also _biot_savart_within_film
   * (solve_film.py:415-437) with dz = 0.  tgt [m,2], src [n,2], scalar dz, out [m] */
  SCB_BS_FILM_TO_FILM = 0,
  /* sources/current.py:13-57 _biot_savart_2d_z: tgt [m,3], src [n,3], out [m] */
  SCB_BS_Z = 1,
  /* sources/current.py:60-110 _biot_savart_2d_vector: out [m,3] */
  SCB_BS_VECTOR = 2,
  /* solution.py:917-928 vector potential: tgt [m,3], src [n,3], out [m,2] */
  SCB_BS_VECTOR_POTENTIAL = 3,
  /* solve_film.py:393-412 _get_boundary_effective_field: tgt [m,2], src = edge centres [n,2],
   * J = edge normals [n,2], area = stream * length [n, nsets], out [m, nsets].  The edge geometry
   * (centres, normals, r^-3 of every pair) is shared by the nsets stream sets. */
  SCB_BS_BOUNDARY = 4
};

/* out = prefactor * sum_j area_j * kernel(tgt_i, src_j, J_j).  nsets > 1 evaluates `nsets`
 * current-density sets J[nsets, n, 2] against the same geometry, out[nsets, m(, c)]; for
 * SCB_BS_BOUNDARY the sets are the columns of area[n, nsets] and out[m, nsets] (see above).
 * Every kind evaluates r^-3 (SCB_BS_VECTOR_POTENTIAL: r^-1) of a pair once for up to 8 sets
 * (passes of 8 / 4 / 2 / 1 sets).  Every set of an SCB_BS_Z, SCB_BS_VECTOR or
 * SCB_BS_VECTOR_POTENTIAL call has the bits of an nsets = 1 call on that set alone: the passes
 * share its arithmetic and its split of the sources, which depends only on (m, n). */
int scb_biot_savart(int kind, int64_t m, const double* tgt, int64_t n, const double* src,
                    const double* area, const double* J, double dz, double prefactor,
                    int64_t nsets, double* out, scb_stream_t stream);

/* One Jacobi step of the film-to-film iteration for ONE target film (solver/solve.py:495-515: the
 * sum of biot_savart_film_to_film over every other film) in a single launch.  The sources are the
 * packed vertices of all films: src [n,3] = (x, y, z0 of the owning film's layer), area [n] (0 for
 * padding rows), J [n, nsets, 2] (source-major: the layout the per-iteration J exchange delivers).
 * Sources in [skip_lo, skip_hi) -- the target film's own segment -- are left out.
 *   out[i, s] = prefactor * sum_j area_j (Jx[j,s] (y_i - y_j) - Jy[j,s] (x_i - x_j)) r_ij^-3,
 *   r_ij^2 = (x_i - x_j)^2 + (y_i - y_j)^2 + (tgt_z - z_j)^2;   tgt [m,2], out [m, nsets]. */
int scb_film_coupling(int64_t m, const double* tgt, double tgt_z, int64_t n, const double* src,
                      const double* area, const double* J, int64_t skip_lo, int64_t skip_hi,
                      double prefactor, int64_t nsets, double* out, scb_stream_t stream);

/* scb_film_coupling with every film moved rigidly, per set: set r moves film f by shift[r][f] =
 * (dx, dy, dz), shift [nsets, nfilms, 3].  The targets belong to film `dst` (0 <= dst < nfilms);
 * src_film [n] (int32, device) is the film of every packed source row, < 0 for padding rows, which
 * never move.  Set r equals, bit for bit, an nsets = 1 scb_film_coupling call on the moved inputs
 *   tgt' = (x_i + shift[r][dst].x, y_i + shift[r][dst].y),  tgt_z' = tgt_z + shift[r][dst].z,
 *   src'_j = src_j + shift[r][src_film[j]]  (componentwise),  J column r,
 * because the passes use that call's arithmetic (dx = fl(x_t + o_t) - fl(x_s + o_s), likewise dy and dz;
 * r^2 = fma(dx, dx, dy dy) + dz^2) and its split of the sources.  Every set has its own geometry, so
 * nothing is shared between sets: passes of 2 / 1 sets. */
int scb_film_coupling_translated(int64_t m, const double* tgt, double tgt_z, int64_t n, const double* src,
                                 const double* area, const double* J, int64_t skip_lo, int64_t skip_hi,
                                 double prefactor, int64_t nsets, int64_t dst, const int32_t* src_film,
                                 int64_t nfilms, const double* shift, double* out, scb_stream_t stream);

/* Field of a film's own sheet current at its vertices for `nsets` current-density sets
 * (solve_film.py:415-437 _biot_savart_within_film; the self field of a film with transport terminals):
 *   out[i, s] = prefactor * sum_j area_j (Jx[j,s] (y_i - y_j) - Jy[j,s] (x_i - x_j)) r_ij^-3,
 * tgt [m,2] (vertices), src [n,2] (triangle centroids), area [n], J [n, nsets, 2] (source-major: the
 * layout scb_spmv produces for the triangle gradients), out [m, nsets].  Every full pass of 64 sets runs
 * as a GEMM on the fp64 tensor cores (K = 2 n) whose r^-3 operand is evaluated in the mma fragment
 * layout and shared by the 64 sets; the remaining sets run as tiled N-body sums on the CUDA cores in
 * passes of 8 / 4 / 2 / 1 (faster below 32 sets, even at 32, measured).  Fixed summation order:
 * bit-reproducible.  n = 0 writes zeros; m = 0 does nothing. */
int scb_biot_savart_within_film(int64_t m, const double* tgt, int64_t n, const double* src,
                                const double* area, const double* J, double prefactor, int64_t nsets,
                                double* out, scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Pairwise distances (K20): distance.py:5-84 cdist / (sq)euclidean_distance_2d/3d
 *   out[m, n] = |XA_i - XB_j|  (squared != 0: squared distance), dim = 2 or 3.  HBM-write bound.
 * ------------------------------------------------------------------------------------ */
int scb_cdist(int dim, int squared, int64_t m, const double* XA, int64_t n, const double* XB,
              double* out, scb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Diagnostics: roofline denominators measured in place (bench.py).  Launches a register-resident
 * issue-rate loop of the fp64 tensor-core atom (kind 0: mma.sync m8n8k4 f64 = DMMA.8x8x4) or of DFMA
 * (kind 1), one 512-thread CTA per SM.  *flop_host (HOST pointer, may be NULL) <- flop executed by the
 * launch; the caller times the launch with CUDA events.  scratch: scb_diag_scratch_elems() doubles.
 * ------------------------------------------------------------------------------------ */
int scb_diag_issue_rate(int kind, int64_t iters, double* scratch, double* flop_host, scb_stream_t stream);
int64_t scb_diag_scratch_elems(void);

#ifdef __cplusplus
}
#endif
#endif /* SCB_H */
