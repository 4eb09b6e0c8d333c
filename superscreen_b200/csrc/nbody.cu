// Tiled fp64 N-body style pair sums (K13, K15-K18, the row sums of the kernel matrix and the
// film-to-film coupling of the Jacobi iteration).
//
// One templated kernel.  A thread owns TPT = 2 targets (coalesced: target k of thread t in CTA b is
// (b * TPT + k) * 256 + t); the sources are staged through shared memory in tiles of 256 and every
// thread walks the whole tile, so all lanes of a warp read the SAME shared-memory word (broadcast,
// one wavefront per load) and the operands of a source are loaded once for TPT pairs.
// Parallelism for small target sets (a film's own vertices: 2k-60k targets) comes from splitting
// the SOURCES over gridDim.y CTAs, never from sub-dividing a warp: the partial sums go to a
// stream-ordered scratch buffer [split][target][acc] and a second tiny kernel adds them in split
// order.  Split count and chunk size depend only on (m, n), so results are bit-reproducible and no
// float atomics are used.  Million-point field evaluations run unsplit.
//
// fp64 CUDA-core bound: ~16-20 DFMA-class operations per pair (SURVEY.md section 8d).
//
// Reference kernels restated (file:line under /root/reference/superscreen):
//   distance.py:87-115 + device/mesh.py:454-458 (row sums / Q @ (w*g))
//   solver/solve.py:28-73 biot_savart_film_to_film (+ its sum over films, :495-515),
//   solver/solve_film.py:393-437
//   sources/current.py:13-110 _biot_savart_2d_z/_vector, solution.py:917-928 vector potential
#include "scb_common.cuh"

namespace scb {

enum : int {
  NB_FILM_TO_FILM = SCB_BS_FILM_TO_FILM,
  NB_Z = SCB_BS_Z,
  NB_VECTOR = SCB_BS_VECTOR,
  NB_VECPOT = SCB_BS_VECTOR_POTENTIAL,
  NB_BOUNDARY = SCB_BS_BOUNDARY,
  NB_KERNEL = 16,    // sum_{j != i} q_ij * payload_j[r], r < NR   (in-plane, 1/r^3)
  NB_COUPLING = 17,  // film-to-film over the packed sources of all films (scb_film_coupling)
  NB_COUPLING_T = 18,  // NB_COUPLING with a per-set shift of every film (scb_film_coupling_translated)
};

constexpr int kTile = 256;
constexpr int TPT = 2;  // targets per thread

struct NbodyParams {
  int64_t m;              // targets
  const double* tgt;      // [m,2] or [m,3]
  int64_t n;              // sources
  const double* src;      // [*,2] or [*,3] (indexed through src_idx when given)
  const int64_t* src_idx; // optional gather list for NB_KERNEL
  const double* area;     // [*] per-source weight; NB_BOUNDARY: [n, ldv] per-source, per-set strengths
  const double* J;        // [*,2] (biot-savart), v [*, ldv] (NB_KERNEL), [n, ldv] (NB_COUPLING, ldv = 2 nsets)
  int64_t ldv;            // row stride of v / J (NB_BOUNDARY: of area, = nsets)
  int64_t ldo;            // row stride of out (NB_KERNEL: = ldv; NB_COUPLING, NB_BOUNDARY: nsets)
  int64_t rhs0;           // first rhs column / current-density set handled by this launch
  double dz2;             // film-to-film: squared layer distance
  double tgt_z;           // NB_COUPLING: z of the target film
  int64_t skip_lo, skip_len;  // NB_COUPLING: sources [skip_lo, skip_lo + skip_len) are left out
  int64_t sld;            // NB_COUPLING: source row (x, y, z) = 3, or (x, y) = 2 for sources in the target plane
  double prefactor;
  double* out;
  int accumulate;
  int64_t chunk;          // sources per CTA; gridDim.y CTAs cover the sources
  double* partial;        // [gridDim.y][m][NACC] partial sums when gridDim.y > 1
};

// NB_COUPLING_T: set r moves the sources of film f by shift[r][f] and the targets by shift[r][dst].
// A second kernel argument, so that NbodyParams (and the code of the other kinds) stays as it is.
struct ShiftTable {
  const int32_t* src_film;  // [n] film of every packed source row (< 0: padding, never moved)
  const double* shift;      // [nsets][nfilms][3]
  int64_t nfilms, dst;
};

template <int KIND, int NR>
struct Traits {
  static constexpr int tdim = (KIND == NB_Z || KIND == NB_VECTOR || KIND == NB_VECPOT) ? 3 : 2;
  static constexpr bool coupling = KIND == NB_COUPLING || KIND == NB_COUPLING_T;
  // NR = right-hand sides (NB_KERNEL), current-density sets sharing the geometry (film-to-film, NB_Z,
  // NB_VECTOR, NB_VECPOT), boundary stream sets sharing the edges (NB_BOUNDARY) or sets with a geometry each
  // (NB_COUPLING_T)
  // source geometries per tile: NB_COUPLING_T stages the shifted sources of every set, the others share one
  static constexpr int ngeo = KIND == NB_COUPLING_T ? NR : 1;
  // NB_Z keeps two sums per set (Jx dy, Jy dx) and subtracts them only in nbody_store, NB_VECTOR four
  // (Jx dy, Jy dx, Jx dz, Jy dz), NB_VECPOT two (Jx, Jy)
  static constexpr int nacc = (KIND == NB_Z || KIND == NB_VECPOT) ? 2 * NR : (KIND == NB_VECTOR ? 4 * NR : NR);
  static constexpr int npay = KIND == NB_KERNEL ? NR : 2 * NR;
  static constexpr bool has_sz = tdim == 3 || coupling;
};

// final value(s) of target i from its complete sums
template <int KIND, int NR>
__device__ __forceinline__ void nbody_store(const NbodyParams& p, int64_t i, const double (&acc)[Traits<KIND, NR>::nacc]) {
  const double pf = p.prefactor;
  if (KIND == NB_KERNEL) {
#pragma unroll
    for (int r = 0; r < NR; r++) {
      double* o = p.out + i * p.ldo + p.rhs0 + r;
      *o = p.accumulate ? *o + pf * acc[r] : pf * acc[r];
    }
  } else if (Traits<KIND, NR>::coupling || KIND == NB_BOUNDARY) {
#pragma unroll
    for (int r = 0; r < NR; r++) p.out[i * p.ldo + p.rhs0 + r] = pf * acc[r];
  } else if (KIND == NB_Z) {
#pragma unroll
    for (int r = 0; r < NR; r++) p.out[r * p.m + i] = pf * (acc[2 * r] - acc[2 * r + 1]);
  } else if (KIND == NB_VECTOR) {
#pragma unroll
    for (int r = 0; r < NR; r++) {
      const int64_t t = r * p.m + i;
      p.out[3 * t] = pf * acc[4 * r + 3];
      p.out[3 * t + 1] = -(pf * acc[4 * r + 2]);
      p.out[3 * t + 2] = pf * (acc[4 * r] - acc[4 * r + 1]);
    }
  } else if (KIND == NB_VECPOT) {
#pragma unroll
    for (int r = 0; r < NR; r++) {
      const int64_t t = r * p.m + i;
      p.out[2 * t] = pf * acc[2 * r];
      p.out[2 * t + 1] = pf * acc[2 * r + 1];
    }
  } else if (KIND == NB_FILM_TO_FILM) {
#pragma unroll
    for (int r = 0; r < NR; r++) p.out[r * p.m + i] = pf * acc[r];
  }
}

template <int KIND, int NR>
__global__ void __launch_bounds__(256) nbody_kernel(NbodyParams p, ShiftTable st) {
  using T = Traits<KIND, NR>;
  constexpr int TD = T::tdim;
  constexpr int NACC = T::nacc;
  constexpr int NPAY = T::npay;
  constexpr int NG = T::ngeo;
  constexpr bool SHIFTED = KIND == NB_COUPLING_T;
  __shared__ double sx[NG * kTile], sy[NG * kTile], sz[T::has_sz ? NG * kTile : 1];
  __shared__ double spay[NPAY][kTile];

  const int tid = threadIdx.x;
  int64_t ti[TPT];
  double tx[TPT], ty[TPT], tz[TPT];
#pragma unroll
  for (int k = 0; k < TPT; k++) {
    ti[k] = (blockIdx.x * (int64_t)TPT + k) * 256 + tid;
    const bool ok = ti[k] < p.m;
    tx[k] = ok ? p.tgt[TD * ti[k]] : 0.0;
    ty[k] = ok ? p.tgt[TD * ti[k] + 1] : 0.0;
    tz[k] = (ok && TD == 3) ? p.tgt[TD * ti[k] + 2] : 0.0;
  }
  // NB_COUPLING_T: the targets of every set, moved by the target film's shift once (registers)
  double gx[TPT][NG], gy[TPT][NG], gz[NG];
  if (SHIFTED) {
#pragma unroll
    for (int g = 0; g < NG; g++) {
      const double* o = st.shift + ((p.rhs0 + g) * st.nfilms + st.dst) * 3;
      gz[g] = p.tgt_z + o[2];
#pragma unroll
      for (int k = 0; k < TPT; k++) {
        gx[k][g] = tx[k] + o[0];
        gy[k][g] = ty[k] + o[1];
      }
    }
  }
  double acc[TPT][NACC];
#pragma unroll
  for (int k = 0; k < TPT; k++)
#pragma unroll
    for (int a = 0; a < NACC; a++) acc[k][a] = 0.0;

  // this CTA's slice of the (virtual, skip range removed) source index space
  const int64_t n_eff = p.n - (T::coupling ? p.skip_len : 0);
  const int64_t lo = blockIdx.y * p.chunk;
  const int64_t hi = (lo + p.chunk) < n_eff ? (lo + p.chunk) : n_eff;
  for (int64_t base = lo; base < hi; base += kTile) {
    const int64_t v = base + tid;
    __syncthreads();
    if (v < hi) {
      const int64_t j = (T::coupling && v >= p.skip_lo) ? v + p.skip_len : v;
      const int64_t js = p.src_idx ? p.src_idx[j] : j;
      const double w = p.area[js];
      if (SHIFTED) {
        // every set's shifted source and dz^2, staged once per tile (the arithmetic of a one-set call on
        // shifted inputs: (x + o) rounded, then the differences)
        const int f = st.src_film[js];
        const double x = p.src[3 * js], y = p.src[3 * js + 1], z = p.src[3 * js + 2];
        const double* Jj = p.J + js * p.ldv + 2 * p.rhs0;
#pragma unroll
        for (int g = 0; g < NG; g++) {
          const double* o = st.shift + ((p.rhs0 + g) * st.nfilms + (f < 0 ? 0 : f)) * 3;
          sx[g * kTile + tid] = f < 0 ? x : x + o[0];
          sy[g * kTile + tid] = f < 0 ? y : y + o[1];
          const double dz = gz[g] - (f < 0 ? z : z + o[2]);
          sz[g * kTile + tid] = dz * dz;
          spay[2 * g][tid] = w * Jj[2 * g];
          spay[2 * g + 1][tid] = w * Jj[2 * g + 1];
        }
      } else if (KIND == NB_COUPLING) {
        sx[tid] = p.src[p.sld * js];
        sy[tid] = p.src[p.sld * js + 1];
        const double dz = p.tgt_z - (p.sld == 3 ? p.src[3 * js + 2] : p.tgt_z);
        sz[tid] = dz * dz;
        const double* Jj = p.J + js * p.ldv + 2 * p.rhs0;
#pragma unroll
        for (int r = 0; r < NR; r++) {
          spay[2 * r][tid] = w * Jj[2 * r];
          spay[2 * r + 1][tid] = w * Jj[2 * r + 1];
        }
      } else {
        sx[tid] = p.src[TD * js];
        sy[tid] = p.src[TD * js + 1];
        if (TD == 3) sz[tid] = p.src[TD * js + 2];
        if (KIND == NB_KERNEL) {
#pragma unroll
          for (int r = 0; r < NR; r++) spay[r][tid] = p.J ? w * p.J[js * p.ldv + p.rhs0 + r] : w;
        } else if (KIND == NB_BOUNDARY) {
#pragma unroll
          for (int r = 0; r < NR; r++) {
            const double wr = p.area[js * p.ldv + p.rhs0 + r];
            spay[2 * r][tid] = wr * p.J[2 * js];
            spay[2 * r + 1][tid] = wr * p.J[2 * js + 1];
          }
        } else {  // NB_FILM_TO_FILM, NB_Z, NB_VECTOR, NB_VECPOT: J [NR, n, 2]
#pragma unroll
          for (int r = 0; r < NR; r++) {
            spay[2 * r][tid] = w * p.J[(r * p.n + js) * 2];
            spay[2 * r + 1][tid] = w * p.J[(r * p.n + js) * 2 + 1];
          }
        }
      }
    }
    __syncthreads();
    const int cnt = (int)((hi - base) < kTile ? (hi - base) : kTile);
#pragma unroll 2
    for (int jj = 0; jj < cnt; jj++) {
      const double xs0 = sx[jj], ys0 = sy[jj];
      const double zs0 = T::has_sz ? sz[jj] : 0.0;
      double pay[NPAY];
#pragma unroll
      for (int q = 0; q < NPAY; q++) pay[q] = spay[q][jj];
      // NG geometries, each shared by NR / NG sets (NG = 1: one r^-3 per pair for all sets)
#pragma unroll
      for (int g = 0; g < NG; g++) {
        const double xs = g == 0 ? xs0 : sx[g * kTile + jj], ys = g == 0 ? ys0 : sy[g * kTile + jj];
        const double zs = g == 0 ? zs0 : sz[g * kTile + jj];
#pragma unroll
        for (int k = 0; k < TPT; k++) {
          const double dx = (SHIFTED ? gx[k][g] : tx[k]) - xs, dy = (SHIFTED ? gy[k][g] : ty[k]) - ys;
          double r2 = fma(dx, dx, dy * dy);
          double dzv = 0.0;
          if (TD == 3) {
            dzv = tz[k] - zs;
            r2 = fma(dzv, dzv, r2);
          } else if (T::coupling) {
            r2 += zs;
          } else if (KIND == NB_FILM_TO_FILM) {
            r2 += p.dz2;
          }
          if (KIND == NB_VECPOT) {  // one r^-1 per pair for every set of the pass
            const double inv = inv_r1(r2);
#pragma unroll
            for (int r = 0; r < NR; r++) {
              acc[k][2 * r] = fma(pay[2 * r], inv, acc[k][2 * r]);
              acc[k][2 * r + 1] = fma(pay[2 * r + 1], inv, acc[k][2 * r + 1]);
            }
          } else {
            double k3 = inv_r3(r2);
            if (KIND == NB_KERNEL) {
              k3 = r2 > 0.0 ? k3 : 0.0;  // q_ii = 0 (distance.py:104-105)
#pragma unroll
              for (int r = 0; r < NR; r++) acc[k][r] = fma(pay[r], k3, acc[k][r]);
            } else if (KIND == NB_FILM_TO_FILM || T::coupling) {
              const double kdy = k3 * dy, kdx = k3 * dx;
#pragma unroll
              for (int r = g * (NR / NG); r < (g + 1) * (NR / NG); r++)
                acc[k][r] = fma(pay[2 * r], kdy, fma(-pay[2 * r + 1], kdx, acc[k][r]));
            } else if (KIND == NB_BOUNDARY) {
#pragma unroll
              for (int r = 0; r < NR; r++) acc[k][r] = fma(-k3, fma(pay[2 * r], dx, pay[2 * r + 1] * dy), acc[k][r]);
            } else if (KIND == NB_Z) {
#pragma unroll
              for (int r = 0; r < NR; r++) {
                acc[k][2 * r] = fma(k3 * pay[2 * r], dy, acc[k][2 * r]);              // Jx_dy
                acc[k][2 * r + 1] = fma(k3 * pay[2 * r + 1], dx, acc[k][2 * r + 1]);  // Jy_dx
              }
            } else {                                        // NB_VECTOR
#pragma unroll
              for (int r = 0; r < NR; r++) {
                const double px = k3 * pay[2 * r], py = k3 * pay[2 * r + 1];
                acc[k][4 * r] = fma(px, dy, acc[k][4 * r]);           // Jx_dy
                acc[k][4 * r + 1] = fma(py, dx, acc[k][4 * r + 1]);   // Jy_dx
                acc[k][4 * r + 2] = fma(px, dzv, acc[k][4 * r + 2]);  // Jx_dz
                acc[k][4 * r + 3] = fma(py, dzv, acc[k][4 * r + 3]);  // Jy_dz
              }
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < TPT; k++) {
    if (ti[k] >= p.m) continue;
    if (gridDim.y == 1) {
      nbody_store<KIND, NR>(p, ti[k], acc[k]);
    } else {
      double* o = p.partial + ((int64_t)blockIdx.y * p.m + ti[k]) * NACC;
#pragma unroll
      for (int a = 0; a < NACC; a++) o[a] = acc[k][a];
    }
  }
}

// adds the per-split partial sums of a target in split order and stores the final value(s).
// A group of NACC consecutive lanes owns one target (lane a of the group adds accumulator a over the
// splits: coalesced reads, NACC times more loads in flight than one thread per target), the group's
// totals meet in the lane that stores them through one shared-memory row per target.
template <int KIND, int NR>
__global__ void __launch_bounds__(128) nbody_reduce_kernel(NbodyParams p, int nsplit) {
  constexpr int NACC = Traits<KIND, NR>::nacc;
  constexpr int TPB = 128 / NACC;  // targets per CTA (NACC in {1, 2, 4, 8, 16, 32})
  static_assert(128 % NACC == 0, "accumulator count must divide the CTA size");
  __shared__ double tot[TPB][NACC + 1];
  const int a = threadIdx.x % NACC, t = threadIdx.x / NACC;
  const int64_t i = blockIdx.x * (int64_t)TPB + t;
  if (i < p.m) {
    const double* o = p.partial + i * NACC + a;
    const int64_t stride = p.m * NACC;
    double s0 = 0.0;
#pragma unroll 8
    for (int y = 0; y < nsplit; y++) s0 += o[y * stride];  // split order: same sum as before
    tot[t][a] = s0;
  }
  __syncthreads();
  if (i < p.m && a == 0) {
    double acc[NACC];
#pragma unroll
    for (int q = 0; q < NACC; q++) acc[q] = tot[t][q];
    nbody_store<KIND, NR>(p, i, acc);
  }
}

static bool g_pool_set[64] = {};

template <int KIND, int NR>
static int launch_nbody(NbodyParams p, cudaStream_t s, ShiftTable st = {}) {
  if (p.m == 0) return SCB_OK;
  constexpr int NACC = Traits<KIND, NR>::nacc;
  const int64_t n_eff = p.n - (Traits<KIND, NR>::coupling ? p.skip_len : 0);
  const int64_t ctas_x = ceil_div(p.m, 256 * TPT);
  // One balanced wave: every CTA does the same amount of work, so the source range is split until the
  // grid just fills the resident-CTA capacity of the device (a CTA keeps at least one source tile).
  // NB_Z, NB_VECTOR and NB_VECPOT passes of several sets split as the single-set pass does, whatever their own
  // occupancy: the split fixes the summation order, so every set of a multi-set call has the bits of a one-set
  // call.  NB_COUPLING_T passes split as the one-set NB_COUPLING pass does, for the same reason.
  constexpr int CAP_NR = (KIND == NB_Z || KIND == NB_VECTOR || KIND == NB_VECPOT || KIND == NB_COUPLING_T) ? 1 : NR;
  constexpr int CAP_KIND = KIND == NB_COUPLING_T ? NB_COUPLING : KIND;
  static int capacity = 0;  // per instantiation; all devices of a node are identical
  if (capacity == 0) {
    int per_sm = 0, sms = 0, dev = 0;
    SCB_CUDA(cudaGetDevice(&dev));
    SCB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nbody_kernel<CAP_KIND, CAP_NR>, 256, 0));
    SCB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    capacity = per_sm * sms > 0 ? per_sm * sms : 148;
  }
  int64_t split = capacity / ctas_x;
  const int64_t max_split = n_eff / kTile;
  if (split > max_split) split = max_split;
  if (split < 1) split = 1;
  p.chunk = n_eff > 0 ? ceil_div(n_eff, split) : 1;
  split = n_eff > 0 ? ceil_div(n_eff, p.chunk) : 1;
  p.partial = nullptr;
  if (split > 1) {
    int dev = 0;
    SCB_CUDA(cudaGetDevice(&dev));
    if (!g_pool_set[dev & 63]) {  // keep freed scratch in the stream-ordered pool instead of returning it to the OS
      cudaMemPool_t pool;
      SCB_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
      uint64_t keep = ~0ull;
      SCB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
      g_pool_set[dev & 63] = true;
    }
    SCB_CUDA(cudaMallocAsync(&p.partial, sizeof(double) * (size_t)(split * p.m * NACC), s));
  }
  nbody_kernel<KIND, NR><<<dim3((unsigned)ctas_x, (unsigned)split), 256, 0, s>>>(p, st);
  SCB_LAUNCH_CHECK();
  if (split > 1) {
    nbody_reduce_kernel<KIND, NR><<<(unsigned)ceil_div(p.m, 128 / NACC), 128, 0, s>>>(p, (int)split);
    SCB_LAUNCH_CHECK();
    SCB_CUDA(cudaFreeAsync(p.partial, s));
  }
  return SCB_OK;
}

// ---------------------------------------------------------------------------------------
// Many right-hand sides: the same sum as NB_KERNEL, as a GEMM on the fp64 tensor cores whose A
// operand (the kernel matrix) is never stored -- every lane evaluates the r^-3 entry that the
// mma.sync m8n8k4 A fragment assigns to it (row = target g, k = source t) and feeds it straight
// to DMMA against a shared-memory tile of the payload matrix  P[j][r] = w_j v[j][r].
// CTA: 64 targets (8 warps x one 8-row tile) x NC = 8 CT right-hand sides; sources in tiles of 32,
// double-buffered through registers.  One r^-3 evaluation now serves NC columns.
// ---------------------------------------------------------------------------------------
constexpr int kGemmSrc = 32;

__device__ __forceinline__ void dmma_nb(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

template <int CT>
__global__ void __launch_bounds__(256) kernel_gemm_kernel(NbodyParams p) {
  constexpr int NC = 8 * CT;
  constexpr int PLD = NC + 4;                    // conflict-free B fragments (ld % 16 == 4)
  constexpr int PER = kGemmSrc * NC / 256;       // payload entries staged per thread
  __shared__ double sx[2][kGemmSrc], sy[2][kGemmSrc];
  __shared__ double sp[2][kGemmSrc * PLD];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t i = blockIdx.x * 64ll + warp * 8 + g;
  const bool active = i < p.m;
  const double tx = active ? p.tgt[2 * i] : 0.0, ty = active ? p.tgt[2 * i + 1] : 0.0;
  double acc[CT][2];
#pragma unroll
  for (int c = 0; c < CT; c++) acc[c][0] = acc[c][1] = 0.0;

  double rpay[PER], rx = 0.0, ry = 0.0;
  auto fetch = [&](int64_t base) {
    // sources past the end: far away and weightless
    if (tid < kGemmSrc) {
      const int64_t j = base + tid;
      const int64_t js = j < p.n ? (p.src_idx ? p.src_idx[j] : j) : -1;
      rx = js >= 0 ? p.src[2 * js] : 1e100;
      ry = js >= 0 ? p.src[2 * js + 1] : 1e100;
    }
#pragma unroll
    for (int q = 0; q < PER; q++) {
      const int e = tid + 256 * q;
      const int r = e / NC, c = e % NC;
      const int64_t j = base + r;
      double v = 0.0;
      if (j < p.n) {
        const int64_t js = p.src_idx ? p.src_idx[j] : j;
        v = p.area[js] * p.J[js * p.ldv + p.rhs0 + c];
      }
      rpay[q] = v;
    }
  };
  auto stash = [&](int buf) {
    if (tid < kGemmSrc) {
      sx[buf][tid] = rx;
      sy[buf][tid] = ry;
    }
#pragma unroll
    for (int q = 0; q < PER; q++) {
      const int e = tid + 256 * q;
      sp[buf][(e / NC) * PLD + e % NC] = rpay[q];
    }
  };
  fetch(0);
  stash(0);
  __syncthreads();
  int buf = 0;
  for (int64_t base = 0; base < p.n; base += kGemmSrc) {
    const bool more = base + kGemmSrc < p.n;
    if (more) fetch(base + kGemmSrc);
#pragma unroll
    for (int ks = 0; ks < kGemmSrc / 4; ks++) {
      const int j = ks * 4 + t;
      const double dx = tx - sx[buf][j], dy = ty - sy[buf][j];
      const double r2 = dx * dx + dy * dy;
      double k3 = inv_r3(r2);
      k3 = r2 > 0.0 ? k3 : 0.0;  // q_ii = 0 (distance.py:104-105)
#pragma unroll
      for (int c = 0; c < CT; c++) dmma_nb(acc[c][0], acc[c][1], k3, sp[buf][j * PLD + c * 8 + g]);
    }
    if (more) stash(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }
  if (!active) return;
  const double pf = p.prefactor;
#pragma unroll
  for (int c = 0; c < CT; c++)
#pragma unroll
    for (int e = 0; e < 2; e++) {
      double* o = p.out + i * p.ldv + p.rhs0 + c * 8 + 2 * t + e;
      *o = p.accumulate ? *o + pf * acc[c][e] : pf * acc[c][e];
    }
}

template <int CT>
static int launch_kernel_gemm(const NbodyParams& p, cudaStream_t s) {
  kernel_gemm_kernel<CT><<<(unsigned)ceil_div(p.m, 64), 256, 0, s>>>(p);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

// ---------------------------------------------------------------------------------------
// Within-film field of many current-density sets (solve_film.py:415-437) on the fp64 tensor cores:
//   out[i, s] = sum_j a_j (Jx[j,s] dy - Jy[j,s] dx) r_ij^-3   as a GEMM with K = 2 n_src,
//   A[i, 2j] = dy r^-3,  A[i, 2j+1] = -dx r^-3  (dx = x_i - x_j),   P[2j + c, s] = a_j J[j, s, c].
// A is evaluated in the mma.sync m8n8k4 A-fragment layout and never stored.  A k-step covers two
// sources (lanes t = 0, 1: source 0, components x, y; t = 2, 3: source 1), so a group of four sources
// spans two k-steps: lane (g, t) evaluates r^-3 of target g and source t of the group once, and each
// k-step fetches the (source, component) entry its fragment needs from lane (g, 2h + t/2) by shuffle.
// One r^-3 then serves NC = 8 CT sets.  CTA: 64 targets (8 warps x 8 rows); sources in tiles of 16
// (32 k rows), double-buffered through registers as in kernel_gemm_kernel.  Every output is summed
// by one lane in a fixed order: no atomics, bit-reproducible.
// ---------------------------------------------------------------------------------------
constexpr int kWfSrc = 16;

template <int CT>
__global__ void __launch_bounds__(256, 2) within_film_gemm_kernel(NbodyParams p) {
  constexpr int NC = 8 * CT;
  constexpr int KR = 2 * kWfSrc;                 // k rows of a source tile
  constexpr int PLD = NC + 4;                    // conflict-free B fragments (ld % 16 == 4)
  constexpr int PER = KR * NC / 256;             // payload entries staged per thread
  __shared__ double sx[2][kWfSrc], sy[2][kWfSrc];
  __shared__ double sp[2][KR * PLD];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t i = blockIdx.x * 64ll + warp * 8 + g;
  const bool active = i < p.m;
  const double tx = active ? p.tgt[2 * i] : 0.0, ty = active ? p.tgt[2 * i + 1] : 0.0;
  double acc[CT][2];
#pragma unroll
  for (int c = 0; c < CT; c++) acc[c][0] = acc[c][1] = 0.0;

  double rpay[PER], rx = 0.0, ry = 0.0;
  auto fetch = [&](int64_t base) {
    // sources past the end: far away and weightless
    if (tid < kWfSrc) {
      const int64_t j = base + tid;
      rx = j < p.n ? p.src[2 * j] : 1e100;
      ry = j < p.n ? p.src[2 * j + 1] : 1e100;
    }
#pragma unroll
    for (int q = 0; q < PER; q++) {
      const int e = tid + 256 * q;               // (source, set, component), component fastest: coalesced
      const int64_t j = base + e / (2 * NC);
      rpay[q] = j < p.n ? p.area[j] * p.J[j * p.ldv + 2 * p.rhs0 + e % (2 * NC)] : 0.0;
    }
  };
  auto stash = [&](int buf) {
    if (tid < kWfSrc) {
      sx[buf][tid] = rx;
      sy[buf][tid] = ry;
    }
#pragma unroll
    for (int q = 0; q < PER; q++) {
      const int e = tid + 256 * q;
      const int jl = e / (2 * NC), sc = e % (2 * NC);
      sp[buf][(2 * jl + (sc & 1)) * PLD + (sc >> 1)] = rpay[q];
    }
  };
  fetch(0);
  stash(0);
  __syncthreads();
  int buf = 0;
  for (int64_t base = 0; base < p.n; base += kWfSrc) {
    const bool more = base + kWfSrc < p.n;
    if (more) fetch(base + kWfSrc);
#pragma unroll
    for (int kk = 0; kk < kWfSrc / 4; kk++) {
      const int j = kk * 4 + t;
      const double dx = tx - sx[buf][j], dy = ty - sy[buf][j];
      const double k3 = inv_r3(fma(dx, dx, dy * dy));
      const double ay = k3 * dy, ax = -(k3 * dx);
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int from = (lane & ~3) | (2 * h + (t >> 1));
        const double vy = __shfl_sync(0xffffffffu, ay, from);
        const double vx = __shfl_sync(0xffffffffu, ax, from);
        const double a = (t & 1) ? vx : vy;
        const int krow = (kk * 2 + h) * 4 + t;
#pragma unroll
        for (int c = 0; c < CT; c++) dmma_nb(acc[c][0], acc[c][1], a, sp[buf][krow * PLD + c * 8 + g]);
      }
    }
    if (more) stash(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }
  if (!active) return;
  const double pf = p.prefactor;
#pragma unroll
  for (int c = 0; c < CT; c++)
#pragma unroll
    for (int e = 0; e < 2; e++) p.out[i * p.ldo + p.rhs0 + c * 8 + 2 * t + e] = pf * acc[c][e];
}

// Sets per pass of within_film_gemm_kernel in scb_biot_savart_within_film.  Measured on a B200 (1000 W limit)
// at 20k vertices x 40k triangles against 8-set CUDA-core passes: 0.71x at 16 sets, 1.01x at 32, 1.17x at 64
// (DESIGN.md 4.5), so only full 64-set passes use it.
constexpr int64_t kWithinFilmGemmSets = 64;

// out[i, rhs0..] (+)= prefactor * sum_{j in src, r_ij > 0} q_ij w_j v[j, rhs0..]
int nbody_kernel_sum(int64_t m, const double* tgt, int64_t n, const double* src,
                     const int64_t* src_idx, const double* w, const double* v, int64_t ldv,
                     int64_t nrhs, double prefactor, double* out, int accumulate, cudaStream_t s) {
  NbodyParams p{};
  p.m = m; p.tgt = tgt; p.n = n; p.src = src; p.src_idx = src_idx; p.area = w; p.J = v;
  p.ldv = ldv; p.ldo = ldv; p.prefactor = prefactor; p.out = out; p.accumulate = accumulate;
  int64_t r = 0;
  // 16 or more right-hand sides: tensor-core GEMM against the on-the-fly kernel matrix
  while (v != nullptr && nrhs - r >= 16) {
    p.rhs0 = r;
    int rc;
    if (nrhs - r >= 64) { rc = launch_kernel_gemm<8>(p, s); r += 64; }
    else if (nrhs - r >= 32) { rc = launch_kernel_gemm<4>(p, s); r += 32; }
    else { rc = launch_kernel_gemm<2>(p, s); r += 16; }
    if (rc) return rc;
  }
  while (r < nrhs) {
    p.rhs0 = r;
    int rc;
    if (nrhs - r >= 8) { rc = launch_nbody<NB_KERNEL, 8>(p, s); r += 8; }
    else if (nrhs - r >= 4) { rc = launch_nbody<NB_KERNEL, 4>(p, s); r += 4; }
    else if (nrhs - r >= 2) { rc = launch_nbody<NB_KERNEL, 2>(p, s); r += 2; }
    else { rc = launch_nbody<NB_KERNEL, 1>(p, s); r += 1; }
    if (rc) return rc;
  }
  return SCB_OK;
}

// out[i, j] = |XA_i - XB_j| (or its square): one thread per 2 adjacent columns, 128-bit stores
template <int DIM>
__global__ void cdist_kernel(int squared, int64_t m, const double* __restrict__ XA, int64_t n,
                             const double* __restrict__ XB, double* __restrict__ out) {
  const int64_t j = 2 * (blockIdx.x * (int64_t)blockDim.x + threadIdx.x);
  const int64_t i0 = blockIdx.y * 16ll;
  if (j >= n) return;
  double b[2][3];
#pragma unroll
  for (int k = 0; k < 2; k++)
#pragma unroll
    for (int d = 0; d < DIM; d++) b[k][d] = (j + k < n) ? XB[(j + k) * DIM + d] : 0.0;
  for (int64_t i = i0; i < i0 + 16 && i < m; i++) {
    double v[2];
#pragma unroll
    for (int k = 0; k < 2; k++) {
      double r2 = 0.0;
#pragma unroll
      for (int d = 0; d < DIM; d++) {
        const double t = XA[i * DIM + d] - b[k][d];
        r2 = fma(t, t, r2);
      }
      v[k] = squared ? r2 : sqrt(r2);
    }
    if (j + 1 < n && (n % 2 == 0)) {
      *reinterpret_cast<double2*>(out + i * n + j) = make_double2(v[0], v[1]);
    } else {
      out[i * n + j] = v[0];
      if (j + 1 < n) out[i * n + j + 1] = v[1];
    }
  }
}

__global__ void qdw_finish_kernel(int64_t n, const double* __restrict__ C, double* qdw) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) qdw[i] = C[i] + qdw[i];
}

}  // namespace scb

using namespace scb;

extern "C" int scb_kernel_diagonal(int64_t n, const double* sites, const double* weights,
                                   const double* C, double* qdw, scb_stream_t stream) {
  SCB_CHECK_ARG(n > 0, "n must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = nbody_kernel_sum(n, sites, n, sites, nullptr, weights, nullptr, 1, 1, kOneOver4Pi, qdw, 0, s);
  if (rc) return rc;
  qdw_finish_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(n, C, qdw);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}

extern "C" int scb_biot_savart(int kind, int64_t m, const double* tgt, int64_t n, const double* src,
                               const double* area, const double* J, double dz, double prefactor,
                               int64_t nsets, double* out, scb_stream_t stream) {
  SCB_CHECK_ARG(m >= 0 && n >= 0 && nsets >= 1, "bad sizes");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t ocomp = kind == SCB_BS_VECTOR ? 3 : (kind == SCB_BS_VECTOR_POTENTIAL ? 2 : 1);
  if (m == 0) return SCB_OK;  // no evaluation points: nothing to write
  if (n == 0) {               // no sources: the field vanishes
    SCB_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)(m * ocomp * nsets), s));
    return SCB_OK;
  }
  if (kind == SCB_BS_BOUNDARY) {
    // edge geometry shared by every set: strengths area[n, nsets], out[m, nsets]
    NbodyParams p{};
    p.m = m; p.tgt = tgt; p.n = n; p.src = src; p.area = area; p.J = J;
    p.ldv = nsets; p.ldo = nsets; p.prefactor = prefactor; p.out = out;
    for (int64_t k = 0; k < nsets;) {
      p.rhs0 = k;
      int rc;
      if (nsets - k >= 8) { rc = launch_nbody<NB_BOUNDARY, 8>(p, s); k += 8; }
      else if (nsets - k >= 4) { rc = launch_nbody<NB_BOUNDARY, 4>(p, s); k += 4; }
      else if (nsets - k >= 2) { rc = launch_nbody<NB_BOUNDARY, 2>(p, s); k += 2; }
      else { rc = launch_nbody<NB_BOUNDARY, 1>(p, s); k += 1; }
      if (rc) return rc;
    }
    return SCB_OK;
  }
  int64_t k = 0;
  while (k < nsets) {
    NbodyParams p{};
    p.m = m; p.tgt = tgt; p.n = n; p.src = src; p.area = area; p.J = J + k * n * 2;
    p.dz2 = dz * dz; p.prefactor = prefactor; p.out = out + k * m * ocomp;
    int rc;
    int64_t step = 1;
    switch (kind) {
      case SCB_BS_FILM_TO_FILM:
        // current-density sets that share the geometry are evaluated together (one r^-3 per pair)
        if (nsets - k >= 8) { rc = launch_nbody<NB_FILM_TO_FILM, 8>(p, s); step = 8; }
        else if (nsets - k >= 4) { rc = launch_nbody<NB_FILM_TO_FILM, 4>(p, s); step = 4; }
        else if (nsets - k >= 2) { rc = launch_nbody<NB_FILM_TO_FILM, 2>(p, s); step = 2; }
        else rc = launch_nbody<NB_FILM_TO_FILM, 1>(p, s);
        break;
      case SCB_BS_Z:  // as film-to-film: one r^-3 per pair serves every set of a pass
        if (nsets - k >= 8) { rc = launch_nbody<NB_Z, 8>(p, s); step = 8; }
        else if (nsets - k >= 4) { rc = launch_nbody<NB_Z, 4>(p, s); step = 4; }
        else if (nsets - k >= 2) { rc = launch_nbody<NB_Z, 2>(p, s); step = 2; }
        else rc = launch_nbody<NB_Z, 1>(p, s);
        break;
      case SCB_BS_VECTOR:  // one r^-3 per pair for the sets of a pass
        if (nsets - k >= 8) { rc = launch_nbody<NB_VECTOR, 8>(p, s); step = 8; }
        else if (nsets - k >= 4) { rc = launch_nbody<NB_VECTOR, 4>(p, s); step = 4; }
        else if (nsets - k >= 2) { rc = launch_nbody<NB_VECTOR, 2>(p, s); step = 2; }
        else rc = launch_nbody<NB_VECTOR, 1>(p, s);
        break;
      case SCB_BS_VECTOR_POTENTIAL:  // one r^-1 per pair for the sets of a pass
        if (nsets - k >= 8) { rc = launch_nbody<NB_VECPOT, 8>(p, s); step = 8; }
        else if (nsets - k >= 4) { rc = launch_nbody<NB_VECPOT, 4>(p, s); step = 4; }
        else if (nsets - k >= 2) { rc = launch_nbody<NB_VECPOT, 2>(p, s); step = 2; }
        else rc = launch_nbody<NB_VECPOT, 1>(p, s);
        break;
      default: set_error("scb_biot_savart: unknown kind %d", kind); return SCB_ERR_INVALID;
    }
    if (rc) return rc;
    k += step;
  }
  return SCB_OK;
}

extern "C" int scb_film_coupling(int64_t m, const double* tgt, double tgt_z, int64_t n, const double* src,
                                 const double* area, const double* J, int64_t skip_lo, int64_t skip_hi,
                                 double prefactor, int64_t nsets, double* out, scb_stream_t stream) {
  SCB_CHECK_ARG(m >= 0 && n >= 0 && nsets >= 1, "bad sizes");
  SCB_CHECK_ARG(0 <= skip_lo && skip_lo <= skip_hi && skip_hi <= n, "skip range must lie inside [0, n]");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0) return SCB_OK;
  if (skip_lo == 0 && skip_hi == n) {  // no other film: the field vanishes
    SCB_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)(m * nsets), s));
    return SCB_OK;
  }
  NbodyParams p{};
  p.m = m; p.tgt = tgt; p.tgt_z = tgt_z; p.n = n; p.src = src; p.area = area; p.J = J; p.ldv = 2 * nsets;
  p.skip_lo = skip_lo; p.skip_len = skip_hi - skip_lo; p.prefactor = prefactor; p.out = out; p.ldo = nsets;
  p.sld = 3;
  int64_t k = 0;
  while (k < nsets) {
    p.rhs0 = k;
    int rc;
    if (nsets - k >= 8) { rc = launch_nbody<NB_COUPLING, 8>(p, s); k += 8; }
    else if (nsets - k >= 4) { rc = launch_nbody<NB_COUPLING, 4>(p, s); k += 4; }
    else if (nsets - k >= 2) { rc = launch_nbody<NB_COUPLING, 2>(p, s); k += 2; }
    else { rc = launch_nbody<NB_COUPLING, 1>(p, s); k += 1; }
    if (rc) return rc;
  }
  return SCB_OK;
}

extern "C" int scb_film_coupling_translated(int64_t m, const double* tgt, double tgt_z, int64_t n, const double* src,
                                            const double* area, const double* J, int64_t skip_lo, int64_t skip_hi,
                                            double prefactor, int64_t nsets, int64_t dst, const int32_t* src_film,
                                            int64_t nfilms, const double* shift, double* out, scb_stream_t stream) {
  SCB_CHECK_ARG(m >= 0 && n >= 0 && nsets >= 1, "bad sizes");
  SCB_CHECK_ARG(0 <= skip_lo && skip_lo <= skip_hi && skip_hi <= n, "skip range must lie inside [0, n]");
  SCB_CHECK_ARG(nfilms >= 1 && 0 <= dst && dst < nfilms, "dst must lie in [0, nfilms)");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0) return SCB_OK;
  if (skip_lo == 0 && skip_hi == n) {  // no other film: the field vanishes
    SCB_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)(m * nsets), s));
    return SCB_OK;
  }
  NbodyParams p{};
  p.m = m; p.tgt = tgt; p.tgt_z = tgt_z; p.n = n; p.src = src; p.area = area; p.J = J; p.ldv = 2 * nsets;
  p.skip_lo = skip_lo; p.skip_len = skip_hi - skip_lo; p.prefactor = prefactor; p.out = out; p.ldo = nsets;
  p.sld = 3;
  const ShiftTable st{src_film, shift, nfilms, dst};
  // No r^-3 to share between sets: a pass of several sets only saves target loads and launches.  Passes
  // of 2 (80 registers, 20 KB of shared memory: 3 CTAs per SM); a 4-set pass needs 136 registers, one CTA.
  int64_t k = 0;
  while (k < nsets) {
    p.rhs0 = k;
    int rc;
    if (nsets - k >= 2) { rc = launch_nbody<NB_COUPLING_T, 2>(p, s, st); k += 2; }
    else { rc = launch_nbody<NB_COUPLING_T, 1>(p, s, st); k += 1; }
    if (rc) return rc;
  }
  return SCB_OK;
}

extern "C" int scb_biot_savart_within_film(int64_t m, const double* tgt, int64_t n, const double* src,
                                           const double* area, const double* J, double prefactor, int64_t nsets,
                                           double* out, scb_stream_t stream) {
  SCB_CHECK_ARG(m >= 0 && n >= 0 && nsets >= 1, "bad sizes");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0) return SCB_OK;
  if (n == 0) {
    SCB_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)(m * nsets), s));
    return SCB_OK;
  }
  NbodyParams p{};
  p.m = m; p.tgt = tgt; p.n = n; p.src = src; p.area = area; p.J = J; p.ldv = 2 * nsets; p.ldo = nsets;
  p.sld = 2; p.prefactor = prefactor; p.out = out;  // (NB_COUPLING: sources in the target plane, nothing skipped)
  int64_t k = 0;
  for (; nsets - k >= kWithinFilmGemmSets; k += kWithinFilmGemmSets) {
    p.rhs0 = k;
    within_film_gemm_kernel<kWithinFilmGemmSets / 8><<<(unsigned)ceil_div(m, 64), 256, 0, s>>>(p);
    SCB_LAUNCH_CHECK();
  }
  while (k < nsets) {
    p.rhs0 = k;
    int rc;
    if (nsets - k >= 8) { rc = launch_nbody<NB_COUPLING, 8>(p, s); k += 8; }
    else if (nsets - k >= 4) { rc = launch_nbody<NB_COUPLING, 4>(p, s); k += 4; }
    else if (nsets - k >= 2) { rc = launch_nbody<NB_COUPLING, 2>(p, s); k += 2; }
    else { rc = launch_nbody<NB_COUPLING, 1>(p, s); k += 1; }
    if (rc) return rc;
  }
  return SCB_OK;
}

extern "C" int scb_cdist(int dim, int squared, int64_t m, const double* XA, int64_t n, const double* XB,
                         double* out, scb_stream_t stream) {
  SCB_CHECK_ARG(dim == 2 || dim == 3, "dim must be 2 or 3");
  SCB_CHECK_ARG(m >= 0 && n >= 0, "bad sizes");
  if (m == 0 || n == 0) return SCB_OK;
  dim3 grid((unsigned)ceil_div(ceil_div(n, 2), 128), (unsigned)ceil_div(m, 16));
  if (dim == 2)
    cdist_kernel<2><<<grid, 128, 0, (cudaStream_t)stream>>>(squared, m, XA, n, XB, out);
  else
    cdist_kernel<3><<<grid, 128, 0, (cudaStream_t)stream>>>(squared, m, XA, n, XB, out);
  SCB_LAUNCH_CHECK();
  return SCB_OK;
}
