// knn_grid.cuh -- exact K-nearest-neighbour search over the Gaussian means on a uniform grid, written as host+device
// inline functions so the SAME search runs in the sm_100a kernel (knn.cu) and in the CPU unit test (tests/hostmath, g++).
//
// Reference behaviour replaced (SURVEY §8(f)-2, compactness-based densification and the neighbour penalties):
//   utils/ops.py:103-114  nearest_neighbor(mean)            -> knn_points(mean, mean, K=2), column 1
//   utils/ops.py:117-134  K_nearest_neighbors(mean, K, ...) -> knn_points(query, mean, K), columns 1..K-1
// called by gs/gaussian_splatting.py:682-691 (densify_by_compatness), :1032-1046 (NN_penalty_loss), :1048-1094
// (compat_penalty_loss).  `knn_points` is pytorch3d.ops.knn_points -- a third-party dependency that is neither vendored
// in the reference nor pinned in its requirements.txt (utils/ops.py:7-14 imports it optionally) and is absent here.  Its
// published contract is restated: for every query the K points with the smallest SQUARED Euclidean distance, sorted
// ascending, returned as (dists [.,K] fp32, idx [.,K] int64); a query that is itself one of the points is its own first
// neighbour (distance 0), which is why the reference drops column 0.  Tie order among equal distances is not part of
// that contract; here it is fixed (smaller point index first) so the result is deterministic and CPU == GPU bit for bit.
//
// Search: points are bucketed into cubic cells (edge h, ~2 points per cell); a query visits the cells at Chebyshev
// distance r = 0, 1, 2, ... from its own cell.  After shell r everything inside the cube of (2r+1)^3 cells is known,
// so the K-th best distance is final as soon as it is smaller than the distance from the query to the nearest face of
// that cube that still has cells behind it (minus a rounding slack).  Cells are numbered x-fastest, so the x-extent of a
// shell row is ONE contiguous run of the cell-sorted point array.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "gsb200_math.cuh"

// (GSB_HD is `static` on the host, which member functions cannot be)
#if defined(__CUDACC__)
#define GSB_HD_MEMBER __host__ __device__ __forceinline__
#else
#define GSB_HD_MEMBER inline
#endif

namespace gsb {

constexpr int kKnnMaxK = 32;
constexpr int kKnnMaxAxisCells = 1024;

struct alignas(16) KnnPt {
  float x, y, z;
  int32_t i;  // index of the point in the caller's array
};

struct KnnGrid {
  float lo[3];
  float h, inv_h;
  float slack;     // bound on the position error of a cell assignment (fp32 rounding of (x - lo) * inv_h)
  int32_t g[3];    // cells per axis, >= 1
  int32_t cells;   // g[0] * g[1] * g[2] <= max_cells
};

GSB_HD int knn_imax(int a, int b) { return a > b ? a : b; }
GSB_HD int knn_imin(int a, int b) { return a < b ? a : b; }

// order-preserving map float -> uint32 (for atomicMin / atomicMax of a bounding box)
GSB_HD uint32_t knn_f2ord(float f) {
  uint32_t u;
#if defined(__CUDA_ARCH__)
  u = __float_as_uint(f);
#else
  memcpy(&u, &f, 4);
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
GSB_HD float knn_ord2f(uint32_t u) {
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  float f;
#if defined(__CUDA_ARCH__)
  f = __uint_as_float(u);
#else
  memcpy(&f, &u, 4);
#endif
  return f;
}

// The box the grid spans: the bounding box of the points, clipped per axis to mean +- 3 sigma.  Points (and queries)
// outside it fall into the border cells (knn_cell_axis clamps) -- the search stays exact for ANY box, a border face just
// never bounds the covered radius -- so a few far-away floaters do not coarsen the cells of the whole scene.
GSB_HD void knn_robust_box(const float* bmin, const float* bmax, const double* sum, const double* sumsq, uint32_t n,
                           float* lo, float* hi) {
  for (int a = 0; a < 3; ++a) {
    lo[a] = bmin[a];
    hi[a] = bmax[a];
    if (n > 0) {
      const double m = sum[a] / (double)n;
      double var = sumsq[a] / (double)n - m * m;
      if (!(var > 0.0)) var = 0.0;
      const double sd = sqrt(var);
      const float l3 = (float)(m - 3.0 * sd), h3 = (float)(m + 3.0 * sd);
      if (l3 > lo[a] && l3 <= hi[a]) lo[a] = l3;   // comparisons are false for NaN / inf statistics: box unchanged
      if (h3 < hi[a] && h3 >= lo[a]) hi[a] = h3;
    }
  }
}

// Grid over the box [lo, hi] of n points: about two points per cell for a roughly isotropic cloud, at most
// `max_cells` cells (the caller sized the cell table for that) and kKnnMaxAxisCells per axis.
GSB_HD KnnGrid knn_make_grid(const float* lo, const float* hi, uint32_t n, uint32_t max_cells) {
  KnnGrid G;
  float ext[3], emax = 0.f, amax = 0.f;
  for (int a = 0; a < 3; ++a) {
    G.lo[a] = lo[a];
    ext[a] = hi[a] - lo[a];
    if (!(ext[a] > 0.f)) ext[a] = 0.f;  // also catches NaN (empty / degenerate input)
    emax = fmaxf(emax, ext[a]);
    amax = fmaxf(amax, fmaxf(fabsf(lo[a]), fabsf(hi[a])));
  }
  float h = 1.0f;
  if (emax > 0.f) h = emax / fmaxf(1.0f, cbrtf(0.5f * (float)n));  // isotropic start; grown until the budgets hold
  bool converged = false;
  for (int it = 0; it < 96 && !converged; ++it) {
    G.h = h;
    G.inv_h = 1.0f / h;
    double c = 1.0;
    bool axis_ok = true;
    for (int a = 0; a < 3; ++a) {
      const float fa = floorf(ext[a] * G.inv_h) + 1.0f;  // the formula knn_cell_axis clamps against
      if (!(fa <= (float)kKnnMaxAxisCells)) axis_ok = false;
      G.g[a] = axis_ok ? (int32_t)fa : kKnnMaxAxisCells;
      c *= (double)G.g[a];
    }
    G.cells = (int32_t)(c < 2.0e9 ? c : 2.0e9);
    converged = axis_ok && c <= (double)(max_cells < 1u ? 1u : max_cells);
    h *= 1.25f;
  }
  if (!converged) {  // non-finite bounding box: one cell, i.e. an exhaustive scan per query (still exact)
    G.h = 1.0f; G.inv_h = 1.0f;
    G.g[0] = G.g[1] = G.g[2] = 1;
    G.cells = 1;
  }
  G.slack = 4e-6f * (amax + emax) + 1e-30f;
  return G;
}

GSB_HD int knn_cell_axis(float x, float lo, float inv_h, int g) {
  const float f = floorf((x - lo) * inv_h);
  int c = (f >= (float)g) ? g - 1 : ((f > 0.f) ? (int)f : 0);  // NaN -> 0
  return c;
}
GSB_HD uint32_t knn_cell_id(const KnnGrid& G, float x, float y, float z) {
  const int cx = knn_cell_axis(x, G.lo[0], G.inv_h, G.g[0]);
  const int cy = knn_cell_axis(y, G.lo[1], G.inv_h, G.g[1]);
  const int cz = knn_cell_axis(z, G.lo[2], G.inv_h, G.g[2]);
  return (uint32_t)((cz * G.g[1] + cy) * G.g[0] + cx);
}

// squared distance as the sum of three separately rounded squares (no FMA contraction: same value on CPU and GPU)
GSB_HD float knn_dist2(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = ax - bx, dy = ay - by, dz = az - bz;
  return add_rn(add_rn(mul_rn(dx, dx), mul_rn(dy, dy)), mul_rn(dz, dz));
}

// sorted insert into the K best (ascending by (distance, index))
template <int K> GSB_HD void knn_insert(float (&bd)[K], int32_t (&bi)[K], float d, int32_t i) {
  if (!(d < bd[K - 1] || (d == bd[K - 1] && i < bi[K - 1]))) return;
  bd[K - 1] = d;
  bi[K - 1] = i;
#pragma unroll
  for (int j = K - 1; j > 0; --j) {
    const bool sw = (bd[j] < bd[j - 1]) || (bd[j] == bd[j - 1] && bi[j] < bi[j - 1]);
    if (sw) {
      const float td = bd[j]; bd[j] = bd[j - 1]; bd[j - 1] = td;
      const int32_t ti = bi[j]; bi[j] = bi[j - 1]; bi[j - 1] = ti;
    }
  }
}

// The shell walk of the search.  pts: the n points sorted by cell id; cell_start[c] .. cell_start[c+1]: the points of
// cell c (cell_start has G.cells + 1 entries).  L: the K best so far -- L.insert(d, i) offers a candidate, L.kth() is
// the current K-th best distance (+inf while fewer than K are known).  Returns the number of shells visited.
template <class List>
GSB_HD int knn_walk(const KnnGrid& G, const KnnPt* pts, const int32_t* cell_start, float qx, float qy, float qz,
                    List& L) {
  const float q[3] = {qx, qy, qz};
  int c[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) c[a] = knn_cell_axis(q[a], G.lo[a], G.inv_h, G.g[a]);
  int rmax = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) rmax = knn_imax(rmax, knn_imax(c[a], G.g[a] - 1 - c[a]));
  int r = 0;
  for (;; ++r) {
    const int z0 = knn_imax(c[2] - r, 0), z1 = knn_imin(c[2] + r, G.g[2] - 1);
    const int y0 = knn_imax(c[1] - r, 0), y1 = knn_imin(c[1] + r, G.g[1] - 1);
    const int x0 = knn_imax(c[0] - r, 0), x1 = knn_imin(c[0] + r, G.g[0] - 1);
    for (int z = z0; z <= z1; ++z) {
      const bool zedge = (z == c[2] - r) || (z == c[2] + r);
      for (int y = y0; y <= y1; ++y) {
        const bool edge = zedge || (y == c[1] - r) || (y == c[1] + r);
        const int row = (z * G.g[1] + y) * G.g[0];
        // on a face of the cube the whole x-extent belongs to the shell (one contiguous run); elsewhere only its two ends
        const int nseg = edge ? 1 : 2;
        for (int sgm = 0; sgm < nseg; ++sgm) {
          int xa, xb;
          if (edge) { xa = x0; xb = x1; }
          else if (sgm == 0) { xa = xb = c[0] - r; if (xa < 0) continue; }
          else { xa = xb = c[0] + r; if (xa > G.g[0] - 1 || r == 0) continue; }
          const int s0 = cell_start[row + xa], s1 = cell_start[row + xb + 1];
          for (int s = s0; s < s1; ++s) {
            const KnnPt p = pts[s];
            L.insert(knn_dist2(p.x, p.y, p.z, qx, qy, qz), p.i);
          }
        }
      }
    }
    if (r >= rmax) break;  // the cube covers the grid
    // distance to the nearest face of the cube that still has cells behind it
    float dmin = INFINITY;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (c[a] - r > 0) dmin = fminf(dmin, q[a] - (G.lo[a] + (float)(c[a] - r) * G.h));
      if (c[a] + r < G.g[a] - 1) dmin = fminf(dmin, (G.lo[a] + (float)(c[a] + r + 1) * G.h) - q[a]);
    }
    const float safe = dmin - G.slack;
    if (safe > 0.f && L.kth() < safe * safe) break;  // strict: an uncovered point cannot even tie
  }
  return r + 1;
}

// the K best in registers (sorted insert network of knn_insert)
template <int K>
struct KnnRegList {
  float (&bd)[K];
  int32_t (&bi)[K];
  GSB_HD_MEMBER void insert(float d, int32_t i) { knn_insert<K>(bd, bi, d, i); }
  GSB_HD_MEMBER float kth() const { return bd[K - 1]; }
};

// The K nearest points of (qx, qy, qz) (see knn_walk).  On return bd / bi hold the neighbours in ascending order;
// slots beyond the number of points are (+inf, -1).  Returns the number of shells visited (statistics).
template <int K>
GSB_HD int knn_query(const KnnGrid& G, const KnnPt* pts, const int32_t* cell_start, float qx, float qy, float qz,
                     float (&bd)[K], int32_t (&bi)[K]) {
#pragma unroll
  for (int j = 0; j < K; ++j) { bd[j] = INFINITY; bi[j] = -1; }
  KnnRegList<K> L{bd, bi};
  return knn_walk(G, pts, cell_start, qx, qy, qz, L);
}

// The same K best as a strided list in memory (slot j at d[j * S], i[j * S]; shared memory on the device, where K
// pairs would not fit in registers): insertion by shifting from the end, the order of knn_insert.
template <int K, int S>
struct KnnStridedList {
  float* d;
  int32_t* i;
  float wd;    // the K-th best, cached
  int32_t wi;
  GSB_HD_MEMBER void init() {
    for (int j = 0; j < K; ++j) { d[j * S] = INFINITY; i[j * S] = -1; }
    wd = INFINITY; wi = -1;
  }
  GSB_HD_MEMBER void insert(float dd, int32_t ii) {
    if (!(dd < wd || (dd == wd && ii < wi))) return;
    int j = K - 1;
    while (j > 0) {
      const float pd = d[(j - 1) * S];
      const int32_t pi = i[(j - 1) * S];
      if (!(dd < pd || (dd == pd && ii < pi))) break;
      d[j * S] = pd; i[j * S] = pi;
      --j;
    }
    d[j * S] = dd; i[j * S] = ii;
    wd = d[(K - 1) * S]; wi = i[(K - 1) * S];
  }
  GSB_HD_MEMBER float kth() const { return wd; }
};

}  // namespace gsb
