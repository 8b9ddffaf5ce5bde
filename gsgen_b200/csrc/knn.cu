// knn.cu -- exact K-nearest neighbours of the Gaussian means on the device (SURVEY §8(f)-2: the neighbour search behind
// compactness-based densification and the NN / compactness penalties; reference: utils/ops.py:103-134 over
// pytorch3d.ops.knn_points, called from gs/gaussian_splatting.py:682-691, :1032-1094).
//
// pytorch3d's knn_points is a brute-force O(N^2) kernel (every query scans every point).  Here the points are bucketed
// into a uniform grid and every query walks cell shells until its K-th best distance is provably final
// (knn_grid.cuh -- the search itself is host+device code, the CPU test-suite runs the same function):
//
//   k_knn_stats    bounding box (ordered-uint atomics) + per-axis sum / sum of squares (double atomics), one pass
//   k_knn_grid     one thread: box clipped to mean +- 3 sigma -> KnnGrid in device memory (no host round trip)
//   k_knn_keys     cell id per point
//   cub::DeviceRadixSort (cell id -> point index), bits_for(max_cells) key bits
//   k_knn_gather   points in cell order as 16-byte records (x, y, z, index)
//   k_knn_cells    cell_start[c] = lower_bound(sorted keys, c), c = 0 .. cells
//   k_knn_query<K> one thread per query; self-queries are issued in cell order so a warp's lanes walk the same cells
//
// Everything is enqueued on the caller's stream; nothing synchronises.  Work: N * (27 cells * ~2 points) distance
// evaluations for a uniform cloud instead of N^2.
#include <cub/device/device_radix_sort.cuh>

#include "gsb200_common.cuh"
#include "kernels.cuh"
#include "knn_grid.cuh"

namespace gsb {

struct KnnStats {
  uint32_t bmin[3], bmax[3];  // knn_f2ord encoded
  double sum[3], sumsq[3];
};

__global__ void __launch_bounds__(256)
k_knn_stats_init(KnnStats* st) {
  if (threadIdx.x < 3) {
    st->bmin[threadIdx.x] = 0xffffffffu;
    st->bmax[threadIdx.x] = 0u;
    st->sum[threadIdx.x] = 0.0;
    st->sumsq[threadIdx.x] = 0.0;
  }
}

__global__ void __launch_bounds__(256)
k_knn_stats(uint32_t n, const float* __restrict__ pts, KnnStats* st) {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  double s[3] = {0, 0, 0}, ss[3] = {0, 0, 0};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float v = pts[3 * (size_t)i + a];
      lo[a] = fminf(lo[a], v);
      hi[a] = fmaxf(hi[a], v);
      s[a] += (double)v;
      ss[a] += (double)v * (double)v;
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
      hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
      s[a] += __shfl_xor_sync(0xffffffffu, s[a], o);
      ss[a] += __shfl_xor_sync(0xffffffffu, ss[a], o);
    }
  }
  // block level: the 8 warp results meet in shared memory, one thread per (axis, quantity) folds them and issues the
  // block's ONE atomic for it (measured round 2 with an atomic per warp: 108 us for 1M points -- 113 k atomics on 12
  // addresses serialise in L2)
  __shared__ float s_lo[8][3], s_hi[8][3];
  __shared__ double s_s[8][3], s_ss[8][3];
  const int warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { s_lo[warp][a] = lo[a]; s_hi[warp][a] = hi[a]; s_s[warp][a] = s[a]; s_ss[warp][a] = ss[a]; }
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    const int a = threadIdx.x % 3, what = threadIdx.x / 3;  // 0 min, 1 max, 2 sum, 3 sum of squares
    if (what == 0) {
      float m = INFINITY;
      for (int w = 0; w < nwarp; ++w) m = fminf(m, s_lo[w][a]);
      if (m < INFINITY) atomicMin(&st->bmin[a], knn_f2ord(m));   // (INFINITY: no non-NaN value seen on this axis)
    } else if (what == 1) {
      float m = -INFINITY;
      for (int w = 0; w < nwarp; ++w) m = fmaxf(m, s_hi[w][a]);
      if (m > -INFINITY) atomicMax(&st->bmax[a], knn_f2ord(m));
    } else if (what == 2) {
      double t = 0.0;
      for (int w = 0; w < nwarp; ++w) t += s_s[w][a];
      atomicAdd(&st->sum[a], t);
    } else {
      double t = 0.0;
      for (int w = 0; w < nwarp; ++w) t += s_ss[w][a];
      atomicAdd(&st->sumsq[a], t);
    }
  }
}

__global__ void k_knn_grid(uint32_t n, uint32_t max_cells, const KnnStats* st, KnnGrid* grid) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float bmin[3], bmax[3], lo[3], hi[3];
  double sum[3], sumsq[3];
  for (int a = 0; a < 3; ++a) {
    bmin[a] = knn_ord2f(st->bmin[a]);
    bmax[a] = knn_ord2f(st->bmax[a]);
    if (!(bmin[a] <= bmax[a])) { bmin[a] = 0.f; bmax[a] = 0.f; }  // no finite point: any box is exact
    sum[a] = st->sum[a];
    sumsq[a] = st->sumsq[a];
  }
  knn_robust_box(bmin, bmax, sum, sumsq, n, lo, hi);
  *grid = knn_make_grid(lo, hi, n, max_cells);
}

__global__ void __launch_bounds__(256)
k_knn_keys(uint32_t n, const float* __restrict__ pts, const KnnGrid* __restrict__ grid, uint32_t* __restrict__ keys,
           int32_t* __restrict__ vals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const KnnGrid G = *grid;
  keys[i] = knn_cell_id(G, pts[3 * (size_t)i], pts[3 * (size_t)i + 1], pts[3 * (size_t)i + 2]);
  vals[i] = (int32_t)i;
}

__global__ void __launch_bounds__(256)
k_knn_gather(uint32_t n, const float* __restrict__ pts, const int32_t* __restrict__ perm, KnnPt* __restrict__ sorted) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const int32_t i = perm[s];
  KnnPt p;
  p.x = pts[3 * (size_t)i];
  p.y = pts[3 * (size_t)i + 1];
  p.z = pts[3 * (size_t)i + 2];
  p.i = i;
  sorted[s] = p;
}

__global__ void __launch_bounds__(256)
k_knn_cells(uint32_t n, const uint32_t* __restrict__ skeys, const KnnGrid* __restrict__ grid,
            int32_t* __restrict__ cell_start) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > (uint32_t)grid->cells) return;
  uint32_t lo = 0, hi = n;  // first position whose key is >= c
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (skeys[mid] < c) lo = mid + 1; else hi = mid;
  }
  cell_start[c] = (int32_t)lo;
}

// One thread per query.  order != nullptr: thread t answers query order[t] (the points query themselves, in cell
// order, so neighbouring lanes walk the same cells and their loads coalesce / broadcast).
template <int KT>
__global__ void __launch_bounds__(128, (KT <= 16 ? 4 : 2))
k_knn_query(uint32_t nq, const float* __restrict__ queries, const int32_t* __restrict__ order,
            const KnnGrid* __restrict__ grid, const KnnPt* __restrict__ sorted, const int32_t* __restrict__ cell_start,
            int K, int64_t* __restrict__ idx_out, float* __restrict__ d2_out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nq) return;
  const uint32_t j = order ? (uint32_t)order[t] : t;
  const KnnGrid G = *grid;
  float bd[KT];
  int32_t bi[KT];
  knn_query<KT>(G, sorted, cell_start, queries[3 * (size_t)j], queries[3 * (size_t)j + 1], queries[3 * (size_t)j + 2],
                bd, bi);
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (k < K) {
      idx_out[(size_t)j * K + k] = (int64_t)bi[k];
      if (d2_out) d2_out[(size_t)j * K + k] = bd[k];
    }
  }
}

static int knn_bits_for(uint32_t n) {
  int b = 1;
  while (b < 32 && (1ull << b) < (unsigned long long)n) ++b;
  return b;
}

// The grid over `n` points on `st` (stats -> grid -> cell keys -> radix sort -> gather -> cell table), in the
// context's knn_* buffers.  Shared by the neighbour search below and the normal estimate (normals.cu).
int knn_build_index(gsb200_ctx* ctx, const float* points, uint32_t n, KnnIndex* out, cudaStream_t st) {
  // the cell table is sized on the host from N alone (the grid itself is chosen on the device)
  const uint32_t max_cells = 4u * n + 64u;
  int rc;
  if ((rc = ctx->knn_small.reserve(sizeof(KnnStats) + sizeof(KnnGrid) + 64))) return rc;
  KnnStats* stats = ctx->knn_small.as<KnnStats>();
  KnnGrid* grid = reinterpret_cast<KnnGrid*>(reinterpret_cast<unsigned char*>(ctx->knn_small.p) +
                                             ((sizeof(KnnStats) + 15) / 16) * 16);
  const size_t n1 = n ? n : 1;
  for (int k = 0; k < 2; ++k) {
    if ((rc = ctx->knn_keys[k].reserve(n1 * 4))) return rc;
    if ((rc = ctx->knn_vals[k].reserve(n1 * 4))) return rc;
  }
  if ((rc = ctx->knn_pts.reserve(n1 * sizeof(KnnPt)))) return rc;
  if ((rc = ctx->knn_cells.reserve(((size_t)max_cells + 1) * 4))) return rc;

  k_knn_stats_init<<<1, 32, 0, st>>>(stats);
  GSB_LAUNCH_CHECK();
  const unsigned blocks = (n + 255) / 256;
  if (n) {
    const unsigned sblocks = blocks < (unsigned)ctx->sm_count * 8 ? blocks : (unsigned)ctx->sm_count * 8;
    k_knn_stats<<<sblocks, 256, 0, st>>>(n, points, stats);
    GSB_LAUNCH_CHECK();
  }
  k_knn_grid<<<1, 32, 0, st>>>(n, max_cells, stats, grid);
  GSB_LAUNCH_CHECK();
  uint32_t* k0 = ctx->knn_keys[0].as<uint32_t>();
  uint32_t* k1 = ctx->knn_keys[1].as<uint32_t>();
  int32_t* v0 = ctx->knn_vals[0].as<int32_t>();
  int32_t* v1 = ctx->knn_vals[1].as<int32_t>();
  if (n) {
    k_knn_keys<<<blocks, 256, 0, st>>>(n, points, grid, k0, v0);
    GSB_LAUNCH_CHECK();
    const int end_bit = knn_bits_for(max_cells);
    size_t bytes = 0;
    GSB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, k0, k1, v0, v1, (int)n, 0, end_bit, st));
    if ((rc = ctx->cub_tmp.reserve(bytes))) return rc;
    GSB_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, bytes, k0, k1, v0, v1, (int)n, 0, end_bit, st));
    k_knn_gather<<<blocks, 256, 0, st>>>(n, points, v1, ctx->knn_pts.as<KnnPt>());
    GSB_LAUNCH_CHECK();
  }
  k_knn_cells<<<(max_cells + 1 + 255) / 256, 256, 0, st>>>(n, k1, grid, ctx->knn_cells.as<int32_t>());
  GSB_LAUNCH_CHECK();
  out->grid = grid;
  out->sorted = ctx->knn_pts.as<KnnPt>();
  out->cell_start = ctx->knn_cells.as<int32_t>();
  out->order = v1;
  return GSB200_OK;
}

int knn_device(gsb200_ctx* ctx, const float* points, uint32_t n, const float* queries, uint32_t nq, int K,
               int64_t* idx_out, float* d2_out, cudaStream_t st) {
  GSB_CHECK(K >= 1 && K <= kKnnMaxK, GSB200_ERR_UNSUPPORTED, "knn: K = %d outside [1, %d]", K, kKnnMaxK);
  GSB_CHECK(n <= 0x7fffffffu / 4u, GSB200_ERR_INVALID, "knn: %u points exceed the int32 index range", n);
  const bool self = (queries == nullptr);
  if (self) { queries = points; nq = n; }
  if (nq == 0) return GSB200_OK;
  GSB_CHECK(points != nullptr || n == 0, GSB200_ERR_INVALID, "knn: points is NULL");
  GSB_CHECK(idx_out != nullptr, GSB200_ERR_INVALID, "knn: idx_out is NULL");
  KnnIndex ix;
  int rc;
  if ((rc = knn_build_index(ctx, points, n, &ix, st))) return rc;
  const int32_t* order = self ? ix.order : nullptr;
  const unsigned qblocks = (nq + 127) / 128;
  const KnnGrid* grid = ix.grid;
  const KnnPt* sp = ix.sorted;
  const int32_t* cs = ix.cell_start;
  if (K <= 2) k_knn_query<2><<<qblocks, 128, 0, st>>>(nq, queries, order, grid, sp, cs, K, idx_out, d2_out);
  else if (K <= 4) k_knn_query<4><<<qblocks, 128, 0, st>>>(nq, queries, order, grid, sp, cs, K, idx_out, d2_out);
  else if (K <= 8) k_knn_query<8><<<qblocks, 128, 0, st>>>(nq, queries, order, grid, sp, cs, K, idx_out, d2_out);
  else if (K <= 16) k_knn_query<16><<<qblocks, 128, 0, st>>>(nq, queries, order, grid, sp, cs, K, idx_out, d2_out);
  else k_knn_query<32><<<qblocks, 128, 0, st>>>(nq, queries, order, grid, sp, cs, K, idx_out, d2_out);
  GSB_LAUNCH_CHECK();
  return GSB200_OK;
}

}  // namespace gsb

using namespace gsb;

extern "C" {

int gsb200_knn(gsb200_ctx* ctx, const float* points, uint32_t n_points, const float* queries, uint32_t n_queries,
               int32_t K, int64_t* idx, float* dist2, gsb200_stream stream) {
  GSB_CHECK(ctx != nullptr, GSB200_ERR_INVALID, "null context");
  GSB_CUDA(cudaSetDevice(ctx->device));
  return knn_device(ctx, points, n_points, queries, n_queries, (int)K, idx, dist2, (cudaStream_t)stream);
}

}  // extern "C"
