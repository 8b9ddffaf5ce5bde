// normals.cu -- per-point normals of a point cloud on the device: K-neighbourhood PCA with pytorch3d's sign
// disambiguation (reference: utils/ops.py:62-72 estimate_normal over pytorch3d.ops.estimate_pointcloud_normals, used
// by gs/gaussian_splatting.py:1186-1196 and :1423-1466 for cfg.normal_as_rgb, and by utils/relight.py).
//
// pytorch3d gathers the [N, K, 3] neighbourhoods of a brute-force knn_points, forms [N, 3, 3] covariances and runs a
// batched eigensolver.  Here one fused kernel does all of it per point, nothing of size [N, K] is written unless the
// backward needs the neighbour indices:
//
//   knn_build_index   the uniform grid of knn.cu (stats -> grid -> keys -> radix sort -> gather -> cell table)
//   k_normals<KT>     (KT = 16, 32; k_normals_smem for 64) one thread per point, in cell order: knn_query<KT> (knn_grid.cuh, exact, ties by index) ->
//                     mean + covariance -> 3x3 Jacobi -> smallest eigenvector -> sign (normals.cuh)
//   k_normals_bwd<KT> one thread per point: the same frame from the saved indices, dL/dC from the eigenvector
//                     perturbation, scattered to the K neighbours with atomics
//
// KT in {16, 32, 64} bounds K; the neighbour lists live in registers, for KT = 64 in shared memory
// (k_normals_smem).  This file is compiled with -fmad=false
// (gsgen_b200/build.py) so the kernels evaluate normals.cuh exactly as the g++ host build does.
#include "gsb200_common.cuh"
#include "kernels.cuh"
#include "knn_grid.cuh"
#include "normals.cuh"

namespace gsb {

// neighbour lists as normals.cuh reads them: a column of a per-block shared array (stride S), or a row of the [n, K]
// index array in global memory
template <int S>
struct NrmStridedNbr {
  const int32_t* base;
  __device__ __forceinline__ int32_t operator[](int k) const { return base[k * S]; }
};
struct NrmRowNbr {
  const int32_t* base;
  __device__ __forceinline__ int32_t operator[](int k) const { return __ldg(base + k); }
};

template <int KT>
__global__ void __launch_bounds__(128, 2)
k_normals(uint32_t n, const float* __restrict__ pts, const int32_t* __restrict__ order,
          const KnnGrid* __restrict__ grid, const KnnPt* __restrict__ sorted, const int32_t* __restrict__ cell_start,
          int K, int disambiguate, float* __restrict__ normals, int32_t* __restrict__ nbr_out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint32_t j = (uint32_t)order[t];
  const KnnGrid G = *grid;
  const float p[3] = {pts[3 * (size_t)j], pts[3 * (size_t)j + 1], pts[3 * (size_t)j + 2]};
  int32_t bi[KT];
  {
    float bd[KT];
    knn_query<KT>(G, sorted, cell_start, p[0], p[1], p[2], bd, bi);
  }
  if (nbr_out) {
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) nbr_out[(size_t)j * K + k] = bi[k];
  }
  NrmFrame f;
  float nv[3];
  nrm_estimate<KT>(pts, bi, K, p, disambiguate != 0, nv, f);
  normals[3 * (size_t)j] = nv[0];
  normals[3 * (size_t)j + 1] = nv[1];
  normals[3 * (size_t)j + 2] = nv[2];
}

// K in (32, 64]: 64 (distance, index) pairs in registers spill (255 registers, measured), so the sorted list lives in
// shared memory instead -- 64 threads x 64 slots x 8 B = 32 KB per block, column layout (slot k of thread t at
// [k * 64 + t]: the lanes of a warp hit 32 consecutive banks).  Same search, same insertion order, same result.
constexpr int kNrmSmemBlock = 64;
__global__ void __launch_bounds__(kNrmSmemBlock)
k_normals_smem(uint32_t n, const float* __restrict__ pts, const int32_t* __restrict__ order,
               const KnnGrid* __restrict__ grid, const KnnPt* __restrict__ sorted,
               const int32_t* __restrict__ cell_start, int K, int disambiguate, float* __restrict__ normals,
               int32_t* __restrict__ nbr_out) {
  constexpr int KT = kNrmMaxK, S = kNrmSmemBlock;
  __shared__ float s_d[KT * S];
  __shared__ int32_t s_i[KT * S];
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint32_t j = (uint32_t)order[t];
  const KnnGrid G = *grid;
  const float p[3] = {pts[3 * (size_t)j], pts[3 * (size_t)j + 1], pts[3 * (size_t)j + 2]};
  KnnStridedList<KT, S> L{s_d + threadIdx.x, s_i + threadIdx.x, 0.f, 0};
  L.init();
  knn_walk(G, sorted, cell_start, p[0], p[1], p[2], L);
  const NrmStridedNbr<S> bi{s_i + threadIdx.x};
  if (nbr_out) {
    for (int k = 0; k < K; ++k) nbr_out[(size_t)j * K + k] = bi[k];
  }
  NrmFrame f;
  float nv[3];
  nrm_estimate<KT>(pts, bi, K, p, disambiguate != 0, nv, f);
  normals[3 * (size_t)j] = nv[0];
  normals[3 * (size_t)j + 1] = nv[1];
  normals[3 * (size_t)j + 2] = nv[2];
}

template <int KT>
__global__ void __launch_bounds__(128)
k_normals_bwd(uint32_t n, const float* __restrict__ pts, int K, int disambiguate, const int32_t* __restrict__ nbr,
              const float* __restrict__ grad_normals, float* __restrict__ grad_points) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const float g[3] = {grad_normals[3 * (size_t)j], grad_normals[3 * (size_t)j + 1], grad_normals[3 * (size_t)j + 2]};
  if (g[0] == 0.f && g[1] == 0.f && g[2] == 0.f) return;
  const float p[3] = {pts[3 * (size_t)j], pts[3 * (size_t)j + 1], pts[3 * (size_t)j + 2]};
  const NrmRowNbr bi{nbr + (size_t)j * K};
  NrmFrame f;
  float nv[3];
  nrm_estimate<KT>(pts, bi, K, p, false, nv, f);
  const float sgn = disambiguate ? nrm_sign<KT>(pts, bi, K, p, nv) : 1.f;
  float M[6];
  if (!nrm_grad_matrix(f, sgn, g, (float)K, M)) return;
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (k < K) {
      float e[3];
      nrm_centred(pts, bi[k], p, f, e);
      float* o = grad_points + 3 * (size_t)bi[k];
      atomicAdd(o, M[0] * e[0] + M[1] * e[1] + M[2] * e[2]);
      atomicAdd(o + 1, M[1] * e[0] + M[3] * e[1] + M[4] * e[2]);
      atomicAdd(o + 2, M[2] * e[0] + M[4] * e[1] + M[5] * e[2]);
    }
  }
}

static int normals_check(uint32_t n, int K) {
  GSB_CHECK(K >= 1 && K <= kNrmMaxK, GSB200_ERR_UNSUPPORTED, "estimate_normals: K = %d outside [1, %d]", K, kNrmMaxK);
  GSB_CHECK(n <= 0x7fffffffu / 4u, GSB200_ERR_INVALID, "estimate_normals: %u points exceed the int32 index range", n);
  GSB_CHECK(n == 0 || (uint32_t)K <= n, GSB200_ERR_INVALID,
            "estimate_normals: K = %d neighbours requested from %u points", K, n);
  return GSB200_OK;
}

int normals_device(gsb200_ctx* ctx, const float* points, uint32_t n, int K, int disambiguate, float* normals,
                   int32_t* nbr_idx, cudaStream_t st) {
  int rc;
  if ((rc = normals_check(n, K))) return rc;
  if (n == 0) return GSB200_OK;
  GSB_CHECK(points != nullptr, GSB200_ERR_INVALID, "estimate_normals: points is NULL");
  GSB_CHECK(normals != nullptr, GSB200_ERR_INVALID, "estimate_normals: normals is NULL");
  KnnIndex ix;
  if ((rc = knn_build_index(ctx, points, n, &ix, st))) return rc;
  const unsigned blocks = (n + 127) / 128;
  if (K <= 16)
    k_normals<16><<<blocks, 128, 0, st>>>(n, points, ix.order, ix.grid, ix.sorted, ix.cell_start, K, disambiguate,
                                          normals, nbr_idx);
  else if (K <= 32)
    k_normals<32><<<blocks, 128, 0, st>>>(n, points, ix.order, ix.grid, ix.sorted, ix.cell_start, K, disambiguate,
                                          normals, nbr_idx);
  else
    k_normals_smem<<<(n + kNrmSmemBlock - 1) / kNrmSmemBlock, kNrmSmemBlock, 0, st>>>(
        n, points, ix.order, ix.grid, ix.sorted, ix.cell_start, K, disambiguate, normals, nbr_idx);
  GSB_LAUNCH_CHECK();
  return GSB200_OK;
}

int normals_backward_device(const float* points, uint32_t n, int K, int disambiguate, const int32_t* nbr_idx,
                            const float* grad_normals, float* grad_points, cudaStream_t st) {
  int rc;
  if ((rc = normals_check(n, K))) return rc;
  if (n == 0) return GSB200_OK;
  GSB_CHECK(points != nullptr && nbr_idx != nullptr && grad_normals != nullptr && grad_points != nullptr,
            GSB200_ERR_INVALID, "estimate_normals_backward: NULL argument");
  const unsigned blocks = (n + 127) / 128;
  if (K <= 16)
    k_normals_bwd<16><<<blocks, 128, 0, st>>>(n, points, K, disambiguate, nbr_idx, grad_normals, grad_points);
  else if (K <= 32)
    k_normals_bwd<32><<<blocks, 128, 0, st>>>(n, points, K, disambiguate, nbr_idx, grad_normals, grad_points);
  else
    k_normals_bwd<64><<<blocks, 128, 0, st>>>(n, points, K, disambiguate, nbr_idx, grad_normals, grad_points);
  GSB_LAUNCH_CHECK();
  return GSB200_OK;
}

}  // namespace gsb

using namespace gsb;

extern "C" {

int gsb200_estimate_normals(gsb200_ctx* ctx, const float* points, uint32_t n_points, int32_t K, int32_t disambiguate,
                            float* normals, int32_t* nbr_idx, gsb200_stream stream) {
  GSB_CHECK(ctx != nullptr, GSB200_ERR_INVALID, "null context");
  GSB_CUDA(cudaSetDevice(ctx->device));
  return normals_device(ctx, points, n_points, (int)K, (int)disambiguate, normals, nbr_idx, (cudaStream_t)stream);
}

int gsb200_estimate_normals_backward(gsb200_ctx* ctx, const float* points, uint32_t n_points, int32_t K,
                                     int32_t disambiguate, const int32_t* nbr_idx, const float* grad_normals,
                                     float* grad_points, gsb200_stream stream) {
  GSB_CHECK(ctx != nullptr, GSB200_ERR_INVALID, "null context");
  GSB_CUDA(cudaSetDevice(ctx->device));
  return normals_backward_device(points, n_points, (int)K, (int)disambiguate, nbr_idx, grad_normals, grad_points,
                                 (cudaStream_t)stream);
}

}  // extern "C"
