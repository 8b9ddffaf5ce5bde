// normals.cuh -- per-point normal of a K-neighbourhood (local PCA), written as host+device inline functions so the SAME
// arithmetic runs in the sm_100a kernels (normals.cu) and in the CPU unit test (tests/hostmath/normals_host.cpp, g++).
//
// Reference behaviour replaced: utils/ops.py:62-72 estimate_normal(pos, neighborhood_size, disambiguate_directions) ->
// pytorch3d.ops.estimate_pointcloud_normals, used by gs/gaussian_splatting.py:1186-1196 (`normal`, normal_type
// "estimated") for cfg.normal_as_rgb and by utils/relight.py.  pytorch3d (0.7) is third party and absent here; its
// contract (estimate_pointcloud_local_coord_frames + _disambiguate_vector_directions) is restated from its documented
// behaviour, it could not be run against this code:
//   neighbourhood  knn_points(p, p, K): the K nearest points, the point itself included (ties: smaller index first)
//   covariance     C = (1/K) sum_k (x_k - mu)(x_k - mu)^T, mu = mean_k x_k
//   normal         the eigenvector of the smallest eigenvalue of C
//   disambiguation proj_k = n . (x_k - p) relative to the point p itself; n_pos = #{proj_k > 0}; flip n if n_pos < K/2
// Ours (pytorch3d leaves them undefined): a zero (or non-finite) covariance -- coincident neighbours, K = 1 -- gives
// n = (0, 0, 1) before the flip and a zero gradient.
//
// Arithmetic: every quantity is formed relative to the query point p (d_k = x_k - p), which keeps the fp32 covariance
// free of the cancellation |x|^2 - |mu|^2 would suffer far from the origin.  The 3x3 eigenproblem is solved by cyclic
// Jacobi rotations on C / max|C_ij| (only +, *, /, sqrt: correctly rounded on both compilers, and normals.cu is built
// with -fmad=false, so the host build and the kernels agree bit for bit).
#pragma once
#include <math.h>
#include <stdint.h>

#include "gsb200_math.cuh"

namespace gsb {

constexpr int kNrmMaxK = 64;
constexpr int kNrmSweeps = 12;           // Jacobi sweeps at most (3x3: converged to fp32 after ~5)
constexpr float kNrmGapGuard = 1e-6f;    // backward: eigen gaps <= 1e-6 * max(lambda_2, 1e-30) contribute zero

// One neighbourhood's PCA.  lam ascending, v[i][c] = component i of the unit eigenvector c (of C, unscaled).
struct NrmFrame {
  float m[3];      // mean of d_k = x_k - p
  float lam[3];
  float v[3][3];
  bool degenerate;  // zero / non-finite covariance: no eigenvectors
};

// one Jacobi rotation zeroing a[P][Q]; R is the third index
template <int P, int Q, int R>
GSB_HD void nrm_jacobi_rot(float (&a)[3][3], float (&v)[3][3], bool late) {
  const float apq = a[P][Q];
  if (apq == 0.f) return;
  const float g = 100.f * fabsf(apq);
  if (late && fabsf(a[P][P]) + g == fabsf(a[P][P]) && fabsf(a[Q][Q]) + g == fabsf(a[Q][Q])) {
    a[P][Q] = a[Q][P] = 0.f;  // below the rounding of both diagonal entries
    return;
  }
  const float h = a[Q][Q] - a[P][P];
  float t;
  if (fabsf(h) + g == fabsf(h)) {
    t = apq / h;  // tan of the rotation angle ~ apq / h when |h| >> |apq| (theta^2 would overflow)
  } else {
    const float theta = 0.5f * h / apq;
    t = 1.f / (fabsf(theta) + sqrtf(theta * theta + 1.f));
    if (theta < 0.f) t = -t;
  }
  const float c = 1.f / sqrtf(t * t + 1.f), s = t * c, tau = s / (1.f + c), th = t * apq;
  a[P][P] -= th;
  a[Q][Q] += th;
  a[P][Q] = a[Q][P] = 0.f;
  const float arp = a[R][P], arq = a[R][Q];
  a[R][P] = a[P][R] = arp - s * (arq + tau * arp);
  a[R][Q] = a[Q][R] = arq + s * (arp - tau * arq);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const float vrp = v[r][P], vrq = v[r][Q];
    v[r][P] = vrp - s * (vrq + tau * vrp);
    v[r][Q] = vrq + s * (vrp - tau * vrq);
  }
}

// sort eigenpair I before J when lam[J] < lam[I]
template <int I, int J>
GSB_HD void nrm_order(float (&lam)[3], float (&v)[3][3]) {
  if (lam[J] < lam[I]) {
    const float t = lam[I]; lam[I] = lam[J]; lam[J] = t;
#pragma unroll
    for (int r = 0; r < 3; ++r) { const float u = v[r][I]; v[r][I] = v[r][J]; v[r][J] = u; }
  }
}

// PCA of the K nearest neighbours nbr[0..K) (indices into pts [n,3]) of the point p.  KT: compile-time bound of K;
// nbr: anything indexable -- a register array, a shared-memory column or a row of the saved [n, K] indices.
template <int KT, class Nbr>
GSB_HD void nrm_frame(const float* pts, const Nbr& nbr, int K, const float p[3], NrmFrame& f) {
  float s[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (k < K) {
      const int32_t i = nbr[k];
#pragma unroll
      for (int a = 0; a < 3; ++a) s[a] += pts[3 * (size_t)i + a] - p[a];
    }
  }
  const float fk = (float)K;
#pragma unroll
  for (int a = 0; a < 3; ++a) f.m[a] = s[a] / fk;
  float c[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // xx xy xz yy yz zz
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (k < K) {
      const int32_t i = nbr[k];
      float e[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) e[a] = (pts[3 * (size_t)i + a] - p[a]) - f.m[a];
      c[0] += e[0] * e[0]; c[1] += e[0] * e[1]; c[2] += e[0] * e[2];
      c[3] += e[1] * e[1]; c[4] += e[1] * e[2]; c[5] += e[2] * e[2];
    }
  }
  float scale = 0.f;
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    c[q] = c[q] / fk;
    scale = fmaxf(scale, fabsf(c[q]));
  }
  // (fmaxf drops NaN: a NaN entry is caught by the finiteness test of the sum)
  const float probe = c[0] + c[1] + c[2] + c[3] + c[4] + c[5];
  f.degenerate = !(scale > 0.f && scale < INFINITY && probe - probe == 0.f);
  if (f.degenerate) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      f.lam[a] = 0.f;
#pragma unroll
      for (int b = 0; b < 3; ++b) f.v[a][b] = (a == b) ? 1.f : 0.f;
    }
    return;
  }
  float A[3][3];
  A[0][0] = c[0] / scale; A[0][1] = A[1][0] = c[1] / scale; A[0][2] = A[2][0] = c[2] / scale;
  A[1][1] = c[3] / scale; A[1][2] = A[2][1] = c[4] / scale; A[2][2] = c[5] / scale;
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) f.v[a][b] = (a == b) ? 1.f : 0.f;
  for (int sweep = 0; sweep < kNrmSweeps; ++sweep) {
    if (fabsf(A[0][1]) + fabsf(A[0][2]) + fabsf(A[1][2]) == 0.f) break;
    const bool late = sweep >= 4;
    nrm_jacobi_rot<0, 1, 2>(A, f.v, late);
    nrm_jacobi_rot<0, 2, 1>(A, f.v, late);
    nrm_jacobi_rot<1, 2, 0>(A, f.v, late);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) f.lam[a] = A[a][a] * scale;
  nrm_order<0, 1>(f.lam, f.v);
  nrm_order<1, 2>(f.lam, f.v);
  nrm_order<0, 1>(f.lam, f.v);
}

// the normal of a frame before disambiguation: unit eigenvector of the smallest eigenvalue, (0, 0, 1) if degenerate
GSB_HD void nrm_unit(const NrmFrame& f, float n[3]) {
  if (f.degenerate) { n[0] = 0.f; n[1] = 0.f; n[2] = 1.f; return; }
  const float l = sqrtf(f.v[0][0] * f.v[0][0] + f.v[1][0] * f.v[1][0] + f.v[2][0] * f.v[2][0]);
  n[0] = f.v[0][0] / l; n[1] = f.v[1][0] / l; n[2] = f.v[2][0] / l;
}

// pytorch3d's _disambiguate_vector_directions for one vector: -1 if fewer than half of the neighbours lie strictly on
// the positive side of n (measured from p), else +1
template <int KT, class Nbr>
GSB_HD float nrm_sign(const float* pts, const Nbr& nbr, int K, const float p[3], const float n[3]) {
  int pos = 0;
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (k < K) {
      const int32_t i = nbr[k];
      const float proj = n[0] * (pts[3 * (size_t)i] - p[0]) + n[1] * (pts[3 * (size_t)i + 1] - p[1]) +
                         n[2] * (pts[3 * (size_t)i + 2] - p[2]);
      pos += proj > 0.f ? 1 : 0;
    }
  }
  return (2 * pos < K) ? -1.f : 1.f;
}

// Forward for one point: n (unit), flipped by the disambiguation when asked.
template <int KT, class Nbr>
GSB_HD void nrm_estimate(const float* pts, const Nbr& nbr, int K, const float p[3], bool disambiguate,
                         float n[3], NrmFrame& f) {
  nrm_frame<KT>(pts, nbr, K, p, f);
  nrm_unit(f, n);
  if (disambiguate) {
    const float sg = nrm_sign<KT>(pts, nbr, K, p, n);
    n[0] *= sg; n[1] *= sg; n[2] *= sg;
  }
}

// Backward for one point, neighbour set and sign held constant.  With n = s v0 and the first-order perturbation
// dv0 = sum_{j=1,2} v_j (v_j^T dC v0) / (lam0 - lam_j), dL = g^T dn = tr(G^T dC) for
// G = s sum_j (g . v_j) / (lam0 - lam_j) v_j v0^T; C = (1/K) sum_k e_k e_k^T with e_k = x_k - mu gives
// dL/dx_k = (1/K)(G + G^T) e_k (the mu term cancels: sum_k e_k = 0).  Returns M = (G + G^T) / K as xx xy xz yy yz zz;
// the caller adds M e_k to the gradient of neighbour k.  Gaps |lam0 - lam_j| <= 1e-6 max(lam2, 1e-30) contribute zero
// (torch.linalg.eigh's backward would return inf / NaN there); a degenerate frame has M = 0.  Returns false if M = 0.
GSB_HD bool nrm_grad_matrix(const NrmFrame& f, float sgn, const float g[3], float K, float M[6]) {
#pragma unroll
  for (int q = 0; q < 6; ++q) M[q] = 0.f;
  if (f.degenerate) return false;
  const float floor_ = kNrmGapGuard * fmaxf(f.lam[2], 1e-30f);
  float G[3][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
  bool any = false;
#pragma unroll
  for (int j = 1; j < 3; ++j) {
    const float gap = f.lam[0] - f.lam[j];
    if (!(fabsf(gap) > floor_)) continue;
    const float w = sgn * (g[0] * f.v[0][j] + g[1] * f.v[1][j] + g[2] * f.v[2][j]) / gap;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) G[a][b] += w * f.v[a][j] * f.v[b][0];
    any = true;
  }
  if (!any) return false;
  M[0] = (G[0][0] + G[0][0]) / K; M[1] = (G[0][1] + G[1][0]) / K; M[2] = (G[0][2] + G[2][0]) / K;
  M[3] = (G[1][1] + G[1][1]) / K; M[4] = (G[1][2] + G[2][1]) / K; M[5] = (G[2][2] + G[2][2]) / K;
  return true;
}

// e_k = (x_k - p) - m, the centred neighbour the gradient matrix acts on
GSB_HD void nrm_centred(const float* pts, int32_t i, const float p[3], const NrmFrame& f, float e[3]) {
#pragma unroll
  for (int a = 0; a < 3; ++a) e[a] = (pts[3 * (size_t)i + a] - p[a]) - f.m[a];
}

}  // namespace gsb
