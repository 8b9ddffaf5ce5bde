// normals_host.cpp -- TEST INFRASTRUCTURE.  g++ build of the normal estimate's per-point math
// (gsgen_b200/csrc/normals.cuh) over the same grid search the kernels use (knn_grid.cuh), so the CPU test-suite can
// check it against a float64 reference and the GPU test-suite can compare the kernels with it.  Never loaded by the
// product path.
#include "../../gsgen_b200/csrc/knn_grid.cuh"
#include "../../gsgen_b200/csrc/normals.cuh"

#include <algorithm>
#include <vector>

using namespace gsb;

namespace {

struct Index {
  KnnGrid G;
  std::vector<KnnPt> sp;
  std::vector<int32_t> cell_start;
  std::vector<int> perm;
};

// knn_build_index on the host: bounding box -> knn_make_grid -> cell ids -> stable sort by cell -> cell table
void build_index(int n, const float* pts, Index& ix) {
  float bmin[3] = {INFINITY, INFINITY, INFINITY}, bmax[3] = {-INFINITY, -INFINITY, -INFINITY}, lo[3], hi[3];
  double sum[3] = {0, 0, 0}, sumsq[3] = {0, 0, 0};
  for (int i = 0; i < n; ++i)
    for (int a = 0; a < 3; ++a) {
      const float v = pts[3 * i + a];
      bmin[a] = fminf(bmin[a], v); bmax[a] = fmaxf(bmax[a], v);
      sum[a] += (double)v; sumsq[a] += (double)v * (double)v;
    }
  for (int a = 0; a < 3; ++a)
    if (!(bmin[a] <= bmax[a])) { bmin[a] = 0.f; bmax[a] = 0.f; }
  knn_robust_box(bmin, bmax, sum, sumsq, (uint32_t)n, lo, hi);
  ix.G = knn_make_grid(lo, hi, (uint32_t)n, 4u * (uint32_t)n + 64u);
  std::vector<uint32_t> key(n);
  ix.perm.resize(n);
  for (int i = 0; i < n; ++i) {
    key[i] = knn_cell_id(ix.G, pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]);
    ix.perm[i] = i;
  }
  std::stable_sort(ix.perm.begin(), ix.perm.end(), [&](int a, int b) { return key[a] < key[b]; });
  ix.sp.resize(n > 0 ? n : 1);
  std::vector<uint32_t> skey(n);
  for (int s = 0; s < n; ++s) {
    const int i = ix.perm[s];
    ix.sp[s] = KnnPt{pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], i};
    skey[s] = key[i];
  }
  ix.cell_start.resize(ix.G.cells + 1);
  for (int c = 0; c <= ix.G.cells; ++c)
    ix.cell_start[c] = (int32_t)(std::lower_bound(skey.begin(), skey.end(), (uint32_t)c) - skey.begin());
}

// the K nearest of point j into nbr[0..KT): register list for KT <= 32, the strided list (the kernel's shared-memory
// list) for KT = 64
template <int KT>
void query(const Index& ix, const float* p, int32_t (&nbr)[KT]) {
  if constexpr (KT <= 32) {
    float bd[KT];
    knn_query<KT>(ix.G, ix.sp.data(), ix.cell_start.data(), p[0], p[1], p[2], bd, nbr);
  } else {
    float d[KT];
    KnnStridedList<KT, 1> L{d, nbr, 0.f, 0};
    L.init();
    knn_walk(ix.G, ix.sp.data(), ix.cell_start.data(), p[0], p[1], p[2], L);
  }
}

template <int KT>
void forward(int n, const float* pts, const Index& ix, int K, int disambiguate, float* normals, int* nbr_out,
             float* lam, int* degenerate) {
  for (int j = 0; j < n; ++j) {
    const float* p = pts + 3 * j;
    int32_t bi[KT];
    query<KT>(ix, p, bi);
    for (int k = 0; k < K; ++k) nbr_out[(long long)j * K + k] = bi[k];
    NrmFrame f;
    nrm_estimate<KT>(pts, bi, K, p, disambiguate != 0, normals + 3 * j, f);
    for (int a = 0; a < 3; ++a) lam[3 * j + a] = f.lam[a];
    degenerate[j] = f.degenerate ? 1 : 0;
  }
}

template <int KT>
void backward(int n, const float* pts, int K, int disambiguate, const int* nbr, const float* g, float* grad) {
  for (int j = 0; j < n; ++j) {
    const float* p = pts + 3 * j;
    int32_t bi[KT];
    for (int k = 0; k < KT; ++k) bi[k] = (k < K) ? nbr[(long long)j * K + k] : 0;
    NrmFrame f;
    float nv[3];
    nrm_estimate<KT>(pts, bi, K, p, false, nv, f);
    const float sgn = disambiguate ? nrm_sign<KT>(pts, bi, K, p, nv) : 1.f;
    float M[6];
    if (!nrm_grad_matrix(f, sgn, g + 3 * j, (float)K, M)) continue;
    for (int k = 0; k < K; ++k) {
      float e[3];
      nrm_centred(pts, bi[k], p, f, e);
      float* o = grad + 3 * (long long)bi[k];
      o[0] += M[0] * e[0] + M[1] * e[1] + M[2] * e[2];
      o[1] += M[1] * e[0] + M[3] * e[1] + M[4] * e[2];
      o[2] += M[2] * e[0] + M[4] * e[1] + M[5] * e[2];
    }
  }
}

}  // namespace

extern "C" {

// gsb200_estimate_normals on the host.  nbr [n,K] always written; lam [n,3] the eigenvalues (ascending), degenerate [n]
// 1 where the covariance was zero / non-finite.  Returns 1 on K outside [1, 64] or K > n.
int hn_normals(int n, const float* pts, int K, int disambiguate, float* normals, int* nbr, float* lam,
               int* degenerate) {
  if (K < 1 || K > kNrmMaxK || K > n) return 1;
  Index ix;
  build_index(n, pts, ix);
  if (K <= 16) forward<16>(n, pts, ix, K, disambiguate, normals, nbr, lam, degenerate);
  else if (K <= 32) forward<32>(n, pts, ix, K, disambiguate, normals, nbr, lam, degenerate);
  else forward<64>(n, pts, ix, K, disambiguate, normals, nbr, lam, degenerate);
  return 0;
}

// gsb200_estimate_normals_backward on the host: ADDS into grad [n,3] (sequential sums)
int hn_normals_backward(int n, const float* pts, int K, int disambiguate, const int* nbr, const float* g,
                        float* grad) {
  if (K < 1 || K > kNrmMaxK || K > n) return 1;
  if (K <= 16) backward<16>(n, pts, K, disambiguate, nbr, g, grad);
  else if (K <= 32) backward<32>(n, pts, K, disambiguate, nbr, g, grad);
  else backward<64>(n, pts, K, disambiguate, nbr, g, grad);
  return 0;
}
}
