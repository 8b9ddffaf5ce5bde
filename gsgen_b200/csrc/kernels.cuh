// kernels.cuh -- declarations shared between the translation units of libgsb200.so
#pragma once
#include "gsb200_common.cuh"

namespace gsb {

enum PayKind { PAY_RGB = 0, PAY_SCALAR = 1, PAY_SH = 2 };

// Arguments of the composite kernels (forward and backward).  Passed by value (< 4 KB).
struct CompositeArgs {
  // per-Gaussian records
  const Splat* splat = nullptr;   // [N] geometry records (32 B)
  const float4* pay = nullptr;    // [N] (r,g,b,depth) or (scalar,-,-,-); unused for SH
  const float* sh = nullptr;      // [N,3,C*C]
  // sorted tile lists
  const int32_t* ids = nullptr;
  const int32_t* start = nullptr;
  const int32_t* end = nullptr;
  // view
  const float* topleft_ptr = nullptr;  // device float[2] (reference API) or nullptr -> tlx/tly
  float tlx = 0.f, tly = 0.f;
  float psx = 0.f, psy = 0.f;
  int H = 0, W = 0, tiles_w = 0, tiles_h = 0;
  float thresh = 1e-4f;
  const float* c9_ptr = nullptr;       // device float[>=9] (reference API) or nullptr -> c9
  float c9[9] = {0};
  const float* bg = nullptr;           // [H,W,3] per-pixel background (RGB) or nullptr
  const float* bg_rgb = nullptr;       // device float[3] constant background (SH) or nullptr
  int device = 0;                      // current CUDA device (per-device one-time kernel attributes)
  int write_empty = 0;                 // 1: empty tiles are written (fused path owns the output buffers)
  // forward outputs
  float* out = nullptr;                // [H,W,3] or [H,W] (scalar)
  float* T = nullptr;                  // [H,W] or nullptr
  float* depth = nullptr;              // extras (RGB fused), all three or none
  float* opacity = nullptr;
  float* z2 = nullptr;
  // backward inputs: saved forward images + upstream gradients (nullptr = zero gradient)
  const float* fin = nullptr;          // final rgb (incl. background) or scalar image
  const float* gout = nullptr;
  const float* fin_depth = nullptr; const float* g_depth = nullptr;
  const float* fin_opacity = nullptr; const float* g_opacity = nullptr;
  const float* fin_z2 = nullptr; const float* g_z2 = nullptr;
  // backward outputs (accumulated with float reductions)
  float* grad_mean = nullptr;          // [N,2]      reference layout
  float* grad_cov = nullptr;           // [N,4]
  float* grad_pay = nullptr;           // [N,3] colour, [>=N] scalar or [N,3,C*C] sh
  float* grad_alpha = nullptr;         // [N]
  float* ggeom = nullptr;              // [N,8] fused gradient record (replaces grad_mean/cov/alpha)
  float* gpay = nullptr;               // [N,4] fused colour gradient record
  float* g_bg = nullptr;               // [H,W,3] or nullptr
  // optional counters (profiling only): [0] += D_eff of the tile (1 + last list index any pixel needed),
  // [1] += list entries actually staged into shared memory
  unsigned long long* stats = nullptr;
};

// preprocess.cu
int launch_cull_bsphere(uint32_t N, const float* mean, const float* svec, const float* normal, const float* pts,
                        uint8_t* mask, float thresh, cudaStream_t st);
int launch_project_fwd(uint32_t N, const float* mean, const float* qvec, const float* svec, const Camera& cam,
                       float* mean2d, float* cov2d, float* JW, float* depth, cudaStream_t st);
int launch_project_bwd(uint32_t N, const float* mean, const float* qvec, const float* svec, const Camera& cam,
                       const float* g_m2, const float* g_cov, const float* g_depth, float* g_mean, float* g_qvec,
                       float* g_svec, cudaStream_t st);
int launch_aabb_count(uint32_t N, const float* mean2d, const float* cov2d, int tile, float fx, float fy, float cx,
                      float cy, int W, int H, float D, int32_t* tl, int32_t* br, unsigned long long* total,
                      cudaStream_t st);
int launch_count_from_aabb(uint32_t N, const int32_t* tl, const int32_t* br, int32_t* count, ushort4* rect,
                           unsigned long long* total, cudaStream_t st);
int launch_pack_splats(uint32_t N, const float* mean2d, const float* cov2d, const float* alpha, const float* payload,
                       int pay_kind, Splat* splat, float4* pay, cudaStream_t st);
int launch_preprocess(uint32_t N, const float* mean, const float* qvec, const float* svec, const float* alpha,
                      const float* color, int act, const Camera& cam, float* mean2d, float* cov2d, float* depthg,
                      uint8_t* mask, float* radii2d, Splat* splat, float4* pay, ushort4* rect, int32_t* count,
                      uint32_t* dkeys, int32_t* perm0, unsigned long long* total, cudaStream_t st);
int launch_project_bwd_fused(uint32_t N, const float* mean, const float* qvec, const float* svec,
                             const float* alpha, const float* color, int act, const uint8_t* mask, const Camera& cam, const float4* ggeom, const float4* gpay,
                             float* g_mean, float* g_qvec, float* g_svec, float* g_alpha, float* g_color,
                             float* g_mean2d, int accumulate, uint8_t* touched, cudaStream_t st);

// optimizer.cu
struct AdamFields {
  int n;
  unsigned long long begin[9];  // field f covers [begin[f], begin[f+1]); begin[n] = total
  float step_size[8];           // lr_f / (1 - beta1^step)
};
int launch_adam_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, unsigned long long total,
                     const AdamFields& fields, const AdamScalars& k, cudaStream_t st);

// binning.cu
int begin_total(gsb200_ctx* ctx, cudaStream_t st);    // zero the device-side duplicate counter
int request_total(gsb200_ctx* ctx, cudaStream_t st);  // async D2H copy + event
int wait_total(gsb200_ctx* ctx, int64_t* h_total);    // host waits for that event only
int reserve_depth_sort(gsb200_ctx* ctx, uint32_t N);   // dkeys / perm / incl for N Gaussians
int sort_depths_and_scan(gsb200_ctx* ctx, uint32_t N, const float* depth, cudaStream_t st, bool keys_ready = false);
int bin_and_sort(gsb200_ctx* ctx, uint32_t N, int64_t D, int tiles_h, int tiles_w, int32_t* ids_out, int32_t* start,
                 int32_t* end, cudaStream_t st, bool padded = false);
int launch_max_list(uint32_t T, const int32_t* start, const int32_t* end, int32_t* out, cudaStream_t st);

// composite_fwd.cu / composite_bwd.cu
int launch_composite_fwd(int pay_kind, int C, bool extras, const CompositeArgs& a, cudaStream_t st);
int launch_composite_bwd(int pay_kind, int C, bool extras, bool fused, const CompositeArgs& a, cudaStream_t st);
// composite_bwd_sh.cu (round 2): SH degree >= 1 with the direct vector-reduction flush
int launch_composite_bwd_sh(int C, bool fused, const CompositeArgs& a, cudaStream_t st);

// knn.cu: exact K nearest neighbours on a uniform grid (queries == nullptr: the points query themselves)
int knn_device(gsb200_ctx* ctx, const float* points, uint32_t n, const float* queries, uint32_t nq, int K,
               int64_t* idx_out, float* d2_out, cudaStream_t st);
// the grid behind it, built on `st` in the context's knn_* buffers: points sorted by cell, the cell table, and `order`
// (order[s] = index of the point in sorted slot s, i.e. the points in cell order)
struct KnnGrid;
struct KnnPt;
struct KnnIndex {
  const KnnGrid* grid;
  const KnnPt* sorted;
  const int32_t* cell_start;
  const int32_t* order;
};
int knn_build_index(gsb200_ctx* ctx, const float* points, uint32_t n, KnnIndex* out, cudaStream_t st);
// normals.cu: per-point normals of the points' K-neighbourhoods (include/gsb200.h Part 7)
int normals_device(gsb200_ctx* ctx, const float* points, uint32_t n, int K, int disambiguate, float* normals,
                   int32_t* nbr_idx, cudaStream_t st);
int normals_backward_device(const float* points, uint32_t n, int K, int disambiguate, const int32_t* nbr_idx,
                            const float* grad_normals, float* grad_points, cudaStream_t st);

// Opt a kernel in to more than 48 KB of dynamic shared memory.  Called before every launch: the attribute is per
// (function, device) and the call is a few hundred ns -- cheaper than a lock-protected per-device cache, and correct
// when several host threads drive different devices through the same library (round-1 advice: the lazy
// `static bool attr_set[64]` was an unsynchronised init).
inline cudaError_t ensure_max_dyn_smem(const void* func, int bytes, int /*device*/) {
  return cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

}  // namespace gsb
