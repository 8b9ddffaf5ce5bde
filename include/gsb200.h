/*
 * gsb200.h -- C ABI of libgsb200.so: the B200-native (sm_100a) replacement for the hot path of
 * gsgen3d/gsgen's `_gs` PyTorch extension (gs/src/bindings.cpp:5-82, gs/src/render.h:3-155).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer (tensor.data_ptr()) unless the name starts with `h_`;
 *     fp32 / int32 / uint8 exactly as the reference's CHECK_DC_FLOAT / CHECK_DC_INT contracts
 *     (gs/src/include/common.h:46-54); tensors are contiguous.
 *   - the caller owns all outputs (reference render.h: every op mutates pre-allocated tensors and
 *     returns void); gradient buffers of the reference-compatible ops are ACCUMULATED into (the
 *     caller zero-fills them, gs/renderer.py:1223-1226).
 *   - every entry point returns GSB200_OK or an error code and never exits the process (the
 *     reference printf+exit(-1)s on CUDA errors, common.h:56-72); the message is available from
 *     gsb200_last_error().  The Python shim raises RuntimeError like TORCH_CHECK does.
 *   - `stream` is a cudaStream_t (the reference launches on the legacy default stream,
 *     render.cu:505 only for SH); all work is enqueued on it, nothing synchronises unless stated.
 *   - tile_size must be 16 (every reference config, conf/base.yaml:132); other values return
 *     GSB200_ERR_UNSUPPORTED.
 */
#ifndef GSB200_H_
#define GSB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the only exported symbols of libgsb200.so */
#endif

#define GSB200_OK 0
#define GSB200_ERR_INVALID 1     /* contract violation (TORCH_CHECK in the reference)            */
#define GSB200_ERR_CUDA 2        /* CUDA runtime / launch error                                   */
#define GSB200_ERR_UNSUPPORTED 3 /* e.g. tile_size != 16, SH C outside 1..4 (render.cu:507-545)   */
#define GSB200_ERR_MISMATCH 4    /* duplicate count != gaussian_ids size (aabb_culling.h:228)      */
#define GSB200_ERR_OVERFLOW 5    /* asynchronous-count mode: the view's tile lists exceeded the capacity */

typedef struct gsb200_ctx gsb200_ctx; /* per-device scratch arena + saved state of one view       */
typedef void* gsb200_stream;           /* cudaStream_t                                              */

const char* gsb200_last_error(void);
int gsb200_version(void);
int gsb200_ctx_create(int device, gsb200_ctx** out);
int gsb200_ctx_destroy(gsb200_ctx* ctx);

/* Per-context options.
 *   GSB200_OPT_BWD_SH_VARIANT  0 (default): SH backward flushes a warp's partial sums straight to global memory with
 *                              vector reductions (csrc/composite_bwd_sh.cu); 1: round-1 kernel (per-batch shared
 *                              accumulator).  Both implement vol_render_sh.h:353-455; kept switchable for A/B timing.
 *   GSB200_OPT_ASYNC_COUNT     0 (default): gsb200_render_forward waits for the view's duplicate count (16 bytes;
 *                              the one host wait of a view -- the reference blocks twice, gs/culling.py:33-35 and
 *                              aabb_culling.h:227).  1: NO host wait anywhere in forward or backward, so the host can
 *                              run many views ahead of the GPU (a descheduled host thread no longer stalls the
 *                              device): the tile sort covers a capacity learnt from the earlier views of this context
 *                              (largest N_with_dub seen + 1/8; the first view of a context, or after N / the image
 *                              size changed, is synchronous), *h_num_dup is -1, and the exact count travels through a
 *                              ring of pinned slots that later calls on the context poll without blocking.  A view
 *                              whose lists exceeded the capacity is reported as GSB200_ERR_OVERFLOW by the first
 *                              render_forward / render_backward on the context that sees its count (usually the
 *                              view's own backward) or by gsb200_view_stats, which waits for all counts in flight:
 *                              that view's images / gradients are truncated -- render it again (capacity raised).
 */
#define GSB200_OPT_BWD_SH_VARIANT 1
#define GSB200_OPT_ASYNC_COUNT 2
int gsb200_ctx_set_option(gsb200_ctx* ctx, int option, int64_t value);

/* ================================================================================================
 * Part 1 -- one entry point per hot-path function of the reference `_gs` module, same argument
 * order and meaning (shape arguments the reference reads from tensor sizes are explicit here).
 * ============================================================================================== */

/* _gs.culling_gaussian_bsphere  render.h:3-5, render.cu:16-44, culling.h:11-34.
 * mask[i] = sphere(mean_i, thresh*max(svec_i)) intersects the 6-plane frustum.  qvec is unused
 * (as in the reference) and may be NULL.  mask is a bool tensor (1 byte / element). */
int gsb200_culling_gaussian_bsphere(const float* mean, const float* qvec, const float* svec,
                                    const float* normal, const float* pts, uint8_t* mask, uint32_t N,
                                    float thresh, gsb200_stream stream);

/* _gs.tile_culling_aabb_start_end  render.h:65-68, render.cu:381-398, aabb_culling.h:192-260.
 * Duplicates each Gaussian over its tile rectangle with key (tile<<32)|float_bits(depth), sorts
 * (cub::DeviceRadixSort), writes gaussian_ids[D] (sorted) and start/end[T] (-1 for empty tiles).
 * Synchronises once to verify the duplicate count against D (the reference's host assert). */
int gsb200_tile_culling_aabb_start_end(gsb200_ctx* ctx, const int32_t* aabb_topleft,
                                       const int32_t* aabb_bottomright, int32_t* gaussian_ids,
                                       int32_t* start, int32_t* end, const float* depth, uint32_t N,
                                       uint32_t N_with_dub, uint32_t n_tiles_h, uint32_t n_tiles_w,
                                       gsb200_stream stream);

/* _gs.tile_based_vol_rendering_start_end_with_T  render.h:151-155, vol_render.h:994-1079, and
 * _gs.tile_based_vol_rendering_start_end (render.h:70-76) when T == NULL.
 * out[H,W,3] / T[H,W] must be pre-initialised (zeros / ones): empty tiles are left untouched. */
int gsb200_tile_based_vol_rendering_start_end_with_T(
    gsb200_ctx* ctx, const float* mean, const float* cov, const float* color, const float* alpha,
    const int32_t* start, const int32_t* end, const int32_t* gaussian_ids, float* out,
    const float* topleft, uint32_t N, uint32_t N_with_dub, uint32_t tile_size, uint32_t n_tiles_h,
    uint32_t n_tiles_w, float pixel_size_x, float pixel_size_y, uint32_t H, uint32_t W, float thresh,
    float* T, gsb200_stream stream);

/* _gs.tile_based_vol_rendering_backward_start_end  render.h:78-84, vol_render.h:866-992.
 * `out` is the saved forward output INCLUDING the background term (gs/renderer.py:1182,1190). */
int gsb200_tile_based_vol_rendering_backward_start_end(
    gsb200_ctx* ctx, const float* mean, const float* cov, const float* color, const float* alpha,
    const int32_t* start, const int32_t* end, const int32_t* gaussian_ids, const float* out,
    float* grad_mean, float* grad_cov, float* grad_color, float* grad_alpha, const float* grad_out,
    const float* topleft, uint32_t N, uint32_t N_with_dub, uint32_t tile_size, uint32_t n_tiles_h,
    uint32_t n_tiles_w, float pixel_size_x, float pixel_size_y, uint32_t H, uint32_t W, float thresh,
    gsb200_stream stream);

/* _gs.tile_based_vol_rendering_scalar  render.h:134-141, vol_render_scalar.h:47-102.
 * scalar may hold more than N entries (A.9-16); only indices < N are read. */
int gsb200_tile_based_vol_rendering_scalar(
    gsb200_ctx* ctx, const float* mean, const float* cov, const float* scalar, const float* alpha,
    const int32_t* start, const int32_t* end, const int32_t* gaussian_ids, float* out,
    const float* topleft, uint32_t N, uint32_t N_with_dub, uint32_t tile_size, uint32_t n_tiles_h,
    uint32_t n_tiles_w, float pixel_size_x, float pixel_size_y, uint32_t H, uint32_t W, float thresh,
    float* T, gsb200_stream stream);

/* _gs.tile_based_vol_rendering_scalar_backward  render.h:143-149, vol_render_scalar.h:148-234. */
int gsb200_tile_based_vol_rendering_scalar_backward(
    gsb200_ctx* ctx, const float* mean, const float* cov, const float* scalar, const float* alpha,
    const int32_t* start, const int32_t* end, const int32_t* gaussian_ids, const float* out,
    float* grad_mean, float* grad_cov, float* grad_scalar, float* grad_alpha, const float* grad_out,
    const float* topleft, uint32_t N, uint32_t N_with_dub, uint32_t tile_size, uint32_t n_tiles_h,
    uint32_t n_tiles_w, float pixel_size_x, float pixel_size_y, uint32_t H, uint32_t W, float thresh,
    gsb200_stream stream);

/* _gs.tile_based_vol_rendering_sh (render.h:86-93, vol_render_sh.h:171-266) and
 * _gs.tile_based_vol_rendering_sh_with_bg (render.h:119-124, vol_render_bg.h:12-129) when
 * bg_rgb != NULL.  sh_coeffs is [N,3,C*C]; c2w: the first NINE floats are read as a packed 3x3. */
int gsb200_tile_based_vol_rendering_sh(
    gsb200_ctx* ctx, const float* mean, const float* cov, const float* sh_coeffs, const float* alpha,
    const int32_t* start, const int32_t* end, const int32_t* gaussian_ids, float* out,
    const float* topleft, const float* c2w, uint32_t N, uint32_t N_with_dub, uint32_t tile_size,
    uint32_t n_tiles_h, uint32_t n_tiles_w, float pixel_size_x, float pixel_size_y, uint32_t H,
    uint32_t W, uint32_t C, float thresh, const float* bg_rgb, gsb200_stream stream);

/* _gs.tile_based_vol_rendering_backward_sh (render.h:95-101, vol_render_sh.h:353-480) and
 * _gs.tile_based_vol_rendering_backward_sh_with_bg (render.h:126-132, vol_render_bg.h:131-266). */
int gsb200_tile_based_vol_rendering_backward_sh(
    gsb200_ctx* ctx, const float* mean, const float* cov, const float* sh_coeffs, const float* alpha,
    const int32_t* start, const int32_t* end, const int32_t* gaussian_ids, const float* out,
    float* grad_mean, float* grad_cov, float* grad_sh_coeffs, float* grad_alpha,
    const float* grad_out, const float* topleft, const float* c2w, uint32_t N, uint32_t N_with_dub,
    uint32_t tile_size, uint32_t n_tiles_h, uint32_t n_tiles_w, float pixel_size_x,
    float pixel_size_y, uint32_t H, uint32_t W, uint32_t C, float thresh, const float* bg_rgb,
    gsb200_stream stream);

/* ================================================================================================
 * Part 2 -- the torch-op stages of the reference hot path as single fused kernels.
 * ============================================================================================== */

/* gs.renderer.project_gaussians  gs/renderer.py:391-421 (+ project_pts :381-388, jacobian :366-378,
 * utils/transforms.py:34-46).  h_c2w: 12 host floats (row-major [3,4]).  JW may be NULL. */
int gsb200_project_gaussians_forward(const float* mean, const float* qvec, const float* svec,
                                     const float* h_c2w, uint32_t N, float* mean2d, float* cov2d,
                                     float* JW, float* depth, gsb200_stream stream);

/* autograd of the above (J constant, mean2d denominator detached iff depth_detach).
 * grad_mean[N,3] / grad_qvec[N,4] / grad_svec[N,3] are WRITTEN. */
int gsb200_project_gaussians_backward(const float* mean, const float* qvec, const float* svec,
                                      const float* h_c2w, uint32_t N, int depth_detach,
                                      const float* grad_mean2d, const float* grad_cov2d,
                                      const float* grad_depth, float* grad_mean, float* grad_qvec,
                                      float* grad_svec, gsb200_stream stream);

/* gs.culling.tile_culling_aabb_count  gs/culling.py:8-37 + utils/camera.py:301-314.
 * Writes aabb_topleft / aabb_bottomright [N,2] int32 tile coords (x,y) and returns the duplicate
 * count in *h_N_with_dub (synchronises, like the reference's .item()). */
int gsb200_tile_culling_aabb_count(gsb200_ctx* ctx, const float* mean2d, const float* cov2d,
                                   uint32_t N, uint32_t tile_size, float fx, float fy, float cx,
                                   float cy, uint32_t W, uint32_t H, float D, int32_t* aabb_topleft,
                                   int32_t* aabb_bottomright, int64_t* h_N_with_dub,
                                   gsb200_stream stream);

/* ================================================================================================
 * Part 3 -- the whole view in two calls (what GaussianSplattingRenderer.render_one,
 * gs/gaussian_splatting.py:1198-1421, and SHRenderer.forward, gs/sh_renderer.py:227-361, orchestrate
 * from ~60 torch kernels + 5 extension calls): cull + project + AABB + count -> scan -> key emit ->
 * radix sort -> ranges -> composite (RGB + depth + opacity + depth^2 in ONE walk, or SH).
 * No stream compaction: culled Gaussians simply own zero duplicates, indices are global.
 * ============================================================================================== */
typedef struct gsb200_camera {
  float c2w[12];              /* row-major [3,4]                                                  */
  float fx, fy, cx, cy;
  int32_t W, H;
  float frustum_normals[18];  /* CameraInfo.get_frustum, utils/camera.py:260-294                  */
  float frustum_pts[18];
  float frustum_radius;       /* conf/base.yaml:134  (6.0)                                        */
  float tile_radius;          /* conf/base.yaml:135  (6.0)                                        */
  float T_thresh;             /* conf/base.yaml:136  (1e-4)                                       */
  int32_t skip_frustum_culling;
  int32_t depth_detach;
} gsb200_camera;

#define GSB200_ACT_SVEC_EXP 1      /* svec  = exp(raw)      conf/renderer/base.yaml:14 */
#define GSB200_ACT_ALPHA_SIGMOID 2 /* alpha = sigmoid(raw)  :15 */
#define GSB200_ACT_COLOR_SIGMOID 4 /* color = sigmoid(raw)  :16 (RGB path; SH coefficients have no activation) */
typedef struct gsb200_view_in {
  uint32_t N;
  const float* mean;   /* [N,3]                                                                   */
  const float* qvec;   /* [N,4] (w,x,y,z)                                                         */
  const float* svec;   /* [N,3] post-activation (raw when act & GSB200_ACT_SVEC_EXP)               */
  const float* alpha;  /* [N]   post-activation (raw when act & GSB200_ACT_ALPHA_SIGMOID)          */
  const float* color;  /* [N,3] post-activation RGB (raw when act & ..COLOR_SIGMOID); NULL with sh  */
  const float* sh;     /* [N,3,C*C] or NULL                                                       */
  int32_t C;           /* SH template parameter (degree+1), 1..4                                  */
  float sh_c2w9[9];    /* the nine floats the SH kernels read as rotation rows (A.7)              */
  const float* bg;     /* [H,W,3] per-pixel background (RGB path) or NULL                         */
  const float* bg_rgb; /* [3] constant background (SH path) or NULL                               */
  int32_t act;         /* GSB200_ACT_* bits: the tensors above are the RAW leaves                     */
                       /* (svec_before_activation ... gs/gaussian_splatting.py:113-123) and the        */
                       /* activation runs inside the front-end kernel; render_backward then returns    */
                       /* gradients w.r.t. the raw leaves.  0 = post-activation tensors (as _gs takes) */
} gsb200_view_in;

typedef struct gsb200_view_out {
  float* rgb;      /* [H,W,3]  (includes the background term)                                     */
  float* T;        /* [H,W]    final transmittance                                                */
  float* depth;    /* [H,W] or NULL  (RGB path, rgb_only=False)                                   */
  float* opacity;  /* [H,W] or NULL                                                               */
  float* z2;       /* [H,W] or NULL  (sum w*depth^2; z_var = z2 - depth^2 is the caller's)        */
  float* mean2d;   /* [N,2]  by-products the reference exposes to autograd / densification        */
  float* cov2d;    /* [N,4]                                                                       */
  float* depthg;   /* [N]                                                                         */
  uint8_t* mask;   /* [N]                                                                         */
  float* radii2d;  /* [N] or NULL: m + sqrt(max(m^2-det,0)) (gaussian_splatting.py:1240-1245)     */
  int64_t* h_num_dup; /* host out (nullable): N_with_dub (-1 in asynchronous-count mode)           */
  int64_t* h_generation; /* host out (nullable): stamp of this forward; pass it to render_backward   */
} gsb200_view_out;

int gsb200_render_forward(gsb200_ctx* ctx, const gsb200_camera* cam, const gsb200_view_in* in,
                          const gsb200_view_out* out, gsb200_stream stream);

typedef struct gsb200_view_grads {
  /* upstream gradients (NULL = zero) and the saved forward images */
  const float* g_rgb;     const float* rgb;      /* [H,W,3]                                        */
  const float* g_depth;   const float* depth;    /* [H,W]                                          */
  const float* g_opacity; const float* opacity;
  const float* g_z2;      const float* z2;
  const float* T;                                 /* [H,W] (for g_bg)                               */
  const uint8_t* mask;                            /* [N] frustum mask written by the forward        */
  /* outputs: WRITTEN (culled Gaussians get zeros), or -- when `accumulate` != 0 -- ADDED to what the buffers
   * hold, so that a multi-view step sums straight into one flat gradient buffer (the NCCL all-reduce operand)
   * without a zero-fill + add pass per view */
  float* g_mean;    /* [N,3]                                                                       */
  float* g_qvec;    /* [N,4]                                                                       */
  float* g_svec;    /* [N,3]                                                                       */
  float* g_alpha;   /* [N]                                                                         */
  float* g_color;   /* [N,3] (RGB path) or NULL                                                    */
  float* g_sh;      /* [N,3,C*C] (SH path) or NULL; always accumulated into (zero-fill it first)   */
  float* g_mean2d;  /* [N,2] or NULL: gradient w.r.t. the projected mean (densification statistic,  */
                    /*                gaussian_splatting.py:464-469)                                */
  float* g_bg;      /* [H,W,3] or NULL: nan_to_num(g_rgb * T) (gs/renderer.py:1282)                 */
  int32_t accumulate;
  int64_t generation; /* 0 = unchecked; else must equal the stamp render_forward returned: a context holds the  */
                      /* binning + splat records of ONE view, and a later forward on it overwrites them           */
  uint8_t* touched;   /* [N] or NULL: touched[i] = 1 is written for every Gaussian the composite backward sent a   */
                      /* gradient to (never cleared here: OR over the views of a step) -- the rows a sparse         */
                      /* multi-GPU all-reduce has to carry (gsb200_rows_pack)                                       */
} gsb200_view_grads;

int gsb200_render_backward(gsb200_ctx* ctx, const gsb200_camera* cam, const gsb200_view_in* in,
                           const gsb200_view_grads* g, gsb200_stream stream);

/* Stage timing for the roofline report: when enabled, render_forward / render_backward bracket their stages
 * with CUDA events on the caller's stream (no extra synchronisation inside the timed region).
 * gsb200_ctx_get_profile synchronises the device and returns the sums since the last reset:
 *   h_ms[0] cull+project+AABB+count   h_ms[1] scan + count read-back   h_ms[2] key emit + radix sort + ranges
 *   h_ms[3] composite forward         h_ms[4] gradient memset + composite backward
 *   h_ms[5] projection backward
 *   h_counts[0] forward calls  [1] backward calls  [2] sum N_with_dub  [3] sum D_eff (1 + last list index any
 *   pixel of a tile needed, SURVEY.md §8(d))  [4] sum list entries staged into shared memory by the forward */
int gsb200_ctx_set_profiling(gsb200_ctx* ctx, int enable);
int gsb200_ctx_get_profile(gsb200_ctx* ctx, float* h_ms /*[6]*/, int64_t* h_counts /*[5]*/, int reset);

/* per-view statistics of the last forward on ctx (synchronises the stream): h_out[0]=N_with_dub,
 * h_out[1]=number of Gaussians passing the frustum test, h_out[2]=longest tile list.  In asynchronous-count
 * mode this is where a forward-only caller learns the count; returns GSB200_ERR_OVERFLOW (numbers valid) when
 * the view's lists were truncated. */
int gsb200_view_stats(gsb200_ctx* ctx, int64_t* h_out, gsb200_stream stream);

/* ================================================================================================
 * Part 4 -- the step after the gradient all-reduce (SURVEY.md §8(f)-3): torch.optim.Adam as the reference
 * configures it (conf/base.yaml:8-11, eps 1e-15; gs/gaussian_splatting.py:398-419, one param group and one
 * learning-rate schedule per field) applied to the FLAT fp32 buffers the multi-GPU path already owns
 * ([mean | qvec | svec | alpha | color or sh], gsgen_b200/parallel.py) in one streaming pass:
 * 16 B read + 12 B written per parameter.  `fields` tile [0, total) in ascending order; `lr` is the value the
 * field's scheduler returns for this step (update_lr, gaussian_splatting.py:451-454); `step` counts from 1 as
 * torch's state["step"]; gradients are multiplied by `grad_scale` first (1 = torch semantics; 1/global_batch
 * turns the SUM all-reduce into a mean).  lr / betas / eps are doubles because torch holds them as Python floats and
 * forms 1-beta and lr/(1-beta^step) in double before rounding to fp32.
 * ============================================================================================== */
typedef struct gsb200_adam_field {
  uint64_t begin;  /* first element of the field in the flat buffers */
  uint64_t count;  /* elements                                       */
  double lr;       /* Python float of the param group, as torch receives it */
} gsb200_adam_field;

int gsb200_adam_step(gsb200_ctx* ctx, float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                     uint64_t total, const gsb200_adam_field* fields, int32_t n_fields /* <= 8 */, double beta1,
                     double beta2, double eps, int64_t step, float grad_scale, gsb200_stream stream);

/* ================================================================================================
 * Part 5 -- device-side row movers of the Gaussian arena (SURVEY.md §8(f)-2).  The arena is four flat fp32 buffers
 * (parameters, gradients, exp_avg, exp_avg_sq) with one field-major layout: field f occupies `capacity * width_f`
 * floats starting at `field_off[f]`, its first N rows are live (gsgen_b200/store.py).
 *
 * gsb200_store_compact: what prune_by_mask + prune_optimizer do to every tensor and both Adam moments
 * (gs/gaussian_splatting.py:421-449, :528-549): rows with remove_mask != 0 disappear, the order of the others is
 * kept.  OUT OF PLACE: buffer b is read from h_src[b] and written to h_dst[b] (the arena's shadow buffer; the caller
 * swaps them); rows [n_keep, zero_upto) of the destination are zero-filled (dead rows carry zero gradient / moments).
 * One prefix sum + ONE mover launch for all fields of all buffers; synchronises once to return the new row count.
 *
 * gsb200_store_append: what densify_on_optimizer does (:481-522): k new rows behind row N of every field -- the
 * parameter buffer h_dst[0] receives h_rows[f] ([k, width_f], device), the other buffers' new rows are zeroed
 * (torch.cat with zeros_like).  One launch; the caller guarantees N + k <= capacity.
 * ============================================================================================== */
int gsb200_store_compact(gsb200_ctx* ctx, const float* const* h_src /*[n_bufs] device pointers*/,
                         float* const* h_dst /*[n_bufs]*/, int32_t n_bufs /* <= 4 */,
                         const uint64_t* h_field_off /*[n_fields]*/, const uint32_t* h_field_width /*[n_fields]*/,
                         int32_t n_fields /* <= 8 */, uint32_t N, uint32_t zero_upto, const uint8_t* remove_mask /*[N]*/,
                         uint32_t* h_n_keep, gsb200_stream stream);
int gsb200_store_append(gsb200_ctx* ctx, float* const* h_dst /*[n_bufs]; [0] = parameters*/, int32_t n_bufs,
                        const float* const* h_rows /*[n_fields] device pointers to [k,width_f]*/,
                        const uint64_t* h_field_off, const uint32_t* h_field_width, int32_t n_fields, uint32_t N,
                        uint32_t k, gsb200_stream stream);

/* Sparse gradient all-reduce (SURVEY.md §8(e)).  A view sends gradients only to the Gaussians in front of the
 * T < T_thresh horizon (measured: 10 % of C3's Gaussians per view, 36 % over the 8 views of a step), so the flat
 * gradient buffer the ranks all-reduce is mostly zeros.  With gsb200_view_grads.touched the backward marks the rows it
 * wrote; the ranks MAX-reduce that byte mask (1 B / Gaussian) and then:
 * gsb200_rows_pack: idx[0 .. n_keep) := the ids of the rows with keep[i] != 0, in order (prefix sum + scatter; idx is
 * the caller's [N] int32 buffer, reused by unpack), *h_n_keep = their number (ONE stream synchronisation: the
 * collective's count is a host quantity), and -- if n_keep * row_floats <= packed_capacity -- one launch that gathers
 * those rows of every field into `packed`, field f starting at n_keep * (widths before f): n_keep * row_floats
 * contiguous floats for ONE collective.
 * gsb200_rows_unpack: the reduced rows back into the flat buffer (rows not kept are left as they are: zero). */
int gsb200_rows_pack(gsb200_ctx* ctx, const float* flat, float* packed, uint64_t packed_capacity /* floats */,
                     const uint64_t* h_field_off, const uint32_t* h_field_width, int32_t n_fields, uint32_t N,
                     const uint8_t* keep /*[N]*/, int32_t* idx /*[N] out*/, uint32_t* h_n_keep, gsb200_stream stream);
int gsb200_rows_unpack(gsb200_ctx* ctx, float* flat, const float* packed, const uint64_t* h_field_off,
                       const uint32_t* h_field_width, int32_t n_fields, uint32_t N, const int32_t* idx,
                       uint32_t n_keep, gsb200_stream stream);

/* ================================================================================================
 * Part 6 -- K nearest neighbours of the Gaussian means (SURVEY.md §8(f)-2: the search behind compactness-based
 * densification, gs/gaussian_splatting.py:634-743, and the NN / compactness penalties, :1032-1094).  Replaces
 * utils/ops.py:103-134 `nearest_neighbor` / `K_nearest_neighbors`, i.e. pytorch3d.ops.knn_points(query, mean, K)
 * (third-party, brute force): for every query the K points with the smallest squared Euclidean distance, ascending,
 * ties by smaller point index.  points [n_points,3] fp32; queries [n_queries,3] fp32 or NULL = the points query
 * themselves (every point is then its own first neighbour, distance 0, which the reference drops); idx
 * [n_queries,K] int64 (-1 where fewer than K points exist), dist2 [n_queries,K] fp32 or NULL (+inf there).
 * 1 <= K <= 32.  Uniform-grid shell search, exact; everything on `stream`, no synchronisation.
 * ============================================================================================== */
int gsb200_knn(gsb200_ctx* ctx, const float* points, uint32_t n_points, const float* queries, uint32_t n_queries,
               int32_t K, int64_t* idx, float* dist2, gsb200_stream stream);

/* ================================================================================================
 * Part 7 -- per-point normals of a point cloud (the Gaussian means): utils/ops.py:62-72 estimate_normal, i.e.
 * pytorch3d.ops.estimate_pointcloud_normals(points, K, disambiguate_directions), used by gs/gaussian_splatting.py
 * for cfg.normal_as_rgb and by utils/relight.py.  For every point: its K nearest points (itself included, the exact
 * search of Part 6), C = (1/K) sum_k (x_k - mu)(x_k - mu)^T, the unit eigenvector of C's smallest eigenvalue; with
 * disambiguate != 0 it is negated when fewer than K/2 neighbours x_k satisfy n . (x_k - p) > 0.  A zero or non-finite
 * covariance gives (0, 0, 1) before that flip.  1 <= K <= 64 and K <= n_points (GSB200_ERR_UNSUPPORTED /
 * GSB200_ERR_INVALID otherwise).
 *
 * gsb200_estimate_normals: points [n,3] fp32 -> normals [n,3] fp32; nbr_idx [n,K] int32 receives the neighbour
 * indices (ascending distance, ties by index) for the backward, or is NULL (then nothing of size [n,K] is written).
 * gsb200_estimate_normals_backward: ADDS dL/dpoints to grad_points [n,3] for dL/dnormals = grad_normals [n,3], with the
 * forward's neighbour sets (nbr_idx) and signs held constant (the sign is recomputed: pass the forward's disambiguate).
 * An eigen gap |lam_0 - lam_j| <= 1e-6 max(lam_2, 1e-30) contributes zero instead of inf / NaN.  Atomic accumulation:
 * not bitwise reproducible.  Both run on `stream` without synchronising.
 * ============================================================================================== */
int gsb200_estimate_normals(gsb200_ctx* ctx, const float* points, uint32_t n_points, int32_t K, int32_t disambiguate,
                            float* normals, int32_t* nbr_idx, gsb200_stream stream);
int gsb200_estimate_normals_backward(gsb200_ctx* ctx, const float* points, uint32_t n_points, int32_t K,
                                     int32_t disambiguate, const int32_t* nbr_idx, const float* grad_normals,
                                     float* grad_points, gsb200_stream stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* GSB200_H_ */
