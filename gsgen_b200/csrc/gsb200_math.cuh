// gsb200_math.cuh -- per-Gaussian math of the hot path, written as host+device inline functions so
// the same code runs in the sm_100a kernels and in the CPU unit test (tests/hostmath, g++).
//
// Reference semantics restated (paths relative to the reference repo, see SURVEY.md App. A):
//   A.2 frustum sphere test      gs/src/include/culling.h:11-20, kernels.h:156-170
//   A.3 EWA projection           gs/renderer.py:366-421, utils/transforms.py:34-46 (kornia 0.6.0 quat->R)
//   A.4 AABB tile rectangle      gs/culling.py:16-35, utils/camera.py:301-314
//   A.6 2-D Gaussian evaluation  gs/src/include/kernels.h:172-224 (cov inverted per pixel, q<0 -> 1000)
//   A.7 SH basis / pixel ray     gs/src/include/shencoder.h:13-56, vol_render_sh.h:48-65
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define GSB_HD __host__ __device__ __forceinline__
#else
#define GSB_HD static inline
#endif

namespace gsb {

constexpr float kMinRenderAlpha = 0.00392156862745098f;  // common.h:89  1/255
constexpr float kAlphaClamp = 0.99f;                     // vol_render.h:212
// G = exp(-q/2) = exp2(-(u^2+v^2)) with (u,v) = s * L d,  s = sqrt(0.5*log2(e))
constexpr double kCholScale = 0.84932180028801907;  // sqrt(0.5 * 1.4426950408889634)
constexpr float kInvCholScale2 = 1.3862943611198906f;  // 1/s^2 = 2 ln 2

// mul / add that must NOT be contracted into an FMA (they mirror separate torch kernels)
#if defined(__CUDA_ARCH__)
GSB_HD float mul_rn(float a, float b) { return __fmul_rn(a, b); }
GSB_HD float add_rn(float a, float b) { return __fadd_rn(a, b); }
GSB_HD int f2i_rz(float a) { return __float2int_rz(a); }  // saturating, NaN -> 0
#else
GSB_HD float mul_rn(float a, float b) { volatile float r = a * b; return r; }
GSB_HD float add_rn(float a, float b) { volatile float r = a + b; return r; }
GSB_HD int f2i_rz(float a) {
  if (!(a == a)) return 0;
  if (a >= 2147483648.0f) return 2147483647;
  if (a <= -2147483648.0f) return (-2147483647 - 1);
  return (int)a;
}
#endif

struct Camera {      // one view; plain floats so it can be passed by value to kernels
  float R[9];        // c2w[:3,:3] row-major (columns = right, down, lookat)
  float t[3];        // c2w[:3,3]
  float fx, fy, cx, cy;
  int W, H;
  int tiles_w, tiles_h;
  float fn[18], fp[18];  // frustum plane normals / points (CameraInfo.get_frustum)
  float frustum_radius;  // 6.0  conf/base.yaml:134
  float tile_radius;     // 6.0  conf/base.yaml:135
  int skip_frustum;
  int depth_detach;      // conf/renderer/base.yaml depth_detach (default True)
};

// ---- parameter activations of the fused front end (SURVEY §8(f)-1) ------------------------------------
// The reference keeps svec / alpha / color as raw leaves and applies an activation in a property on every
// access (gs/gaussian_splatting.py:113-123); every shipped config uses exp / sigmoid / sigmoid
// (conf/renderer/base.yaml:14-16, utils/activations.py:36-45).  With `act` bits set the fused kernels take the
// RAW leaves and return gradients w.r.t. them; the formulas are torch's (exp -> y, sigmoid -> y(1-y)).
enum : int { kActSvecExp = 1, kActAlphaSigmoid = 2, kActColorSigmoid = 4 };
GSB_HD float act_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }
GSB_HD float act_svec(float raw, int act) { return (act & kActSvecExp) ? expf(raw) : raw; }
GSB_HD float act_alpha(float raw, int act) { return (act & kActAlphaSigmoid) ? act_sigmoid(raw) : raw; }
GSB_HD float act_color(float raw, int act) { return (act & kActColorSigmoid) ? act_sigmoid(raw) : raw; }
// chain rule: gradient w.r.t. the raw leaf from the gradient w.r.t. the activated value y
GSB_HD float act_svec_bwd(float g, float y, int act) { return (act & kActSvecExp) ? g * y : g; }
GSB_HD float act_alpha_bwd(float g, float y, int act) { return (act & kActAlphaSigmoid) ? g * ((1.0f - y) * y) : g; }
GSB_HD float act_color_bwd(float g, float y, int act) { return (act & kActColorSigmoid) ? g * ((1.0f - y) * y) : g; }

// ---- Adam on the flat parameter buffer (SURVEY §8(f)-3) ---------------------------------------------------
// torch.optim.Adam(amsgrad=False, weight_decay=0) as the reference configures it (conf/base.yaml:8-11: eps 1e-15;
// gs/gaussian_splatting.py:398-419: one param group per field, lr from the field's scheduler).  Same expression
// order as torch's kernels: lerp, mul+addcmul, sqrt / bias_correction2_sqrt + eps, addcdiv.
struct AdamScalars {
  float beta2, one_minus_beta1, one_minus_beta2, eps, bc2_sqrt, grad_scale;
};
GSB_HD void adam_update(float& p, float g, float& m, float& v, float step_size, const AdamScalars& k) {
  g *= k.grad_scale;
  m = m + k.one_minus_beta1 * (g - m);
  v = v * k.beta2;
  v = v + (k.one_minus_beta2 * g) * g;
  const float denom = sqrtf(v) / k.bc2_sqrt + k.eps;
  p = p - step_size * (m / denom);
}

// ---- A.2 -----------------------------------------------------------------------------------------
GSB_HD bool sphere_in_frustum(const float m[3], float r, const float* fn, const float* fp) {
#pragma unroll
  for (int p = 0; p < 6; ++p) {
    float d = (m[0] - fp[3 * p]) * fn[3 * p] + (m[1] - fp[3 * p + 1]) * fn[3 * p + 1] +
              (m[2] - fp[3 * p + 2]) * fn[3 * p + 2];
    if (!(d > -r)) return false;
  }
  return true;
}

// ---- A.3 -----------------------------------------------------------------------------------------
// kornia 0.6.0 quaternion_to_rotation_matrix(order=WXYZ): normalise (eps 1e-12) then unit-quaternion matrix
GSB_HD void quat_to_rotmat(const float q[4], float R[9], float qn[4], float* inv_norm) {
  float n = sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  float inv = 1.0f / fmaxf(n, 1e-12f);
  float w = q[0] * inv, x = q[1] * inv, y = q[2] * inv, z = q[3] * inv;
  qn[0] = w; qn[1] = x; qn[2] = y; qn[3] = z;
  *inv_norm = inv;
  float tx = 2.0f * x, ty = 2.0f * y, tz = 2.0f * z;
  float twx = tx * w, twy = ty * w, twz = tz * w;
  float txx = tx * x, txy = ty * x, txz = tz * x;
  float tyy = ty * y, tyz = tz * y, tzz = tz * z;
  R[0] = 1.0f - (tyy + tzz); R[1] = txy - twz;          R[2] = txz + twy;
  R[3] = txy + twz;          R[4] = 1.0f - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy;          R[7] = tyz + twx;          R[8] = 1.0f - (txx + tyy);
}

struct Proj {        // forward intermediates the backward re-uses
  float p[3];        // camera-space point  p = Rc^T (x - t)
  float T2[6];       // first two rows of J*W (J detached): 2x3 row-major
  float Rq[9];       // rotation of the normalised quaternion
  float qn[4];
  float inv_qnorm;
  float A[6];        // T2 * (Rq diag(s)): 2x3 ; cov2d = A A^T
  float mean2d[2];
  float cov[4];
  float depth;
};

GSB_HD void project_gaussian(const float x[3], const float q[4], const float s[3], const Camera& cam, Proj& o) {
  // project_pts (gs/renderer.py:381-388): W (pts + d), W = Rc^T, d = -t
  float dx = x[0] - cam.t[0], dy = x[1] - cam.t[1], dz = x[2] - cam.t[2];
  const float* Rc = cam.R;
#pragma unroll
  for (int i = 0; i < 3; ++i) o.p[i] = fmaf(Rc[6 + i], dz, fmaf(Rc[3 + i], dy, Rc[i] * dx));
  float px = o.p[0], py = o.p[1], pz = o.p[2];
  // jacobian (gs/renderer.py:366-378), rows 0 and 1 only (cov2d = (J W S W^T J^T)[:2,:2])
  float j00 = 1.0f / pz, j02 = -px / pz / pz, j12 = -py / pz / pz;
  // JW = J W ; W[i][k] = Rc[k][i]
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    o.T2[k] = fmaf(j02, Rc[3 * k + 2], j00 * Rc[3 * k + 0]);
    o.T2[3 + k] = fmaf(j12, Rc[3 * k + 2], j00 * Rc[3 * k + 1]);
  }
  quat_to_rotmat(q, o.Rq, o.qn, &o.inv_qnorm);
  // A = T2 * M, M[k][j] = Rq[k][j]*s[j]  (utils/transforms.py:40: svec.unsqueeze(-2) * R)
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float acc = o.T2[3 * r] * o.Rq[j];
      acc = fmaf(o.T2[3 * r + 1], o.Rq[3 + j], acc);
      acc = fmaf(o.T2[3 * r + 2], o.Rq[6 + j], acc);
      o.A[3 * r + j] = acc * s[j];
    }
  const float* A = o.A;
  o.cov[0] = fmaf(A[2], A[2], fmaf(A[1], A[1], A[0] * A[0]));
  o.cov[1] = fmaf(A[2], A[5], fmaf(A[1], A[4], A[0] * A[3]));
  o.cov[2] = o.cov[1];
  o.cov[3] = fmaf(A[5], A[5], fmaf(A[4], A[4], A[3] * A[3]));
  o.depth = pz;
  o.mean2d[0] = px / pz;
  o.mean2d[1] = py / pz;
}

// backward of project_gaussian.  g_cov = [g0 g1; g2 g3], J is a constant (renderer.py:365 @no_grad),
// mean2d's denominator is detached when cam.depth_detach (renderer.py:414-419).
GSB_HD void project_gaussian_bwd(const float s[3], const Camera& cam, const Proj& f, const float g_m2[2],
                                 const float g_cov[4], float g_depth, float g_x[3], float g_q[4], float g_s[3]) {
  const float* A = f.A;
  float gs01 = g_cov[1] + g_cov[2];
  float gA[6];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    gA[j] = 2.0f * g_cov[0] * A[j] + gs01 * A[3 + j];
    gA[3 + j] = gs01 * A[j] + 2.0f * g_cov[3] * A[3 + j];
  }
  float gR[9];
#pragma unroll
  for (int j = 0; j < 3; ++j) g_s[j] = 0.0f;
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float gM = f.T2[k] * gA[j] + f.T2[3 + k] * gA[3 + j];
      g_s[j] = fmaf(gM, f.Rq[3 * k + j], g_s[j]);
      gR[3 * k + j] = gM * s[j];
    }
  float w = f.qn[0], x = f.qn[1], y = f.qn[2], z = f.qn[3];
  float gw = 2.0f * (-z * gR[1] + y * gR[2] + z * gR[3] - x * gR[5] - y * gR[6] + x * gR[7]);
  float gx = 2.0f * (y * gR[1] + z * gR[2] + y * gR[3] - 2.0f * x * gR[4] - w * gR[5] + z * gR[6] + w * gR[7] -
                     2.0f * x * gR[8]);
  float gy = 2.0f * (-2.0f * y * gR[0] + x * gR[1] + w * gR[2] + x * gR[3] + z * gR[5] - w * gR[6] + z * gR[7] -
                     2.0f * y * gR[8]);
  float gz = 2.0f * (-2.0f * z * gR[0] - w * gR[1] + x * gR[2] + w * gR[3] - 2.0f * z * gR[4] + y * gR[5] +
                     x * gR[6] + y * gR[7]);
  float dotq = w * gw + x * gx + y * gy + z * gz;
  g_q[0] = (gw - w * dotq) * f.inv_qnorm;
  g_q[1] = (gx - x * dotq) * f.inv_qnorm;
  g_q[2] = (gy - y * dotq) * f.inv_qnorm;
  g_q[3] = (gz - z * dotq) * f.inv_qnorm;
  float pz = f.p[2];
  float gp[3] = {g_m2[0] / pz, g_m2[1] / pz, g_depth};
  if (!cam.depth_detach) gp[2] -= (g_m2[0] * f.p[0] + g_m2[1] * f.p[1]) / (pz * pz);
  const float* Rc = cam.R;
#pragma unroll
  for (int j = 0; j < 3; ++j) g_x[j] = Rc[3 * j] * gp[0] + Rc[3 * j + 1] * gp[1] + Rc[3 * j + 2] * gp[2];
}

// largest eigenvalue of cov2d, gs/gaussian_splatting.py:1240-1245
GSB_HD float radius2d(const float cov[4]) {
  float m = (cov[0] + cov[3]) * 0.5f;
  float det = cov[0] * cov[3] - cov[1] * cov[2];
  return m + sqrtf(fmaxf(m * m - det, 0.0f));
}

// ---- A.4 -----------------------------------------------------------------------------------------
// Integer tile rectangle of the sqrt(D*cov) AABB; bit-exact restatement of the torch op sequence
// (separate mul / add kernels, truncating int cast, clamp, floor-div).  rect = {x0,y0,x1,y1} in tiles.
GSB_HD void aabb_tiles(const float m2[2], float c00, float c11, float D, float fx, float fy, float cx, float cy,
                       int W, int H, int tile, int rect[4]) {
  float ex = sqrtf(mul_rn(D, c00)), ey = sqrtf(mul_rn(D, c11));
  float tlx = add_rn(m2[0], -ex), tly = add_rn(m2[1], -ey);
  float brx = add_rn(m2[0], ex), bry = add_rn(m2[1], ey);
  int x0 = f2i_rz(add_rn(mul_rn(tlx, fx), cx)), y0 = f2i_rz(add_rn(mul_rn(tly, fy), cy));
  int x1 = f2i_rz(add_rn(mul_rn(brx, fx), cx)), y1 = f2i_rz(add_rn(mul_rn(bry, fy), cy));
  x0 = x0 < 0 ? 0 : (x0 > W - 1 ? W - 1 : x0);
  x1 = x1 < 0 ? 0 : (x1 > W - 1 ? W - 1 : x1);
  y0 = y0 < 0 ? 0 : (y0 > H - 1 ? H - 1 : y0);
  y1 = y1 < 0 ? 0 : (y1 > H - 1 ? H - 1 : y1);
  rect[0] = x0 / tile; rect[1] = y0 / tile; rect[2] = x1 / tile; rect[3] = y1 / tile;
}

// ---- A.6 -----------------------------------------------------------------------------------------
// Per-Gaussian "splat record": everything a pixel needs to evaluate a*G without a division.
//   G(d) = exp(-0.5 d^T S^-1 d) with S^-1 from the reference's per-pixel formula
//          q = ((dx*c3 - dy*c2)*dx + (-dx*c1 + dy*c0)*dy) / (c0*c3 - c1*c2)     (kernels.h:172-224)
//        = dx^2*A + 2*dx*dy*B + dy^2*Cc,  A = c3/det, B = -(c1+c2)/(2 det), Cc = c0/det
//   Cholesky S^-1 = L^T L (L upper-triangular) evaluated in fp64 once per Gaussian, scaled so that
//   G = exp2(-(u^2+v^2)), u = p0*dx + p1*dy, v = p2*dy: a sum of squares, no cancellation in q.
//   (hx,hy): half-extents (camera-plane units) of the region where a*G >= 1/255 can hold, inflated by
//   1e-4 -- used only to skip whole warps; the per-pixel test stays the arbiter.
// A covariance that is not positive definite (reference: undefined / q<0 -> G=exp(-500)=0) never contributes.
struct Splat {
  float mx, my, p0, p1;  // float4 #0
  float p2, a, hx, hy;   // float4 #1
};

GSB_HD Splat make_splat(const float m2[2], const float cov[4], float alpha) {
  Splat s;
  s.mx = m2[0]; s.my = m2[1];
  double c0 = cov[0], c1 = cov[1], c2 = cov[2], c3 = cov[3];
  double det = c0 * c3 - c1 * c2;
  double b = 0.5 * (c1 + c2);
  float a = fminf(alpha, kAlphaClamp);
  // NaN alpha must be tested before the clamp: fminf(NaN, 0.99f) is 0.99f
  bool ok = (det > 0.0) && (c0 > 0.0) && (c3 > 0.0) && (det == det) && (alpha == alpha);
  double A = c3 / det, B = -b / det, Cc = c0 / det;
  double l00 = sqrt(A), l01 = B / l00, l11sq = Cc - l01 * l01;
  ok = ok && (l11sq > 0.0) && (l00 == l00) && (l00 < 1e18) && (l11sq < 1e36);
  if (!ok) {
    s.p0 = 0.f; s.p1 = 0.f; s.p2 = 0.f; s.a = 0.f; s.hx = -1.f; s.hy = -1.f;
    return s;
  }
  s.p0 = (float)(kCholScale * l00);
  s.p1 = (float)(kCholScale * l01);
  s.p2 = (float)(kCholScale * sqrt(l11sq));
  s.a = a;
  double a255 = 255.0 * (double)a;
  if (!(a255 > 1.0)) {
    s.hx = -1.f; s.hy = -1.f;  // a*G < 1/255 for every pixel
  } else {
    double qmax = 2.0 * log(a255) * (1.0 + 1e-6) + 1e-6;
    double dq = A * Cc - B * B;  // det(S^-1)
    s.hx = (float)(sqrt(qmax * Cc / dq) * (1.0 + 1e-4)) + 1e-6f;
    s.hy = (float)(sqrt(qmax * A / dq) * (1.0 + 1e-4)) + 1e-6f;
  }
  return s;
}

// ---- A.7 -----------------------------------------------------------------------------------------
template <int C>
GSB_HD void sh_basis(float x, float y, float z, float* o) {
  float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
  o[0] = 0.28209479177387814f;
  if (C <= 1) return;
  o[1] = -0.48860251190291987f * y;
  o[2] = 0.48860251190291987f * z;
  o[3] = -0.48860251190291987f * x;
  if (C <= 2) return;
  o[4] = 1.0925484305920792f * xy;
  o[5] = -1.0925484305920792f * yz;
  o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
  o[7] = -1.0925484305920792f * xz;
  o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
  if (C <= 3) return;
  o[9] = 0.59004358992664352f * y * (-3.0f * x2 + y2);
  o[10] = 2.8906114426405538f * xy * z;
  o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2);
  o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
  o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2);
  o[14] = 1.4453057213202769f * z * (x2 - y2);
  o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
}

// vol_render_sh.h:48-65: dir = normalize(rows(c2w_first_9_floats) . (posx, posy, 1))
GSB_HD void pixel_dir(float posx, float posy, const float* c9, float d[3]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) d[r] = c9[3 * r] * posx + c9[3 * r + 1] * posy + c9[3 * r + 2];
  float len = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  d[0] /= len; d[1] /= len; d[2] /= len;
}

}  // namespace gsb
