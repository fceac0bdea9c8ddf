// tracker_device.cuh -- per-pixel device functions of the tracker reductions, shared by the
// stand-alone step kernels (tracker_kernels.cu) and the persistent Gauss-Newton kernel
// (gn_tiled.cu).  Arithmetic spec: SURVEY.md Appendix A1-A5 / Core/Cuda/reduce.cu.
#pragma once
#include "tracker_kernels.cuh"

namespace cfb {
namespace dev {

__device__ __forceinline__ float ldplane(const PlanarMap& m, int plane_row, int x) {
  return __ldg(row_ptr(m.p, m.pitch, plane_row) + x);
}

// 27 upper-triangular products + row6^2 + inlier (JtJJtrSE3 order, types.cuh:101-112)
__device__ __forceinline__ void accumulate_se3(float (&acc)[32], const float (&row)[7], bool found) {
  int k = 0;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i; j < 7; ++j) acc[k++] += row[i] * row[j];
  acc[27] += row[6] * row[6];
  acc[28] += found ? 1.f : 0.f;
}

// ------------------------------------------------------------------------------------------ ICP
__device__ __forceinline__ void icp_pixel(const IcpArgs& a, const IcpPose& P, int x, int y,
                                          float (&acc)[32]) {
  const int rows = a.rows;
  float3 vcurr = make_float3(ldplane(a.vmap_curr, y, x), ldplane(a.vmap_curr, y + rows, x),
                             ldplane(a.vmap_curr, y + 2 * rows, x));
  const float3 tcurr = make_float3(P.tcurr[0], P.tcurr[1], P.tcurr[2]);
  const float3 tprev = make_float3(P.tprev[0], P.tprev[1], P.tprev[2]);
  float3 vcurr_g = mul(P.Rcurr, vcurr) + tcurr;
  float3 vcurr_cp = mul(P.Rprev_inv, vcurr_g - tprev);

  int ux = __float2int_rn(vcurr_cp.x * a.intr.fx / vcurr_cp.z + a.intr.cx);
  int uy = __float2int_rn(vcurr_cp.y * a.intr.fy / vcurr_cp.z + a.intr.cy);

  float row[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  bool found = false;
  if (ux < 0 || uy < 0 || ux >= a.cols || uy >= rows || vcurr_cp.z < 0) {
    if (a.error_map) row_ptr(a.error_map, a.error_pitch, y)[x] = 0.0f;
  } else {
    float3 vprev_g = make_float3(ldplane(a.vmap_g_prev, uy, ux), ldplane(a.vmap_g_prev, uy + rows, ux),
                                 ldplane(a.vmap_g_prev, uy + 2 * rows, ux));
    float3 ncurr = make_float3(ldplane(a.nmap_curr, y, x), ldplane(a.nmap_curr, y + rows, x),
                               ldplane(a.nmap_curr, y + 2 * rows, x));
    float3 ncurr_g = mul(P.Rcurr, ncurr);
    float3 nprev_g = make_float3(ldplane(a.nmap_g_prev, uy, ux), ldplane(a.nmap_g_prev, uy + rows, ux),
                                 ldplane(a.nmap_g_prev, uy + 2 * rows, ux));
    float dist = norm(vprev_g - vcurr_g);
    float sine = norm(cross(ncurr_g, nprev_g));
    if (a.error_map) row_ptr(a.error_map, a.error_pitch, y)[x] = isfinite(dist) ? dist : 0.0f;
    found = (sine < a.angleThres && dist <= a.distThres && !isnan(ncurr.x) && !isnan(nprev_g.x));
    if (found) {
      float3 s_cp = vcurr_cp;  // Rprev_inv * (vcurr_g - tprev), same expression as above
      float3 d_cp = mul(P.Rprev_inv, vprev_g - tprev);
      float3 n_cp = mul(P.Rprev_inv, nprev_g);
      float3 c = cross(s_cp, n_cp);
      row[0] = n_cp.x;
      row[1] = n_cp.y;
      row[2] = n_cp.z;
      row[3] = c.x;
      row[4] = c.y;
      row[5] = c.z;
      row[6] = dot(n_cp, s_cp - d_cp);
    }
  }
  accumulate_se3(acc, row, found);
}

// --------------------------------------------------------------------------------- RGB residual
__device__ __forceinline__ bool rgb_residual_pixel(const RgbResidualArgs& a, const RgbWarp& Wp, int j0,
                                                   int i, DataTerm& corres, int& sq) {
  corres.valid = false;
  corres.zero = make_short2(0, 0);
  corres.one = make_short2(0, 0);
  corres.diff = 0.f;
  sq = 0;
  const int cols = a.cols, rows = a.rows;
  if (!(j0 < cols - 5 && i < rows - 1)) return false;
  // all 16 loads are issued unconditionally (a short-circuit && would serialise 16 L2 round trips)
  unsigned nz = 1u;
  for (int u = max(i - 2, 0); u < min(i + 2, rows); u++) {
    const unsigned char* r = row_ptr(a.nextImage, a.img_pitch, u);
    for (int v = max(j0 - 2, 0); v < min(j0 + 2, cols); v++) nz &= (unsigned)(__ldg(r + v) > 0);
  }
  if (!nz) return false;
  short valx = __ldg(row_ptr(a.dIdx, a.grad_pitch, i) + j0);
  short valy = __ldg(row_ptr(a.dIdy, a.grad_pitch, i) + j0);
  float mTwo = (float)((valx * valx) + (valy * valy));
  if (!(mTwo >= a.minScale)) return false;
  const int y = i, x = j0;
  float d1 = __ldg(row_ptr(a.nextDepth, a.depth_pitch, y) + x);
  if (isnan(d1)) return false;
  const float* k = Wp.krkinv.m;
  float transformed_d1 = d1 * (k[6] * x + k[7] * y + k[8]) + Wp.kt[2];
  int u0 = __float2int_rn((d1 * (k[0] * x + k[1] * y + k[2]) + Wp.kt[0]) / transformed_d1);
  int v0 = __float2int_rn((d1 * (k[3] * x + k[4] * y + k[5]) + Wp.kt[1]) / transformed_d1);
  if (!(u0 >= 0 && v0 >= 0 && u0 < cols && v0 < rows)) return false;
  float d0 = __ldg(row_ptr(a.lastDepth, a.depth_pitch, v0) + u0);
  unsigned char li = __ldg(row_ptr(a.lastImage, a.img_pitch, v0) + u0);
  if (!(d0 > 0 && fabsf(transformed_d1 - d0) <= a.maxDepthDelta && li != 0)) return false;
  corres.zero = make_short2((short)u0, (short)v0);
  corres.one = make_short2((short)x, (short)y);
  corres.diff = (float)__ldg(row_ptr(a.nextImage, a.img_pitch, y) + x) - (float)li;
  corres.valid = true;
  sq = (int)(corres.diff * corres.diff);  // float -> int truncation, reduce.cu:851
  return true;
}

// ------------------------------------------------------------------------------------- RGB step
__device__ __forceinline__ void rgb_step_pixel(const RgbStepArgs& a, float sigma, const DataTerm& c,
                                               float (&acc)[32]) {
  float row[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  bool found = c.valid;
  if (found) {
    float w = sigma + fabsf(c.diff);
    w = w > 1.19209290E-07F ? 1.0f / w : 1.0f;
    if (sigma == -1.f) w = 1.f;
    row[6] = -w * c.diff;
    const float* cp = (const float*)((const char*)a.cloud + (size_t)c.zero.y * a.cloud_pitch) + 3 * c.zero.x;
    float3 P = make_float3(__ldg(cp), __ldg(cp + 1), __ldg(cp + 2));
    float invz = (float)(1.0 / (double)P.z);
    float dI_dx_val = w * a.sobelScale * (float)__ldg(row_ptr(a.dIdx, a.grad_pitch, c.one.y) + c.one.x);
    float dI_dy_val = w * a.sobelScale * (float)__ldg(row_ptr(a.dIdy, a.grad_pitch, c.one.y) + c.one.x);
    float v0 = dI_dx_val * a.fx * invz;
    float v1 = dI_dy_val * a.fy * invz;
    float v2 = -(v0 * P.x + v1 * P.y) * invz;
    row[0] = v0;
    row[1] = v1;
    row[2] = v2;
    row[3] = -P.z * v1 + P.y * v2;
    row[4] = P.z * v0 - P.x * v2;
    row[5] = -P.y * v0 + P.x * v1;
  }
  accumulate_se3(acc, row, found);
}

// ------------------------------------------------------------------------------------------ SO3
__device__ __forceinline__ float2 so3_gradient(const unsigned char* img, size_t pitch, int x, int y) {
  const unsigned char* r = row_ptr(img, pitch, y);
  float actu = (float)__ldg(r + x);
  float back = (float)__ldg(r + x - 1), fore = (float)__ldg(r + x + 1);
  float2 g;
  g.x = ((back + actu) / 2.0f) - ((fore + actu) / 2.0f);
  back = (float)__ldg(row_ptr(img, pitch, y - 1) + x);
  fore = (float)__ldg(row_ptr(img, pitch, y + 1) + x);
  g.y = ((back + actu) / 2.0f) - ((fore + actu) / 2.0f);
  return g;
}

__device__ __forceinline__ void so3_pixel(const unsigned char* lastImage, const unsigned char* nextImage,
                                          size_t img_pitch, int cols, int rows, const Mat33& imageBasis,
                                          const Mat33& kinv, const Mat33& krlr, int x, int y, float (&acc)[32]) {
    float3 unwarped = make_float3((float)x, (float)y, 1.0f);
    float3 warped = mul(imageBasis, unwarped);
    int wx = __float2int_rn(warped.x / warped.z), wy = __float2int_rn(warped.y / warped.z);
    bool found = (wx >= 1 && wx < cols - 1 && wy >= 1 && wy < rows - 1 && x >= 1 && x < cols - 1 &&
                  y >= 1 && y < rows - 1);
    float row[4] = {0.f, 0.f, 0.f, 0.f};
    if (found) {
      float2 gN = so3_gradient(nextImage, img_pitch, wx, wy);
      float2 gL = so3_gradient(lastImage, img_pitch, x, y);
      float gx = (gN.x + gL.x) / 2.0f, gy = (gN.y + gL.y) / 2.0f;
      float3 point = mul(kinv, unwarped);
      float z2 = point.z * point.z;
      const float* K = krlr.m;
      float3 left = make_float3(
          ((point.z * (K[3] * gy + K[0] * gx)) - (gy * K[6] * y) - (gx * K[6] * x)) / z2,
          ((point.z * (K[4] * gy + K[1] * gx)) - (gy * K[7] * y) - (gx * K[7] * x)) / z2,
          ((point.z * (K[5] * gy + K[2] * gx)) - (gy * K[8] * y) - (gx * K[8] * x)) / z2);
      float3 jac = cross(left, point);
      row[0] = jac.x;
      row[1] = jac.y;
      row[2] = jac.z;
      row[3] = -((float)__ldg(row_ptr(nextImage, img_pitch, wy) + wx) -
                 (float)__ldg(row_ptr(lastImage, img_pitch, y) + x));
    }
    int q = 0;
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
      for (int r = p; r < 4; ++r) acc[q++] += row[p] * row[r];
    acc[9] += row[3] * row[3];
    acc[10] += found ? 1.f : 0.f;
}

}  // namespace dev
}  // namespace cfb
