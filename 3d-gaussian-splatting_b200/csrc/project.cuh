// Per-Gaussian projection math shared by the legacy (global_culling) and fused kernels.
// Behaviour follows reference gaussian.cu:1131-1336 (forward) and :1371-1576 (backward);
// the arithmetic is re-derived (only the two image-plane rows of J*W are formed and
// cov2d = (J W R S)(J W R S)^T), it is not a transcription.
#pragma once
#include "gs_common.cuh"

struct GsCam {
  float r[9];
  float t[3];
};

struct GsProj {
  float x, y, depth;   // x/z, y/z, |p_c|
  float a, b, c, d;    // 2x2 covariance in normalised image-plane units
  bool visible;
};

struct GsRot {
  float m[9];
};

__device__ __forceinline__ GsRot gs_quat_to_rot(float w, float x, float y, float z) {
  GsRot R;
  R.m[0] = 1.f - 2.f * y * y - 2.f * z * z;
  R.m[1] = 2.f * x * y - 2.f * z * w;
  R.m[2] = 2.f * x * z + 2.f * y * w;
  R.m[3] = 2.f * x * y + 2.f * z * w;
  R.m[4] = 1.f - 2.f * x * x - 2.f * z * z;
  R.m[5] = 2.f * y * z - 2.f * x * w;
  R.m[6] = 2.f * x * z - 2.f * y * w;
  R.m[7] = 2.f * y * z + 2.f * x * w;
  R.m[8] = 1.f - 2.f * x * x - 2.f * y * y;
  return R;
}

__device__ __forceinline__ void gs_world_to_cam(const GsCam& cam, const float p[3], float pc[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
    pc[i] = cam.r[i * 3 + 0] * p[0] + cam.r[i * 3 + 1] * p[1] + cam.r[i * 3 + 2] * p[2] + cam.t[i];
}

// rows 0,1 of J*W with J = d(x/z, y/z)/d p_c evaluated at the un-clamped p_c
__device__ __forceinline__ void gs_jw_rows(const GsCam& cam, const float pc[3], float jw0[3], float jw1[3]) {
  float iz = 1.f / pc[2];
  float jx = -pc[0] / (pc[2] * pc[2]);
  float jy = -pc[1] / (pc[2] * pc[2]);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    jw0[k] = iz * cam.r[0 * 3 + k] + jx * cam.r[2 * 3 + k];
    jw1[k] = iz * cam.r[1 * 3 + k] + jy * cam.r[2 * 3 + k];
  }
}

// q (w,x,y,z) must be normalised and s activated by the caller.
__device__ __forceinline__ GsProj gs_project(const GsCam& cam, const float p[3], const float q[4],
                                             const float s[3], float near_plane, float half_w, float half_h) {
  GsProj o;
  o.visible = false;
  float pc[3];
  gs_world_to_cam(cam, p, pc);
  if (!(pc[2] > near_plane)) return o;                       // :1208  (z <= near culled)
  o.x = pc[0] / pc[2];
  o.y = pc[1] / pc[2];
  o.depth = sqrtf(pc[0] * pc[0] + pc[1] * pc[1] + pc[2] * pc[2]);
  if (fabsf(o.x) >= half_w || fabsf(o.y) >= half_h) return o;  // :1220
  o.visible = true;
  float jw0[3], jw1[3];
  gs_jw_rows(cam, pc, jw0, jw1);
  GsRot R = gs_quat_to_rot(q[0], q[1], q[2], q[3]);
  float m0[3], m1[3];                                         // M = (JW)(RS), 2x3
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    m0[c] = (jw0[0] * R.m[0 * 3 + c] + jw0[1] * R.m[1 * 3 + c] + jw0[2] * R.m[2 * 3 + c]) * s[c];
    m1[c] = (jw1[0] * R.m[0 * 3 + c] + jw1[1] * R.m[1 * 3 + c] + jw1[2] * R.m[2 * 3 + c]) * s[c];
  }
  o.a = m0[0] * m0[0] + m0[1] * m0[1] + m0[2] * m0[2];
  o.b = m0[0] * m1[0] + m0[1] * m1[1] + m0[2] * m1[2];
  o.c = o.b;
  o.d = m1[0] * m1[0] + m1[1] * m1[1] + m1[2] * m1[2];
  return o;
}

// Backward of gs_project for a visible Gaussian.  g_xyd = dL/d(x/z, y/z, depth),
// g_cov = dL/d(a,b,c,d).  Outputs dL/dp (world), dL/dq (wrt the NORMALISED quaternion
// entries as independent variables, like the reference), dL/ds (activated scale) and, when
// gcam is non-null, this Gaussian's share of dL/d(cam.r[9], cam.t[3]) (12 floats, written):
// p_c = R p + t and JW = J R with J detached, as for every other gradient here.
__device__ __forceinline__ void gs_project_backward(const GsCam& cam, const float p[3], const float q[4],
                                                    const float s[3], const float g_xyd[3],
                                                    const float g_cov[4], float gp[3], float gq[4],
                                                    float gs[3], float* gcam = nullptr) {
  float pc[3];
  gs_world_to_cam(cam, p, pc);
  float r = sqrtf(pc[0] * pc[0] + pc[1] * pc[1] + pc[2] * pc[2]);
  float iz = 1.f / pc[2];
  float ir = 1.f / r;
  float gc[3];
  gc[0] = g_xyd[0] * iz + g_xyd[2] * pc[0] * ir;                         // :1404-1406
  gc[1] = g_xyd[1] * iz + g_xyd[2] * pc[1] * ir;
  gc[2] = -(g_xyd[0] * pc[0] + g_xyd[1] * pc[1]) * iz * iz + g_xyd[2] * pc[2] * ir;
#pragma unroll
  for (int k = 0; k < 3; ++k) gp[k] = cam.r[0 * 3 + k] * gc[0] + cam.r[1 * 3 + k] * gc[1] + cam.r[2 * 3 + k] * gc[2];

  float jw0[3], jw1[3];
  gs_jw_rows(cam, pc, jw0, jw1);
  GsRot R = gs_quat_to_rot(q[0], q[1], q[2], q[3]);
  float m0[3], m1[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    m0[c] = (jw0[0] * R.m[0 * 3 + c] + jw0[1] * R.m[1 * 3 + c] + jw0[2] * R.m[2 * 3 + c]) * s[c];
    m1[c] = (jw1[0] * R.m[0 * 3 + c] + jw1[1] * R.m[1 * 3 + c] + jw1[2] * R.m[2 * 3 + c]) * s[c];
  }
  // cov3 gradient G3 = JW2^T G2 JW2; d(RS) = (G3 + G3^T) RS = JW2^T (G2 + G2^T) M   (:1440-1519)
  float s00 = 2.f * g_cov[0], s01 = g_cov[1] + g_cov[2], s11 = 2.f * g_cov[3];
  float h0[3], h1[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    h0[c] = s00 * m0[c] + s01 * m1[c];
    h1[c] = s01 * m0[c] + s11 * m1[c];
  }
  float grs[9];
#pragma unroll
  for (int rr = 0; rr < 3; ++rr)
#pragma unroll
    for (int c = 0; c < 3; ++c) grs[rr * 3 + c] = jw0[rr] * h0[c] + jw1[rr] * h1[c];
  if (gcam) {
    // mean: dL/dt = gc, dL/dR[a][b] = gc[a] p[b].  Covariance: dL/d(JW)[r][k] = sum_c h_r[c] RS[k][c], chained
    // through the image-plane rows (iz, 0, jx), (0, iz, jy) of J (gs_jw_rows).
    const float jx = -pc[0] / (pc[2] * pc[2]);
    const float jy = -pc[1] / (pc[2] * pc[2]);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      gcam[9 + a] = gc[a];
#pragma unroll
      for (int b = 0; b < 3; ++b) gcam[a * 3 + b] = gc[a] * p[b];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float gjw0 = 0.f, gjw1 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float rs = R.m[k * 3 + c] * s[c];
        gjw0 += h0[c] * rs;
        gjw1 += h1[c] * rs;
      }
      gcam[k] += iz * gjw0;
      gcam[3 + k] += iz * gjw1;
      gcam[6 + k] += jx * gjw0 + jy * gjw1;
    }
  }
  float gR[9];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    gs[c] = grs[0 * 3 + c] * R.m[0 * 3 + c] + grs[1 * 3 + c] * R.m[1 * 3 + c] + grs[2 * 3 + c] * R.m[2 * 3 + c];  // :1522-1526
#pragma unroll
    for (int rr = 0; rr < 3; ++rr) gR[rr * 3 + c] = grs[rr * 3 + c] * s[c];
  }
  float w = q[0], x = q[1], y = q[2], z = q[3];
  gq[0] = 2.f * (-z * gR[1] + y * gR[2] + z * gR[3] - x * gR[5] - y * gR[6] + x * gR[7]);
  gq[1] = 2.f * (y * gR[1] + z * gR[2] + y * gR[3] - 2.f * x * gR[4] - w * gR[5] + z * gR[6] + w * gR[7] - 2.f * x * gR[8]);
  gq[2] = 2.f * (-2.f * y * gR[0] + x * gR[1] + w * gR[2] + x * gR[3] + z * gR[5] - w * gR[6] + z * gR[7] - 2.f * y * gR[8]);
  gq[3] = 2.f * (-2.f * z * gR[0] - w * gR[1] + x * gR[2] + w * gR[3] - 2.f * z * gR[4] + y * gR[5] + x * gR[6] + y * gR[7]);
}

// Tile rectangle covered by a Gaussian, method 2 "prob2" (gaussian.cu:226-242): axis aligned
// bbox of the `thresh` iso-probability ellipse; float->uint32 casts truncate / saturate.
struct GsTileGrid {
  float lx, ly, leftmost, topmost, t2;   // t2 = -2*logf(thresh)
  int ntx, nty;
};

__device__ __forceinline__ bool gs_tile_rect(const GsTileGrid& g, float cx, float cy, float a, float b, float c,
                                             float d, uint32_t& tx0, uint32_t& tx1, uint32_t& ty0, uint32_t& ty1) {
  float det = a * d - b * c;
  if (det <= 0.f) return false;                                              // :227
  float ai = (float)((double)d / ((double)det + 1e-14));                     // :229
  float di = (float)((double)a / ((double)det + 1e-14));                     // :232
  float shift_x = sqrtf(di * g.t2 * det);
  float shift_y = sqrtf(ai * g.t2 * det);
  float right = cx + shift_x, left = cx - shift_x;
  float top = cy - shift_y, bottom = cy + shift_y;
  ty0 = (uint32_t)fmaxf((top - g.topmost) / g.ly, 0.f);                      // :241
  ty1 = (uint32_t)((bottom - g.topmost) / g.ly + 1.f);
  tx0 = (uint32_t)fmaxf((left - g.leftmost) / g.lx, 0.f);                    // :242
  tx1 = (uint32_t)((right - g.leftmost) / g.lx + 1.f);
  ty1 = min(ty1, (uint32_t)g.nty);
  tx1 = min(tx1, (uint32_t)g.ntx);
  return (ty1 > ty0) && (tx1 > tx0);
}
