// Per-Gaussian kernels: projection + cull + 2-D covariance (forward / backward), legacy
// helpers (world2camera, jacobian) and the fused frame-path variants that also apply the
// parameter activations and the tile-rectangle rule.  All HBM-bound streaming kernels.
#include "internal.h"

namespace {

constexpr int kBlock = 256;

__global__ void __launch_bounds__(kBlock) jacobian_kernel(const float* __restrict__ pc, int n,
                                                           float* __restrict__ jac) {
  int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  float u0 = pc[3 * i], u1 = pc[3 * i + 1], u2 = pc[3 * i + 2];   // gaussian.cu:10-39
  float rs = rsqrtf(u0 * u0 + u1 * u1 + u2 * u2);
  float* j = jac + 9 * (size_t)i;
  j[0] = 1.f / u2;
  j[1] = 0.f;
  j[2] = -u0 / (u2 * u2);
  j[3] = 0.f;
  j[4] = 1.f / u2;
  j[5] = -u1 / (u2 * u2);
  j[6] = rs * u0;
  j[7] = rs * u1;
  j[8] = rs * u2;
}

// ---------------------------------------------------------------------------------------
// Fused frame path.  Activations (splatter.py:519-524,:539-540) are applied in-register.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void load_activated(const float* __restrict__ quat, const float* __restrict__ scale,
                                               int i, int scale_act, float q[4], float s[3], float raw_s[3],
                                               float& qnorm) {
  float4 q4 = reinterpret_cast<const float4*>(quat)[i];
  qnorm = sqrtf(q4.x * q4.x + q4.y * q4.y + q4.z * q4.z + q4.w * q4.w);
  q[0] = q4.x / qnorm;
  q[1] = q4.y / qnorm;
  q[2] = q4.z / qnorm;
  q[3] = q4.w / qnorm;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    raw_s[k] = scale[3 * i + k];
    s[k] = (scale_act == GS_SCALE_ABS) ? (fabsf(raw_s[k]) + 1e-4f) : expf(raw_s[k]);
  }
}

__global__ void __launch_bounds__(kBlock) fused_project_kernel(
    const float* __restrict__ pos, const float* __restrict__ rgb, const float* __restrict__ opa,
    const float* __restrict__ quat, const float* __restrict__ scale, int n, int d, int scale_act, GsCam cam,
    GsTileGrid grid, float near_plane, float half_w, float half_h, GsRec* __restrict__ rec,
    uint32_t* __restrict__ count, uint32_t* __restrict__ dkey, int64_t* __restrict__ mask,
    unsigned int* __restrict__ n_visible) {
  int i = blockIdx.x * kBlock + threadIdx.x;
  bool vis = false;
  uint32_t cnt = 0;
  if (i < n) {
    float p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
    float q[4], s[3], raw_s[3], qn;
    load_activated(quat, scale, i, scale_act, q, s, raw_s, qn);
    GsProj o = gs_project(cam, p, q, s, near_plane, half_w, half_h);
    vis = o.visible;
    if (mask) mask[i] = o.visible ? 1 : 0;
    if (o.visible) {
      uint32_t tx0, tx1, ty0, ty1;
      if (gs_tile_rect(grid, o.x, o.y, o.a, o.b, o.c, o.d, tx0, tx1, ty0, ty1)) {
        cnt = (tx1 - tx0) * (ty1 - ty0);
        GsConic k = gs_make_conic(o.a, o.b, o.c, o.d);
        float op = gs_sigmoid(opa[i]);
        GsRec* r = rec + i;
        r->a = make_float4(o.x, o.y, k.ca, k.cb);
        // RGB colour = sigmoid(logit) (splatter.py:539); SH coefficients stay raw and are gathered
        // from the parameter tensor by the pack pass
        float cr = 0.f, cg = 0.f, cb = 0.f;
        if (d == 3) {
          cr = gs_sigmoid(rgb[3 * i]);
          cg = gs_sigmoid(rgb[3 * i + 1]);
          cb = gs_sigmoid(rgb[3 * i + 2]);
        }
        r->b = make_float4(k.cc, log2f(op), cr, cg);
        r->c = make_float4(cb, o.depth, __uint_as_float(tx0 | (ty0 << 16)),
                           __uint_as_float((tx1 - tx0) | ((ty1 - ty0) << 16)));
        r->d = make_uint4(0u, 0u, 0u, 0u);   // whole 32-byte sectors: a half-written sector is a DRAM read-modify-write (ECC)
      }
    }
    count[i] = cnt;
    // depth sort key: positive float bits order like the floats; Gaussians without instances last
    dkey[i] = cnt ? __float_as_uint(o.depth) : 0xffffffffu;
  }
  // 64-bit instance total next to the visible count (counters[2..3]): the u32 scans that follow
  // would wrap silently for M >= 2^32 (e.g. diverged scales: every Gaussian on every tile); the
  // host sizes the frame from this total and refuses instead
  __shared__ unsigned long long wsum[kBlock / 32];
  unsigned long long c64 = cnt;
#pragma unroll
  for (int o = 16; o; o >>= 1) c64 += __shfl_xor_sync(0xffffffffu, c64, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c64;
  int nv = __syncthreads_count(vis);
  if (threadIdx.x == 0) {
    unsigned long long tot = 0;
#pragma unroll
    for (int w = 0; w < kBlock / 32; ++w) tot += wsum[w];
    if (nv) atomicAdd(n_visible, (unsigned int)nv);
    if (tot) atomicAdd(reinterpret_cast<unsigned long long*>(n_visible + 2), tot);
  }
}

// Segment-sums the per-instance gradient records of each Gaussian (its instances occupy the
// contiguous rows offsets_g[i] .. + count[i]) and chains them to the RAW parameters.  No
// atomics anywhere: the result is deterministic.  Row layout (GW floats): d/d{x, y, ca, cb, cc,
// l2o} then D colour gradients (activated RGB for D == 3, raw SH coefficients otherwise).
// Destination of a run of `cnt` consecutive gradient floats that would land at `local` in this
// rank's flat bucket.  W == 0: the bucket itself.  W > 0 (data-parallel push, SURVEY.md §8e): the
// bucket is cut into W slices of `per` floats owned by rank 0..W-1; floats of another rank's slice
// are stored straight into slot `rank` of that owner's staging buffer over NVLink, so the reduce
// half of the gradient exchange overlaps this kernel.  Returns nullptr when the run straddles two
// slices (the caller then stores element by element).
template <int W>
__device__ __forceinline__ float* push_dst(const GsGradPush& P, float* local, int cnt) {
  if (W == 0) return local;
  const uint32_t idx = (uint32_t)(local - P.bucket);
  const uint32_t owner = idx / P.per;
  if (cnt > 1 && (idx + (uint32_t)cnt - 1) / P.per != owner) return nullptr;
  if (owner == (uint32_t)P.rank) return local;
  float* st = P.staging[0];
#pragma unroll
  for (int p = 1; p < (W > 0 ? W : 1); ++p)
    if (owner == (uint32_t)p) st = P.staging[p];
  return st + (size_t)P.rank * P.per + (idx - owner * P.per);
}

template <int W, int CNT>
__device__ __forceinline__ void push_store(const GsGradPush& P, float* local, const float* v) {
  float* dst = push_dst<W>(P, local, CNT);
  if (dst) {
#pragma unroll
    for (int k = 0; k < CNT; ++k) dst[k] = v[k];
  } else {
#pragma unroll
    for (int k = 0; k < CNT; ++k) *push_dst<W>(P, local + k, 1) = v[k];
  }
}

// Sum of the 12 camera-gradient floats of the block's 256 Gaussians, in double, in a fixed order (xor butterfly in
// each warp, then warps 0..7): one partial row per block, partial[blockIdx.x][12].
__device__ __forceinline__ void camgrad_block_reduce(const float gcam[12], double* __restrict__ partial) {
  __shared__ double red[kBlock / 32][12];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    double v = (double)gcam[k];
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kBlock / 32; ++w) s += red[w][threadIdx.x];
    partial[(size_t)blockIdx.x * 12 + threadIdx.x] = s;
  }
}

// DEPTH (maps frames, D == 3): float 9 of the rows is d/d|p_c| and is chained to pos; otherwise the depth is only a
// sort key.  CAMGRAD (RGB, one GPU): also the camera gradient of the block's Gaussians, one partial row per block
// into cam_partial (summed by camgrad_finish_kernel); every thread of the block takes part in that reduction.
template <int D, int GW, int W, bool DEPTH = false, bool CAMGRAD = false>
__global__ void __launch_bounds__(kBlock) fused_project_bwd_kernel(
    const float* __restrict__ pos, const float* __restrict__ rgb, const float* __restrict__ opa,
    const float* __restrict__ quat, const float* __restrict__ scale, int n, int scale_act, GsCam cam,
    float near_plane, float half_w, float half_h, const uint32_t* __restrict__ offsets_g,
    const uint32_t* __restrict__ count, const float* __restrict__ grad_inst,
    const uint32_t* __restrict__ row_epoch, uint32_t epoch, float* __restrict__ g_pos,
    float* __restrict__ g_rgb, float* __restrict__ g_opa, float* __restrict__ g_quat, float* __restrict__ g_scale,
    GsGradPush push, double* __restrict__ cam_partial) {
  static_assert(!CAMGRAD || (D == 3 && W == 0), "camera gradients: RGB colour on one GPU only");
  int i = blockIdx.x * kBlock + threadIdx.x;
  // SH colour on one GPU: the warp writes its coefficient gradients together (below), so threads past n stay
  constexpr bool kStagedRgb = (D != 3) && (W == 0);
  const bool valid = i < n;
  if (!valid && !kStagedRgb && !CAMGRAD) return;
  float gp[3] = {0.f, 0.f, 0.f}, gq_raw[4] = {0.f, 0.f, 0.f, 0.f}, gs_raw[3] = {0.f, 0.f, 0.f};
  float gcam[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) gcam[k] = 0.f;
  float go = 0.f;
  float acc[GW];
#pragma unroll
  for (int k = 0; k < GW; ++k) acc[k] = 0.f;
  const uint32_t cnt = valid ? count[i] : 0u;
  if (cnt > 0) {
    const uint32_t o0 = offsets_g[i], o1 = o0 + cnt;   // this Gaussian's contiguous gradient rows
    // issue the parameter loads BEFORE the row loop so that both round trips to HBM overlap
    float p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
    float q[4], s[3], raw_s[3], qn;
    load_activated(quat, scale, i, scale_act, q, s, raw_s, qn);
    const float opa_raw = opa[i];
    float rgb_raw[3] = {0.f, 0.f, 0.f};
    if (D == 3) {
      rgb_raw[0] = rgb[3 * i];
      rgb_raw[1] = rgb[3 * i + 1];
      rgb_raw[2] = rgb[3 * i + 2];
    }
    // (measured slower: loading the tags and rows of 4 instances at once - 0.180 vs 0.168 ms, 80 registers; a
    //  warp-cooperative version streaming the 32 Gaussians' contiguous row span through shared memory - 0.238 ms)
    for (uint32_t r = o0; r < o1; ++r) {
      if (row_epoch[r] != epoch) continue;     // instance not reached by its (saturated) tile: zero gradient
      const float4* row = reinterpret_cast<const float4*>(grad_inst + (size_t)r * GW);
#pragma unroll
      for (int qq = 0; qq < GW / 4; ++qq) {
        const float4 v = row[qq];
        acc[4 * qq] += v.x;
        acc[4 * qq + 1] += v.y;
        acc[4 * qq + 2] += v.z;
        acc[4 * qq + 3] += v.w;
      }
    }
    GsProj o = gs_project(cam, p, q, s, near_plane, half_w, half_h);
    // conic (ca, cb, cc) = (d, b+c, a) * sc,  sc = log2e / (2 det + 1e-14)
    float det = o.a * o.d - o.b * o.c;
    double pn = 2.0 * (double)det + 1e-14;
    float sc = (float)((double)GS_LOG2E / pn);
    float kk = 2.f * sc * sc / GS_LOG2E;                      // d sc / d det = -kk
    float gsc = acc[2] * o.d + acc[3] * (o.b + o.c) + acc[4] * o.a;
    float gcov[4];
    gcov[0] = acc[4] * sc - gsc * kk * o.d;                   // d det/da =  d
    gcov[1] = acc[3] * sc + gsc * kk * o.c;                   // d det/db = -c
    gcov[2] = acc[3] * sc + gsc * kk * o.b;                   // d det/dc = -b
    gcov[3] = acc[2] * sc - gsc * kk * o.a;                   // d det/dd =  a
    static_assert(!DEPTH || D == 3, "the depth gradient has a row slot in the RGB layout only");
    float gxyd[3] = {acc[0], acc[1], DEPTH ? acc[9] : 0.f};   // depth: sort key, + map gradient in maps frames
    float gq[4], gsv[3];
    gs_project_backward(cam, p, q, s, gxyd, gcov, gp, gq, gsv, CAMGRAD ? gcam : nullptr);
    // quat normalisation backward: q = r/|r|
    float dot = q[0] * gq[0] + q[1] * gq[1] + q[2] * gq[2] + q[3] * gq[3];
#pragma unroll
    for (int k = 0; k < 4; ++k) gq_raw[k] = (gq[k] - q[k] * dot) / qn;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (scale_act == GS_SCALE_ABS)
        gs_raw[k] = gsv[k] * (raw_s[k] > 0.f ? 1.f : (raw_s[k] < 0.f ? -1.f : 0.f));
      else
        gs_raw[k] = gsv[k] * expf(fminf(fmaxf(raw_s[k], -1.f), 1.f));   // renderer.py:98-100
    }
    float op = gs_sigmoid(opa_raw);
    // l2o = log2(op):  d/d logit = d_l2o / (op ln2) * op (1-op) = d_l2o (1-op) / ln2
    go = acc[5] * (1.f - op) / GS_LN2;
    if (D == 3) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        float c = gs_sigmoid(rgb_raw[k]);
        acc[6 + k] *= c * (1.f - c);
      }
    }
  }
  if (CAMGRAD && !valid) {
    // past n: no rows to store, zeros to the camera-gradient reduction below
  } else if (W == 0) {
    if constexpr (kStagedRgb) {
      // The 32 Gaussians of a warp own 32 * D contiguous floats of g_rgb.  One strided 4-byte store per coefficient
      // makes every store a partial-sector write (read-modify-write under ECC: 8x the bytes; 0.45 / 0.91 ms at
      // D = 27 / 48 against 0.17 ms for RGB): the rows go through shared memory and leave as whole sectors.
      // D = 48: two passes of 24 floats (96-byte, sector-aligned pieces); D = 27: the whole 32 x 108-byte span.
      constexpr int HW = (D % 8 == 0) ? D / 2 : D;
      __shared__ float stage[kBlock / 32][32][HW + 1];
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
      const int i0 = blockIdx.x * kBlock + warp * 32;
      const int nrow = min(32, n - i0);
#pragma unroll
      for (int pass = 0; pass < D / HW; ++pass) {
        __syncwarp();
#pragma unroll
        for (int k = 0; k < HW; ++k) stage[warp][lane][k] = acc[6 + pass * HW + k];
        __syncwarp();
        if (HW == D) {
          float* dst = g_rgb + (size_t)i0 * D;
          for (int t = lane; t < nrow * D; t += 32) dst[t] = stage[warp][t / D][t % D];
        } else {
          for (int t = lane; t < nrow * HW; t += 32) {
            const int g = t / HW, c = t % HW;
            g_rgb[(size_t)(i0 + g) * D + pass * HW + c] = stage[warp][g][c];
          }
        }
      }
      if (!valid) return;
    } else {
#pragma unroll
      for (int k = 0; k < D; ++k) g_rgb[(size_t)i * D + k] = acc[6 + k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      g_pos[3 * i + k] = gp[k];
      g_scale[3 * i + k] = gs_raw[k];
    }
    reinterpret_cast<float4*>(g_quat)[i] = make_float4(gq_raw[0], gq_raw[1], gq_raw[2], gq_raw[3]);
    g_opa[i] = go;
  } else {
    push_store<W, 3>(push, g_pos + 3 * (size_t)i, gp);
    push_store<W, 3>(push, g_scale + 3 * (size_t)i, gs_raw);
    push_store<W, D>(push, g_rgb + (size_t)i * D, acc + 6);
    // a quaternion is 4 floats at a 16-byte aligned bucket offset and `per` is a multiple of 4:
    // it never straddles two slices
    *reinterpret_cast<float4*>(push_dst<W>(push, g_quat + 4 * (size_t)i, 1)) =
        make_float4(gq_raw[0], gq_raw[1], gq_raw[2], gq_raw[3]);
    push_store<W, 1>(push, g_opa + i, &go);
  }
  if constexpr (CAMGRAD) camgrad_block_reduce(gcam, cam_partial);
}

// Sums the partial rows of the projection backward in block order, in double: warp k owns float k of the camera
// gradient (lane stride over the rows, then a fixed xor butterfly).  No atomics: bit-deterministic.  nblocks == 0
// (no Gaussian) writes zeros.
__global__ void __launch_bounds__(12 * 32) camgrad_finish_kernel(const double* __restrict__ partial, int nblocks,
                                                                 float* __restrict__ out) {
  const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += partial[(size_t)b * 12 + k];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[k] = (float)s;
}

}  // namespace

// The legacy API passes rot/tran as DEVICE pointers (torch tensors); the kernels read
// them through the read-only path so that no host synchronisation is needed.
namespace {
__global__ void __launch_bounds__(kBlock) project_fwd_kernel_p(const float* pos, const float* quat,
                                                                const float* scale, const float* rot,
                                                                const float* tran, int n, float near_plane,
                                                                float half_w, float half_h, float* res_pos,
                                                                float* res_cov, int64_t* mask) {
  GsCam cam;
#pragma unroll
  for (int k = 0; k < 9; ++k) cam.r[k] = __ldg(rot + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) cam.t[k] = __ldg(tran + k);
  int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  float p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
  float4 q4 = reinterpret_cast<const float4*>(quat)[i];
  float q[4] = {q4.x, q4.y, q4.z, q4.w};
  float s[3] = {scale[3 * i], scale[3 * i + 1], scale[3 * i + 2]};
  GsProj o = gs_project(cam, p, q, s, near_plane, half_w, half_h);
  if (!o.visible) return;
  mask[i] = 1;
  res_pos[3 * i] = o.x;
  res_pos[3 * i + 1] = o.y;
  res_pos[3 * i + 2] = o.depth;
  reinterpret_cast<float4*>(res_cov)[i] = make_float4(o.a, o.b, o.c, o.d);
}

__global__ void __launch_bounds__(kBlock) project_bwd_kernel_p(const float* pos, const float* quat,
                                                                const float* scale, const float* rot,
                                                                const float* tran, int n, const float* go_pos,
                                                                const float* go_cov, const int64_t* mask,
                                                                float* gi_pos, float* gi_quat, float* gi_scale) {
  GsCam cam;
#pragma unroll
  for (int k = 0; k < 9; ++k) cam.r[k] = __ldg(rot + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) cam.t[k] = __ldg(tran + k);
  int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  if (mask[i] == 0) return;
  float p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
  float4 q4 = reinterpret_cast<const float4*>(quat)[i];
  float q[4] = {q4.x, q4.y, q4.z, q4.w};
  float s[3] = {scale[3 * i], scale[3 * i + 1], scale[3 * i + 2]};
  float gx[3] = {go_pos[3 * i], go_pos[3 * i + 1], go_pos[3 * i + 2]};
  float4 gc4 = reinterpret_cast<const float4*>(go_cov)[i];
  float gc[4] = {gc4.x, gc4.y, gc4.z, gc4.w};
  float gp[3], gq[4], gs[3];
  gs_project_backward(cam, p, q, s, gx, gc, gp, gq, gs);
  gi_pos[3 * i] = gp[0];
  gi_pos[3 * i + 1] = gp[1];
  gi_pos[3 * i + 2] = gp[2];
  reinterpret_cast<float4*>(gi_quat)[i] = make_float4(gq[0], gq[1], gq[2], gq[3]);
  gi_scale[3 * i] = gs[0];
  gi_scale[3 * i + 1] = gs[1];
  gi_scale[3 * i + 2] = gs[2];
}

__global__ void __launch_bounds__(kBlock) w2c_fwd_kernel_p(const float* pos, const float* rot, const float* tran,
                                                            int n, float* res) {
  GsCam cam;
#pragma unroll
  for (int k = 0; k < 9; ++k) cam.r[k] = __ldg(rot + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) cam.t[k] = __ldg(tran + k);
  int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  float p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
  float pc[3];
  gs_world_to_cam(cam, p, pc);
  res[3 * i] = pc[0];
  res[3 * i + 1] = pc[1];
  res[3 * i + 2] = pc[2];
}

__global__ void __launch_bounds__(kBlock) w2c_bwd_kernel_p(const float* go, const float* rot, int n, float* gi) {
  float r[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) r[k] = __ldg(rot + k);
  int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  float g[3] = {go[3 * i], go[3 * i + 1], go[3 * i + 2]};
#pragma unroll
  for (int k = 0; k < 3; ++k) gi[3 * i + k] = g[0] * r[k] + g[1] * r[3 + k] + g[2] * r[6 + k];
}
}  // namespace

static inline int grid_for(int n) { return (n + kBlock - 1) / kBlock; }

extern "C" int gs_project_fwd(const float* pos, const float* quat, const float* scale, const float* rot,
                              const float* tran, int n, float near_plane, float half_width, float half_height,
                              float* res_pos, float* res_cov, int64_t* mask, gs_stream_t stream) {
  if (n < 0) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_project_fwd: n < 0");
  if (n == 0) return 0;
  project_fwd_kernel_p<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(pos, quat, scale, rot, tran, n, near_plane,
                                                                        half_width, half_height, res_pos, res_cov,
                                                                        mask);
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch();
  return 0;
}

extern "C" int gs_project_bwd(const float* pos, const float* quat, const float* scale, const float* rot,
                              const float* tran, const float* gradout_pos, const float* gradout_cov,
                              const int64_t* mask, int n, float* gradin_pos, float* gradin_quat,
                              float* gradin_scale, gs_stream_t stream) {
  if (n < 0) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_project_bwd: n < 0");
  if (n == 0) return 0;
  project_bwd_kernel_p<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(pos, quat, scale, rot, tran, n, gradout_pos,
                                                                        gradout_cov, mask, gradin_pos, gradin_quat,
                                                                        gradin_scale);
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch();
  return 0;
}

extern "C" int gs_w2c_fwd(const float* pos, const float* rot, const float* tran, int n, float* res,
                          gs_stream_t stream) {
  if (n <= 0) return n == 0 ? 0 : gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_w2c_fwd: n < 0");
  w2c_fwd_kernel_p<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(pos, rot, tran, n, res);
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch();
  return 0;
}

extern "C" int gs_w2c_bwd(const float* grad_out, const float* rot, int n, float* grad_in, gs_stream_t stream) {
  if (n <= 0) return n == 0 ? 0 : gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_w2c_bwd: n < 0");
  w2c_bwd_kernel_p<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(grad_out, rot, n, grad_in);
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch();
  return 0;
}

extern "C" int gs_jacobian(const float* pos_cam, int n, float* jac, gs_stream_t stream) {
  if (n <= 0) return n == 0 ? 0 : gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_jacobian: n < 0");
  jacobian_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(pos_cam, n, jac);
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch();
  return 0;
}

cudaError_t gs_launch_fused_project(const float* pos, const float* rgb, const float* opa, const float* quat,
                                    const float* scale, int n, int d, int scale_act, const GsCam& cam,
                                    const GsTileGrid& grid, float near_plane, float half_w, float half_h,
                                    GsRec* rec, uint32_t* count, uint32_t* dkey, int64_t* mask,
                                    unsigned int* n_visible, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  fused_project_kernel<<<grid_for(n), kBlock, 0, st>>>(pos, rgb, opa, quat, scale, n, d, scale_act, cam, grid,
                                                       near_plane, half_w, half_h, rec, count, dkey, mask, n_visible);
  return cudaGetLastError();
}

cudaError_t gs_launch_fused_project_bwd(const float* pos, const float* rgb, const float* opa, const float* quat,
                                        const float* scale, int n, int d, int scale_act, const GsCam& cam,
                                        float near_plane, float half_w, float half_h, const uint32_t* offsets_g,
                                        const uint32_t* count, const float* grad_inst, const uint32_t* row_epoch, uint32_t epoch,
                                        float* g_pos, float* g_rgb, float* g_opa,
                                        float* g_quat, float* g_scale, const GsGradPush& push, cudaStream_t st,
                                        bool depth_grad, double* cam_partial) {
  if (n == 0) return cudaSuccess;
  if (cam_partial && (d != 3 || push.world != 0)) return cudaErrorInvalidValue;
#define GS_LAUNCH_PBWD_RGB(DEPTH, CAMGRAD)                                                                          \
  fused_project_bwd_kernel<3, GS_GREC, 0, DEPTH, CAMGRAD><<<grid_for(n), kBlock, 0, st>>>(                         \
      pos, rgb, opa, quat, scale, n, scale_act, cam, near_plane, half_w, half_h, offsets_g, count, grad_inst,       \
      row_epoch, epoch, g_pos, g_rgb, g_opa, g_quat, g_scale, push, cam_partial)
  if (cam_partial) {
    if (depth_grad) GS_LAUNCH_PBWD_RGB(true, true);
    else GS_LAUNCH_PBWD_RGB(false, true);
    return cudaGetLastError();
  }
  if (depth_grad) {
    if (d != 3 || push.world != 0) return cudaErrorInvalidValue;
    GS_LAUNCH_PBWD_RGB(true, false);
    return cudaGetLastError();
  }
#undef GS_LAUNCH_PBWD_RGB
#define GS_LAUNCH_PBWD(D, GW, W)                                                                                    \
  fused_project_bwd_kernel<D, GW, W><<<grid_for(n), kBlock, 0, st>>>(pos, rgb, opa, quat, scale, n, scale_act, cam, \
                                                                     near_plane, half_w, half_h, offsets_g, count, \
                                                                     grad_inst, row_epoch, epoch, g_pos, g_rgb,    \
                                                                     g_opa, g_quat, g_scale, push, nullptr)
#define GS_LAUNCH_PBWD_W(D, GW)                  \
  switch (push.world) {                          \
    case 0: GS_LAUNCH_PBWD(D, GW, 0); break;     \
    case 2: GS_LAUNCH_PBWD(D, GW, 2); break;     \
    case 4: GS_LAUNCH_PBWD(D, GW, 4); break;     \
    case 8: GS_LAUNCH_PBWD(D, GW, 8); break;     \
    default: return cudaErrorInvalidValue;       \
  }
  if (d == 3) { GS_LAUNCH_PBWD_W(3, GS_GREC) }
  else if (d == 27) { GS_LAUNCH_PBWD_W(27, 36) }
  else { GS_LAUNCH_PBWD_W(48, 56) }
#undef GS_LAUNCH_PBWD_W
#undef GS_LAUNCH_PBWD
  return cudaGetLastError();
}

size_t gs_camgrad_partial_bytes(int n) { return (size_t)grid_for(n) * 12 * sizeof(double); }

cudaError_t gs_launch_camgrad_finish(const double* cam_partial, int n, float* grad_cam, cudaStream_t st) {
  camgrad_finish_kernel<<<1, 12 * 32, 0, st>>>(cam_partial, n > 0 ? grid_for(n) : 0, grad_cam);
  return cudaGetLastError();
}
