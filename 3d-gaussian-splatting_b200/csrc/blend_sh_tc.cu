// Tile blend with per-pixel SH colour on the 5th-generation tensor cores (tcgen05, accumulators in TMEM).
//
// The two dense contractions of the SH path (reference gaussian.cu:936-948 forward colour, :665-689 backward)
//   logit[pixel, (instance, channel)] = sum_q SH_q(pixel) * coef[instance, channel, q]                  (forward + backward)
//   d coef[(instance, channel), q]    = sum_pixel d logit[pixel, (instance, channel)] * SH_q(pixel)     (backward)
// are the only GEMM-shaped work of the rasterizer: 3K (forward) / 2 * 3K (backward) FMAs per (pixel, instance), i.e.
// 27 of the 57 and 54 of the 137 instructions the scalar kernels (blend_sh.cu) issue per warp and 32 pairs at K = 9.
// Here ONE THREAD OWNS ONE PIXEL:
//   * a tile is 256 pixels = two M = 128 accumulator blocks; the SH basis of the tile is written once to shared
//     memory as bf16 hi + lo parts (x = hi + lo to 2^-17) in the no-swizzle canonical layout, whose image is at the
//     same time the K-major A operand of the first and the MN-major B operand of the second contraction;
//   * per round of 16 instances the raw coefficients (gathered by cp.async, as in blend_sh.cu) are split into
//     bf16 hi / lo K-major B operands [48 x 16] (pre-multiplied by -log2 e), three MMAs per block
//     (hi*hi + hi*lo + lo*hi, fp32 accumulate: logits to ~2e-5 relative) leave the logits of 16 instances x 3
//     channels in 48 TMEM columns of the lane (= pixel) that blends them: tcgen05.ld 32x32b hands every thread
//     its own pixel's row, so the front-to-back recurrence stays a plain sequential loop;
//   * backward: the per-(pixel, instance) logit gradients are written back to shared memory as the MN-major A
//     operand [96 rows = (hi | lo) x 3 channels x 16 instances, K = 256 pixels] and contracted with the basis
//     image (N = 32 = hi | lo) by 16 K = 16 MMAs; the six geometry sums per instance keep the warp-shuffle reduction.
// Layouts / descriptor encodings: tc_common.cuh (validated by profiles/r2_micro/umma_probe.cu).
#include <cstddef>

#include "internal.h"
#include "sh_common.cuh"
#include "tc_common.cuh"

namespace {

using namespace gs_sh;
using namespace gs_tc;

constexpr int TC_J = 16;     // instances per round
constexpr int TC_NT = 256;   // threads per CTA = pixels per tile

template <int K, int STAGES>
struct TcStage {
  float4 R[STAGES][TC_J * 4];
  float S[STAGES][TC_J * sh_sw(K)];
  uint64_t full[STAGES];
};

// TC_NT / 16 threads per instance: record (3 x 16 B), first gradient row (backward), raw coefficients
template <int K, int STAGES, bool BWD>
__device__ __forceinline__ void tc_gather(TcStage<K, STAGES>& sm, int stage, const GsRec* __restrict__ grec,
                                          const float* __restrict__ rgb, const uint32_t* __restrict__ ids,
                                          const uint32_t* __restrict__ goff, int base, int n, int tid) {
  constexpr int SW = sh_sw(K), D = 3 * K, TPI = TC_NT / TC_J;   // threads per instance
  static_assert(TPI >= 4, "the record pieces and the row offset need four threads");
  const int i = tid / TPI, l = tid % TPI;
  if (i < n) {
    const uint32_t id = ids[base + i];
    const uint32_t dr = gs_smem_u32(&sm.R[stage][i * 4]);
    if (l < 3) {
      const float4* src4 = reinterpret_cast<const float4*>(grec + id) + l;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dr + 16u * l), "l"(src4) : "memory");
    } else if (BWD && l == 3) {
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dr + 48u), "l"(goff + id) : "memory");
    }
    const float* src = rgb + (size_t)id * D;
    const uint32_t ds = gs_smem_u32(&sm.S[stage][i * SW]);
    if ((D * 4) % 16 == 0) {
      for (int q = l; q < D / 4; q += TPI)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ds + 16u * q), "l"(src + 4 * q) : "memory");
    } else {
      for (int q = l; q < D; q += TPI)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(ds + 4u * q), "l"(src + q) : "memory");
    }
  }
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(gs_smem_u32(&sm.full[stage])) : "memory");
}

// raw coefficients of one round -> K-major bf16 operands [n = channel * 16 + instance][q], scaled by -log2 e
// (the blend needs 2^(-logit * log2 e)); element (n, q) lives in 16-byte unit (q / 8) * 48 + n.  q >= K stays 0.
template <int K>
__device__ __forceinline__ void tc_split_coefs(const float* __restrict__ S, uint4* __restrict__ bc_hi,
                                               uint4* __restrict__ bc_lo, int tid) {
  constexpr int SW = sh_sw(K);
  if ((unsigned)tid < 96u) {
    const int n = tid % 48, g = tid / 48, c = n >> 4, j = n & 15;
    const float* src = S + j * SW + c * K + g * 8;
    uint32_t h[4], l[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float v0 = (g * 8 + 2 * w < K) ? -GS_LOG2E * src[2 * w] : 0.f;
      const float v1 = (g * 8 + 2 * w + 1 < K) ? -GS_LOG2E * src[2 * w + 1] : 0.f;
      split_bf16x2(v0, v1, h[w], l[w]);
    }
    bc_hi[g * 48 + n] = make_uint4(h[0], h[1], h[2], h[3]);
    bc_lo[g * 48 + n] = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// SH basis of this thread's pixel -> bf16 hi / lo operand image: 16-byte unit (q / 8) * 256 + pixel
template <int K>
__device__ __forceinline__ void tc_store_basis(const float* sh, uint4* __restrict__ img_hi, uint4* __restrict__ img_lo,
                                               int pixel) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float v0 = (g * 8 + 2 * w < K) ? sh[g * 8 + 2 * w] : 0.f;
      const float v1 = (g * 8 + 2 * w + 1 < K) ? sh[g * 8 + 2 * w + 1] : 0.f;
      split_bf16x2(v0, v1, h[w], l[w]);
    }
    img_hi[g * 256 + pixel] = make_uint4(h[0], h[1], h[2], h[3]);
    img_lo[g * 256 + pixel] = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// logits of one round: D[block][pixel, n] = basis[pixel, :] . coef[n, :]   (3 MMAs per 128-pixel block)
__device__ __forceinline__ void tc_issue_logits(uint32_t tm, const uint4* img_hi, const uint4* img_lo, const uint4* bc_hi,
                                                const uint4* bc_lo, uint64_t* bar) {
  constexpr uint32_t idesc = idesc_bf16(0, 0, 128, 48);
  const uint64_t b_hi = smem_desc(gs_smem_u32(bc_hi), 768, 128), b_lo = smem_desc(gs_smem_u32(bc_lo), 768, 128);
#pragma unroll
  for (int b = 0; b < 2; ++b) {
    const uint64_t a_hi = smem_desc(gs_smem_u32(img_hi) + b * 2048, 4096, 128);
    const uint64_t a_lo = smem_desc(gs_smem_u32(img_lo) + b * 2048, 4096, 128);
    mma_bf16(tm + b * 48, a_hi, b_hi, idesc, 0);
    mma_bf16(tm + b * 48, a_hi, b_lo, idesc, 1);
    mma_bf16(tm + b * 48, a_lo, b_hi, idesc, 1);
  }
  mma_commit(bar);
}

// three sigmoids from v_c = -logit_c * log2 e with ONE reciprocal (see blend_sh.cu)
__device__ __forceinline__ void tc_colours(float v0, float v1, float v2, float* col) {
  const float d0 = 1.f + gs_ex2(fminf(v0, 40.f)), d1 = 1.f + gs_ex2(fminf(v1, 40.f)), d2 = 1.f + gs_ex2(fminf(v2, 40.f));
  const float d01 = d0 * d1;
  const float r = gs_rcp(d01 * d2);
  col[2] = r * d01;
  const float r2 = r * d2;
  col[0] = r2 * d1;
  col[1] = r2 * d0;
}

// ---------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------
template <int K>
struct TcFwdSmem {
  uint4 img_hi[2 * 256];
  uint4 img_lo[2 * 256];
  uint4 bc_hi[2 * 48];
  uint4 bc_lo[2 * 48];
  TcStage<K, 4> st;
  uint64_t mma_bar;
  uint32_t tmem_base;
};

template <int K>
__global__ void __launch_bounds__(TC_NT) blend_sh_fwd_tc_kernel(const GsRec* __restrict__ grec, const float* __restrict__ rgb,
                                                                const uint32_t* __restrict__ ids,
                                                                const int* __restrict__ tile_accum, int wp, int hp, int ntx,
                                                                float fx, float fy, const float* __restrict__ rays_o,
                                                                const float* __restrict__ lefttop,
                                                                const float* __restrict__ vdx, const float* __restrict__ vdy,
                                                                float* __restrict__ image, int* __restrict__ tile_neff,
                                                                float* __restrict__ final_img, GsCrop crop) {
  constexpr int STAGES = 4, TCOLS = 128;
  __shared__ __align__(128) TcFwdSmem<K> sm;
  const int tile = blockIdx.x, tid = threadIdx.x, warp = tid >> 5;
  const int tx = tile % ntx, ty = tile / ntx;
  const int ix = tx * GS_TILE + (tid & 15), iy = ty * GS_TILE + (tid >> 4);
  const int start = tile_accum[tile];
  const int cnt = tile_accum[tile + 1] - start;
  float T = 1.f, cr = 0.f, cg = 0.f, cb = 0.f;
  int consumed = cnt;
  if (cnt > 0) {                                              // uniform over the CTA
    const int nchunks = (cnt + TC_J - 1) / TC_J;
    if (tid == 0) {
      for (int s = 0; s < STAGES; ++s) gs_mbar_init(&sm.st.full[s], TC_NT);
      gs_mbar_init(&sm.mma_bar, 1);
      gs_fence_barrier_init();
    }
    if (warp == 0) tmem_alloc<TCOLS>(&sm.tmem_base);
    {
      float sh[16];
      pixel_sh<K>(ix, iy, rays_o, lefttop, vdx, vdy, sh);
      tc_store_basis<K>(sh, sm.img_hi, sm.img_lo, tid);
    }
    if (tid < 96) {                                           // q >= K columns of the coefficient operand stay zero
      sm.bc_hi[tid] = make_uint4(0, 0, 0, 0);
      sm.bc_lo[tid] = make_uint4(0, 0, 0, 0);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tm = sm.tmem_base;
    const uint32_t trow = tm + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(warp >> 2) * 48u;
    const float px = gs_pixel_coord(ix, wp, fx), py = gs_pixel_coord(iy, hp, fy);
    for (int k = 0; k < STAGES - 1 && k < nchunks; ++k)
      tc_gather<K, STAGES, false>(sm.st, k, grec, rgb, ids, nullptr, start + k * TC_J, min(TC_J, cnt - k * TC_J), tid);

    for (int k = 0; k < nchunks; ++k) {
      const int stage = k % STAGES;
      gs_mbar_wait(&sm.st.full[stage], (uint32_t)((k / STAGES) & 1));
      const int n = min(TC_J, cnt - k * TC_J);
      tc_split_coefs<K>(sm.st.S[stage], sm.bc_hi, sm.bc_lo, tid);
      fence_smem_to_async();
      fence_before_sync();
      // every thread has finished round k - 1 (its TMEM reads, its staged rows); all pixels saturated -> done
      if (__syncthreads_and(!(T > GS_T_STOP))) {
        consumed = k * TC_J;
        break;
      }
      if (warp == 0) {
        if (elect_one()) {
          fence_after_sync();
          tc_issue_logits(tm, sm.img_hi, sm.img_lo, sm.bc_hi, sm.bc_lo, &sm.mma_bar);
        }
        __syncwarp();
      }
      if (k + STAGES - 1 < nchunks) {
        const int kn = k + STAGES - 1;
        tc_gather<K, STAGES, false>(sm.st, kn % STAGES, grec, rgb, ids, nullptr, start + kn * TC_J,
                                    min(TC_J, cnt - kn * TC_J), tid);
      }
      gs_mbar_wait(&sm.mma_bar, (uint32_t)(k & 1));
      fence_after_sync();
      const float4* R = sm.st.R[stage];
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        if (h * 8 >= n) break;
        if (__all_sync(0xffffffffu, !(T > GS_T_STOP))) break;
        float lr[8], lg[8], lb[8];
        tmem_ld8x3(trow + h * 8, trow + 16 + h * 8, trow + 32 + h * 8, lr, lg, lb);
        const float4* Rh = R + 32 * h;
        // one (pixel, instance) pair; a saturated pixel blends nothing (w = 0), without a divergent branch
        auto pair = [&](const float4 a, const float4 b4, float l0, float l1, float l2) {
          const float dx = px - a.x, dy = py - a.y;
          const float eu = fmaf(a.z, dx, -a.w * dy);
          const float ev = fmaf(-b4.x * dy, dy, b4.y);
          const float alpha = gs_ex2(fmaf(-dx, eu, ev));
          const float w = (T > GS_T_STOP) ? alpha * T : 0.f;
          float col[3];
          tc_colours(l0, l1, l2, col);
          cr = fmaf(col[0], w, cr);
          cg = fmaf(col[1], w, cg);
          cb = fmaf(col[2], w, cb);
          T -= w;
        };
        if (h * 8 + 8 <= n) {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) pair(Rh[4 * jj], Rh[4 * jj + 1], lr[jj], lg[jj], lb[jj]);
        } else {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj)
            if (h * 8 + jj < n) pair(Rh[4 * jj], Rh[4 * jj + 1], lr[jj], lg[jj], lb[jj]);
        }
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<TCOLS>(tm);
  }
  float* o = image + ((size_t)iy * wp + ix) * 3;
  o[0] = cr;
  o[1] = cg;
  o[2] = cb;
  if (final_img) gs_store_final(final_img, ix, iy, crop.left, crop.top, crop.width, crop.height, cr, cg, cb);
  if (tile_neff && tid == 0) tile_neff[tile] = consumed;
}

// ---------------------------------------------------------------------------------------
// backward
// grad row (GS_SH_GREC(K) floats): d/d{x, y, ca, cb, cc, l2o}, d/d coef[0..3K)
// ---------------------------------------------------------------------------------------
template <int K>
struct TcBwdSmem {
  // A operand of the coefficient-gradient contraction, MN-major: 16-byte unit G * 256 + pixel holds the 8 rows
  // (instances 8h .. 8h+7 of channel c, hi or lo part) G = part * 6 + c * 2 + h of that pixel.  The M = 128
  // instruction reads 16 groups: the last four fall into img_hi / img_lo, which MUST follow (their rows are unused).
  uint4 dct[12 * 256];
  uint4 img_hi[2 * 256];
  uint4 img_lo[2 * 256];
  uint4 bc_hi[2 * 48];
  uint4 bc_lo[2 * 48];
  TcStage<K, 4> st;
  float part[2][8][TC_J][8];   // per-warp sums of the six geometry values (by round parity)
  float epi[48][17];           // (lo part) . basis, staged for the thread that owns the hi row
  uint64_t mma_bar, mma2_bar;
  uint32_t tmem_base;
};

template <int K>
__global__ void __launch_bounds__(TC_NT) blend_sh_bwd_tc_kernel(const GsRec* __restrict__ grec, const float* __restrict__ rgb,
                                                                const uint32_t* __restrict__ ids,
                                                                const uint32_t* __restrict__ goff,
                                                                const int* __restrict__ tile_accum, int wp, int hp, int ntx,
                                                                float fx, float fy, const float* __restrict__ rays_o,
                                                                const float* __restrict__ lefttop,
                                                                const float* __restrict__ vdx, const float* __restrict__ vdy,
                                                                const float* __restrict__ image,
                                                                const float* __restrict__ grad_image,
                                                                float* __restrict__ grad_inst, int grad_is_final, GsCrop crop,
                                                                uint32_t* __restrict__ row_epoch, uint32_t epoch,
                                                                int* __restrict__ tile_neff_b) {
  constexpr int STAGES = 4, TCOLS = 256, NV = sh_nv(K), GREC = (NV + 3) / 4 * 4;
  constexpr uint32_t D2COL = 96;                            // logits: columns [0, 96); gradient accumulators: 2 x 32
  static_assert(offsetof(TcBwdSmem<K>, img_hi) == 12 * 256 * 16 && offsetof(TcBwdSmem<K>, img_lo) == 14 * 256 * 16,
                "the basis image must follow the gradient operand: descriptors address both as one region");
  extern __shared__ __align__(128) uint8_t tc_smem_raw[];
  TcBwdSmem<K>& sm = *reinterpret_cast<TcBwdSmem<K>*>(tc_smem_raw);
  const int tile = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tx = tile % ntx, ty = tile / ntx;
  const int ix = tx * GS_TILE + (tid & 15), iy = ty * GS_TILE + (tid >> 4);
  const int start = tile_accum[tile];
  const int cnt = tile_accum[tile + 1] - start;
  if (cnt == 0) return;
  const int nchunks = (cnt + TC_J - 1) / TC_J;
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) gs_mbar_init(&sm.st.full[s], TC_NT);
    gs_mbar_init(&sm.mma_bar, 1);
    gs_mbar_init(&sm.mma2_bar, 1);
    gs_fence_barrier_init();
  }
  if (warp == 0) tmem_alloc<TCOLS>(&sm.tmem_base);
  {
    float sh[16];
    pixel_sh<K>(ix, iy, rays_o, lefttop, vdx, vdy, sh);
    tc_store_basis<K>(sh, sm.img_hi, sm.img_lo, tid);
  }
  if (tid < 96) {
    sm.bc_hi[tid] = make_uint4(0, 0, 0, 0);
    sm.bc_lo[tid] = make_uint4(0, 0, 0, 0);
  }
  float T = 1.f, R, gr, gg, gb;
  {
    const size_t off = ((size_t)iy * wp + ix) * 3;
    const float raw[3] = {image[off], image[off + 1], image[off + 2]};
    if (!grad_is_final) {
      gr = grad_image[off];
      gg = grad_image[off + 1];
      gb = grad_image[off + 2];
    } else {
      gs_load_final_grad(grad_image, raw, ix, iy, crop.left, crop.top, crop.width, crop.height, gr, gg, gb);
    }
    R = gr * raw[0] + gg * raw[1] + gb * raw[2];
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = sm.tmem_base;
  const uint32_t tlane = (uint32_t)((warp & 3) * 32) << 16;
  const uint32_t trow = tm + tlane + (uint32_t)(warp >> 2) * 48u;
  const float px = gs_pixel_coord(ix, wp, fx), py = gs_pixel_coord(iy, hp, fy);
  for (int k = 0; k < STAGES - 1 && k < nchunks; ++k)
    tc_gather<K, STAGES, true>(sm.st, k, grec, rgb, ids, goff, start + k * TC_J, min(TC_J, cnt - k * TC_J), tid);

  // coefficient-gradient rows of the previous round: its contraction ran while this round's operands were prepared.
  // Rows 0 .. 95 of the accumulators live in TMEM lanes 0 .. 95 (warps 0 .. 2): (hi part) x (basis hi | lo) in rows
  // 0 .. 47, (lo part) x basis hi in rows 48 .. 95, summed by the thread that owns the hi row.
  // (np, Rp: instance count and staged records of THAT round - its stage is not refilled before the next barrier)
  auto epilogue = [&](int np, const float4* Rp) {
    if (warp < 3) {
      float a[32], b[32];
      tmem_ld32(tm + tlane + D2COL, a);
      tmem_ld32(tm + tlane + D2COL + 32, b);
      if (tid >= 48) {
#pragma unroll
        for (int q = 0; q < 16; ++q) sm.epi[tid - 48][q] = a[q] + b[q];
      }
      gs_bar_sync(1, 96);
      if (tid < 48) {
        const int c = tid >> 4, j = tid & 15;
        if (j < np) {
          const float4 cc = Rp[4 * j + 2];
          const uint32_t rxy = __float_as_uint(cc.z), rwh = __float_as_uint(cc.w);
          const uint32_t slot = __float_as_uint(Rp[4 * j + 3].x) + ((uint32_t)ty - (rxy >> 16)) * (rwh & 0xffffu) +
                                ((uint32_t)tx - (rxy & 0xffffu));
          float* out = grad_inst + (size_t)slot * GREC + 6 + c * K;
#pragma unroll
          for (int q = 0; q < K; ++q) out[q] = ((a[q] + b[q]) + (a[16 + q] + b[16 + q])) + sm.epi[tid][q];
        }
      }
    }
  };

  // one (pixel, instance) pair: blend state update, logit gradients dc[3], geometry values v[0..5]
  auto pair = [&](const float4 a, const float4 b4, float l0, float l1, float l2, float* dc, float* v) {
    const float dx = px - a.x, dy = py - a.y;
    const float eu = fmaf(a.z, dx, -a.w * dy);
    const float ev = fmaf(-b4.x * dy, dy, b4.y);
    const float alpha = gs_ex2(fmaf(-dx, eu, ev));
    const bool live = T > GS_T_STOP;                        // saturated pixels contribute exactly nothing
    const float w = live ? alpha * T : 0.f;
    float col[3];
    tc_colours(l0, l1, l2, col);
    const float gc = fmaf(gr, col[0], fmaf(gg, col[1], gb * col[2]));
    R = fmaf(-gc, w, R);
    const float rc = gs_rcp(1.0000001f - alpha);
    const float dal = fmaf(T, gc, -R * rc);
    const float e = live ? dal * alpha : 0.f;
    T -= w;
    const float ex = e * dx, ey = e * dy;
    v[0] = ex;
    v[1] = ey;
    v[2] = ex * dx;
    v[3] = ex * dy;
    v[4] = ey * dy;
    v[5] = e;
    v[6] = 0.f;
    v[7] = 0.f;
    // d colour_c / d logit_c = sigma'(.)      (gaussian.cu:666-674)
    dc[0] = gr * w * col[0] * (1.f - col[0]);
    dc[1] = gg * w * col[1] * (1.f - col[1]);
    dc[2] = gb * w * col[2] * (1.f - col[2]);
  };

  // Schedule of round k (ONE CTA-wide barrier per round; the tensor core works one step ahead / behind):
  //   wait logits(k)  ->  [96 threads: split the coefficients of round k + 1]  ->  first 8 instances  ->
  //   wait contraction(k - 1) (it read sm.dct)  ->  store their rows  ->  [warps 0-2: coefficient rows of round k - 1]
  //   ->  second 8 instances  ->  barrier + "all pixels saturated" vote  ->  issue logits(k + 1), then contraction(k)
  //   ->  [warp 4: geometry rows of round k]  ->  gather round k + 3.
  // What orders every producer / consumer pair (B(k) = the barrier of round k):
  //   staged records / coefficients   cp.async -> stage mbarrier (full[s]) -> every reader waits on it; a stage is refilled
  //                                   (round k + 3 into the stage of round k - 1) after B(k), its last readers (blend of
  //                                   k - 1, geometry rows, coefficient rows of k - 1) all run before B(k)
  //   bc_hi / bc_lo                   written (warps 5-7) after their wait on logits(k); read by logits(k + 1), issued after B(k)
  //   TMEM logits                     written by logits(k + 1) after B(k); all tcgen05.ld of round k precede B(k)
  //   sm.dct                          written after the wait on contraction(k - 1); read by contraction(k), issued after B(k)
  //   TMEM gradient accumulators      written by contraction(k) after B(k); read (warps 0-2) in round k + 1 after its mbarrier,
  //                                   before B(k + 1), after which contraction(k + 1) overwrites them
  //   sm.part[k & 1]                  written in round k; read by warp 4 after B(k); rewritten in round k + 2, after B(k + 1)
  //   sm.epi                          warps 0-2 only, named barrier 1; the next use lies behind B(k)
  int consumed = cnt, n_prev = 0, st_prev = 0;
  uint32_t par_prev = 0;
  gs_mbar_wait(&sm.st.full[0], 0);
  tc_split_coefs<K>(sm.st.S[0], sm.bc_hi, sm.bc_lo, tid);
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    if (elect_one()) {
      fence_after_sync();
      tc_issue_logits(tm, sm.img_hi, sm.img_lo, sm.bc_hi, sm.bc_lo, &sm.mma_bar);
    }
    __syncwarp();
  }
  for (int k = 0; k < nchunks; ++k) {
    const int stage = k % STAGES;
    const int n = min(TC_J, cnt - k * TC_J);
    gs_mbar_wait(&sm.st.full[stage], (uint32_t)((k / STAGES) & 1));   // records of this round
    gs_mbar_wait(&sm.mma_bar, (uint32_t)(k & 1));
    fence_after_sync();
    if (k + 1 < nchunks) {                                  // logits(k) are complete: the coefficient operand is free
      gs_mbar_wait(&sm.st.full[(k + 1) % STAGES], (uint32_t)(((k + 1) / STAGES) & 1));
      tc_split_coefs<K>(sm.st.S[(k + 1) % STAGES], sm.bc_hi, sm.bc_lo, tid - 160);   // warps 5 .. 7
    }
    const float4* Rr = sm.st.R[stage];
    float(*part)[8] = sm.part[k & 1][warp];
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      uint32_t hw[3][4], lw[3][4];
      const bool have = h * 8 < n;                          // uniform
      const bool idle = have && __all_sync(0xffffffffu, !(T > GS_T_STOP));
      if (have && !idle) {
        float lr[8], lg[8], lb[8];
        tmem_ld8x3(trow + h * 8, trow + 16 + h * 8, trow + 32 + h * 8, lr, lg, lb);
        const float4* Rh = Rr + 32 * h;
        float* ph = &part[h * 8][(lane >> 2) & 7];
        if (h * 8 + 8 <= n) {                               // all eight instances exist: no per-instance tests
#pragma unroll
          for (int jp = 0; jp < 4; ++jp) {
            float dc[2][3];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int jj = 2 * jp + u;
              float v[8];
              pair(Rh[4 * jj], Rh[4 * jj + 1], lr[jj], lg[jj], lb[jj], dc[u], v);
              const float r = reduce8(v, lane);
              if ((lane & 3) == 0) ph[jj * 8] = r;
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) split_bf16x2(dc[0][c], dc[1][c], hw[c][jp], lw[c][jp]);
          }
        } else {
#pragma unroll
          for (int jp = 0; jp < 4; ++jp) {
            float dc[2][3];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int jj = 2 * jp + u;
              dc[u][0] = dc[u][1] = dc[u][2] = 0.f;
              if (h * 8 + jj < n) {
                float v[8];
                pair(Rh[4 * jj], Rh[4 * jj + 1], lr[jj], lg[jj], lb[jj], dc[u], v);
                const float r = reduce8(v, lane);
                if ((lane & 3) == 0) ph[jj * 8] = r;
              }
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) split_bf16x2(dc[0][c], dc[1][c], hw[c][jp], lw[c][jp]);
          }
        }
      } else if (idle) {
        // nothing left to blend in this warp: the rows of this half round are zeros
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int q = 0; q < 4; ++q) hw[c][q] = lw[c][q] = 0u;
        part[h * 8 + (lane >> 2)][lane & 3] = 0.f;
        part[h * 8 + (lane >> 2)][4 + (lane & 3)] = 0.f;
      }
      if (h == 0 && n_prev > 0) {                           // the previous contraction has read sm.dct
        gs_mbar_wait(&sm.mma2_bar, par_prev);
        fence_after_sync();
      }
      if (have) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          sm.dct[(c * 2 + h) * 256 + tid] = make_uint4(hw[c][0], hw[c][1], hw[c][2], hw[c][3]);
          sm.dct[(6 + c * 2 + h) * 256 + tid] = make_uint4(lw[c][0], lw[c][1], lw[c][2], lw[c][3]);
        }
      }
      if (h == 0 && n_prev > 0) epilogue(n_prev, sm.st.R[(k - 1) % STAGES]);
    }
    fence_smem_to_async();
    fence_before_sync();
    const bool done = __syncthreads_and(!(T > GS_T_STOP)) != 0;   // operands of both contractions complete
    const bool more = !done && k + 1 < nchunks;
    if (warp == 0) {
      if (elect_one()) {
        fence_after_sync();
        if (more) tc_issue_logits(tm, sm.img_hi, sm.img_lo, sm.bc_hi, sm.bc_lo, &sm.mma_bar);
        constexpr uint32_t idesc2 = idesc_bf16(1, 1, 128, 32);
        const uint32_t a0 = gs_smem_u32(sm.dct), b0 = gs_smem_u32(sm.img_hi);
#pragma unroll
        for (int s = 0; s < 16; ++s)
          mma_bf16(tm + D2COL + (uint32_t)(s & 1) * 32u, smem_desc(a0 + s * 256, 128, 4096), smem_desc(b0 + s * 256, 128, 4096),
                   idesc2, s >= 2);
        mma_commit(&sm.mma2_bar);
      }
      __syncwarp();
    }
    // geometry rows (while the tensor core contracts): threads 128 .. 143, one instance each
    if (tid >= 128 && tid < 128 + n) {
      const int j = tid - 128;
      float s[6];
#pragma unroll
      for (int u = 0; u < 6; ++u) {
        float t = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) t += sm.part[k & 1][w8][j][u];
        s[u] = t;
      }
      const float4 a = Rr[4 * j];
      const float4 b4 = Rr[4 * j + 1];
      const float4 cc = Rr[4 * j + 2];
      const uint32_t rxy = __float_as_uint(cc.z), rwh = __float_as_uint(cc.w);
      const uint32_t slot = __float_as_uint(Rr[4 * j + 3].x) + ((uint32_t)ty - (rxy >> 16)) * (rwh & 0xffffu) +
                            ((uint32_t)tx - (rxy & 0xffffu));
      float* out = grad_inst + (size_t)slot * GREC;
      out[0] = GS_LN2 * (2.f * a.z * s[0] - a.w * s[1]);
      out[1] = GS_LN2 * (2.f * b4.x * s[1] - a.w * s[0]);
      out[2] = -GS_LN2 * s[2];
      out[3] = GS_LN2 * s[3];
      out[4] = -GS_LN2 * s[4];
      out[5] = GS_LN2 * s[5];
      row_epoch[slot] = epoch;
    }
    n_prev = n;
    par_prev = (uint32_t)(k & 1);
    st_prev = stage;
    if (done) {
      consumed = min(cnt, (k + 1) * TC_J);
      break;
    }
    // stage (k + 3) % 4 held round k - 1, whose records were last read before this round's barrier
    if (k + STAGES - 1 < nchunks) {
      const int kn = k + STAGES - 1;
      tc_gather<K, STAGES, true>(sm.st, kn % STAGES, grec, rgb, ids, goff, start + kn * TC_J, min(TC_J, cnt - kn * TC_J),
                                 tid);
    }
  }
  __syncthreads();
  if (n_prev > 0) {
    gs_mbar_wait(&sm.mma2_bar, par_prev);
    fence_after_sync();
    epilogue(n_prev, sm.st.R[st_prev]);
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc<TCOLS>(tm);
  if (tile_neff_b && tid == 0) tile_neff_b[tile] = consumed;
}

}  // namespace

cudaError_t gs_launch_blend_sh_fwd_tc(const GsRec* grec, const float* rgb, const uint32_t* ids, int d,
                                      const int* tile_accum, const GsFrameGeom& g, const GsRayPtrs& r, float* image,
                                      int* tile_neff, float* final_img, const GsCrop& crop, cudaStream_t st) {
#define GS_SHF_TC(K)                                                                                                  \
  blend_sh_fwd_tc_kernel<K><<<g.n_tiles, TC_NT, 0, st>>>(grec, rgb, ids, tile_accum, g.wp, g.hp, g.ntx, g.fx, g.fy,     \
                                                         r.rays_o, r.lefttop, r.dx, r.dy, image, tile_neff, final_img, \
                                                         crop)
  if (d == 27) GS_SHF_TC(9); else GS_SHF_TC(16);
#undef GS_SHF_TC
  return cudaGetLastError();
}

cudaError_t gs_launch_blend_sh_bwd_tc(const GsRec* grec, const float* rgb, const uint32_t* ids, const uint32_t* goff, int d,
                                      const int* tile_accum, const GsFrameGeom& g, const GsRayPtrs& r, const float* image,
                                      const float* grad_image, float* grad_inst, int grad_is_final, const GsCrop& crop,
                                      uint32_t* row_epoch, uint32_t epoch, int* tile_neff_b, cudaStream_t st) {
  if (!row_epoch) return cudaErrorInvalidValue;   // unprocessed rows are left stale: the consumer needs the epoch tags
#define GS_SHB_TC(K)                                                                                                  \
  do {                                                                                                                \
    /* per device and cheap: set on every launch rather than cached in a process-wide flag */                        \
    cudaError_t e = cudaFuncSetAttribute(blend_sh_bwd_tc_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                         (int)sizeof(TcBwdSmem<K>));                                                  \
    if (e != cudaSuccess) return e;                                                                                   \
    blend_sh_bwd_tc_kernel<K><<<g.n_tiles, TC_NT, sizeof(TcBwdSmem<K>), st>>>(                                          \
        grec, rgb, ids, goff, tile_accum, g.wp, g.hp, g.ntx, g.fx, g.fy, r.rays_o, r.lefttop, r.dx, r.dy, image,       \
        grad_image, grad_inst, grad_is_final, crop, row_epoch, epoch, tile_neff_b);                                   \
  } while (0)
  if (d == 27) GS_SHB_TC(9); else GS_SHB_TC(16);
#undef GS_SHB_TC
  return cudaGetLastError();
}
