// Per-tile front-to-back alpha compositing, forward and backward (the hot kernels).
//
// Semantics: reference gaussian.cu:806-970 (draw_kernel) and :440-803 (draw_backward_kernel):
// 16x16 pixel tiles, each tile blends its (depth-sorted) instance range front to back,
// a pixel stops before an instance once its transmittance is < 1e-4, no alpha clamp, no
// 1/255 skip, black background (the MAPS instantiations of the gather path - an extension - also write depth and
// alpha maps and composite over a background colour; DESIGN.md §9).  Design (not the reference's):
//   * each tile's range is contiguous in three packed record streams (see gs_common.cuh) and is
//     staged into shared memory by 1-D bulk async copies (cp.async.bulk -> UBLKCP, mbarrier
//     complete_tx), double buffered; one elected thread issues, nobody spends LSU slots on it;
//   * per (pixel, instance): one ex2 (opacity folded into the exponent) and ~15 FP32 ops;
//     no FP64, no division in the forward loop;
//   * whole-warp and whole-CTA early exit once every pixel is saturated, so a tile's tail is
//     never read (M_eff accounting);
//   * backward: one warp x 8 pixels per thread per tile; six partial sums per (thread, instance) go to shared
//     memory and a second phase of 4 threads per instance reduces them and writes ONE record per instance
//     (no atomics, deterministic).
#include <cstdlib>
#include <type_traits>

#include "internal.h"

namespace {

// =======================================================================================
// forward
// =======================================================================================
constexpr int FWD_CH = 128;                  // instances per staging chunk
constexpr int FWD_PX = 4;                    // each thread owns a row of 4 adjacent pixels
constexpr int FWD_THREADS = 256 / FWD_PX;    // 2 warps per tile
constexpr int FWD_STAGES = 2;

template <typename SM>
__device__ __forceinline__ void issue_chunk(SM& sm, int stage, const float4* __restrict__ pA,
                                            const float2* __restrict__ pB, const float4* __restrict__ pC,
                                            int base, int n, int shift) {
  uint32_t bytes_a = (uint32_t)n * 16u;
  uint32_t nb = (uint32_t)(n + shift + 1) & ~1u;
  uint32_t bytes_b = nb * 8u;
  gs_mbar_expect_tx(&sm.full[stage], 2u * bytes_a + bytes_b);
  gs_bulk_g2s(sm.A[stage], pA + base, bytes_a, &sm.full[stage]);
  gs_bulk_g2s(sm.C[stage], pC + base, bytes_a, &sm.full[stage]);
  gs_bulk_g2s(sm.B[stage], pB + (base - shift), bytes_b, &sm.full[stage]);
}

// ---- two ways a tile's sorted range reaches shared memory -------------------------------------------
// packed : three contiguous record streams written by the pack pass (and by the legacy draw API);
//          one thread issues three 1-D bulk copies per chunk.
// gather : NO pack pass - every thread of the CTA issues, for "its" instances of the next chunk, the 16-byte
//          cp.async pieces of the Gaussian's record straight from GsRec rec[N] through the sorted id list and
//          arrives on the stage's mbarrier when they have landed (cp.async.mbarrier.arrive; barrier count = CTA
//          threads).  The per-instance record in shared memory is {a, b, c, d} (gs_common.cuh GsRec).
template <int CH, int STAGES>
struct PackedRing {
  float4 A[STAGES][CH];
  float4 C[STAGES][CH];
  float2 B[STAGES][CH + 2];
  uint64_t full[STAGES];
};

template <bool GATHER>
struct StageView;
template <>
struct StageView<false> {
  const float4* A;
  const float4* C;
  const float2* B;
  __device__ __forceinline__ float4 a(int j) const { return A[j]; }
  __device__ __forceinline__ float2 b(int j) const { return B[j]; }
  __device__ __forceinline__ float4 c(int j) const { return C[j]; }                   // r, g, b, (slot)
  __device__ __forceinline__ uint32_t slot(int j, int, int) const { return __float_as_uint(C[j].w); }
  __device__ __forceinline__ float depth(int) const { return 0.f; }                    // not staged (maps: gather only)
};
template <>
struct StageView<true> {
  const float4* R;                                                                     // [CH][RECW]
  int recw;
  __device__ __forceinline__ float4 a(int j) const { return R[j * recw]; }
  __device__ __forceinline__ float2 b(int j) const {
    const float4 t = R[j * recw + 1];
    return make_float2(t.x, t.y);
  }
  __device__ __forceinline__ float4 c(int j) const {
    const float4 t = R[j * recw + 1];
    return make_float4(t.z, t.w, R[j * recw + 2].x, 0.f);
  }
  __device__ __forceinline__ float depth(int j) const { return R[j * recw + 2].y; }   // |p_c| (maps frames)
  // gradient row of this (Gaussian, tile) instance: first row of the Gaussian + rank of the tile in its rectangle
  __device__ __forceinline__ uint32_t slot(int j, int tx, int ty) const {
    const float4 cc = R[j * recw + 2];
    const uint32_t rxy = __float_as_uint(cc.z), rwh = __float_as_uint(cc.w);
    const uint32_t off = __float_as_uint(R[j * recw + 3].x);
    return off + ((uint32_t)ty - (rxy >> 16)) * (rwh & 0xffffu) + ((uint32_t)tx - (rxy & 0xffffu));
  }
};

template <int CH, int STAGES, int RECW>
struct GatherRing {
  float4 rec[STAGES][CH * RECW];
  uint64_t full[STAGES];
};

// ids of "this thread's" instances of one chunk, loaded one chunk boundary ahead of their use so that the
// dependent record copies never wait for the id load
template <int NT, int CH>
struct GatherIds {
  uint32_t id[(CH + NT - 1) / NT];
  __device__ __forceinline__ void load(const uint32_t* __restrict__ ids, int base, int n, int tid) {
#pragma unroll
    for (int u = 0; u < (CH + NT - 1) / NT; ++u) {
      const int i = tid + u * NT;
      id[u] = i < n ? __ldg(ids + base + i) : 0u;
    }
  }
};

// RECW = 3: {a, b, c} (forward); RECW = 4: {a, b, c, (first gradient row of the Gaussian, -, -, -)} (backward: the
// 4th piece comes from offsets_g[id], a 4-byte cp.async - patching it into rec[] from another kernel cost more)
template <typename SM, int NT, int CH, int RECW>
__device__ __forceinline__ void gather_issue(SM& sm, int stage, const GsRec* __restrict__ grec,
                                             const uint32_t* __restrict__ goff, const GatherIds<NT, CH>& g, int n,
                                             int tid) {
  // 16-byte cp.async (LDGSTS) pieces: one warp-wide instruction moves a piece of 32 instances.  (Measured: one
  // 1-D bulk copy per instance, i.e. ~6 M tiny TMA requests per frame, made both blend kernels ~15 % slower.)
#pragma unroll
  for (int u = 0; u < (CH + NT - 1) / NT; ++u) {
    const int i = tid + u * NT;
    if (i < n) {
      const float4* src = reinterpret_cast<const float4*>(grec + g.id[u]);
      const uint32_t dst = gs_smem_u32(&sm.rec[stage][i * RECW]);
#pragma unroll
      for (int q = 0; q < 3; ++q)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * q), "l"(src + q) : "memory");
      if (RECW == 4)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 48u), "l"(goff + g.id[u]) : "memory");
    }
  }
  // this thread's arrival on the stage barrier (count = CTA threads) fires when its copies have landed
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(gs_smem_u32(&sm.full[stage])) : "memory");
}

// Per (thread, instance): 3 broadcast LDS + 4 row-shared FP32 ops (dy, cb*dy, cc*dy, l2o-cc*dy^2)
// + 4 pixels x (dx, u, exponent, MUFU.EX2, setp, mul, sel, 3 FFMA colour, T update) = 12.75
// issue slots per (pixel, instance) instead of 17-18 with one pixel per thread.
// MAPS (gather path only): one more FFMA per (pixel, instance) accumulates the depth map; the epilogue adds T * bg to
// the colour and stores depth and alpha = 1 - T.
template <bool GATHER, bool MAPS>
__global__ void __launch_bounds__(FWD_THREADS) blend_fwd_kernel(const float4* __restrict__ pA,
                                                                 const float2* __restrict__ pB,
                                                                 const float4* __restrict__ pC,
                                                                 const GsRec* __restrict__ grec,
                                                                 const uint32_t* __restrict__ ids,
                                                                 const int* __restrict__ tile_accum, int wp, int hp,
                                                                 int ntx, float fx, float fy,
                                                                 float* __restrict__ image,
                                                                 int* __restrict__ tile_neff,
                                                                 float* __restrict__ final_img, GsCrop crop,
                                                                 GsMapsFwd maps) {
  static_assert(!MAPS || GATHER, "depth / alpha maps read the depth from the gathered records");
  using Smem =
      typename std::conditional<GATHER, GatherRing<FWD_CH, FWD_STAGES, 3>, PackedRing<FWD_CH, FWD_STAGES>>::type;
  __shared__ __align__(16) Smem sm;
  const int tile = blockIdx.x;
  const int tid = threadIdx.x;
  const int tx = tile % ntx, ty = tile / ntx;
  // thread -> a row of FWD_PX adjacent pixels (ix0 .. ix0+FWD_PX-1, iy)
  constexpr int TPR = GS_TILE / FWD_PX;
  const int ix0 = tx * GS_TILE + (tid % TPR) * FWD_PX;
  const int iy = ty * GS_TILE + (tid / TPR);
  float px[FWD_PX];
#pragma unroll
  for (int p = 0; p < FWD_PX; ++p) px[p] = gs_pixel_coord(ix0 + p, wp, fx);
  const float py = gs_pixel_coord(iy, hp, fy);

  const int start = tile_accum[tile];
  const int cnt = tile_accum[tile + 1] - start;
  const int shift = start & 1;
  const int nchunks = (cnt + FWD_CH - 1) / FWD_CH;

  if (tid == 0) {
    for (int s = 0; s < FWD_STAGES; ++s) gs_mbar_init(&sm.full[s], GATHER ? FWD_THREADS : 1);
    gs_fence_barrier_init();
  }
  __syncthreads();
  GatherIds<FWD_THREADS, FWD_CH> gid;
  if constexpr (GATHER) {
    for (int k = 0; k < FWD_STAGES && k < nchunks; ++k) {
      gid.load(ids, start + k * FWD_CH, min(FWD_CH, cnt - k * FWD_CH), tid);
      gather_issue<Smem, FWD_THREADS, FWD_CH, 3>(sm, k, grec, nullptr, gid, min(FWD_CH, cnt - k * FWD_CH), tid);
    }
    if (FWD_STAGES < nchunks) gid.load(ids, start + FWD_STAGES * FWD_CH, min(FWD_CH, cnt - FWD_STAGES * FWD_CH), tid);
  } else if (tid == 0) {
    for (int k = 0; k < FWD_STAGES && k < nchunks; ++k)
      issue_chunk<Smem>(sm, k, pA, pB, pC, start + k * FWD_CH, min(FWD_CH, cnt - k * FWD_CH), shift);
  }

  float T[FWD_PX], cr[FWD_PX], cg[FWD_PX], cb[FWD_PX];
  float dd[FWD_PX];                                   // depth map (MAPS only)
#pragma unroll
  for (int p = 0; p < FWD_PX; ++p) {
    T[p] = 1.f;
    cr[p] = cg[p] = cb[p] = 0.f;
    dd[p] = 0.f;
  }
  int consumed = cnt;
  int k = 0;
  for (; k < nchunks; ++k) {
    const int stage = k % FWD_STAGES;
    gs_mbar_wait(&sm.full[stage], (uint32_t)((k / FWD_STAGES) & 1));
    const int n = min(FWD_CH, cnt - k * FWD_CH);
    StageView<GATHER> sv;
    if constexpr (GATHER) {
      sv.R = sm.rec[stage];
      sv.recw = 3;
    } else {
      sv.A = sm.A[stage];
      sv.C = sm.C[stage];
      sv.B = sm.B[stage] + shift;
    }

#define GS_FWD_BODY(J)                                                                      \
  {                                                                                         \
    const float4 a = sv.a(J);                                                               \
    const float2 b = sv.b(J);                                                               \
    const float4 c = sv.c(J);                                                               \
    float dep = 0.f;                                                                        \
    if constexpr (MAPS) dep = sv.depth(J);                                                  \
    const float dy = py - a.y;                                                              \
    const float m1 = a.w * dy;                                                              \
    const float ev = fmaf(-b.x * dy, dy, b.y);                                              \
    _Pragma("unroll") for (int p = 0; p < FWD_PX; ++p) {                                    \
      const float dx = px[p] - a.x;                                                         \
      const float eu = fmaf(a.z, dx, -m1);                                                  \
      const float alpha = gs_ex2(fmaf(-dx, eu, ev)); /* l2o - (ca dx^2 - cb dx dy + cc dy^2) */ \
      const float w = (T[p] > GS_T_STOP) ? alpha * T[p] : 0.f;                              \
      cr[p] = fmaf(c.x, w, cr[p]);                                                          \
      cg[p] = fmaf(c.y, w, cg[p]);                                                          \
      cb[p] = fmaf(c.z, w, cb[p]);                                                          \
      if constexpr (MAPS) dd[p] = fmaf(dep, w, dd[p]);                                      \
      T[p] -= w;                                                                            \
    }                                                                                       \
  }
    int j = 0;
    bool warp_dead = false;
    for (; j + 4 <= n; j += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) GS_FWD_BODY(j + u)
      bool dead = true;
#pragma unroll
      for (int p = 0; p < FWD_PX; ++p) dead = dead && !(T[p] > GS_T_STOP);
      if (__all_sync(0xffffffffu, dead)) {
        warp_dead = true;
        break;
      }
    }
    if (!warp_dead)
      for (; j < n; ++j) GS_FWD_BODY(j)
#undef GS_FWD_BODY

    bool dead = true;
#pragma unroll
    for (int p = 0; p < FWD_PX; ++p) dead = dead && !(T[p] > GS_T_STOP);
    const int all_dead = __syncthreads_and(dead);
    if (all_dead) {
      consumed = min(cnt, (k + 1) * FWD_CH);
      break;
    }
    if (k + FWD_STAGES < nchunks) {
      const int kn = k + FWD_STAGES;            // every thread is past the barrier above: the stage is free
      if constexpr (GATHER) {
        gather_issue<Smem, FWD_THREADS, FWD_CH, 3>(sm, stage, grec, nullptr, gid, min(FWD_CH, cnt - kn * FWD_CH), tid);
        if (kn + 1 < nchunks) gid.load(ids, start + (kn + 1) * FWD_CH, min(FWD_CH, cnt - (kn + 1) * FWD_CH), tid);
      } else if (tid == 0)
        issue_chunk<Smem>(sm, stage, pA, pB, pC, start + kn * FWD_CH, min(FWD_CH, cnt - kn * FWD_CH), shift);
    }
  }
  // drain copies that were issued but never consumed (early exit) before the CTA retires
  if (tid == 0 && k < nchunks) {
    for (int kk = k + 1; kk < nchunks && kk < k + FWD_STAGES; ++kk)
      gs_mbar_wait(&sm.full[kk % FWD_STAGES], (uint32_t)((kk / FWD_STAGES) & 1));
  }
  if constexpr (MAPS) {
    // background behind the remaining transmittance; depth and alpha planes (FWD_PX floats = 16-byte aligned rows)
    float av[FWD_PX];
#pragma unroll
    for (int p = 0; p < FWD_PX; ++p) {
      cr[p] = fmaf(T[p], maps.bg_r, cr[p]);
      cg[p] = fmaf(T[p], maps.bg_g, cg[p]);
      cb[p] = fmaf(T[p], maps.bg_b, cb[p]);
      av[p] = 1.f - T[p];
    }
    float4* od = reinterpret_cast<float4*>(maps.depth + (size_t)iy * wp + ix0);
    float4* oa = reinterpret_cast<float4*>(maps.alpha + (size_t)iy * wp + ix0);
#pragma unroll
    for (int q = 0; q < FWD_PX / 4; ++q) {
      od[q] = make_float4(dd[4 * q], dd[4 * q + 1], dd[4 * q + 2], dd[4 * q + 3]);
      oa[q] = make_float4(av[4 * q], av[4 * q + 1], av[4 * q + 2], av[4 * q + 3]);
    }
    if (maps.depth_final) {
#pragma unroll
      for (int p = 0; p < FWD_PX; ++p) {
        const int x = ix0 + p - crop.left, y = iy - crop.top;
        if (x >= 0 && x < crop.width && y >= 0 && y < crop.height) {
          maps.depth_final[(size_t)y * crop.width + x] = dd[p];
          maps.alpha_final[(size_t)y * crop.width + x] = av[p];
        }
      }
    }
  }
  // FWD_PX pixels x 3 channels = FWD_PX * 12 contiguous, 16-byte aligned bytes
  {
    float ob[FWD_PX * 3];
#pragma unroll
    for (int p = 0; p < FWD_PX; ++p) {
      ob[3 * p] = cr[p];
      ob[3 * p + 1] = cg[p];
      ob[3 * p + 2] = cb[p];
    }
    float4* o = reinterpret_cast<float4*>(image + ((size_t)iy * wp + ix0) * 3);
#pragma unroll
    for (int q = 0; q < FWD_PX * 3 / 4; ++q) o[q] = make_float4(ob[4 * q], ob[4 * q + 1], ob[4 * q + 2], ob[4 * q + 3]);
  }
  if (final_img) {
#pragma unroll
    for (int p = 0; p < FWD_PX; ++p)
      gs_store_final(final_img, ix0 + p, iy, crop.left, crop.top, crop.width, crop.height, cr[p], cg[p], cb[p]);
  }
  if (tile_neff && tid == 0) tile_neff[tile] = consumed;
}

// =======================================================================================
// backward
// =======================================================================================
// Cross-thread reduction WITHOUT shuffles: every thread accumulates, over its own row of
// PX pixels, six partial sums per instance (S0, Sx, Sxx, Cr, Cg, Cb; dy is shared by the row) and
// stores them to shared memory ([instance][quarter][thread][6], strides chosen so that both the
// 8-byte stores and the 8-byte loads of the second phase are bank-conflict free).  After R = NT/4
// instances a second phase gives each instance to 4 threads: each sums one quarter of the source
// threads (4 pixel rows: Sy = sum dy S0, Sxy = sum dy Sx, Syy = sum dy^2 S0 are formed per row), two
// xor-shuffles combine the quarters, and each of the 4 lanes stores one 16-byte piece of the
// instance's gradient record.  ~13 instructions per (thread, instance) instead of ~42 for a
// recursive-halving shuffle network; fixed summation order => bit-deterministic.
constexpr int BWD_PX = 8;                    // each thread owns a row of 8 adjacent pixels
constexpr int BWD_THREADS = 256 / BWD_PX;    // one warp per tile

// Per-path constants.  gather: the best configuration of the round-2 sweeps (profiles/r2_sweeps.md), 32-instance
// chunks 3 deep, 4 instances per unrolled step.  packed (legacy draw API, gs_tune("gather", 0)): 64-instance chunks
// 2 deep, unroll 2.
template <bool GATHER, bool MAPS>
struct BwdCfg {
  static constexpr int PX = BWD_PX, NT = BWD_THREADS;
  static constexpr int TPR = GS_TILE / PX;                   // threads per pixel row
  static constexpr int RQ = 4;                               // reducer threads per instance in the second phase
  static constexpr int R = NT / RQ;                          // instances per reduction round
  static constexpr int SQ = NT / RQ;                         // source threads per reducer ("part")
  static constexpr int ROWS = SQ / TPR;                      // pixel rows per reducer
  // floats per (source thread, instance): 6, or 8 for a maps frame - the 7th sum (and a pad) then sits in a
  // [part][source thread][2] block behind the [part][source thread][6] one, so both store streams keep their stride
  static constexpr int PW = MAPS ? 8 : 6;
  // strides (floats) of the partial buffer [instance][part][source thread][6 (+2)]: part stride = 32/RQ and
  // instance stride = 2 (mod 32) make the 8-byte loads of a half-warp (16 / RQ instances x RQ parts) hit
  // 16 distinct bank pairs; the 8-byte stores of 16 consecutive source threads (stride 6, resp. 2) are conflict free
  static constexpr int QS = (SQ * PW + 31) / 32 * 32 + 32 / RQ;
  static constexpr int IS = RQ * QS + 2 - (RQ * QS) % 32 + ((RQ * QS) % 32 > 2 ? 32 : 0);
  static constexpr int CH = GATHER ? 32 : 64;                // instances per staging chunk
  static constexpr int STAGES = GATHER ? 3 : 2;              // staging ring depth
  static constexpr int UNR = GATHER ? 4 : 2;                 // instances per unrolled step of the first phase
  static constexpr int MINB = GATHER ? 10 : 16;              // __launch_bounds__ min blocks (register cap)
};

template <bool GATHER, bool MAPS>
struct BwdSmem : std::conditional<GATHER, GatherRing<BwdCfg<GATHER, MAPS>::CH, BwdCfg<GATHER, MAPS>::STAGES, 4>,
                                  PackedRing<BwdCfg<GATHER, MAPS>::CH, BwdCfg<GATHER, MAPS>::STAGES>>::type {
  float part[BwdCfg<GATHER, MAPS>::R * BwdCfg<GATHER, MAPS>::IS];
  float pyt[GS_TILE];
};

// Upstream gradients of the depth and alpha maps for a thread's row of PX pixels (MAPS only)
template <int PX>
struct MapsGrad {
  float gd[PX], ga[PX];
};

// one instance x this thread's row of PX pixels: recompute alpha, analytic d/d alpha, six partial sums.
// MAPS: depth and alpha act as two more channels with per-instance "colours" d_i and 1 (gc += gD d_i + gA), and a
// 7th sum gD w (the gradient of the instance's depth) goes to dst_d.
template <int PX, bool MAPS = false>
__device__ __forceinline__ void bwd_row(const float4 a, const float2 b, const float4 c, const float (&px)[PX],
                                        const float py, float (&T)[PX], float (&Rr)[PX], const float (&gr)[PX],
                                        const float (&gg)[PX], const float (&gb)[PX], float2* __restrict__ dst,
                                        const float dep = 0.f, const MapsGrad<PX>* mg = nullptr,
                                        float2* __restrict__ dst_d = nullptr) {
  float s0 = 0.f, sx = 0.f, sxx = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f, cd = 0.f;
  const float dy = py - a.y;
  const float m1 = a.w * dy;
  const float ev = fmaf(-b.x * dy, dy, b.y);
#pragma unroll
  for (int p = 0; p < PX; ++p) {
    const float dx = px[p] - a.x;
    const float eu = fmaf(a.z, dx, -m1);
    float alpha = gs_ex2(fmaf(-dx, eu, ev));                     // l2o - (ca dx^2 - cb dx dy + cc dy^2)
    alpha = (T[p] > GS_T_STOP) ? alpha : 0.f;                    // early stop (:578): no weight, no gradient
    const float w = alpha * T[p];
    float gc = fmaf(gr[p], c.x, fmaf(gg[p], c.y, gb[p] * c.z));
    if constexpr (MAPS) {
      gc = fmaf(mg->gd[p], dep, gc + mg->ga[p]);
      cd = fmaf(mg->gd[p], w, cd);
    }
    Rr[p] = fmaf(-gc, w, Rr[p]);                                 // sum_c g_c (out_c - C_c^{<=i})
    const float rc = gs_rcp(1.0000001f - alpha);                 // 1/(1 - alpha + 1e-7)  (:721)
    const float dal = fmaf(T[p], gc, -Rr[p] * rc);               // d L / d alpha            (:710-722)
    const float e = dal * alpha;
    T[p] -= w;
    const float ex = e * dx;
    s0 += e;
    sx += ex;
    sxx = fmaf(ex, dx, sxx);
    c0 = fmaf(gr[p], w, c0);
    c1 = fmaf(gg[p], w, c1);
    c2 = fmaf(gb[p], w, c2);
  }
  dst[0] = make_float2(s0, sx);
  dst[1] = make_float2(sxx, c0);
  dst[2] = make_float2(c1, c2);
  if constexpr (MAPS) dst_d[0] = make_float2(cd, 0.f);
}

// Thread 0 (packed) or every thread (gather) issues the copies of the next chunk at the chunk boundaries.
// MAPS (gather path only): gradients of the depth / alpha maps too; d/d depth_i goes to float 9 of the gradient row.
template <bool GATHER, bool MAPS>
__global__ void __launch_bounds__(BWD_THREADS, BwdCfg<GATHER, MAPS>::MINB)
    blend_bwd_kernel(const float4* __restrict__ pA, const float2* __restrict__ pB, const float4* __restrict__ pC,
                     const GsRec* __restrict__ grec, const uint32_t* __restrict__ ids,
                     const uint32_t* __restrict__ goff, const int* __restrict__ tile_accum, int wp, int hp, int ntx, float fx, float fy,
                     const float* __restrict__ image, const float* __restrict__ grad_image,
                     float* __restrict__ grad_inst, int grad_is_final, GsCrop crop, uint32_t* __restrict__ row_epoch,
                     uint32_t epoch, int* __restrict__ tile_neff_b, GsMapsBwd maps) {
  using Cfg = BwdCfg<GATHER, MAPS>;
  constexpr int PX = Cfg::PX, NT = Cfg::NT, TPR = Cfg::TPR, RQ = Cfg::RQ, R = Cfg::R, SQ = Cfg::SQ, QS = Cfg::QS,
                IS = Cfg::IS, ROWS = Cfg::ROWS, CH = Cfg::CH, STAGES = Cfg::STAGES, UNR = Cfg::UNR;
  static_assert(IS % 2 == 0 && QS % 2 == 0 && IS % 32 == 2 && QS % 32 == 32 / RQ, "partial buffer strides");
  static_assert(NT == 32, "one warp per tile: warp votes and __syncwarp order the phases");
  static_assert(!MAPS || GATHER, "depth / alpha maps read the depth from the gathered records");
  static_assert(PX % 4 == 0, "float4 rows of the image / map planes");
  using Smem = BwdSmem<GATHER, MAPS>;
  __shared__ __align__(16) Smem sm;
  const int tile = blockIdx.x;
  const int tid = threadIdx.x;
  const int start = tile_accum[tile];
  const int cnt = tile_accum[tile + 1] - start;
  if (cnt == 0) return;
  const int nchunks = (cnt + CH - 1) / CH;
  const int tx = tile % ntx, ty = tile / ntx;
  const int shift = start & 1;
  if (tid < GS_TILE) sm.pyt[tid] = gs_pixel_coord(ty * GS_TILE + tid, hp, fy);
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) gs_mbar_init(&sm.full[s], GATHER ? NT : 1);
    gs_fence_barrier_init();
  }
  __syncthreads();
  GatherIds<NT, CH> gid;
  if constexpr (GATHER) {
    for (int k = 0; k < STAGES && k < nchunks; ++k) {
      gid.load(ids, start + k * CH, min(CH, cnt - k * CH), tid);
      gather_issue<Smem, NT, CH, 4>(sm, k, grec, goff, gid, min(CH, cnt - k * CH), tid);
    }
    if (STAGES < nchunks) gid.load(ids, start + STAGES * CH, min(CH, cnt - STAGES * CH), tid);
  } else if (tid == 0) {
    for (int k = 0; k < STAGES && k < nchunks; ++k)
      issue_chunk<Smem>(sm, k, pA, pB, pC, start + k * CH, min(CH, cnt - k * CH), shift);
  }
  const int ix0 = tx * GS_TILE + (tid % TPR) * PX;
  const int iy = ty * GS_TILE + (tid / TPR);
  float px[PX];
#pragma unroll
  for (int p = 0; p < PX; ++p) px[p] = gs_pixel_coord(ix0 + p, wp, fx);
  const float py = sm.pyt[tid / TPR];

  float T[PX], Rr[PX], gr[PX], gg[PX], gb[PX];
  {
    const size_t off = ((size_t)iy * wp + ix0) * 3;     // PX*12 contiguous, 16-byte aligned bytes
    const float4* im = reinterpret_cast<const float4*>(image + off);
    float gbuf[PX * 3], ibuf[PX * 3];
#pragma unroll
    for (int q = 0; q < PX * 3 / 4; ++q) {
      const float4 i4 = im[q];
      ibuf[4 * q] = i4.x; ibuf[4 * q + 1] = i4.y; ibuf[4 * q + 2] = i4.z; ibuf[4 * q + 3] = i4.w;
    }
    if (!grad_is_final) {
      const float4* gi = reinterpret_cast<const float4*>(grad_image + off);
#pragma unroll
      for (int q = 0; q < PX * 3 / 4; ++q) {
        const float4 g4 = gi[q];
        gbuf[4 * q] = g4.x; gbuf[4 * q + 1] = g4.y; gbuf[4 * q + 2] = g4.z; gbuf[4 * q + 3] = g4.w;
      }
    } else {
#pragma unroll
      for (int p = 0; p < PX; ++p)
        gs_load_final_grad(grad_image, ibuf + 3 * p, ix0 + p, iy, crop.left, crop.top, crop.width, crop.height,
                           gbuf[3 * p], gbuf[3 * p + 1], gbuf[3 * p + 2]);
    }
#pragma unroll
    for (int p = 0; p < PX; ++p) {
      gr[p] = gbuf[3 * p];
      gg[p] = gbuf[3 * p + 1];
      gb[p] = gbuf[3 * p + 2];
      Rr[p] = gr[p] * ibuf[3 * p] + gg[p] * ibuf[3 * p + 1] + gb[p] * ibuf[3 * p + 2];
      T[p] = 1.f;
    }
  }
  MapsGrad<PX> mg;
  if constexpr (MAPS) {
    // the suffix sum starts at g . image + gD depth + gA alpha (the raw maps of the forward)
    const size_t po = (size_t)iy * wp + ix0;          // PX floats = 16-byte aligned rows of the [Hp,Wp] planes
    float dv[PX], av[PX];
#pragma unroll
    for (int q = 0; q < PX / 4; ++q) {
      const float4 d4 = reinterpret_cast<const float4*>(maps.depth + po)[q];
      const float4 a4 = reinterpret_cast<const float4*>(maps.alpha + po)[q];
      dv[4 * q] = d4.x; dv[4 * q + 1] = d4.y; dv[4 * q + 2] = d4.z; dv[4 * q + 3] = d4.w;
      av[4 * q] = a4.x; av[4 * q + 1] = a4.y; av[4 * q + 2] = a4.z; av[4 * q + 3] = a4.w;
    }
    if (!grad_is_final) {
#pragma unroll
      for (int q = 0; q < PX / 4; ++q) {
        const float4 d4 = reinterpret_cast<const float4*>(maps.grad_depth + po)[q];
        const float4 a4 = reinterpret_cast<const float4*>(maps.grad_alpha + po)[q];
        mg.gd[4 * q] = d4.x; mg.gd[4 * q + 1] = d4.y; mg.gd[4 * q + 2] = d4.z; mg.gd[4 * q + 3] = d4.w;
        mg.ga[4 * q] = a4.x; mg.ga[4 * q + 1] = a4.y; mg.ga[4 * q + 2] = a4.z; mg.ga[4 * q + 3] = a4.w;
      }
    } else {
      // cropped [H,W] gradients: no clamp on the maps, nothing outside the crop
#pragma unroll
      for (int p = 0; p < PX; ++p) {
        const int x = ix0 + p - crop.left, y = iy - crop.top;
        const bool in = x >= 0 && x < crop.width && y >= 0 && y < crop.height;
        mg.gd[p] = in ? maps.grad_depth[(size_t)y * crop.width + x] : 0.f;
        mg.ga[p] = in ? maps.grad_alpha[(size_t)y * crop.width + x] : 0.f;
      }
    }
#pragma unroll
    for (int p = 0; p < PX; ++p) Rr[p] = fmaf(mg.gd[p], dv[p], fmaf(mg.ga[p], av[p], Rr[p]));
  }
  // this thread's slot in the partial buffer: quarter tid / SQ, position tid % SQ
  float2* const my_part = reinterpret_cast<float2*>(sm.part + (tid / SQ) * QS + (tid % SQ) * 6);
  float2* const my_part_d = reinterpret_cast<float2*>(sm.part + (tid / SQ) * QS + SQ * 6 + (tid % SQ) * 2);
  // second-phase role: instance ri of the round, quarter rq of the source threads
  const int ri = tid / RQ, rq = tid % RQ;
  const float2* const red_src = reinterpret_cast<const float2*>(sm.part + ri * IS + rq * QS);
  const float2* const red_src_d = reinterpret_cast<const float2*>(sm.part + ri * IS + rq * QS + SQ * 6);

  int consumed = cnt;
  bool finished = false;
  int k = 0;
  for (; k < nchunks && !finished; ++k) {
    const int stage = k % STAGES;
    gs_mbar_wait(&sm.full[stage], (uint32_t)((k / STAGES) & 1));
    const int n = min(CH, cnt - k * CH);
    StageView<GATHER> sv;
    if constexpr (GATHER) {
      sv.R = sm.rec[stage];
      sv.recw = 4;
    } else {
      sv.A = sm.A[stage];
      sv.C = sm.C[stage];
      sv.B = sm.B[stage] + shift;
    }

    for (int sub = 0; sub < n; sub += R) {
      const int nr = min(R, n - sub);
      // ---- phase 1: per-thread partial sums of up to R instances
      int j = 0;
      bool wdead = false;
      for (; j + UNR <= nr; j += UNR) {
        if (UNR >= 4 || (j & 3) == 0) {
          bool dead = true;
#pragma unroll
          for (int p = 0; p < PX; ++p) dead = dead && !(T[p] > GS_T_STOP);
          if (__all_sync(0xffffffffu, dead)) {
            wdead = true;
            break;
          }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u)
          bwd_row<PX, MAPS>(sv.a(sub + j + u), sv.b(sub + j + u), sv.c(sub + j + u), px, py, T, Rr, gr, gg, gb,
                            my_part + (j + u) * (IS / 2), MAPS ? sv.depth(sub + j + u) : 0.f, &mg,
                            my_part_d + (j + u) * (IS / 2));
      }
      if (!wdead)
        for (; j < nr; ++j)
          bwd_row<PX, MAPS>(sv.a(sub + j), sv.b(sub + j), sv.c(sub + j), px, py, T, Rr, gr, gg, gb,
                            my_part + j * (IS / 2), MAPS ? sv.depth(sub + j) : 0.f, &mg, my_part_d + j * (IS / 2));
      bool dead = true;
#pragma unroll
      for (int p = 0; p < PX; ++p) dead = dead && !(T[p] > GS_T_STOP);
      __syncwarp();
      const int all_dead = __all_sync(0xffffffffu, dead);
      // ---- phase 2: 4 threads per instance, one quarter of the source threads (4 pixel rows) each
      {
        float S0 = 0.f, Sx = 0.f, Sxx = 0.f, Sy = 0.f, Sxy = 0.f, Syy = 0.f, C0 = 0.f, C1 = 0.f, C2 = 0.f, Cd = 0.f;
        const bool act = ri < nr;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        float2 b = make_float2(0.f, 0.f);
        if (act) {
          a = sv.a(sub + ri);
          b = sv.b(sub + ri);
        }
        if (act && ri < j) {                       // j: instances the warp really processed (warp-uniform)
#pragma unroll
          for (int r = 0; r < ROWS; ++r) {
            float2 u0 = red_src[(r * TPR) * 3], u1 = red_src[(r * TPR) * 3 + 1], u2 = red_src[(r * TPR) * 3 + 2];
#pragma unroll
            for (int t = 1; t < TPR; ++t) {
              const float2 w0 = red_src[(r * TPR + t) * 3], w1 = red_src[(r * TPR + t) * 3 + 1],
                           w2 = red_src[(r * TPR + t) * 3 + 2];
              u0.x += w0.x; u0.y += w0.y; u1.x += w1.x; u1.y += w1.y; u2.x += w2.x; u2.y += w2.y;
            }
            const float dyr = sm.pyt[ROWS * rq + r] - a.y;
            S0 += u0.x;
            Sx += u0.y;
            Sxx += u1.x;
            C0 += u1.y;
            C1 += u2.x;
            C2 += u2.y;
            Sy = fmaf(dyr, u0.x, Sy);
            Sxy = fmaf(dyr, u0.y, Sxy);
            Syy = fmaf(dyr * dyr, u0.x, Syy);
            if constexpr (MAPS) {
              float ud = red_src_d[r * TPR].x;
#pragma unroll
              for (int t = 1; t < TPR; ++t) ud += red_src_d[r * TPR + t].x;
              Cd += ud;
            }
          }
        }
#define GS_RED4(V)                                   \
  V += __shfl_xor_sync(0xffffffffu, V, 1);           \
  V += __shfl_xor_sync(0xffffffffu, V, 2);
        GS_RED4(S0) GS_RED4(Sx) GS_RED4(Sxx) GS_RED4(Sy) GS_RED4(Sxy) GS_RED4(Syy) GS_RED4(C0) GS_RED4(C1) GS_RED4(C2)
        if constexpr (MAPS) { GS_RED4(Cd) }
#undef GS_RED4
        if (act) {
          const uint32_t slot = sv.slot(sub + ri, tx, ty);
          float4* out = reinterpret_cast<float4*>(grad_inst + (size_t)slot * GS_GREC);
          // d/dx, d/dy, d/dca, d/dcb  |  d/dcc, d/dl2o, d/dr, d/dg  |  d/db (, d/ddepth: maps frames)
          if (rq == 0)
            out[0] = make_float4(GS_LN2 * (2.f * a.z * Sx - a.w * Sy), GS_LN2 * (2.f * b.x * Sy - a.w * Sx),
                                 -GS_LN2 * Sxx, GS_LN2 * Sxy);
          else if (rq == 1)
            out[1] = make_float4(-GS_LN2 * Syy, GS_LN2 * S0, C0, C1);
          else if (rq == 2)
            out[2] = make_float4(C2, MAPS ? Cd : 0.f, 0.f, 0.f);
          else if (rq == 3 && row_epoch)
            row_epoch[slot] = epoch;               // marks the row as written in this frame
        }
      }
      __syncwarp();                               // the partial buffer may be overwritten now
      if (all_dead) {
        consumed = min(cnt, k * CH + sub + nr);
        finished = true;
        break;
      }
    }
    if constexpr (GATHER) {
      if (!finished && k + STAGES < nchunks) {   // every thread is past the barrier: the stage is free
        const int kn = k + STAGES;
        gather_issue<Smem, NT, CH, 4>(sm, stage, grec, goff, gid, min(CH, cnt - kn * CH), tid);
        if (kn + 1 < nchunks) gid.load(ids, start + (kn + 1) * CH, min(CH, cnt - (kn + 1) * CH), tid);
      }
    } else if (tid == 0 && !finished && k + STAGES < nchunks) {
      const int kn = k + STAGES;                 // every thread is past the barrier: the stage is free
      issue_chunk<Smem>(sm, stage, pA, pB, pC, start + kn * CH, min(CH, cnt - kn * CH), shift);
    }
  }
  if (tid == 0) {
    if (finished) {
      // drain copies that were issued but never consumed before the CTA may retire (k was incremented past the
      // chunk that finished): chunks k .. k + STAGES - 2 are in flight
      for (int kk = k; kk < nchunks && kk < k + STAGES - 1; ++kk)
        gs_mbar_wait(&sm.full[kk % STAGES], (uint32_t)((kk / STAGES) & 1));
    }
    if (tile_neff_b) tile_neff_b[tile] = consumed;
  }
  // the unread tail of a saturated tile has zero gradient: with an epoch array the rows are simply
  // left stale (the consumer skips rows whose tag is not this frame's); otherwise write zeros
  if (row_epoch || GATHER) return;              // (the gather path always runs with an epoch array)
  for (int t = consumed + tid; t < cnt; t += NT) {
    const uint32_t slot = __float_as_uint(pC[start + t].w);
    float4* out = reinterpret_cast<float4*>(grad_inst + (size_t)slot * GS_GREC);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    out[0] = z;
    out[1] = z;
    out[2] = z;
  }
}

// =======================================================================================
// legacy boundary helpers: per-instance tensors <-> packed record streams
// =======================================================================================
__global__ void __launch_bounds__(256) legacy_pack_kernel(const float* __restrict__ pos, const float* __restrict__ rgb,
                                                           const float* __restrict__ opa,
                                                           const float* __restrict__ cov, int m,
                                                           float4* __restrict__ pA, float2* __restrict__ pB,
                                                           float4* __restrict__ pC) {
  int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= m) return;
  float4 cv = reinterpret_cast<const float4*>(cov)[i];
  GsConic k = gs_make_conic(cv.x, cv.y, cv.z, cv.w);
  pA[i] = make_float4(pos[3 * i], pos[3 * i + 1], k.ca, k.cb);
  pB[i] = make_float2(k.cc, log2f(opa[i]));
  pC[i] = make_float4(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], __uint_as_float((uint32_t)i));
}

__global__ void __launch_bounds__(256) legacy_unpack_grads_kernel(const float* __restrict__ grad_inst,
                                                                   const float* __restrict__ opa,
                                                                   const float* __restrict__ cov, int m,
                                                                   float* __restrict__ g_pos,
                                                                   float* __restrict__ g_rgb,
                                                                   float* __restrict__ g_opa,
                                                                   float* __restrict__ g_cov) {
  int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= m) return;
  const float4* row = reinterpret_cast<const float4*>(grad_inst + (size_t)i * GS_GREC);
  float4 v0 = row[0], v1 = row[1], v2 = row[2];
  float4 cv = reinterpret_cast<const float4*>(cov)[i];
  float det = cv.x * cv.w - cv.y * cv.z;
  double pn = 2.0 * (double)det + 1e-14;
  float sc = (float)((double)GS_LOG2E / pn);
  float kk = 2.f * sc * sc / GS_LOG2E;
  float gsc = v0.z * cv.w + v0.w * (cv.y + cv.z) + v1.x * cv.x;
  g_pos[3 * i] = v0.x;
  g_pos[3 * i + 1] = v0.y;                                    // z column untouched (gaussian.cu:785-786)
  reinterpret_cast<float4*>(g_cov)[i] = make_float4(v1.x * sc - gsc * kk * cv.w, v0.w * sc + gsc * kk * cv.z,
                                                    v0.w * sc + gsc * kk * cv.y, v0.z * sc - gsc * kk * cv.x);
  g_opa[i] = opa[i] > 0.f ? v1.y / (opa[i] * GS_LN2) : 0.f;   // opacity exactly 0: alpha == 0 everywhere, log2 undefined
  g_rgb[3 * i] = v1.z;
  g_rgb[3 * i + 1] = v1.w;
  g_rgb[3 * i + 2] = v2.x;
}

// SH variants: third stream row = {coef[0..d), slot, pad}; gradient row = {6 geometry, d coefficient}
__global__ void __launch_bounds__(256) legacy_pack_sh_kernel(const float* __restrict__ pos,
                                                              const float* __restrict__ rgb,
                                                              const float* __restrict__ opa,
                                                              const float* __restrict__ cov, int m, int d, int sw,
                                                              float4* __restrict__ pA, float2* __restrict__ pB,
                                                              float* __restrict__ pS) {
  int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= m) return;
  float4 cv = reinterpret_cast<const float4*>(cov)[i];
  GsConic k = gs_make_conic(cv.x, cv.y, cv.z, cv.w);
  pA[i] = make_float4(pos[3 * i], pos[3 * i + 1], k.ca, k.cb);
  pB[i] = make_float2(k.cc, log2f(opa[i]));
  float* row = pS + (size_t)i * sw;
  const float* src = rgb + (size_t)i * d;
  for (int q = 0; q < d; ++q) row[q] = src[q];
  row[d] = __uint_as_float((uint32_t)i);
}

__global__ void __launch_bounds__(256) legacy_unpack_grads_sh_kernel(const float* __restrict__ grad_inst, int gw,
                                                                      const float* __restrict__ opa,
                                                                      const float* __restrict__ cov, int m, int d,
                                                                      float* __restrict__ g_pos,
                                                                      float* __restrict__ g_rgb,
                                                                      float* __restrict__ g_opa,
                                                                      float* __restrict__ g_cov) {
  int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= m) return;
  const float* row = grad_inst + (size_t)i * gw;
  float4 cv = reinterpret_cast<const float4*>(cov)[i];
  float det = cv.x * cv.w - cv.y * cv.z;
  double pn = 2.0 * (double)det + 1e-14;
  float sc = (float)((double)GS_LOG2E / pn);
  float kk = 2.f * sc * sc / GS_LOG2E;
  float d_ca = row[2], d_cb = row[3], d_cc = row[4];
  float gsc = d_ca * cv.w + d_cb * (cv.y + cv.z) + d_cc * cv.x;
  g_pos[3 * i] = row[0];
  g_pos[3 * i + 1] = row[1];
  reinterpret_cast<float4*>(g_cov)[i] = make_float4(d_cc * sc - gsc * kk * cv.w, d_cb * sc + gsc * kk * cv.z,
                                                    d_cb * sc + gsc * kk * cv.y, d_ca * sc - gsc * kk * cv.x);
  g_opa[i] = opa[i] > 0.f ? row[5] / (opa[i] * GS_LN2) : 0.f;
  for (int q = 0; q < d; ++q) g_rgb[(size_t)i * d + q] = row[6 + q];
}

struct LegacyWs {
  float4* pA;
  float2* pB;
  float4* pC;
  float* grad_inst;
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// d == 3: pC is the float4 colour stream; d == 27 / 48: pC aliases the SH stream (sw floats / row)
inline size_t legacy_ws_layout(int m, int d, LegacyWs* ws, char* base) {
  size_t off = 0;
  size_t mm = (size_t)(m > 0 ? m : 0);
  size_t crow = d == 3 ? 16 : (size_t)gs_sh_stream_width(d) * 4;
  size_t grow = d == 3 ? (size_t)GS_GREC * 4 : (size_t)gs_sh_grad_width(d) * 4;
  if (ws) ws->pA = reinterpret_cast<float4*>(base + off);
  off += align_up(mm * 16, 256);
  if (ws) ws->pC = reinterpret_cast<float4*>(base + off);
  off += align_up(mm * crow + 16, 256);
  if (ws) ws->pB = reinterpret_cast<float2*>(base + off);
  off += align_up((mm + 2) * 8, 256);
  if (ws) ws->grad_inst = reinterpret_cast<float*>(base + off);
  off += align_up(mm * grow, 256);
  return off;
}

}  // namespace

cudaError_t gs_launch_blend_fwd(const float4* pA, const float2* pB, const float4* pC, const GsRec* grec,
                                const uint32_t* ids, const int* tile_accum, const GsFrameGeom& g, float* image,
                                int* tile_neff, float* final_img, const GsCrop& crop, cudaStream_t st) {
  const auto kernel = grec ? blend_fwd_kernel<true, false> : blend_fwd_kernel<false, false>;
  kernel<<<g.n_tiles, FWD_THREADS, 0, st>>>(pA, pB, pC, grec, ids, tile_accum, g.wp, g.hp, g.ntx, g.fx, g.fy, image,
                                            tile_neff, final_img, crop, GsMapsFwd{});
  return cudaGetLastError();
}

cudaError_t gs_launch_blend_bwd(const float4* pA, const float2* pB, const float4* pC, const GsRec* grec,
                                const uint32_t* ids, const uint32_t* goff, const int* tile_accum, const GsFrameGeom& g,
                                const float* image,
                                const float* grad_image, float* grad_inst, int grad_is_final, const GsCrop& crop,
                                uint32_t* row_epoch, uint32_t epoch, int* tile_neff_b, cudaStream_t st) {
  if (grec && !row_epoch) return cudaErrorInvalidValue;
  const auto kernel = grec ? blend_bwd_kernel<true, false> : blend_bwd_kernel<false, false>;
  kernel<<<g.n_tiles, BWD_THREADS, 0, st>>>(pA, pB, pC, grec, ids, goff, tile_accum, g.wp, g.hp, g.ntx, g.fx, g.fy, image,
                                            grad_image, grad_inst, grad_is_final, crop, row_epoch, epoch, tile_neff_b,
                                            GsMapsBwd{});
  return cudaGetLastError();
}

cudaError_t gs_launch_blend_fwd_maps(const GsRec* grec, const uint32_t* ids, const int* tile_accum, const GsFrameGeom& g,
                                     float* image, int* tile_neff, float* final_img, const GsCrop& crop,
                                     const GsMapsFwd& maps, cudaStream_t st) {
  // grec / ids may be null: a frame without tile instances (no Gaussian, or none visible, on a context that never
  // had one) never reads them - every tile is empty and renders the background with depth = alpha = 0
  if (!maps.depth || !maps.alpha || (final_img != nullptr) != (maps.depth_final != nullptr) ||
      (maps.depth_final != nullptr) != (maps.alpha_final != nullptr))
    return cudaErrorInvalidValue;
  blend_fwd_kernel<true, true><<<g.n_tiles, FWD_THREADS, 0, st>>>(nullptr, nullptr, nullptr, grec, ids, tile_accum, g.wp,
                                                                   g.hp, g.ntx, g.fx, g.fy, image, tile_neff, final_img,
                                                                   crop, maps);
  return cudaGetLastError();
}

cudaError_t gs_launch_blend_bwd_maps(const GsRec* grec, const uint32_t* ids, const uint32_t* goff, const int* tile_accum,
                                     const GsFrameGeom& g, const float* image, const float* grad_image, float* grad_inst,
                                     int grad_is_final, const GsCrop& crop, uint32_t* row_epoch, uint32_t epoch,
                                     int* tile_neff_b, const GsMapsBwd& maps, cudaStream_t st) {
  // only launched for frames with tile instances (an empty frame has no blend backward), so the records exist
  if (!grec || !ids || !goff || !row_epoch || !maps.depth || !maps.alpha || !maps.grad_depth || !maps.grad_alpha)
    return cudaErrorInvalidValue;
  blend_bwd_kernel<true, true><<<g.n_tiles, BWD_THREADS, 0, st>>>(nullptr, nullptr, nullptr, grec, ids, goff, tile_accum,
                                                                  g.wp, g.hp, g.ntx, g.fx, g.fy, image, grad_image,
                                                                  grad_inst, grad_is_final, crop, row_epoch, epoch,
                                                                  tile_neff_b, maps);
  return cudaGetLastError();
}

extern "C" size_t gs_draw_workspace_bytes(int m, int d) {
  if (d != 3 && gs_sh_basis_count(d) == 0) return 0;
  return legacy_ws_layout(m, d, nullptr, nullptr);
}

static int check_draw_args(const char* fn, int m, int d, int wp, int hp, int weight_normalize, int sigmoid,
                           size_t ws_bytes, void* ws) {
  if (m < 0 || wp <= 0 || hp <= 0 || (wp % GS_TILE) || (hp % GS_TILE))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, fn);
  if (weight_normalize || sigmoid || (d != 3 && gs_sh_basis_count(d) == 0)) return gs_set_error_msg(GS_ERR_UNSUPPORTED, fn);
  if (m > 0 && (ws == nullptr || ws_bytes < gs_draw_workspace_bytes(m, d)))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, fn);
  return 0;
}

extern "C" int gs_draw_fwd(const float* pos, const float* rgb, const float* opa, const float* cov,
                           const int* tile_n_point_accum, int m, int d, int width_padded, int height_padded,
                           float focal_x, float focal_y, int weight_normalize, int sigmoid, const float* rays_o,
                           const float* lefttop, const float* vec_dx, const float* vec_dy, float* image,
                           void* workspace, size_t workspace_bytes, gs_stream_t stream) {
  int rc = check_draw_args("gs_draw_fwd: bad/unsupported arguments", m, d, width_padded, height_padded,
                           weight_normalize, sigmoid, workspace_bytes, workspace);
  if (rc) return rc;
  if (d != 3 && (!rays_o || !lefttop || !vec_dx || !vec_dy))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_draw_fwd: SH colour needs rays_o / lefttop / vec_dx / vec_dy");
  cudaStream_t st = (cudaStream_t)stream;
  LegacyWs ws{};
  legacy_ws_layout(m, d, &ws, static_cast<char*>(workspace));
  if (m > 0) {
    if (d == 3)
      legacy_pack_kernel<<<(m + 255) / 256, 256, 0, st>>>(pos, rgb, opa, cov, m, ws.pA, ws.pB, ws.pC);
    else
      legacy_pack_sh_kernel<<<(m + 255) / 256, 256, 0, st>>>(pos, rgb, opa, cov, m, d, gs_sh_stream_width(d), ws.pA,
                                                             ws.pB, reinterpret_cast<float*>(ws.pC));
    GS_CUDA_TRY(cudaGetLastError());
    gs_count_launch();
  }
  GsFrameGeom g{};
  g.wp = width_padded;
  g.hp = height_padded;
  g.ntx = width_padded / GS_TILE;
  g.nty = height_padded / GS_TILE;
  g.n_tiles = g.ntx * g.nty;
  g.fx = focal_x;
  g.fy = focal_y;
  if (d == 3) {
    GS_CUDA_TRY(gs_launch_blend_fwd(ws.pA, ws.pB, ws.pC, nullptr, nullptr, tile_n_point_accum, g, image, nullptr, nullptr,
                                    GsCrop{}, st));
  } else {
    GsRayPtrs r{rays_o, lefttop, vec_dx, vec_dy};
    GS_CUDA_TRY(gs_launch_blend_sh_fwd(ws.pA, ws.pB, reinterpret_cast<float*>(ws.pC), nullptr, nullptr, nullptr, nullptr, d,
                                       tile_n_point_accum, g, r,
                                       image, nullptr, nullptr, GsCrop{}, st));
  }
  gs_count_launch();
  return 0;
}

extern "C" int gs_draw_bwd(const float* pos, const float* rgb, const float* opa, const float* cov,
                           const int* tile_n_point_accum, int m, int d, int width_padded, int height_padded,
                           float focal_x, float focal_y, int weight_normalize, int sigmoid, const float* rays_o,
                           const float* lefttop, const float* vec_dx, const float* vec_dy, const float* image,
                           const float* grad_image, float* grad_pos, float* grad_rgb, float* grad_opa,
                           float* grad_cov, void* workspace, size_t workspace_bytes, gs_stream_t stream) {
  int rc = check_draw_args("gs_draw_bwd: bad/unsupported arguments", m, d, width_padded, height_padded,
                           weight_normalize, sigmoid, workspace_bytes, workspace);
  if (rc) return rc;
  if (m == 0) return 0;
  if (d != 3 && (!rays_o || !lefttop || !vec_dx || !vec_dy))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_draw_bwd: SH colour needs rays_o / lefttop / vec_dx / vec_dy");
  cudaStream_t st = (cudaStream_t)stream;
  LegacyWs ws{};
  legacy_ws_layout(m, d, &ws, static_cast<char*>(workspace));
  if (d == 3)
    legacy_pack_kernel<<<(m + 255) / 256, 256, 0, st>>>(pos, rgb, opa, cov, m, ws.pA, ws.pB, ws.pC);
  else
    legacy_pack_sh_kernel<<<(m + 255) / 256, 256, 0, st>>>(pos, rgb, opa, cov, m, d, gs_sh_stream_width(d), ws.pA,
                                                           ws.pB, reinterpret_cast<float*>(ws.pC));
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch();
  GsFrameGeom g{};
  g.wp = width_padded;
  g.hp = height_padded;
  g.ntx = width_padded / GS_TILE;
  g.nty = height_padded / GS_TILE;
  g.n_tiles = g.ntx * g.nty;
  g.fx = focal_x;
  g.fy = focal_y;
  if (d == 3) {
    GS_CUDA_TRY(gs_launch_blend_bwd(ws.pA, ws.pB, ws.pC, nullptr, nullptr, nullptr, tile_n_point_accum, g, image,
                                    grad_image,
                                    ws.grad_inst, 0,
                                    GsCrop{}, nullptr, 0u, nullptr, st));
    legacy_unpack_grads_kernel<<<(m + 255) / 256, 256, 0, st>>>(ws.grad_inst, opa, cov, m, grad_pos, grad_rgb,
                                                              grad_opa, grad_cov);
  } else {
    GsRayPtrs r{rays_o, lefttop, vec_dx, vec_dy};
    GS_CUDA_TRY(gs_launch_blend_sh_bwd(ws.pA, ws.pB, reinterpret_cast<float*>(ws.pC), nullptr, nullptr, nullptr, nullptr, d,
                                       tile_n_point_accum, g, r,
                                       image, grad_image, ws.grad_inst, 0, GsCrop{}, nullptr, 0u, nullptr, st));
    legacy_unpack_grads_sh_kernel<<<(m + 255) / 256, 256, 0, st>>>(ws.grad_inst, gs_sh_grad_width(d), opa, cov, m, d,
                                                                 grad_pos, grad_rgb, grad_opa, grad_cov);
  }
  GS_CUDA_TRY(cudaGetLastError());
  gs_count_launch(2);   // blend backward + unpack
  return 0;
}
