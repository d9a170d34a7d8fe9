// Shared device helpers for libgs_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define GS_TILE 16
#define GS_LOG2E 1.4426950408889634f
#define GS_LN2 0.6931471805599453f
// Early stop: the reference tests `accum < 0.0001` with a double literal
// (gaussian.cu:906,:578); for a float accum that is exactly `accum <= 1e-4f`
// (1e-4f is the largest float below the double 0.0001).
#define GS_T_STOP 1e-4f

#define GS_CUDA_TRY(expr)                                  \
  do {                                                     \
    cudaError_t _e = (expr);                               \
    if (_e != cudaSuccess) return gs_set_error(_e, #expr); \
  } while (0)

int gs_set_error(cudaError_t e, const char* what);
int gs_set_error_msg(int code, const char* what);

// ---- packed per-instance record streams consumed by the blend kernels ------------------
// A[i] = {x, y, ca, cb}       centre (normalised image plane) + conic * log2e / (2det+1e-14)
// B[i] = {cc, l2o}            third conic term, log2(opacity)
// C[i] = {r, g, b, slot}      activated colour, slot = destination row of this instance's
//                             gradient record (int bits)
// alpha(px,py) = exp2(l2o - (ca*dx*dx - cb*dx*dy + cc*dy*dy)),  dx = px-x, dy = py-y
//   == opa * __expf(-(d*dx^2 - (b+c)*dx*dy + a*dy^2) / (2*det + 1e-14))   (gaussian.cu:920-926)
// Per-Gaussian record produced by the fused projection (one 64-byte line = two sectors, so the
// post-sort gather touches 2 sectors per instance instead of 5 separate arrays).
struct __align__(64) GsRec {
  float4 a;      // x, y, ca, cb
  float4 b;      // cc, l2o, r, g
  float4 c;      // b, depth, rect(tx0 | ty0<<16) bits, rect(w | h<<16) bits
  uint4 d;       // offsets[g] (first instance row), unused x3
};

struct GsConic {
  float ca, cb, cc;
};

__device__ __forceinline__ GsConic gs_make_conic(float a, float b, float c, float d) {
  // (2*det + 1e-14) is evaluated in double in the reference (double literal).
  float det = a * d - b * c;
  double pn = 2.0 * (double)det + 1e-14;
  float s = (float)((double)GS_LOG2E / pn);
  GsConic k;
  k.ca = d * s;
  k.cb = (b + c) * s;
  k.cc = a * s;
  return k;
}

__device__ __forceinline__ float gs_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float gs_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float gs_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---- mbarrier + 1-D bulk async copy (TMA engine, UBLKCP in SASS) -----------------------
__device__ __forceinline__ uint32_t gs_smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void gs_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gs_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void gs_fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void gs_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gs_smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void gs_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          gs_smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(gs_smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void gs_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  uint32_t addr = gs_smem_u32(bar);
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!ok);
}

// named barrier over a SUBSET of the CTA's warps.  `n` = number of participating threads (multiple of 32).
__device__ __forceinline__ void gs_bar_sync(int id, int n) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory");
}

// pixel centre in normalised image-plane units, gaussian.cu:839-840 (double arithmetic,
// `w/2` is an unsigned integer division)
__device__ __forceinline__ float gs_pixel_coord(int idx, int extent, float focal) {
  return (float)(((double)idx + 0.5 - (double)(extent / 2)) / (double)focal);
}

// ---- fused clamp + crop helpers (reference splatter.py:652-653) ---------------------------
__device__ __forceinline__ void gs_store_final(float* __restrict__ final_img, int ix, int iy, int left, int top,
                                               int width, int height, float r, float g, float b) {
  const int x = ix - left, y = iy - top;
  if (x >= 0 && x < width && y >= 0 && y < height) {
    float* o = final_img + ((size_t)y * width + x) * 3;
    o[0] = fminf(fmaxf(r, 0.f), 1.f);
    o[1] = fminf(fmaxf(g, 0.f), 1.f);
    o[2] = fminf(fmaxf(b, 0.f), 1.f);
  }
}
// gradient of the final (clamped, cropped) image seen from the raw padded image: torch.clamp
// passes the gradient where 0 <= v <= 1; pixels outside the crop receive none
__device__ __forceinline__ void gs_load_final_grad(const float* __restrict__ grad_final, const float* raw3, int ix,
                                                   int iy, int left, int top, int width, int height, float& gr,
                                                   float& gg, float& gb) {
  const int x = ix - left, y = iy - top;
  gr = gg = gb = 0.f;
  if (x >= 0 && x < width && y >= 0 && y < height) {
    const float* g = grad_final + ((size_t)y * width + x) * 3;
    gr = (raw3[0] >= 0.f && raw3[0] <= 1.f) ? g[0] : 0.f;
    gg = (raw3[1] >= 0.f && raw3[1] <= 1.f) ? g[1] : 0.f;
    gb = (raw3[2] >= 0.f && raw3[2] <= 1.f) ? g[2] : 0.f;
  }
}
