// Internal (non-ABI) launcher declarations shared between the translation units of libgs_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gs_b200.h"
#include "project.cuh"

// Width (floats) of one per-instance gradient record written by the blend backward:
// {d_x, d_y, d_ca, d_cb, d_cc, d_l2o, d_r, d_g, d_b} (+ 3 pad so rows are 16-byte aligned)
#define GS_GREC 12

struct GsFrameGeom {
  int width, height, wp, hp, ntx, nty, n_tiles;
  float fx, fy;
};

// Optional fused post-processing of reference splatter.py:652-653 (clamp to [0,1] + centre crop):
// forward additionally writes final[height,width,3]; backward takes the gradient of that final
// image (clamp mask from the raw padded image, zero outside the crop) instead of a padded one.
struct GsCrop {
  int left, top, width, height;
};

// Depth / alpha maps and a background colour (gs_render_forward_maps; RGB gather path only).  Per pixel, over the
// instances the colour blend uses: image += T_end * bg, depth = sum w_i d_i (d_i = |p_c|, GsRec.c.y), alpha = 1 - T_end.
// Forward: raw padded planes [Hp,Wp]; the cropped [H,W] planes (no clamp) when the final layout is requested.
struct GsMapsFwd {
  float* depth;
  float* alpha;
  float* depth_final;           // nullable (with final_img == nullptr)
  float* alpha_final;
  float bg_r, bg_g, bg_b;
};
// Backward: the forward's raw planes and the gradients of the depth / alpha maps (padded, or cropped [H,W] when
// grad_is_final; zero outside the crop, no clamp mask)
struct GsMapsBwd {
  const float* depth;
  const float* alpha;
  const float* grad_depth;
  const float* grad_alpha;
};

// world-space ray setup for per-pixel SH (reference splatter.py:305-321), DEVICE pointers to 3 floats each
struct GsRayPtrs {
  const float *rays_o, *lefttop, *dx, *dy;
};

// Run-time tuning knobs (the defaults are the shipped configuration).  Set with gs_tune("name", value) or the
// environment variable GS_TUNE_<NAME> (read once; an out-of-range value there keeps the default).
struct GsTuning {
  int gather;       // fused frame path (RGB and SH): 1 = no pack pass, blend kernels gather records from rec[N]; 0 = packed streams
  int sh_tc;        // SH blend on the tensor cores (blend_sh_tc.cu, gather path only): bit 0 = forward, bit 1 = backward
};
GsTuning& gs_tuning();

// every launch of one of OUR kernels is counted (bench.py reports the count of the timed region)
void gs_count_launch(int n = 1);

// ---- blend_sh.cu -----------------------------------------------------------------------
int gs_sh_basis_count(int d);      // 27 -> 9, 48 -> 16, else 0
int gs_sh_stream_width(int d);     // floats per instance row of the SH stream (coefficients + slot, padded)
int gs_sh_grad_width(int d);       // floats per instance gradient row (6 geometry + d coefficients, padded)
// grec != nullptr: gather path (records from rec[N], raw coefficients from the parameter tensor rgb[N, d])
cudaError_t gs_launch_blend_sh_fwd(const float4* pA, const float2* pB, const float* pS, const GsRec* grec,
                                   const float* rgb, const uint32_t* ids, const uint32_t* goff /*offsets_g*/, int d,
                                   const int* tile_accum,
                                   const GsFrameGeom& g, const GsRayPtrs& r, float* image, int* tile_neff,
                                   float* final_img, const GsCrop& crop, cudaStream_t st);
cudaError_t gs_launch_blend_sh_bwd(const float4* pA, const float2* pB, const float* pS, const GsRec* grec,
                                   const float* rgb, const uint32_t* ids, const uint32_t* goff /*offsets_g*/, int d,
                                   const int* tile_accum,
                                   const GsFrameGeom& g, const GsRayPtrs& r, const float* image,
                                   const float* grad_image, float* grad_inst, int grad_is_final, const GsCrop& crop,
                                   uint32_t* row_epoch, uint32_t epoch, int* tile_neff_b, cudaStream_t st);

// ---- blend_sh_tc.cu (tcgen05 / TMEM) -----------------------------------------------------
cudaError_t gs_launch_blend_sh_fwd_tc(const GsRec* grec, const float* rgb, const uint32_t* ids, int d,
                                      const int* tile_accum, const GsFrameGeom& g, const GsRayPtrs& r, float* image,
                                      int* tile_neff, float* final_img, const GsCrop& crop, cudaStream_t st);
cudaError_t gs_launch_blend_sh_bwd_tc(const GsRec* grec, const float* rgb, const uint32_t* ids, const uint32_t* goff, int d,
                                      const int* tile_accum, const GsFrameGeom& g, const GsRayPtrs& r, const float* image,
                                      const float* grad_image, float* grad_inst, int grad_is_final, const GsCrop& crop,
                                      uint32_t* row_epoch, uint32_t epoch, int* tile_neff_b, cudaStream_t st);

// ---- project.cu ------------------------------------------------------------------------
cudaError_t gs_launch_fused_project(const float* pos, const float* rgb, const float* opa, const float* quat,
                                    const float* scale, int n, int d, int scale_act, const GsCam& cam,
                                    const GsTileGrid& grid, float near_plane, float half_w, float half_h,
                                    GsRec* rec, uint32_t* count, uint32_t* dkey, int64_t* mask,
                                    unsigned int* n_visible, cudaStream_t st);

// Data-parallel gradient push (device view of gs_grad_push): world == 0 disables it.
struct GsGradPush {
  float* bucket;                  // this rank's flat gradient bucket (the five grad pointers lie inside)
  float* staging[GS_MAX_PEERS];   // staging[p] = rank p's staging buffer [world][per] as mapped here
  uint32_t per;                   // floats per slice (multiple of 4)
  int rank, world;
};

cudaError_t gs_launch_fused_project_bwd(const float* pos, const float* rgb, const float* opa, const float* quat,
                                        const float* scale, int n, int d, int scale_act, const GsCam& cam,
                                        float near_plane, float half_w, float half_h, const uint32_t* offsets_g,
                                        const uint32_t* count, const float* grad_inst, const uint32_t* row_epoch, uint32_t epoch,
                                        float* g_pos, float* g_rgb, float* g_opa,
                                        float* g_quat, float* g_scale, const GsGradPush& push, cudaStream_t st,
                                        bool depth_grad = false /*maps frame: chain float 9 of the rows to pos*/,
                                        double* cam_partial = nullptr /*camera gradient: [blocks][12] partial rows*/);
// Camera gradient (gs_ctx_set_camera_grad; RGB, one GPU): bytes of the partial rows the projection backward of n
// Gaussians writes, and the one-block kernel that sums them in a fixed order into grad_cam[12] (zeros when n == 0).
size_t gs_camgrad_partial_bytes(int n);
cudaError_t gs_launch_camgrad_finish(const double* cam_partial, int n, float* grad_cam, cudaStream_t st);

// ---- binning.cu ------------------------------------------------------------------------
cudaError_t gs_launch_emit_keys(const GsRec* rec, const uint32_t* perm, const uint32_t* offsets_sorted, int n, int ntx,
                                void* keys, int key_bytes, uint32_t* vals, cudaStream_t st);
cudaError_t gs_launch_tile_ranges(const void* keys, int key_bytes, long long m, int n_tiles, int* tile_accum,
                                  cudaStream_t st);

cudaError_t gs_launch_pack_sorted(const void* keys, int key_bytes, const uint32_t* vals, long long m, int n_tiles,
                                  int ntx, const GsRec* rec, const uint32_t* offsets_g, float4* pA, float2* pB, float4* pC,
                                  int* tile_accum, cudaStream_t st);

cudaError_t gs_launch_pack_sorted_sh(const void* keys, int key_bytes, const uint32_t* vals, long long m, int n_tiles,
                                     int ntx, const GsRec* rec, const uint32_t* offsets_g, const float* rgb, int d, int sw,
                                     float4* pA, float2* pB, float* pS, int* tile_accum, cudaStream_t st);
cudaError_t gs_launch_iota(uint32_t* out, int n, cudaStream_t st);

// ---- blend.cu --------------------------------------------------------------------------
// grec / ids != nullptr: gather path (records pulled straight from rec[N] through the sorted id list; the packed
// stream pointers are ignored); else the packed streams written by the pack pass / the legacy draw API.
cudaError_t gs_launch_blend_fwd(const float4* pA, const float2* pB, const float4* pC, const GsRec* grec,
                                const uint32_t* ids, const int* tile_accum, const GsFrameGeom& g, float* image,
                                int* tile_neff, float* final_img, const GsCrop& crop, cudaStream_t st);

cudaError_t gs_launch_blend_bwd(const float4* pA, const float2* pB, const float4* pC, const GsRec* grec,
                                const uint32_t* ids, const uint32_t* goff /*offsets_g (gather path)*/,
                                const int* tile_accum, const GsFrameGeom& g, const float* image,
                                const float* grad_image, float* grad_inst /*[M,GS_GREC] rows addressed by slot*/,
                                int grad_is_final, const GsCrop& crop, uint32_t* row_epoch /*nullable (packed only)*/,
                                uint32_t epoch, int* tile_neff_b /*nullable: instances the backward consumed per tile*/,
                                cudaStream_t st);

// Maps frame (gather path).  The backward additionally writes d/d depth_i = sum g_D w into float 9 of every gradient row.
cudaError_t gs_launch_blend_fwd_maps(const GsRec* grec, const uint32_t* ids, const int* tile_accum, const GsFrameGeom& g,
                                     float* image, int* tile_neff, float* final_img, const GsCrop& crop,
                                     const GsMapsFwd& maps, cudaStream_t st);
cudaError_t gs_launch_blend_bwd_maps(const GsRec* grec, const uint32_t* ids, const uint32_t* goff, const int* tile_accum,
                                     const GsFrameGeom& g, const float* image, const float* grad_image, float* grad_inst,
                                     int grad_is_final, const GsCrop& crop, uint32_t* row_epoch, uint32_t epoch,
                                     int* tile_neff_b, const GsMapsBwd& maps, cudaStream_t st);
