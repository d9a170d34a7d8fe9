/*
 * gs_b200.h — C ABI of libgs_b200.so: B200-native (sm_100a) differentiable tile rasterizer.
 *
 * This is the drop-in boundary for the hot path of WangFeng18/3d-gaussian-splatting
 * (projection + 3D->2D covariance, (tile|depth) sort, front-to-back alpha blend, and the
 * backward of all of it).  The reference exposes that path as a torch/pybind11 module
 * named `gaussian` (reference src/bindings.cpp:21-50); our pybind shim
 * (3d-gaussian-splatting_b200/csrc/bindings.cpp) keeps that Python-visible surface and
 * forwards every call to the functions below.  Everything here is plain C:
 *   - raw DEVICE pointers (unless a name ends in `_host`), explicit sizes,
 *   - a trailing `gs_stream_t` (a `cudaStream_t`; NULL = legacy default stream),
 *   - return value: 0 on success, otherwise a `cudaError_t` code (or GS_ERR_* < 0),
 *   - no function allocates or synchronises unless its comment says so.
 * All tensors are dense row-major float32 unless stated; indices int32; mask int64.
 */
#ifndef GS_B200_H
#define GS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gs_stream_t; /* cudaStream_t */

#define GS_ERR_INVALID_ARG (-1)
#define GS_ERR_UNSUPPORTED (-2)
#define GS_ERR_NO_FORWARD (-3)

/* ABI version of this header (bumped on any signature change). */
int gs_abi_version(void);
/* Human-readable text of the last error on this host thread ("" if none). */
const char* gs_last_error(void);
/* Blend-path knobs (defaults = the shipped configuration; environment GS_TUNE_GATHER / GS_TUNE_SH_TC, read once):
 *   "gather"  1 (default) = the fused frame's blend kernels gather records through the sorted id list;
 *             0 = a pack pass writes record streams first (the legacy draw API's kernels)
 *   "sh_tc"   0..3, default 3: SH blend of the gather path on the tensor cores, bit 0 = forward, bit 1 = backward
 *             (0 = the scalar kernels)
 * An unknown name or a value out of range returns GS_ERR_INVALID_ARG and leaves the knob unchanged.
 * Process-wide, not thread-safe. */
int gs_tune(const char* name, int value);
/* New: current value of a gs_tune knob (e.g. to restore it after an experiment). */
int gs_tune_get(const char* name, int* value);
/* Number of kernels of THIS library launched by the process so far (library kernels such as CUB's are not
 * counted); bench.py reports the difference over its timed region as `gpu_launches`. */
unsigned long long gs_kernel_launches(void);

/* ---------------------------------------------------------------------------------------
 * Legacy per-stage entry points == the reference's `gaussian` module functions.
 * ------------------------------------------------------------------------------------- */

/* global_culling — reference bindings.cpp:48, gaussian.cu:1338-1369 (kernel :1182-1336).
 * quat/scale are PRE-activated (splatter.py:519-524).  res_pos[n,3]=(x/z,y/z,|p_c|),
 * res_cov[n,2,2], mask[n] int64; outputs must be zero-filled by the caller (culled rows
 * are left untouched, like the reference). */
int gs_project_fwd(const float* pos, const float* quat, const float* scale, const float* rot,
                   const float* tran, int n, float near_plane, float half_width, float half_height,
                   float* res_pos, float* res_cov, int64_t* mask, gs_stream_t stream);

/* global_culling_backward — bindings.cpp:49, gaussian.cu:1578-1609 (kernel :1371-1576).
 * The projection Jacobian is treated as constant (no d cov2d / d pos), as in the reference. */
int gs_project_bwd(const float* pos, const float* quat, const float* scale, const float* rot,
                   const float* tran, const float* gradout_pos, const float* gradout_cov,
                   const int64_t* mask, int n, float* gradin_pos, float* gradin_quat,
                   float* gradin_scale, gs_stream_t stream);

/* calc_tile_list — bindings.cpp:44, gaussian.cu:254-335.  method 0 "dist" (:101-136),
 * 1 "prob" (:138-195), 2 "prob2" (:197-250).  tile_top/bottom/left/right[n_tiles] are only
 * read by methods 0/1.  tile_n_point[T] is incremented (may exceed max_per_tile; entries
 * beyond capacity are dropped, caller clamps — splatter.py:586). */
int gs_tile_list(const float* pos /*[n,3]*/, const float* cov /*[n,4]*/, int n,
                 const float* tile_top, const float* tile_bottom, const float* tile_left,
                 const float* tile_right, int n_tiles, int* tile_n_point, int* tile_gaussian_list,
                 int max_per_tile, float thresh, int method, float tile_length_x, float tile_length_y,
                 int n_tiles_x, int n_tiles_y, float leftmost, float topmost, gs_stream_t stream);

/* gather_gaussians — bindings.cpp:45, gaussian.cu:359-381. */
int gs_gather(const int* tile_n_point_accum /*[T+1]*/, const int* tile_gaussian_list /*[T,list_stride]*/,
              int n_tiles, int list_stride, int max_points_for_tile, int* gathered_list /*[M]*/,
              int* tile_ids_for_points /*[M]*/, gs_stream_t stream);

/* Scratch bytes needed by gs_draw_fwd / gs_draw_bwd for m tile-instances with colour width
 * d (3 = RGB, 27 = SH degree 2). */
size_t gs_draw_workspace_bytes(int m, int d);

/* draw — bindings.cpp:46, gaussian.cu:973-1043 (kernel :806-970).  Inputs are the already
 * (tile, depth)-sorted per-instance tensors pos[m,3], rgb[m,d], opa[m], cov[m,2,2] and
 * tile_n_point_accum[T+1]; image[Hp,Wp,3] is fully overwritten.  d = 3 or 27
 * (use_sh_coeff).  `weight_normalize` / `sigmoid` must be 0 (GS_ERR_UNSUPPORTED
 * otherwise: the reference never enables them, splatter.py:627, train.py:377).
 * rays_o/lefttop/vec_dx/vec_dy[3] are only read when d == 27 (splatter.py:305-321). */
int gs_draw_fwd(const float* pos, const float* rgb, const float* opa, const float* cov,
                const int* tile_n_point_accum, int m, int d, int width_padded, int height_padded,
                float focal_x, float focal_y, int weight_normalize, int sigmoid,
                const float* rays_o, const float* lefttop, const float* vec_dx, const float* vec_dy,
                float* image, void* workspace, size_t workspace_bytes, gs_stream_t stream);

/* draw_backward — bindings.cpp:47, gaussian.cu:1045-1129 (kernel :440-803).
 * grad_pos[m,3] (z column untouched), grad_rgb[m,d], grad_opa[m], grad_cov[m,2,2] receive the
 * per-instance gradients (every row of the listed columns is written). */
int gs_draw_bwd(const float* pos, const float* rgb, const float* opa, const float* cov,
                const int* tile_n_point_accum, int m, int d, int width_padded, int height_padded,
                float focal_x, float focal_y, int weight_normalize, int sigmoid,
                const float* rays_o, const float* lefttop, const float* vec_dx, const float* vec_dy,
                const float* image, const float* grad_image,
                float* grad_pos, float* grad_rgb, float* grad_opa, float* grad_cov,
                void* workspace, size_t workspace_bytes, gs_stream_t stream);

/* world2camera / world2camera_backward / jacobian — bindings.cpp:24-26,
 * gaussian.cu:71-76, :95-99, :41-47 (deprecated cudaculling=0 path). */
int gs_w2c_fwd(const float* pos, const float* rot, const float* tran, int n, float* res, gs_stream_t stream);
int gs_w2c_bwd(const float* grad_out, const float* rot, int n, float* grad_in, gs_stream_t stream);
int gs_jacobian(const float* pos_cam, int n, float* jac /*[n,3,3]*/, gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Fused frame path (additive; replaces the PyTorch glue of splatter.py:513-655 and the
 * autograd glue around it): parameters -> image, grad_image -> parameter gradients.
 * ------------------------------------------------------------------------------------- */

typedef struct gs_ctx gs_ctx; /* owns device workspaces; one per (device, in-flight frame).  NOT thread-safe:
                                 use a context from one host thread / one stream at a time; it holds the
                                 intermediate state of its LAST forward only. */

typedef struct gs_camera {
  int width, height;          /* un-padded image size; render target is padded to x16 */
  float focal_x, focal_y;     /* principal point = image centre (splatter.py:499-500)  */
  float rot[9];               /* world->camera rotation, row-major                      */
  float tran[3];
  float near_plane;           /* splatter.py: near=0.3                                   */
  float tile_thresh;          /* bbox probability threshold, train.py:310 (0.05)         */
} gs_camera;

typedef struct gs_frame_info {
  int n_gaussians;            /* N                                                       */
  int n_visible;              /* Nc: passed near + 1.2x frustum cull                     */
  long long n_instances;      /* M : tile-instances binned                               */
  long long n_instances_eff;  /* M_eff: instances actually consumed before every pixel   */
                              /*        of their tile saturated (filled by forward)      */
  int width_padded, height_padded, n_tiles;
  int max_tile_count;
  long long n_instances_eff_bwd; /* instances the last BACKWARD consumed (sub-chunk granular); -1 if none ran */
} gs_frame_info;

/* scale_activation: 0 = abs()+1e-4 (splatter.py:521), 1 = trunc_exp (splatter.py:524). */
#define GS_SCALE_ABS 0
#define GS_SCALE_EXP 1

int gs_ctx_create(gs_ctx** out);           /* binds to the current CUDA device            */
/* Optional: workspaces of this context come from the caller's allocator instead of cudaMalloc / cudaFree
 * (which synchronise the stream when a buffer has to grow, e.g. after every densification).  `alloc` returns
 * device memory usable on `stream` (NULL = out of memory), `free_fn` releases it stream-ordered (the caller's
 * allocator must keep the block alive until the work already enqueued on that stream has finished - PyTorch's
 * caching allocator does; the torch shim installs it).  Pass NULL, NULL to go back to cudaMalloc. */
typedef void* (*gs_alloc_fn)(size_t bytes, void* user, gs_stream_t stream);
typedef void (*gs_free_fn)(void* ptr, void* user);
int gs_ctx_set_allocator(gs_ctx* ctx, gs_alloc_fn alloc, gs_free_fn free_fn, void* user);
void gs_ctx_destroy(gs_ctx* ctx);          /* frees workspaces (synchronises the device)  */

/* Raw parameters (splatter.py:399-406): pos[n,3], rgb[n,d] (logits if d==3, SH coefficients
 * channel-major [c*K+k] if d==27), opa[n] logits, quat[n,4] wxyz un-normalised, scale[n,3]
 * raw.  Writes image[Hp,Wp,3] (un-clamped, padded; black background) and, if non-NULL,
 * culling_mask[n] int64 (train.py:150).  Performs ONE host synchronisation on `stream`
 * (reads back the instance count M to size the sort). */
int gs_render_forward(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                      const float* quat, const float* scale, int n, int d, int scale_activation,
                      const gs_camera* cam_host, float* image, int64_t* culling_mask,
                      gs_stream_t stream);

/* Backward of the most recent gs_render_forward on `ctx` (same parameter pointers).
 * grad_image[Hp,Wp,3]; `image` is the forward output.  Writes (overwrites, all n rows)
 * grad_pos[n,3], grad_rgb[n,d], grad_opa[n], grad_quat[n,4], grad_scale[n,3]:
 * gradients wrt the RAW parameters (activation backward included).  No synchronisation. */
int gs_render_backward(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                       const float* quat, const float* scale, const float* image,
                       const float* grad_image, float* grad_pos, float* grad_rgb, float* grad_opa,
                       float* grad_quat, float* grad_scale, gs_stream_t stream);

/* Same as gs_render_forward / gs_render_backward with the post-processing of reference
 * splatter.py:652-653 fused in: forward additionally writes image_final[height,width,3] =
 * centre crop of clamp(image_raw_padded, 0, 1); backward takes grad_final[height,width,3], the
 * gradient of that final image (clamp passes gradients where 0 <= raw <= 1; padding gets none). */
int gs_render_forward_final(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                            const float* quat, const float* scale, int n, int d, int scale_activation,
                            const gs_camera* cam_host, float* image_raw_padded, float* image_final,
                            int64_t* culling_mask, gs_stream_t stream);
int gs_render_backward_final(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                             const float* quat, const float* scale, const float* image_raw_padded,
                             const float* grad_final, float* grad_pos, float* grad_rgb, float* grad_opa,
                             float* grad_quat, float* grad_scale, gs_stream_t stream);

/* New (an extension, not a replacement of a reference function; the reference composites colour on black only):
 * the frame of gs_render_forward[_final] plus a depth map, an alpha map and a background colour.
 * For a pixel, over exactly the instances (and the early stop) of the colour blend, w_i = alpha_i T_i:
 *   image = sum w_i c_i + T_end * background     (background_host: 3 host floats; NULL = black = gs_render_forward)
 *   depth = sum w_i d_i,  d_i = |R p_i + t|       (the depth of global_culling's res_pos[:,2] and of the sort key;
 *                                                  accumulated, not normalised: expected depth = depth / alpha)
 *   alpha = 1 - T_end
 * Writes image_raw_padded[Hp,Wp,3] (un-clamped), depth_raw_padded[Hp,Wp], alpha_raw_padded[Hp,Wp] and, when the
 * three final pointers are set (all NULL or all set), image_final[height,width,3] = crop(clamp(image, 0, 1)),
 * depth_final / alpha_final[height,width] = crop(.) with NO clamp.  Same launches and one host synchronisation,
 * like gs_render_forward.  GS_ERR_UNSUPPORTED (reason in gs_last_error) for d != 3 (SH colour), with
 * gs_tune("gather", 0), and while a gs_ctx_set_grad_push configuration is active. */
int gs_render_forward_maps(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                           const float* quat, const float* scale, int n, int d, int scale_activation,
                           const gs_camera* cam_host, const float* background_host,
                           float* image_raw_padded, float* depth_raw_padded, float* alpha_raw_padded,
                           float* image_final, float* depth_final, float* alpha_final,
                           int64_t* culling_mask, gs_stream_t stream);
/* New.  Backward of the most recent gs_render_forward_maps on ctx: the gradient of
 * <grad_image, image> + <grad_depth, depth> + <grad_alpha, alpha> wrt the five RAW parameters (overwrites all n rows,
 * like gs_render_backward).  The raw planes are the forward's outputs.  grad_is_final = 0: padded gradients
 * ([Hp,Wp,3], [Hp,Wp], [Hp,Wp]); 1: gradients of the final outputs ([height,width,3], [height,width] x 2; the image
 * clamp passes gradient where 0 <= raw <= 1, the maps have no clamp, the padding gets none).  Pass zero-filled
 * planes for outputs without a gradient.  pos receives the direct depth term through d_i; the background is a
 * constant (no gradient).  GS_ERR_NO_FORWARD if the last forward on ctx was not a maps forward; GS_ERR_UNSUPPORTED
 * as for the forward.  No synchronisation. */
int gs_render_backward_maps(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                            const float* quat, const float* scale, const float* image_raw_padded,
                            const float* depth_raw_padded, const float* alpha_raw_padded,
                            const float* grad_image, const float* grad_depth, const float* grad_alpha,
                            int grad_is_final, float* grad_pos, float* grad_rgb, float* grad_opa,
                            float* grad_quat, float* grad_scale, gs_stream_t stream);

/* New (an extension; the reference treats the camera as a constant): camera pose gradients.  While grad_cam is set
 * (a DEVICE pointer to 12 floats, 4-byte aligned; NULL clears it), every gs_render_backward, gs_render_backward_final
 * and gs_render_backward_maps on ctx also overwrites grad_cam with the gradient of the same L as the parameter
 * gradients (<grad_image, image>, plus <grad_depth, depth> + <grad_alpha, alpha> for a maps frame) wrt the camera of
 * ctx's last forward:
 *   grad_cam[0..9)  = dL/d rot   (row-major; the 9 entries as independent variables, no SO(3) projection: chain it to
 *                                 a quaternion / axis-angle parametrisation on the caller's side)
 *   grad_cam[9..12) = dL/d tran
 * Conventions as for the parameters: the projection Jacobian J is detached (p_c = R p + t and J R both carry R), the
 * 1.2x frustum cull, the near plane, the tile binning and the sort order are constants, and in plain frames the depth
 * is a sort key only (maps frames add the depth map's d_i = |R p_i + t|).  Deterministic (no atomics); the backward
 * launches one more kernel.  A frame without instances writes zeros.  Refused at backward time with
 * GS_ERR_UNSUPPORTED (reason in gs_last_error) for d != 3 (SH colour: the per-pixel SH basis depends on the camera
 * through the ray directions, which is not differentiated) and while a gs_ctx_set_grad_push configuration is active,
 * whichever of the two was set first.  GS_ERR_INVALID_ARG for a null ctx or a misaligned pointer. */
int gs_ctx_set_camera_grad(gs_ctx* ctx, float* grad_cam);

/* Per-stage device timing with CUDA events recorded on the frame's stream (off by default).
 * gs_frame_stage_ms fills out[GS_N_STAGES] with the milliseconds of the last frame's stages:
 * 0 project, 1 depth sort of Gaussians + scan + M readback, 2 key emit, 3 tile-id radix sort,
 * 4 range + pack, 5 blend forward,
 * 6 blend backward, 7 project backward (-1 where not available).  Synchronises `stream`. */
#define GS_N_STAGES 8
int gs_ctx_set_timing(gs_ctx* ctx, int enable);
int gs_frame_stage_ms(gs_ctx* ctx, float* out_host, gs_stream_t stream);

/* M (tile-instances) of the last forward on ctx, -1 if none; no synchronisation (the forward
 * already read it back). */
long long gs_frame_instances(gs_ctx* ctx);

/* Statistics of the last forward on ctx (host struct; synchronises `stream` for M_eff). */
int gs_frame_stats(gs_ctx* ctx, gs_frame_info* out_host, gs_stream_t stream);

/* Exposes the last frame's sorted instance list for parity tests: copies
 * min(capacity, M) entries of the sorted Gaussian ids into gauss_idx (device int32) and
 * T+1 entries into tile_accum (device int32).  Either pointer may be NULL. */
int gs_frame_sorted(gs_ctx* ctx, int* gauss_idx, long long capacity, int* tile_accum, gs_stream_t stream);

/* Per-tile consumed instance counts of the last forward (device int32 [T]): tile t's blend stopped
 * after tile_consumed[t] of its tile_accum[t+1]-tile_accum[t] instances because every pixel had
 * saturated (M_eff = their sum).  For parity tests / roofline accounting. */
int gs_frame_tile_consumed(gs_ctx* ctx, int* tile_consumed, gs_stream_t stream);

/* End-to-end convenience with HOST buffers (bench `e2e` leg and plain-C callers): copies
 * the camera + grad_image from host, runs forward + backward on device-resident parameters,
 * copies the padded image back.  Host buffers should be pinned.  Synchronises. */
int gs_render_forward_backward_host(gs_ctx* ctx, const float* pos, const float* rgb, const float* opa,
                                    const float* quat, const float* scale, int n, int d,
                                    int scale_activation, const gs_camera* cam_host,
                                    const float* grad_image_host, float* image_host,
                                    float* grad_pos, float* grad_rgb, float* grad_opa,
                                    float* grad_quat, float* grad_scale, gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Next-row widening (SURVEY.md §8 f-2): fused Adam over the flat parameter / gradient buckets.
 * Replaces torch.optim.Adam over the five parameter groups of reference train.py:56-64 (same
 * update as torch's single-tensor Adam, no weight decay / amsgrad).  `param`, `grad`, `exp_avg`,
 * `exp_avg_sq` are flat device buffers of n floats (n % 4 == 0) split into n_seg (<= 8) segments
 * ending at seg_end_host[s] (ascending multiples of 4) with learning rate lr_host[s]; `step` is
 * the 1-based step count used for the bias corrections. */
int gs_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                 const long long* seg_end_host, const float* lr_host, int n_seg, float beta1, float beta2,
                 float eps, int step, gs_stream_t stream);

/* Densification on the device (SURVEY.md §8 f-2; reference splatter.py:122-228 `adaptive_control`, called
 * from train.py:156-172): prune Gaussians with opacity logit <= opa_logit_min or activated-scale norm >=
 * delete_thresh; of the kept ones whose aggregated |grad| (max or mean over xyz) exceeds grad_thresh, CLONE the
 * small ones (norm <= tau; the copy is moved by -grad * clone_dt) and SPLIT the large ones (scale / 1.6, or
 * - log 1.6 for the exp activation; both halves re-positioned at pos + R (s_act * z), z ~ N(0, I) supplied by the
 * caller so that data-parallel replicas draw identical samples).
 *   gs_densify_plan : code[n+1] (bit0 keep, bit1 clone, bit2 split) and dst[3][n+1] = exclusive scans of the
 *                     three flags (dst[b][n] = totals: n_keep, n_clone, n_split).  No synchronisation.
 *   gs_densify_apply: writes the n_keep + n_clone + n_split rows of the new parameter arrays, laid out like the
 *                     reference's torch.cat: kept (in order), clones (in order), second split samples (in order).
 *                     normals: [2][n_split][3].  Output arrays are caller-allocated. */
size_t gs_densify_workspace_bytes(int n);
int gs_densify_plan(const float* opa, const float* scale, const float* grad, int n, int scale_activation,
                    float opa_logit_min, float delete_thresh, float grad_thresh, int grad_agg_max, float tau,
                    int use_clone, int use_split, unsigned char* code, int* dst, void* workspace,
                    size_t workspace_bytes, gs_stream_t stream);
int gs_densify_apply(const float* pos, const float* rgb, const float* opa, const float* quat, const float* scale,
                     int n, int d, const unsigned char* code, const int* dst, const float* grad, float clone_dt,
                     const float* normals, int n_keep, int n_clone, int n_split, int scale_activation,
                     float* out_pos, float* out_rgb, float* out_opa, float* out_quat, float* out_scale,
                     gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Next-row widening (SURVEY.md §8 f-3): the training loss of reference train.py:99-107 on the device,
 * forward and backward in two kernels, producing the image gradient in the layout
 * gs_render_backward_final consumes.  image / grad_image: [height, width, 3] float32; target: same
 * shape, float32 or float16 (`target_is_half`; reference `ground_truth` is float16, splatter.py:478).
 *   L1   = mean |image - target|                                             (train.py:99)
 *   SSIM = torchmetrics StructuralSimilarityIndexMeasure(data_range=1.0): 11x11 Gaussian window,
 *          sigma 1.5, k1 0.01, k2 0.03, mean over the pixels whose window is inside the image and
 *          over channels                                                      (train.py:72,101-104)
 *   out3 (device) = { w_l1 * L1 + w_ssim * SSIM + bias,  L1,  SSIM }
 *   grad_image (nullable) = d out3[0] / d image.
 * train.py:107's loss (1 - w) l1 + w (1 - ssim) is w_l1 = 1 - w, w_ssim = -w, bias = w.
 * height and width must exceed 10.  No allocation, no synchronisation. */
size_t gs_loss_workspace_bytes(int height, int width);
int gs_loss_l1_ssim(const float* image, const void* target, int target_is_half, int height, int width,
                    float w_l1, float w_ssim, float bias, float* grad_image, float* out3, void* workspace,
                    size_t workspace_bytes, gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Multi-GPU exchange step (SURVEY.md §8e; new - the reference is single-GPU): in-place SUM of
 * the flat gradient bucket across `world` GPUs of one NVSwitch domain through an NVLS multicast
 * mapping.  `multicast_ptr` is the multicast address of a symmetric buffer holding each rank's
 * n_floats (multiple of 4) gradients at the same offset; rank r reduces and re-broadcasts slice r
 * (multimem.ld_reduce + multimem.st).  The caller orders it between two cross-rank barriers
 * (all buckets written before; all slices visible after).  No synchronisation inside. */
int gs_allreduce_multimem_f32(void* multicast_ptr, long long n_floats, int rank, int world,
                              gs_stream_t stream);

/* The same exchange over plain peer mappings (no multicast needed): `peer_ptrs` is a HOST array
 * of `world` (2, 4 or 8) device pointers, entry p = rank p's copy of the bucket as mapped into
 * this process (entry `rank` = the local copy).  Rank r sums slice r over all copies and stores
 * the sum into all of them.  Same barrier contract as above. */
#define GS_MAX_PEERS 8
int gs_allreduce_p2p_f32(void* const* peer_ptrs, long long n_floats, int rank, int world,
                         gs_stream_t stream);

/* Exchange fused into the backward ("push"): the flat bucket is cut into `world` slices of `per`
 * floats (multiple of 4; world * per >= bucket length, < 2^32); rank r owns slice r.  While a
 * context has a push configuration, gs_render_backward[_final] stores every gradient float that
 * belongs to ANOTHER rank's slice straight into slot `rank` of that owner's staging buffer
 * (staging[p] = rank p's [world][per] float buffer as mapped into this process) from inside the
 * projection-backward kernel, and only its own slice into `bucket` - the reduce half of the
 * exchange overlaps the kernel.  The five gradient pointers of the backward call must lie inside
 * [bucket, bucket + world * per).  gs_allreduce_push_finish_f32 (after a cross-rank barrier)
 * completes it: rank r sums its own slice with the world-1 pushed contributions and stores the sum
 * into every rank's bucket (`peer_buckets`: host array of `world` device pointers); a second
 * barrier makes all slices visible.  world must be 2, 4 or 8.  NULL clears the configuration. */
typedef struct gs_grad_push {
  int world, rank;
  long long per;
  float* bucket;
  float* staging[GS_MAX_PEERS];
} gs_grad_push;
int gs_ctx_set_grad_push(gs_ctx* ctx, const gs_grad_push* push);
int gs_allreduce_push_finish_f32(void* const* peer_buckets, const float* staging_local, long long n_floats,
                                 long long per, int rank, int world, gs_stream_t stream);
/* The same second half with the broadcast done by the NVSwitch: the sum of rank r's slice is written once
 * through `bucket_multicast` (the NVLS multicast address of the symmetric bucket; `bucket_local` is this
 * rank's own mapping of it) with multimem.st and lands in all `world` buckets. */
int gs_allreduce_push_finish_mc_f32(void* bucket_multicast, const float* bucket_local, const float* staging_local,
                                    long long n_floats, long long per, int rank, int world, gs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GS_B200_H */
