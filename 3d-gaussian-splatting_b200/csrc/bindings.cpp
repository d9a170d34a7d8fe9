// torch / pybind11 shim: the Python module `gaussian` with the exact symbol surface of the
// reference's extension (reference src/bindings.cpp:21-50: 12 functions + classes Tiles and
// Gaussian3ds), so the reference's renderer.py / splatter.py import and run unchanged.
// This is the ONLY libtorch-dependent translation unit; every function validates its tensors
// (the reference does not — SURVEY.md §8b) and forwards raw pointers + the CURRENT CUDA stream
// to the C ABI of libgs_b200.so (include/gs_b200.h).  Additive: class `RenderContext`
// (fused frame path) used by our splatter.py.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDACachingAllocator.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <string>
#include <vector>

#include "../../include/gs_b200.h"

namespace gsb200 {

#define GS_CHECK_F32(x)                                                                         \
  TORCH_CHECK((x).is_cuda(), #x " must be a CUDA tensor");                                      \
  TORCH_CHECK((x).is_contiguous(), #x " must be contiguous");                                   \
  TORCH_CHECK((x).scalar_type() == at::kFloat, #x " must be float32")
#define GS_CHECK_I32(x)                                                                         \
  TORCH_CHECK((x).is_cuda(), #x " must be a CUDA tensor");                                      \
  TORCH_CHECK((x).is_contiguous(), #x " must be contiguous");                                   \
  TORCH_CHECK((x).scalar_type() == at::kInt, #x " must be int32")
#define GS_CHECK_I64(x)                                                                         \
  TORCH_CHECK((x).is_cuda(), #x " must be a CUDA tensor");                                      \
  TORCH_CHECK((x).is_contiguous(), #x " must be contiguous");                                   \
  TORCH_CHECK((x).scalar_type() == at::kLong, #x " must be int64")

static inline void check_rc(int rc, const char* fn) {
  TORCH_CHECK(rc == 0, fn, " failed (", rc, "): ", gs_last_error());
}
static inline gs_stream_t cur_stream() { return (gs_stream_t)at::cuda::getCurrentCUDAStream().stream(); }
static inline const float* fp(const torch::Tensor& t) { return t.data_ptr<float>(); }
static inline float* fpm(torch::Tensor& t) { return t.data_ptr<float>(); }

// Same attribute names as reference common.hpp:36-74; distinct C++ types so both modules can
// live in one interpreter during parity tests.
struct TilesPy {
  torch::Tensor top, bottom, left, right;
};
struct Gaussian3dsPy {
  torch::Tensor pos, rgb, opa, quat, scale, cov;
};

void culling(torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor) {
  // reference gaussian.cu:6-8 is a stub that prints a string; nothing calls it.
}

void world2camera(torch::Tensor pos, torch::Tensor rot, torch::Tensor trans, torch::Tensor res) {
  GS_CHECK_F32(pos); GS_CHECK_F32(rot); GS_CHECK_F32(trans); GS_CHECK_F32(res);
  TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3 && res.sizes() == pos.sizes() && rot.numel() == 9 && trans.numel() == 3,
              "world2camera: bad shapes");
  c10::cuda::CUDAGuard guard(pos.device());
  check_rc(gs_w2c_fwd(fp(pos), fp(rot), fp(trans), (int)pos.size(0), fpm(res), cur_stream()), "world2camera");
}

void world2camera_backward(torch::Tensor grad_out, torch::Tensor rot, torch::Tensor grad_inp) {
  GS_CHECK_F32(grad_out); GS_CHECK_F32(rot); GS_CHECK_F32(grad_inp);
  TORCH_CHECK(grad_out.dim() == 2 && grad_out.size(1) == 3 && grad_inp.sizes() == grad_out.sizes() && rot.numel() == 9,
              "world2camera_backward: bad shapes");
  c10::cuda::CUDAGuard guard(grad_out.device());
  check_rc(gs_w2c_bwd(fp(grad_out), fp(rot), (int)grad_out.size(0), fpm(grad_inp), cur_stream()),
           "world2camera_backward");
}

void jacobian(torch::Tensor pos_camera_space, torch::Tensor jac) {
  GS_CHECK_F32(pos_camera_space); GS_CHECK_F32(jac);
  TORCH_CHECK(pos_camera_space.dim() == 2 && pos_camera_space.size(1) == 3 &&
                  jac.numel() == pos_camera_space.size(0) * 9, "jacobian: bad shapes");
  c10::cuda::CUDAGuard guard(jac.device());
  check_rc(gs_jacobian(fp(pos_camera_space), (int)pos_camera_space.size(0), fpm(jac), cur_stream()), "jacobian");
}

void calc_tile_list(Gaussian3dsPy& g, TilesPy& tiles, torch::Tensor tile_n_point, torch::Tensor tile_gaussian_list,
                    float thresh, int method, float tile_length_x, float tile_length_y, int n_tiles_x, int n_tiles_y,
                    float leftmost, float topmost) {
  GS_CHECK_F32(g.pos); GS_CHECK_I32(tile_n_point); GS_CHECK_I32(tile_gaussian_list);
  TORCH_CHECK(g.pos.dim() == 2 && g.pos.size(1) == 3, "calc_tile_list: pos must be [n,3]");
  TORCH_CHECK(tile_gaussian_list.dim() == 2 && tile_gaussian_list.size(0) == tile_n_point.size(0),
              "calc_tile_list: tile_gaussian_list must be [n_tiles, max_points]");
  TORCH_CHECK(method >= 0 && method <= 2, "calc_tile_list: method must be 0, 1 or 2");
  int n = (int)g.pos.size(0);
  int n_tiles = (int)tile_n_point.size(0);
  const float *top = nullptr, *bottom = nullptr, *left = nullptr, *right = nullptr, *cov = nullptr;
  if (method != 0) {
    GS_CHECK_F32(g.cov);
    TORCH_CHECK(g.cov.numel() == (int64_t)n * 4, "calc_tile_list: cov must be [n,2,2]");
    cov = fp(g.cov);
  }
  if (method != 2) {
    GS_CHECK_F32(tiles.top); GS_CHECK_F32(tiles.bottom); GS_CHECK_F32(tiles.left); GS_CHECK_F32(tiles.right);
    TORCH_CHECK(tiles.top.numel() == n_tiles && tiles.bottom.numel() == n_tiles && tiles.left.numel() == n_tiles &&
                    tiles.right.numel() == n_tiles, "calc_tile_list: tile bounds must have n_tiles entries");
    top = fp(tiles.top); bottom = fp(tiles.bottom); left = fp(tiles.left); right = fp(tiles.right);
  } else {
    TORCH_CHECK((int64_t)n_tiles_x * n_tiles_y == n_tiles, "calc_tile_list: n_tiles_x*n_tiles_y != len(tile_n_point)");
  }
  c10::cuda::CUDAGuard guard(g.pos.device());
  check_rc(gs_tile_list(fp(g.pos), cov, n, top, bottom, left, right, n_tiles, tile_n_point.data_ptr<int>(),
                        tile_gaussian_list.data_ptr<int>(), (int)tile_gaussian_list.size(1), thresh, method,
                        tile_length_x, tile_length_y, n_tiles_x, n_tiles_y, leftmost, topmost, cur_stream()),
           "calc_tile_list");
}

void gather_gaussians(torch::Tensor tile_n_point_accum, torch::Tensor tile_gaussian_list, torch::Tensor gathered_list,
                      torch::Tensor tile_ids_for_points, int max_points_for_tile) {
  GS_CHECK_I32(tile_n_point_accum); GS_CHECK_I32(tile_gaussian_list); GS_CHECK_I32(gathered_list);
  GS_CHECK_I32(tile_ids_for_points);
  TORCH_CHECK(tile_gaussian_list.dim() == 2 && tile_n_point_accum.numel() == tile_gaussian_list.size(0) + 1,
              "gather_gaussians: bad shapes");
  TORCH_CHECK(gathered_list.numel() == tile_ids_for_points.numel(), "gather_gaussians: output sizes differ");
  c10::cuda::CUDAGuard guard(gathered_list.device());
  check_rc(gs_gather(tile_n_point_accum.data_ptr<int>(), tile_gaussian_list.data_ptr<int>(),
                     (int)tile_gaussian_list.size(0), (int)tile_gaussian_list.size(1), max_points_for_tile,
                     gathered_list.data_ptr<int>(), tile_ids_for_points.data_ptr<int>(), cur_stream()),
           "gather_gaussians");
}

static void check_draw_inputs(const torch::Tensor& pos, const torch::Tensor& rgb, const torch::Tensor& opa,
                              const torch::Tensor& cov, const torch::Tensor& accum, const torch::Tensor& img,
                              bool use_sh_coeff) {
  GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(cov); GS_CHECK_I32(accum); GS_CHECK_F32(img);
  int64_t m = pos.size(0);
  TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3, "draw: pos must be [m,3]");
  if (use_sh_coeff) {   // 27 = degree 2 (the reference's layout [c*9+k]); 48 = degree 3 extension [c*16+k]
    TORCH_CHECK(rgb.dim() == 2 && rgb.size(0) == m && (rgb.size(1) == 27 || rgb.size(1) == 48),
                "draw: SH rgb must be [m,27] or [m,48]");
  } else {
    TORCH_CHECK(rgb.numel() == m * 3, "draw: rgb must be [m,3]");
  }
  TORCH_CHECK(opa.numel() == m && cov.numel() == m * 4, "draw: opa must be [m], cov [m,2,2]");
  TORCH_CHECK(img.dim() == 3 && img.size(2) == 3 && img.size(0) % 16 == 0 && img.size(1) % 16 == 0,
              "draw: image must be [Hp,Wp,3] with Hp,Wp multiples of 16");
  TORCH_CHECK(accum.numel() == (img.size(0) / 16) * (img.size(1) / 16) + 1, "draw: tile_n_point_accum must be [T+1]");
}

void draw(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor cov, torch::Tensor tile_n_point_accum,
          torch::Tensor res, float focal_x, float focal_y, bool weight_normalize, bool sigmoid, bool fast,
          torch::Tensor rays_o, torch::Tensor lefttop_pos, torch::Tensor vec_dx, torch::Tensor vec_dy,
          bool use_sh_coeff) {
  (void)fast;   // both exp flavours of the reference are within 2 ulp of ex2.approx; one code path
  check_draw_inputs(pos, rgb, opa, cov, tile_n_point_accum, res, use_sh_coeff);
  c10::cuda::CUDAGuard guard(pos.device());
  int m = (int)pos.size(0), d = use_sh_coeff ? (int)rgb.size(1) : 3;
  auto ws = torch::empty({(int64_t)gs_draw_workspace_bytes(m, d)}, pos.options().dtype(at::kByte));
  const float *ro = nullptr, *lt = nullptr, *dx = nullptr, *dy = nullptr;
  if (use_sh_coeff) {
    GS_CHECK_F32(rays_o); GS_CHECK_F32(lefttop_pos); GS_CHECK_F32(vec_dx); GS_CHECK_F32(vec_dy);
    ro = fp(rays_o); lt = fp(lefttop_pos); dx = fp(vec_dx); dy = fp(vec_dy);
  }
  check_rc(gs_draw_fwd(fp(pos), fp(rgb), fp(opa), fp(cov), tile_n_point_accum.data_ptr<int>(), m, d, (int)res.size(1),
                       (int)res.size(0), focal_x, focal_y, weight_normalize, sigmoid, ro, lt, dx, dy, fpm(res),
                       ws.data_ptr(), (size_t)ws.numel(), cur_stream()),
           "draw");
}

void draw_backward(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor cov,
                   torch::Tensor tile_n_point_accum, torch::Tensor output, torch::Tensor grad_output,
                   torch::Tensor grad_pos, torch::Tensor grad_rgb, torch::Tensor grad_opa, torch::Tensor grad_cov,
                   float focal_x, float focal_y, bool weight_normalize, bool sigmoid, bool fast, torch::Tensor rays_o,
                   torch::Tensor lefttop_pos, torch::Tensor vec_dx, torch::Tensor vec_dy, bool use_sh_coeff) {
  (void)fast;
  check_draw_inputs(pos, rgb, opa, cov, tile_n_point_accum, output, use_sh_coeff);
  GS_CHECK_F32(grad_pos); GS_CHECK_F32(grad_rgb); GS_CHECK_F32(grad_opa); GS_CHECK_F32(grad_cov);
  TORCH_CHECK(grad_output.is_cuda() && grad_output.scalar_type() == at::kFloat, "grad_output must be a float32 CUDA tensor");
  TORCH_CHECK(grad_output.sizes() == output.sizes(), "draw_backward: grad_output shape != output shape");
  TORCH_CHECK(grad_pos.sizes() == pos.sizes() && grad_rgb.numel() == rgb.numel() && grad_opa.numel() == opa.numel() &&
                  grad_cov.numel() == cov.numel(), "draw_backward: gradient buffers must match their inputs");
  c10::cuda::CUDAGuard guard(pos.device());
  auto go = grad_output.contiguous();   // autograd may hand us a strided view (crop backward)
  int m = (int)pos.size(0), d = use_sh_coeff ? (int)rgb.size(1) : 3;
  auto ws = torch::empty({(int64_t)gs_draw_workspace_bytes(m, d)}, pos.options().dtype(at::kByte));
  const float *ro = nullptr, *lt = nullptr, *dx = nullptr, *dy = nullptr;
  if (use_sh_coeff) {
    GS_CHECK_F32(rays_o); GS_CHECK_F32(lefttop_pos); GS_CHECK_F32(vec_dx); GS_CHECK_F32(vec_dy);
    ro = fp(rays_o); lt = fp(lefttop_pos); dx = fp(vec_dx); dy = fp(vec_dy);
  }
  check_rc(gs_draw_bwd(fp(pos), fp(rgb), fp(opa), fp(cov), tile_n_point_accum.data_ptr<int>(), m, d,
                       (int)output.size(1), (int)output.size(0), focal_x, focal_y, weight_normalize, sigmoid, ro, lt,
                       dx, dy, fp(output), fp(go), fpm(grad_pos), fpm(grad_rgb), fpm(grad_opa), fpm(grad_cov),
                       ws.data_ptr(), (size_t)ws.numel(), cur_stream()),
           "draw_backward");
}

void global_culling(torch::Tensor pos, torch::Tensor quat, torch::Tensor scale, torch::Tensor current_rot,
                    torch::Tensor current_tran, torch::Tensor res_pos, torch::Tensor res_cov,
                    torch::Tensor culling_mask, float near, float half_width, float half_height) {
  GS_CHECK_F32(pos); GS_CHECK_F32(quat); GS_CHECK_F32(scale); GS_CHECK_F32(current_rot); GS_CHECK_F32(current_tran);
  GS_CHECK_F32(res_pos); GS_CHECK_F32(res_cov); GS_CHECK_I64(culling_mask);
  int64_t n = pos.size(0);
  TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3 && quat.numel() == n * 4 && scale.numel() == n * 3 &&
                  current_rot.numel() == 9 && current_tran.numel() == 3 && res_pos.numel() == n * 3 &&
                  res_cov.numel() == n * 4 && culling_mask.numel() == n, "global_culling: bad shapes");
  c10::cuda::CUDAGuard guard(pos.device());
  check_rc(gs_project_fwd(fp(pos), fp(quat), fp(scale), fp(current_rot), fp(current_tran), (int)n, near, half_width,
                          half_height, fpm(res_pos), fpm(res_cov), culling_mask.data_ptr<int64_t>(), cur_stream()),
           "global_culling");
}

void global_culling_backward(torch::Tensor pos, torch::Tensor quat, torch::Tensor scale, torch::Tensor current_rot,
                             torch::Tensor current_tran, torch::Tensor gradout_pos, torch::Tensor gradout_cov,
                             torch::Tensor culling_mask, torch::Tensor gradinput_pos, torch::Tensor gradinput_quat,
                             torch::Tensor gradinput_scale) {
  GS_CHECK_F32(pos); GS_CHECK_F32(quat); GS_CHECK_F32(scale); GS_CHECK_F32(current_rot); GS_CHECK_F32(current_tran);
  GS_CHECK_I64(culling_mask); GS_CHECK_F32(gradinput_pos); GS_CHECK_F32(gradinput_quat); GS_CHECK_F32(gradinput_scale);
  int64_t n = pos.size(0);
  TORCH_CHECK(gradout_pos.is_cuda() && gradout_cov.is_cuda() && gradout_pos.scalar_type() == at::kFloat &&
                  gradout_cov.scalar_type() == at::kFloat, "global_culling_backward: gradients must be float32 CUDA");
  TORCH_CHECK(gradout_pos.numel() == n * 3 && gradout_cov.numel() == n * 4 && culling_mask.numel() == n &&
                  gradinput_pos.numel() == n * 3 && gradinput_quat.numel() == n * 4 && gradinput_scale.numel() == n * 3,
              "global_culling_backward: bad shapes");
  c10::cuda::CUDAGuard guard(pos.device());
  auto gp = gradout_pos.contiguous();
  auto gc = gradout_cov.contiguous();
  check_rc(gs_project_bwd(fp(pos), fp(quat), fp(scale), fp(current_rot), fp(current_tran), fp(gp), fp(gc),
                          culling_mask.data_ptr<int64_t>(), (int)n, fpm(gradinput_pos), fpm(gradinput_quat),
                          fpm(gradinput_scale), cur_stream()),
           "global_culling_backward");
}

// ---- additive: fused frame path ----------------------------------------------------------
struct RenderContext {
  gs_ctx* ctx = nullptr;
  int device = -1;
  // The context holds the intermediate state of ONE forward.  Every forward gets an id; a
  // backward that names another id is refused instead of silently using the wrong frame.
  int64_t frame = 0;
  int64_t frame_id() const { return frame; }
  void check_frame(int64_t expected, const char* fn) const {
    TORCH_CHECK(expected < 0 || expected == frame, fn, ": this RenderContext has rendered another frame (id ", frame,
                ") since the forward being differentiated (id ", expected,
                "); run backward before the next forward, or use one RenderContext / Splatter per in-flight frame");
  }
  static void* torch_alloc(size_t bytes, void*, gs_stream_t stream) {
    try {
      return c10::cuda::CUDACachingAllocator::raw_alloc_with_stream(bytes, (cudaStream_t)stream);
    } catch (...) {
      return nullptr;
    }
  }
  static void torch_free(void* p, void*) { c10::cuda::CUDACachingAllocator::raw_delete(p); }
  RenderContext() {
    check_rc(gs_ctx_create(&ctx), "gs_ctx_create");
    cudaGetDevice(&device);
    // workspaces from PyTorch's stream-ordered caching allocator: growth needs no device synchronisation
    check_rc(gs_ctx_set_allocator(ctx, &torch_alloc, &torch_free, nullptr), "gs_ctx_set_allocator");
  }
  ~RenderContext() { gs_ctx_destroy(ctx); }
  RenderContext(const RenderContext&) = delete;
  RenderContext& operator=(const RenderContext&) = delete;

  static gs_camera make_cam(int width, int height, float fx, float fy, const torch::Tensor& rot,
                            const torch::Tensor& tran, float near, float thresh) {
    TORCH_CHECK(!rot.is_cuda() && !tran.is_cuda(), "RenderContext: rot/tran must be CPU tensors (camera is host data)");
    auto r = rot.to(at::kFloat).contiguous();
    auto t = tran.to(at::kFloat).contiguous();
    TORCH_CHECK(r.numel() == 9 && t.numel() == 3, "RenderContext: rot must be 3x3, tran 3");
    gs_camera cam{};
    cam.width = width;
    cam.height = height;
    cam.focal_x = fx;
    cam.focal_y = fy;
    memcpy(cam.rot, r.data_ptr<float>(), sizeof(cam.rot));
    memcpy(cam.tran, t.data_ptr<float>(), sizeof(cam.tran));
    cam.near_plane = near;
    cam.tile_thresh = thresh;
    return cam;
  }

  // returns (image[Hp,Wp,3], culling_mask[n] int64)
  std::tuple<torch::Tensor, torch::Tensor> forward(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa,
                                                   torch::Tensor quat, torch::Tensor scale, int width, int height,
                                                   float fx, float fy, torch::Tensor rot, torch::Tensor tran,
                                                   float near, float thresh, int scale_activation) {
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    int64_t n = pos.size(0);
    TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3 && opa.numel() == n && quat.numel() == n * 4 &&
                    scale.numel() == n * 3 && rgb.dim() == 2 && rgb.size(0) == n && n < (int64_t(1) << 31),
                "RenderContext.forward: bad shapes");
    TORCH_CHECK(pos.device().index() == device, "RenderContext was created on another device");
    c10::cuda::CUDAGuard guard(pos.device());
    gs_camera cam = make_cam(width, height, fx, fy, rot, tran, near, thresh);
    int wp = (width + 15) / 16 * 16, hp = (height + 15) / 16 * 16;
    auto image = torch::empty({hp, wp, 3}, pos.options());
    auto mask = torch::empty({n}, pos.options().dtype(at::kLong));
    check_rc(gs_render_forward(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), (int)n, (int)rgb.size(1),
                               scale_activation, &cam, fpm(image), mask.data_ptr<int64_t>(), cur_stream()),
             "gs_render_forward");
    ++frame;
    return {image, mask};
  }

  std::vector<torch::Tensor> backward(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat,
                                      torch::Tensor scale, torch::Tensor image, torch::Tensor grad_image) {
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    GS_CHECK_F32(image);
    TORCH_CHECK(grad_image.is_cuda() && grad_image.scalar_type() == at::kFloat && grad_image.sizes() == image.sizes(),
                "RenderContext.backward: grad_image must match image");
    c10::cuda::CUDAGuard guard(pos.device());
    auto gi = grad_image.contiguous();
    auto g_pos = torch::empty_like(pos), g_rgb = torch::empty_like(rgb), g_opa = torch::empty_like(opa),
         g_quat = torch::empty_like(quat), g_scale = torch::empty_like(scale);
    check_rc(gs_render_backward(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), fp(image), fp(gi), fpm(g_pos),
                                fpm(g_rgb), fpm(g_opa), fpm(g_quat), fpm(g_scale), cur_stream()),
             "gs_render_backward");
    return {g_pos, g_rgb, g_opa, g_quat, g_scale};
  }

  // data-parallel gradient push (gs_grad_push): pointers as integers (symmetric-memory mappings)
  void set_grad_push(int64_t bucket_ptr, std::vector<int64_t> staging_ptrs, int64_t per, int rank) {
    gs_grad_push p{};
    p.world = (int)staging_ptrs.size();
    TORCH_CHECK(p.world <= GS_MAX_PEERS, "set_grad_push: at most ", GS_MAX_PEERS, " ranks");
    p.rank = rank;
    p.per = per;
    p.bucket = reinterpret_cast<float*>(static_cast<uintptr_t>(bucket_ptr));
    for (int k = 0; k < p.world; ++k) p.staging[k] = reinterpret_cast<float*>(static_cast<uintptr_t>(staging_ptrs[k]));
    check_rc(gs_ctx_set_grad_push(ctx, &p), "gs_ctx_set_grad_push");
  }
  void clear_grad_push() { check_rc(gs_ctx_set_grad_push(ctx, nullptr), "gs_ctx_set_grad_push"); }

  // camera pose gradient (gs_ctx_set_camera_grad): every backward on this context also overwrites grad_cam[12] =
  // (d/d rot row-major, d/d tran) while it is set; None clears it.  The tensor must outlive its use.
  void set_camera_grad(c10::optional<torch::Tensor> grad_cam) {
    float* p = nullptr;
    if (grad_cam) {
      const torch::Tensor& g = *grad_cam;
      GS_CHECK_F32(g);
      TORCH_CHECK(g.numel() == 12, "set_camera_grad: grad_cam must have 12 elements (9 rot + 3 tran)");
      TORCH_CHECK(g.device().index() == device, "set_camera_grad: grad_cam is on another device than the RenderContext");
      p = g.data_ptr<float>();
    }
    check_rc(gs_ctx_set_camera_grad(ctx, p), "gs_ctx_set_camera_grad");
  }

  void set_timing(bool on) { check_rc(gs_ctx_set_timing(ctx, on ? 1 : 0), "gs_ctx_set_timing"); }
  std::vector<float> stage_ms() {
    std::vector<float> v(GS_N_STAGES, -1.f);
    check_rc(gs_frame_stage_ms(ctx, v.data(), cur_stream()), "gs_frame_stage_ms");
    return v;
  }

  // fused clamp + centre crop: returns (final[H,W,3], raw padded[Hp,Wp,3], mask)
  std::tuple<torch::Tensor, torch::Tensor, torch::Tensor> forward_final(
      torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat, torch::Tensor scale, int width,
      int height, float fx, float fy, torch::Tensor rot, torch::Tensor tran, float near, float thresh,
      int scale_activation) {
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    int64_t n = pos.size(0);
    TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3 && opa.numel() == n && quat.numel() == n * 4 &&
                    scale.numel() == n * 3 && rgb.dim() == 2 && rgb.size(0) == n && n < (int64_t(1) << 31),
                "RenderContext.forward: bad shapes");
    TORCH_CHECK(pos.device().index() == device, "RenderContext was created on another device");
    c10::cuda::CUDAGuard guard(pos.device());
    gs_camera cam = make_cam(width, height, fx, fy, rot, tran, near, thresh);
    int wp = (width + 15) / 16 * 16, hp = (height + 15) / 16 * 16;
    auto raw = torch::empty({hp, wp, 3}, pos.options());
    auto fin = torch::empty({height, width, 3}, pos.options());
    auto mask = torch::empty({n}, pos.options().dtype(at::kLong));
    check_rc(gs_render_forward_final(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), (int)n, (int)rgb.size(1),
                                     scale_activation, &cam, fpm(raw), fpm(fin), mask.data_ptr<int64_t>(),
                                     cur_stream()),
             "gs_render_forward_final");
    ++frame;
    return {fin, raw, mask};
  }

  void backward_final_into(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat,
                           torch::Tensor scale, torch::Tensor raw, torch::Tensor grad_final, torch::Tensor g_pos,
                           torch::Tensor g_rgb, torch::Tensor g_opa, torch::Tensor g_quat, torch::Tensor g_scale,
                           int64_t expected_frame) {
    check_frame(expected_frame, "RenderContext.backward_final_into");
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    GS_CHECK_F32(raw); GS_CHECK_F32(g_pos); GS_CHECK_F32(g_rgb); GS_CHECK_F32(g_opa); GS_CHECK_F32(g_quat);
    GS_CHECK_F32(g_scale);
    TORCH_CHECK(grad_final.is_cuda() && grad_final.scalar_type() == at::kFloat && grad_final.dim() == 3 &&
                    grad_final.size(2) == 3, "RenderContext.backward_final_into: grad_final must be [H,W,3] float32");
    TORCH_CHECK(g_pos.numel() == pos.numel() && g_rgb.numel() == rgb.numel() && g_opa.numel() == opa.numel() &&
                    g_quat.numel() == quat.numel() && g_scale.numel() == scale.numel(),
                "RenderContext.backward_final_into: gradient buffers must match their parameters");
    TORCH_CHECK(reinterpret_cast<uintptr_t>(g_quat.data_ptr()) % 16 == 0, "grad_quat must be 16-byte aligned");
    c10::cuda::CUDAGuard guard(pos.device());
    auto gf = grad_final.contiguous();
    check_rc(gs_render_backward_final(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), fp(raw), fp(gf), fpm(g_pos),
                                      fpm(g_rgb), fpm(g_opa), fpm(g_quat), fpm(g_scale), cur_stream()),
             "gs_render_backward_final");
  }

  void backward_into(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat, torch::Tensor scale,
                     torch::Tensor image, torch::Tensor grad_image, torch::Tensor g_pos, torch::Tensor g_rgb,
                     torch::Tensor g_opa, torch::Tensor g_quat, torch::Tensor g_scale, int64_t expected_frame) {
    check_frame(expected_frame, "RenderContext.backward_into");
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    GS_CHECK_F32(image); GS_CHECK_F32(g_pos); GS_CHECK_F32(g_rgb); GS_CHECK_F32(g_opa); GS_CHECK_F32(g_quat);
    GS_CHECK_F32(g_scale);
    TORCH_CHECK(grad_image.is_cuda() && grad_image.scalar_type() == at::kFloat && grad_image.sizes() == image.sizes(),
                "RenderContext.backward_into: grad_image must match image");
    TORCH_CHECK(g_pos.numel() == pos.numel() && g_rgb.numel() == rgb.numel() && g_opa.numel() == opa.numel() &&
                    g_quat.numel() == quat.numel() && g_scale.numel() == scale.numel(),
                "RenderContext.backward_into: gradient buffers must match their parameters");
    TORCH_CHECK(reinterpret_cast<uintptr_t>(g_quat.data_ptr()) % 16 == 0, "grad_quat must be 16-byte aligned");
    c10::cuda::CUDAGuard guard(pos.device());
    auto gi = grad_image.contiguous();
    check_rc(gs_render_backward(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), fp(image), fp(gi), fpm(g_pos),
                                fpm(g_rgb), fpm(g_opa), fpm(g_quat), fpm(g_scale), cur_stream()),
             "gs_render_backward");
  }

  // depth / alpha maps + background (gs_render_forward_maps): returns [image, depth, alpha, image_raw, depth_raw,
  // alpha_raw, mask]; with final = false the first three are the raw padded planes themselves
  std::vector<torch::Tensor> forward_maps(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat,
                                          torch::Tensor scale, int width, int height, float fx, float fy,
                                          torch::Tensor rot, torch::Tensor tran, float near, float thresh,
                                          int scale_activation, c10::optional<std::vector<double>> background,
                                          bool final_layout) {
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    int64_t n = pos.size(0);
    TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3 && opa.numel() == n && quat.numel() == n * 4 &&
                    scale.numel() == n * 3 && rgb.dim() == 2 && rgb.size(0) == n && n < (int64_t(1) << 31),
                "RenderContext.forward_maps: bad shapes");
    TORCH_CHECK(pos.device().index() == device, "RenderContext was created on another device");
    float bg[3] = {0.f, 0.f, 0.f};
    if (background) {
      TORCH_CHECK(background->size() == 3, "RenderContext.forward_maps: background must have 3 values (r, g, b)");
      for (int k = 0; k < 3; ++k) bg[k] = (float)(*background)[k];
    }
    c10::cuda::CUDAGuard guard(pos.device());
    gs_camera cam = make_cam(width, height, fx, fy, rot, tran, near, thresh);
    int wp = (width + 15) / 16 * 16, hp = (height + 15) / 16 * 16;
    auto raw = torch::empty({hp, wp, 3}, pos.options());
    auto dpad = torch::empty({hp, wp}, pos.options());
    auto araw = torch::empty({hp, wp}, pos.options());
    torch::Tensor fin = raw, dfin = dpad, afin = araw;
    if (final_layout) {
      fin = torch::empty({height, width, 3}, pos.options());
      dfin = torch::empty({height, width}, pos.options());
      afin = torch::empty({height, width}, pos.options());
    }
    auto mask = torch::empty({n}, pos.options().dtype(at::kLong));
    check_rc(gs_render_forward_maps(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), (int)n, (int)rgb.size(1),
                                    scale_activation, &cam, bg, fpm(raw), fpm(dpad), fpm(araw),
                                    final_layout ? fpm(fin) : nullptr, final_layout ? fpm(dfin) : nullptr,
                                    final_layout ? fpm(afin) : nullptr, mask.data_ptr<int64_t>(), cur_stream()),
             "gs_render_forward_maps");
    ++frame;
    return {fin, dfin, afin, raw, dpad, araw, mask};
  }

  void backward_maps_into(torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat,
                          torch::Tensor scale, torch::Tensor raw, torch::Tensor depth_raw, torch::Tensor alpha_raw,
                          torch::Tensor grad_image, torch::Tensor grad_depth, torch::Tensor grad_alpha, bool grad_is_final,
                          torch::Tensor g_pos, torch::Tensor g_rgb, torch::Tensor g_opa, torch::Tensor g_quat,
                          torch::Tensor g_scale, int64_t expected_frame) {
    check_frame(expected_frame, "RenderContext.backward_maps_into");
    GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale);
    GS_CHECK_F32(raw); GS_CHECK_F32(depth_raw); GS_CHECK_F32(alpha_raw);
    GS_CHECK_F32(g_pos); GS_CHECK_F32(g_rgb); GS_CHECK_F32(g_opa); GS_CHECK_F32(g_quat); GS_CHECK_F32(g_scale);
    TORCH_CHECK(raw.dim() == 3 && raw.size(2) == 3 && depth_raw.dim() == 2 && depth_raw.size(0) == raw.size(0) &&
                    depth_raw.size(1) == raw.size(1) && alpha_raw.sizes() == depth_raw.sizes(),
                "RenderContext.backward_maps_into: raw planes must be [Hp,Wp,3], [Hp,Wp], [Hp,Wp]");
    for (const torch::Tensor* t : {&grad_image, &grad_depth, &grad_alpha})
      TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kFloat,
                  "RenderContext.backward_maps_into: gradients must be float32 CUDA tensors");
    TORCH_CHECK(grad_image.dim() == 3 && grad_image.size(2) == 3 && grad_depth.dim() == 2 &&
                    grad_depth.size(0) == grad_image.size(0) && grad_depth.size(1) == grad_image.size(1) &&
                    grad_alpha.sizes() == grad_depth.sizes(),
                "RenderContext.backward_maps_into: gradients must be [H,W,3], [H,W], [H,W]");
    TORCH_CHECK(grad_is_final || grad_image.sizes() == raw.sizes(),
                "RenderContext.backward_maps_into: padded gradients must match the raw planes");
    TORCH_CHECK(g_pos.numel() == pos.numel() && g_rgb.numel() == rgb.numel() && g_opa.numel() == opa.numel() &&
                    g_quat.numel() == quat.numel() && g_scale.numel() == scale.numel(),
                "RenderContext.backward_maps_into: gradient buffers must match their parameters");
    TORCH_CHECK(reinterpret_cast<uintptr_t>(g_quat.data_ptr()) % 16 == 0, "grad_quat must be 16-byte aligned");
    c10::cuda::CUDAGuard guard(pos.device());
    auto gi = grad_image.contiguous(), gd = grad_depth.contiguous(), ga = grad_alpha.contiguous();
    check_rc(gs_render_backward_maps(ctx, fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), fp(raw), fp(depth_raw),
                                     fp(alpha_raw), fp(gi), fp(gd), fp(ga), grad_is_final ? 1 : 0, fpm(g_pos),
                                     fpm(g_rgb), fpm(g_opa), fpm(g_quat), fpm(g_scale), cur_stream()),
             "gs_render_backward_maps");
  }

  int64_t last_instances() { return (int64_t)gs_frame_instances(ctx); }

  py::dict stats() {
    gs_frame_info fi{};
    check_rc(gs_frame_stats(ctx, &fi, cur_stream()), "gs_frame_stats");
    py::dict d;
    d["n_gaussians"] = fi.n_gaussians;
    d["n_visible"] = fi.n_visible;
    d["n_instances"] = fi.n_instances;
    d["n_instances_eff"] = fi.n_instances_eff;
    d["width_padded"] = fi.width_padded;
    d["height_padded"] = fi.height_padded;
    d["n_tiles"] = fi.n_tiles;
    d["max_tile_count"] = fi.max_tile_count;
    d["n_instances_eff_bwd"] = fi.n_instances_eff_bwd;
    return d;
  }

  // (sorted gaussian ids [M] int32, tile_n_point_accum [T+1] int32) of the last forward
  std::tuple<torch::Tensor, torch::Tensor> sorted_instances() {
    gs_frame_info fi{};
    check_rc(gs_frame_stats(ctx, &fi, cur_stream()), "gs_frame_stats");
    auto opts = torch::TensorOptions().device(torch::kCUDA, device).dtype(at::kInt);
    auto idx = torch::empty({(int64_t)fi.n_instances}, opts);
    auto accum = torch::empty({(int64_t)fi.n_tiles + 1}, opts);
    check_rc(gs_frame_sorted(ctx, idx.data_ptr<int>(), fi.n_instances, accum.data_ptr<int>(), cur_stream()),
             "gs_frame_sorted");
    return {idx, accum};
  }

  // consumed instances per tile [T] int32 of the last forward (M_eff = sum)
  torch::Tensor tile_consumed() {
    gs_frame_info fi{};
    check_rc(gs_frame_stats(ctx, &fi, cur_stream()), "gs_frame_stats");
    auto out = torch::empty({(int64_t)fi.n_tiles}, torch::TensorOptions().device(torch::kCUDA, device).dtype(at::kInt));
    check_rc(gs_frame_tile_consumed(ctx, out.data_ptr<int>(), cur_stream()), "gs_frame_tile_consumed");
    return out;
  }
};

// fused Adam over flat buffers (SURVEY.md §8 f-2); seg_ends / lrs are small host lists
void adam_step(torch::Tensor param, torch::Tensor grad, torch::Tensor exp_avg, torch::Tensor exp_avg_sq,
               std::vector<int64_t> seg_ends, std::vector<double> lrs, double beta1, double beta2, double eps,
               int64_t step) {
  GS_CHECK_F32(param); GS_CHECK_F32(grad); GS_CHECK_F32(exp_avg); GS_CHECK_F32(exp_avg_sq);
  int64_t n = param.numel();
  TORCH_CHECK(grad.numel() == n && exp_avg.numel() == n && exp_avg_sq.numel() == n, "adam_step: size mismatch");
  TORCH_CHECK(seg_ends.size() == lrs.size() && !seg_ends.empty() && seg_ends.back() == n,
              "adam_step: segments must cover the flat buffer");
  for (auto* t : {&param, &grad, &exp_avg, &exp_avg_sq})
    TORCH_CHECK(reinterpret_cast<uintptr_t>(t->data_ptr()) % 16 == 0, "adam_step: buffers must be 16-byte aligned");
  std::vector<long long> ends(seg_ends.begin(), seg_ends.end());
  std::vector<float> lr(lrs.begin(), lrs.end());
  c10::cuda::CUDAGuard guard(param.device());
  check_rc(gs_adam_step(fpm(param), fp(grad), fpm(exp_avg), fpm(exp_avg_sq), n, ends.data(), lr.data(), (int)ends.size(),
                        (float)beta1, (float)beta2, (float)eps, (int)step, cur_stream()),
           "gs_adam_step");
}

// fused L1 + SSIM loss (SURVEY.md §8 f-3, reference train.py:99-107): returns (out3 = {total, l1, ssim}, grad_image)
std::tuple<torch::Tensor, torch::Tensor> loss_l1_ssim(torch::Tensor image, torch::Tensor target, double w_l1,
                                                      double w_ssim, double bias, bool want_grad) {
  GS_CHECK_F32(image);
  TORCH_CHECK(target.is_cuda() && target.is_contiguous() &&
                  (target.scalar_type() == at::kFloat || target.scalar_type() == at::kHalf),
              "loss_l1_ssim: target must be a contiguous float32 / float16 CUDA tensor");
  TORCH_CHECK(image.dim() == 3 && image.size(2) == 3 && target.sizes() == image.sizes(),
              "loss_l1_ssim: image and target must both be [H, W, 3]");
  TORCH_CHECK(image.size(0) > 10 && image.size(1) > 10, "loss_l1_ssim: the image must be larger than the 11x11 window");
  c10::cuda::CUDAGuard guard(image.device());
  const int h = (int)image.size(0), w = (int)image.size(1);
  auto ws = torch::empty({(int64_t)gs_loss_workspace_bytes(h, w)}, image.options().dtype(at::kByte));
  auto out3 = torch::empty({3}, image.options());
  torch::Tensor grad = want_grad ? torch::empty_like(image) : torch::Tensor();
  check_rc(gs_loss_l1_ssim(fp(image), target.data_ptr(), target.scalar_type() == at::kHalf ? 1 : 0, h, w, (float)w_l1,
                           (float)w_ssim, (float)bias, want_grad ? fpm(grad) : nullptr, fpm(out3), ws.data_ptr(),
                           (size_t)ws.numel(), cur_stream()),
           "gs_loss_l1_ssim");
  return {out3, grad};
}

// densification (SURVEY.md §8 f-2): returns the five new parameter tensors + (n_deleted, n_clone, n_split)
std::tuple<std::vector<torch::Tensor>, std::vector<int64_t>> densify(
    torch::Tensor pos, torch::Tensor rgb, torch::Tensor opa, torch::Tensor quat, torch::Tensor scale, torch::Tensor grad,
    int scale_activation, double opa_logit_min, double delete_thresh, double grad_thresh, bool grad_agg_max, double tau,
    bool use_clone, bool use_split, double clone_dt, c10::optional<at::Generator> gen) {
  GS_CHECK_F32(pos); GS_CHECK_F32(rgb); GS_CHECK_F32(opa); GS_CHECK_F32(quat); GS_CHECK_F32(scale); GS_CHECK_F32(grad);
  const int64_t n = pos.size(0);
  TORCH_CHECK(pos.dim() == 2 && pos.size(1) == 3 && rgb.dim() == 2 && rgb.size(0) == n && opa.numel() == n &&
                  quat.numel() == 4 * n && scale.numel() == 3 * n && grad.numel() == 3 * n && n < (int64_t(1) << 31),
              "densify: bad shapes");
  c10::cuda::CUDAGuard guard(pos.device());
  auto bopt = pos.options().dtype(at::kByte);
  auto code = torch::empty({n + 1}, bopt);
  auto dst = torch::empty({3, n + 1}, pos.options().dtype(at::kInt));
  auto ws = torch::empty({(int64_t)gs_densify_workspace_bytes((int)n)}, bopt);
  check_rc(gs_densify_plan(fp(opa), fp(scale), fp(grad), (int)n, scale_activation, (float)opa_logit_min,
                           (float)delete_thresh, (float)grad_thresh, grad_agg_max ? 1 : 0, (float)tau, use_clone ? 1 : 0,
                           use_split ? 1 : 0, code.data_ptr<uint8_t>(), dst.data_ptr<int>(), ws.data_ptr(),
                           (size_t)ws.numel(), cur_stream()),
           "gs_densify_plan");
  int64_t nk = n, nc = 0, nsp = 0;
  if (n > 0) {
    auto tot = dst.index({torch::indexing::Slice(), n}).cpu();        // the one host sync: sizes of the new arrays
    nk = tot[0].item<int>(); nc = tot[1].item<int>(); nsp = tot[2].item<int>();
  }
  const int64_t m = nk + nc + nsp;
  const int64_t d = rgb.size(1);
  auto z = torch::randn({2, nsp, 3}, gen, pos.options());              // torch's generator: identical on every DP rank
  std::vector<torch::Tensor> out = {torch::empty({m, 3}, pos.options()), torch::empty({m, d}, pos.options()),
                                    torch::empty({m}, pos.options()), torch::empty({m, 4}, pos.options()),
                                    torch::empty({m, 3}, pos.options())};
  check_rc(gs_densify_apply(fp(pos), fp(rgb), fp(opa), fp(quat), fp(scale), (int)n, (int)d, code.data_ptr<uint8_t>(),
                            dst.data_ptr<int>(), fp(grad), (float)clone_dt, fp(z), (int)nk, (int)nc, (int)nsp,
                            scale_activation, fpm(out[0]), fpm(out[1]), fpm(out[2]), fpm(out[3]), fpm(out[4]),
                            cur_stream()),
           "gs_densify_apply");
  return {out, {n - nk, nc, nsp}};
}

// NVLS in-place all-reduce of a symmetric flat buffer (multicast address as an integer)
void allreduce_multimem(int64_t multicast_ptr, int64_t n_floats, int rank, int world, int device) {
  c10::cuda::CUDAGuard guard(c10::Device(c10::kCUDA, (c10::DeviceIndex)device));
  check_rc(gs_allreduce_multimem_f32(reinterpret_cast<void*>(static_cast<uintptr_t>(multicast_ptr)), n_floats, rank,
                                     world, cur_stream()),
           "gs_allreduce_multimem_f32");
}

void allreduce_p2p(std::vector<int64_t> peer_ptrs, int64_t n_floats, int rank, int world, int device) {
  c10::cuda::CUDAGuard guard(c10::Device(c10::kCUDA, (c10::DeviceIndex)device));
  TORCH_CHECK((int)peer_ptrs.size() == world, "allreduce_p2p: need one pointer per rank");
  std::vector<void*> ptrs;
  for (int64_t p : peer_ptrs) ptrs.push_back(reinterpret_cast<void*>(static_cast<uintptr_t>(p)));
  check_rc(gs_allreduce_p2p_f32(ptrs.data(), n_floats, rank, world, cur_stream()), "gs_allreduce_p2p_f32");
}

void allreduce_push_finish(std::vector<int64_t> bucket_ptrs, int64_t staging_local, int64_t n_floats, int64_t per,
                           int rank, int world, int device) {
  c10::cuda::CUDAGuard guard(c10::Device(c10::kCUDA, (c10::DeviceIndex)device));
  TORCH_CHECK((int)bucket_ptrs.size() == world, "allreduce_push_finish: need one bucket pointer per rank");
  std::vector<void*> ptrs;
  for (int64_t p : bucket_ptrs) ptrs.push_back(reinterpret_cast<void*>(static_cast<uintptr_t>(p)));
  check_rc(gs_allreduce_push_finish_f32(ptrs.data(), reinterpret_cast<const float*>(static_cast<uintptr_t>(staging_local)),
                                        n_floats, per, rank, world, cur_stream()),
           "gs_allreduce_push_finish_f32");
}

void allreduce_push_finish_mc(int64_t bucket_multicast, int64_t bucket_local, int64_t staging_local, int64_t n_floats,
                              int64_t per, int rank, int world, int device) {
  c10::cuda::CUDAGuard guard(c10::Device(c10::kCUDA, (c10::DeviceIndex)device));
  check_rc(gs_allreduce_push_finish_mc_f32(reinterpret_cast<void*>(static_cast<uintptr_t>(bucket_multicast)),
                                           reinterpret_cast<const float*>(static_cast<uintptr_t>(bucket_local)),
                                           reinterpret_cast<const float*>(static_cast<uintptr_t>(staging_local)), n_floats,
                                           per, rank, world, cur_stream()),
           "gs_allreduce_push_finish_mc_f32");
}

}  // namespace gsb200

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  using namespace gsb200;
  m.doc() = "B200-native drop-in for the reference `gaussian` extension (libgs_b200 C ABI underneath)";
  m.def("culling", &culling, "gaussian culling (no-op stub, as in the reference)");
  m.def("world2camera", &world2camera, "world to camera (CUDA)");
  m.def("world2camera_backward", &world2camera_backward, "world to camera backward (CUDA)");
  m.def("jacobian", &jacobian, "jacobian (CUDA)");

  py::class_<TilesPy>(m, "Tiles")
      .def(py::init<>())
      .def_readwrite("top", &TilesPy::top)
      .def_readwrite("bottom", &TilesPy::bottom)
      .def_readwrite("left", &TilesPy::left)
      .def_readwrite("right", &TilesPy::right);

  py::class_<Gaussian3dsPy>(m, "Gaussian3ds")
      .def(py::init<>())
      .def_readwrite("pos", &Gaussian3dsPy::pos)
      .def_readwrite("rgb", &Gaussian3dsPy::rgb)
      .def_readwrite("opa", &Gaussian3dsPy::opa)
      .def_readwrite("quat", &Gaussian3dsPy::quat)
      .def_readwrite("scale", &Gaussian3dsPy::scale)
      .def_readwrite("cov", &Gaussian3dsPy::cov);

  m.def("calc_tile_list", &calc_tile_list, "calc tile list (CUDA)");
  m.def("gather_gaussians", &gather_gaussians, "gather gaussian (CUDA)");
  m.def("draw", &draw, "draw (CUDA)");
  m.def("draw_backward", &draw_backward, "draw backward (CUDA)");
  m.def("global_culling", &global_culling, "global culling (CUDA)");
  m.def("global_culling_backward", &global_culling_backward, "global culling backward (CUDA)");

  py::class_<RenderContext>(m, "RenderContext")
      .def(py::init<>())
      .def("forward", &RenderContext::forward)
      .def("backward", &RenderContext::backward)
      .def("backward_into", &RenderContext::backward_into, py::arg("pos"), py::arg("rgb"), py::arg("opa"),
           py::arg("quat"), py::arg("scale"), py::arg("image"), py::arg("grad_image"), py::arg("g_pos"),
           py::arg("g_rgb"), py::arg("g_opa"), py::arg("g_quat"), py::arg("g_scale"), py::arg("expected_frame") = -1)
      .def("forward_final", &RenderContext::forward_final)
      .def("backward_final_into", &RenderContext::backward_final_into, py::arg("pos"), py::arg("rgb"),
           py::arg("opa"), py::arg("quat"), py::arg("scale"), py::arg("raw"), py::arg("grad_final"),
           py::arg("g_pos"), py::arg("g_rgb"), py::arg("g_opa"), py::arg("g_quat"), py::arg("g_scale"),
           py::arg("expected_frame") = -1)
      .def("forward_maps", &RenderContext::forward_maps, py::arg("pos"), py::arg("rgb"), py::arg("opa"),
           py::arg("quat"), py::arg("scale"), py::arg("width"), py::arg("height"), py::arg("fx"), py::arg("fy"),
           py::arg("rot"), py::arg("tran"), py::arg("near"), py::arg("thresh"), py::arg("scale_activation"),
           py::arg("background") = py::none(), py::arg("final") = true)
      .def("backward_maps_into", &RenderContext::backward_maps_into, py::arg("pos"), py::arg("rgb"), py::arg("opa"),
           py::arg("quat"), py::arg("scale"), py::arg("raw"), py::arg("depth_raw"), py::arg("alpha_raw"),
           py::arg("grad_image"), py::arg("grad_depth"), py::arg("grad_alpha"), py::arg("grad_is_final"),
           py::arg("g_pos"), py::arg("g_rgb"), py::arg("g_opa"), py::arg("g_quat"), py::arg("g_scale"),
           py::arg("expected_frame") = -1)
      .def("frame_id", &RenderContext::frame_id)
      .def("last_instances", &RenderContext::last_instances)
      .def("stats", &RenderContext::stats)
      .def("set_timing", &RenderContext::set_timing)
      .def("set_grad_push", &RenderContext::set_grad_push)
      .def("clear_grad_push", &RenderContext::clear_grad_push)
      .def("set_camera_grad", &RenderContext::set_camera_grad, py::arg("grad_cam"))
      .def("stage_ms", &RenderContext::stage_ms)
      .def("sorted_instances", &RenderContext::sorted_instances)
      .def("tile_consumed", &RenderContext::tile_consumed);
  m.def("allreduce_push_finish", &allreduce_push_finish, "second half of the pushed gradient exchange");
  m.def("allreduce_push_finish_mc", &allreduce_push_finish_mc,
        "second half of the pushed gradient exchange, broadcast through the NVSwitch (multimem.st)");
  m.def("allreduce_p2p", &allreduce_p2p, "peer-to-peer two-shot in-place all-reduce of a symmetric buffer");
  m.def("allreduce_multimem", &allreduce_multimem, "NVLS multimem in-place all-reduce of a symmetric buffer");
  m.def("densify", &densify, "prune / clone / split on the device (reference splatter.py:122-228)", py::arg("pos"),
        py::arg("rgb"), py::arg("opa"), py::arg("quat"), py::arg("scale"), py::arg("grad"), py::arg("scale_activation"),
        py::arg("opa_logit_min"), py::arg("delete_thresh"), py::arg("grad_thresh"), py::arg("grad_agg_max"), py::arg("tau"),
        py::arg("use_clone"), py::arg("use_split"), py::arg("clone_dt"), py::arg("generator") = py::none());
  m.def("loss_l1_ssim", &loss_l1_ssim, "fused L1 + SSIM loss, forward + image gradient (CUDA)");
  m.def("adam_step", &adam_step, "fused Adam over flat parameter / gradient buffers (CUDA)");
  m.def("tune", [](const std::string& name, int value) { check_rc(gs_tune(name.c_str(), value), "gs_tune"); },
        "set a blend-path knob: gather (0 packed, 1 gather) or sh_tc (0..3); see include/gs_b200.h gs_tune");
  m.def("tuned", [](const std::string& name) {
          int v = 0;
          check_rc(gs_tune_get(name.c_str(), &v), "gs_tune_get");
          return v;
        },
        "current value of a gs_tune knob (gather, sh_tc)");
  m.def("kernel_launches", []() { return (int64_t)gs_kernel_launches(); },
        "kernels of libgs_b200 launched by this process so far");
  m.attr("abi_version") = gs_abi_version();
}
