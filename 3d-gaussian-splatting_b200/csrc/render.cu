// Frame orchestration for the fused path: owns device workspaces and strings the stages
//   project -> depth sort of the N Gaussians + scan -> emit in depth order -> stable tile-id
//   radix sort of the M instances (CUB onesweep, 2 passes at 1080p) -> range+pack -> blend
// and the backward  blend_bwd -> project_bwd (segment-sum + chain rule).
// Replaces the PyTorch glue of reference splatter.py:513-655 (4 boolean-mask compactions, the
// dense [T, N/20] tile list, cumsum, two 4-tensor gathers, fp32-key torch.sort, >= 7 host
// syncs) with 7 launches and ONE 8-byte readback (the instance count M sizes the sort).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "internal.h"

// count of the Gaussian at depth-sorted position i (0 for the sentinel item i == n)
struct GsCountInSortedOrder {
  const uint32_t* count;
  const uint32_t* perm;
  uint32_t n;
  __host__ __device__ __forceinline__ uint32_t operator()(uint32_t i) const { return i < n ? count[perm[i]] : 0u; }
};

// ---- error plumbing ---------------------------------------------------------------------
static thread_local char g_err[512] = {0};

int gs_set_error(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return (int)e;
}
int gs_set_error_msg(int code, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s", what);
  return code;
}
extern "C" const char* gs_last_error(void) { return g_err; }
extern "C" int gs_abi_version(void) { return 2; }

static int tune_env(const char* env, int dflt, int max) {
  const char* e = getenv(env);
  const int v = e ? atoi(e) : dflt;
  return v >= 0 && v <= max ? v : dflt;
}
GsTuning& gs_tuning() {
  static GsTuning t = {tune_env("GS_TUNE_GATHER", 1, 1), tune_env("GS_TUNE_SH_TC", 3, 3)};
  return t;
}
// the knob called `name` (nullptr if there is none) and its largest valid value; every range starts at 0
static int* tune_knob(const char* name, int& max) {
  GsTuning& t = gs_tuning();
  if (!strcmp(name, "gather")) {
    max = 1;
    return &t.gather;
  }
  if (!strcmp(name, "sh_tc")) {
    max = 3;
    return &t.sh_tc;
  }
  return nullptr;
}
extern "C" int gs_tune(const char* name, int value) {
  if (!name) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_tune: null name");
  int max = 0;
  int* v = tune_knob(name, max);
  if (!v) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_tune: unknown knob");
  if (value < 0 || value > max) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_tune: value out of range");
  *v = value;
  return 0;
}
extern "C" int gs_tune_get(const char* name, int* value) {
  if (!name || !value) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_tune_get: null argument");
  int max = 0;
  const int* v = tune_knob(name, max);
  if (!v) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_tune_get: unknown knob");
  *value = *v;
  return 0;
}

#include <atomic>
static std::atomic<unsigned long long> g_launches{0};
void gs_count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
extern "C" unsigned long long gs_kernel_launches(void) { return g_launches.load(std::memory_order_relaxed); }

// ---- growable device buffer -------------------------------------------------------------
// Workspaces come from the caller's allocator when one is installed (gs_ctx_set_allocator: the torch shim
// passes PyTorch's stream-ordered caching allocator, so growth - e.g. after every densification - needs no
// device synchronisation and the memory shows up in torch's accounting); else cudaMalloc / cudaFree with a
// stream synchronisation before a buffer is replaced.
struct GsAllocator {
  gs_alloc_fn alloc = nullptr;
  gs_free_fn free = nullptr;
  void* user = nullptr;
};
static thread_local const GsAllocator* g_cur_alloc = nullptr;   // allocator of the context being served

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  const GsAllocator* owner = nullptr;       // allocator the current block came from (nullptr: cudaMalloc)
  void drop(cudaStream_t st, bool sync) {
    if (!p) return;
    if (owner && owner->free) {
      owner->free(p, owner->user);          // stream-ordered allocator: no synchronisation needed
    } else {
      if (sync) cudaStreamSynchronize(st);
      cudaFree(p);
    }
    p = nullptr;
    cap = 0;
  }
  cudaError_t reserve(size_t bytes, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    drop(st, true);
    size_t want = bytes + bytes / 8 + 256;   // slack so M jitter between frames does not realloc
    const GsAllocator* a = g_cur_alloc;
    if (a && a->alloc) {
      p = a->alloc(want, a->user, (gs_stream_t)st);
      if (!p) return cudaErrorMemoryAllocation;
      owner = a;
    } else {
      cudaError_t e = cudaMalloc(&p, want);
      if (e != cudaSuccess) return e;
      owner = nullptr;
    }
    cap = want;
    return cudaSuccess;
  }
  void release() { drop(nullptr, false); }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

struct gs_ctx {
  int device = 0;
  GsAllocator allocator{};
  // per Gaussian
  DevBuf rec, count, offsets, dkey_in, dkey_out, perm, iota, offsets_g;
  size_t iota_n = 0;
  // per instance
  DevBuf keys_in, keys_out, vals_in, vals_out, pA, pB, pC, grad_inst, row_epoch;
  uint32_t epoch = 0;                      // tag of the current backward in row_epoch[]
  // per tile / misc
  DevBuf tile_accum, tile_neff, tile_neff_b, cub_tmp, counters, img_dev, gimg_dev, rays;
  DevBuf cam_partial;                     // camera gradient: one [12] double row per projection-backward block
  float* host_rays = nullptr;             // pinned: rays_o, lefttop, dx, dy (SH colour only)
  unsigned long long* host_m = nullptr;   // pinned: {M}
  cudaEvent_t ev_m = nullptr;             // marks the completion of the M read-back
  // state of the last forward
  bool have_forward = false, have_backward = false, gather = false;
  bool maps = false;                      // the last forward also wrote depth / alpha maps (gs_render_forward_maps)
  int n = 0, d = 3, scale_act = 0;
  long long m = 0;
  GsCam cam{};
  GsTileGrid grid{};
  GsFrameGeom geom{};
  float near_plane = 0.f, half_w = 0.f, half_h = 0.f;
  int64_t* mask_ptr = nullptr;
  // optional per-stage timing (CUDA events on the frame's stream)
  bool timing = false;
  cudaEvent_t ev[GS_N_STAGES + 2] = {};
  bool ev_ok = false;
  bool ev_fwd_valid = false, ev_bwd_valid = false;
  // data-parallel gradient push (gs_ctx_set_grad_push); world == 0: off
  GsGradPush push{};
  // camera gradient output (gs_ctx_set_camera_grad; device, 12 floats); nullptr: off
  float* grad_cam = nullptr;
};

// stage boundaries: event i is recorded BEFORE stage i; stage i lasts ev[i+1]-ev[i]
//  forward : 0 project | 1 scan+readback | 2 emit keys | 3 radix sort | 4 pack | 5 blend fwd | (6 end)
//  backward: 7 blend bwd | 8 project bwd | (9 end)
static inline void gs_mark(gs_ctx* c, int i, cudaStream_t st) {
  if (c->timing && c->ev_ok) cudaEventRecord(c->ev[i], st);
}

extern "C" int gs_ctx_create(gs_ctx** out) {
  if (!out) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_create: null out");
  gs_ctx* c = new (std::nothrow) gs_ctx();
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_create: out of host memory");
  GS_CUDA_TRY(cudaGetDevice(&c->device));
  cudaError_t e = cudaMallocHost(reinterpret_cast<void**>(&c->host_m), 64);
  if (e == cudaSuccess) e = cudaMallocHost(reinterpret_cast<void**>(&c->host_rays), 64);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_m, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    delete c;
    return gs_set_error(e, "cudaMallocHost");
  }
  *out = c;
  return 0;
}

extern "C" void gs_ctx_destroy(gs_ctx* c) {
  if (!c) return;
  // the buffers live on the device that was current at creation, which need not be current now
  int cur = -1;
  const bool switched = cudaGetDevice(&cur) == cudaSuccess && cur != c->device && cudaSetDevice(c->device) == cudaSuccess;
  cudaDeviceSynchronize();
  DevBuf* bufs[] = {&c->rec, &c->count, &c->offsets, &c->dkey_in, &c->dkey_out, &c->perm, &c->iota, &c->offsets_g, &c->keys_in, &c->keys_out,
                    &c->vals_in, &c->vals_out, &c->pA, &c->pB, &c->pC, &c->grad_inst, &c->row_epoch, &c->tile_accum, &c->tile_neff,
                    &c->tile_neff_b, &c->cub_tmp, &c->counters, &c->img_dev, &c->gimg_dev, &c->rays, &c->cam_partial};
  for (DevBuf* b : bufs) b->release();
  if (c->host_m) cudaFreeHost(c->host_m);
  if (c->host_rays) cudaFreeHost(c->host_rays);
  if (c->ev_m) cudaEventDestroy(c->ev_m);
  if (c->ev_ok)
    for (cudaEvent_t e : c->ev) cudaEventDestroy(e);
  if (switched) cudaSetDevice(cur);
  delete c;
}

// a ctx owns buffers on the device that was current at gs_ctx_create; using it under another
// current device would launch on the wrong GPU
static int gs_check_device(int want, const char* who) {
  int dev = -1;
  GS_CUDA_TRY(cudaGetDevice(&dev));
  if (dev != want) {
    char msg[160];
    snprintf(msg, sizeof(msg), "%s: ctx belongs to device %d but device %d is current", who, want, dev);
    return gs_set_error_msg(GS_ERR_INVALID_ARG, msg);
  }
  return 0;
}

static int ceil_log2(unsigned v) {
  int b = 0;
  while ((1u << b) < v) ++b;
  return b;
}

// a maps frame needs the RGB gather path and one GPU's gradient layout; returns 0 or the refusal
static int check_maps_supported(const gs_ctx* c, int d, const char* fn) {
  char msg[200];
  const char* why = nullptr;
  if (d != 3)
    why = "depth / alpha maps need RGB colour (d == 3); SH colour is not supported";
  else if (gs_tuning().gather == 0)
    why = "depth / alpha maps need the gather path (gs_tune(\"gather\", 0) is set)";
  else if (c->push.world != 0)
    why = "depth / alpha maps do not support the data-parallel gradient push (gs_ctx_set_grad_push is active)";
  if (!why) return 0;
  snprintf(msg, sizeof(msg), "%s: %s", fn, why);
  return gs_set_error_msg(GS_ERR_UNSUPPORTED, msg);
}

// camera gradients need RGB colour on one GPU; returns 0 or the refusal
static int check_camgrad_supported(const gs_ctx* c, const char* fn) {
  char msg[260];
  const char* why = nullptr;
  if (c->d != 3)
    why = "camera gradients need RGB colour (d == 3); with SH colour the per-pixel SH basis depends on the camera "
          "through the ray directions, which is not differentiated";
  else if (c->push.world != 0)
    why = "camera gradients do not support the data-parallel gradient push (gs_ctx_set_grad_push is active)";
  if (!why) return 0;
  snprintf(msg, sizeof(msg), "%s: %s", fn, why);
  return gs_set_error_msg(GS_ERR_UNSUPPORTED, msg);
}

static int render_forward_impl(gs_ctx* c, const float* pos, const float* rgb, const float* opa, const float* quat,
                               const float* scale, int n, int d, int scale_activation, const gs_camera* cam,
                               float* image, float* final_img, int64_t* culling_mask, gs_stream_t stream,
                               const GsMapsFwd* maps = nullptr) {
  if (!c || !cam || n < 0) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward: bad arguments");
  if (d != 3 && gs_sh_basis_count(d) == 0)
    return gs_set_error_msg(GS_ERR_UNSUPPORTED, "gs_render_forward: colour width must be 3 (RGB), 27 (SH deg 2) or 48 (SH deg 3)");
  if (cam->width <= 0 || cam->height <= 0 || !(cam->focal_x > 0.f) || !(cam->focal_y > 0.f))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward: bad camera");
  if (!(cam->tile_thresh > 0.f && cam->tile_thresh < 1.f))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward: tile_thresh must be in (0, 1)");
  if (!image || (n > 0 && (!pos || !rgb || !opa || !quat || !scale)))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward: null tensor pointer");
  if (maps)
    if (int rc = check_maps_supported(c, d, "gs_render_forward_maps")) return rc;
  if (int rc = gs_check_device(c->device, "gs_render_forward")) return rc;
  g_cur_alloc = &c->allocator;
  cudaStream_t st = (cudaStream_t)stream;
  c->have_forward = false;
  c->maps = false;
  c->have_backward = false;

  GsFrameGeom g{};
  g.width = cam->width;
  g.height = cam->height;
  g.wp = (cam->width + GS_TILE - 1) / GS_TILE * GS_TILE;     // splatter.py:259-260
  g.hp = (cam->height + GS_TILE - 1) / GS_TILE * GS_TILE;
  g.ntx = g.wp / GS_TILE;
  g.nty = g.hp / GS_TILE;
  g.n_tiles = g.ntx * g.nty;
  g.fx = cam->focal_x;
  g.fy = cam->focal_y;
  if (g.ntx > 65535 || g.nty > 65535) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward: image too large");

  // Host scalars are formed in double then narrowed, like the Python floats that the reference
  // passes through pybind (splatter.py:279-282, :532-533).
  GsTileGrid grid{};
  grid.lx = (float)(16.0 / (double)cam->focal_x);
  grid.ly = (float)(16.0 / (double)cam->focal_y);
  grid.leftmost = (float)(-(double)g.wp / 2.0 / (double)cam->focal_x);
  grid.topmost = (float)(-(double)g.hp / 2.0 / (double)cam->focal_y);
  grid.t2 = -2.f * logf(cam->tile_thresh);
  grid.ntx = g.ntx;
  grid.nty = g.nty;
  GsCam dc{};
  memcpy(dc.r, cam->rot, sizeof(dc.r));
  memcpy(dc.t, cam->tran, sizeof(dc.t));
  float half_w = (float)((double)cam->width * 1.2 / 2.0 / (double)cam->focal_x);
  float half_h = (float)((double)cam->height * 1.2 / 2.0 / (double)cam->focal_y);

  size_t N = (size_t)n;
  GS_CUDA_TRY(c->rec.reserve(N * sizeof(GsRec), st));
  GS_CUDA_TRY(c->count.reserve((N + 1) * 4, st));
  GS_CUDA_TRY(c->offsets.reserve((N + 1) * 4, st));
  GS_CUDA_TRY(c->dkey_in.reserve(N * 4 + 4, st));
  GS_CUDA_TRY(c->dkey_out.reserve(N * 4 + 4, st));
  GS_CUDA_TRY(c->perm.reserve(N * 4 + 4, st));
  GS_CUDA_TRY(c->offsets_g.reserve((N + 1) * 4, st));
  GS_CUDA_TRY(c->tile_accum.reserve((size_t)(g.n_tiles + 1) * 4, st));
  GS_CUDA_TRY(c->tile_neff.reserve((size_t)g.n_tiles * 4, st));
  GS_CUDA_TRY(c->tile_neff_b.reserve((size_t)g.n_tiles * 4, st));
  GS_CUDA_TRY(c->counters.reserve(64, st));
  if (c->iota_n < N) {   // 0..N-1 values for the depth sort (kept across frames)
    GS_CUDA_TRY(c->iota.reserve(N * 4 + 4, st));
    GS_CUDA_TRY(gs_launch_iota(c->iota.as<uint32_t>(), n, st));
    gs_count_launch();
    c->iota_n = N;
  }

  if (d != 3) {
    // world-space ray set-up for per-pixel SH, reference splatter.py:305-321 (RayInfo):
    // c2w = inverse(w2c); rays_o = -c2w t; lefttop = c2w (((-Wp/2+.5)/fx, (-Hp/2+.5)/fy, 1) - t)
    GS_CUDA_TRY(c->rays.reserve(64, st));
    double m3[9], inv[9];
    for (int k = 0; k < 9; ++k) m3[k] = cam->rot[k];
    double det3 = m3[0] * (m3[4] * m3[8] - m3[5] * m3[7]) - m3[1] * (m3[3] * m3[8] - m3[5] * m3[6]) +
                  m3[2] * (m3[3] * m3[7] - m3[4] * m3[6]);
    inv[0] = (m3[4] * m3[8] - m3[5] * m3[7]) / det3;
    inv[1] = (m3[2] * m3[7] - m3[1] * m3[8]) / det3;
    inv[2] = (m3[1] * m3[5] - m3[2] * m3[4]) / det3;
    inv[3] = (m3[5] * m3[6] - m3[3] * m3[8]) / det3;
    inv[4] = (m3[0] * m3[8] - m3[2] * m3[6]) / det3;
    inv[5] = (m3[2] * m3[3] - m3[0] * m3[5]) / det3;
    inv[6] = (m3[3] * m3[7] - m3[4] * m3[6]) / det3;
    inv[7] = (m3[1] * m3[6] - m3[0] * m3[7]) / det3;
    inv[8] = (m3[0] * m3[4] - m3[1] * m3[3]) / det3;
    double lt[3] = {(-(double)g.wp / 2 + 0.5) / cam->focal_x - cam->tran[0],
                    (-(double)g.hp / 2 + 0.5) / cam->focal_y - cam->tran[1], 1.0 - cam->tran[2]};
    for (int k = 0; k < 3; ++k) {
      c->host_rays[k] = (float)(-(inv[3 * k] * cam->tran[0] + inv[3 * k + 1] * cam->tran[1] + inv[3 * k + 2] * cam->tran[2]));
      c->host_rays[3 + k] = (float)(inv[3 * k] * lt[0] + inv[3 * k + 1] * lt[1] + inv[3 * k + 2] * lt[2]);
      c->host_rays[6 + k] = (float)(inv[3 * k] / cam->focal_x);
      c->host_rays[9 + k] = (float)(inv[3 * k + 1] / cam->focal_y);
    }
    GS_CUDA_TRY(cudaMemcpyAsync(c->rays.p, c->host_rays, 48, cudaMemcpyHostToDevice, st));
  }
  // 1. projection + activations + tile rectangle
  c->ev_fwd_valid = false;
  gs_mark(c, 0, st);
  GS_CUDA_TRY(cudaMemsetAsync(c->counters.p, 0, 64, st));
  GS_CUDA_TRY(cudaMemsetAsync(c->count.as<uint32_t>() + N, 0, 4, st));
  GS_CUDA_TRY(gs_launch_fused_project(pos, rgb, opa, quat, scale, n, d, scale_activation, dc, grid, cam->near_plane,
                                      half_w, half_h, c->rec.as<GsRec>(), c->count.as<uint32_t>(),
                                      c->dkey_in.as<uint32_t>(), culling_mask, c->counters.as<unsigned int>(), st));
  if (n > 0) gs_count_launch();
  // 2. (a) exclusive scan of the tile counts in Gaussian-id order -> gradient-row bases and M;
  //    (b) stable depth sort of the N Gaussians; (c) scan of the counts in depth order (the
  //    count gather is fused into the scan's input iterator) -> instance emission offsets
  gs_mark(c, 1, st);
  size_t tmp_bytes = 0, tmp2 = 0, tmp3 = 0;
  if (n > 0)
    GS_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, c->dkey_in.as<uint32_t>(),
                                                c->dkey_out.as<uint32_t>(), c->iota.as<uint32_t>(),
                                                c->perm.as<uint32_t>(), n, 0, 32, st));
  GsCountInSortedOrder cnt_it_fn{c->count.as<uint32_t>(), c->perm.as<uint32_t>(), (uint32_t)n};
  cub::CountingInputIterator<uint32_t> idx_it(0);
  cub::TransformInputIterator<uint32_t, GsCountInSortedOrder, cub::CountingInputIterator<uint32_t>> cnt_it(idx_it,
                                                                                                            cnt_it_fn);
  GS_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp2, cnt_it, c->offsets.as<uint32_t>(), n + 1, st));
  GS_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp3, c->count.as<uint32_t>(), c->offsets_g.as<uint32_t>(),
                                            n + 1, st));
  if (tmp2 > tmp_bytes) tmp_bytes = tmp2;
  if (tmp3 > tmp_bytes) tmp_bytes = tmp3;
  GS_CUDA_TRY(c->cub_tmp.reserve(tmp_bytes, st));
  GS_CUDA_TRY(cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp3, c->count.as<uint32_t>(), c->offsets_g.as<uint32_t>(),
                                            n + 1, st));
  // the one host round trip of the frame: M = offsets_g[N] is known right after the first scan, so
  // its read-back is enqueued BEFORE the depth sort and the host waits on an event recorded there -
  // the GPU keeps sorting while the host wakes up and enqueues the rest of the frame (no bubble)
  *c->host_m = 0;
  GS_CUDA_TRY(cudaMemcpyAsync(c->host_m, c->counters.as<unsigned int>() + 2, 8, cudaMemcpyDeviceToHost, st));
  GS_CUDA_TRY(cudaEventRecord(c->ev_m, st));
  if (n > 0)
    GS_CUDA_TRY(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, tmp_bytes, c->dkey_in.as<uint32_t>(),
                                                c->dkey_out.as<uint32_t>(), c->iota.as<uint32_t>(),
                                                c->perm.as<uint32_t>(), n, 0, 32, st));
  GS_CUDA_TRY(cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp2, cnt_it, c->offsets.as<uint32_t>(), n + 1, st));
  GS_CUDA_TRY(cudaEventSynchronize(c->ev_m));
  // 64-bit total accumulated by the projection kernel (== offsets_g[N] whenever the u32 scans did
  // not wrap); instance indices are 32-bit from here on
  if (*c->host_m >= (1ull << 31))
    return gs_set_error_msg(GS_ERR_UNSUPPORTED, "gs_render_forward: more than 2^31 tile instances");
  long long m = (long long)*c->host_m;
  size_t M = (size_t)m;

  const bool gather = gs_tuning().gather != 0;   // RGB and SH: no pack pass
  gs_mark(c, 2, st);
  // tile-id sort key width (GS_TILE_KEY_BYTES=4 forces the wide path, for tests)
  static const int forced_key = getenv("GS_TILE_KEY_BYTES") ? atoi(getenv("GS_TILE_KEY_BYTES")) : 0;
  const int key_bytes = (g.n_tiles <= 65536 && forced_key != 4) ? 2 : 4;
  const size_t crow = d == 3 ? 16 : (size_t)gs_sh_stream_width(d) * 4;   // colour / SH stream row bytes
  if (!gather) {
    GS_CUDA_TRY(c->pA.reserve(M * 16 + 16, st));
    GS_CUDA_TRY(c->pC.reserve(M * crow + 16, st));
    GS_CUDA_TRY(c->pB.reserve((M + 2) * 8, st));
  }
  if (m > 0) {
    GS_CUDA_TRY(c->keys_in.reserve(M * 4 + 16, st));
    GS_CUDA_TRY(c->keys_out.reserve(M * 4 + 16, st));
    GS_CUDA_TRY(c->vals_in.reserve(M * 4, st));
    GS_CUDA_TRY(c->vals_out.reserve(M * 4, st));
    // 3. instances in (depth, id) order: tile-id keys + Gaussian-id values
    GS_CUDA_TRY(gs_launch_emit_keys(c->rec.as<GsRec>(), c->perm.as<uint32_t>(), c->offsets.as<uint32_t>(), n, g.ntx,
                                    c->keys_in.p, key_bytes, c->vals_in.as<uint32_t>(), st));
    gs_count_launch();
    // 4. stable radix sort on the tile id only -> (tile, depth, id)
    gs_mark(c, 3, st);
    int end_bit = ceil_log2((unsigned)g.n_tiles);
    if (end_bit < 1) end_bit = 1;
    size_t sort_tmp = 0;
    if (key_bytes == 2) {
      GS_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, c->keys_in.as<uint16_t>(),
                                                  c->keys_out.as<uint16_t>(), c->vals_in.as<uint32_t>(),
                                                  c->vals_out.as<uint32_t>(), (int)m, 0, end_bit, st));
      GS_CUDA_TRY(c->cub_tmp.reserve(sort_tmp, st));
      GS_CUDA_TRY(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, sort_tmp, c->keys_in.as<uint16_t>(),
                                                  c->keys_out.as<uint16_t>(), c->vals_in.as<uint32_t>(),
                                                  c->vals_out.as<uint32_t>(), (int)m, 0, end_bit, st));
    } else {
      GS_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, c->keys_in.as<uint32_t>(),
                                                  c->keys_out.as<uint32_t>(), c->vals_in.as<uint32_t>(),
                                                  c->vals_out.as<uint32_t>(), (int)m, 0, end_bit, st));
      GS_CUDA_TRY(c->cub_tmp.reserve(sort_tmp, st));
      GS_CUDA_TRY(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, sort_tmp, c->keys_in.as<uint32_t>(),
                                                  c->keys_out.as<uint32_t>(), c->vals_in.as<uint32_t>(),
                                                  c->vals_out.as<uint32_t>(), (int)m, 0, end_bit, st));
    }
  }
  // 5. tile ranges + packed sorted record streams
  if (m == 0) gs_mark(c, 3, st);
  gs_mark(c, 4, st);
  if (gather) {
    // no pack pass: only the tile ranges are derived from the sorted keys; the blend kernels pull the records
    // of their tile straight from rec[N] through the sorted id list
    GS_CUDA_TRY(gs_launch_tile_ranges(c->keys_out.p, key_bytes, m, g.n_tiles, c->tile_accum.as<int>(), st));
  } else if (d == 3) {
    GS_CUDA_TRY(gs_launch_pack_sorted(c->keys_out.p, key_bytes, c->vals_out.as<uint32_t>(), m, g.n_tiles, g.ntx,
                                      c->rec.as<GsRec>(), c->offsets_g.as<uint32_t>(), c->pA.as<float4>(),
                                      c->pB.as<float2>(), c->pC.as<float4>(), c->tile_accum.as<int>(), st));
  } else {
    GS_CUDA_TRY(gs_launch_pack_sorted_sh(c->keys_out.p, key_bytes, c->vals_out.as<uint32_t>(), m, g.n_tiles, g.ntx,
                                         c->rec.as<GsRec>(), c->offsets_g.as<uint32_t>(), rgb, d,
                                         gs_sh_stream_width(d), c->pA.as<float4>(), c->pB.as<float2>(),
                                         c->pC.as<float>(), c->tile_accum.as<int>(), st));
  }
  if (m > 0) gs_count_launch();   // pack, or the tile-range pass of the gather path
  // 6. blend (+ optional fused clamp & centre crop, splatter.py:652-653 / :267-272)
  GsCrop crop{(g.wp - g.width) / 2, (g.hp - g.height) / 2, g.width, g.height};
  gs_mark(c, 5, st);
  if (maps) {
    GS_CUDA_TRY(gs_launch_blend_fwd_maps(c->rec.as<GsRec>(), c->vals_out.as<uint32_t>(), c->tile_accum.as<int>(), g, image,
                                         c->tile_neff.as<int>(), final_img, crop, *maps, st));
  } else if (d == 3) {
    GS_CUDA_TRY(gs_launch_blend_fwd(c->pA.as<float4>(), c->pB.as<float2>(), c->pC.as<float4>(),
                                    gather ? c->rec.as<GsRec>() : nullptr, c->vals_out.as<uint32_t>(),
                                    c->tile_accum.as<int>(), g, image, c->tile_neff.as<int>(), final_img, crop, st));
  } else {
    const float* rp = c->rays.as<float>();
    GsRayPtrs rays{rp, rp + 3, rp + 6, rp + 9};
    GS_CUDA_TRY(gs_launch_blend_sh_fwd(c->pA.as<float4>(), c->pB.as<float2>(), c->pC.as<float>(),
                                       gather ? c->rec.as<GsRec>() : nullptr, rgb, c->vals_out.as<uint32_t>(),
                                       c->offsets_g.as<uint32_t>(), d,
                                       c->tile_accum.as<int>(), g, rays, image, c->tile_neff.as<int>(), final_img,
                                       crop, st));
  }
  gs_count_launch();   // blend forward
  gs_mark(c, 6, st);
  c->ev_fwd_valid = c->timing && c->ev_ok;

  c->have_forward = true;
  c->maps = maps != nullptr;
  c->gather = gather;
  c->n = n;
  c->d = d;
  c->scale_act = scale_activation;
  c->m = m;
  c->cam = dc;
  c->grid = grid;
  c->geom = g;
  c->near_plane = cam->near_plane;
  c->half_w = half_w;
  c->half_h = half_h;
  return 0;
}

extern "C" int gs_render_forward(gs_ctx* c, const float* pos, const float* rgb, const float* opa, const float* quat,
                                 const float* scale, int n, int d, int scale_activation, const gs_camera* cam,
                                 float* image, int64_t* culling_mask, gs_stream_t stream) {
  return render_forward_impl(c, pos, rgb, opa, quat, scale, n, d, scale_activation, cam, image, nullptr, culling_mask,
                             stream);
}

extern "C" int gs_render_forward_final(gs_ctx* c, const float* pos, const float* rgb, const float* opa,
                                       const float* quat, const float* scale, int n, int d, int scale_activation,
                                       const gs_camera* cam, float* image_raw_padded, float* image_final,
                                       int64_t* culling_mask, gs_stream_t stream) {
  if (!image_final) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward_final: null image_final");
  return render_forward_impl(c, pos, rgb, opa, quat, scale, n, d, scale_activation, cam, image_raw_padded, image_final,
                             culling_mask, stream);
}

static int render_backward_impl(gs_ctx* c, const float* pos, const float* rgb, const float* opa, const float* quat,
                                const float* scale, const float* image, const float* grad_image, int grad_is_final,
                                float* grad_pos, float* grad_rgb, float* grad_opa, float* grad_quat,
                                float* grad_scale, gs_stream_t stream, const GsMapsBwd* maps = nullptr) {
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_backward: null ctx");
  if (!c->have_forward) return gs_set_error_msg(GS_ERR_NO_FORWARD, "gs_render_backward: no forward on this ctx");
  if (c->grad_cam)
    if (int rc = check_camgrad_supported(c, maps ? "gs_render_backward_maps" : "gs_render_backward")) return rc;
  if (maps) {
    if (!c->maps)
      return gs_set_error_msg(GS_ERR_NO_FORWARD,
                              "gs_render_backward_maps: the last forward on this ctx was not gs_render_forward_maps");
    if (int rc = check_maps_supported(c, c->d, "gs_render_backward_maps")) return rc;
    if (!maps->depth || !maps->alpha || !maps->grad_depth || !maps->grad_alpha)
      return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_backward_maps: null map pointer");
  }
  if (!image || !grad_image || !grad_pos || !grad_rgb || !grad_opa || !grad_quat || !grad_scale ||
      (c->n > 0 && (!pos || !rgb || !opa || !quat || !scale)))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_backward: null tensor pointer");
  if (int rc = gs_check_device(c->device, "gs_render_backward")) return rc;
  g_cur_alloc = &c->allocator;
  cudaStream_t st = (cudaStream_t)stream;
  size_t M = (size_t)c->m;
  const int d = c->d;
  const size_t grow = d == 3 ? (size_t)GS_GREC * 4 : (size_t)gs_sh_grad_width(d) * 4;
  GS_CUDA_TRY(c->grad_inst.reserve(M * grow + 16, st));
  if (c->grad_cam) GS_CUDA_TRY(c->cam_partial.reserve(gs_camgrad_partial_bytes(c->n), st));
  {
    // one u32 tag per gradient row: rows written by this backward carry `epoch`; the tails of
    // saturated tiles are never written nor read (saves ~0.2 GB of HBM writes + reads at C3)
    const size_t before = c->row_epoch.cap;            // (a caching allocator may hand the same address back)
    GS_CUDA_TRY(c->row_epoch.reserve(M * 4 + 16, st));
    if (c->row_epoch.cap != before || c->epoch == 0xffffffffu) {
      GS_CUDA_TRY(cudaMemsetAsync(c->row_epoch.p, 0, c->row_epoch.cap, st));
      c->epoch = 0;
    }
    ++c->epoch;
  }
  c->ev_bwd_valid = false;
  GsCrop crop{(c->geom.wp - c->geom.width) / 2, (c->geom.hp - c->geom.height) / 2, c->geom.width, c->geom.height};
  gs_mark(c, 7, st);
  if (c->m > 0) {
    if (maps) {
      GS_CUDA_TRY(gs_launch_blend_bwd_maps(c->rec.as<GsRec>(), c->vals_out.as<uint32_t>(), c->offsets_g.as<uint32_t>(),
                                           c->tile_accum.as<int>(), c->geom, image, grad_image, c->grad_inst.as<float>(),
                                           grad_is_final, crop, c->row_epoch.as<uint32_t>(), c->epoch,
                                           c->tile_neff_b.as<int>(), *maps, st));
    } else if (d == 3) {
      GS_CUDA_TRY(gs_launch_blend_bwd(c->pA.as<float4>(), c->pB.as<float2>(), c->pC.as<float4>(),
                                      c->gather ? c->rec.as<GsRec>() : nullptr, c->vals_out.as<uint32_t>(),
                                      c->offsets_g.as<uint32_t>(), c->tile_accum.as<int>(), c->geom, image, grad_image,
                                      c->grad_inst.as<float>(),
                                      grad_is_final, crop, c->row_epoch.as<uint32_t>(), c->epoch,
                                      c->tile_neff_b.as<int>(), st));
    } else {
      const float* rp = c->rays.as<float>();
      GsRayPtrs rays{rp, rp + 3, rp + 6, rp + 9};
      GS_CUDA_TRY(gs_launch_blend_sh_bwd(c->pA.as<float4>(), c->pB.as<float2>(), c->pC.as<float>(),
                                         c->gather ? c->rec.as<GsRec>() : nullptr, rgb, c->vals_out.as<uint32_t>(),
                                         c->offsets_g.as<uint32_t>(), d,
                                         c->tile_accum.as<int>(), c->geom, rays, image, grad_image,
                                         c->grad_inst.as<float>(), grad_is_final, crop,
                                         c->row_epoch.as<uint32_t>(), c->epoch, c->tile_neff_b.as<int>(), st));
    }
    gs_count_launch();
    c->have_backward = true;
  }
  gs_mark(c, 8, st);
  if (c->push.world) {
    // every gradient segment must lie inside the sliced bucket, quaternions on 16-byte offsets
    const float* lo = c->push.bucket;
    const float* hi = lo + (size_t)c->push.world * c->push.per;
    const size_t nn = (size_t)c->n;
    const float* seg[5] = {grad_pos, grad_rgb, grad_opa, grad_quat, grad_scale};
    const size_t len[5] = {3 * nn, (size_t)d * nn, nn, 4 * nn, 3 * nn};
    for (int k = 0; k < 5; ++k)
      if (seg[k] < lo || seg[k] + len[k] > hi)
        return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_backward: gradient buffers are not inside the push bucket");
    if ((grad_quat - lo) % 4)
      return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_backward: grad_quat must sit on a 16-byte bucket offset");
  }
  GS_CUDA_TRY(gs_launch_fused_project_bwd(pos, rgb, opa, quat, scale, c->n, d, c->scale_act, c->cam, c->near_plane,
                                          c->half_w, c->half_h, c->offsets_g.as<uint32_t>(), c->count.as<uint32_t>(),
                                          c->grad_inst.as<float>(), c->row_epoch.as<uint32_t>(), c->epoch,
                                          grad_pos, grad_rgb, grad_opa, grad_quat, grad_scale, c->push, st,
                                          maps != nullptr, c->grad_cam ? c->cam_partial.as<double>() : nullptr));
  if (c->n > 0) gs_count_launch();
  if (c->grad_cam) {
    GS_CUDA_TRY(gs_launch_camgrad_finish(c->cam_partial.as<double>(), c->n, c->grad_cam, st));
    gs_count_launch();
  }
  gs_mark(c, 9, st);
  c->ev_bwd_valid = c->timing && c->ev_ok;
  return 0;
}

extern "C" int gs_render_backward(gs_ctx* c, const float* pos, const float* rgb, const float* opa, const float* quat,
                                  const float* scale, const float* image, const float* grad_image, float* grad_pos,
                                  float* grad_rgb, float* grad_opa, float* grad_quat, float* grad_scale,
                                  gs_stream_t stream) {
  return render_backward_impl(c, pos, rgb, opa, quat, scale, image, grad_image, 0, grad_pos, grad_rgb, grad_opa,
                              grad_quat, grad_scale, stream);
}

extern "C" int gs_render_backward_final(gs_ctx* c, const float* pos, const float* rgb, const float* opa,
                                        const float* quat, const float* scale, const float* image_raw_padded,
                                        const float* grad_final, float* grad_pos, float* grad_rgb, float* grad_opa,
                                        float* grad_quat, float* grad_scale, gs_stream_t stream) {
  return render_backward_impl(c, pos, rgb, opa, quat, scale, image_raw_padded, grad_final, 1, grad_pos, grad_rgb,
                              grad_opa, grad_quat, grad_scale, stream);
}

extern "C" int gs_render_forward_maps(gs_ctx* c, const float* pos, const float* rgb, const float* opa, const float* quat,
                                      const float* scale, int n, int d, int scale_activation, const gs_camera* cam,
                                      const float* background_host, float* image_raw_padded, float* depth_raw_padded,
                                      float* alpha_raw_padded, float* image_final, float* depth_final, float* alpha_final,
                                      int64_t* culling_mask, gs_stream_t stream) {
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward_maps: null ctx");
  if (!depth_raw_padded || !alpha_raw_padded)
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward_maps: null depth / alpha plane");
  const bool fin = image_final != nullptr;
  if ((depth_final != nullptr) != fin || (alpha_final != nullptr) != fin)
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward_maps: the three final outputs must be all NULL or all set");
  GsMapsFwd maps{depth_raw_padded, alpha_raw_padded, depth_final, alpha_final, 0.f, 0.f, 0.f};
  if (background_host) {
    maps.bg_r = background_host[0];
    maps.bg_g = background_host[1];
    maps.bg_b = background_host[2];
  }
  return render_forward_impl(c, pos, rgb, opa, quat, scale, n, d, scale_activation, cam, image_raw_padded, image_final,
                             culling_mask, stream, &maps);
}

extern "C" int gs_render_backward_maps(gs_ctx* c, const float* pos, const float* rgb, const float* opa,
                                       const float* quat, const float* scale, const float* image_raw_padded,
                                       const float* depth_raw_padded, const float* alpha_raw_padded,
                                       const float* grad_image, const float* grad_depth, const float* grad_alpha,
                                       int grad_is_final, float* grad_pos, float* grad_rgb, float* grad_opa,
                                       float* grad_quat, float* grad_scale, gs_stream_t stream) {
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_backward_maps: null ctx");
  GsMapsBwd maps{depth_raw_padded, alpha_raw_padded, grad_depth, grad_alpha};
  return render_backward_impl(c, pos, rgb, opa, quat, scale, image_raw_padded, grad_image, grad_is_final ? 1 : 0,
                              grad_pos, grad_rgb, grad_opa, grad_quat, grad_scale, stream, &maps);
}

extern "C" int gs_ctx_set_grad_push(gs_ctx* c, const gs_grad_push* p) {
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_grad_push: null ctx");
  if (!p) {
    c->push = GsGradPush{};
    return 0;
  }
  if (!(p->world == 2 || p->world == 4 || p->world == 8) || p->rank < 0 || p->rank >= p->world || p->per <= 0 ||
      (p->per % 4) || (unsigned long long)p->per * (unsigned)p->world >= (1ull << 32) || !p->bucket ||
      reinterpret_cast<uintptr_t>(p->bucket) % 16)
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_grad_push: bad configuration");
  GsGradPush g{};
  g.bucket = p->bucket;
  g.per = (uint32_t)p->per;
  g.rank = p->rank;
  g.world = p->world;
  for (int k = 0; k < p->world; ++k) {
    if (!p->staging[k] || reinterpret_cast<uintptr_t>(p->staging[k]) % 16)
      return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_grad_push: staging pointers must be 16-byte aligned");
    g.staging[k] = p->staging[k];
  }
  c->push = g;
  return 0;
}

extern "C" int gs_ctx_set_camera_grad(gs_ctx* c, float* grad_cam) {
  // the pointer is checked first so that both refusals need no context
  if (reinterpret_cast<uintptr_t>(grad_cam) % alignof(float))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_camera_grad: grad_cam must be 4-byte aligned");
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_camera_grad: null ctx");
  c->grad_cam = grad_cam;
  return 0;
}

extern "C" int gs_ctx_set_allocator(gs_ctx* c, gs_alloc_fn alloc, gs_free_fn free_fn, void* user) {
  if (!c || ((alloc == nullptr) != (free_fn == nullptr)))
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_allocator: null ctx, or only one of alloc / free given");
  c->allocator.alloc = alloc;        // blocks already held keep the allocator they came from (DevBuf::owner)
  c->allocator.free = free_fn;
  c->allocator.user = user;
  return 0;
}

extern "C" long long gs_frame_instances(gs_ctx* c) { return (c && c->have_forward) ? c->m : -1; }

extern "C" int gs_frame_stats(gs_ctx* c, gs_frame_info* out, gs_stream_t stream) {
  if (!c || !out) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_frame_stats: null argument");
  if (!c->have_forward) return gs_set_error_msg(GS_ERR_NO_FORWARD, "gs_frame_stats: no forward on this ctx");
  cudaStream_t st = (cudaStream_t)stream;
  int T = c->geom.n_tiles;
  int* h = static_cast<int*>(malloc(sizeof(int) * (size_t)(3 * T + 1)));
  if (!h) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_frame_stats: out of host memory");
  unsigned int nvis = 0;
  cudaError_t e = cudaMemcpyAsync(h, c->tile_accum.p, sizeof(int) * (size_t)(T + 1), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(h + T + 1, c->tile_neff.p, sizeof(int) * (size_t)T, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && c->have_backward)
    e = cudaMemcpyAsync(h + 2 * T + 1, c->tile_neff_b.p, sizeof(int) * (size_t)T, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&nvis, c->counters.p, 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    free(h);
    return gs_set_error(e, "gs_frame_stats copy");
  }
  long long meff = 0, meff_b = 0;
  int mx = 0;
  for (int t = 0; t < T; ++t) {
    int cnt = h[t + 1] - h[t];
    if (cnt > mx) mx = cnt;
    meff += h[T + 1 + t];
    if (c->have_backward && cnt > 0) meff_b += h[2 * T + 1 + t];
  }
  free(h);
  out->n_gaussians = c->n;
  out->n_visible = (int)nvis;
  out->n_instances = c->m;
  out->n_instances_eff = meff;
  out->n_instances_eff_bwd = c->have_backward ? meff_b : -1;
  out->width_padded = c->geom.wp;
  out->height_padded = c->geom.hp;
  out->n_tiles = T;
  out->max_tile_count = mx;
  return 0;
}

extern "C" int gs_frame_sorted(gs_ctx* c, int* gauss_idx, long long capacity, int* tile_accum, gs_stream_t stream) {
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_frame_sorted: null ctx");
  if (!c->have_forward) return gs_set_error_msg(GS_ERR_NO_FORWARD, "gs_frame_sorted: no forward on this ctx");
  cudaStream_t st = (cudaStream_t)stream;
  if (gauss_idx && c->m > 0) {
    long long k = capacity < c->m ? capacity : c->m;
    if (k > 0)
      GS_CUDA_TRY(cudaMemcpyAsync(gauss_idx, c->vals_out.p, sizeof(int) * (size_t)k, cudaMemcpyDeviceToDevice, st));
  }
  if (tile_accum)
    GS_CUDA_TRY(cudaMemcpyAsync(tile_accum, c->tile_accum.p, sizeof(int) * (size_t)(c->geom.n_tiles + 1),
                                cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int gs_frame_tile_consumed(gs_ctx* c, int* tile_consumed, gs_stream_t stream) {
  if (!c || !tile_consumed) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_frame_tile_consumed: null argument");
  if (!c->have_forward) return gs_set_error_msg(GS_ERR_NO_FORWARD, "gs_frame_tile_consumed: no forward on this ctx");
  GS_CUDA_TRY(cudaMemcpyAsync(tile_consumed, c->tile_neff.p, sizeof(int) * (size_t)c->geom.n_tiles,
                              cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

extern "C" int gs_render_forward_backward_host(gs_ctx* c, const float* pos, const float* rgb, const float* opa,
                                               const float* quat, const float* scale, int n, int d,
                                               int scale_activation, const gs_camera* cam,
                                               const float* grad_image_host, float* image_host, float* grad_pos,
                                               float* grad_rgb, float* grad_opa, float* grad_quat, float* grad_scale,
                                               gs_stream_t stream) {
  if (!c || !cam || !grad_image_host || !image_host)
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward_backward_host: null argument");
  if (cam->width <= 0 || cam->height <= 0)
    return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_render_forward_backward_host: bad camera");
  cudaStream_t st = (cudaStream_t)stream;
  g_cur_alloc = &c->allocator;
  int wp = (cam->width + GS_TILE - 1) / GS_TILE * GS_TILE, hp = (cam->height + GS_TILE - 1) / GS_TILE * GS_TILE;
  size_t img_bytes = (size_t)wp * hp * 3 * sizeof(float);
  DevBuf& img_dev = c->img_dev;
  DevBuf& gimg_dev = c->gimg_dev;
  GS_CUDA_TRY(img_dev.reserve(img_bytes, st));
  GS_CUDA_TRY(gimg_dev.reserve(img_bytes, st));
  GS_CUDA_TRY(cudaMemcpyAsync(gimg_dev.p, grad_image_host, img_bytes, cudaMemcpyHostToDevice, st));
  int rc = gs_render_forward(c, pos, rgb, opa, quat, scale, n, d, scale_activation, cam, img_dev.as<float>(), nullptr,
                             stream);
  if (rc) return rc;
  rc = gs_render_backward(c, pos, rgb, opa, quat, scale, img_dev.as<float>(), gimg_dev.as<float>(), grad_pos, grad_rgb,
                          grad_opa, grad_quat, grad_scale, stream);
  if (rc) return rc;
  GS_CUDA_TRY(cudaMemcpyAsync(image_host, img_dev.p, img_bytes, cudaMemcpyDeviceToHost, st));
  GS_CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int gs_ctx_set_timing(gs_ctx* c, int enable) {
  if (!c) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_ctx_set_timing: null ctx");
  if (enable && !c->ev_ok) {
    for (cudaEvent_t& e : c->ev) GS_CUDA_TRY(cudaEventCreate(&e));
    c->ev_ok = true;
  }
  c->timing = enable != 0;
  c->ev_fwd_valid = c->ev_bwd_valid = false;
  return 0;
}

extern "C" int gs_frame_stage_ms(gs_ctx* c, float* out, gs_stream_t stream) {
  if (!c || !out) return gs_set_error_msg(GS_ERR_INVALID_ARG, "gs_frame_stage_ms: null argument");
  for (int i = 0; i < GS_N_STAGES; ++i) out[i] = -1.f;
  if (!c->ev_ok) return 0;
  GS_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  if (c->ev_fwd_valid)
    for (int i = 0; i < 6; ++i) GS_CUDA_TRY(cudaEventElapsedTime(&out[i], c->ev[i], c->ev[i + 1]));
  if (c->ev_bwd_valid)
    for (int i = 6; i < 8; ++i) GS_CUDA_TRY(cudaEventElapsedTime(&out[i], c->ev[i + 1], c->ev[i + 2]));
  return 0;
}
