"""Autograd operator boundary — host-side mirror of the reference's renderer.py.

Same public names, positional argument order, return values and zero-fill/ownership
conventions as reference renderer.py (`draw` :89, `trunc_exp` :102,
`world2camera_func` :119, `global_culling` :158), so code written against the
reference keeps working; underneath, every op calls the sm_100a kernels of
libgs_b200 through the `gaussian` extension in this directory.  Additive:
`render_frame`, one autograd node for the whole frame (fused path), and `render_frame_maps`,
the same frame with depth / alpha maps and a background colour.  All three frames also differentiate
the camera pose (`rot`, `tran`) when a pose tensor requires grad (RGB colour only).

The product path never falls back to PyTorch/CPU math: importing this module
without the built extension raises.
"""
from __future__ import annotations

import torch

try:
    import gaussian
except ImportError as e:  # pragma: no cover - fail loudly, never fall back
    raise ImportError(
        "the `gaussian` CUDA extension is not built; run "
        "`python 3d-gaussian-splatting_b200/build.py` (needs nvcc, sm_100a)") from e


def _f32(t):
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


class _Drawer(torch.autograd.Function):
    """Tile blend of sorted per-instance tensors (reference renderer.py:6-87)."""

    @staticmethod
    def forward(ctx, gaussians_pos, gaussians_rgb, gaussians_opa, gaussians_cov, tile_n_point_accum,
                padded_height, padded_width, focal_x, focal_y, render_weight_normalize=False,
                sigmoid=False, use_sh_coeff=False, fast=False, rays_o=None, lefttop_pos=None,
                vec_dx=None, vec_dy=None):
        pos, rgb, opa, cov = (_f32(gaussians_pos), _f32(gaussians_rgb), _f32(gaussians_opa), _f32(gaussians_cov))
        accum = tile_n_point_accum.contiguous()
        image = torch.empty(padded_height, padded_width, 3, device=pos.device, dtype=torch.float32)
        dummy = pos.new_zeros(3)
        rays = [dummy if r is None else _f32(r) for r in (rays_o, lefttop_pos, vec_dx, vec_dy)]
        gaussian.draw(pos, rgb, opa, cov, accum, image, focal_x, focal_y, render_weight_normalize, sigmoid,
                      fast, rays[0], rays[1], rays[2], rays[3], use_sh_coeff)
        ctx.save_for_backward(pos, rgb, opa, cov, accum, image, *rays)
        ctx.cfg = (focal_x, focal_y, render_weight_normalize, sigmoid, fast, use_sh_coeff)
        return image

    @staticmethod
    def backward(ctx, grad_output):
        pos, rgb, opa, cov, accum, image, rays_o, lefttop_pos, vec_dx, vec_dy = ctx.saved_tensors
        focal_x, focal_y, weight_normalize, sigmoid, fast, use_sh_coeff = ctx.cfg
        g_pos = torch.zeros_like(pos)          # z column stays 0 (depth is only a sort key)
        g_rgb = torch.empty_like(rgb)
        g_opa = torch.empty_like(opa)
        g_cov = torch.empty_like(cov)
        gaussian.draw_backward(pos, rgb, opa, cov, accum, image, _f32(grad_output), g_pos, g_rgb, g_opa, g_cov,
                               focal_x, focal_y, weight_normalize, sigmoid, fast, rays_o, lefttop_pos, vec_dx,
                               vec_dy, use_sh_coeff)
        return (g_pos, g_rgb, g_opa, g_cov) + (None,) * 13


draw = _Drawer.apply


class _trunc_exp(torch.autograd.Function):
    """exp with a clamped-gradient backward (reference renderer.py:91-100)."""

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return torch.exp(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * torch.exp(x.clamp(-1, 1))


trunc_exp = _trunc_exp.apply


class _world2camera(torch.autograd.Function):
    """p @ R^T + t and its adjoint (reference renderer.py:104-117; deprecated path)."""

    @staticmethod
    def forward(ctx, pos, rot, tran):
        pos, rot, tran = _f32(pos), _f32(rot), _f32(tran)
        ctx.save_for_backward(rot)
        res = torch.empty_like(pos)
        gaussian.world2camera(pos, rot, tran, res)
        return res

    @staticmethod
    def backward(ctx, grad_out):
        (rot,) = ctx.saved_tensors
        grad_out = _f32(grad_out)
        grad_inp = torch.empty_like(grad_out)
        gaussian.world2camera_backward(grad_out, rot, grad_inp)
        return grad_inp, None, None


world2camera_func = _world2camera.apply


class _GlobalCulling(torch.autograd.Function):
    """Projection + near/frustum cull + 2-D covariance (reference renderer.py:121-156)."""

    @staticmethod
    def forward(ctx, pos, quat, scale, current_rot, current_tran, near, half_width, half_height):
        pos, quat, scale = _f32(pos), _f32(quat), _f32(scale)
        rot, tran = _f32(current_rot), _f32(current_tran)
        n = pos.shape[0]
        res_pos = torch.zeros_like(pos)                       # culled rows must read 0
        res_cov = torch.zeros((n, 2, 2), device=pos.device, dtype=torch.float32)
        culling_mask = torch.zeros(n, dtype=torch.long, device=pos.device)
        gaussian.global_culling(pos, quat, scale, rot, tran, res_pos, res_cov, culling_mask,
                                near, half_width, half_height)
        ctx.save_for_backward(culling_mask, pos, quat, scale, rot, tran)
        ctx.mark_non_differentiable(culling_mask)
        return res_pos, res_cov, culling_mask

    @staticmethod
    def backward(ctx, gradout_pos, gradout_cov, _grad_mask):
        culling_mask, pos, quat, scale, rot, tran = ctx.saved_tensors
        g_pos = torch.zeros_like(pos)
        g_quat = torch.zeros_like(quat)
        g_scale = torch.zeros_like(scale)
        gaussian.global_culling_backward(pos, quat, scale, rot, tran, _f32(gradout_pos), _f32(gradout_cov),
                                         culling_mask, g_pos, g_quat, g_scale)
        return g_pos, g_quat, g_scale, None, None, None, None, None


global_culling = _GlobalCulling.apply


# ----------------------------------------------------------------------------------------
# additive: the whole frame as one autograd node (fused path)
# ----------------------------------------------------------------------------------------
SCALE_ACTIVATIONS = {"abs": 0, "exp": 1}


_flat_grad_allocator = None


def set_flat_grad_allocator(fn):
    """Install `fn(numel, device) -> 1-D fp32 tensor (16-byte aligned)` (or `(tensor, push)` with
    push = (bucket_ptr, staging_ptrs, per, rank) for `RenderContext.set_grad_push`) as the source of the flat
    gradient bucket the fused backward writes into (None restores torch.empty).  Data-parallel
    runs use it to place the bucket in symmetric memory so the gradient exchange runs in place over
    NVLink (dp.NvlsGradBucket): the backward kernel's stores ARE the collective's send buffer."""
    global _flat_grad_allocator
    _flat_grad_allocator = fn


def _flat_grads(tensors):
    """Five gradient views carved out of ONE flat buffer (order pos, rgb, opa, quat, scale; each
    segment 16-byte aligned for the kernel's float4 stores) so that the data-parallel all-reduce
    runs in place on a single bucket (dp.GradBucket)."""
    sizes = [t.numel() for t in tensors]
    starts, o = [], 0
    for n in sizes:
        starts.append(o)
        o += (n + 3) // 4 * 4
    push = None
    if _flat_grad_allocator is not None:
        flat = _flat_grad_allocator(o, tensors[0].device)
        if isinstance(flat, tuple):                      # (bucket, push configuration) - see dp.py
            flat, push = flat
        assert flat.numel() >= o and flat.dtype == torch.float32 and flat.data_ptr() % 16 == 0
    else:
        flat = torch.empty(o, device=tensors[0].device, dtype=torch.float32)
    outs = []
    for t, n, b in zip(tensors, sizes, starts):
        outs.append(flat[b:b + n].view(t.shape))
        if n % 4:
            flat[b + n:b + (n + 3) // 4 * 4].zero_()     # keep the (<= 3 float) pads finite
    return outs, push


def _apply_push(rctx, push):
    """Route this backward's gradient stores: plain bucket, or (data-parallel push) other ranks'
    slices straight into their owners' staging buffers over NVLink (gs_grad_push)."""
    if push is None:
        rctx.clear_grad_push()
    else:
        rctx.set_grad_push(*push)


# positions of rot / tran among the inputs of the three frame Functions (ctx.needs_input_grad)
_ROT, _TRAN = 10, 11


def _save_pose(ctx, rot, tran):
    ctx.pose = [(t.shape, t.dtype, t.device) if isinstance(t, torch.Tensor) else None for t in (rot, tran)]


def _backward_with_pose(ctx, pos, run):
    """Runs `run()` (the context's backward); when rot or tran needs a gradient, the same backward also writes the
    camera gradient (gs_ctx_set_camera_grad, one more kernel), returned as (grad_rot, grad_tran) in each input's
    shape, dtype and device.  Otherwise nothing changes and (None, None) is returned."""
    want = [ctx.needs_input_grad[_ROT], ctx.needs_input_grad[_TRAN]]
    if not any(want):
        run()
        return None, None
    gcam = torch.empty(12, device=pos.device, dtype=torch.float32)
    ctx.rctx.set_camera_grad(gcam)
    try:
        run()
    finally:
        ctx.rctx.set_camera_grad(None)
    out = []
    for w, part, meta in zip(want, (gcam[:9], gcam[9:]), ctx.pose):
        out.append(part.reshape(meta[0]).to(dtype=meta[1], device=meta[2]) if w else None)
    return tuple(out)


class _RenderFrame(torch.autograd.Function):
    """raw parameters -> padded un-clamped image, replacing splatter.py:513-634's glue.

    `rctx` is a `gaussian.RenderContext` (owns device workspaces; holds the state of
    the latest forward, so backward must run before the next forward on the same ctx).
    """

    @staticmethod
    def forward(ctx, rctx, pos, rgb, opa, quat, scale, width, height, focal_x, focal_y, rot, tran,
                near, tile_thresh, scale_activation):
        pos, rgb, opa, quat, scale = (_f32(t.detach()) for t in (pos, rgb, opa, quat, scale))
        image, mask = rctx.forward(pos, rgb, opa, quat, scale, int(width), int(height), float(focal_x),
                                   float(focal_y), rot.detach().cpu(), tran.detach().cpu(), float(near),
                                   float(tile_thresh), SCALE_ACTIVATIONS[scale_activation])
        ctx.rctx = rctx
        ctx.frame = rctx.frame_id()
        _save_pose(ctx, rot, tran)
        ctx.save_for_backward(pos, rgb, opa, quat, scale, image)
        ctx.mark_non_differentiable(mask)
        return image, mask

    @staticmethod
    def backward(ctx, grad_image, _grad_mask):
        pos, rgb, opa, quat, scale, image = ctx.saved_tensors
        outs, push = _flat_grads((pos, rgb, opa, quat, scale))
        _apply_push(ctx.rctx, push)
        g_rot, g_tran = _backward_with_pose(
            ctx, pos, lambda: ctx.rctx.backward_into(pos, rgb, opa, quat, scale, image, _f32(grad_image), *outs,
                                                     ctx.frame))
        return (None, outs[0], outs[1], outs[2], outs[3], outs[4]) + (None,) * 4 + (g_rot, g_tran) + (None,) * 3


render_frame = _RenderFrame.apply


class _RenderFrameFinal(torch.autograd.Function):
    """Like `render_frame`, with reference splatter.py:652-653 (clamp to [0,1] + centre crop)
    fused into the blend kernels: returns the final HxWx3 image; backward consumes its gradient
    directly (no clamp / pad kernels, no padded gradient image)."""

    @staticmethod
    def forward(ctx, rctx, pos, rgb, opa, quat, scale, width, height, focal_x, focal_y, rot, tran,
                near, tile_thresh, scale_activation):
        pos, rgb, opa, quat, scale = (_f32(t.detach()) for t in (pos, rgb, opa, quat, scale))
        final, raw, mask = rctx.forward_final(pos, rgb, opa, quat, scale, int(width), int(height), float(focal_x),
                                              float(focal_y), rot.detach().cpu(), tran.detach().cpu(), float(near),
                                              float(tile_thresh), SCALE_ACTIVATIONS[scale_activation])
        ctx.rctx = rctx
        ctx.frame = rctx.frame_id()
        _save_pose(ctx, rot, tran)
        ctx.save_for_backward(pos, rgb, opa, quat, scale, raw)
        ctx.mark_non_differentiable(mask)
        return final, mask

    @staticmethod
    def backward(ctx, grad_final, _grad_mask):
        pos, rgb, opa, quat, scale, raw = ctx.saved_tensors
        outs, push = _flat_grads((pos, rgb, opa, quat, scale))
        _apply_push(ctx.rctx, push)
        g_rot, g_tran = _backward_with_pose(
            ctx, pos, lambda: ctx.rctx.backward_final_into(pos, rgb, opa, quat, scale, raw, _f32(grad_final), *outs,
                                                           ctx.frame))
        return (None, outs[0], outs[1], outs[2], outs[3], outs[4]) + (None,) * 4 + (g_rot, g_tran) + (None,) * 3


render_frame_final = _RenderFrameFinal.apply


class _RenderFrameMaps(torch.autograd.Function):
    """The frame of `render_frame` / `render_frame_final` plus a depth map (sum_i w_i |p_c,i|, not normalised), an
    alpha map (1 - T_end) and a constant background colour (image += T_end * bg), all from the blend kernels in one
    pass.  final=True: crop(clamp(image)) [H,W,3], crop(depth), crop(alpha) [H,W] (maps not clamped); else the
    padded raw planes.  RGB colour only; the background gets no gradient."""

    @staticmethod
    def forward(ctx, rctx, pos, rgb, opa, quat, scale, width, height, focal_x, focal_y, rot, tran,
                near, tile_thresh, scale_activation, background, final):
        pos, rgb, opa, quat, scale = (_f32(t.detach()) for t in (pos, rgb, opa, quat, scale))
        image, depth, alpha, raw, draw_, araw, mask = rctx.forward_maps(
            pos, rgb, opa, quat, scale, int(width), int(height), float(focal_x), float(focal_y), rot.detach().cpu(),
            tran.detach().cpu(), float(near), float(tile_thresh), SCALE_ACTIVATIONS[scale_activation], background,
            bool(final))
        ctx.rctx = rctx
        ctx.frame = rctx.frame_id()
        _save_pose(ctx, rot, tran)
        ctx.final = bool(final)
        ctx.save_for_backward(pos, rgb, opa, quat, scale, raw, draw_, araw)
        ctx.mark_non_differentiable(mask)
        return image, depth, alpha, mask

    @staticmethod
    def backward(ctx, grad_image, grad_depth, grad_alpha, _grad_mask):
        # autograd hands zeros for an output that received no gradient (materialised grads)
        pos, rgb, opa, quat, scale, raw, draw_, araw = ctx.saved_tensors
        outs, push = _flat_grads((pos, rgb, opa, quat, scale))
        _apply_push(ctx.rctx, push)
        g_rot, g_tran = _backward_with_pose(
            ctx, pos, lambda: ctx.rctx.backward_maps_into(pos, rgb, opa, quat, scale, raw, draw_, araw,
                                                          _f32(grad_image), _f32(grad_depth), _f32(grad_alpha),
                                                          ctx.final, *outs, ctx.frame))
        return (None, outs[0], outs[1], outs[2], outs[3], outs[4]) + (None,) * 4 + (g_rot, g_tran) + (None,) * 5


def render_frame_maps(rctx, pos, rgb, opa, quat, scale, width, height, focal_x, focal_y, rot, tran, near,
                      tile_thresh, scale_activation, background=None, final=True):
    """One autograd node: raw parameters -> (image, depth, alpha, culling_mask).  `background`: None (black) or
    three floats.  A None gradient for any of the three images counts as zeros.  See `_RenderFrameMaps`."""
    bg = None if background is None else [float(x) for x in background]
    if bg is not None and len(bg) != 3:
        raise ValueError("background must have 3 values (r, g, b)")
    return _RenderFrameMaps.apply(rctx, pos, rgb, opa, quat, scale, width, height, focal_x, focal_y, rot, tran, near,
                                  tile_thresh, scale_activation, bg, final)
