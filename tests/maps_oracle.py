"""CPU oracle for the depth / alpha maps and the background colour of a maps frame
(`renderer.render_frame_maps`, `Splatter.render_maps`, gs_render_forward_maps).

An extension of `gs_oracle` (the reference composites colour on black only and has no maps), kept
beside the tests so that the pinned oracle stays as it is.  It adds no blend of its own: depth and
alpha are two more colour channels whose per-instance "colours" are d_i = |p_c,i| and 1, so both
maps are `gs_oracle.draw` of the colour rows (d_i, 1, 0) over the same sorted instances - same
weights w_i, same constant early-stop mask - and the background enters as (1 - alpha) * bg.  The
front end (activations, projection, culling, binning, exact (tile, depth, id) order) is
`gs_oracle`'s too.  Gradients come from autograd (fp64 in the tests).  RGB colour only, like the
kernels.
"""
from __future__ import annotations

import torch

import gs_oracle as O


def draw_maps(pos, rgb, opa, cov, depth, tile_n_point_accum, Hp, Wp, fx, fy, background=None, tiles=None):
    """Blend sorted per-instance tensors (pos[M,3], rgb[M,3] activated, opa[M] activated, cov[M,2,2],
    depth[M]).  Returns (image[Hp,Wp,3] = sum w c + T_end bg, depth[Hp,Wp] = sum w d,
    alpha[Hp,Wp] = sum w = 1 - T_end).  Tiles outside `tiles` are not blended: depth and alpha 0 there."""
    img = O.draw(pos, rgb, opa, cov, tile_n_point_accum, Hp, Wp, fx, fy, tiles=tiles)
    rows = torch.stack([depth, torch.ones_like(depth), torch.zeros_like(depth)], dim=-1)
    da = O.draw(pos, rows, opa, cov, tile_n_point_accum, Hp, Wp, fx, fy, tiles=tiles)
    dmap, amap = da[..., 0], da[..., 1]
    if background is not None:
        bg = torch.as_tensor(background, dtype=img.dtype).reshape(1, 1, 3)
        img = img + (1 - amap).unsqueeze(-1) * bg
    return img, dmap, amap


def crop2(cam: O.Camera, m):
    """Centre crop of an [Hp,Wp] plane (splatter.py:267-272), no clamp."""
    return cam.crop(m.unsqueeze(-1)).squeeze(-1)


def render_maps(pos, rgb, opa, quat, scale, cam: O.Camera, thresh=0.05, scale_activation="abs", background=None,
                tiles=None, depth_key=None, detach_depth=False, return_aux=False):
    """A maps frame on raw parameters: (crop(clamp(image)) [H,W,3], crop(depth) [H,W], crop(alpha) [H,W]).
    d_i = |p_c,i| = global_culling's res_pos[:,2]; `detach_depth` cuts its direct gradient to pos (tests isolate
    that term by differencing)."""
    dt = pos.dtype
    rot, tran = cam.rot.to(dt), cam.tran.to(dt)
    nq, ns, opa_a, rgb_a = O.preactivate(quat, scale, opa, rgb, scale_activation)
    rp, rc, mask = O.global_culling(pos, nq, ns, rot, tran, cam.near, cam.half_w, cam.half_h)
    idx = torch.nonzero(mask.bool()).squeeze(-1)
    p_c, c_c, rgb_c, opa_c = rp[idx], rc[idx], rgb_a[idx], opa_a[idx]
    rects = O.tile_rects(p_c[:, :2], c_c, thresh, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                         cam.topmost)
    gi, accum = O.bin_and_sort(p_c, c_c, rects, cam.ntx, cam.nty, None if depth_key is None else depth_key[idx])
    d_c = p_c[:, 2].detach() if detach_depth else p_c[:, 2]
    gd, acc_d = gi, accum
    if tiles is not None:                  # gather only the instances of the requested tiles
        a64 = accum.to(torch.int64)
        keep = torch.zeros(a64.numel() - 1, dtype=torch.int64)
        parts = []
        for t in sorted(int(x) for x in tiles):
            parts.append(gi[int(a64[t]):int(a64[t + 1])])
            keep[t] = int(a64[t + 1] - a64[t])
        gd = torch.cat(parts) if parts else gi[:0]
        acc_d = torch.zeros_like(a64)
        acc_d[1:] = torch.cumsum(keep, 0)
    img, dmap, amap = draw_maps(p_c[gd], rgb_c[gd], opa_c[gd], c_c[gd], d_c[gd], acc_d, cam.Hp, cam.Wp, cam.fx,
                                cam.fy, background, tiles)
    out = (cam.crop(torch.clamp(img, 0, 1)), crop2(cam, dmap), crop2(cam, amap))
    if return_aux:
        return out + (dict(padded=img, padded_depth=dmap, padded_alpha=amap, mask=mask, accum=accum,
                           gauss_idx=idx[gi]),)
    return out
