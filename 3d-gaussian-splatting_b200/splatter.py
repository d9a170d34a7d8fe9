"""Scene + per-frame pipeline: host-side mirror of the reference's `Splatter`
(reference splatter.py:323-655) on top of the fused B200 frame path.

Same constructor as the reference (`Splatter(colmap_path, image_path, near=..., ...)`,
splatter.py:324-345) and the surface train.py / visergui.py touch (train.py:57-61,:67,:99,:150,
:161-171,:190,:198-199,:234; visergui.py:137-149): `gaussian_3ds.{pos,rgb,opa,quat,scale}`
(nn.Parameters; opa / rgb logits, wxyz quaternion, raw scale), `gaussian_3ds.adaptive_control`,
`reset_opa`, `forward(camera_id, extrinsics, intrinsics)` -> clamped, centre-cropped HxWx3 image,
`ground_truth`, `imgs`, `culling_mask` (int64), `n_tile_gaussians`, `n_gaussians`, `device`,
`scale_activation`, `set_camera`, `switch_resolution`.  Additionally
`Splatter.from_tensors(gaussians, views, ...)` builds a scene without COLMAP (synthetic
benchmarks / tests) and `render_maps(...)` returns depth and alpha maps with the image, over an
optional background colour.

The per-frame work of reference `project_and_culling` + `render` (:513-634: 4 boolean-mask
compactions, the dense [T, N/20] list, cumsum, two 4-tensor gathers, fp32-key sort, >= 7 host
syncs) and the clamp + crop of `forward` (:652-653) is ONE autograd node here
(`renderer.render_frame_final`).
"""
from __future__ import annotations

import math
import os
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

import gaussian
from renderer import render_frame, render_frame_final, render_frame_maps

EPS = 1e-4
SH_C0 = 0.28209479177387814


def inverse_sigmoid(y):
    return -math.log(1 / y - 1)


def quat_to_rotmat(q):
    """wxyz -> R (reference utils.py:318-333)."""
    w, x, y, z = q.unbind(-1)
    return torch.stack([1 - 2 * y * y - 2 * z * z, 2 * x * y - 2 * z * w, 2 * x * z + 2 * y * w,
                        2 * x * y + 2 * z * w, 1 - 2 * x * x - 2 * z * z, 2 * y * z - 2 * x * w,
                        2 * x * z - 2 * y * w, 2 * y * z + 2 * x * w, 1 - 2 * x * x - 2 * y * y],
                       dim=-1).reshape(q.shape[:-1] + (3, 3))


class Gaussian3ds(nn.Module):
    """Parameter holder + densification (reference splatter.py:39-228, init_values=True branch)."""

    def __init__(self, pos, rgb, opa, quat, scale):
        super().__init__()
        self.pos = nn.Parameter(pos)
        self.rgb = nn.Parameter(rgb)
        self.opa = nn.Parameter(opa)
        self.quat = nn.Parameter(quat)
        self.scale = nn.Parameter(scale)

    def reset_opa(self):                                        # reference splatter.py:119-120
        with torch.no_grad():
            self.opa.fill_(inverse_sigmoid(0.01))

    def get_gaussian_3d_cov(self, scale_activation="abs"):      # reference splatter.py:100-114
        R = quat_to_rotmat(self.quat)
        s = self.scale.abs() + EPS if scale_activation == "abs" else torch.exp(self.scale)
        RS = R * s.unsqueeze(-2)
        return RS @ RS.transpose(-1, -2)

    @torch.no_grad()
    def adaptive_control(self, grad, taus, delete_thresh, scale_activation="abs", grad_thresh=0.0002,
                         grad_aggregation="max", use_clone=True, use_split=True, clone_dt=0.01, generator=None):
        """Prune / clone / split (reference splatter.py:122-228, same signature as train.py:160-171 calls it):
        delete Gaussians with opacity below sigmoid^-1(0.02) or a scale norm above `delete_thresh`; where the
        accumulated position gradient exceeds `grad_thresh`, clone the small ones (moved against the gradient)
        and split the large ones (scale / 1.6, two positions sampled from the un-shrunk Gaussian itself).
        Runs on the device (`gaussian.densify`: classify -> scans -> one kernel that writes the new arrays);
        the split samples come from torch's CUDA generator, so data-parallel replicas that seed torch
        identically stay identical.  Parameters are re-created: the caller rebuilds its optimizer
        (train.py:173-181)."""
        if scale_activation not in ("abs", "exp"):
            raise ValueError("scale_activation must be 'abs' or 'exp'")
        if grad_aggregation not in ("max", "mean"):
            raise ValueError("grad_aggregation must be 'max' or 'mean'")
        g = grad.detach()
        if g.dtype != torch.float32 or not g.is_contiguous():
            g = g.float().contiguous()
        args = [t.detach().contiguous() for t in (self.pos, self.rgb, self.opa, self.quat, self.scale)]
        new, (n_deleted, n_clone, n_split) = gaussian.densify(
            *args, g, 0 if scale_activation == "abs" else 1, inverse_sigmoid(0.02), float(delete_thresh),
            float(grad_thresh), grad_aggregation == "max", float(taus), bool(use_clone), bool(use_split),
            float(clone_dt), generator)
        self.pos, self.rgb, self.opa, self.quat, self.scale = (nn.Parameter(t) for t in new)
        return dict(deleted=int(n_deleted), cloned=int(n_clone), split=int(n_split), total=self.pos.shape[0])


class Tiles:
    """Padded render-target geometry (reference splatter.py:255-272)."""

    def __init__(self, width, height, focal_x, focal_y):
        self.width, self.height = int(width), int(height)
        self.padded_width = int(math.ceil(self.width / 16)) * 16
        self.padded_height = int(math.ceil(self.height / 16)) * 16
        self.focal_x, self.focal_y = float(focal_x), float(focal_y)
        self.n_tile_x = self.padded_width // 16
        self.n_tile_y = self.padded_height // 16

    def __len__(self):
        return self.n_tile_x * self.n_tile_y

    def crop(self, image):
        top = (self.padded_height - self.height) // 2
        left = (self.padded_width - self.width) // 2
        return image[top:top + self.height, left:left + self.width, :]


class Splatter(nn.Module):
    def __init__(self, colmap_path, image_path, near=0.3, jacobian_calc="cuda", render_downsample=1,
                 use_sh_coeff=False, render_weight_normalize=False, opa_init_value=0.1, scale_init_value=0.02,
                 tile_culling_method="prob2", tile_culling_dist_thresh=0.5, tile_culling_prob_thresh=0.1,
                 debug=0, scale_activation="abs", cudaculling=1, load_ckpt=None, debug_align=False,
                 fast_drawing=True, test=False, images: Optional[List[torch.Tensor]] = None, device=None):
        """Reference signature (splatter.py:324-345).  `colmap_path` may also be a dict of raw
        parameter tensors (pos, rgb, opa, quat, scale) with `image_path` a list of view dicts
        (width, height, focal_x, focal_y, rot[3,3], tran[3]) - see `from_tensors`.

        Options that selected slower variants of the same maths in the reference are accepted and
        ignored (`jacobian_calc`, `cudaculling`, `fast_drawing`, `debug`, `debug_align`); options
        whose result would differ are refused (`render_weight_normalize`, tile culling methods other
        than "prob2", which is train.py's default, train.py:311)."""
        super().__init__()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if render_weight_normalize:
            raise NotImplementedError("render_weight_normalize is not supported (the reference never enables it)")
        if tile_culling_method != "prob2":
            raise NotImplementedError("the fused path implements tile_culling_method='prob2' (train.py's default); "
                                      "methods 'dist' / 'prob' are available through gaussian.calc_tile_list")
        self.use_sh_coeff = bool(use_sh_coeff)
        self.near = near
        self.render_downsample = render_downsample
        self.tile_culling_method = tile_culling_method
        self.tile_culling_prob_thresh = tile_culling_prob_thresh
        self.scale_activation = scale_activation
        self.debug = debug
        self.test = test
        self.imgs: List[torch.Tensor] = []
        self.views: List[dict] = []
        if isinstance(colmap_path, dict):
            params = {k: colmap_path[k] for k in ("pos", "rgb", "opa", "quat", "scale")}
            self._set_views(image_path)
            self.imgs = [] if images is None else [im.to(self.device) for im in images]
        else:
            params = self._load_colmap(colmap_path, image_path, opa_init_value, scale_init_value)
        if load_ckpt is not None:                                   # reference splatter.py:417-424
            ckpt = torch.load(load_ckpt, map_location="cpu", weights_only=False)   # nn.Parameters, train.py:284-290
            params = {k: ckpt[k].detach() for k in ("pos", "rgb", "opa", "quat", "scale")}
        if self.use_sh_coeff != (params["rgb"].shape[1] != 3):
            raise ValueError("use_sh_coeff must match the colour width (3 = RGB logits, 27 / 48 = SH)")
        to = dict(device=self.device, dtype=torch.float32)
        self.gaussian_3ds = Gaussian3ds(*(params[k].detach().to(**to).contiguous()
                                         for k in ("pos", "rgb", "opa", "quat", "scale")))
        with torch.cuda.device(self.device):                      # the context lives on self.device, not on the current one
            self._rctx = gaussian.RenderContext()
        self.ground_truth = None
        self.culling_mask = None
        self.n_tile_gaussians = 0
        self.n_gaussians = self.gaussian_3ds.pos.shape[0]
        self.current_view = None
        self.current_camera = None
        self.tile_info = None
        if self.views and not self.test:
            self.set_camera(0)

    @classmethod
    def from_tensors(cls, gaussians, views, images=None, **kw):
        kw.setdefault("tile_culling_prob_thresh", 0.05)            # train.py:310
        return cls(gaussians, views, images=images, **kw)

    # -- scene loading ----------------------------------------------------------------------
    def _set_views(self, views: Sequence[dict]):
        self.views = [dict(v) for v in views]
        for v in self.views:                     # the camera is host data
            v["rot"] = torch.as_tensor(np.asarray(v["rot"]), dtype=torch.float32).cpu().contiguous()
            v["tran"] = torch.as_tensor(np.asarray(v["tran"]), dtype=torch.float32).cpu().contiguous()

    def _load_colmap(self, colmap_path, image_path, opa_init_value, scale_init_value):
        """reference splatter.py:363-412: points -> parameters (colour logits, opacity logit,
        identity rotation, scale = mean distance to the 3 nearest neighbours x scale_init_value)."""
        import colmap_io
        from scipy.spatial import cKDTree
        self.colmap_path, self.image_path = colmap_path, image_path
        self.cameras = colmap_io.read_cameras_binary(os.path.join(colmap_path, "cameras.bin"))
        self.images_info = colmap_io.read_images_binary(os.path.join(colmap_path, "images.bin"))
        pts = colmap_io.read_points3d_binary(os.path.join(colmap_path, "points3D.bin"))
        if not self.test:
            self.parse_imgs()
        xyz = np.stack([p.xyz for p in pts.values()]).astype(np.float32)
        rgb = np.stack([p.rgb for p in pts.values()]).astype(np.float32) / 255.0
        rgb = np.clip(rgb, 1e-4, 1 - 1e-4)
        logit = torch.from_numpy(-np.log(1 / rgb - 1))
        if self.use_sh_coeff:                                      # utils.py:345-348
            sh = torch.zeros(len(xyz), 3, 9)
            sh[:, :, 0] = logit / SH_C0
            colour = sh.flatten(1)
        else:
            colour = logit
        dist, _ = cKDTree(xyz).query(xyz, k=4)
        s = torch.from_numpy(dist[:, 1:].mean(axis=1).astype(np.float32)) * scale_init_value
        if self.scale_activation == "exp":
            s = s.log()
        n = len(xyz)
        return dict(pos=torch.from_numpy(xyz), rgb=colour.float(),
                    opa=torch.full((n,), inverse_sigmoid(opa_init_value)),
                    quat=torch.tensor([1.0, 0, 0, 0]).repeat(n, 1), scale=s.unsqueeze(1).repeat(1, 3))

    def parse_imgs(self):
        """reference splatter.py:429-452: every registered image that exists on disk becomes a view
        (w2c pose from COLMAP's qvec / tvec) with its uint8 ground truth kept on the GPU."""
        import colmap_io
        import cv2
        self.imgs, views = [], []
        for img_id in sorted(self.images_info):
            info = self.images_info[img_id]
            cam = self.cameras[info.camera_id]
            fn = os.path.join(self.image_path, info.name)
            if not os.path.exists(fn):
                continue
            im = cv2.cvtColor(cv2.imread(fn), cv2.COLOR_BGR2RGB)
            self.imgs.append(torch.from_numpy(im).to(torch.uint8).to(self.device))
            fy = cam.params[1] if cam.model != "SIMPLE_PINHOLE" else cam.params[0]
            views.append(dict(width=im.shape[1], height=im.shape[0], focal_x=cam.params[0] / self.render_downsample,
                              focal_y=fy / self.render_downsample, rot=colmap_io.qvec_to_rotmat(info.qvec),
                              tran=np.asarray(info.tvec), camera_id=info.camera_id))
        self._set_views(views)

    def switch_resolution(self, downsample_factor):                 # reference splatter.py:454-463
        if downsample_factor == self.render_downsample:
            return
        self.image_path = self.image_path.replace(f"images_{self.render_downsample}", f"images_{downsample_factor}")
        self.render_downsample = downsample_factor
        self.parse_imgs()
        self.current_camera = None
        self.set_camera(0)

    # -- camera -----------------------------------------------------------------------------
    def set_camera(self, idx, extrinsics=None, intrinsics=None):
        """reference splatter.py:465-511 (idx=None: free camera from the GUI).  On the free-camera path, torch
        tensors in `extrinsics` reach the renderer as they are, so a pose that requires grad receives gradients
        (pose refinement; the kernels get a host copy); other array types become constant float32 host tensors.
        Views addressed by index keep their stored constant pose."""
        if idx is None:
            def pose(x):
                if isinstance(x, torch.Tensor):
                    return x
                return torch.as_tensor(np.asarray(x), dtype=torch.float32).cpu().contiguous()
            v = dict(width=int(math.ceil(intrinsics["width"])), height=int(math.ceil(intrinsics["height"])),
                     focal_x=float(intrinsics["focal_x"]), focal_y=float(intrinsics["focal_y"]),
                     rot=pose(extrinsics["rot"]), tran=pose(extrinsics["tran"]))
            self.ground_truth = None
        else:
            v = self.views[idx]
            self.ground_truth = (self.imgs[idx].to(torch.float16) / 255.) if idx < len(self.imgs) else None
        self.current_view = self.current_camera = v
        self.current_w2c_rot = v["rot"]
        self.current_w2c_tran = v["tran"]
        self.tile_info = Tiles(v["width"], v["height"], v["focal_x"], v["focal_y"])

    # -- frame ------------------------------------------------------------------------------
    def render_padded(self):
        """Padded, un-clamped image (what reference `render` returns, splatter.py:563-634)."""
        g, v = self.gaussian_3ds, self.current_view
        image, mask = render_frame(self._rctx, g.pos, g.rgb, g.opa, g.quat, g.scale, v["width"], v["height"],
                                   v["focal_x"], v["focal_y"], v["rot"], v["tran"], self.near,
                                   self.tile_culling_prob_thresh, self.scale_activation)
        self.culling_mask = mask
        self.n_gaussians = g.pos.shape[0]
        return image

    def forward(self, camera_id=None, extrinsics=None, intrinsics=None):
        """reference splatter.py:643-655; clamp(0,1) + centre crop (:652-653) run inside the blend
        kernels (`render_frame_final`)."""
        self.set_camera(camera_id, extrinsics, intrinsics)
        g, v = self.gaussian_3ds, self.current_view
        image, mask = render_frame_final(self._rctx, g.pos, g.rgb, g.opa, g.quat, g.scale, v["width"], v["height"],
                                         v["focal_x"], v["focal_y"], v["rot"], v["tran"], self.near,
                                         self.tile_culling_prob_thresh, self.scale_activation)
        self.culling_mask = mask
        self.n_gaussians = g.pos.shape[0]
        self.n_tile_gaussians = self._rctx.last_instances()         # train.py:198 reads it every step
        return image

    def render_maps(self, camera_id=None, extrinsics=None, intrinsics=None, background=None):
        """Like `forward`, plus the depth and alpha maps, over an optional constant background colour
        (three floats; None = black, i.e. `forward`'s image).  Returns (image [H,W,3] clamped to [0,1],
        depth [H,W] = sum_i w_i |p_c,i| (not normalised: expected depth = depth / alpha), alpha [H,W] =
        1 - final transmittance), all differentiable; the maps are not clamped.  RGB colour only."""
        self.set_camera(camera_id, extrinsics, intrinsics)
        g, v = self.gaussian_3ds, self.current_view
        image, depth, alpha, mask = render_frame_maps(self._rctx, g.pos, g.rgb, g.opa, g.quat, g.scale, v["width"],
                                                      v["height"], v["focal_x"], v["focal_y"], v["rot"], v["tran"],
                                                      self.near, self.tile_culling_prob_thresh, self.scale_activation,
                                                      background=background, final=True)
        self.culling_mask = mask
        self.n_gaussians = g.pos.shape[0]
        self.n_tile_gaussians = self._rctx.last_instances()
        return image, depth, alpha

    def forward_unfused_post(self, camera_id=None, extrinsics=None, intrinsics=None):
        """Same image through the padded raw render + torch clamp/crop (kept for cross-checks)."""
        self.set_camera(camera_id, extrinsics, intrinsics)
        padded = self.render_padded()
        return self.tile_info.crop(torch.clamp(padded, 0, 1))

    def save_checkpoint(self, path, optimizer=None, iteration=None, trainer_state=None):
        """reference Trainer.save_checkpoint (train.py:283-291) + resume state; see checkpoint.py."""
        import checkpoint
        return checkpoint.save_checkpoint(self, path, optimizer, iteration, trainer_state)

    def frame_stats(self):
        s = self._rctx.stats()
        self.n_tile_gaussians = int(s["n_instances"])
        return s
