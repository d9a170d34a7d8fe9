"""Shared helpers for the parity tests (CPU oracle <-> CUDA path)."""
import os

import numpy as np
import torch

import gs_oracle as O
import synthetic as S

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def scene(n, w, h, seed=0, k=0, sh_dim=3, opa_range=(0.05, 0.9), sigma_px=(0.6, 5.0)):
    v = S.make_view(w, h, k)
    g = S.make_gaussians(n, w, h, seed, sh_dim, opa_range, sigma_px)
    cam = O.Camera(w, h, v.fx, v.fy, v.rot, v.tran, v.near)
    return g, v, cam


def sorted_instances_cpu(g, cam, thresh=0.05, scale_activation="abs", use_sh=False, dtype=torch.float32):
    """Oracle front-end: activated, culled, binned and exactly sorted per-instance tensors
    (what reference splatter.py hands to `draw`)."""
    p = {k: v.to(dtype) for k, v in g.items()}
    nq, ns, opa_a, rgb_a = O.preactivate(p["quat"], p["scale"], p["opa"], p["rgb"], scale_activation, use_sh)
    rp, rc, mask = O.global_culling(p["pos"], nq, ns, cam.rot.to(dtype), cam.tran.to(dtype), cam.near,
                                    cam.half_w, cam.half_h)
    idx = torch.nonzero(mask.bool()).squeeze(-1)
    p_c, c_c = rp[idx], rc[idx]
    rects = O.tile_rects(p_c[:, :2], c_c, thresh, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                         cam.topmost)
    gi, accum = O.bin_and_sort(p_c, c_c, rects, cam.ntx, cam.nty)
    return dict(pos=p_c[gi].contiguous(), rgb=rgb_a[idx][gi].contiguous(), opa=opa_a[idx][gi].contiguous(),
                cov=c_c[gi].contiguous(), accum=accum, gauss_idx=idx[gi])


def rel_err(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def abs_err(a, b):
    return float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max())


def load_golden(name):
    path = os.path.join(GOLDEN, name)
    if not os.path.exists(path):
        return None
    z = np.load(path)
    return {k: torch.from_numpy(z[k]) for k in z.files}


def require_golden(name):
    """A committed fixture of tests/golden/ (written by tests/golden/make_golden.py); missing is an error."""
    gold = load_golden(name)
    assert gold is not None, f"tests/golden/{name} is missing"
    return gold


def assert_matches_golden_frame(sp, img, gold, img_atol, grad_rtol):
    """A rendered frame and the five parameter gradients of Splatter `sp` against a fixture that
    holds the image on a pixel sample (`pix`, `image`) and the gradients on a row sample (`rows`)."""
    assert abs_err(img.detach().reshape(-1, 3).cpu()[gold["pix"].long()], gold["image"]) < img_atol
    r = gold["rows"].long()
    for name in ("pos", "rgb", "opa", "quat", "scale"):
        assert rel_err(getattr(sp.gaussian_3ds, name).grad.cpu()[r], gold["grad_" + name]) < grad_rtol, name


def device_depth_keys(g, cam, dev, scale_activation="abs"):
    """float32 depth |p_c| of every Gaussian as the CUDA path computes it (legacy
    `global_culling`, same device function as the fused projection); culled rows are 0.  Used as
    the oracle's sort key so that ulp-level depth ties cannot make the two sides order
    differently (the order is only defined up to such ties - SURVEY.md hazard 4)."""
    import renderer
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"], scale_activation)
    rp, _, _ = renderer.global_culling(g["pos"].to(dev), nq.to(dev).contiguous(), ns.to(dev).contiguous(),
                                       cam.rot.to(dev), cam.tran.to(dev), cam.near, cam.half_w, cam.half_h)
    return rp[:, 2].detach().cpu()
