"""GPU checks of the camera pose gradient: pose tensors that require grad on the free-camera path of `Splatter`
(`forward`, `render_maps`), through `gs_ctx_set_camera_grad`, against autograd of the fp64 oracle with respect to the
camera's `rot` / `tran` (J detached, as for every other gradient); plus identities, determinism, launch counts,
refusals and an end-to-end pose recovery."""
import math

import pytest
import torch

import gs_oracle as O
import maps_oracle as MO
import synthetic as S
from helpers import device_depth_keys, rel_err, scene

pytestmark = pytest.mark.gpu

CAM_RTOL = 1e-3
NAMES = ("pos", "rgb", "opa", "quat", "scale")
BG = (0.2, 0.5, 1.0)
CONFIGS = [
    (2000, 128, 96, 0, (0.005, 0.05)),     # safe regime, no saturation
    (10000, 256, 256, 0, (0.05, 0.9)),     # C1
    (8000, 200, 120, 2, (0.05, 0.9)),      # rotated view (culling), non-multiple-of-16 size
    (5000, 96, 64, 0, (0.6, 0.98)),        # opaque: early termination everywhere
]


def _splatter(g, views, dev, **kw):
    import splatter
    vs = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran) for v in views]
    return splatter.Splatter.from_tensors(g, vs, device=dev, **kw)


def _intr(v):
    return dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy)


def _pose(v, dev=None, grad=True):
    rot = v.rot.clone().to(dev or "cpu").requires_grad_(grad)
    tran = v.tran.clone().to(dev or "cpu").requires_grad_(grad)
    return rot, tran


def _upstream(h, w, seed=0):
    gi = S.make_grad_output(h, w, seed) * (h * w)
    gen = torch.Generator().manual_seed(seed + 11)
    return gi, torch.rand(h, w, generator=gen) * 2 - 1, torch.rand(h, w, generator=gen) * 2 - 1


def _oracle(g, cam, ups, maps, tiles=None):
    """(grad_cam[12] fp64, parameter grads) of <ups, outputs> through the oracle, pose as leaves."""
    rot = cam.rot.double().clone().requires_grad_(True)
    tran = cam.tran.double().clone().requires_grad_(True)
    c2 = O.Camera(cam.width, cam.height, cam.fx, cam.fy, rot, tran, cam.near)
    p = {k: v.double().clone().requires_grad_(True) for k, v in g.items()}
    dk = device_depth_keys(g, cam, torch.device("cuda", 0))
    if maps:
        outs = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], c2, background=BG, tiles=tiles,
                              depth_key=dk)
        loss = sum((o * u.double()).sum() for o, u in zip(outs, ups))
    else:
        out = O.render(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], c2, tiles=tiles, depth_key=dk)
        loss = (out * ups[0].double()).sum()
    loss.backward()
    grads = {k: (p[k].grad if p[k].grad is not None else torch.zeros_like(p[k])) for k in p}
    return torch.cat([rot.grad.reshape(-1), tran.grad]), grads


def _run(sp, v, ups, maps, pose, dev):
    """Forward + backward on the free-camera path; returns (grad_cam or None, parameter grads)."""
    for p in sp.gaussian_3ds.parameters():
        p.grad = None
    rot, tran = pose
    ex = dict(rot=rot, tran=tran)
    if maps:
        outs = sp.render_maps(None, extrinsics=ex, intrinsics=_intr(v), background=BG)
        torch.autograd.backward(list(outs), [u.to(dev) for u in ups])
    else:
        sp(None, extrinsics=ex, intrinsics=_intr(v)).backward(ups[0].to(dev))
    gcam = None
    if rot.requires_grad or tran.requires_grad:    # a pose part without requires_grad reads as zeros here
        gcam = torch.cat([(t.grad if t.grad is not None else torch.zeros_like(t)).detach().cpu().reshape(-1)
                          for t in (rot, tran)])
    return gcam, [getattr(sp.gaussian_3ds, n).grad.clone() for n in NAMES]


@pytest.mark.parametrize("maps", [False, True], ids=["final", "maps+bg"])
@pytest.mark.parametrize("n,w,h,k,opa", CONFIGS, ids=["safe", "C1", "rotated", "opaque"])
def test_camera_grad_vs_oracle(gs, cuda, n, w, h, k, opa, maps):
    g, v, cam = scene(n, w, h, k=k, opa_range=opa)
    ups = _upstream(h, w)
    ocam, _ = _oracle(g, cam, ups, maps)
    sp = _splatter(g, [v], cuda)
    pose = _pose(v)
    gcam, grads = _run(sp, v, ups, maps, pose, cuda)
    assert pose[0].grad.shape == (3, 3) and pose[1].grad.shape == (3,) and gcam.dtype == torch.float32
    err = rel_err(gcam, ocam)
    print(f"camera gradient rel err {err:.2e}")
    assert err < CAM_RTOL, (gcam, ocam)
    # the five parameter gradients are those of a run without camera gradients
    _, ref = _run(sp, v, ups, maps, _pose(v, grad=False), cuda)
    print(f"parameter gradients bit-equal with / without camera gradients: "
          f"{all(torch.equal(a, b) for a, b in zip(grads, ref))}")
    for name, a, b in zip(NAMES, grads, ref):
        assert rel_err(a, b) < 1e-6, name


def test_camera_grad_packed_path_matches_gather(gs, cuda):
    """The projection backward is shared: the packed path (gs_tune("gather", 0)) gives the same camera gradient."""
    gaussian, _ = gs
    n, w, h = 8000, 200, 120
    g, v, _ = scene(n, w, h, k=2)
    ups = _upstream(h, w)
    sp = _splatter(g, [v], cuda)
    gather, _ = _run(sp, v, ups, False, _pose(v), cuda)
    old = gaussian.tuned("gather")
    gaussian.tune("gather", 0)
    try:
        packed, _ = _run(sp, v, ups, False, _pose(v), cuda)
    finally:
        gaussian.tune("gather", old)
    assert gaussian.tuned("gather") == old
    assert rel_err(packed, gather) < 1e-5


def _c3(cuda):
    n, w, h = 2_400_000, 1920, 1080
    g, v, cam = scene(n, w, h, k=0)
    return g, v, cam, _splatter(g, [v], cuda)


def test_camera_grad_full_size_sampled_tiles(gs, cuda):
    """C3 RGB (2.4 M Gaussians, 1080p), maps frame with image, depth and alpha gradients only on sampled tiles (the
    heaviest, the most skipped tail, one in between): the camera gradient matches the oracle restricted to them."""
    g, v, cam, sp = _c3(cuda)
    w, h = v.width, v.height
    with torch.no_grad():
        sp.render_maps(0)
    _, accum = sp._rctx.sorted_instances()
    acc = accum.long().cpu()
    counts = acc[1:] - acc[:-1]
    tail = counts - sp._rctx.tile_consumed().long().cpu()
    top = (cam.Hp - h) // 2
    inside = torch.zeros(cam.nty, cam.ntx, dtype=torch.bool)
    inside[(top + 15) // 16:(top + h) // 16] = True
    inside = inside.reshape(-1)
    heavy = int(torch.where(inside, counts, -1).argmax())
    skip = int(torch.where(inside, tail, -1).argmax())
    busy = (inside & (counts > 0)).nonzero().squeeze(-1)
    tiles = sorted({heavy, skip, int(busy[len(busy) // 3])})
    assert int(counts[heavy]) > 3 * 128 and int(tail[skip]) > 0
    mask_px = torch.zeros(cam.Hp, cam.Wp, dtype=torch.bool)
    for t in tiles:
        ty, tx = divmod(t, cam.ntx)
        mask_px[ty * 16:(ty + 1) * 16, tx * 16:(tx + 1) * 16] = True
    mask_f = cam.crop(mask_px.unsqueeze(-1)).squeeze(-1)
    gi, gd, ga = _upstream(h, w)
    ups = (gi * mask_f.unsqueeze(-1), gd * mask_f, ga * mask_f)
    ocam, _ = _oracle(g, cam, ups, True, tiles=torch.tensor(tiles))
    gcam, _ = _run(sp, v, ups, True, _pose(v), cuda)
    err = rel_err(gcam, ocam)
    print(f"C3 sampled-tile camera gradient rel err {err:.2e}")
    assert err < CAM_RTOL, (gcam, ocam)


def test_camera_grad_translation_identity_full_size(gs, cuda):
    """C3, full image gradient: p_c = R p + t with J detached, so grad_tran = R sum_i grad_pos_i; checked against
    the sum of the magnitudes it is made of."""
    g, v, cam, sp = _c3(cuda)
    ups = _upstream(v.height, v.width)
    gcam, grads = _run(sp, v, ups, False, _pose(v), cuda)
    R = v.rot.double().to(cuda)
    rg = grads[0].double() @ R.T                                  # R grad_pos_i, per Gaussian
    expect = rg.sum(0).cpu()
    bound = 1e-4 * rg.abs().sum(0).cpu()
    dev = (gcam[9:].double() - expect).abs()
    print(f"translation identity: |diff| {dev.tolist()} bound {bound.tolist()}")
    assert bool((dev <= bound).all()) and float(bound.min()) > 0


def test_camera_grad_determinism_and_launches(gs, cuda):
    gaussian, _ = gs
    n, w, h = 8000, 200, 120
    g, v, _ = scene(n, w, h, k=2)
    ups = _upstream(h, w)
    sp = _splatter(g, [v], cuda)

    def counted(pose, maps=False):
        torch.cuda.synchronize()
        k0 = gaussian.kernel_launches()
        out = _run(sp, v, ups, maps, pose, cuda)
        torch.cuda.synchronize()
        return out, gaussian.kernel_launches() - k0

    counted(_pose(v, grad=False))                 # a context's first frame also fills its 0..N-1 sort values
    (_, gp), l_plain = counted(_pose(v, grad=False))
    (c1, g1), l_cam = counted(_pose(v))
    (c2, g2), _ = counted(_pose(v))
    assert torch.equal(c1, c2) and all(torch.equal(a, b) for a, b in zip(g1, g2))
    assert l_cam == l_plain + 1
    (c3, _), l_maps_cam = counted(_pose(v), maps=True)
    (_, _), l_maps = counted(_pose(v, grad=False), maps=True)
    assert l_maps_cam == l_maps + 1 and l_maps == l_plain
    # only one of the two pose tensors requires grad: the other gets none, the count is the same
    rot, tran = v.rot.clone().requires_grad_(True), v.tran.clone()
    (c4, _), l_rot = counted((rot, tran))
    assert l_rot == l_cam and tran.grad is None and torch.equal(c4[:9], c1[:9])


def test_camera_grad_zero_without_instances(gs, cuda):
    """Frames without a single tile instance on fresh contexts (a scene behind the camera, one beside the view):
    the camera gradient is exactly zero, as are the parameter gradients."""
    w, h = 64, 48
    v = S.make_view(w, h, 0)
    for shift in ((0.0, 0.0, -100.0), (50.0, 0.0, 0.0)):
        g = S.make_gaussians(100, w, h)
        g["pos"] += torch.tensor(shift)
        sp = _splatter(g, [v], cuda)
        ups = _upstream(h, w)
        for maps in (False, True):
            gcam, grads = _run(sp, v, ups, maps, _pose(v), cuda)
            assert sp.n_tile_gaussians == 0
            assert float(gcam.abs().max()) == 0.0, (shift, maps)
            assert all(float(t.abs().max()) == 0.0 for t in grads)


def test_camera_grad_refusals(gs, cuda):
    gaussian, renderer = gs
    g, v, _ = scene(500, 64, 48)
    # SH colour: refused with the reason; the setter is cleared again after the exception
    gsh, _, _ = scene(500, 64, 48, sh_dim=27)
    sp_sh = _splatter(gsh, [v], cuda, use_sh_coeff=True)
    img = sp_sh(None, extrinsics=dict(zip(("rot", "tran"), _pose(v))), intrinsics=_intr(v))
    with pytest.raises(RuntimeError, match="RGB colour"):
        img.sum().backward()
    img = sp_sh(None, extrinsics=dict(rot=v.rot, tran=v.tran), intrinsics=_intr(v))
    img.sum().backward()                          # a backward without pose gradients runs again on that context
    # wrong buffers
    sp = _splatter(g, [v], cuda)
    rctx = sp._rctx
    for bad, msg in ((torch.zeros(12), "CUDA"), (torch.zeros(12, device=cuda, dtype=torch.float64), "float32"),
                     (torch.zeros(11, device=cuda), "12 elements"), (torch.zeros(24, device=cuda)[::2], "contiguous")):
        with pytest.raises(RuntimeError, match=msg):
            rctx.set_camera_grad(bad)
    # data-parallel gradient push: refused at backward time whichever of the two was set first
    gp = sp.gaussian_3ds
    args = [t.detach() for t in (gp.pos, gp.rgb, gp.opa, gp.quat, gp.scale)]
    grads = [torch.empty_like(t) for t in args]
    gcam = torch.zeros(12, device=cuda)
    bucket = torch.zeros(64, device=cuda)
    for cam_first in (True, False):
        fin, raw, _ = rctx.forward_final(*args, 64, 48, v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, 0)
        try:
            if cam_first:
                rctx.set_camera_grad(gcam)
            rctx.set_grad_push(bucket.data_ptr(), [bucket.data_ptr(), bucket.data_ptr()], 32, 0)
            if not cam_first:
                rctx.set_camera_grad(gcam)
            with pytest.raises(RuntimeError, match="gradient push"):
                rctx.backward_final_into(*args, raw, torch.zeros_like(fin), *grads)
        finally:
            rctx.clear_grad_push()
            rctx.set_camera_grad(None)
    # usable again, pose gradients included
    gcam_ok, _ = _run(sp, v, _upstream(48, 64), False, _pose(v), cuda)
    assert bool(torch.isfinite(gcam_ok).all()) and float(gcam_ok.abs().max()) > 0


def _axis_angle(w):
    """Rodrigues: axis-angle [3] -> rotation [3,3], differentiable (w != 0)."""
    th = w.norm()
    k = w / th
    K = torch.zeros(3, 3, dtype=w.dtype, device=w.device)
    K[0, 1], K[0, 2], K[1, 0], K[1, 2], K[2, 0], K[2, 1] = -k[2], k[1], k[2], -k[0], -k[1], k[0]
    return torch.eye(3, dtype=w.dtype, device=w.device) + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


POSE_STEPS = 150
POSE_LR_ROT = 1e-3          # rad
POSE_LR_TRAN = 4e-3         # scene units (the camera is 4 units from the scene centre)


def test_pose_recovery_end_to_end(gs, cuda):
    """C1 scene (10 k Gaussians, 256x256): from a pose perturbed by 1 deg of rotation and 2 % of the scene depth in
    translation, Adam on the L1 image loss over the pose alone (axis-angle in torch) recovers it: both errors fall
    below 10 % of their initial values in a fixed number of steps."""
    n, w, h = 10000, 256, 256
    g, v, _ = scene(n, w, h, k=0)
    sp = _splatter(g, [v], cuda)
    for p in sp.gaussian_3ds.parameters():
        p.requires_grad_(False)
    R0, t0 = v.rot.double().to(cuda), v.tran.double().to(cuda)
    with torch.no_grad():
        target = sp(None, extrinsics=dict(rot=v.rot, tran=v.tran), intrinsics=_intr(v)).clone()
    axis = torch.tensor([0.3, 1.0, -0.5], dtype=torch.float64)
    w_err = (axis / axis.norm() * math.radians(1.0)).to(cuda)
    dt = torch.tensor([0.6, -0.5, 0.62], dtype=torch.float64)
    dt = (dt / dt.norm() * 0.02 * float(v.tran.norm())).to(cuda)
    omega = w_err.clone().requires_grad_(True)      # R = exp([omega]) R0
    tran = (t0 + dt).clone().requires_grad_(True)
    opt = torch.optim.Adam([dict(params=[omega], lr=POSE_LR_ROT), dict(params=[tran], lr=POSE_LR_TRAN)])
    e_rot0, e_tran0 = float(omega.norm()), float((tran - t0).norm())
    for _ in range(POSE_STEPS):
        opt.zero_grad()
        rot = _axis_angle(omega) @ R0
        img = sp(None, extrinsics=dict(rot=rot, tran=tran), intrinsics=_intr(v))
        (img - target).abs().mean().backward()
        opt.step()
    e_rot, e_tran = float(omega.norm()), float((tran - t0).detach().norm())
    print(f"pose recovery: rotation {math.degrees(e_rot0):.3f} -> {math.degrees(e_rot):.4f} deg, "
          f"translation {e_tran0:.4f} -> {e_tran:.5f}")
    assert e_rot < 0.1 * e_rot0 and e_tran < 0.1 * e_tran0
