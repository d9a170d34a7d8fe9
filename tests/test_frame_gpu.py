"""GPU parity of the fused frame path (parameters -> image -> parameter gradients) against
the CPU oracle, the committed golden fixtures and the reference build's whole pipeline (its
outputs stored in tests/golden/ref_frame.npz); plus size-independent properties at
BASELINE.json's full sizes (P3/P5/P6 of SURVEY.md §8c).
"""
import os

import pytest
import torch

import gs_oracle as O
import synthetic as S
from helpers import (abs_err, assert_matches_golden_frame, device_depth_keys, load_golden, rel_err, require_golden,
                     scene)

pytestmark = pytest.mark.gpu

IMG_ATOL = 1e-4
GRAD_RTOL = 1e-3


def _splatter(g, views, dev, **kw):
    import splatter
    vs = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran) for v in views]
    return splatter.Splatter.from_tensors(g, vs, device=dev, **kw)


def _oracle_frame(g, cam, grad_out, dtype=torch.float64, **kw):
    p = {k: v.to(dtype).clone().requires_grad_(True) for k, v in g.items()}
    if torch.cuda.is_available():       # sort on the device's own fp32 depth keys (ulp-tie robust)
        kw = dict(kw, depth_key=device_depth_keys(g, cam, torch.device("cuda", 0), kw.get("scale_activation", "abs")))
    img, aux = O.render(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, return_aux=True, **kw)
    img.backward(grad_out.to(dtype))
    return img.detach(), {k: p[k].grad for k in p}, aux


@pytest.mark.parametrize("n,w,h,k,opa", [
    (2000, 128, 96, 0, (0.005, 0.05)),     # safe regime, no saturation
    (10000, 256, 256, 0, (0.05, 0.9)),     # C1: BASELINE configs[0]
    (8000, 200, 120, 2, (0.05, 0.9)),      # rotated view (culling), non-multiple-of-16 size
    (5000, 96, 64, 0, (0.6, 0.98)),        # opaque: early termination everywhere
])
def test_fused_frame_vs_oracle(gs, cuda, n, w, h, k, opa):
    g, v, cam = scene(n, w, h, k=k, opa_range=opa)
    go = S.make_grad_output(h, w, 0) * (h * w)            # O(1) upstream gradient
    oimg, ograds, aux = _oracle_frame(g, cam, go)
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    assert img.shape == (h, w, 3)
    assert abs_err(img, oimg) < IMG_ATOL
    img.backward(go.to(cuda))
    gp = sp.gaussian_3ds
    for name in ("pos", "rgb", "opa", "quat", "scale"):
        assert rel_err(getattr(gp, name).grad, ograds[name]) < GRAD_RTOL, name
    # culling mask: int64, identical to the oracle's (train.py:150 consumes it)
    assert sp.culling_mask.dtype == torch.int64
    assert int((sp.culling_mask.cpu() != aux["mask"]).sum()) <= 1
    # P3: our (tile, depth) order is the oracle's exact order
    st = sp.frame_stats()
    assert st["n_instances"] == int(aux["accum"][-1])
    idx, accum = sp._rctx.sorted_instances()
    assert torch.equal(accum.cpu(), aux["accum"])
    # the oracle sorted the device's own fp32 depth keys -> exactly the same (tile, depth, id) order
    assert torch.equal(idx.cpu().long(), aux["gauss_idx"])


@pytest.mark.parametrize("sh_tc", [3, 0], ids=["tensor-core", "scalar"])
@pytest.mark.parametrize("sh_dim,opa", [(27, (0.005, 0.05)), (27, (0.3, 0.95)), (48, (0.05, 0.9))])
def test_fused_frame_sh_vs_oracle(gs, cuda, sh_dim, opa, sh_tc):
    """Both SH blend kernel families (blend_sh_tc.cu: tcgen05 contractions with bf16 hi/lo operands, the default;
    blend_sh.cu: scalar fp32) against the fp64 oracle, at the tolerances of BASELINE.json's north_star."""
    n, w, h = 2500, 112, 80
    g, v, cam = scene(n, w, h, k=1, sh_dim=sh_dim, opa_range=opa)
    go = S.make_grad_output(h, w, 0) * (h * w)
    oimg, ograds, aux = _oracle_frame(g, cam, go, use_sh_coeff=True)
    gs[0].tune("sh_tc", sh_tc)
    try:
        sp = _splatter(g, [v], cuda, use_sh_coeff=True)
        img = sp(0)
        assert abs_err(img, oimg) < IMG_ATOL
        img.backward(go.to(cuda))
        for name in ("pos", "rgb", "opa", "quat", "scale"):
            assert rel_err(getattr(sp.gaussian_3ds, name).grad, ograds[name]) < GRAD_RTOL, name
    finally:
        gs[0].tune("sh_tc", 3)


def test_fused_frame_vs_reference_pipeline(gs, cuda):
    """P5: whole reference pipeline (its CUDA build + its renderer.py + the splatter.py call
    sequence; outputs in tests/golden/ref_frame.npz) vs our fused path on a C1-class scene inside
    the reference's safe regime."""
    import golden_cases as GC
    # a scene inside the reference's own limits (capacity MAXP = n//20, no fp32 sort-key ties)
    n, w, h = 2000, 192, 128
    g, v, cam, go = GC.frame_case(n, w, h, (0.005, 0.05), (0.4, 1.5), 2)
    assert GC.reference_key_collisions(g, cam)[0] == 0
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    img.backward(go.to(cuda))
    assert_matches_golden_frame(sp, img, require_golden("ref_frame.npz"), IMG_ATOL, GRAD_RTOL)


def test_legacy_boundary_drop_in(gs, cuda):
    """The reference's splatter.py call sequence runs unchanged on OUR `gaussian` module
    (+ our renderer.py) and agrees with the fused path."""
    import ref_pipeline
    gaussian, renderer = gs
    import golden_cases as GC
    n, w, h = 2000, 192, 128
    g, v, cam, go = GC.frame_case(n, w, h, (0.05, 0.6), (0.4, 1.5), 6)      # capacity n//20 respected
    assert GC.reference_key_collisions(g, cam)[0] == 0
    go = go.to(cuda)
    frame = ref_pipeline.LegacyFrame(gaussian, renderer, w, h, v.fx, v.fy, v.rot.to(cuda), v.tran.to(cuda))
    p = {k: t.to(cuda).clone().requires_grad_(True) for k, t in g.items()}
    limg = frame(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"])
    limg.backward(go)
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    img.backward(go)
    assert abs_err(img, limg) < IMG_ATOL
    for name in ("pos", "rgb", "opa", "quat", "scale"):
        assert rel_err(getattr(sp.gaussian_3ds, name).grad, p[name].grad) < GRAD_RTOL, name


def test_fused_frame_vs_golden(gs, cuda):
    gold = load_golden("frame_c1.npz")
    if gold is None:
        pytest.skip("tests/golden/frame_c1.npz not generated yet")
    import golden_cases as GC
    g, v, cam, go = GC.frame_inputs()
    assert (int(gold["n"]), int(gold["w"]), int(gold["h"])) == (g["pos"].shape[0], v.width, v.height)
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    assert abs_err(img, gold["image"]) < IMG_ATOL
    img.backward(go.to(cuda))
    for name in ("pos", "rgb", "opa", "quat", "scale"):
        assert rel_err(getattr(sp.gaussian_3ds, name).grad, gold["grad_" + name]) < GRAD_RTOL, name


def test_fused_clamp_crop_equals_torch_post(gs, cuda):
    """Splatter.forward (clamp + crop inside the kernels) == padded render + torch clamp/crop,
    image and gradients, on a near-saturated scene whose size needs padding on both axes.
    (With sigmoid colours and a black background sum_i w_i c_i <= 1, so the clamp only ever
    guards rounding; the crop / zero-padding of the gradient is what this exercises.)"""
    g, v, cam = scene(6000, 200, 120, k=0, opa_range=(0.3, 0.95))
    g["rgb"] = g["rgb"] + 3.0                      # bright colours: accumulated colour exceeds 1
    go = (S.make_grad_output(120, 200, 3) * (120 * 200)).to(cuda)
    res = []
    for fused in (True, False):
        sp = _splatter(g, [v], cuda)
        img = sp(0) if fused else sp.forward_unfused_post(0)
        img.backward(go)
        res.append((img.detach(), [p.grad.clone() for p in sp.gaussian_3ds.parameters()]))
    assert float(res[1][0].max()) > 0.9
    assert torch.equal(res[0][0], res[1][0])
    for a, b in zip(res[0][1], res[1][1]):
        assert rel_err(a, b) < 1e-6


def test_edge_cases(gs, cuda):
    v = S.make_view(64, 48, 0)
    # empty scene
    g0 = S.make_gaussians(0, 64, 48)
    sp = _splatter(g0, [v], cuda)
    img = sp(0)
    assert img.shape == (48, 64, 3) and float(img.abs().max()) == 0
    # everything behind the camera -> all culled, zero gradients
    g = S.make_gaussians(100, 64, 48)
    g["pos"][:, 2] -= 100.0
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    assert float(img.abs().max()) == 0 and int(sp.culling_mask.sum()) == 0
    img.sum().backward()
    assert float(sp.gaussian_3ds.pos.grad.abs().max()) == 0
    # a single Gaussian in the middle of the image
    g = S.make_gaussians(1, 64, 48)
    g["pos"][:] = 0
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    cam = O.Camera(64, 48, v.fx, v.fy, v.rot, v.tran)
    oimg = O.render(g["pos"], g["rgb"], g["opa"], g["quat"], g["scale"], cam)
    assert abs_err(img, oimg) < IMG_ATOL and float(img.max()) > 0
    # free camera through extrinsics/intrinsics (visergui.py:137-149 path)
    img2 = sp(None, dict(rot=v.rot.numpy(), tran=v.tran.numpy()),
              dict(width=64, height=48, focal_x=v.fx, focal_y=v.fy))
    assert torch.equal(img, img2)


@pytest.mark.parametrize("n,w,h", [(500_000, 1920, 1080), (2_400_000, 1920, 1080)])
def test_full_size_properties(gs, cuda, n, w, h):
    """BASELINE configs[1]/[2] sizes: properties that need no CPU oracle."""
    g, v, cam = scene(n, w, h, k=0)
    sp = _splatter(g, [v], cuda)
    go1 = S.make_grad_output(h, w, 0).to(cuda) * (h * w)
    go2 = S.make_grad_output(h, w, 5).to(cuda) * (h * w)

    def run(go):
        for p in sp.gaussian_3ds.parameters():
            p.grad = None
        img = sp(0)
        img.backward(go)
        return img.detach().clone(), [p.grad.clone() for p in sp.gaussian_3ds.parameters()]

    img_a, ga = run(go1)
    img_b, gb = run(go1)
    assert torch.equal(img_a, img_b)                               # forward deterministic
    for x, y in zip(ga, gb):
        assert torch.equal(x, y)                                   # backward deterministic (no atomics)
    assert bool(torch.isfinite(img_a).all()) and float(img_a.min()) >= 0 and float(img_a.max()) <= 1
    st = sp.frame_stats()
    idx, accum = sp._rctx.sorted_instances()
    acc = accum.long()
    assert int(acc[0]) == 0 and int(acc[-1]) == st["n_instances"] and bool((acc[1:] >= acc[:-1]).all())
    assert st["n_instances_eff"] <= st["n_instances"]
    # sortedness: depth non-decreasing inside every tile (sampled tiles)
    pos = sp.gaussian_3ds.pos.detach()
    pc = pos @ v.rot.to(cuda).T + v.tran.to(cuda)
    depth = pc.norm(dim=-1)
    for t in torch.linspace(0, acc.numel() - 2, 64).long().tolist():
        s, e = int(acc[t]), int(acc[t + 1])
        d = depth[idx[s:e].long()]
        assert bool((d[1:] >= d[:-1] - 1e-5).all())
    # backward is linear in the upstream gradient
    _, g2 = run(go2)
    _, g12 = run(go1 + go2)
    for x, y, z in zip(ga, g2, g12):
        assert rel_err(x + y, z) < 1e-3
    # oracle spot check on a tile sub-sample (P6): 6 tiles of the padded image
    tiles = torch.linspace(0, cam.ntx * cam.nty - 1, 6).long()
    oimg, aux = O.render(g["pos"], g["rgb"], g["opa"], g["quat"], g["scale"], cam, tiles=tiles, return_aux=True)
    padded = aux["padded"]
    img_p = torch.zeros(cam.Hp, cam.Wp, 3)
    top, left = (cam.Hp - h) // 2, (cam.Wp - w) // 2
    img_p[top:top + h, left:left + w] = img_a.cpu()
    for t in tiles.tolist():
        ty, tx = divmod(t, cam.ntx)
        a = img_p[ty * 16:(ty + 1) * 16, tx * 16:(tx + 1) * 16]
        b = padded[ty * 16:(ty + 1) * 16, tx * 16:(tx + 1) * 16].clamp(0, 1)
        if ty * 16 >= top and (ty + 1) * 16 <= top + h:
            assert abs_err(a, b) < IMG_ATOL


def test_training_loop_converges(gs, cuda):
    """§8f-1: the reference's train_step (L1 + Adam over the five parameter groups) on top of the
    fused path: the loss must fall on a small synthetic multi-view scene."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "train_dp", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "train_dp.py"))
    td = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(td)
    sp, gts = td.build(20000, 160, 96, 4, cuda)
    hist, ips = td.train(sp, gts, 60, 1, 0, log_every=20)
    assert hist[-1][1] < 0.6 * hist[0][1], hist
    assert hist[-1][2] > hist[0][2] + 2.0


def test_wide_tile_keys_path_matches(gs, cuda):
    """Images with more than 65536 tiles sort 32-bit tile keys; that path (forced through
    GS_TILE_KEY_BYTES=4 in a fresh process) must give bit-identical results."""
    import os
    import subprocess
    import sys
    code = r"""
import sys, torch, hashlib
sys.path[:0] = [r'%s', r'%s', r'%s']
import splatter, synthetic as S
v = S.make_view(200, 120, 1); g = S.make_gaussians(5000, 200, 120, 4)
sp = splatter.Splatter.from_tensors(g, [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran)])
img = sp(0); img.backward(S.make_grad_output(120, 200, 0).cuda() * 24000)
h = hashlib.sha1(img.detach().cpu().numpy().tobytes())
for p in sp.gaussian_3ds.parameters(): h.update(p.grad.cpu().numpy().tobytes())
print(h.hexdigest())
""" % tuple(p for p in sys.path[:3])
    outs = []
    for kb in ("2", "4"):
        env = dict(os.environ, GS_TILE_KEY_BYTES=kb)
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(r.stdout.strip().splitlines()[-1])
    assert outs[0] == outs[1] and len(outs[0]) == 40


def test_exp_scale_activation_and_extreme_gaussians(gs, cuda):
    """scale_activation="exp" (trunc_exp, renderer.py:91-100: clamped-gradient backward) and shapes
    that stress binning: one Gaussian covering every tile, needle-thin ones, negative raw scales."""
    n, w, h = 1500, 128, 96
    g, v, cam = scene(n, w, h, k=0, opa_range=(0.05, 0.8))
    g["scale"] = torch.log(g["scale"])                       # raw = log(sigma) for the exp activation
    g["scale"][0] = torch.log(torch.tensor([2.0, 2.0, 2.0]))  # huge: bbox covers the whole image
    g["pos"][0] = torch.tensor([0.0, 0.0, 0.0])
    g["scale"][1] = torch.tensor([1.2, 1.1, 1.3])            # raw > 1: hits the clamp in trunc_exp's backward
    go = S.make_grad_output(h, w, 0) * (h * w)
    oimg, ograds, aux = _oracle_frame(g, cam, go, scale_activation="exp")
    sp = _splatter(g, [v], cuda, scale_activation="exp")
    img = sp(0)
    assert abs_err(img, oimg) < IMG_ATOL
    img.backward(go.to(cuda))
    for name in ("pos", "rgb", "opa", "quat", "scale"):
        assert rel_err(getattr(sp.gaussian_3ds, name).grad, ograds[name]) < GRAD_RTOL, name
    counts = aux["accum"][1:] - aux["accum"][:-1]
    assert int(counts.min()) >= 1                              # the huge Gaussian is in every tile
    # a degenerate needle (sigma ratio 1e4): det(cov2d) is pure fp32 rounding noise, so whether it is
    # binned at all is arbitrary (gaussian.cu:227 `det <= 0`) - only require a finite result
    g["scale"][2] = torch.tensor([-9.0, 1.2, -9.0])
    sp = _splatter(g, [v], cuda, scale_activation="exp")
    img = sp(0)
    img.backward(go.to(cuda))
    assert bool(torch.isfinite(img).all())
    assert all(bool(torch.isfinite(p.grad).all()) for p in sp.gaussian_3ds.parameters())
    # abs activation with negative raw scales: |s| + 1e-4, gradient sign follows the raw value
    g2, v2, cam2 = scene(800, 96, 64, k=0)
    g2["scale"] = -g2["scale"]
    oimg2, ograds2, _ = _oracle_frame(g2, cam2, S.make_grad_output(64, 96, 0) * (64 * 96))
    sp2 = _splatter(g2, [v2], cuda)
    img2 = sp2(0)
    assert abs_err(img2, oimg2) < IMG_ATOL
    img2.backward((S.make_grad_output(64, 96, 0) * (64 * 96)).to(cuda))
    assert rel_err(sp2.gaussian_3ds.scale.grad, ograds2["scale"]) < GRAD_RTOL


def test_instance_count_overflow_is_refused(gs, cuda):
    """Diverged scales (every Gaussian on every tile) make M = N*T exceed the 32-bit instance index:
    2^31 <= M < 2^32, and M >= 2^32 where a u32 scan would wrap to a small, plausible value.  Both
    must raise (the reference silently truncates at N/20 per tile) and leave the context usable."""
    w, h = 1920, 1080                                          # T = 8160
    for n in (300_000, 600_000):                               # M = 2.4e9 (>2^31), 4.9e9 (>2^32)
        g = {"pos": torch.zeros(n, 3), "rgb": torch.zeros(n, 3), "opa": torch.zeros(n),
             "quat": torch.tensor([[1.0, 0.0, 0.0, 0.0]]).repeat(n, 1), "scale": torch.full((n, 3), 30.0)}
        v = S.make_view(w, h, 0)
        sp = _splatter(g, [v], cuda)
        with pytest.raises(RuntimeError, match="2\\^31 tile instances"):
            with torch.no_grad():
                sp(0)
    small, vs, _ = scene(500, 64, 48)
    sp = _splatter(small, [vs], cuda)
    assert bool(torch.isfinite(sp(0)).all())


def test_bad_arguments_are_refused(gs, cuda):
    g, v, cam = scene(100, 64, 48)
    for thresh in (0.0, 1.0, -1.0):
        sp = _splatter(g, [v], cuda, tile_culling_prob_thresh=thresh)
        with pytest.raises(RuntimeError, match="tile_thresh"):
            sp(0)


def test_stale_forward_is_refused(gs, cuda):
    """One RenderContext holds one frame: differentiating an older frame after another forward
    must raise instead of silently using the wrong intermediate state."""
    g, v, cam = scene(500, 64, 48)
    sp = _splatter(g, [v, S.make_view(64, 48, 1)], cuda)
    img0 = sp(0)
    with torch.no_grad():
        sp(1)                                   # e.g. a test render between forward and backward
    with pytest.raises(RuntimeError, match="another frame"):
        img0.sum().backward()
    img1 = sp(1)                                # normal use keeps working
    img1.sum().backward()
    assert sp.gaussian_3ds.pos.grad is not None


def test_splatter_reference_constructor_on_colmap_dataset(gs, cuda, tmp_path):
    """The reference's own construction path (train.py:374-392): Splatter(colmap_dir, image_dir,
    <reference kwargs>) on a synthetic COLMAP model + PNG images, then the train-step surface
    train.py uses: forward(camera_id) vs ground_truth, backward, culling_mask accumulation,
    adaptive_control + optimizer rebuild, reset_opa, n_tile_gaussians / n_gaussians."""
    import cv2
    import numpy as np
    import colmap_io as C
    import splatter
    w, h, n_views = 160, 96, 4
    teacher = S.make_gaussians(4000, w, h, 0)
    views = [S.make_view(w, h, k) for k in range(n_views)]
    vd = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran) for v in views]
    sp_t = splatter.Splatter.from_tensors(teacher, vd, device=cuda)
    sparse, imgdir = tmp_path / "sparse" / "0", tmp_path / "images_1"
    os.makedirs(sparse), os.makedirs(imgdir)
    cams = {1: C.Camera(1, "PINHOLE", w, h, np.array([views[0].fx, views[0].fy, w / 2, h / 2]))}
    imgs = {}
    for k, v in enumerate(views):
        with torch.no_grad():
            im = (sp_t(k).clamp(0, 1) * 255).byte().cpu().numpy()
        cv2.imwrite(str(imgdir / f"v{k}.png"), im[..., ::-1])
        imgs[k + 1] = C.Image(k + 1, C.rotmat_to_qvec(v.rot.numpy()), v.tran.numpy(), 1, f"v{k}.png")
    pts = {i: C.Point3D(i, teacher["pos"][i].numpy(), (torch.sigmoid(teacher["rgb"][i]) * 255).byte().numpy(), 0.0)
           for i in range(0, 4000, 2)}
    C.write_cameras_binary(sparse / "cameras.bin", cams)
    C.write_images_binary(sparse / "images.bin", imgs)
    C.write_points3d_binary(sparse / "points3D.bin", pts)

    sp = splatter.Splatter(str(sparse), str(imgdir), render_weight_normalize=False, render_downsample=1,
                           use_sh_coeff=False, scale_init_value=0.5, opa_init_value=0.3, tile_culling_method="prob2",
                           tile_culling_dist_thresh=0.5, tile_culling_prob_thresh=0.05, debug=0, scale_activation="abs",
                           cudaculling=1, load_ckpt=None, fast_drawing=True, test=False)
    assert len(sp.imgs) == n_views and sp.gaussian_3ds.pos.shape == (2000, 3) and sp.gaussian_3ds.quat.shape == (2000, 4)
    assert torch.allclose(sp.views[2]["rot"], views[2].rot, atol=1e-5) and abs(sp.views[0]["focal_x"] - views[0].fx) < 1e-3
    g3 = sp.gaussian_3ds

    def make_opt():
        return torch.optim.Adam([{"params": g3.opa, "lr": 0.03}, {"params": g3.rgb, "lr": 0.03},
                                 {"params": g3.pos, "lr": 0.003}, {"params": g3.scale, "lr": 0.003},
                                 {"params": g3.quat, "lr": 0.003}], betas=(0.9, 0.99))
    opt = make_opt()
    accum = torch.zeros_like(g3.pos)
    counter = torch.zeros(g3.pos.shape[0], device=cuda)
    losses = []
    for it in range(40):
        opt.zero_grad()
        img = sp(it % n_views)
        assert img.shape == (h, w, 3) and sp.ground_truth.shape == (h, w, 3) and sp.ground_truth.dtype == torch.float16
        loss = (img - sp.ground_truth).abs().mean()             # train.py:99
        loss.backward()
        opt.step()
        accum += g3.pos.grad.abs()                              # train.py:149-150
        counter += sp.culling_mask.to(torch.float32)
        losses.append(float(loss))
        assert sp.n_tile_gaussians > 0 and sp.n_gaussians == g3.pos.shape[0]
    assert losses[-1] < losses[0]
    n0 = g3.pos.shape[0]
    info = g3.adaptive_control(accum / (counter + 1e-3).unsqueeze(-1), taus=0.02, delete_thresh=1.5,
                               scale_activation=sp.scale_activation, grad_thresh=1e-7, use_clone=True, use_split=True,
                               grad_aggregation="max", clone_dt=0.01)
    assert info["total"] == g3.pos.shape[0] == n0 - info["deleted"] + info["cloned"] + info["split"]
    assert info["cloned"] + info["split"] > 0
    opt = make_opt()                                            # train.py:173-181
    g3.reset_opa()
    img = sp(0)
    (img - sp.ground_truth).abs().mean().backward()
    opt.step()
    assert g3.pos.grad.shape[0] == info["total"] and bool(torch.isfinite(g3.pos).all())


def test_c_abi_host_buffer_entry_point(gs, cuda):
    """gs_render_forward_backward_host called straight through ctypes (no torch types in the
    signature): device-resident parameters, HOST image / gradient buffers; must reproduce the
    Python path bit for bit."""
    import ctypes
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "3d-gaussian-splatting_b200")
    lib = ctypes.CDLL(os.path.join(pkg, "libgs_b200.so"))

    class Cam(ctypes.Structure):
        _fields_ = [("width", ctypes.c_int), ("height", ctypes.c_int), ("focal_x", ctypes.c_float),
                    ("focal_y", ctypes.c_float), ("rot", ctypes.c_float * 9), ("tran", ctypes.c_float * 3),
                    ("near_plane", ctypes.c_float), ("tile_thresh", ctypes.c_float)]
    n, w, h = 3000, 112, 80                                  # padded to 112 x 80
    g, v, cam = scene(n, w, h, k=1)
    sp = _splatter(g, [v], cuda)
    gpad = torch.zeros(cam.Hp, cam.Wp, 3)
    gpad[:h, :w] = S.make_grad_output(h, w, 0) * (h * w)
    raw = sp.render_padded()
    raw.backward(gpad.to(cuda))
    want = [p.grad.clone() for p in sp.gaussian_3ds.parameters()]

    P = ctypes.c_void_p
    lib.gs_last_error.restype = ctypes.c_char_p
    ctx = P()
    assert lib.gs_ctx_create(ctypes.byref(ctx)) == 0
    c = Cam(w, h, v.fx, v.fy, (ctypes.c_float * 9)(*v.rot.flatten().tolist()), (ctypes.c_float * 3)(*v.tran.tolist()),
            0.3, 0.05)
    dev = {k: t.to(cuda).contiguous() for k, t in g.items()}
    grads = {k: torch.empty_like(t) for k, t in dev.items()}
    gimg_host = gpad.contiguous().pin_memory()
    img_host = torch.empty(cam.Hp, cam.Wp, 3).pin_memory()
    lib.gs_render_forward_backward_host.argtypes = [P] * 6 + [ctypes.c_int] * 3 + [ctypes.POINTER(Cam)] + [P] * 8
    torch.cuda.synchronize()
    rc = lib.gs_render_forward_backward_host(
        ctx, dev["pos"].data_ptr(), dev["rgb"].data_ptr(), dev["opa"].data_ptr(), dev["quat"].data_ptr(),
        dev["scale"].data_ptr(), n, 3, 0, ctypes.byref(c), gimg_host.data_ptr(), img_host.data_ptr(),
        grads["pos"].data_ptr(), grads["rgb"].data_ptr(), grads["opa"].data_ptr(), grads["quat"].data_ptr(),
        grads["scale"].data_ptr(), None)
    assert rc == 0, lib.gs_last_error()
    assert torch.equal(img_host, raw.detach().cpu())
    for a, b in zip((grads[k] for k in ("pos", "rgb", "opa", "quat", "scale")), want):
        assert torch.equal(a, b)
    # error conventions: unsupported colour width -> GS_ERR_UNSUPPORTED (-2) with a message, no crash
    rc = lib.gs_render_forward_backward_host(
        ctx, dev["pos"].data_ptr(), dev["rgb"].data_ptr(), dev["opa"].data_ptr(), dev["quat"].data_ptr(),
        dev["scale"].data_ptr(), n, 5, 0, ctypes.byref(c), gimg_host.data_ptr(), img_host.data_ptr(),
        grads["pos"].data_ptr(), grads["rgb"].data_ptr(), grads["opa"].data_ptr(), grads["quat"].data_ptr(),
        grads["scale"].data_ptr(), None)
    assert rc == -2 and b"colour width" in lib.gs_last_error()
    lib.gs_ctx_destroy.argtypes = [P]
    lib.gs_ctx_destroy(ctx)


def test_fused_flat_adam_matches_torch_adam(gs, cuda):
    """§8 f-2: FlatAdam (one kernel over the flat bucket) == torch.optim.Adam with the reference's
    five parameter groups, over several steps with per-group learning rates that change."""
    import optim
    import renderer
    torch.manual_seed(0)
    n = 1001                                                   # odd: exercises the padded segments
    shapes = dict(pos=(n, 3), rgb=(n, 3), opa=(n,), quat=(n, 4), scale=(n, 3))
    init = {k: torch.randn(s, device=cuda) for k, s in shapes.items()}
    pa = {k: torch.nn.Parameter(v.clone()) for k, v in init.items()}
    pb = {k: torch.nn.Parameter(v.clone()) for k, v in init.items()}
    order = ("opa", "rgb", "pos", "scale", "quat")            # train.py:56-64 group order
    lrs = dict(opa=0.03, rgb=0.03, pos=0.003, scale=0.004, quat=0.005)
    oa = optim.FlatAdam([{"params": pa[k], "lr": lrs[k]} for k in order], betas=(0.9, 0.99))
    ob = torch.optim.Adam([{"params": pb[k], "lr": lrs[k]} for k in order], betas=(0.9, 0.99))
    for it in range(6):
        grads, _ = renderer._flat_grads(tuple(pa[k] for k in ("pos", "rgb", "opa", "quat", "scale")))
        for gv, k in zip(grads, ("pos", "rgb", "opa", "quat", "scale")):
            gv.copy_(torch.randn_like(gv) * (0.1 + it))
            pa[k].grad = gv
            pb[k].grad = gv.clone()
        for grp_a, grp_b in zip(oa.param_groups, ob.param_groups):       # lr schedule, train.py:184-185
            grp_a["lr"] = grp_b["lr"] = grp_b["lr"] * 0.9
        oa.step()
        ob.step()
        oa.zero_grad()
        ob.zero_grad()
    for k in shapes:
        assert rel_err(pa[k], pb[k]) < 2e-6, k
    # the parameters now alias one flat buffer, in bucket order
    assert pa["pos"].data.untyped_storage().data_ptr() == pa["scale"].data.untyped_storage().data_ptr()


def test_checkpoint_schema_and_exact_resume(gs, cuda, tmp_path):
    """§8 f-4: `save_checkpoint` writes the reference's five keys (train.py:283-291) + resume state; training
    N steps, saving, training M more == loading into a fresh scene + optimizer and training M steps, bit for bit;
    a reference-style file (five keys only) loads too."""
    import checkpoint
    import optim
    import splatter
    n, w, h = 3000, 128, 96
    g, v, cam = scene(n, w, h, k=0)
    teacher, _, _ = scene(n, w, h, seed=3, k=0)
    vd = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran)]
    with torch.no_grad():
        gt = splatter.Splatter.from_tensors(teacher, vd, device=cuda)(0)

    def make(gauss):
        sp = splatter.Splatter.from_tensors(gauss, vd, device=cuda)
        g3 = sp.gaussian_3ds
        opt = optim.FlatAdam([{"params": g3.opa, "lr": 0.03}, {"params": g3.rgb, "lr": 0.03}, {"params": g3.pos, "lr": 0.003},
                              {"params": g3.scale, "lr": 0.003}, {"params": g3.quat, "lr": 0.003}], betas=(0.9, 0.99))
        return sp, opt

    def train(sp, opt, steps):
        for _ in range(steps):
            opt.zero_grad()
            (sp(0) - gt).abs().mean().backward()
            opt.step()

    sp, opt = make(g)
    train(sp, opt, 5)
    path = str(tmp_path / "exp" / "ckpt.pth")
    sp.save_checkpoint(path, optimizer=opt, iteration=5, trainer_state={"grad_counter": 3})
    train(sp, opt, 4)
    want = {k: getattr(sp.gaussian_3ds, k).detach().clone() for k in checkpoint.KEYS}

    raw = torch.load(path, map_location="cpu", weights_only=False)
    assert [k for k in raw if k != "resume"] == list(checkpoint.KEYS) and raw["pos"].shape == (n, 3)
    assert raw["resume"]["iteration"] == 5 and raw["resume"]["trainer"]["grad_counter"] == 3

    sp2, opt2 = make(g)
    checkpoint.load_checkpoint(path, sp2, None)
    sp2b, opt2 = make({k: getattr(sp2.gaussian_3ds, k).detach().cpu() for k in checkpoint.KEYS})
    checkpoint.load_checkpoint(path, None, opt2)
    train(sp2b, opt2, 4)
    for k in checkpoint.KEYS:
        assert torch.equal(getattr(sp2b.gaussian_3ds, k).detach(), want[k]), k

    # a file as the reference writes it (train.py:284-291: the nn.Parameters, nothing else) loads as well
    ref_style = str(tmp_path / "ref_ckpt.pth")
    torch.save({k: getattr(sp.gaussian_3ds, k) for k in ("pos", "opa", "rgb", "quat", "scale")}, ref_style)
    sp3 = splatter.Splatter(g, vd, device=cuda, tile_culling_prob_thresh=0.05, load_ckpt=ref_style)
    assert torch.equal(sp3.gaussian_3ds.pos.detach(), want["pos"])
    assert checkpoint.load_checkpoint(ref_style, sp3).get("resume") is None


@pytest.mark.parametrize("act,agg,sh", [("abs", "max", 3), ("exp", "mean", 27)])
def test_densification_kernel_vs_oracle(gs, cuda, act, agg, sh):
    """§8 f-2: `Gaussian3ds.adaptive_control` (device kernels) == the torch restatement of reference
    splatter.py:122-228 given the same normals, element for element, incl. layout and counts."""
    import densify_oracle as DO
    import splatter
    n, w, h = 5000, 128, 96
    g, v, cam = scene(n, w, h, k=0, sh_dim=sh)
    if act == "exp":
        g["scale"] = torch.log(g["scale"])
    gen = torch.Generator().manual_seed(7)
    g["opa"] = g["opa"] - 3.0 * (torch.rand(n, generator=gen) < 0.2)          # some below the prune threshold
    g["scale"][::50] = 2.0 if act == "abs" else 1.0                              # some above delete_thresh
    grad = torch.randn(n, 3, generator=gen) * 3e-4
    vd = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran)]
    sp = splatter.Splatter.from_tensors(g, vd, device=cuda, use_sh_coeff=sh != 3, scale_activation=act)
    norm = (g["scale"].norm(dim=-1) if act == "abs" else g["scale"].exp().norm(dim=-1))
    tau = float(norm.median())
    torch.cuda.manual_seed(123)
    info = sp.gaussian_3ds.adaptive_control(grad.to(cuda), taus=tau, delete_thresh=1.5, scale_activation=act,
                                            grad_thresh=2e-4, grad_aggregation=agg, use_clone=True, use_split=True,
                                            clone_dt=0.01)
    torch.cuda.manual_seed(123)
    z = torch.randn(2, info["split"], 3, device=cuda).cpu()
    want, oinfo = DO.adaptive_control(g["pos"], g["rgb"], g["opa"], g["quat"], g["scale"], grad, tau, 1.5, act, 2e-4, agg,
                                      True, True, 0.01, z=z)
    assert (info["deleted"], info["cloned"], info["split"]) == (oinfo["deleted"], oinfo["cloned"], oinfo["split"])
    assert info["deleted"] > 0 and info["cloned"] > 0 and info["split"] > 0
    assert info["total"] == n - info["deleted"] + info["cloned"] + info["split"]
    for name, t in zip(("pos", "rgb", "opa", "quat", "scale"), want):
        got = getattr(sp.gaussian_3ds, name).detach().cpu()
        assert got.shape == t.shape, name
        assert rel_err(got, t) < 1e-6, name
    assert bool(torch.isfinite(sp(0)).all())                  # the new scene renders
    # clone / split switched off (train.py passes False inside the opacity-reset interval): prune only
    n1 = sp.gaussian_3ds.pos.shape[0]
    info2 = sp.gaussian_3ds.adaptive_control(torch.zeros(n1, 3, device=cuda), taus=tau, delete_thresh=1.5,
                                             scale_activation=act, use_clone=False, use_split=False)
    assert info2["cloned"] == 0 and info2["split"] == 0 and info2["total"] == n1 - info2["deleted"]


def test_workspaces_come_from_the_torch_allocator_and_grow(gs, cuda):
    """gs_ctx_set_allocator: the torch shim hands PyTorch's caching allocator to the context, so the frame's
    workspaces are visible in torch's accounting and a growing scene (densification) re-allocates without
    cudaMalloc / a device synchronisation; results stay identical to a fresh context."""
    import splatter
    torch.cuda.synchronize()
    g1, v, cam = scene(3000, 160, 96, k=0)
    g2, _, _ = scene(30000, 160, 96, seed=3, k=0)
    vd = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran)]
    sp = splatter.Splatter.from_tensors(g1, vd, device=cuda)
    m0 = torch.cuda.memory_allocated(cuda)
    img = sp(0)
    img.sum().backward()
    m1 = torch.cuda.memory_allocated(cuda)
    assert m1 - m0 > 3000 * 64                       # at least the record array lives in torch's pool now
    # the same context serves a 10x larger scene (what adaptive_control does to a Splatter) ...
    with torch.no_grad():
        for name in ("pos", "rgb", "opa", "quat", "scale"):
            setattr(sp.gaussian_3ds, name, torch.nn.Parameter(g2[name].to(cuda)))
    go = S.make_grad_output(96, 160, 0).to(cuda) * (96 * 160)
    img2 = sp(0)
    img2.backward(go)
    assert torch.cuda.memory_allocated(cuda) > m1
    # ... with the same result as a fresh context
    sp_f = splatter.Splatter.from_tensors(g2, vd, device=cuda)
    img3 = sp_f(0)
    img3.backward(go)
    assert torch.equal(img2, img3)
    for a, b in zip(sp.gaussian_3ds.parameters(), sp_f.gaussian_3ds.parameters()):
        assert torch.equal(a.grad, b.grad)
    del sp, sp_f, img, img2, img3
    torch.cuda.synchronize()
