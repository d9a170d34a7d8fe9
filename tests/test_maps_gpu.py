"""GPU checks of the maps frame (`renderer.render_frame_maps`, `Splatter.render_maps`): depth / alpha maps and a
background colour from the blend kernels, against the fp64 maps oracle (tests/maps_oracle.py), plus identities with
the plain frame, determinism, launch counts and refusals."""
import pytest
import torch

import gs_oracle as O
import maps_oracle as MO
import synthetic as S
from helpers import abs_err, device_depth_keys, rel_err, scene

pytestmark = pytest.mark.gpu

IMG_ATOL = 1e-4
GRAD_RTOL = 1e-3
NAMES = ("pos", "rgb", "opa", "quat", "scale")
BG = (0.2, 0.5, 1.0)


def _splatter(g, views, dev, **kw):
    import splatter
    vs = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran) for v in views]
    return splatter.Splatter.from_tensors(g, vs, device=dev, **kw)


def _upstream(h, w, which, seed=0):
    """(g_image [H,W,3], g_depth [H,W], g_alpha [H,W]) with the outputs not in `which` set to zero."""
    gi = S.make_grad_output(h, w, seed) * (h * w)
    gen = torch.Generator().manual_seed(seed + 11)
    gd = torch.rand(h, w, generator=gen) * 2 - 1
    ga = torch.rand(h, w, generator=gen) * 2 - 1
    z = lambda t, k: t if k in which else torch.zeros_like(t)   # noqa: E731
    return z(gi, "image"), z(gd, "depth"), z(ga, "alpha")


def _oracle_maps(g, cam, ups, background=None, tiles=None):
    p = {k: v.double().clone().requires_grad_(True) for k, v in g.items()}
    dk = device_depth_keys(g, cam, torch.device("cuda", 0))
    outs = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, background=background,
                          tiles=tiles, depth_key=dk, return_aux=True)
    loss = sum((o * u.double()).sum() for o, u in zip(outs[:3], ups))
    loss.backward()
    grads = {k: (p[k].grad if p[k].grad is not None else torch.zeros_like(p[k])) for k in p}
    return [o.detach() for o in outs[:3]], grads, outs[3]


CONFIGS = [
    (2000, 128, 96, 0, (0.005, 0.05)),     # safe regime, no saturation
    (10000, 256, 256, 0, (0.05, 0.9)),     # C1
    (8000, 200, 120, 2, (0.05, 0.9)),      # rotated view (culling), non-multiple-of-16 size
    (5000, 96, 64, 0, (0.6, 0.98)),        # opaque: early termination everywhere
]
CASES = {"image": ("image",), "depth": ("depth",), "alpha": ("alpha",), "all+bg": ("image", "depth", "alpha")}


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("n,w,h,k,opa", CONFIGS, ids=["safe", "C1", "rotated", "opaque"])
def test_maps_frame_vs_oracle(gs, cuda, n, w, h, k, opa, case):
    g, v, cam = scene(n, w, h, k=k, opa_range=opa)
    bg = BG if case == "all+bg" else None
    ups = _upstream(h, w, CASES[case])
    (oimg, odep, oalp), ograds, _ = _oracle_maps(g, cam, ups, background=bg)
    sp = _splatter(g, [v], cuda)
    img, dep, alp = sp.render_maps(0, background=bg)
    assert img.shape == (h, w, 3) and dep.shape == (h, w) and alp.shape == (h, w)
    assert abs_err(img, oimg) < IMG_ATOL
    assert abs_err(alp, oalp) < 1e-4
    assert abs_err(dep, odep) < 1e-4 * float(odep.abs().max())
    torch.autograd.backward([img, dep, alp], [u.to(cuda) for u in ups])
    for name in NAMES:
        assert rel_err(getattr(sp.gaussian_3ds, name).grad, ograds[name]) < GRAD_RTOL, (name, case)
    assert sp.n_tile_gaussians == sp.frame_stats()["n_instances"] > 0


def test_maps_full_size_sampled_tiles(gs, cuda):
    """C3 RGB (2.4 M Gaussians, 1080p): map gradients only on sampled tiles - the heaviest tile (several chunks)
    and the tile with the most skipped tail among them.  Maps there and the gradients of their Gaussians match the
    fp64 oracle; every other gradient is exactly 0."""
    n, w, h = 2_400_000, 1920, 1080
    g, v, cam = scene(n, w, h, k=0)
    sp = _splatter(g, [v], cuda)
    with torch.no_grad():
        sp.render_maps(0)
    idx, accum = sp._rctx.sorted_instances()
    acc = accum.long().cpu()
    counts = acc[1:] - acc[:-1]
    tail = counts - sp._rctx.tile_consumed().long().cpu()
    top = (cam.Hp - h) // 2
    inside = torch.zeros(cam.nty, cam.ntx, dtype=torch.bool)
    inside[(top + 15) // 16:(top + h) // 16] = True                     # tiles fully inside the crop (rows)
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
    _, gd, ga = _upstream(h, w, ("depth", "alpha"))
    gd, ga = gd * mask_f, ga * mask_f
    gi = torch.zeros(h, w, 3)
    (_, odep, oalp), ograds, aux = _oracle_maps(g, cam, (gi, gd, ga), tiles=torch.tensor(tiles))
    for p in sp.gaussian_3ds.parameters():
        p.grad = None
    img, dep, alp = sp.render_maps(0)
    torch.autograd.backward([dep, alp], [gd.to(cuda), ga.to(cuda)])
    dcpu, acpu = dep.detach().cpu(), alp.detach().cpu()
    assert abs_err(acpu[mask_f], oalp[mask_f]) < 1e-4
    assert abs_err(dcpu[mask_f], odep[mask_f]) < 1e-4 * float(odep[mask_f].abs().max())
    # Gaussians with an instance on a sampled tile vs all others
    sel = torch.zeros(n, dtype=torch.bool)
    for t in tiles:
        sel[idx[int(acc[t]):int(acc[t + 1])].long().cpu()] = True
    for name in NAMES:
        got = getattr(sp.gaussian_3ds, name).grad.cpu()
        assert float(got[~sel].abs().max()) == 0.0, name
        assert rel_err(got[sel], ograds[name][sel]) < GRAD_RTOL, name


def test_maps_empty_views_render_the_background(gs, cuda):
    """Frames without a single tile instance, each on a FRESH context (no workspace from an earlier frame): an
    empty scene, and a scene entirely behind the camera.  image = bg, depth = alpha = 0; all gradients 0."""
    w, h = 64, 48
    v = S.make_view(w, h, 0)
    bg = torch.tensor(BG, device=cuda)
    empty = S.make_gaussians(0, w, h)
    sp = _splatter(empty, [v], cuda)
    with torch.no_grad():
        img, dep, alp = sp.render_maps(0, background=BG)
    assert torch.equal(img, bg.expand(h, w, 3)) and float(dep.abs().max()) == 0 and float(alp.abs().max()) == 0
    behind = S.make_gaussians(100, w, h)
    behind["pos"][:, 2] -= 100.0
    sp = _splatter(behind, [v], cuda)
    img, dep, alp = sp.render_maps(0, background=BG)
    assert int(sp.culling_mask.sum()) == 0 and sp.n_tile_gaussians == 0
    assert torch.equal(img.detach(), bg.expand(h, w, 3))
    assert float(dep.detach().abs().max()) == 0 and float(alp.detach().abs().max()) == 0
    gi, gd, ga = _upstream(h, w, ("image", "depth", "alpha"))
    torch.autograd.backward([img, dep, alp], [gi.to(cuda), gd.to(cuda), ga.to(cuda)])
    for name in NAMES:
        assert float(getattr(sp.gaussian_3ds, name).grad.abs().max()) == 0.0, name
    # the padded raw layout of render_frame_maps on the same (still instance-free) context
    import renderer
    g3 = sp.gaussian_3ds
    with torch.no_grad():
        raw, draw_, araw, _ = renderer.render_frame_maps(sp._rctx, g3.pos, g3.rgb, g3.opa, g3.quat, g3.scale, w, h,
                                                         v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, "abs", background=BG,
                                                         final=False)
    assert raw.shape == (48, 64, 3) and torch.equal(raw, bg.expand(48, 64, 3))
    assert float(draw_.abs().max()) == 0 and float(araw.abs().max()) == 0


def test_maps_identities(gs, cuda):
    """Black background + zero map gradients == the plain final frame; final maps == crop of the raw maps; two maps
    frames are bit-identical; a maps frame launches as many kernels as a plain frame."""
    gaussian, renderer = gs
    n, w, h = 8000, 200, 120
    g, v, cam = scene(n, w, h, k=2, opa_range=(0.05, 0.9))
    go = (S.make_grad_output(h, w, 0) * (h * w)).to(cuda)
    sp = _splatter(g, [v], cuda)
    gp = sp.gaussian_3ds

    def run(maps):
        for p in gp.parameters():
            p.grad = None
        k0 = gaussian.kernel_launches()
        if maps:
            img, dep, alp = sp.render_maps(0)
            torch.autograd.backward([img], [go])     # no gradient for depth / alpha: zeros
        else:
            img = sp(0)
            img.backward(go)
        torch.cuda.synchronize()
        return img.detach().clone(), [p.grad.clone() for p in gp.parameters()], gaussian.kernel_launches() - k0

    run(False)                                       # a context's first frame also fills its 0..N-1 sort values
    img_p, gr_p, l_p = run(False)
    img_m, gr_m, l_m = run(True)
    assert torch.equal(img_p, img_m)
    bit_equal = all(torch.equal(a, b) for a, b in zip(gr_p, gr_m))
    print(f"maps vs plain gradients bit-equal: {bit_equal}")
    for a, b in zip(gr_p, gr_m):
        assert rel_err(b, a) < 1e-6
    assert l_p == l_m
    # final planes are the exact crop of the raw planes
    rctx = sp._rctx
    with torch.no_grad():
        fin, dfin, afin, raw, draw_, araw, _ = rctx.forward_maps(
            gp.pos.detach(), gp.rgb.detach(), gp.opa.detach(), gp.quat.detach(), gp.scale.detach(), w, h, v.fx, v.fy,
            v.rot, v.tran, 0.3, 0.05, 0, [0.2, 0.5, 1.0], True)
    assert torch.equal(fin, cam.crop(raw.clamp(0, 1)))
    assert torch.equal(dfin, cam.crop(draw_.unsqueeze(-1)).squeeze(-1))
    assert torch.equal(afin, cam.crop(araw.unsqueeze(-1)).squeeze(-1))
    assert float(araw.max()) <= 1.0 and float(araw.min()) >= 0.0
    # determinism of the whole maps frame
    _, gd, ga = _upstream(h, w, ("depth", "alpha"))

    def run_full():
        for p in gp.parameters():
            p.grad = None
        outs = sp.render_maps(0, background=BG)
        torch.autograd.backward(list(outs), [go, gd.to(cuda), ga.to(cuda)])
        return [o.detach().clone() for o in outs] + [p.grad.clone() for p in gp.parameters()]

    a, b = run_full(), run_full()
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_maps_refusals(gs, cuda):
    gaussian, renderer = gs
    g, v, cam = scene(500, 64, 48)
    # SH colour
    gsh, _, _ = scene(500, 64, 48, sh_dim=27)
    sp_sh = _splatter(gsh, [v], cuda, use_sh_coeff=True)
    with pytest.raises(RuntimeError, match="RGB colour"):
        sp_sh.render_maps(0)
    sp = _splatter(g, [v], cuda)
    # packed path
    gather = gaussian.tuned("gather")
    assert gather != 0
    gaussian.tune("gather", 0)
    try:
        with pytest.raises(RuntimeError, match="gather path"):
            sp.render_maps(0)
    finally:
        gaussian.tune("gather", gather)
    assert gaussian.tuned("gather") == gather
    img, dep, alp = sp.render_maps(0)              # usable again
    (img.sum() + dep.sum() + alp.sum()).backward()
    # maps backward after a plain forward
    gp = sp.gaussian_3ds
    args = [t.detach() for t in (gp.pos, gp.rgb, gp.opa, gp.quat, gp.scale)]
    rctx = sp._rctx
    outs = rctx.forward_maps(*args, 64, 48, v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, 0, None, True)
    with torch.no_grad():
        sp(0)
    grads = [torch.empty_like(t) for t in args]
    with pytest.raises(RuntimeError, match="not gs_render_forward_maps"):
        rctx.backward_maps_into(*args, outs[3], outs[4], outs[5], torch.zeros_like(outs[0]), torch.zeros_like(outs[1]),
                                torch.zeros_like(outs[2]), True, *grads)
    # wrong shapes / dtypes
    outs = rctx.forward_maps(*args, 64, 48, v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, 0, None, True)
    with pytest.raises(RuntimeError, match="gradients must be"):
        rctx.backward_maps_into(*args, outs[3], outs[4], outs[5], torch.zeros_like(outs[0]),
                                torch.zeros(47, 64, device=cuda), torch.zeros_like(outs[2]), True, *grads)
    with pytest.raises(RuntimeError, match="float32"):
        rctx.backward_maps_into(*args, outs[3], outs[4], outs[5], torch.zeros_like(outs[0]),
                                torch.zeros_like(outs[1]).double(), torch.zeros_like(outs[2]), True, *grads)
    with pytest.raises(RuntimeError, match="float32"):
        rctx.forward_maps(args[0].double(), *args[1:], 64, 48, v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, 0, None, True)
    with pytest.raises(RuntimeError, match="3 values"):
        rctx.forward_maps(*args, 64, 48, v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, 0, [1.0, 0.0], True)
    with pytest.raises(ValueError, match="3 values"):
        sp.render_maps(0, background=(1.0, 0.0))
    # data-parallel gradient push: refused rather than silently wrong (the configuration is only validated here)
    bucket = torch.zeros(64, device=cuda)
    rctx.set_grad_push(bucket.data_ptr(), [bucket.data_ptr(), bucket.data_ptr()], 32, 0)
    try:
        with pytest.raises(RuntimeError, match="gradient push"):
            rctx.forward_maps(*args, 64, 48, v.fx, v.fy, v.rot, v.tran, 0.3, 0.05, 0, None, True)
    finally:
        rctx.clear_grad_push()
