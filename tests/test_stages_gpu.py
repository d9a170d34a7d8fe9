"""GPU parity of the legacy per-stage boundary (the reference's `gaussian` module surface)
against the CPU oracle and against the reference's own CUDA build on identical inputs (its
outputs stored in tests/golden/ref_*.npz by tests/golden/make_golden.py).  Protocol P1/P2/P4
of SURVEY.md §8c.

Tolerances (BASELINE.json north_star): image <= 1e-4 abs per pixel; gradients <= 1e-3
relative (max |delta| / max |reference| per tensor); projection 1e-5 relative.
"""
import numpy as np
import pytest
import torch

import golden_cases as GC
import gs_oracle as O
from helpers import abs_err, rel_err, require_golden, scene, sorted_instances_cpu

pytestmark = pytest.mark.gpu

IMG_ATOL = 1e-4
GRAD_RTOL = 1e-3


def _proj_inputs(n, w, h, k, dev, seed=0):
    g, v, cam = scene(n, w, h, seed=seed, k=k)
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    return g, cam, nq.contiguous(), ns.contiguous()


@pytest.mark.parametrize("k", [0, 1, 3])
def test_global_culling_forward_backward_vs_oracle(gs, cuda, k):
    gaussian, renderer = gs
    g, cam, nq, ns = _proj_inputs(5000, 256, 256, k, cuda)
    # oracle (fp64 for a clean reference)
    pos64 = g["pos"].double().requires_grad_(True)
    q64 = nq.double().requires_grad_(True)
    s64 = ns.double().requires_grad_(True)
    rp, rc, m = O.global_culling(pos64, q64, s64, cam.rot.double(), cam.tran.double(), cam.near, cam.half_w, cam.half_h)
    gen = torch.Generator().manual_seed(7)
    go_p = torch.randn(rp.shape, generator=gen, dtype=torch.float64)
    go_c = torch.randn(rc.shape, generator=gen, dtype=torch.float64)
    (rp * go_p).sum().backward(retain_graph=True)
    (rc * go_c).sum().backward()
    # ours
    pos = g["pos"].to(cuda).requires_grad_(True)
    q = nq.to(cuda).requires_grad_(True)
    s = ns.to(cuda).requires_grad_(True)
    op, oc, om = renderer.global_culling(pos, q, s, cam.rot.to(cuda), cam.tran.to(cuda), cam.near, cam.half_w, cam.half_h)
    assert om.dtype == torch.int64
    # mask may only differ for points within rounding distance of the frustum planes
    mm = (om.cpu() != m)
    assert int(mm.sum()) <= 2
    keep = ~mm
    assert 0 < int(m.sum()) <= m.numel()
    assert rel_err(op.cpu()[keep], rp[keep]) < 1e-5
    assert rel_err(oc.cpu()[keep], rc[keep]) < 2e-5
    (op * go_p.float().to(cuda)).sum().backward(retain_graph=True)
    (oc * go_c.float().to(cuda)).sum().backward()
    assert rel_err(pos.grad.cpu()[keep], pos64.grad[keep]) < 1e-4
    assert rel_err(q.grad.cpu()[keep], q64.grad[keep]) < 1e-4
    assert rel_err(s.grad.cpu()[keep], s64.grad[keep]) < 1e-4
    # culled rows: outputs and gradients are exactly zero
    culled = (om == 0)
    if int(culled.sum()):
        assert float(op[culled].abs().max()) == 0 and float(pos.grad[culled].abs().max()) == 0


def test_global_culling_vs_reference_build(gs, cuda):
    """Against the reference build's outputs on the same inputs (tests/golden/ref_culling.npz: the
    full mask, everything else on a sample of visible rows)."""
    gaussian, renderer = gs
    gold = require_golden("ref_culling.npz")
    g, cam, nq, ns = _proj_inputs(20000, 640, 360, 1, cuda)
    pos = g["pos"].to(cuda).requires_grad_(True)
    q = nq.to(cuda).requires_grad_(True)
    s = ns.to(cuda).requires_grad_(True)
    op, oc, om = renderer.global_culling(pos, q, s, cam.rot.to(cuda), cam.tran.to(cuda), cam.near, cam.half_w,
                                         cam.half_h)
    gen = torch.Generator().manual_seed(3)
    gp = torch.randn(op.shape, generator=gen).to(cuda)
    gc = torch.randn(oc.shape, generator=gen).to(cuda)
    ((op * gp).sum() + (oc * gc).sum()).backward()
    assert torch.equal(om.cpu().bool(), gold["mask"])
    r = gold["rows"].long()
    a = [t.detach().cpu()[r] for t in (op, oc, pos.grad, q.grad, s.grad)]
    # depth (the sort key) is bit-identical to the reference kernel's: same ordering keys
    assert torch.equal(a[0][:, 2], gold["res_pos"][:, 2])
    assert rel_err(a[0], gold["res_pos"]) < 1e-5 and rel_err(a[1], gold["res_cov"]) < 2e-5
    for x, k in zip(a[2:], ("grad_pos", "grad_quat", "grad_scale")):
        assert rel_err(x, gold[k]) < 1e-4, k


def _tile_lists(gmod, pos, cov, cam, dev, thresh=0.05, maxp=None):
    T = cam.ntx * cam.nty
    n = pos.shape[0]
    maxp = maxp or max(n // 2, 8)
    cnt = torch.zeros(T, dtype=torch.int32, device=dev)
    lst = torch.full((T, maxp), -1, dtype=torch.int32, device=dev)
    cobj = gmod.Gaussian3ds()
    cobj.pos, cobj.cov = pos.to(dev).contiguous(), cov.to(dev).contiguous()
    cobj.rgb = torch.zeros(n, 3, device=dev)
    cobj.opa = torch.zeros(n, device=dev)
    tiles = gmod.Tiles()
    gmod.calc_tile_list(cobj, tiles, cnt, lst, thresh, 2, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                        cam.topmost)
    return cnt, lst


def _per_tile_sets(cnt, lst):
    cnt, lst = cnt.cpu(), lst.cpu()
    return [sorted(lst[t, :int(cnt[t])].tolist()) for t in range(cnt.numel())]


def test_tile_binning_and_gather_vs_oracle(gs, cuda):
    gaussian, _ = gs
    g, v, cam = scene(6000, 320, 200, k=0)
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    rp, rc, m = O.global_culling(g["pos"], nq, ns, cam.rot, cam.tran, cam.near, cam.half_w, cam.half_h)
    idx = torch.nonzero(m.bool()).squeeze(-1)
    pos, cov = rp[idx].contiguous(), rc[idx].contiguous()
    tx0, tx1, ty0, ty1 = O.tile_rects(pos[:, :2], cov, 0.05, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                                      cam.topmost)
    want = [[] for _ in range(cam.ntx * cam.nty)]
    for i in range(pos.shape[0]):
        for ty in range(int(ty0[i]), int(ty1[i])):
            for tx in range(int(tx0[i]), int(tx1[i])):
                want[ty * cam.ntx + tx].append(i)
    cnt, lst = _tile_lists(gaussian, pos, cov, cam, cuda)
    got = _per_tile_sets(cnt, lst)
    flips = sum(len(set(a) ^ set(b)) for a, b in zip(got, want))
    total = sum(len(w) for w in want)
    assert total > 0 and flips <= max(2, total // 20000), (flips, total)
    # gather_gaussians: compacts the dense lists in tile order
    accum = torch.zeros(cnt.numel() + 1, dtype=torch.int32, device=cuda)
    accum[1:] = torch.cumsum(cnt, 0)
    M = int(accum[-1])
    gathered = torch.empty(M, dtype=torch.int32, device=cuda)
    tids = torch.empty(M, dtype=torch.int32, device=cuda)
    gaussian.gather_gaussians(accum, lst, gathered, tids, int(cnt.max()))
    acc = accum.cpu()
    gat, tid = gathered.cpu(), tids.cpu()
    for t in (0, 5, cnt.numel() // 2, cnt.numel() - 1):
        s, e = int(acc[t]), int(acc[t + 1])
        assert sorted(gat[s:e].tolist()) == got[t]
        assert bool((tid[s:e] == t).all())


def _assert_same_sets(sets, gold, prefix=""):
    """Per-tile sets equal to the reference build's, compared through GC.tile_set_digest."""
    for k, a in GC.tile_set_digest(sets).items():
        assert np.array_equal(a, gold[prefix + k].numpy()), prefix + k


def test_tile_binning_vs_reference_build(gs, cuda):
    gaussian, _ = gs
    g, v, cam = scene(30000, 640, 368, k=0)
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    rp, rc, m = O.global_culling(g["pos"], nq, ns, cam.rot, cam.tran, cam.near, cam.half_w, cam.half_h)
    idx = torch.nonzero(m.bool()).squeeze(-1)
    pos, cov = rp[idx].contiguous(), rc[idx].contiguous()
    _assert_same_sets(_per_tile_sets(*_tile_lists(gaussian, pos, cov, cam, cuda)), require_golden("ref_tiles.npz"))


def _draw_case(n, w, h, opa_range, seed=0):
    g, v, cam = scene(n, w, h, seed=seed, opa_range=opa_range)
    inst = sorted_instances_cpu(g, cam)
    gen = torch.Generator().manual_seed(seed + 11)
    grad_img = (torch.rand(cam.Hp, cam.Wp, 3, generator=gen) * 2 - 1)
    return cam, inst, grad_img


def _run_draw(R, inst, cam, grad_img, dev):
    t = {k: inst[k].to(dev).float().contiguous().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
    accum = inst["accum"].to(dev)
    dummy = torch.zeros(3, device=dev)
    img = R.draw(t["pos"], t["rgb"], t["opa"], t["cov"], accum, cam.Hp, cam.Wp, cam.fx, cam.fy, False, False, False,
                 True, dummy, dummy, dummy, dummy)
    img.backward(grad_img.to(dev))
    return img.detach(), {k: t[k].grad for k in t}


def _oracle_draw(inst, cam, grad_img):
    t = {k: inst[k].double().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
    img = O.draw(t["pos"], t["rgb"], t["opa"], t["cov"], inst["accum"], cam.Hp, cam.Wp, cam.fx, cam.fy)
    img.backward(grad_img.double())
    return img.detach(), {k: t[k].grad for k in t}


@pytest.mark.parametrize("case", ["safe", "opaque", "many_chunks"])
def test_draw_forward_backward_vs_oracle(gs, cuda, case):
    _, renderer = gs
    if case == "safe":          # no pixel saturates: pure arithmetic parity
        cam, inst, gi = _draw_case(4000, 128, 96, (0.005, 0.05))
    elif case == "opaque":      # early termination + whole-tile early exit
        cam, inst, gi = _draw_case(6000, 96, 64, (0.5, 0.95), seed=1)
    else:                       # several staging chunks per tile (count > 256) with saturation
        cam, inst, gi = _draw_case(20000, 64, 64, (0.05, 0.6), seed=2)
    img, grads = _run_draw(renderer, inst, cam, gi, cuda)
    oimg, ograds = _oracle_draw(inst, cam, gi)
    assert abs_err(img, oimg) < IMG_ATOL
    assert rel_err(grads["rgb"], ograds["rgb"]) < GRAD_RTOL
    assert rel_err(grads["opa"], ograds["opa"]) < GRAD_RTOL
    assert rel_err(grads["cov"], ograds["cov"]) < GRAD_RTOL
    assert rel_err(grads["pos"][:, :2], ograds["pos"][:, :2]) < GRAD_RTOL
    assert float(grads["pos"][:, 2].abs().max()) == 0.0      # depth: sort key only


def _assert_matches_reference_draw(img, grads, gold):
    """Image on the stored pixel sample, gradients on the stored instance sample."""
    assert abs_err(img.reshape(-1, 3).cpu()[gold["pix"].long()], gold["image"]) < IMG_ATOL
    r = gold["rows"].long()
    for k in ("rgb", "opa", "cov"):
        assert rel_err(grads[k].cpu()[r], gold["grad_" + k]) < GRAD_RTOL, k
    assert rel_err(grads["pos"][:, :2].cpu()[r], gold["grad_pos"]) < GRAD_RTOL


def test_draw_vs_reference_build_safe_regime(gs, cuda):
    """P4: the sorted inputs the reference build was given (tests/golden/ref_draw.npz holds its
    outputs), inside its safe regime (per-tile count <= 500, no pixel reaching T < 1e-4;
    SURVEY.md §8c hazards 1-3)."""
    _, renderer = gs
    cam, inst, gi = _draw_case(4000, 256, 256, (0.005, 0.05))
    counts = inst["accum"][1:] - inst["accum"][:-1]
    assert int(counts.max()) <= 500
    _assert_matches_reference_draw(*_run_draw(renderer, inst, cam, gi, cuda), require_golden("ref_draw.npz"))


def test_draw_edge_cases(gs, cuda):
    gaussian, renderer = gs
    # empty instance list: black image, no crash
    accum = torch.zeros(4 * 2 + 1, dtype=torch.int32, device=cuda)
    z = torch.zeros(0, device=cuda)
    img = renderer.draw(z.reshape(0, 3), z.reshape(0, 3), z, z.reshape(0, 2, 2), accum, 32, 64, 50.0, 50.0)
    assert img.shape == (32, 64, 3) and float(img.abs().max()) == 0.0
    # unsupported flags fail loudly instead of silently differing (weight_normalize / sigmoid)
    with pytest.raises(RuntimeError):
        renderer.draw(z.reshape(0, 3), z.reshape(0, 3), z, z.reshape(0, 2, 2), accum, 32, 64, 50.0, 50.0, True)
    # wrong dtype / device are rejected by the shim (the reference would silently corrupt)
    with pytest.raises(RuntimeError):
        gaussian.global_culling(torch.zeros(4, 3), torch.zeros(4, 4), torch.zeros(4, 3), torch.eye(3), torch.zeros(3),
                                torch.zeros(4, 3), torch.zeros(4, 2, 2), torch.zeros(4, dtype=torch.long), 0.3, 1.0, 1.0)


def test_world2camera_and_jacobian(gs, cuda):
    gaussian, renderer = gs
    gen = torch.Generator().manual_seed(5)
    p = torch.randn(1000, 3, generator=gen)
    p[:, 2] += 4
    rot = torch.linalg.qr(torch.randn(3, 3, generator=gen))[0].contiguous()
    tran = torch.randn(3, generator=gen)
    pc = p.to(cuda).requires_grad_(True)
    out = renderer.world2camera_func(pc, rot.to(cuda), tran.to(cuda))
    assert rel_err(out, p @ rot.T + tran) < 1e-6
    gout = torch.randn(1000, 3, generator=gen)
    out.backward(gout.to(cuda))
    assert rel_err(pc.grad, gout @ rot) < 1e-6
    jac = torch.empty(1000, 3, 3, device=cuda)
    gaussian.jacobian(p.to(cuda).contiguous(), jac)
    x, y, z = p.unbind(-1)
    r = p.norm(dim=-1)
    zero = torch.zeros_like(x)
    want = torch.stack([1 / z, zero, -x / z ** 2, zero, 1 / z, -y / z ** 2, x / r, y / r, z / r], -1).reshape(-1, 3, 3)
    assert rel_err(jac, want) < 1e-5


# ---- SH colour (use_sh_coeff): per-pixel ray SH evaluated inside the blend -----------------
def _sh_case(n, w, h, sh_dim, opa_range, seed=0):
    g, v, cam = scene(n, w, h, seed=seed, sh_dim=sh_dim, opa_range=opa_range)
    inst = sorted_instances_cpu(g, cam, use_sh=True)
    gen = torch.Generator().manual_seed(seed + 21)
    grad_img = torch.rand(cam.Hp, cam.Wp, 3, generator=gen) * 2 - 1
    rays = O.ray_info(cam.rot, cam.tran, cam.Hp, cam.Wp, cam.fx, cam.fy)
    return cam, inst, grad_img, rays


def _run_draw_sh(R, inst, cam, grad_img, rays, dev):
    t = {k: inst[k].to(dev).float().contiguous().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
    r = [x.to(dev).float().contiguous() for x in rays]
    img = R.draw(t["pos"], t["rgb"], t["opa"], t["cov"], inst["accum"].to(dev), cam.Hp, cam.Wp, cam.fx, cam.fy, False,
                 False, True, True, r[0], r[1], r[2], r[3])
    img.backward(grad_img.to(dev))
    return img.detach(), {k: t[k].grad for k in t}


@pytest.mark.parametrize("sh_dim,case", [(27, "safe"), (27, "opaque"), (48, "safe"), (48, "opaque")])
def test_draw_sh_forward_backward_vs_oracle(gs, cuda, sh_dim, case):
    _, renderer = gs
    if case == "safe":
        cam, inst, gi, rays = _sh_case(1500, 96, 64, sh_dim, (0.005, 0.05))
    else:
        cam, inst, gi, rays = _sh_case(3000, 64, 48, sh_dim, (0.4, 0.95), seed=3)
    img, grads = _run_draw_sh(renderer, inst, cam, gi, rays, cuda)
    t = {k: inst[k].double().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
    r64 = [x.double() for x in rays]
    oimg = O.draw(t["pos"], t["rgb"], t["opa"], t["cov"], inst["accum"], cam.Hp, cam.Wp, cam.fx, cam.fy, True, *r64)
    oimg.backward(gi.double())
    assert abs_err(img, oimg) < IMG_ATOL
    for k in ("rgb", "opa", "cov"):
        assert rel_err(grads[k], t[k].grad) < GRAD_RTOL, k
    assert rel_err(grads["pos"][:, :2], t["pos"].grad[:, :2]) < GRAD_RTOL


def test_draw_sh_vs_reference_build(gs, cuda):
    """P4 for SH-27 inside the reference's safe regime (<= 160 instances per tile in backward);
    the reference build's outputs are tests/golden/ref_draw_sh.npz."""
    _, renderer = gs
    cam, inst, gi, rays = _sh_case(2500, 256, 192, 27, (0.005, 0.05))
    counts = inst["accum"][1:] - inst["accum"][:-1]
    assert int(counts.max()) <= 160
    _assert_matches_reference_draw(*_run_draw_sh(renderer, inst, cam, gi, rays, cuda),
                                   require_golden("ref_draw_sh.npz"))


# ---- legacy tile-culling methods 0 ("dist") and 1 ("prob"): brute force over (Gaussian, tile) ----
def _tile_bounds(cam, dev):
    left = torch.linspace(-cam.Wp / 2, cam.Wp / 2, cam.ntx + 1)[:-1]
    top = torch.linspace(-cam.Hp / 2, cam.Hp / 2, cam.nty + 1)[:-1]
    l = (left / cam.fx).repeat(cam.nty)
    r = ((left + 16) / cam.fx).repeat(cam.nty)
    t = (top / cam.fy).repeat_interleave(cam.ntx)
    b = ((top + 16) / cam.fy).repeat_interleave(cam.ntx)
    return [x.float().contiguous().to(dev) for x in (t, b, l, r)]


def _legacy_lists(gmod, method, pos, cov, cam, thresh, dev):
    T = cam.ntx * cam.nty
    n = pos.shape[0]
    cnt = torch.zeros(T, dtype=torch.int32, device=dev)
    lst = torch.full((T, n), -1, dtype=torch.int32, device=dev)
    cobj = gmod.Gaussian3ds()
    cobj.pos, cobj.cov = pos.to(dev).contiguous(), cov.to(dev).contiguous()
    cobj.rgb, cobj.opa = torch.zeros(n, 3, device=dev), torch.zeros(n, device=dev)
    tiles = gmod.Tiles()
    tiles.top, tiles.bottom, tiles.left, tiles.right = _tile_bounds(cam, dev)
    gmod.calc_tile_list(cobj, tiles, cnt, lst, thresh, method, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                        cam.topmost)
    return _per_tile_sets(cnt, lst)


def _small_projected_scene():
    g, v, cam = scene(1500, 160, 96, k=0)
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    rp, rc, m = O.global_culling(g["pos"], nq, ns, cam.rot, cam.tran, cam.near, cam.half_w, cam.half_h)
    idx = torch.nonzero(m.bool()).squeeze(-1)
    return rp[idx].contiguous(), rc[idx].contiguous(), cam


def test_tile_methods_dist_and_prob_vs_torch(gs, cuda):
    gaussian, _ = gs
    pos, cov, cam = _small_projected_scene()
    t, b, l, r = [x.cpu() for x in _tile_bounds(cam, cuda)]
    # method 0 "dist" (gaussian.cu:101-136): centre distance^2 to the tile centre < thresh
    thresh0 = (cam.tile_lx / 0.5) ** 2                                       # splatter.py:576
    cx, cy = (l + r) / 2, (t + b) / 2
    d2 = (pos[:, 0:1] - cx[None]) ** 2 + (pos[:, 1:2] - cy[None]) ** 2        # [n, T]
    want0 = [sorted(torch.nonzero(d2[:, k] < thresh0).squeeze(-1).tolist()) for k in range(t.numel())]
    got0 = _legacy_lists(gaussian, 0, pos, cov, cam, thresh0, cuda)
    flips0 = sum(len(set(a) ^ set(w)) for a, w in zip(got0, want0))
    assert sum(map(len, want0)) > 0 and flips0 <= 2
    # method 1 "prob" (gaussian.cu:138-195): bbox of the thresh-ellipse overlaps the tile
    a, bb, c, d = cov.reshape(-1, 4).unbind(-1)
    det = a * d - bb * c
    t2 = -2 * torch.log(torch.tensor(0.05))
    sx = torch.sqrt(a / (det + 1e-14) * t2 * det)
    sy = torch.sqrt(d / (det + 1e-14) * t2 * det)
    hit = ~((r[None] < (pos[:, 0:1] - sx[:, None])) | ((pos[:, 0:1] + sx[:, None]) < l[None]) |
            (b[None] < (pos[:, 1:2] - sy[:, None])) | ((pos[:, 1:2] + sy[:, None]) < t[None])) & (det > 0)[:, None]
    want1 = [sorted(torch.nonzero(hit[:, k]).squeeze(-1).tolist()) for k in range(t.numel())]
    got1 = _legacy_lists(gaussian, 1, pos, cov, cam, 0.05, cuda)
    flips1 = sum(len(set(a_) ^ set(w)) for a_, w in zip(got1, want1))
    assert sum(map(len, want1)) > 0 and flips1 <= 2


def test_tile_methods_dist_and_prob_vs_reference_build(gs, cuda):
    gaussian, _ = gs
    gold = require_golden("ref_tile_methods.npz")
    pos, cov, cam = _small_projected_scene()
    for method, thresh in ((0, (cam.tile_lx / 0.5) ** 2), (1, 0.05)):
        _assert_same_sets(_legacy_lists(gaussian, method, pos, cov, cam, thresh, cuda), gold, f"m{method}_")
