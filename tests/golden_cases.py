"""Golden-vector cases shared by tests/golden/make_golden.py (runs the REFERENCE's CUDA
build on a GPU and writes tests/golden/*.npz) and tests/test_oracle.py (checks the CPU
oracle against those files).  All inputs are regenerated from seeds; the .npz files hold
the reference's outputs (plus the few inputs that are themselves oracle-derived)."""
import numpy as np
import torch

import gs_oracle as O
import synthetic as S
from helpers import abs_err, rel_err, scene, sorted_instances_cpu

CASES = {
    "project.npz": dict(n=2000, w=256, h=256, k=1),
    "tiles.npz": dict(n=3000, w=320, h=200, k=0),
    "draw_rgb.npz": dict(n=1500, w=128, h=96, opa=(0.005, 0.05)),
    "draw_sh.npz": dict(n=1000, w=128, h=96, opa=(0.005, 0.05), sh_dim=27),      # max tile <= 160
    # whole-pipeline case: must sit inside the reference's own limits (SURVEY.md hazards 1, 4):
    # max tile count 86 <= MAXP = n//20 = 100 (dense-list capacity, splatter.py:569) and NO two
    # instances of a tile collide in the reference's quantised fp32 sort key (splatter.py:610-612)
    "frame_c1.npz": dict(n=2000, w=192, h=128, opa=(0.005, 0.05), sigma=(0.4, 1.5), seed=0),
}


def project_inputs():
    c = CASES["project.npz"]
    g, v, cam = scene(c["n"], c["w"], c["h"], k=c["k"])
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    gen = torch.Generator().manual_seed(101)
    go_pos = torch.randn(c["n"], 3, generator=gen)
    go_cov = torch.randn(c["n"], 2, 2, generator=gen)
    return g["pos"], nq.contiguous(), ns.contiguous(), cam, go_pos, go_cov


def tiles_inputs():
    c = CASES["tiles.npz"]
    g, v, cam = scene(c["n"], c["w"], c["h"], k=c["k"])
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    rp, rc, m = O.global_culling(g["pos"], nq, ns, cam.rot, cam.tran, cam.near, cam.half_w, cam.half_h)
    idx = torch.nonzero(m.bool()).squeeze(-1)
    return rp[idx].contiguous(), rc[idx].contiguous(), cam


def draw_inputs():
    c = CASES["draw_rgb.npz"]
    g, v, cam = scene(c["n"], c["w"], c["h"], opa_range=c["opa"])
    inst = sorted_instances_cpu(g, cam)
    gen = torch.Generator().manual_seed(202)
    grad_img = torch.rand(cam.Hp, cam.Wp, 3, generator=gen) * 2 - 1
    return inst, cam, grad_img


def draw_sh_inputs():
    c = CASES["draw_sh.npz"]
    g, v, cam = scene(c["n"], c["w"], c["h"], opa_range=c["opa"], sh_dim=c["sh_dim"])
    inst = sorted_instances_cpu(g, cam, use_sh=True)
    gen = torch.Generator().manual_seed(303)
    grad_img = torch.rand(cam.Hp, cam.Wp, 3, generator=gen) * 2 - 1
    rays = O.ray_info(cam.rot, cam.tran, cam.Hp, cam.Wp, cam.fx, cam.fy)
    return inst, cam, grad_img, rays


def frame_inputs():
    c = CASES["frame_c1.npz"]
    return frame_case(c["n"], c["w"], c["h"], c["opa"], c["sigma"], c["seed"])


def frame_case(n, w, h, opa, sigma, seed):
    g, v, cam = scene(n, w, h, seed=seed, opa_range=opa, sigma_px=sigma)
    go = S.make_grad_output(h, w, seed) * (h * w)
    return g, v, cam, go


def reference_key_collisions(g, cam):
    """(# same-tile neighbours that tie/invert under the reference's fp32 composite key,
    max tile count, MAXP) for a scene - emulated on the CPU with the oracle front end."""
    inst = sorted_instances_cpu(g, cam)
    acc = inst["accum"].long()
    cnt = acc[1:] - acc[:-1]
    depth = inst["pos"][:, 2].float()
    tile = torch.repeat_interleave(torch.arange(cnt.numel()), cnt).float()
    key = depth + tile * (depth.max() + 1)
    bad = int(((key[1:] <= key[:-1]) & (tile[1:] == tile[:-1])).sum())
    return bad, int(cnt.max()), g["pos"].shape[0] // 20


def sample(rows, k, seed=0):
    """A fixed, seeded sample of at most k entries of the index tensor `rows`.  The first j entries
    of a sample are the sample for k = j, so a stored sample can be shortened without re-running."""
    rows = torch.as_tensor(rows).flatten()
    perm = torch.randperm(rows.numel(), generator=torch.Generator().manual_seed(seed))
    return rows[perm[:k]]


def tile_set_digest(sets):
    """Per-tile count, sum and sum of squares of the Gaussian ids in each tile's list: equal digests
    mean equal per-tile sets for any change short of a coincidence in all three."""
    ids = [torch.tensor(s, dtype=torch.int64) for s in sets]
    return dict(counts=np.array([i.numel() for i in ids], dtype=np.int32),
                sum=np.array([int(i.sum()) for i in ids], dtype=np.int64),
                sum_sq=np.array([int((i * i).sum()) for i in ids], dtype=np.int64))


def check_oracle_against(name, gold):
    if name == "project.npz":
        pos, nq, ns, cam, go_pos, go_cov = project_inputs()
        p = pos.double().requires_grad_(True)
        q = nq.double().requires_grad_(True)
        s = ns.double().requires_grad_(True)
        rp, rc, m = O.global_culling(p, q, s, cam.rot.double(), cam.tran.double(), cam.near, cam.half_w, cam.half_h)
        ((rp * go_pos.double()).sum() + (rc * go_cov.double()).sum()).backward()
        assert int((m != gold["mask"]).sum()) <= 1
        keep = m == gold["mask"]
        assert rel_err(rp[keep], gold["res_pos"][keep]) < 1e-5
        assert rel_err(rc[keep], gold["res_cov"][keep]) < 2e-5
        assert rel_err(p.grad[keep], gold["grad_pos"][keep]) < 1e-4
        assert rel_err(q.grad[keep], gold["grad_quat"][keep]) < 1e-4
        assert rel_err(s.grad[keep], gold["grad_scale"][keep]) < 1e-4
    elif name == "tiles.npz":
        pos, cov, cam = tiles_inputs()
        tx0, tx1, ty0, ty1 = O.tile_rects(pos[:, :2], cov, 0.05, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty,
                                          cam.leftmost, cam.topmost)
        T = cam.ntx * cam.nty
        want = [[] for _ in range(T)]
        for i in range(pos.shape[0]):
            for ty in range(int(ty0[i]), int(ty1[i])):
                for tx in range(int(tx0[i]), int(tx1[i])):
                    want[ty * cam.ntx + tx].append(i)
        counts, flat = gold["counts"].tolist(), gold["flat_ids"].tolist()
        flips, o = 0, 0
        for t in range(T):
            got = flat[o:o + counts[t]]
            o += counts[t]
            flips += len(set(got) ^ set(want[t]))
        assert flips <= 2, flips
    elif name == "draw_rgb.npz":
        inst, cam, grad_img = draw_inputs()
        for k in ("pos", "rgb", "opa", "cov"):          # oracle-derived inputs are stored too
            assert torch.allclose(inst[k], gold["in_" + k], atol=0, rtol=0) or rel_err(inst[k], gold["in_" + k]) < 1e-6
        t = {k: gold["in_" + k].double().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
        img = O.draw(t["pos"], t["rgb"], t["opa"], t["cov"], gold["in_accum"], cam.Hp, cam.Wp, cam.fx, cam.fy)
        img.backward(grad_img.double())
        assert abs_err(img, gold["image"]) < 1e-4
        assert rel_err(t["rgb"].grad, gold["grad_rgb"]) < 1e-3
        assert rel_err(t["opa"].grad, gold["grad_opa"]) < 1e-3
        assert rel_err(t["cov"].grad, gold["grad_cov"]) < 1e-3
        assert rel_err(t["pos"].grad[:, :2], gold["grad_pos"][:, :2]) < 1e-3
    elif name == "draw_sh.npz":
        inst, cam, grad_img, rays = draw_sh_inputs()
        t = {k: gold["in_" + k].double().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
        img = O.draw(t["pos"], t["rgb"], t["opa"], t["cov"], gold["in_accum"], cam.Hp, cam.Wp, cam.fx, cam.fy, True,
                     *[r.double() for r in rays])
        img.backward(grad_img.double())
        assert abs_err(img, gold["image"]) < 1e-4
        for k in ("rgb", "opa", "cov"):
            assert rel_err(t[k].grad, gold["grad_" + k]) < 1e-3, k
        assert rel_err(t["pos"].grad[:, :2], gold["grad_pos"][:, :2]) < 1e-3
    elif name == "frame_c1.npz":
        g, v, cam, go = frame_inputs()
        p = {k: x.double().clone().requires_grad_(True) for k, x in g.items()}
        img = O.render(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam)
        img.backward(go.double())
        assert abs_err(img, gold["image"]) < 1e-4
        for k in ("pos", "rgb", "opa", "quat", "scale"):
            assert rel_err(p[k].grad, gold["grad_" + k]) < 1e-3, k
    else:
        raise KeyError(name)
