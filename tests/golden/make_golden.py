"""Generates tests/golden/*.npz by running the REFERENCE's own CUDA build (oracle/_ref,
built by oracle/build_ref.py from the unmodified sources) on a GPU.  The ref_*.npz fixtures
hold what the GPU parity tests compare our kernels against; two of them (ref_p4_c2_*, the
reference's kernels fed our sorted instance order, and ref_renderer_*, the reference's
renderer.py driving our `gaussian` module) also run our extension to produce their inputs.

Run on the B200 box:   python tests/golden/make_golden.py gpurun_out/golden
then copy the files into tests/golden/ and commit them.  Nothing of ours (kernels or
oracle arithmetic) produces the stored outputs; the oracle only prepares the sorted
per-instance INPUTS of the `draw` case, which are stored alongside.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in ("3d-gaussian-splatting_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))

import golden_cases as GC  # noqa: E402
import gs_oracle as O  # noqa: E402
import ref_pipeline  # noqa: E402


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda", 0)
    gref, rref = ref_pipeline.load_reference()
    assert gref is not None, "oracle/_ref is missing: run oracle/build_ref.py where /root/reference exists"
    cpu = lambda t: t.detach().cpu().numpy()

    # ---- project.npz : global_culling forward + backward -------------------------------
    pos, nq, ns, cam, go_pos, go_cov = GC.project_inputs()
    p = pos.to(dev).requires_grad_(True)
    q = nq.to(dev).requires_grad_(True)
    s = ns.to(dev).requires_grad_(True)
    rp, rc, m = rref.global_culling(p, q, s, cam.rot.to(dev), cam.tran.to(dev), cam.near, cam.half_w, cam.half_h)
    ((rp * go_pos.to(dev)).sum() + (rc * go_cov.to(dev)).sum()).backward()
    np.savez_compressed(os.path.join(out_dir, "project.npz"), res_pos=cpu(rp), res_cov=cpu(rc), mask=cpu(m),
                        grad_pos=cpu(p.grad), grad_quat=cpu(q.grad), grad_scale=cpu(s.grad))

    # ---- tiles.npz : calc_tile_list method 2 --------------------------------------------
    pos2, cov2, cam = GC.tiles_inputs()
    T = cam.ntx * cam.nty
    n = pos2.shape[0]
    cnt = torch.zeros(T, dtype=torch.int32, device=dev)
    lst = torch.full((T, n), -1, dtype=torch.int32, device=dev)
    cobj = gref.Gaussian3ds()
    cobj.pos, cobj.cov = pos2.to(dev), cov2.to(dev)
    cobj.rgb, cobj.opa = torch.zeros(n, 3, device=dev), torch.zeros(n, device=dev)
    tiles = gref.Tiles()
    tiles.top = tiles.bottom = tiles.left = tiles.right = torch.zeros(T, device=dev)
    gref.calc_tile_list(cobj, tiles, cnt, lst, 0.05, 2, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                        cam.topmost)
    cnt_c, lst_c = cnt.cpu(), lst.cpu()
    flat = [sorted(lst_c[t, :int(cnt_c[t])].tolist()) for t in range(T)]
    np.savez_compressed(os.path.join(out_dir, "tiles.npz"), counts=cnt_c.numpy(),
                        flat_ids=np.array([i for f in flat for i in f], dtype=np.int32))

    # ---- draw_rgb.npz : draw + draw_backward on sorted per-instance inputs ----------------
    inst, cam, grad_img = GC.draw_inputs()
    t = {k: inst[k].to(dev).float().contiguous().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
    dummy = torch.zeros(3, device=dev)
    img = rref.draw(t["pos"], t["rgb"], t["opa"], t["cov"], inst["accum"].to(dev), cam.Hp, cam.Wp, cam.fx, cam.fy,
                    False, False, False, True, dummy, dummy, dummy, dummy)
    img.backward(grad_img.to(dev))
    counts = inst["accum"][1:] - inst["accum"][:-1]
    assert int(counts.max()) <= 500, "outside the reference backward's safe regime"
    np.savez_compressed(os.path.join(out_dir, "draw_rgb.npz"), image=cpu(img),
                        in_pos=cpu(inst["pos"]), in_rgb=cpu(inst["rgb"]), in_opa=cpu(inst["opa"]),
                        in_cov=cpu(inst["cov"]), in_accum=cpu(inst["accum"]),
                        grad_pos=cpu(t["pos"].grad), grad_rgb=cpu(t["rgb"].grad), grad_opa=cpu(t["opa"].grad),
                        grad_cov=cpu(t["cov"].grad))

    # ---- draw_sh.npz : draw + draw_backward with per-pixel SH-27 colour ---------------------------
    inst, cam, grad_img, rays = GC.draw_sh_inputs()
    counts = inst["accum"][1:] - inst["accum"][:-1]
    assert int(counts.max()) <= 160, "outside the reference SH backward's safe regime"
    t = {k: inst[k].to(dev).float().contiguous().requires_grad_(True) for k in ("pos", "rgb", "opa", "cov")}
    r = [x.to(dev).float().contiguous() for x in rays]
    img = rref.draw(t["pos"], t["rgb"], t["opa"], t["cov"], inst["accum"].to(dev), cam.Hp, cam.Wp, cam.fx, cam.fy,
                    False, False, True, True, r[0], r[1], r[2], r[3])
    img.backward(grad_img.to(dev))
    np.savez_compressed(os.path.join(out_dir, "draw_sh.npz"), image=cpu(img),
                        in_pos=cpu(inst["pos"]), in_rgb=cpu(inst["rgb"]), in_opa=cpu(inst["opa"]),
                        in_cov=cpu(inst["cov"]), in_accum=cpu(inst["accum"]),
                        grad_pos=cpu(t["pos"].grad), grad_rgb=cpu(t["rgb"].grad), grad_opa=cpu(t["opa"].grad),
                        grad_cov=cpu(t["cov"].grad))

    # ---- frame_c1.npz : the reference's whole per-frame pipeline ---------------------------
    g, v, cam, go = GC.frame_inputs()
    c = GC.CASES["frame_c1.npz"]
    bad, mx, maxp = GC.reference_key_collisions(g, cam)
    assert bad == 0 and mx <= maxp, (bad, mx, maxp)
    frame = ref_pipeline.LegacyFrame(gref, rref, c["w"], c["h"], v.fx, v.fy, v.rot.to(dev), v.tran.to(dev))
    pr = {k: x.to(dev).clone().requires_grad_(True) for k, x in g.items()}
    img = frame(pr["pos"], pr["rgb"], pr["opa"], pr["quat"], pr["scale"])
    img.backward(go.to(dev))
    # inside the reference's own limits: dense-list capacity MAXP = Nc//20 (splatter.py:569) and the
    # backward's 500-instance chunk (SURVEY.md hazards 1, 4)
    assert frame.aux["max_tile"] <= min(500, frame.aux["MAXP"]), frame.aux["max_tile"]
    np.savez_compressed(os.path.join(out_dir, "frame_c1.npz"), n=c["n"], w=c["w"], h=c["h"], image=cpu(img),
                        **{"grad_" + k: cpu(pr[k].grad) for k in pr})
    reference_parity(out_dir, gref, rref, dev)
    print("golden fixtures written to", out_dir, sorted(os.listdir(out_dir)))


# ---- ref_*.npz : what the GPU parity tests compare our kernels against ------------------------
# Each fixture holds the reference's outputs for the inputs the test builds (the same helpers build
# them here), reduced to a seeded sample of rows / pixels (GC.sample) where the full output is large.
K_ROWS, K_PIX = 256, 512
NAMES = ("pos", "rgb", "opa", "quat", "scale")


def _sampled_image(img, k=K_PIX):
    flat = img.detach().reshape(-1, 3).cpu()
    pix = GC.sample(torch.arange(flat.shape[0]), k, seed=1)
    return dict(pix=pix.int().numpy(), image=flat[pix].numpy())


def _sampled_grads(grads, names, k=K_ROWS):
    """Rows where some gradient is non-zero (culled / untouched Gaussians carry exact zeros)."""
    grads = {n: grads[n].detach().cpu() for n in names}
    live = sum(g.reshape(g.shape[0], -1).abs().sum(1) for g in grads.values()) > 0
    rows = GC.sample(torch.nonzero(live).squeeze(-1), k, seed=2)
    return dict(rows=rows.int().numpy(), **{"grad_" + n: grads[n][rows].numpy() for n in names})


def _reference_renderer_on(gmod):
    """The reference's renderer.py (the copy oracle/build_ref.py makes), imported with `gaussian` bound to `gmod`."""
    import importlib.util
    saved = sys.modules.get("gaussian")
    sys.modules["gaussian"] = gmod
    try:
        spec = importlib.util.spec_from_file_location("renderer_ref_on_ours", os.path.join(ref_pipeline.REF_DIR, "renderer.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        if saved is None:
            del sys.modules["gaussian"]
        else:
            sys.modules["gaussian"] = saved
    return mod


def _reference_chain(rref, g, v, cam, gi, accum, go, dev):
    """The reference's own operators (its CUDA build through its unmodified renderer.py) on OUR sorted
    instance order: pre-activations (splatter.py:519-524,539-540) -> global_culling -> gather (a8) ->
    draw -> clamp + crop (splatter.py:652-653) -> backward of all of it."""
    p = {k: t.to(dev).clone().requires_grad_(True) for k, t in g.items()}
    nq = p["quat"] / p["quat"].norm(dim=1, keepdim=True)
    ns = p["scale"].abs() + 1e-4
    _pos, _cov, mask = rref.global_culling(p["pos"], nq, ns, v.rot.to(dev), v.tran.to(dev), cam.near,
                                           cam.half_w, cam.half_h)
    t_pos, t_cov = _pos[gi], _cov[gi]
    t_rgb, t_opa = p["rgb"].sigmoid()[gi], p["opa"].sigmoid()[gi]
    dummy = torch.zeros(3, device=dev)
    rimg_p = rref.draw(t_pos, t_rgb, t_opa, t_cov, accum, cam.Hp, cam.Wp, cam.fx, cam.fy, False, False, False, True,
                       dummy, dummy, dummy, dummy)
    rimg = cam.crop(torch.clamp(rimg_p, 0, 1))
    rimg.backward(go)
    return rimg.detach(), {k: p[k].grad for k in NAMES}, mask


def reference_parity(out_dir, gref, rref, dev):
    import gaussian
    import synthetic as S
    import test_frame_gpu as TF
    import test_scale_parity_gpu as TP
    import test_stages_gpu as TS
    from helpers import scene
    save = lambda name, **kw: np.savez_compressed(os.path.join(out_dir, name), **kw)

    # global_culling forward + backward (test_global_culling_vs_reference_build)
    g, cam, nq, ns = TS._proj_inputs(20000, 640, 360, 1, dev)
    pos, q, s = (t.to(dev).requires_grad_(True) for t in (g["pos"], nq, ns))
    op, oc, om = rref.global_culling(pos, q, s, cam.rot.to(dev), cam.tran.to(dev), cam.near, cam.half_w, cam.half_h)
    gen = torch.Generator().manual_seed(3)
    gp = torch.randn(op.shape, generator=gen).to(dev)
    gc = torch.randn(oc.shape, generator=gen).to(dev)
    ((op * gp).sum() + (oc * gc).sum()).backward()
    rows = GC.sample(torch.nonzero(om.cpu()).squeeze(-1), K_ROWS, seed=2)
    save("ref_culling.npz", mask=om.cpu().bool().numpy(), rows=rows.int().numpy(),
         **{k: t.detach().cpu()[rows].numpy() for k, t in
            dict(res_pos=op, res_cov=oc, grad_pos=pos.grad, grad_quat=q.grad, grad_scale=s.grad).items()})

    # calc_tile_list method 2 (test_tile_binning_vs_reference_build)
    g, v, cam = scene(30000, 640, 368, k=0)
    nq, ns, _, _ = O.preactivate(g["quat"], g["scale"], g["opa"], g["rgb"])
    rp, rc, m = O.global_culling(g["pos"], nq, ns, cam.rot, cam.tran, cam.near, cam.half_w, cam.half_h)
    idx = torch.nonzero(m.bool()).squeeze(-1)
    save("ref_tiles.npz", **GC.tile_set_digest(TS._per_tile_sets(*TS._tile_lists(gref, rp[idx].contiguous(),
                                                                                 rc[idx].contiguous(), cam, dev))))

    # calc_tile_list methods 0 and 1 (test_tile_methods_dist_and_prob_vs_reference_build)
    pos, cov, cam = TS._small_projected_scene()
    out = {}
    for method, thresh in ((0, (cam.tile_lx / 0.5) ** 2), (1, 0.05)):
        for k, a in GC.tile_set_digest(TS._legacy_lists(gref, method, pos, cov, cam, thresh, dev)).items():
            out[f"m{method}_{k}"] = a
    save("ref_tile_methods.npz", **out)

    # draw + draw_backward, RGB and SH-27 (test_draw_vs_reference_build_safe_regime, test_draw_sh_vs_reference_build)
    cam, inst, gi = TS._draw_case(4000, 256, 256, (0.005, 0.05))
    assert int((inst["accum"][1:] - inst["accum"][:-1]).max()) <= 500
    img, grads = TS._run_draw(rref, inst, cam, gi, dev)
    grads["pos"] = grads["pos"][:, :2]
    save("ref_draw.npz", **_sampled_image(img), **_sampled_grads(grads, ("pos", "rgb", "opa", "cov")))
    cam, inst, gi, rays = TS._sh_case(2500, 256, 192, 27, (0.005, 0.05))
    assert int((inst["accum"][1:] - inst["accum"][:-1]).max()) <= 160
    img, grads = TS._run_draw_sh(rref, inst, cam, gi, rays, dev)
    grads["pos"] = grads["pos"][:, :2]
    save("ref_draw_sh.npz", **_sampled_image(img), **_sampled_grads(grads, ("pos", "rgb", "opa", "cov")))

    # the reference's whole per-frame pipeline (test_fused_frame_vs_reference_pipeline)
    n, w, h = 2000, 192, 128
    g, v, cam, go = GC.frame_case(n, w, h, (0.005, 0.05), (0.4, 1.5), 2)
    assert GC.reference_key_collisions(g, cam)[0] == 0
    frame = ref_pipeline.LegacyFrame(gref, rref, w, h, v.fx, v.fy, v.rot.to(dev), v.tran.to(dev))
    p = {k: t.to(dev).clone().requires_grad_(True) for k, t in g.items()}
    img = frame(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"])
    img.backward(go.to(dev))
    assert frame.aux["max_tile"] <= min(500, frame.aux["MAXP"])
    save("ref_frame.npz", **_sampled_image(img), **_sampled_grads({k: p[k].grad for k in NAMES}, NAMES))

    # the reference's renderer.py on OUR `gaussian` module (test_reference_renderer_bound_to_our_module)
    rmod = _reference_renderer_on(gaussian)
    for use_sh in (False, True):
        g, v, cam, go = GC.frame_case(n, w, h, (0.05, 0.6), (0.4, 1.5), 6)
        assert GC.reference_key_collisions(g, cam)[0] == 0
        if use_sh:
            g, v, cam = scene(n, w, h, seed=6, sh_dim=27, opa_range=(0.05, 0.6), sigma_px=(0.4, 1.5))
        wide = torch.zeros(h, w, 6, device=dev)
        wide[..., ::2] = go.to(dev)
        frame = ref_pipeline.LegacyFrame(gaussian, rmod, w, h, v.fx, v.fy, v.rot.to(dev), v.tran.to(dev),
                                         use_sh_coeff=use_sh)
        p = {k: t.to(dev).clone().requires_grad_(True) for k, t in g.items()}
        img = frame(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"])
        assert frame.aux["max_tile"] <= frame.aux["MAXP"]
        img.backward(wide[..., ::2])
        save(f"ref_renderer_{'sh' if use_sh else 'rgb'}.npz", **_sampled_image(img),
             **_sampled_grads({k: p[k].grad for k in NAMES}, NAMES))

    # C2 at full size, the reference's kernels fed our sorted order (test_p4_at_c2)
    n, w, h = 500_000, 1920, 1080
    for regime, opa in (("safe", (0.005, 0.05)), ("standard", (0.05, 0.9))):
        g, v, cam = scene(n, w, h, k=0, opa_range=opa)
        go = (S.make_grad_output(h, w, 0) * (h * w)).to(dev)
        sp = TF._splatter(g, [v], dev)
        img = sp(0)
        img.backward(go)
        assert sp.frame_stats()["max_tile_count"] <= 500
        idx, accum = sp._rctx.sorted_instances()
        rimg, rgrads, mask = _reference_chain(rref, g, v, cam, idx.long(), accum, go, dev)
        print(f"P4@C2[{regime}] ours vs reference, full frame:",
              {k: float((getattr(sp.gaussian_3ds, k).grad - rgrads[k]).abs().max() / rgrads[k].abs().max()) for k in NAMES})
        out = dict(mask=np.packbits(mask.cpu().bool().numpy()), **_sampled_image(rimg), **_sampled_grads(rgrads, NAMES))
        if regime == "standard":
            # the reference's gradients for an upstream gradient restricted to sampled tiles, on a sample
            # of the Gaussians binned into those tiles
            neff = sp._rctx.tile_consumed().cpu().long()
            acc = accum.cpu().long()
            tiles = TP._pick_tiles(acc, neff, cam.ntx, cam.nty, 5)
            gom = S.make_grad_output(h, w, 0) * (h * w) * TP._tile_mask(cam, tiles, h, w)
            _, rg, _ = _reference_chain(rref, g, v, cam, idx.long(), accum, gom.to(dev), dev)
            U = torch.unique(torch.cat([idx.cpu()[int(acc[t]):int(acc[t + 1])].long() for t in tiles]))
            u_ids = GC.sample(U, K_ROWS, seed=3)
            out.update(tiles=np.array(tiles, dtype=np.int32), u_ids=u_ids.int().numpy(),
                       **{"tiles_grad_" + k: rg[k].cpu()[u_ids].numpy() for k in NAMES})
        save(f"ref_p4_c2_{regime}.npz", **out)
        del sp, rgrads
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden"))
