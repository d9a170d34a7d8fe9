"""Parity at BASELINE.json's FULL sizes (SURVEY.md §8c P4@C2 and P6), where tiles hold up to
~2,000 instances, the staging pipeline runs 8-31 chunks per tile, whole tiles saturate and the
epoch-tagged tails of the gradient rows are skipped:

* `test_p4_at_c2`        - C2 (500 k Gaussians, 1080p): the reference build's own `draw` /
                           `draw_backward` (through its unmodified renderer.py) fed OUR sorted
                           per-instance order; image and all five parameter gradients vs the fused path
                           (the reference's outputs are stored in tests/golden/ref_p4_c2_*.npz).
* `test_masked_gradient_at_scale` - C3 (2.4 M, 1080p; RGB, SH-27, SH-48) and C5 (5 M, 4K): the upstream
                           gradient is non-zero only on K sampled tiles (the heaviest tile, the most
                           saturated one, a spread); ALL FIVE parameter gradients are compared with the
                           fp64 CPU oracle run on exactly the Gaussians of those tiles, every other
                           gradient must be exactly zero.
* `test_reference_renderer_bound_to_our_module` - the reference's renderer.py, UNCHANGED, imported
                           with `gaussian` = our extension (SURVEY.md §2 #5), incl. a strided grad_output
                           (its outputs are stored in tests/golden/ref_renderer_*.npz).
"""
import numpy as np
import pytest
import torch

import gs_oracle as O
import synthetic as S
from helpers import abs_err, assert_matches_golden_frame, rel_err, require_golden, scene

pytestmark = pytest.mark.gpu

IMG_ATOL = 1e-4
GRAD_RTOL = 1e-3
NAMES = ("pos", "rgb", "opa", "quat", "scale")


def _splatter(g, views, dev, **kw):
    import splatter
    vs = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran) for v in views]
    return splatter.Splatter.from_tensors(g, vs, device=dev, **kw)


# ------------------------------------------------------------------------------------------
def _tile_mask(cam, tiles, h, w):
    top, left = (cam.Hp - h) // 2, (cam.Wp - w) // 2
    mpad = torch.zeros(cam.Hp, cam.Wp, 1)
    for t in tiles:
        ty, tx = divmod(t, cam.ntx)
        mpad[ty * 16:(ty + 1) * 16, tx * 16:(tx + 1) * 16] = 1.0
    return mpad[top:top + h, left:left + w]


@pytest.mark.parametrize("regime,opa", [("safe", (0.005, 0.05)), ("standard", (0.05, 0.9))])
def test_p4_at_c2(gs, cuda, regime, opa):
    """SURVEY.md §8c "P4@C2": C2 (500 k Gaussians, 1080p; heaviest tile <= 500 instances, inside the limit
    below which the reference's draw_backward does not mix chunks - hazard 1).  The reference build's own
    kernels were fed OUR (tile, depth, id) order, so its fp32 sort-key ties (hazard 4) cannot enter; what
    they computed is tests/golden/ref_p4_c2_<regime>.npz (culling mask, image on a pixel sample, gradients
    on a sample of rows).
      safe     - opacities in [0.005, 0.05]: no pixel reaches T < 1e-4, the reference's backward is exact:
                 image <= 1e-4 and ALL gradients <= 1e-3 are gated against it;
      standard - the benchmark's opacities [0.05, 0.9]: pixels saturate, and the reference's partial-mask
                 shuffle reduction (hazard 3, gaussian.cu:675-772) is no longer exact.  The image is gated
                 against the reference; for the gradients the fp64 oracle arbitrates on sampled tiles: ours
                 must match it to 1e-3, and any disagreement with the reference must be the reference's."""
    gold = require_golden(f"ref_p4_c2_{regime}.npz")
    n, w, h = 500_000, 1920, 1080
    g, v, cam = scene(n, w, h, k=0, opa_range=opa)
    go = (S.make_grad_output(h, w, 0) * (h * w)).to(cuda)
    sp = _splatter(g, [v], cuda)
    img = sp(0)
    img.backward(go)
    st = sp.frame_stats()
    assert st["max_tile_count"] <= 500, st
    idx, accum = sp._rctx.sorted_instances()
    mask = torch.from_numpy(np.unpackbits(gold["mask"].numpy(), count=n).astype(bool))
    assert torch.equal(sp.culling_mask.cpu().bool(), mask)
    assert abs_err(img.detach().reshape(-1, 3).cpu()[gold["pix"].long()], gold["image"]) < IMG_ATOL
    r = gold["rows"].long()
    errs = {k: rel_err(getattr(sp.gaussian_3ds, k).grad.cpu()[r], gold["grad_" + k]) for k in NAMES}
    print(f"P4@C2[{regime}] ours vs reference build, sampled rows: {errs}")
    if regime == "safe":
        assert st["n_instances_eff"] == st["n_instances"]              # nothing saturated
        for k in NAMES:
            assert errs[k] < GRAD_RTOL, (k, errs)
        return
    # standard regime: arbitrate on the fixture's tiles with the fp64 oracle
    tiles = gold["tiles"].tolist()
    gom = S.make_grad_output(h, w, 0) * (h * w) * _tile_mask(cam, tiles, h, w)
    for p_ in sp.gaussian_3ds.parameters():
        p_.grad = None
    sp(0).backward(gom.to(cuda))
    _, U, og = _oracle_on_tiles(g, v, cam, idx.cpu(), accum.cpu().long(), tiles, gom, False)
    # the reference's gradients are stored for a sample of the Gaussians binned into those tiles
    u_ids = gold["u_ids"].long()
    loc = torch.searchsorted(U, u_ids).clamp(max=U.numel() - 1)
    assert torch.equal(U[loc], u_ids)
    for k in NAMES:
        e_ours = rel_err(getattr(sp.gaussian_3ds, k).grad.cpu()[U], og[k])
        e_ref = rel_err(gold["tiles_grad_" + k], og[k][loc])
        print(f"P4@C2[standard] {k}: ours vs oracle {e_ours:.2e}, reference vs oracle (sampled) {e_ref:.2e}, "
              f"ours vs reference (sampled rows) {errs[k]:.2e}")
        assert e_ours < GRAD_RTOL, (k, e_ours)
        assert errs[k] < GRAD_RTOL or e_ref > 10 * e_ours, (k, errs[k], e_ref, e_ours)


# ------------------------------------------------------------------------------------------
def _pick_tiles(accum, neff, ntx, nty, k_spread):
    """heaviest tile, tile with the longest consumed list, tile with the most skipped tail, a spread."""
    cnt = (accum[1:] - accum[:-1]).long()
    tiles = {int(cnt.argmax()), int(neff.argmax()), int((cnt - neff).argmax())}
    inner = [ty * ntx + tx for ty in (1, nty // 3, nty // 2, nty - 2) for tx in (0, ntx // 4, ntx // 2, ntx - 1)]
    for t in inner[:: max(1, len(inner) // k_spread)]:
        tiles.add(int(t))
    return sorted(tiles)


def _oracle_on_tiles(g, v, cam, idx, accum, tiles, go_final, use_sh):
    """fp64 oracle restricted to the Gaussians that the DEVICE binned into `tiles` (binning parity
    P2 and order P3 are checked elsewhere; fp64-vs-fp32 bbox flips at a tile border would otherwise
    make this test flaky at 2.4 M Gaussians).  Returns (padded fp64 image, U, grads on U)."""
    dt = torch.float64
    ids = [idx[int(accum[t]):int(accum[t + 1])].long() for t in tiles]
    U = torch.unique(torch.cat(ids))                                        # ascending Gaussian ids
    p = {k: g[k][U].to(dt).clone().requires_grad_(True) for k in NAMES}
    nq, ns, opa_a, rgb_a = O.preactivate(p["quat"], p["scale"], p["opa"], p["rgb"], "abs", use_sh)
    rp, rc, _ = O.global_culling(p["pos"], nq, ns, cam.rot.to(dt), cam.tran.to(dt), cam.near, cam.half_w, cam.half_h)
    loc = torch.cat([torch.searchsorted(U, i) for i in ids])
    T = cam.ntx * cam.nty
    counts = torch.zeros(T, dtype=torch.int64)
    for t, i in zip(tiles, ids):
        counts[t] = i.numel()
    acc2 = torch.zeros(T + 1, dtype=torch.int64)
    acc2[1:] = torch.cumsum(counts, 0)
    rays = O.ray_info(cam.rot.to(dt), cam.tran.to(dt), cam.Hp, cam.Wp, cam.fx, cam.fy) if use_sh else (None,) * 4
    padded = O.draw(rp[loc], rgb_a[loc], opa_a[loc], rc[loc], acc2.to(torch.int32), cam.Hp, cam.Wp, cam.fx, cam.fy,
                    use_sh, *rays, tiles=torch.tensor(tiles))
    out = cam.crop(torch.clamp(padded, 0, 1))
    out.backward(go_final.to(dt))
    return padded.detach(), U, {k: p[k].grad for k in NAMES}


@pytest.mark.parametrize("label,n,w,h,sh_dim", [
    ("C3-rgb", 2_400_000, 1920, 1080, 3),
    ("C3-sh27", 2_400_000, 1920, 1080, 27),
    ("C3-sh48", 2_400_000, 1920, 1080, 48),
    ("C5-4k", 5_000_000, 3840, 2160, 3),
])
def test_masked_gradient_at_scale(gs, cuda, label, n, w, h, sh_dim):
    use_sh = sh_dim != 3
    g, v, cam = scene(n, w, h, k=0, sh_dim=sh_dim)
    sp = _splatter(g, [v], cuda, use_sh_coeff=use_sh)
    with torch.no_grad():
        sp(0)
    st = sp.frame_stats()
    idx, accum = sp._rctx.sorted_instances()
    idx, accum = idx.cpu(), accum.cpu().long()
    neff = sp._rctx.tile_consumed().cpu().long()
    tiles = _pick_tiles(accum, neff, cam.ntx, cam.nty, 5)
    cnt = accum[1:] - accum[:-1]
    assert int(cnt.max()) == st["max_tile_count"] and int(cnt[tiles].max()) == st["max_tile_count"]
    if w == 1920:
        assert st["max_tile_count"] > 1000            # multi-chunk tiles really are exercised

    # upstream gradient: O(1) values on the sampled tiles only (crop coordinates)
    top, left = (cam.Hp - h) // 2, (cam.Wp - w) // 2
    go = S.make_grad_output(h, w, 0) * (h * w) * _tile_mask(cam, tiles, h, w)

    img = sp(0)
    img.backward(go.to(cuda))
    opad, U, ograds = _oracle_on_tiles(g, v, cam, idx, accum, tiles, go, use_sh)

    # forward on the sampled tiles
    raw = torch.zeros(cam.Hp, cam.Wp, 3, dtype=torch.float64)
    raw[top:top + h, left:left + w] = img.detach().cpu().double()
    for t in tiles:
        ty, tx = divmod(t, cam.ntx)
        r0, r1 = max(ty * 16, top), min((ty + 1) * 16, top + h)
        a = raw[r0:r1, tx * 16:(tx + 1) * 16]
        b = opad[r0:r1, tx * 16:(tx + 1) * 16].clamp(0, 1)
        assert abs_err(a, b) < IMG_ATOL, (label, t)
    # all five gradients on the Gaussians of those tiles; exactly zero everywhere else
    other = torch.ones(n, dtype=torch.bool)
    other[U] = False
    for name in NAMES:
        got = getattr(sp.gaussian_3ds, name).grad.cpu()
        assert bool(torch.isfinite(got).all()), name
        assert rel_err(got[U], ograds[name]) < GRAD_RTOL, (label, name)
        assert float(got[other].abs().max()) == 0.0, (label, name)


# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_sh", [False, True])
def test_reference_renderer_bound_to_our_module(gs, cuda, use_sh):
    """SURVEY.md §2 #5 / §8b: the reference's renderer.py, UNCHANGED, driven by the reference's splatter.py
    call sequence (oracle/ref_pipeline.LegacyFrame) with `gaussian` bound to our module and a strided
    (non-contiguous) upstream gradient; what it computed is tests/golden/ref_renderer_{rgb,sh}.npz.
    The fused path must agree with it."""
    import golden_cases as GC
    n, w, h = 2000, 192, 128
    # a scene inside the reference pipeline's own limits (capacity n//20, no fp32 sort-key ties); the
    # SH variant has the same geometry (the generator draws colours last)
    g, v, cam, go = GC.frame_case(n, w, h, (0.05, 0.6), (0.4, 1.5), 6)
    assert GC.reference_key_collisions(g, cam)[0] == 0
    if use_sh:
        g, v, cam = scene(n, w, h, seed=6, sh_dim=27, opa_range=(0.05, 0.6), sigma_px=(0.4, 1.5))
    sp = _splatter(g, [v], cuda, use_sh_coeff=use_sh)
    img = sp(0)
    img.backward(go.to(cuda))
    gold = require_golden(f"ref_renderer_{'sh' if use_sh else 'rgb'}.npz")
    assert_matches_golden_frame(sp, img, gold, IMG_ATOL, GRAD_RTOL)
