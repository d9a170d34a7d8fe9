"""CPU checks of the maps oracle (tests/maps_oracle.py: depth / alpha maps and a background colour) against
closed forms, and of the argument validation of the two maps entry points of the C ABI.  No GPU needed."""
import ctypes
import math
import os

import torch

import gs_oracle as O
import maps_oracle as MO
from helpers import scene, sorted_instances_cpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "3d-gaussian-splatting_b200")


def _params(g, dtype=torch.float64, grad=False):
    return {k: v.to(dtype).clone().requires_grad_(grad) for k, v in g.items()}


def test_black_background_image_is_the_plain_oracle_image():
    g, v, cam = scene(400, 96, 64, k=1, opa_range=(0.3, 0.95))
    p = _params(g)
    img0, aux0 = O.render(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, return_aux=True)
    img, depth, alpha, aux = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, return_aux=True)
    assert torch.equal(img, img0) and torch.equal(aux["padded"], aux0["padded"])
    assert depth.shape == (64, 96) and alpha.shape == (64, 96)
    assert float(alpha.min()) >= 0 and float(alpha.max()) <= 1 and float(alpha.max()) > 0.5


def _one_gaussian_scene(n):
    v_w, v_h = 64, 48
    g, v, cam = scene(n, v_w, v_h, k=0, opa_range=(0.4, 0.6), sigma_px=(3.0, 4.0))
    g["pos"][0] = torch.tensor([0.02, -0.01, 0.3])
    if n > 1:
        g["pos"][1] = torch.tensor([-0.03, 0.02, 0.1])       # overlaps #0 at another depth
    return g, v, cam


def _alpha_closed_form(p, cam, i):
    """opa * exp(power) of Gaussian i at every padded pixel centre, from the projected conic."""
    nq, ns, opa_a, _ = O.preactivate(p["quat"], p["scale"], p["opa"], p["rgb"])
    rp, rc, _ = O.global_culling(p["pos"], nq, ns, cam.rot.double(), cam.tran.double(), cam.near, cam.half_w,
                                 cam.half_h)
    a, b, c, d = rc[i].reshape(4)
    px = (torch.arange(cam.Wp, dtype=torch.float64) + 0.5 - cam.Wp // 2) / cam.fx
    py = (torch.arange(cam.Hp, dtype=torch.float64) + 0.5 - cam.Hp // 2) / cam.fy
    X = px.reshape(1, -1) - rp[i, 0]
    Y = py.reshape(-1, 1) - rp[i, 1]
    power = -(d * X * X - (b + c) * X * Y + a * Y * Y) / (2 * (a * d - b * c) + 1e-14)
    return (opa_a[i] * torch.exp(power)).detach(), float(rp[i, 2])


def test_one_gaussian_alpha_and_depth_closed_form():
    g, v, cam = _one_gaussian_scene(1)
    p = _params(g)
    _, _, _, aux = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, return_aux=True)
    want_a, depth = _alpha_closed_form(p, cam, 0)
    pc = (p["pos"][0] @ cam.rot.double().T + cam.tran.double()).norm()
    assert math.isclose(depth, float(pc), rel_tol=1e-12)
    acc = aux["accum"]
    cover = torch.zeros(cam.nty * cam.ntx, dtype=torch.bool)
    cover[(acc[1:] - acc[:-1]) > 0] = True
    cover = cover.reshape(cam.nty, cam.ntx).repeat_interleave(16, 0).repeat_interleave(16, 1)
    got_a, got_d = aux["padded_alpha"].detach(), aux["padded_depth"].detach()
    assert float(cover.float().mean()) > 0.05
    assert torch.allclose(got_a[cover], want_a[cover], rtol=0, atol=1e-12)
    assert torch.allclose(got_d[cover], (want_a * depth)[cover], rtol=0, atol=1e-11)
    assert float(got_a[~cover].abs().max()) == 0.0


def test_two_gaussians_alpha_composes():
    g, v, cam = _one_gaussian_scene(2)
    g["scale"][1] = g["scale"][0]                              # same footprint: one tile rectangle
    g["quat"][1] = g["quat"][0]
    p = _params(g)
    _, _, _, aux = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, return_aux=True)
    a1, d1 = _alpha_closed_form(p, cam, 0)
    a2, d2 = _alpha_closed_form(p, cam, 1)
    acc = aux["accum"]
    both = ((acc[1:] - acc[:-1]) == 2).reshape(cam.nty, cam.ntx).repeat_interleave(16, 0).repeat_interleave(16, 1)
    assert float(both.float().mean()) > 0.05
    got = aux["padded_alpha"].detach()
    assert torch.allclose(got[both], (1 - (1 - a1) * (1 - a2))[both], rtol=0, atol=1e-12)
    # depth: the nearer one first (the (tile, depth) order), the farther one behind it
    (an, dn), (af, df) = ((a1, d1), (a2, d2)) if d1 < d2 else ((a2, d2), (a1, d1))
    want_d = an * dn + (1 - an) * af * df
    assert torch.allclose(aux["padded_depth"].detach()[both], want_d[both], rtol=0, atol=1e-11)


def test_background_fills_the_remaining_transmittance():
    g, v, cam = scene(600, 96, 64, k=0, opa_range=(0.05, 0.9))
    p = _params(g)
    bg = (0.2, 0.5, 1.0)
    _, _, _, aux0 = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, return_aux=True)
    img, depth, alpha, aux = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, background=bg,
                                            return_aux=True)
    want = aux0["padded"] + (1 - aux0["padded_alpha"]).unsqueeze(-1) * torch.tensor(bg, dtype=torch.float64)
    assert torch.allclose(aux["padded"], want, rtol=0, atol=1e-14)
    assert torch.equal(aux["padded_depth"], aux0["padded_depth"]) and torch.equal(aux["padded_alpha"], aux0["padded_alpha"])
    assert torch.equal(img, cam.crop(aux["padded"].clamp(0, 1)))
    assert torch.equal(alpha, MO.crop2(cam, aux["padded_alpha"]))
    # an empty tile shows the background
    empty = ((aux["accum"][1:] - aux["accum"][:-1]) == 0).nonzero()
    if len(empty):
        ty, tx = divmod(int(empty[0]), cam.ntx)
        assert torch.equal(aux["padded"][ty * 16, tx * 16], torch.tensor(bg, dtype=torch.float64))


def test_direct_depth_term_of_the_position_gradient():
    """d/d pos with d_i live minus with d_i detached == sum_pixels gD w_i * R^T p_c / |p_c| per Gaussian."""
    g, v, cam = scene(300, 80, 64, k=2, opa_range=(0.1, 0.8))
    gD = torch.rand(64, 80, generator=torch.Generator().manual_seed(5), dtype=torch.float64) * 2 - 1
    grads = []
    for detach in (False, True):
        p = _params(g, grad=True)
        _, depth, _ = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], cam, detach_depth=detach)
        (depth * gD).sum().backward()
        grads.append(p["pos"].grad)
    direct = grads[0] - grads[1]
    # sum_pixels gD w_i per instance: gradient of <gD, depth map> wrt a leaf per-instance depth
    s = sorted_instances_cpu(g, cam, dtype=torch.float64)
    dleaf = s["pos"][:, 2].clone().requires_grad_(True)
    _, dmap, _ = MO.draw_maps(s["pos"], s["rgb"], s["opa"], s["cov"], dleaf, s["accum"], cam.Hp, cam.Wp, cam.fx, cam.fy)
    (MO.crop2(cam, dmap) * gD).sum().backward()
    per_g = torch.zeros(g["pos"].shape[0], dtype=torch.float64).index_add_(0, s["gauss_idx"], dleaf.grad)
    pc = g["pos"].double() @ cam.rot.double().T + cam.tran.double()
    want = per_g.unsqueeze(-1) * ((pc / pc.norm(dim=-1, keepdim=True)) @ cam.rot.double())
    assert float(per_g.abs().max()) > 0
    assert torch.allclose(direct, want, rtol=1e-9, atol=1e-12)


def test_maps_entry_points_validate_without_a_gpu():
    lib = ctypes.CDLL(os.path.join(PKG, "libgs_b200.so"))
    lib.gs_last_error.restype = ctypes.c_char_p
    P, I = ctypes.c_void_p, ctypes.c_int
    lib.gs_render_forward_maps.argtypes = [P] * 6 + [I] * 3 + [P] * 9
    assert lib.gs_render_forward_maps(*([None] * 6), 0, 3, 0, *([None] * 9)) == -1
    assert b"null ctx" in lib.gs_last_error()
    lib.gs_render_backward_maps.argtypes = [P] * 12 + [I] + [P] * 6
    assert lib.gs_render_backward_maps(*([None] * 12), 0, *([None] * 6)) == -1
    assert b"null ctx" in lib.gs_last_error()


def test_tune_knobs_read_back_without_a_gpu():
    """gs_tune_get returns what gs_tune set (so a caller can restore a knob it changed)."""
    lib = ctypes.CDLL(os.path.join(PKG, "libgs_b200.so"))
    lib.gs_last_error.restype = ctypes.c_char_p
    lib.gs_tune.argtypes = [ctypes.c_char_p, ctypes.c_int]
    lib.gs_tune_get.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int)]
    v = ctypes.c_int(-7)
    assert lib.gs_tune_get(b"gather", ctypes.byref(v)) == 0
    before = v.value
    assert lib.gs_tune(b"gather", 0) == 0
    assert lib.gs_tune_get(b"gather", ctypes.byref(v)) == 0 and v.value == 0
    assert lib.gs_tune(b"gather", before) == 0
    assert lib.gs_tune_get(b"gather", ctypes.byref(v)) == 0 and v.value == before
    assert lib.gs_tune_get(b"no_such_knob", ctypes.byref(v)) == -1 and b"unknown knob" in lib.gs_last_error()
    assert lib.gs_tune_get(b"gather", None) == -1
