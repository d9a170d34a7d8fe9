"""CPU checks of the camera pose gradient (gs_ctx_set_camera_grad, `RenderContext.set_camera_grad`, pose tensors
that require grad in the frame Functions).  The reference gradient is autograd of the fp64 oracle with respect to
the camera's `rot` / `tran`: `gs_oracle.global_culling` builds p_c = pos @ rot.T + tran and JW = J @ rot with only J
detached, the convention of the kernels.  Here the oracle itself is checked against identities and the closed form
the projection backward implements, and the new C entry point's argument validation is checked without a device."""
import ctypes
import os

import torch

import gs_oracle as O
import maps_oracle as MO
import synthetic as S
from helpers import scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "3d-gaussian-splatting_b200")


def _pose_leaves(cam):
    rot = cam.rot.double().clone().requires_grad_(True)
    tran = cam.tran.double().clone().requires_grad_(True)
    return rot, tran, O.Camera(cam.width, cam.height, cam.fx, cam.fy, rot, tran, cam.near)


def _params(g):
    return {k: v.double().clone().requires_grad_(True) for k, v in g.items()}


def _grads_plain(g, cam, seed=0):
    rot, tran, c2 = _pose_leaves(cam)
    p = _params(g)
    out = O.render(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], c2)
    gi = S.make_grad_output(cam.height, cam.width, seed).double() * (cam.height * cam.width)
    (out * gi).sum().backward()
    return rot, tran, p


def _grads_maps(g, cam, seed=0):
    rot, tran, c2 = _pose_leaves(cam)
    p = _params(g)
    outs = MO.render_maps(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], c2, background=(0.2, 0.5, 1.0))
    gen = torch.Generator().manual_seed(seed + 5)
    loss = sum((o * (torch.rand(o.shape, generator=gen, dtype=torch.float64) * 2 - 1)).sum() for o in outs)
    loss.backward()
    return rot, tran, p


def _check_translation_identity(rot, tran, p):
    """p_c = R p + t with J detached for both: dL/dt = sum_i dL/dp_c,i = R sum_i dL/dpos_i (R orthonormal)."""
    expect = rot.detach() @ p["pos"].grad.sum(0)
    scale = float((p["pos"].grad @ rot.detach().T).abs().sum())
    assert scale > 0
    assert float((tran.grad - expect).abs().max()) <= 1e-10 * scale, (tran.grad, expect)


def test_oracle_translation_gradient_is_rotated_position_sum_plain():
    for k in (0, 2):
        g, _, cam = scene(400, 64, 48, k=k, seed=3)
        _check_translation_identity(*_grads_plain(g, cam))


def test_oracle_translation_gradient_is_rotated_position_sum_maps():
    for k in (0, 2):
        g, _, cam = scene(400, 64, 48, k=k, seed=4)
        _check_translation_identity(*_grads_maps(g, cam))


def test_oracle_single_gaussian_closed_form():
    """One Gaussian: dL/dt = gc = dL/dp_c from the projected (x/z, y/z) gradient, and dL/dR = gc p^T (mean term)
    plus the covariance term sum_c h_r[c] RS[k][c] chained through the image-plane rows of J - the formula of
    gs_project_backward, evaluated here in fp64 from the oracle's own dL/d(x/z, y/z) and dL/dcov2."""
    w, h = 64, 48
    v = S.make_view(w, h, 1)
    cam = O.Camera(w, h, v.fx, v.fy, v.rot, v.tran, v.near)
    g = S.make_gaussians(1, w, h, seed=2, opa_range=(0.5, 0.6), sigma_px=(3.0, 4.0))
    g["pos"] = torch.tensor([[0.15, -0.1, 0.2]])
    rot, tran, c2 = _pose_leaves(cam)
    p = _params(g)
    out, aux = O.render(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"], c2, return_aux=True)
    assert int(aux["mask"].sum()) == 1
    aux["res_pos"].retain_grad()
    aux["res_cov"].retain_grad()
    gi = S.make_grad_output(h, w, 0).double() * (h * w)
    (out * gi).sum().backward()
    gxy = aux["res_pos"].grad[0]
    G2 = aux["res_cov"].grad[0]
    assert float(gxy[2].abs()) == 0.0                          # plain frame: the depth is a sort key only
    with torch.no_grad():
        R = rot.detach()
        pw = p["pos"][0].detach()
        pc = R @ pw + tran.detach()
        x, y, z = pc.tolist()
        gc = torch.tensor([gxy[0] / z, gxy[1] / z, -(gxy[0] * x + gxy[1] * y) / (z * z)], dtype=torch.float64)
        assert torch.allclose(tran.grad, gc, rtol=1e-10, atol=1e-14)
        nq, ns, _, _ = O.preactivate(p["quat"].detach(), p["scale"].detach(), p["opa"].detach(), p["rgb"].detach())
        RS = O.quat_to_rot(nq)[0] * ns[0].unsqueeze(0)          # RS[k][c] = Rg[k][c] s[c]
        iz, jx, jy = 1 / z, -x / (z * z), -y / (z * z)
        J2 = torch.tensor([[iz, 0, jx], [0, iz, jy]], dtype=torch.float64)
        M = J2 @ R @ RS                                         # rows m0, m1
        H = (G2 + G2.T) @ M                                     # rows h0, h1
        gJW = H @ RS.T                                          # gJW[r][k] = sum_c h_r[c] RS[k][c]
        cov_term = J2.T @ gJW                                   # rows 0 / 1 / 2 of R: iz gJW0, iz gJW1, jx gJW0 + jy gJW1
        expect = torch.outer(gc, pw) + cov_term
    assert float(cov_term.abs().max()) > 1e-3 * float(torch.outer(gc, pw).abs().max())   # both terms matter here
    assert torch.allclose(rot.grad, expect, rtol=1e-9, atol=1e-12), (rot.grad, expect)


def test_set_camera_grad_validates_without_a_gpu():
    """gs_ctx_set_camera_grad checks its pointer, then its context, before touching either."""
    lib = ctypes.CDLL(os.path.join(PKG, "libgs_b200.so"))
    lib.gs_last_error.restype = ctypes.c_char_p
    lib.gs_ctx_set_camera_grad.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    assert lib.gs_ctx_set_camera_grad(None, 0x1002) == -1 and "aligned" in lib.gs_last_error().decode()
    assert lib.gs_ctx_set_camera_grad(None, 0x1000) == -1 and "null ctx" in lib.gs_last_error().decode()
    assert lib.gs_ctx_set_camera_grad(None, None) == -1 and "null ctx" in lib.gs_last_error().decode()
    import sys
    sys.path.insert(0, PKG)
    import gaussian
    assert callable(getattr(gaussian.RenderContext, "set_camera_grad"))
