"""CPU checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/gs_b200.h declares, and the pybind module exposes the reference's surface
(reference src/bindings.cpp:21-50).  No compute calls (no GPU here)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "3d-gaussian-splatting_b200")


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "gs_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(gs_[a-z0-9_]+)\s*\(", txt)))


def test_header_declares_the_expected_entry_points():
    syms = _declared_symbols()
    for s in ("gs_project_fwd", "gs_project_bwd", "gs_tile_list", "gs_gather", "gs_draw_fwd", "gs_draw_bwd",
              "gs_w2c_fwd", "gs_w2c_bwd", "gs_jacobian", "gs_render_forward", "gs_render_backward",
              "gs_ctx_create", "gs_ctx_destroy"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(os.path.join(PKG, "libgs_b200.so"))
    for s in _declared_symbols():
        assert hasattr(lib, s), f"libgs_b200.so does not export {s}"
    lib.gs_abi_version.restype = ctypes.c_int
    assert lib.gs_abi_version() == 2
    lib.gs_draw_workspace_bytes.restype = ctypes.c_size_t
    assert lib.gs_draw_workspace_bytes(0, 3) >= 0
    assert lib.gs_draw_workspace_bytes(1000, 3) >= 1000 * (16 + 16 + 8 + 48)


def test_pybind_module_has_reference_surface():
    import sys
    sys.path.insert(0, PKG)
    import torch  # noqa: F401
    import gaussian
    for name in ("culling", "world2camera", "world2camera_backward", "jacobian", "calc_tile_list",
                 "gather_gaussians", "draw", "draw_backward", "global_culling", "global_culling_backward"):
        assert callable(getattr(gaussian, name)), name
    t = gaussian.Tiles()
    for a in ("top", "bottom", "left", "right"):
        assert hasattr(t, a)
    g = gaussian.Gaussian3ds()
    for a in ("pos", "rgb", "opa", "quat", "scale", "cov"):
        assert hasattr(g, a)
    g.pos = torch.zeros(2, 3)
    assert g.pos.shape == (2, 3)


def test_shim_rejects_cpu_tensors():
    import sys
    import pytest
    sys.path.insert(0, PKG)
    import torch
    import gaussian
    with pytest.raises(RuntimeError):
        gaussian.world2camera(torch.zeros(4, 3), torch.eye(3), torch.zeros(3), torch.zeros(4, 3))


def test_product_path_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under the package may import, call or link it, and
    the package must not carry a CPU fallback for the kernels."""
    bad = []
    for root, _, files in os.walk(PKG):
        if "build" in root.split(os.sep):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(root, f), errors="ignore").read()
                if re.search(r"gs_oracle|ref_pipeline|import\s+oracle|from\s+oracle|oracle/", txt):
                    bad.append(os.path.join(root, f))
    assert not bad, bad


def test_argument_validation_needs_no_gpu():
    """Every entry point validates its arguments before touching CUDA: bad calls return
    GS_ERR_INVALID_ARG (-1) / GS_ERR_UNSUPPORTED (-2) with a message in gs_last_error()."""
    lib = ctypes.CDLL(os.path.join(PKG, "libgs_b200.so"))
    lib.gs_last_error.restype = ctypes.c_char_p
    P, LL, I = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int

    def err():
        return lib.gs_last_error().decode()

    # gradient exchange kernels
    lib.gs_allreduce_multimem_f32.argtypes = [P, LL, I, I, P]
    assert lib.gs_allreduce_multimem_f32(None, 16, 0, 2, None) == -1 and "bad arguments" in err()
    assert lib.gs_allreduce_multimem_f32(0x1000, 15, 0, 2, None) == -1          # not a multiple of 4 floats
    assert lib.gs_allreduce_multimem_f32(0x1008, 16, 0, 2, None) == -1 and "16-byte" in err()
    assert lib.gs_allreduce_multimem_f32(0x1000, 16, 2, 2, None) == -1          # rank out of range
    ptrs = (P * 3)(0x1000, 0x2000, 0x3000)
    lib.gs_allreduce_p2p_f32.argtypes = [ctypes.POINTER(P), LL, I, I, P]
    assert lib.gs_allreduce_p2p_f32(ptrs, 16, 0, 3, None) == -1 and "2, 4 or 8" in err()
    bad = (P * 2)(0x1000, 0x2004)
    assert lib.gs_allreduce_p2p_f32(bad, 16, 0, 2, None) == -1 and "16-byte" in err()
    lib.gs_allreduce_push_finish_f32.argtypes = [ctypes.POINTER(P), P, LL, LL, I, I, P]
    two = (P * 2)(0x1000, 0x2000)
    assert lib.gs_allreduce_push_finish_f32(two, 0x3000, 64, 16, 0, 2, None) == -1   # 2 * per < n
    assert lib.gs_allreduce_push_finish_f32(two, 0x3000, 64, 30, 0, 2, None) == -1   # per not a multiple of 4
    assert lib.gs_allreduce_push_finish_f32(two, None, 64, 32, 0, 2, None) == -1
    # contexts / frames
    lib.gs_ctx_set_grad_push.argtypes = [P, P]
    assert lib.gs_ctx_set_grad_push(None, None) == -1 and "null ctx" in err()
    lib.gs_ctx_create.argtypes = [P]
    assert lib.gs_ctx_create(None) == -1
    lib.gs_frame_instances.argtypes = [P]
    lib.gs_frame_instances.restype = LL
    assert lib.gs_frame_instances(None) == -1
    lib.gs_render_backward.argtypes = [P] * 14
    assert lib.gs_render_backward(*([None] * 14)) == -1 and "null ctx" in err()
    # optimizer
    lib.gs_adam_step.argtypes = [P, P, P, P, LL, P, P, I, ctypes.c_float, ctypes.c_float, ctypes.c_float, I, P]
    ends = (LL * 1)(16)
    lrs = (ctypes.c_float * 1)(1e-3)
    assert lib.gs_adam_step(0x1000, 0x2000, 0x3000, 0x4000, 16, ends, lrs, 1, 0.9, 0.99, 1e-8, 0, None) == -1  # step 0
    assert lib.gs_adam_step(0x1000, 0x2000, 0x3000, 0x4000, 15, ends, lrs, 1, 0.9, 0.99, 1e-8, 1, None) == -1  # n % 4
    assert lib.gs_adam_step(0x1000, 0x2000, 0x3000, 0x4000, 16, ends, lrs, 9, 0.9, 0.99, 1e-8, 1, None) == -1  # > 8 segments


def test_round2_entry_points_and_tune_knobs_validate_without_a_gpu():
    """The entry points added in round 2 (loss, densification, tuning, push-finish through the switch, launch
    counter) reject bad arguments before touching CUDA; gs_tune knows exactly the knobs gather and sh_tc and
    refuses values outside their ranges."""
    lib = ctypes.CDLL(os.path.join(PKG, "libgs_b200.so"))
    lib.gs_last_error.restype = ctypes.c_char_p
    P, LL, I, F = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_float

    def err():
        return lib.gs_last_error().decode()

    lib.gs_loss_workspace_bytes.restype = ctypes.c_size_t
    assert lib.gs_loss_workspace_bytes(1080, 1920) >= 1080 * 1920 * 9 * 4 and lib.gs_loss_workspace_bytes(0, 5) == 0
    lib.gs_loss_l1_ssim.argtypes = [P, P, I, I, I, F, F, F, P, P, P, ctypes.c_size_t, P]
    assert lib.gs_loss_l1_ssim(None, None, 0, 64, 64, 0.9, -0.1, 0.1, None, None, None, 0, None) == -1 and "null" in err()
    assert lib.gs_loss_l1_ssim(0x1000, 0x2000, 0, 8, 64, 0.9, -0.1, 0.1, None, 0x3000, 0x4000, 1 << 30, None) == -1 \
        and "11x11" in err()
    assert lib.gs_loss_l1_ssim(0x1000, 0x2000, 0, 64, 64, 0.9, -0.1, 0.1, None, 0x3000, 0x4000, 16, None) == -1 \
        and "workspace" in err()
    lib.gs_densify_workspace_bytes.restype = ctypes.c_size_t
    assert lib.gs_densify_workspace_bytes(1000) > 0
    lib.gs_densify_plan.argtypes = [P, P, P, I, I, F, F, F, I, F, I, I, P, P, P, ctypes.c_size_t, P]
    assert lib.gs_densify_plan(None, None, None, -1, 0, 0.0, 1.0, 1e-4, 1, 0.1, 1, 1, None, None, None, 0, None) == -1
    assert lib.gs_densify_plan(None, None, None, 10, 0, 0.0, 1.0, 1e-4, 1, 0.1, 1, 1, None, None, None, 0, None) == -1
    lib.gs_densify_apply.argtypes = [P] * 5 + [I, I, P, P, P, F, P, I, I, I, I] + [P] * 6
    assert lib.gs_densify_apply(*([None] * 5), 10, 3, None, None, None, 0.01, None, 5, 0, 2, 0, *([None] * 6)) == -1  # splits need normals
    lib.gs_tune.argtypes = [ctypes.c_char_p, I]
    assert lib.gs_tune(b"no_such_knob", 1) == -1 and "unknown knob" in err()
    assert lib.gs_tune(None, 1) == -1
    lib.gs_tune_get.argtypes = [ctypes.c_char_p, ctypes.POINTER(I)]

    def tuned(knob):
        v = I(-1)
        assert lib.gs_tune_get(knob, ctypes.byref(v)) == 0, knob
        return v.value

    # the two knobs accept every value of their range; the shipped defaults are restored last
    for knob, values, dflt in ((b"gather", (0, 1), 1), (b"sh_tc", (0, 1, 2, 3), 3)):
        for value in values + (dflt,):
            assert lib.gs_tune(knob, value) == 0, (knob, value)
            assert tuned(knob) == value
    # out of range: refused, and the knob keeps its value
    for knob, bad in ((b"sh_tc", 7), (b"sh_tc", -1), (b"gather", 2), (b"gather", -1)):
        before = tuned(knob)
        assert lib.gs_tune(knob, bad) == -1 and "out of range" in err(), (knob, bad)
        assert tuned(knob) == before
    # the knobs of the retired blend-kernel variants are gone
    for knob in (b"fwd_kernel", b"fwd_ch", b"fwd_px", b"bwd_kernel", b"bwd_px", b"bwd_ws", b"bwd_unroll", b"bwd_stages",
                 b"bwd_minb", b"bwd_rq", b"bwd_ch", b"strict"):
        assert lib.gs_tune(knob, 0) == -1 and "unknown knob" in err(), knob
    lib.gs_allreduce_push_finish_mc_f32.argtypes = [P, P, P, LL, LL, I, I, P]
    assert lib.gs_allreduce_push_finish_mc_f32(None, 0x1000, 0x2000, 64, 32, 0, 2, None) == -1
    assert lib.gs_allreduce_push_finish_mc_f32(0x1000, 0x2000, 0x3000, 64, 16, 0, 2, None) == -1      # 2 * per < n
    lib.gs_kernel_launches.restype = ctypes.c_ulonglong
    assert lib.gs_kernel_launches() == 0                                    # nothing launched in this process
    lib.gs_frame_tile_consumed.argtypes = [P, P, P]
    assert lib.gs_frame_tile_consumed(None, None, None) == -1
