"""Cost of the camera pose gradient: plain frame vs the same frame with pose gradients, C3 RGB, in one process.

  python profiles/camgrad_bench.py [--steps 40] [--warmup 5] [--out profiles/camgrad_bench_C3.json]

C3 = 2.4 M Gaussians (synthetic.py, seed 0), 1920x1080, view 0, on the free-camera path of Splatter.forward.
Alternates, step by step,
  plain  : forward + backward of an image gradient, pose tensors constant
  camgrad: the same with rot / tran requiring grad (gs_ctx_set_camera_grad: the projection backward also reduces
           the camera gradient, plus one finishing kernel)
after `--warmup` steps of each.  Reports CUDA-event medians per step, then, in a second pass with the library's
per-stage events on, the median projection-backward stage (which includes the finishing kernel), then, in a third
pass under torch.profiler, the median device time of the projection-backward and finishing kernels.  The card's
name and power limit are read in the same process.  Needs a GPU; writes one JSON file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "3d-gaussian-splatting_b200"))

STAGES = ["project", "depth_sort+scan+readback", "emit_keys", "tile_sort", "pack", "blend_fwd", "blend_bwd",
          "project_bwd"]


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:                      # the measurement still carries torch's device name
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "camgrad_bench_C3.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("camgrad_bench.py needs a CUDA device")
    import gaussian
    import splatter
    import synthetic as S

    dev = torch.device("cuda", 0)
    n, w, h = 2_400_000, 1920, 1080
    g = S.make_gaussians(n, w, h, 0)
    v = S.make_view(w, h, 0)
    intr = dict(width=w, height=h, focal_x=v.fx, focal_y=v.fy)
    sp = splatter.Splatter.from_tensors(g, [dict(intr, rot=v.rot, tran=v.tran)], device=dev)
    params = list(sp.gaussian_3ds.parameters())
    go = (S.make_grad_output(h, w, 0) * (h * w)).to(dev)
    rot = v.rot.clone().requires_grad_(True)
    tran = v.tran.clone().requires_grad_(True)

    def step(pose):
        for p in params + [rot, tran]:
            p.grad = None
        img = sp(None, extrinsics=dict(rot=pose[0], tran=pose[1]), intrinsics=intr)
        img.backward(go)

    legs = {"plain": lambda: step((v.rot, v.tran)), "camgrad": lambda: step((rot, tran))}
    for _ in range(args.warmup):
        for f in legs.values():
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in legs}
    launches = {}
    for _ in range(args.steps):
        for k, f in legs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0 = gaussian.kernel_launches()
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
            launches[k] = gaussian.kernel_launches() - k0
    # per-stage device times (library events), separate pass
    sp._rctx.set_timing(True)
    stage = {k: {s: [] for s in STAGES} for k in legs}
    for _ in range(max(5, args.steps // 4)):
        for k, f in legs.items():
            f()
            for s, ms in zip(STAGES, sp._rctx.stage_ms()):
                stage[k][s].append(ms)
    sp._rctx.set_timing(False)
    # kernel device times (CUPTI through torch.profiler), separate pass
    from torch.profiler import ProfilerActivity, profile
    kern = {"plain": {}, "camgrad": {}}
    for k, f in legs.items():
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(max(5, args.steps // 4)):
                f()
            torch.cuda.synchronize()
        for e in prof.events():
            for short in ("fused_project_bwd_kernel", "camgrad_finish_kernel"):
                if short in e.name and e.device_type == torch.autograd.DeviceType.CUDA:
                    kern[k].setdefault(short, []).append(e.device_time_total / 1000.0)
    st = sp.frame_stats()

    med = {k: statistics.median(t) for k, t in times.items()}
    kmed = {k: {s: statistics.median(t) for s, t in d.items()} for k, d in kern.items()}
    pb = {k: statistics.median(stage[k]["project_bwd"]) for k in legs}
    res = {
        "what": "C3 RGB (2.4 M Gaussians, 1920x1080, view 0), free-camera path: plain final frame vs the same with "
                "rot / tran requiring grad, forward + backward of an image gradient per step, alternating",
        "card": card(),
        "torch": torch.__version__,
        "steps": args.steps, "warmup": args.warmup,
        "step_ms_median": med,
        "step_ms_min": {k: min(t) for k, t in times.items()},
        "step_ms_max": {k: max(t) for k, t in times.items()},
        "camgrad_over_plain": med["camgrad"] / med["plain"],
        "stage_ms_median": {k: {s: statistics.median(x) for s, x in d.items()} for k, d in stage.items()},
        "project_bwd_stage_ms_median": pb,
        "project_bwd_stage_ratio": pb["camgrad"] / pb["plain"],
        "kernel_ms_median_profiler": kmed,
        "kernel_launches_per_step": launches,
        "grad_cam": torch.cat([rot.grad.reshape(-1), tran.grad]).tolist(),
        "n_instances": st["n_instances"],
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"step_ms_median": med, "camgrad_over_plain": res["camgrad_over_plain"],
                      "project_bwd_stage_ms_median": pb, "kernel_ms_median_profiler": kmed, "card": res["card"]}))


if __name__ == "__main__":
    main()
