"""Cost of the depth / alpha maps: plain frame vs maps frame on the C3 RGB scene, in one process.

  python profiles/maps_bench.py [--steps 40] [--warmup 5] [--out profiles/maps_bench_C3.json]

C3 = 2.4 M Gaussians (synthetic.py, seed 0), 1920x1080, view 0.  Alternates, step by step,
  plain : Splatter.forward (render_frame_final) + backward of an image gradient
  maps  : Splatter.render_maps(background=(0.2, 0.5, 1.0)) + backward of non-zero image, depth and alpha gradients
after `--warmup` steps of each.  Reports CUDA-event medians per step (forward + backward), then, in a second pass
with the library's per-stage events on, the median blend forward / backward stage times.  The card's name and power
limit are read in the same process.  Needs a GPU; writes one JSON file.
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

BG = (0.2, 0.5, 1.0)
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "maps_bench_C3.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("maps_bench.py needs a CUDA device")
    import gaussian
    import splatter
    import synthetic as S

    dev = torch.device("cuda", 0)
    n, w, h = 2_400_000, 1920, 1080
    g = S.make_gaussians(n, w, h, 0)
    v = S.make_view(w, h, 0)
    sp = splatter.Splatter.from_tensors(g, [dict(width=w, height=h, focal_x=v.fx, focal_y=v.fy, rot=v.rot,
                                                 tran=v.tran)], device=dev)
    params = list(sp.gaussian_3ds.parameters())
    go = (S.make_grad_output(h, w, 0) * (h * w)).to(dev)
    gen = torch.Generator().manual_seed(11)
    gd = (torch.rand(h, w, generator=gen) * 2 - 1).to(dev)
    ga = (torch.rand(h, w, generator=gen) * 2 - 1).to(dev)

    def plain():
        for p in params:
            p.grad = None
        img = sp(0)
        img.backward(go)

    def maps():
        for p in params:
            p.grad = None
        img, depth, alpha = sp.render_maps(0, background=BG)
        torch.autograd.backward([img, depth, alpha], [go, gd, ga])

    legs = {"plain": plain, "maps": maps}
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
    st = sp.frame_stats()

    med = {k: statistics.median(t) for k, t in times.items()}
    res = {
        "what": "C3 RGB (2.4 M Gaussians, 1920x1080, view 0): plain final frame vs maps frame (background "
                f"{BG}, non-zero image / depth / alpha gradients), forward + backward per step, alternating",
        "card": card(),
        "torch": torch.__version__,
        "steps": args.steps, "warmup": args.warmup,
        "step_ms_median": med,
        "step_ms_min": {k: min(t) for k, t in times.items()},
        "step_ms_max": {k: max(t) for k, t in times.items()},
        "maps_over_plain": med["maps"] / med["plain"],
        "stage_ms_median": {k: {s: statistics.median(v) for s, v in d.items()} for k, d in stage.items()},
        "blend_ratio": {s: statistics.median(stage["maps"][s]) / statistics.median(stage["plain"][s])
                        for s in ("blend_fwd", "blend_bwd")},
        "kernel_launches_per_step": launches,
        "n_instances": st["n_instances"],
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"step_ms_median": med, "maps_over_plain": res["maps_over_plain"],
                      "blend_ratio": res["blend_ratio"], "card": res["card"]}))


if __name__ == "__main__":
    main()
