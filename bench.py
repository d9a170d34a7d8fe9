#!/usr/bin/env python
"""Benchmark of the hot path: render + backward FPS at 1080p, 2.4M Gaussians.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C2|C3|C5] [--colour 3|27|48]
                  [--dump-outputs DIR]

One "step" = one forward + backward of one 1920x1080 view per GPU: raw parameters ->
image -> gradients of all five parameter tensors for a fixed upstream image gradient
(SURVEY.md §8d FPS_fb; no loss / optimizer inside), followed at N > 1 by the exchange of the
gradient bucket (views are sharded one per GPU, Gaussians replicated: weak scaling): our own
kernels over NVLink peer memory (push fused into the projection backward) at N = 2, 4, 8, else one
NCCL all-reduce.  `value` = N views / max-over-ranks step time, inputs resident in HBM.
`e2e`   = the same through the public `Splatter` API with the upstream gradient coming
from pinned HOST memory and the rendered image read back to the host every step.
Also on the line: `stage_ms`, `roofline` (HBM fraction as the metric asks + what really binds),
`gpu_launches` (counted by the library), at N = 1 short legs `sh` (D = 27 / 48) and `opaque_scene`, at
N > 1 `exchange_check` (active exchange vs NCCL, bit-equality across ranks) and `per_rank`.

--impl reference times the reference's own CUDA build (oracle/_ref: unmodified
gaussian.cu + bindings.cpp + renderer.py) driven with the reference's per-frame call
sequence (oracle/ref_pipeline.py) on the same scene, rank 0 only.  If oracle/_ref is
absent it falls back to the CPU oracle port on a tile sub-sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in ("3d-gaussian-splatting_b200", "oracle"):
    sys.path.insert(0, os.path.join(ROOT, _p))

import torch  # noqa: E402


def _ensure_built():
    """In-tree .so files normally travel with the snapshot; build them on a bare checkout."""
    import glob
    pkg = os.path.join(ROOT, "3d-gaussian-splatting_b200")
    if glob.glob(os.path.join(pkg, "gaussian*.so")) and os.path.exists(os.path.join(pkg, "libgs_b200.so")):
        return
    if int(os.environ.get("RANK", "0")) == 0:
        import importlib.util
        spec = importlib.util.spec_from_file_location("gs_b200_build", os.path.join(pkg, "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build_all()
    else:                                   # other ranks wait for rank 0's build
        t0 = time.time()
        while not glob.glob(os.path.join(pkg, "gaussian*.so")) and time.time() - t0 < 900:
            time.sleep(2)
        time.sleep(5)

WORKLOADS = {
    # name: (N gaussians, width, height, forward_only)
    "C2": (500_000, 1920, 1080, False),
    "C3": (2_400_000, 1920, 1080, False),
    "C5": (5_000_000, 3840, 2160, True),
    "tiny": (20_000, 320, 192, False),
}
METRIC = "render+backward FPS @1080p (2.4M Gaussians)"


# ------------------------------------------------------------------------------------------
def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:      # first sample before the timed region
                time.sleep(0.01)
            self.rows.clear()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nm, val in zip(names, r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return world, rank, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world, dev):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------
def timed_loop(step_fn, steps, warmup, world, dev):
    for _ in range(warmup):
        step_fn()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step_fn()
    e1.record()
    barrier(world)
    ms = e0.elapsed_time(e1) / steps
    return max_over_ranks(ms, world, dev)


def cpu_baseline(workload, n_tiles_sample=12, max_threads=32):
    """The CPU oracle (pure PyTorch) on the box's host cores, bounded to roughly half a minute:
    full projection + binning + exact sort of the frame (once), then blend forward + autograd
    backward on a tile sub-sample, extrapolated to all tiles (labelled as such).  PyTorch's CPU
    kernels stop scaling on these small per-tile tensors well before 32 threads, so the thread
    count is capped there and reported as `cores`."""
    import gs_oracle as O
    import synthetic as S
    n, w, h, fwd_only = WORKLOADS[workload]
    cores = min(os.cpu_count() or 1, max_threads)
    torch.set_num_threads(cores)
    v = S.make_view(w, h, 0)
    g = S.make_gaussians(n, w, h, 0)
    cam = O.Camera(w, h, v.fx, v.fy, v.rot, v.tran)
    T = cam.ntx * cam.nty
    tiles = torch.linspace(0, T - 1, n_tiles_sample).long()
    go = S.make_grad_output(h, w, 0)
    p = {k: t.clone().requires_grad_(not fwd_only) for k, t in g.items()}
    with torch.set_grad_enabled(not fwd_only):
        t0 = time.time()
        # front end: activations, projection, culling, binning, exact (tile, depth) sort
        nq, ns, opa_a, rgb_a = O.preactivate(p["quat"], p["scale"], p["opa"], p["rgb"])
        rp, rc, mask = O.global_culling(p["pos"], nq, ns, cam.rot, cam.tran, cam.near, cam.half_w, cam.half_h)
        idx = torch.nonzero(mask.bool()).squeeze(-1)
        p_c, c_c = rp[idx], rc[idx]
        rects = O.tile_rects(p_c[:, :2], c_c, 0.05, cam.tile_lx, cam.tile_ly, cam.ntx, cam.nty, cam.leftmost,
                             cam.topmost)
        gi, accum = O.bin_and_sort(p_c, c_c, rects, cam.ntx, cam.nty)
        s_pos, s_rgb, s_opa, s_cov = p_c[gi], rgb_a[idx][gi], opa_a[idx][gi], c_c[gi]
        t_front = time.time() - t0
        t1 = time.time()
        img = O.draw(s_pos, s_rgb, s_opa, s_cov, accum, cam.Hp, cam.Wp, cam.fx, cam.fy, tiles=tiles)
        t_blend = time.time() - t1
        if not fwd_only:
            t2 = time.time()
            img.backward(torch.ones_like(img) / img.numel())
            t_bwd = time.time() - t2          # blend backward of the sampled tiles + front-end backward
        else:
            t_bwd = 0.0
    est = t_front + (t_blend + t_bwd) * (T / n_tiles_sample)
    return {"value": 1.0 / est, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{workload}: full projection+binning+sort of {n} gaussians ({t_front:.1f}s), blend fwd"
                      f"{'' if fwd_only else '+bwd'} on {n_tiles_sample}/{T} tiles ({t_blend + t_bwd:.1f}s), "
                      f"extrapolated to all tiles; {cores} torch threads"}


# ------------------------------------------------------------------------------------------
def workload_string(name, n, w, h, colour, fwd_only):
    """Identical for both arms (the driver compares it): the scene, not its measured statistics."""
    col = "RGB colour (D=3)" if colour == 3 else f"per-pixel SH colour (D={colour})"
    return (f"{name}: {n} gaussians, {w}x{h}, {col}, {'forward only' if fwd_only else 'forward+backward'}, "
            f"one view per GPU (view k = rank mod 8), seed 0 (SURVEY.md §8d generator)")


def ncu_metrics(workload, colour, kernel):
    """Per-launch counters of `kernel` from the committed `ncu --set full` captures
    (profiles/*_ncu_metrics.json, written by profiles/summarize.py; latest round wins): DRAM traffic,
    executed warp instructions, MUFU (XU pipe) and FMA pipe utilisation.  None if not captured."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for name in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if name.endswith("_ncu_metrics.json"):
            try:
                d = json.load(open(os.path.join(pdir, name)))
                best = d.get(f"{workload}/D{colour}", {}).get(kernel, best)
            except Exception:
                pass
    return best


class Scene:
    """One replica of the benchmark scene on this rank's GPU, driven through the public Splatter API."""

    def __init__(self, workload, colour, dev, exchange="auto", opa_range=(0.05, 0.9)):
        import dp
        import splatter
        import synthetic as S
        self.n, self.w, self.h, self.fwd_only = WORKLOADS[workload]
        g = S.make_gaussians(self.n, self.w, self.h, 0, sh_dim=colour, opa_range=opa_range)
        views = [S.make_view(self.w, self.h, k) for k in range(8)]
        vd = [dict(width=v.width, height=v.height, focal_x=v.fx, focal_y=v.fy, rot=v.rot, tran=v.tran) for v in views]
        self.sp = splatter.Splatter.from_tensors(g, vd, device=dev, use_sh_coeff=colour != 3)
        self.params = list(self.sp.gaussian_3ds.parameters())
        self.bucket = dp.make_grad_bucket(self.params, exchange=exchange)
        self.symmetric = isinstance(self.bucket, dp.SymmetricGradBucket)
        self.go_host = S.make_grad_output(self.h, self.w, 0).pin_memory()
        self.go_dev = self.go_host.to(dev)
        self.dev = dev

    def step(self, view_id, exchange=True, go=None):
        for p in self.params:
            p.grad = None
        if self.fwd_only:
            with torch.no_grad():
                return self.sp(view_id)
        img = self.sp(view_id)
        img.backward(self.go_dev if go is None else go)
        if exchange:
            self.bucket.allreduce()
        return img


def exchange_check(sc, view_id, world, dev):
    """Run on every multi-GPU bench (the driver's GPU-test box has ONE GPU): the gradient bucket summed by the
    active exchange vs NCCL's all-reduce of the same per-rank gradients (the backward is deterministic, so
    two backwards of the same frame give identical local gradients), and bit-equality across ranks."""
    import torch.distributed as dist
    import renderer
    renderer.set_flat_grad_allocator(None)                      # plain bucket, no push: local gradients
    sc.step(view_id, exchange=False)
    ref = torch.cat([p.grad.flatten() for p in sc.params])
    dist.all_reduce(ref)
    if sc.symmetric:
        renderer.set_flat_grad_allocator(sc.bucket.allocator)
    sc.step(view_id, exchange=True)
    got = torch.cat([p.grad.flatten() for p in sc.params])
    err = (got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    digest = got.view(torch.int32).to(torch.int64).sum().reshape(1)
    alld = [torch.zeros_like(digest) for _ in range(world)]
    dist.all_gather(alld, digest)
    return {"mode": (sc.bucket.mode + ("+multimem.st" if getattr(sc.bucket, "push_mc", False) and sc.bucket.mode == "push" else ""))
            if sc.symmetric else "nccl",
            "max_rel_err_vs_nccl": float(err), "bit_equal_across_ranks": bool(all(int(d) == int(alld[0]) for d in alld)),
            "floats": int(got.numel())}


def run_ours(args, world, rank, local):
    import gaussian
    dev = torch.device("cuda", local)
    n, w, h, fwd_only = WORKLOADS[args.workload]
    sc = Scene(args.workload, args.colour, dev, exchange=args.exchange)
    sp, params, bucket = sc.sp, sc.params, sc.bucket
    exchange = "none" if world == 1 else (f"own kernels over symmetric memory ({bucket.mode}"
                                          f"{', broadcast via multimem.st' if getattr(bucket, 'push_mc', False) and bucket.mode == 'push' else ''})"
                                          if sc.symmetric else "NCCL all-reduce")
    view_id = rank % 8
    sp._rctx.set_timing(True)

    xcheck = None
    if world > 1 and not fwd_only:
        xcheck = exchange_check(sc, view_id, world, dev)

    # clocks / throttle reasons are sampled DURING the timed region (nvidia-smi -lms 20 in a side
    # process; the sampler is started, and has delivered its first row, before the warm-up)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = None

    last_img = [None]

    def step_resident():
        last_img[0] = sc.step(view_id)

    for _ in range(args.warmup):
        step_resident()
    barrier(world)
    launches0 = gaussian.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_resident()
    e1.record()
    barrier(world)
    launches = gaussian.kernel_launches() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_img[0], {k: getattr(sp.gaussian_3ds, k).grad
                                                      for k in ("pos", "rgb", "opa", "quat", "scale")})
    last_img[0] = None
    ms_local = e0.elapsed_time(e1) / args.steps
    ms = max_over_ranks(ms_local, world, dev)
    clocks = sampler.stop() if rank == 0 else {}

    # per-stage device times of the last frame (CUDA events on the launching stream)
    stage = sp._rctx.stage_ms()
    st = sp.frame_stats()

    # per-rank compute time without the exchange (separates view imbalance from the collective)
    compute_ms = ms_local
    if world > 1 and not fwd_only:
        import renderer
        renderer.set_flat_grad_allocator(None)
        k2 = max(5, args.steps // 4)
        for _ in range(2):
            sc.step(view_id, exchange=False)
        barrier(world)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(k2):
            sc.step(view_id, exchange=False)
        c1.record()
        torch.cuda.synchronize()
        compute_ms = c0.elapsed_time(c1) / k2
        if sc.symmetric:
            renderer.set_flat_grad_allocator(bucket.allocator)
        barrier(world)

    # ---- e2e: host buffers in the timed region -------------------------------------------
    img_host = torch.empty(h, w, 3, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    go_stages = [torch.empty_like(sc.go_dev) for _ in range(2)]   # double buffered: the H2D of step i+1 overlaps
    bwd_done = [None, None]                                        # the backward of step i, which still reads buffer i
    e2e_it = [0]

    def step_e2e():
        for p in params:
            p.grad = None
        main = torch.cuda.current_stream(dev)
        slot = e2e_it[0] & 1
        e2e_it[0] += 1
        go_stage = go_stages[slot]
        with torch.cuda.stream(copy_stream):
            if bwd_done[slot] is not None:
                copy_stream.wait_event(bwd_done[slot])           # the backward two steps ago has read this buffer
            go_stage.copy_(sc.go_host, non_blocking=True)        # H2D: this step's upstream gradient
            h2d_done = torch.cuda.Event()
            h2d_done.record(copy_stream)
        if fwd_only:
            with torch.no_grad():
                img = sp(view_id)
        else:
            img = sp(view_id)                                    # camera (48 B) goes host->device inside
        fwd_done = torch.cuda.Event()
        fwd_done.record(main)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(fwd_done)
            img_host.copy_(img.detach(), non_blocking=True)      # D2H: the rendered image
        if not fwd_only:
            main.wait_event(h2d_done)
            img.backward(go_stage)
            bucket.allreduce()
            bwd_done[slot] = torch.cuda.Event()
            bwd_done[slot].record(main)
        copy_stream.synchronize()

    ms_e2e = timed_loop(step_e2e, args.steps, max(3, args.warmup // 2), world, dev)

    # per-rank record (every rank contributes; rank 0 prints)
    per_rank = None
    if world > 1:
        import torch.distributed as dist
        mine = torch.tensor([float(view_id), float(st["n_instances"]), float(st["n_instances_eff"]), compute_ms, ms_local],
                            dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": r, "view": int(t[0]), "tile_instances_M": int(t[1]), "consumed_M_eff": int(t[2]),
                     "compute_ms": round(float(t[3]), 4), "step_ms": round(float(t[4]), 4),
                     "exchange_ms": round(float(t[4]) - float(t[3]), 4)} for r, t in enumerate(allr)]
    if rank != 0:
        return None
    M, Meff = int(st["n_instances"]), int(st["n_instances_eff"])
    Meff_b = int(st.get("n_instances_eff_bwd", -1))
    if Meff_b < 0:
        Meff_b = Meff
    T = int(st["n_tiles"])
    P = int(st["width_padded"]) * int(st["height_padded"])
    D = args.colour
    peak, peak_src = measured_peak_gbs()
    bf = 4 * (7 + D) * Meff + 12 * P + 4 * (T + 1)
    bb = 8 * (7 + D) * Meff_b + 24 * P + 4 * (T + 1)             # the backward's OWN consumed count
    blend_f_ms, blend_b_ms = stage[5], stage[6]
    roof_kernel = "blend_bwd" if not fwd_only else "blend_fwd"
    alg_bytes, k_ms = (bb, blend_b_ms) if not fwd_only else (bf, blend_f_ms)
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms and k_ms > 0 else None
    pairs = (Meff_b if not fwd_only else Meff) * 256
    ncu = ncu_metrics(args.workload, D, roof_kernel) or {}
    sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    roof = {"bound": "hbm", "kernel": roof_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": (achieved / peak) if achieved else None, "traffic": ncu.get("dram_bytes"),
            "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full)",
            "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
            # the roof that actually binds: instruction issue (4 warp-instructions / clk / SM) and MUFU (16 / clk / SM)
            "binding": "issue",
            "pairs_per_launch": pairs, "pairs_per_s": pairs / (k_ms * 1e-3) if k_ms and k_ms > 0 else None,
            "pairs_per_clk_per_sm": pairs / (k_ms * 1e-3 * sm_hz * n_sm) if k_ms and k_ms > 0 else None,
            "issue_frac": ncu.get("issue_active_frac"), "mufu_frac": ncu.get("xu_pipe_frac"),
            "fma_pipe_frac": ncu.get("fma_pipe_frac"), "warp_inst_per_launch": ncu.get("warp_inst"),
            "thread_inst_per_pair": (ncu["warp_inst"] * 32.0 / pairs) if ncu.get("warp_inst") and pairs else None,
            "ncu_source": ncu.get("source"),
            "note": "blend is instruction-issue / MUFU bound, not HBM bound (SURVEY.md §8d): the HBM fraction is reported "
                    "because the metric asks for it; issue_frac / mufu_frac come from the committed ncu capture of this "
                    "workload (null if not captured), pairs_per_s is measured live",
            "blend_fwd": {"ms": blend_f_ms, "algorithmic_bytes": bf,
                          "achieved": bf / (blend_f_ms * 1e-3) / 1e9 if blend_f_ms > 0 else None},
            "blend_bwd": {"ms": blend_b_ms, "algorithmic_bytes": bb,
                          "achieved": bb / (blend_b_ms * 1e-3) / 1e9 if blend_b_ms > 0 else None}}
    out = {
        "metric": METRIC if args.workload == "C3" else f"render{'' if fwd_only else '+backward'} FPS ({args.workload})",
        "value": world * 1000.0 / ms, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, n, w, h, D, fwd_only),
                   "tile_instances_M": M, "tile_instances_consumed_M_eff": Meff, "consumed_by_backward": Meff_b,
                   "max_tile_count": st["max_tile_count"],
                   "n_visible": st["n_visible"], "l2": "inputs larger than L2 (per-frame working set "
                                                       f"{(M * 112 + n * 56) / 1e6:.0f} MB >> 126 MB)",
                   "parallelism": f"dp{world} over views, gradient bucket exchange: {exchange}"},
        "clocks": clocks,
        "e2e": {"value": world * 1000.0 / ms_e2e, "unit": "frames/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(sc.go_host.numel() * 4 + 48), "d2h_bytes_per_step": int(img_host.numel() * 4),
                "api": "Splatter.forward(camera_id) + image.backward(grad) with pinned host grad / image buffers"},
        "gpu_launches": int(launches),
        "gpu_launches_note": "kernels of libgs_b200 launched by rank 0 inside the timed region, counted by the library "
                             "(gs_kernel_launches); CUB scan / onesweep sort kernels are library code and not counted",
        "stage_ms": dict(zip(["project", "depth_sort+scan+readback", "emit_keys", "tile_sort", "pack", "blend_fwd",
                              "blend_bwd", "project_bwd"], [round(x, 4) for x in stage])),
        "stage_ms_note": "one frame (the last resident step) on rank 0, CUDA events recorded by the library",
        "roofline": roof,
    }
    if xcheck is not None:
        out["exchange_check"] = xcheck
    if per_rank is not None:
        out["per_rank"] = per_rank
    if world == 1 and args.workload == "C3" and D == 3 and not args.no_extra_legs:
        out["sh"] = sh_legs(dev)
        out["opaque_scene"] = opaque_leg(dev, peak)
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args.workload)
    return out


DUMP_BYTES = 60 << 20


def dump_outputs(out_dir, img, grads):
    """What the last timed step returned to its caller, as float32 .npy files: `image` (pixels as rows
    of 3) and `grad_<name>` for each parameter tensor that has a gradient.  So that the dump stays
    under DUMP_BYTES, arrays longer than k rows keep a fixed sample of k rows (seed 0, one sample per
    row count, rows in ascending order), k chosen from the bytes of one row of every array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"image": img.detach().reshape(-1, 3)}
    arrays.update({"grad_" + k: g for k, g in grads.items() if g is not None})
    k = DUMP_BYTES // sum(4 * a[0].numel() for a in arrays.values())
    samples = {}
    for name, a in arrays.items():
        n = a.shape[0]
        if n > k:
            if n not in samples:
                perm = torch.randperm(n, generator=torch.Generator().manual_seed(0))
                samples[n] = perm[:k].sort().values.to(a.device)
            a = a[samples[n]]
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


def _short_leg(sc, steps=10, warmup=3):
    for _ in range(warmup):
        sc.step(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sc.step(0)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def sh_legs(dev):
    """BASELINE configs[2] as written ("SH degree 3") and the reference's own SH (degree 2): short 10-step
    legs of the same C3 scene with per-pixel SH colour; D=27 also times the reference's CUDA build here."""
    import gc
    res = {}
    for D in (27, 48):
        sc = Scene("C3", D, dev)
        sc.sp._rctx.set_timing(True)
        ms = _short_leg(sc)
        stage = sc.sp._rctx.stage_ms()
        leg = {"value": 1000.0 / ms, "unit": "frames/s", "ms_per_step": ms, "steps": 10, "warmup": 3,
               "blend_fwd_ms": round(stage[5], 4), "blend_bwd_ms": round(stage[6], 4), "pack_ms": round(stage[4], 4)}
        del sc
        gc.collect()
        torch.cuda.empty_cache()
        if D == 27:
            try:
                ref_ms = reference_ms("C3", 27, dev, steps=5, warmup=2)
                if ref_ms:
                    leg["reference_ms_per_step"] = ref_ms
                    leg["vs_reference"] = ref_ms / ms
            except Exception as e:                    # the reference arm is optional here
                leg["reference_error"] = str(e)[:200]
        res[str(D)] = leg
    return res


def opaque_leg(dev, peak):
    """SURVEY.md §8d lever 3: the same C3 geometry with opacities in [0.5, 0.99] - pixels saturate after a few
    instances, the regime where the blend IS closer to HBM-bound; reports its HBM fraction."""
    import gc
    sc = Scene("C3", 3, dev, opa_range=(0.5, 0.99))
    sc.sp._rctx.set_timing(True)
    ms = _short_leg(sc)
    stage = sc.sp._rctx.stage_ms()
    st = sc.sp.frame_stats()
    T, P = int(st["n_tiles"]), int(st["width_padded"]) * int(st["height_padded"])
    mf, mb = int(st["n_instances_eff"]), int(st.get("n_instances_eff_bwd", st["n_instances_eff"]))
    bf = 40 * mf + 12 * P + 4 * (T + 1)
    bb = 80 * mb + 24 * P + 4 * (T + 1)
    out = {"opacity_range": [0.5, 0.99], "ms_per_step": ms, "tile_instances_M": int(st["n_instances"]),
           "consumed_M_eff": mf, "consumed_by_backward": mb,
           "blend_fwd": {"ms": stage[5], "achieved_GBps": bf / (stage[5] * 1e-3) / 1e9, "frac_of_hbm_peak": bf / (stage[5] * 1e-3) / 1e9 / peak},
           "blend_bwd": {"ms": stage[6], "achieved_GBps": bb / (stage[6] * 1e-3) / 1e9, "frac_of_hbm_peak": bb / (stage[6] * 1e-3) / 1e9 / peak}}
    del sc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def reference_ms(workload, colour, dev, steps, warmup):
    """ms per step of the reference's CUDA build on this GPU (None when oracle/_ref is absent)."""
    import ref_pipeline
    import synthetic as S
    n, w, h, fwd_only = WORKLOADS[workload]
    gref, rref = ref_pipeline.load_reference()
    if gref is None:
        return None
    g = S.make_gaussians(n, w, h, 0, sh_dim=colour)
    v = S.make_view(w, h, 0)
    frame = ref_pipeline.LegacyFrame(gref, rref, w, h, v.fx, v.fy, v.rot.to(dev), v.tran.to(dev), use_sh_coeff=colour != 3)
    p = {k: t.to(dev).clone().requires_grad_(True) for k, t in g.items()}
    go = S.make_grad_output(h, w, 0).to(dev)

    def step():
        for t in p.values():
            t.grad = None
        img = frame(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"])
        img.backward(go)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_reference(args, world, rank, local):
    """Reference arm: rank 0 only, one GPU (the reference has no multi-GPU path)."""
    if rank != 0:
        return None
    import ref_pipeline
    import synthetic as S
    n, w, h, fwd_only = WORKLOADS[args.workload]
    gref, rref = ref_pipeline.load_reference()
    if gref is None:
        cb = cpu_baseline(args.workload)
        return {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": 1,
                "steps": 1, "warmup": 0, "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": args.workload, "note": "oracle/_ref absent: CPU oracle port"},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    dev = torch.device("cuda", local)
    if args.colour == 48:
        return {"impl": "reference", "unavailable": "the reference has no SH degree-3 path (calc_sh is called with 9 bases only)"}
    g = S.make_gaussians(n, w, h, 0, sh_dim=args.colour)
    v = S.make_view(w, h, 0)
    frame = ref_pipeline.LegacyFrame(gref, rref, w, h, v.fx, v.fy, v.rot.to(dev), v.tran.to(dev),
                                     use_sh_coeff=args.colour != 3)
    p = {k: t.to(dev).clone().requires_grad_(True) for k, t in g.items()}
    go = S.make_grad_output(h, w, 0).to(dev)

    def step():
        for t in p.values():
            t.grad = None
        if fwd_only:
            with torch.no_grad():
                frame(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"])
        else:
            img = frame(p["pos"], p["rgb"], p["opa"], p["quat"], p["scale"])
            img.backward(go)

    sampler = ClockSampler(local)
    sampler.start()
    ms = timed_loop(step, args.steps, args.warmup, 1, dev)
    clocks = sampler.stop()
    fps = 1000.0 / ms
    return {"impl": "reference", "metric": METRIC if args.workload == "C3" else f"FPS ({args.workload})",
            "value": fps, "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_string(args.workload, n, w, h, args.colour, fwd_only),
                       "impl": "reference CUDA build (oracle/_ref: unmodified gaussian.cu + bindings.cpp + renderer.py, "
                               "-std=c++17 flag only) driven with the call sequence of reference splatter.py:513-655",
                       "tile_instances_M": frame.aux.get("n_instances"), "max_tile_count": frame.aux.get("max_tile"),
                       "note": "reference backward is only valid for <= 500 instances per tile (SURVEY.md hazard 1); "
                               "timing is still that of its stock code path"},
            "clocks": clocks,
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": 0, "kind": "reference",
                             "sample": "the reference has no CPU implementation of this path; this arm is its own "
                                       "CUDA build on the same GPU (the stronger baseline)"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    # NCCL / torchrun helpers write banners to fd 1; keep the contract "ONE JSON line on stdout":
    # everything else goes to stderr, the JSON line is written to the saved original stdout.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-legs", action="store_true",
                    help="skip the short SH (D=27, 48) and opaque-scene legs of the default N=1 C3 run")
    ap.add_argument("--exchange", default="auto", choices=["auto", "multimem", "p2p", "push", "nccl"],
                    help="N>1 gradient exchange: own push / p2p / multimem kernels on a symmetric bucket, NCCL all-reduce, "
                         "or auto (push at N = 2, 4, 8; NCCL otherwise)")
    ap.add_argument("--colour", type=int, default=3, choices=[3, 27, 48],
                    help="3 = RGB (default; the reference's published 2.4M point), 27 = per-pixel SH degree 2 "
                         "(the reference's use_sh_coeff), 48 = SH degree 3 extension")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the image and parameter gradients of the last timed step to DIR/<name>.npy "
                         "(float32; large arrays as a fixed seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    if args.impl != "reference":
        _ensure_built()
    world, rank, local = dist_setup(args.gpus)
    if args.impl == "reference":
        out = run_reference(args, world, rank, local)
    else:
        out = run_ours(args, world, rank, local)
    if rank == 0 and out is not None:
        real_stdout.write(json.dumps(out) + "\n")
        real_stdout.flush()
    if world > 1:
        import torch.distributed as dist
        if args.impl != "reference":
            dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
