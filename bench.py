#!/usr/bin/env python
"""bench.py -- Mpaths/s and Mrays/s of the path-tracing sample loop on N B200s.

A "step" is one pass of the hot path over one frame: BASELINE.json configs[1], the Cornell box
600x600 at 1000 spp, max depth 100 (src/scene.rs:630-730, src/main.rs:28-29).  With N > 1 ranks
(torchrun, one process per GPU) the 1000 samples per pixel are sharded: rank k renders global
samples [k*spp/N, (k+1)*spp/N) of every pixel and the fp32 sum buffers are combined with one NCCL
reduce to rank 0 (strong scaling: the frame is fixed).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` = whole-job Mpaths/s with the scene resident in HBM,
timed with CUDA events on the stream every kernel and the reduce run on, max over ranks.
`e2e` = the same metric through the reference-facing calls with HOST buffers: per step `vk_scene_upload`
of the flattened scene (H2D) and ONE `vk_render` call whose output is the caller's host frame (D2H inside);
with N > 1 ranks each rank's `vk_render_device` slice, the NCCL reduce and the D2H on rank 0.
`roofline` follows SURVEY 8(d): max(algorithmic flops / FP32 peak, algorithmic bytes / bandwidth of the level
the scene's working set lives in), the bound named by whichever is larger.  `other_configs` (N = 1 only)
are short runs of BASELINE.json's other four configurations so that they appear in the driver's record too.
`--impl reference` times the CPU restatement of the reference (oracle/, the Rust itself cannot be
built here) on the host cores with the same config, on a bounded sample of the frame's spp.
`--dump-outputs DIR` writes the frame the last timed step finished (see dump_frame) so that two builds can be
compared output for output: the seeds of the timed steps are fixed, so the same arguments give the same inputs.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIGS = {
    # name: (scene, param, width, height, spp, max_depth, cpu_spp)   -- BASELINE.json configs[0..4]
    "random_spheres": ("random_spheres_demo", 0, 400, 225, 16, 50, 16),
    "cornell": ("cornell_box", 0, 600, 600, 1000, 100, 64),
    "cornell_smoke": ("cornell_smoke", 0, 600, 600, 2000, 100, 32),
    "final_scene": ("final_scene", 0, 800, 800, 10000, 100, 4),
    "stress_1m": ("stress_spheres", 1000, 3840, 2160, 256, 50, 1),
}


def load_json(path, default=None):
    try:
        return json.load(open(path))
    except Exception:
        return default


DUMP_LIMIT = 64 * 10**6  # bytes of --dump-outputs, all files together


def dump_frame(out_dir, frame):
    """The finished (H, W, 3) float32 frame as out_dir/frame.npy.  A frame over DUMP_LIMIT (stress_1m at 4K) is
    replaced by a fixed sample of 2^20 pixels drawn with seed 0: out_dir/frame_sample.npy (N, 3) and the row-major
    pixel indices of that sample as out_dir/frame_sample_pixels.npy (float64, exact below 2^53)."""
    os.makedirs(out_dir, exist_ok=True)
    frame = np.ascontiguousarray(frame, dtype=np.float32)
    if frame.nbytes <= DUMP_LIMIT:
        np.save(os.path.join(out_dir, "frame.npy"), frame)
        return
    px = frame.reshape(-1, 3)
    idx = np.sort(np.random.default_rng(0).choice(len(px), size=1 << 20, replace=False))
    np.save(os.path.join(out_dir, "frame_sample.npy"), px[idx])
    np.save(os.path.join(out_dir, "frame_sample_pixels.npy"), idx.astype(np.float64))


def alg_work(scene_name):
    """Algorithmic flops / bytes per ray segment, counted by the instrumented oracle on the
    reference's own traversal order (profiles/alg_work_per_ray.json, made by profiles/make_alg_work.py)."""
    d = load_json(os.path.join(ROOT, "profiles", "alg_work_per_ray.json"), {})
    return d.get(scene_name)


def ncu_traffic(config, variant):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    summary of one `ncu --set full` capture of this config (profiles/ncu_traffic.json, written by
    profiles/summarize.py from the report); None when no capture of this (config, variant) exists."""
    d = load_json(os.path.join(ROOT, "profiles", "ncu_traffic.json"), {}) or {}
    return (d.get(f"{config}:{variant}") or {}).get("dram_bytes_per_launch")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag = True
        if not self.nv or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        busy = sorted(self.samples)[len(self.samples) // 4:]  # drop idle samples taken around the region
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


VARIANT_NAMES = {1: "megakernel", 2: "wavefront", 3: "staged", 4: "warpq", 5: "stepq"}


def kernel_of(kst, scene):
    flat_program = kst.node_visits == 0  # the flat traversal program visits no BVH node
    return {1: "k_megakernel_flat" if flat_program else ("k_megakernel_dyn" if scene.desc.n_nodes >= 65536 else "k_megakernel"),
            2: "k_wf_extend + k_wf_shade", 3: "k_staged_flat" if flat_program else "k_staged",
            4: "k_warpq_flat" if flat_program else "k_warpq", 5: "k_stepq"}.get(kst.variant, "?")


def make_roofline(config, variant_name, kernel_name, aw, k_rays, k_ms, fp32_peak, l2_gbs, peaks, scene_bytes):
    """SURVEY 8(d): achieved = max(flops_alg * rays/s / FP32 peak, bytes_alg * rays/s / bandwidth of the bound level).
    The level is where the TRAVERSAL working set (nodes + primitives, texels excluded) lives.  SURVEY 8(d): configs 1-4
    are KBs to ~2 MB, L1 / L2 resident and re-read by every ray -> no bandwidth bound is claimed, FP32 issue is the
    roofline; config 5 (64 MB of wide nodes + 20 MB of spheres, random access) is L2-bandwidth bound (peak: the L2 read
    microbenchmark measured live); anything over 100 MB would be HBM (peak: MEASURED_PEAKS.json).
    Units per launch = ray segments traced by that launch (vk_stats.rays)."""
    flops_ray, bytes_ray = aw.get("flops_per_ray"), aw.get("bytes_per_ray")
    if not flops_ray or not k_ms:
        return None
    rate = k_rays / (k_ms * 1e-3)
    f_ach, f_frac = flops_ray * rate / 1e12, flops_ray * rate / 1e12 / fp32_peak
    level = "l1" if scene_bytes <= (4 << 20) else ("l2" if scene_bytes <= (100 << 20) else "hbm")
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    b_peak = {"l1": None, "l2": l2_gbs, "hbm": hbm_peak}[level]
    b_ach = bytes_ray * rate / 1e9 if bytes_ray else None
    b_frac = b_ach / b_peak if (b_ach and b_peak) else None
    views = {"fp32": {"achieved": f_ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": f_frac, "alg_flops_per_ray": flops_ray,
                      "peak_source": "FFMA microbenchmark vk_measure_peaks, measured live (MEASURED_PEAKS.json has no fp32 figure)"},
             "bytes": {"level": level, "achieved": b_ach, "peak": b_peak, "unit": "GB/s", "frac": b_frac, "alg_bytes_per_ray": bytes_ray,
                       "peak_source": {"l1": "traversal working set <= 4 MB, L1 / L2 / constant-bank resident: no bandwidth bound claimed",
                                       "l2": "L2-resident 32 MiB read microbenchmark vk_measure_peaks, measured live",
                                       "hbm": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"}[level]}}
    use_bytes = b_frac is not None and b_frac > f_frac
    r = {"bound": level if use_bytes else "fp32", "achieved": b_ach if use_bytes else f_ach, "peak": b_peak if use_bytes else fp32_peak,
         "unit": "GB/s" if use_bytes else "TFLOP/s", "frac": b_frac if use_bytes else f_frac,
         "traffic": ncu_traffic(config, variant_name), "kernel": kernel_name, "kernel_ms": k_ms, "views": views}
    return r


# short runs of the other BASELINE.json configurations (N = 1): (spp of the short run, why)
OTHER_SPP = {"random_spheres": (16, "full config"), "cornell": (1000, "full config"), "cornell_smoke": (2000, "full config"),
             "final_scene": (64, "64 of the 10 000 spp (the config is quoted over 8 GPUs; throughput does not depend on spp)"),
             "stress_1m": (8, "8 of the 256 spp (throughput does not depend on spp)")}


def other_configs(vb, ctx, args, fp32_peak, l2_gbs, peaks):
    """One warm-up and two timed frames of every other configuration through vk_render_device (scene resident, kernels
    timed by the library's CUDA events on its stream), so that all five appear in the driver-run record."""
    out = []
    for name, (scene_name, param, W, H, spp_full, depth, _) in CONFIGS.items():
        if name == args.config:
            continue
        spp, why = OTHER_SPP[name]
        try:
            scene = vb.Scene(scene_name, seed=1, param=param)
            cam = scene.next_camera()
            ctx.upload(scene)
            import torch
            d_sum = torch.empty(W * H * 3, dtype=torch.float32, device="cuda")
            best = None
            for rep in range(3):
                st = ctx.render_device(cam, vb.render_params(W, H, spp, depth, seed=1 + rep, variant=args.variant), d_sum.data_ptr(), want_stats=True)
                if rep and (best is None or st.ms_kernels < best.ms_kernels):
                    best = st
            vname = VARIANT_NAMES.get(best.variant, str(best.variant))
            kname = kernel_of(best, scene)
            rl = make_roofline(name, vname, kname, alg_work(scene_name) or {}, best.rays, best.ms_kernels, fp32_peak, l2_gbs, peaks,
                               scene.nbytes() - int(scene.desc.n_texel_bytes))
            out.append({"config": name, "workload": f"{scene_name} {W}x{H}, max depth {depth}, {spp} spp measured ({why}; BASELINE.json configs[{list(CONFIGS).index(name)}] is {spp_full} spp)",
                        "ms": best.ms_kernels, "mpaths_per_s": best.paths / best.ms_kernels / 1e3, "mrays_per_s": best.rays / best.ms_kernels / 1e3,
                        "rays_per_path": best.rays / best.paths, "variant": vname, "kernel": kname,
                        "roofline": None if rl is None else {k: rl[k] for k in ("bound", "achieved", "peak", "unit", "frac")}})
            del d_sum
            scene.close()
        except Exception as e:  # a short extra run must never cost the main line
            out.append({"config": name, "error": str(e)})
    return out


def run_reference(args, cfg):
    """The reference's CPU implementation of the path (its C++ restatement, oracle/) on all host
    cores: same scene, resolution, depth; each step renders a bounded `cpu_spp` slice."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import vecchio_b200 as vb
    from oracle import pyoracle as po

    scene_name, param, W, H, spp, depth, cpu_spp = cfg
    scene = vb.Scene(scene_name, seed=1, param=param)
    cam = scene.next_camera()
    o = po.OracleScene(scene)
    cores = os.cpu_count()
    for i in range(args.warmup):
        o.render(cam, vb.render_params(W, H, cpu_spp, depth, seed=100 + i), threads=cores)
    paths = rays = 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        frame, _, st = o.render(cam, vb.render_params(W, H, cpu_spp, depth, seed=200 + i), threads=cores)
        paths += st.paths
        rays += st.rays
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_frame(args.dump_outputs, frame)
    v = paths / dt / 1e6
    line = {"impl": "reference", "metric": "Mpaths/s", "value": v, "unit": "Mpaths/s", "mrays_per_s": rays / dt / 1e6,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: {scene_name} {W}x{H}, max depth {depth}, {cpu_spp} spp per step "
                                   f"(bounded sample of the {spp} spp frame)", "seed": 1},
            "cpu_baseline": {"value": v, "unit": "Mpaths/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps} x {W}x{H}x{cpu_spp} spp, C++ restatement of the reference "
                                       f"(oracle/oracle.cpp, OpenMP dynamic over pixels); the Rust cannot be built (no rustc)"},
            "e2e": {"value": v, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args, cfg):
    import torch
    import torch.distributed as dist

    import vecchio_b200 as vb

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    scene_name, param, W, H, spp, depth, cpu_spp = cfg
    scene = vb.Scene(scene_name, seed=1, param=param)
    cam = scene.next_camera()
    ctx = vb.Context(local_rank)
    ctx.upload(scene)
    info = ctx.device_info()
    # One explicit (non-default) stream for everything that is timed: our kernels, the NCCL
    # reduce, the L2 flush and the CUDA events.
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    # spp sharding: rank k renders global samples [k*spp/N, (k+1)*spp/N)
    from vecchio_b200.sharding import reduce_sums_to_root, spp_slice
    s0, s_count = spp_slice(rank, world, spp)
    s1 = s0 + s_count
    n = W * H * 3
    d_sum = torch.empty(n, dtype=torch.float32, device=dev)
    d_rgb = torch.empty(n, dtype=torch.float32, device=dev)
    h_rgb = torch.empty(n, dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def params(seed):
        return vb.render_params(W, H, spp, depth, seed=seed, spp_begin=s0, spp_count=s1 - s0, variant=args.variant)

    def step_device(seed):
        ctx.render_device(cam, params(seed), d_sum.data_ptr(), want_stats=False)
        reduce_sums_to_root(d_sum, world)  # one NCCL reduce(sum) over NVLink on the same stream
        if rank == 0:
            ctx.finalize_device(d_sum.data_ptr(), d_rgb.data_ptr(), n, spp)

    h_frame = np.empty(n, dtype=np.float32)  # the caller's (pageable) host frame, as a Rust Vec<Vec3> would be

    def step_e2e(seed):
        ctx.upload(scene)  # vk_scene_upload: H2D of the flattened scene (host arrays -> device), every step
        if world == 1:     # the plugin call itself: vk_render(host params) -> host frame (D2H + copy-out inside)
            import ctypes as C
            st_ = vb.vk_stats()
            p_ = params(seed)
            ctx._check(ctx._L.vk_render(ctx._h, C.byref(cam), C.byref(p_), h_frame.ctypes.data, None, C.byref(st_)))
            return
        step_device(seed)
        if rank == 0:
            h_rgb.copy_(d_rgb, non_blocking=True)  # D2H of the finished frame
        stream.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing: W warm-up steps, then exactly K steps -------------------------
    for i in range(args.warmup):
        flush.zero_()
        step_device(1000 + i)
    ctx.flush_stats()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (256 MB memset, ~0.1 ms)
        step_device(1 + i)
    ev1.record(stream)
    barrier()
    clocks = sampler.result()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    st = ctx.flush_stats()
    counts = torch.tensor([st.paths, st.rays, st.dropped_samples, st.launches], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    paths, rays, dropped, launches = [float(x) for x in counts.tolist()]
    value = paths / (ms * 1e-3) / 1e6
    mrays = rays / (ms * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:  # before the kernel-only and e2e runs below reuse the device buffers
        dump_frame(args.dump_outputs, d_rgb.cpu().numpy().reshape(H, W, 3))

    # ---- kernel-only time of the dominant kernel (CUDA events inside the library) ---------------
    kst = ctx.render_device(cam, params(77), d_sum.data_ptr(), want_stats=True)
    k_ms, k_rays, k_paths = kst.ms_kernels, kst.rays, kst.paths
    variant_name = VARIANT_NAMES.get(kst.variant, str(kst.variant))
    kernel_name = kernel_of(kst, scene)

    # ---- end to end through the C ABI with host buffers -----------------------------------------
    for i in range(2):
        step_e2e(2000 + i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(3000 + i)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_paths = float(W) * H * spp * args.steps
    ctx.flush_stats()

    if rank == 0:
        peaks = load_json(os.path.join(ROOT, "MEASURED_PEAKS.json"), {})
        fp32_peak, l2_gbs = ctx.measure_peaks()
        aw = alg_work(scene_name) or {}
        flops_ray, bytes_ray = aw.get("flops_per_ray"), aw.get("bytes_per_ray")
        roofline = make_roofline(args.config, variant_name, kernel_name, aw, k_rays, k_ms, fp32_peak, l2_gbs, peaks, scene.nbytes() - int(scene.desc.n_texel_bytes))
        line = {"metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "mrays_per_s": mrays, "rays_per_path": rays / paths,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{args.config}: {scene_name} {W}x{H} at {spp} spp, max depth {depth} "
                                       f"(BASELINE.json configs[{list(CONFIGS).index(args.config)}])",
                           "parallelism": f"spp-sharded x{world}, NCCL reduce(sum) of {n * 4} B to rank 0" if world > 1 else "single GPU",
                           "seed": "1..K (one per step)", "l2": "256 MB memset between timed steps; scene itself is KB-sized and cache-resident by design",
                           "variant": variant_name, "scene_bytes": scene.nbytes()},
                "e2e": {"value": e2e_paths / e2e_s / 1e6, "unit": "Mpaths/s", "h2d_bytes_per_step": scene.nbytes() + 96 + 56,
                        "d2h_bytes_per_step": n * 4, "ms_per_step": e2e_s / args.steps * 1e3},
                "gpu_launches": int(launches), "dropped_samples": int(dropped), "clocks": clocks, "roofline": roofline,
                "kernel_only": {"mpaths_per_s": k_paths / (k_ms * 1e-3) / 1e6, "mrays_per_s": k_rays / (k_ms * 1e-3) / 1e6, "ms": k_ms},
                "device": info}
        if world == 1 and not args.no_other_configs:
            line["other_configs"] = other_configs(vb, ctx, args, fp32_peak, l2_gbs, peaks)
            ctx.upload(scene)
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as po
            o = po.OracleScene(scene)
            cores = os.cpu_count()
            _, _, cst = o.render(cam, vb.render_params(W, H, cpu_spp, depth, seed=5), threads=cores)
            line["cpu_baseline"] = {"value": cst.paths / cst.seconds / 1e6, "unit": "Mpaths/s", "mrays_per_s": cst.rays / cst.seconds / 1e6,
                                    "cores": cores, "kind": "port",
                                    "sample": f"{W}x{H} at {cpu_spp} spp ({cst.seconds:.1f} s), C++ restatement of the reference "
                                              f"(oracle/), OpenMP over pixels; the Rust reference cannot be built here (no rustc)"}
        print(json.dumps(line), flush=True)
    barrier()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cornell", choices=list(CONFIGS))
    ap.add_argument("--spp", type=int, default=0, help="override the config's spp (reduced-budget runs; say so when quoting)")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short runs of the other four BASELINE.json configurations")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR as .npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = list(CONFIGS[args.config])
    if args.spp:
        cfg[4] = args.spp
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, tuple(cfg))
    else:
        run_ours(args, tuple(cfg))


if __name__ == "__main__":
    main()
