"""Adaptive sampling (vk_render_adaptive) against fixed-spp renders: time, samples used, error and pass costs.

    python scripts/adaptive_bench.py [--errors 1,2,4] [--reps 3] [--out FILE.json]

Workloads: Cornell 600x600 (cap 1000 spp), final_scene 800x800 (cap 1024), random_spheres_demo 400x225 (cap 256),
pass_spp 64 (random spheres: 32), depth 50.  For each workload and max_error:
  - wall (host clock around the call, copy-back included) and kernel time (the call's CUDA-event sum) of the adaptive
    render and of the fixed render at the cap, median of --reps alternated repetitions;
  - samples used = sum(n_p) / (W*H*cap);
  - RMSE in 8-bit units (256 * sqrt(mean), unclamped) against an independent-seed fixed render at 4x the cap;
  - pass costs: pass count, per-pass kernel time (the time of the call capped at (k+1) * pass_spp minus the call capped
    at k * pass_spp: the passes before the cap are the same passes), and pass 0 against a plain vk_render at
    spp = pass_spp (what the list, the square atomics and the select cost);
  - equal-quality comparison: the RMSE of fixed renders at a ladder of spp, and the interpolated spp (and its kernel
    time) at which the fixed render's RMSE equals the adaptive one's.
The device name, its power limit and SM clocks are read in the same run and stored with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import vecchio_b200 as vb  # noqa: E402

WORKLOADS = [  # name, scene, width, height, cap, pass_spp
    ("cornell_600", "cornell_box", 600, 600, 1000, 64),
    ("final_scene_800", "final_scene", 800, 800, 1024, 64),
    ("random_spheres_400x225", "random_spheres_demo", 400, 225, 256, 32),
]
DEPTH = 50


def device_record():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    fields = [x.strip() for x in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(q.split(","), fields)) if len(fields) == 4 else {"error": r.stderr.strip() or "nvidia-smi failed"}


def units8(rgb):
    return 256.0 * np.sqrt(np.maximum(rgb.astype(np.float64), 0.0))


def rmse8(rgb, ref):
    return float(np.sqrt(np.mean((units8(rgb) - units8(ref)) ** 2)))


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def run(ctx, scene, cam, name, W, H, cap, M, errors, reps):
    p = lambda spp, seed=1: vb.render_params(W, H, spp, DEPTH, seed=seed)  # noqa: E731
    ctx.render(cam, p(M))  # warm-up: modules, buffers
    ref, _, _ = ctx.render(cam, p(4 * cap, seed=987654321))
    fixed_wall, fixed_kern = [], []
    for _ in range(reps):
        w, (rgb_fixed, _, st) = timed(lambda: ctx.render(cam, p(cap)))
        fixed_wall.append(w)
        fixed_kern.append(st.ms_kernels)
    fixed = {"spp": cap, "wall_ms": statistics.median(fixed_wall), "kernel_ms": statistics.median(fixed_kern),
             "rmse8": rmse8(rgb_fixed, ref), "variant": st.variant}
    ladder = []
    for spp in sorted({max(M, cap // 8), cap // 4, cap // 2, cap}):
        rgb, _, st = ctx.render(cam, p(spp))
        ladder.append({"spp": spp, "kernel_ms": st.ms_kernels, "rmse8": rmse8(rgb, ref)})
    plain0 = statistics.median([ctx.render(cam, p(M))[2].ms_kernels for _ in range(reps)])
    rows = []
    for e in errors:
        walls, kerns = [], []
        for _ in range(reps):  # the fixed render at the cap is timed above; adaptive calls alternate with it here
            w, (rgb, n, st) = timed(lambda: ctx.render_adaptive(cam, p(cap), M, e))
            walls.append(w)
            kerns.append(st.ms_kernels)
            ctx.render(cam, p(cap))
        passes = int(-(-int(n.max()) // M))
        cum = [0.0]
        for k in range(1, passes + 1):  # kernel time of the call capped after pass k-1
            cum.append(statistics.median([ctx.render_adaptive(cam, p(min(k * M, cap)), M, e)[2].ms_kernels for _ in range(reps)]))
        per_pass = [cum[k + 1] - cum[k] for k in range(passes)]
        per_pass[0] = cum[1]
        active = [int((n > k * M).sum()) for k in range(passes)]
        err = rmse8(rgb, ref)
        # the fixed spp whose RMSE equals the adaptive one's (RMSE falls monotonically along the ladder: interpolate in log)
        eq = None
        for a, b in zip(ladder, ladder[1:]):
            if a["rmse8"] >= err >= b["rmse8"]:
                t = (np.log(a["rmse8"]) - np.log(err)) / max(np.log(a["rmse8"]) - np.log(b["rmse8"]), 1e-12)
                spp_eq = float(np.exp(np.log(a["spp"]) + t * (np.log(b["spp"]) - np.log(a["spp"]))))
                eq = {"spp": spp_eq, "kernel_ms": a["kernel_ms"] + t * (b["kernel_ms"] - a["kernel_ms"])}
        rows.append({
            "max_error": e, "wall_ms": statistics.median(walls), "kernel_ms": statistics.median(kerns),
            "kernel_ms_spread": [min(kerns), max(kerns)], "samples_used": float(n.sum(dtype=np.float64) / (W * H * cap)),
            "paths": int(st.paths), "rays": int(st.rays), "launches": int(st.launches), "variant": int(st.variant),
            "rmse8": err, "passes": passes, "active_pixels_per_pass": active, "pass_kernel_ms": per_pass,
            "pass0_kernel_ms": cum[1], "plain_render_at_pass_spp_kernel_ms": plain0,
            "fixed_at_equal_rmse": eq if eq else "outside the ladder",
            "speedup_vs_fixed_cap_kernel": fixed["kernel_ms"] / statistics.median(kerns),
            "speedup_vs_fixed_equal_rmse_kernel": (eq["kernel_ms"] / statistics.median(kerns)) if eq else None,
        })
        print(json.dumps({"workload": name, **rows[-1]}), flush=True)
    return {"workload": name, "scene": scene.name, "width": W, "height": H, "cap": cap, "pass_spp": M, "depth": DEPTH,
            "fixed_at_cap": fixed, "fixed_ladder": ladder, "adaptive": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--errors", default="1,2,4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    errors = [float(x) for x in a.errors.split(",")]
    ctx = vb.Context(0)
    dev = device_record()
    print(json.dumps({"device": dev}), flush=True)
    out = {"device": dev, "workloads": []}
    for name, scene_name, W, H, cap, M in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        scene = vb.Scene(scene_name)
        cam = scene.next_camera()
        ctx.upload(scene)
        out["workloads"].append(run(ctx, scene, cam, name, W, H, cap, M, errors, a.reps))
    out["device_after"] = device_record()
    ctx.close()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
