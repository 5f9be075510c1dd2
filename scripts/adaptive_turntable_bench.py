"""Adaptive sampling of a batch of frames (vk_render_frames_adaptive_rgb8) against K single adaptive calls and the fixed batch.

    python scripts/adaptive_turntable_bench.py [--ks 1,4,16] [--reps 5] [--out FILE.json]

Workloads (depth 50):
  - random_spheres_demo turntable, 400x225, cap 256, pass_spp 32, max_error 1 and 4;
  - bowser_demo turntable, 400x225, cap 256, pass_spp 32, max_error 1 and 4;
  - Cornell box 600x600 (fixed camera: K copies, frame f with seed + f), cap 1000, pass_spp 64, max_error 4.
For each workload, max_error and K, three ways to render the same K frames, per frame (the call's total / K):
  - batch: one vk_render_frames_adaptive_rgb8 call over the K cameras;
  - sequential: K vk_render_adaptive_rgb8 calls, frame f with seed + f (AUTO picks each frame's kernel itself);
  - fixed: one vk_render_frames_rgb8 call at the cap.
Wall time is a host clock around the call(s), copy-back included; kernel time is the sum of the calls' CUDA-event
kernel time (stats.ms_kernels).  Median and [min, max] of --reps repetitions in which the three alternate.  Also recorded:
samples used (sum of n_p over K * W*H * cap), pass count, and the kernel each way ran.  The device name, its power limit and
SM clock are read in the same run and stored with the numbers."""
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

WORKLOADS = [  # name, scene, width, height, cap, pass_spp, max_errors
    ("random_spheres_400x225", "random_spheres_demo", 400, 225, 256, 32, (1.0, 4.0)),
    ("bowser_400x225", "bowser_demo", 400, 225, 256, 32, (1.0, 4.0)),
    ("cornell_600", "cornell_box", 600, 600, 1000, 64, (4.0,)),
]
DEPTH = 50


def device_record():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    fields = [x.strip() for x in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(q.split(","), fields)) if len(fields) == 4 else {"error": r.stderr.strip() or "nvidia-smi failed"}


def cameras(scene, k):
    """The scene's first k cameras; a fixed-camera scene repeats its one camera (the frames differ by seed)."""
    cams = [scene.next_camera()]
    while len(cams) < k:
        c = scene.next_camera()
        cams.append(c if c is not None else cams[-1])
    return cams


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def run(ctx, name, cams_all, W, H, cap, M, e, ks, reps):
    p = vb.render_params(W, H, cap, DEPTH, seed=1)
    rows = []
    for k in ks:
        cams = cams_all[:k]

        def batch():
            _, n, st = ctx.render_frames_adaptive_rgb8(cams, p, M, e)
            return st.ms_kernels, int(n.sum(dtype=np.uint64)), int(n.max()), st.variant

        def sequential():
            ms, used, top, variants = 0.0, 0, 0, set()
            for f, cam in enumerate(cams):
                q = vb.render_params(W, H, cap, DEPTH, seed=1 + f)
                _, n, st = ctx.render_adaptive_rgb8(cam, q, M, e)
                ms += st.ms_kernels
                used += int(n.sum(dtype=np.uint64))
                top = max(top, int(n.max()))
                variants.add(st.variant)
            return ms, used, top, sorted(variants)

        def fixed():
            _, st = ctx.render_frames_rgb8(cams, p)
            return st.ms_kernels, k * W * H * cap, cap, st.variant

        ways = {"batch": batch, "sequential": sequential, "fixed": fixed}
        for fn in ways.values():  # warm-up: modules, buffers of this K
            fn()
        wall = {w: [] for w in ways}
        kern = {w: [] for w in ways}
        info = {}
        for _ in range(reps):
            for w, fn in ways.items():
                t0 = time.perf_counter()
                ms, used, top, variant = fn()
                wall[w].append((time.perf_counter() - t0) * 1e3 / k)
                kern[w].append(ms / k)
                info[w] = {"samples_used": used / (k * W * H * cap), "passes": -(-top // M) if w != "fixed" else 1, "variant": variant}
        row = {"k": k, "max_error": e}
        for w in ways:
            row[w] = {"wall_ms_per_frame": summary(wall[w]), "kernel_ms_per_frame": summary(kern[w]), **info[w]}
        for w in ("sequential", "fixed"):
            row[f"batch_speedup_vs_{w}_wall"] = statistics.median(wall[w]) / statistics.median(wall["batch"])
            row[f"batch_speedup_vs_{w}_kernel"] = statistics.median(kern[w]) / statistics.median(kern["batch"])
        print(json.dumps({"workload": name, **row}), flush=True)
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="1,4,16")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    ks = [int(x) for x in a.ks.split(",")]
    ctx = vb.Context(0)
    dev = device_record()
    print(json.dumps({"device": dev}), flush=True)
    out = {"device": dev, "depth": DEPTH, "reps": a.reps, "workloads": []}
    for name, scene_name, W, H, cap, M, errors in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        scene = vb.Scene(scene_name)
        cams = cameras(scene, max(ks))
        ctx.upload(scene)
        for e in errors:
            out["workloads"].append({"workload": name, "scene": scene_name, "width": W, "height": H, "cap": cap, "pass_spp": M,
                                     "max_error": e, "rows": run(ctx, name, cams, W, H, cap, M, e, ks, a.reps)})
    out["device_after"] = device_record()
    ctx.close()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
