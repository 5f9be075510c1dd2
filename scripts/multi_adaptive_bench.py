#!/usr/bin/env python3
"""Adaptive sampling split into shards of pixels (vk_adaptive_begin_shard, vk_multi_*adaptive*); writes
profiles/multi_adaptive_bench_b200.json.

    python scripts/multi_adaptive_bench.py [--reps 3] [--base-tree DIR] [--out FILE]

Measured in this one run:
  - balance on one GPU: for N = 2, 4, 8, every shard of N refined once to the one-shot target, one after another on device 0,
    against the unsharded session (N = 1).  Per shard its kernel ms and paths; per N the slowest shard, the mean, their
    ratio (the static balance the ownership rule achieves: the slowest shard sets a multi-GPU refine's time) and the
    unsharded kernel ms over the slowest shard's (the speed-up N devices could reach at best, before the gather).
    Workloads: Cornell 600x600, cap 1000, pass 64, E = 4; the random_spheres turntable K = 16 at 400x225, cap 256, pass
    32, E = 1; the final scene 800x800, cap 1024, pass 64, E = 1.
  - several GPUs, when the machine has them: wall time of vk_multi_render_adaptive_rgb8 (or the frames call) over the first
    N devices against vk_render_adaptive_rgb8 on device 0, for N = 2, 4, 8; "not measured" otherwise.
  - no regression (with --base-tree, a built checkout of the parent): adaptive_refine_bench.py's alternated one-shot
    adaptive calls and bench.py's default configuration, parent against this tree.
The device name, power limit and SM clocks are read in the same run and stored with the numbers."""
import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, ROOT)

DEPTH = 50
# (name, scene, W, H, cap, pass_spp, max_error, frames)
WORKLOADS = [("cornell_600", "cornell_box", 600, 600, 1000, 64, 4.0, 1),
             ("random_spheres_turntable_k16", "random_spheres_demo", 400, 225, 256, 32, 1.0, 16),
             ("final_scene_800", "final_scene", 800, 800, 1024, 64, 1.0, 1)]
SHARDS = (2, 4, 8)


def setup(vb, scene_name, W, H, cap, k):
    from adaptive_refine_bench import turntable
    scene = vb.Scene(scene_name)
    cams = turntable(scene, k)
    return scene, (cams[0] if k == 1 else cams), vb.render_params(W, H, cap, DEPTH, seed=1)


def balance(vb, ctx, reps):
    rows = []
    for name, scene_name, W, H, cap, M, E, k in WORKLOADS:
        scene, cams, p = setup(vb, scene_name, W, H, cap, k)
        ctx.upload(scene)

        def refine_ms(shard):
            s = ctx.adaptive_session(cams, p, M, shard=shard)
            st = s.refine(E)
            s.close()
            return st.ms_kernels, int(st.paths)

        refine_ms(None)  # warm-up: modules, buffers
        whole = [refine_ms(None) for _ in range(reps)]
        row = {"workload": name, "scene": scene_name, "width": W, "height": H, "frames": k, "cap": cap, "pass_spp": M, "max_error": E,
               "unsharded_kernel_ms": statistics.median(w[0] for w in whole), "paths": whole[0][1], "shards": []}
        for n in SHARDS:
            per = []
            for sh in range(n):
                t = [refine_ms((sh, n)) for _ in range(reps)]
                per.append({"shard": sh, "kernel_ms": statistics.median(x[0] for x in t), "paths": t[0][1]})
            ms = [x["kernel_ms"] for x in per]
            assert sum(x["paths"] for x in per) == row["paths"], "the shards' paths do not add up to the unsharded session's"
            r = {"n": n, "per_shard": per, "max_kernel_ms": max(ms), "mean_kernel_ms": statistics.mean(ms),
                 "max_over_mean": max(ms) / statistics.mean(ms), "paths_max_over_mean": max(x["paths"] for x in per) / (row["paths"] / n),
                 "unsharded_over_slowest_shard": row["unsharded_kernel_ms"] / max(ms)}
            row["shards"].append(r)
            print(json.dumps({"workload": name, **{k_: v for k_, v in r.items() if k_ != "per_shard"}}), flush=True)
        rows.append(row)
    return rows


def multi_gpu(vb, ab, reps):
    from conftest import cuda_device_count
    n_dev = cuda_device_count()
    if n_dev < 2:
        return f"not measured: this machine has {n_dev} GPU"
    ctx = vb.Context(0)
    rows = []
    for name, scene_name, W, H, cap, M, E, k in WORKLOADS:
        scene, cams, p = setup(vb, scene_name, W, H, cap, k)
        ctx.upload(scene)
        one = (lambda: ctx.render_adaptive_rgb8(cams, p, M, E)) if k == 1 else (lambda: ctx.render_frames_adaptive_rgb8(cams, p, M, E))
        one()
        row = {"workload": name, "one_gpu_wall_ms": statistics.median(ab.timed(one)[0] for _ in range(reps)), "multi": []}
        ref = one()
        for n in SHARDS:
            if n > n_dev:
                row["multi"].append({"n": n, "wall_ms": "not measured: too few GPUs"})
                continue
            m = vb.MultiContext(list(range(n)))
            m.upload(scene)
            call = (lambda: m.render_adaptive_rgb8(cams, p, M, E)) if k == 1 else (lambda: m.render_frames_adaptive_rgb8(cams, p, M, E))
            got = call()
            same = bool(np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]))
            walls = [ab.timed(call)[0] for _ in range(reps)]
            m.close()
            w = statistics.median(walls)
            row["multi"].append({"n": n, "wall_ms": w, "speedup": row["one_gpu_wall_ms"] / w, "same_image_and_counts": same})
            print(json.dumps({"workload": name, **row["multi"][-1]}), flush=True)
        rows.append(row)
    ctx.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--base-tree", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import adaptive_bench as ab
    import vecchio_b200 as vb
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    dev = ab.device_record()
    print(json.dumps({"device": dev}), flush=True)
    out = {"device": dev, "reps": a.reps, "depth": DEPTH}
    ctx = vb.Context(0)
    out["balance_one_gpu"] = balance(vb, ctx, a.reps)
    ctx.close()
    out["multi_gpu"] = multi_gpu(vb, ab, a.reps)
    if a.base_tree:
        from adaptive_refine_bench import regression
        out["regression"] = {"base_tree": "the parent commit, built the same way", "reps": a.reps,
                             "workloads": regression(a.base_tree, a.reps)}
    out["device_after"] = ab.device_record()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
