#!/usr/bin/env python3
"""Adaptive render sessions (vk_adaptive_*) on one GPU; writes profiles/adaptive_refine_bench_b200.json.

    python scripts/adaptive_refine_bench.py [--reps 3] [--base-tree DIR] [--out FILE]

Three measurements, each in this one run:
  - progressive against one-shot: a session tightened step by step, with a read after each step, against one one-shot call
    at the last target (Cornell 600x600, cap 1000, pass 64: E 8 -> 4 -> 2; random_spheres turntable K = 16 at 400x225,
    cap 256, pass 32: E 4 -> 1).  Wall and kernel ms per step, the levels each refine launched (its passes), medians of
    alternated repetitions.
  - the floor on the final scene (800x800, cap 1024, pass 64, E = 1, min_spp 0 / 256 / 512): RMSE (8-bit units) and samples
    used against an independent 4x reference, and the fixed spp at equal RMSE (scripts/adaptive_bench.py's helpers).
  - no regression: the one-shot adaptive calls of scripts/adaptive_bench.py and scripts/adaptive_turntable_bench.py at one
    target each, and bench.py's default configuration (config 2), timed in child processes that alternate between
    --base-tree (a built checkout of the parent) and this tree.
The device name, its power limit and SM clocks are read in the same run and stored with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, ROOT)

DEPTH = 50
# the one-shot workloads compared against the parent: (name, scene, W, H, cap, pass_spp, max_error, frames)
ONESHOT = [("cornell_600", "cornell_box", 600, 600, 1000, 64, 2.0, 1), ("final_scene_800", "final_scene", 800, 800, 1024, 64, 2.0, 1),
           ("random_spheres_400x225", "random_spheres_demo", 400, 225, 256, 32, 2.0, 1),
           ("random_spheres_turntable_k16", "random_spheres_demo", 400, 225, 256, 32, 1.0, 16)]


def turntable(scene, k):
    cams = []
    while len(cams) < k:
        c = scene.next_camera()
        if c is None:
            break
        cams.append(c)
    return cams


def progressive(vb, ctx, timed, name, scene_name, W, H, cap, M, errors, k, reps):
    scene = vb.Scene(scene_name)
    cams = turntable(scene, k)
    ctx.upload(scene)
    p = vb.render_params(W, H, cap, DEPTH, seed=1)
    one = (lambda: ctx.render_adaptive(cams[0], p, M, errors[-1])) if k == 1 else (lambda: ctx.render_frames_adaptive(cams, p, M, errors[-1]))
    one()  # warm-up: modules, buffers
    steps, oneshot = [[] for _ in errors], []
    for _ in range(reps):  # alternated: the whole progressive sequence, then the one-shot call
        s = ctx.adaptive_session(cams[0] if k == 1 else cams, p, M)
        n0 = s.export()[2]
        for i, e in enumerate(errors):
            w, st = timed(lambda: (s.refine(e), s.read_rgb8())[0])
            n = s.export()[2]
            # the levels this refine launched: every grid level some pixel rendered through (one launch per non-empty level)
            levels = sum(bool(np.any((n0 <= L) & (n > L))) for L in range(0, cap, M))
            steps[i].append({"wall_ms": w, "kernel_ms": st.ms_kernels, "paths": int(st.paths), "launches": int(st.launches),
                             "levels": levels})
            n0 = n
        final = s.export()
        s.close()
        w, (img, n1, st1) = timed(one)
        oneshot.append({"wall_ms": w, "kernel_ms": st1.ms_kernels, "paths": int(st1.paths), "launches": int(st1.launches)})
        assert np.array_equal(final[2].reshape(n1.shape), n1), "the progressive state differs from the one-shot call"
    med = lambda rows, f: statistics.median(r[f] for r in rows)  # noqa: E731
    out_steps = []
    for e, rows in zip(errors, steps):
        out_steps.append({"max_error": e, "wall_ms": med(rows, "wall_ms"), "kernel_ms": med(rows, "kernel_ms"),
                          "paths": rows[0]["paths"], "launches": rows[0]["launches"], "levels": rows[0]["levels"]})
    row = {"workload": name, "scene": scene_name, "width": W, "height": H, "frames": k, "cap": cap, "pass_spp": M,
           "targets": errors, "steps": out_steps,
           "sum_of_steps_wall_ms": sum(r["wall_ms"] for r in out_steps),
           "sum_of_steps_kernel_ms": sum(r["kernel_ms"] for r in out_steps),
           "oneshot": {"max_error": errors[-1], "wall_ms": med(oneshot, "wall_ms"), "kernel_ms": med(oneshot, "kernel_ms"),
                       "paths": oneshot[0]["paths"], "launches": oneshot[0]["launches"]},
           "same_counts_as_oneshot": True}
    print(json.dumps(row), flush=True)
    return row


def floor(vb, ab, ctx, reps, floors=(0, 256, 512)):
    W = H = 800
    cap, M, E = 1024, 64, 1.0
    scene = vb.Scene("final_scene")
    cam = scene.next_camera()
    ctx.upload(scene)
    p = lambda spp, seed=1: vb.render_params(W, H, spp, DEPTH, seed=seed)  # noqa: E731
    ctx.render(cam, p(M))
    ref, _, _ = ctx.render(cam, p(4 * cap, seed=987654321))
    ladder = []
    for spp in (128, 256, 512, 1024):
        rgb, _, st = ctx.render(cam, p(spp))
        ladder.append({"spp": spp, "kernel_ms": st.ms_kernels, "rmse8": ab.rmse8(rgb, ref)})
    rows = []
    for f in floors:
        kerns, walls = [], []
        for _ in range(reps):
            s = ctx.adaptive_session(cam, p(cap), M)
            w, st = ab.timed(lambda: s.refine(E, min_spp=f))
            rgb, n, _ = s.read()
            s.close()
            kerns.append(st.ms_kernels)
            walls.append(w)
        err = ab.rmse8(rgb, ref)
        eq = None
        for a, b in zip(ladder, ladder[1:]):
            if a["rmse8"] >= err >= b["rmse8"]:
                t = (np.log(a["rmse8"]) - np.log(err)) / max(np.log(a["rmse8"]) - np.log(b["rmse8"]), 1e-12)
                spp_eq = float(np.exp(np.log(a["spp"]) + t * (np.log(b["spp"]) - np.log(a["spp"]))))
                eq = {"spp": spp_eq, "kernel_ms": a["kernel_ms"] + t * (b["kernel_ms"] - a["kernel_ms"])}
        rows.append({"min_spp": f, "max_error": E, "rmse8": err, "samples_used": float(n.sum(dtype=np.float64) / (W * H * cap)),
                     "kernel_ms": statistics.median(kerns), "wall_ms": statistics.median(walls),
                     "pixels_at_cap": int((n == cap).sum()), "fixed_at_equal_rmse": eq if eq else "outside the ladder",
                     "x_fixed_at_equal_rmse_kernel": (eq["kernel_ms"] / statistics.median(kerns)) if eq else None})
        print(json.dumps({"workload": "final_scene_800_floor", **rows[-1]}), flush=True)
    return {"workload": "final_scene_800_floor", "width": W, "height": H, "cap": cap, "pass_spp": M, "depth": DEPTH,
            "reference_spp": 4 * cap, "fixed_ladder": ladder, "rows": rows}


def oneshot_child():
    """One timed call of every ONESHOT workload with the package of the tree this script was started from (a child of
    --base-tree or of this tree); prints one JSON line."""
    import time
    import vecchio_b200 as vb
    ctx = vb.Context(0)
    out = {}
    for name, scene_name, W, H, cap, M, E, k in ONESHOT:
        scene = vb.Scene(scene_name)
        cams = turntable(scene, k)
        ctx.upload(scene)
        p = vb.render_params(W, H, cap, DEPTH, seed=1)
        call = (lambda: ctx.render_adaptive(cams[0], p, M, E)) if k == 1 else (lambda: ctx.render_frames_adaptive(cams, p, M, E))
        call()
        t0 = time.perf_counter()
        _, n, st = call()
        out[name] = {"wall_ms": (time.perf_counter() - t0) * 1e3, "kernel_ms": st.ms_kernels, "paths": int(st.paths),
                     "counts_sum": int(n.sum(dtype=np.int64))}
    ctx.close()
    print(json.dumps(out), flush=True)


def regression(base_tree, reps):
    runs = {"base": [], "head": []}
    bench = {"base": [], "head": []}  # bench.py's default configuration (config 2), ms per step
    me = os.path.abspath(__file__)
    for _ in range(reps):
        for tag, tree in (("base", os.path.abspath(base_tree)), ("head", ROOT)):
            r = subprocess.run([sys.executable, me, "--oneshot-child", "--tree", tree], capture_output=True, text=True)
            if r.returncode != 0:
                return {"error": r.stderr[-2000:]}
            runs[tag].append(json.loads(r.stdout.strip().splitlines()[-1]))
            r = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", "5", "--warmup", "2",
                                "--no-other-configs"], cwd=tree, capture_output=True, text=True)
            if r.returncode != 0:
                return {"error": r.stderr[-2000:]}
            bench[tag].append(json.loads(r.stdout.strip().splitlines()[-1])["ms_per_step"])
    out = {"bench_py_config2_ms_per_step": {"base": bench["base"], "head": bench["head"],
                                            "base_median": statistics.median(bench["base"]),
                                            "head_median": statistics.median(bench["head"])}}
    print(json.dumps({"regression": "bench.py", **out["bench_py_config2_ms_per_step"]}), flush=True)
    for name, *_ in ONESHOT:
        b = [x[name] for x in runs["base"]]
        h = [x[name] for x in runs["head"]]
        out[name] = {"base_kernel_ms": statistics.median(x["kernel_ms"] for x in b), "head_kernel_ms": statistics.median(x["kernel_ms"] for x in h),
                     "base_wall_ms": statistics.median(x["wall_ms"] for x in b), "head_wall_ms": statistics.median(x["wall_ms"] for x in h),
                     "same_paths_and_counts": all(x["paths"] == b[0]["paths"] and x["counts_sum"] == b[0]["counts_sum"] for x in b + h)}
        print(json.dumps({"regression": name, **out[name]}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--base-tree", default="")
    ap.add_argument("--out", default="")
    ap.add_argument("--oneshot-child", action="store_true")
    ap.add_argument("--tree", default="")
    a = ap.parse_args()
    if a.oneshot_child:
        sys.path.insert(0, a.tree)
        for m in [m for m in sys.modules if m.startswith("vecchio_b200")]:
            del sys.modules[m]
        return oneshot_child()
    import adaptive_bench as ab
    import vecchio_b200 as vb
    dev = ab.device_record()
    print(json.dumps({"device": dev}), flush=True)
    out = {"device": dev}
    ctx = vb.Context(0)
    out["progressive"] = [progressive(vb, ctx, ab.timed, "cornell_600", "cornell_box", 600, 600, 1000, 64, [8.0, 4.0, 2.0], 1, a.reps),
                          progressive(vb, ctx, ab.timed, "random_spheres_turntable_k16", "random_spheres_demo", 400, 225, 256, 32,
                                      [4.0, 1.0], 16, a.reps)]
    out["floor"] = floor(vb, ab, ctx, a.reps)
    ctx.close()
    if a.base_tree:
        out["regression"] = {"base_tree": "the parent commit, built the same way", "reps": a.reps,
                             "workloads": regression(a.base_tree, a.reps)}
    out["device_after"] = ab.device_record()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
