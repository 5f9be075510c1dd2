"""Per-frame time of a turntable rendered in batches (vk_render_frames_rgb8, K cameras per launch) against the same K
frames rendered one vk_render_rgb8 call each -- the two alternated in the same run, several repetitions, median and
spread reported.  The device name, its power limit and SM clocks are read in the same run and stored with the numbers.

    python scripts/turntable_bench.py [--ks 1,2,4,8,16] [--reps 7] [--out FILE.json]

Workloads: config 1's turntable (random_spheres_demo 400x225, 16 spp, depth 50, its first K cameras), bowser_demo
(400 wide, 16 spp, depth 50) and cornell_box (600x600, 64 spp, depth 100; one camera, so frame f repeats it with
seed + f).  Times are host wall clock around calls that end in a stream synchronise (what the frame program pays per
frame, copy-back included); `kernel_ms` is the CUDA-event kernel time the calls report."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import vecchio_b200 as vb  # noqa: E402

WORKLOADS = [  # name, scene, width, spp, depth
    ("config1_random_spheres", "random_spheres_demo", 400, 16, 50),
    ("bowser", "bowser_demo", 400, 16, 50),
    ("cornell", "cornell_box", 600, 64, 100),
]


def device_record():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    fields = [x.strip() for x in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(q.split(","), fields)) if len(fields) == 4 else {"error": r.stderr.strip() or "nvidia-smi failed"}


def cameras(scene, k):
    cams = []
    while len(cams) < k:
        c = scene.next_camera()
        if c is None:
            break
        cams.append(c)
    while len(cams) < k:  # a fixed camera: the same view, frame f with seed + f
        cams.append(cams[0])
    return cams


def sequential(ctx, cams, width, height, spp, depth, seed):
    ms = 0.0
    t0 = time.perf_counter()
    for f, cam in enumerate(cams):
        _, st = ctx.render_rgb8(cam, vb.render_params(width, height, spp, depth, seed=seed + f))
        ms += st.ms_kernels
    return (time.perf_counter() - t0) * 1e3, ms, st.variant


def batched(ctx, cams, width, height, spp, depth, seed):
    t0 = time.perf_counter()
    _, st = ctx.render_frames_rgb8(cams, vb.render_params(width, height, spp, depth, seed=seed))
    return (time.perf_counter() - t0) * 1e3, st.ms_kernels, st.variant


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="1,2,4,8,16")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ks = [int(k) for k in args.ks.split(",")]
    ctx = vb.Context(0)
    record = {"device": ctx.device_info(), "smi_before": device_record(), "reps": args.reps, "results": []}
    for label, name, width, spp, depth in WORKLOADS:
        scene = vb.Scene(name, seed=1)
        height = scene.height_for(width)
        cams = cameras(scene, max(ks))
        ctx.upload(scene)
        for k in ks:  # warm-up of every shape the timed runs use
            sequential(ctx, cams[:k], width, height, spp, depth, 1)
            batched(ctx, cams[:k], width, height, spp, depth, 1)
        for k in ks:
            seq, bat, seq_k, bat_k = [], [], [], []
            variant = {}
            for rep in range(args.reps):  # alternate which of the two goes first
                runs = [("seq", sequential), ("batch", batched)]
                for mode, fn in (runs if rep % 2 == 0 else runs[::-1]):
                    wall, kern, var = fn(ctx, cams[:k], width, height, spp, depth, 1)
                    (seq if mode == "seq" else bat).append(wall / k)
                    (seq_k if mode == "seq" else bat_k).append(kern / k)
                    variant[mode] = var
            row = {"workload": label, "scene": name, "width": width, "height": height, "spp": spp, "depth": depth, "k": k,
                   "paths_per_launch": {"seq": width * height * spp, "batch": width * height * spp * k},
                   "variant": {m: {1: "megakernel", 4: "warpq", 5: "stepq"}.get(v, str(v)) for m, v in variant.items()},
                   "ms_per_frame_wall": {"seq": summary(seq), "batch": summary(bat)},
                   "ms_per_frame_kernel": {"seq": summary(seq_k), "batch": summary(bat_k)}}
            row["speedup_wall"] = row["ms_per_frame_wall"]["seq"]["median"] / row["ms_per_frame_wall"]["batch"]["median"]
            record["results"].append(row)
            w = row["ms_per_frame_wall"]
            print(f"{label:24s} K={k:2d}  seq {w['seq']['median']:7.3f} ms/frame [{w['seq']['min']:.3f}, {w['seq']['max']:.3f}] "
                  f"({row['variant']['seq']})  batch {w['batch']['median']:7.3f} [{w['batch']['min']:.3f}, {w['batch']['max']:.3f}] "
                  f"({row['variant']['batch']})  x{row['speedup_wall']:.3f}", flush=True)
        scene.close()
    record["smi_after"] = device_record()
    ctx.close()
    text = json.dumps(record, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({"device": record["device"], "smi": record["smi_before"]}))


if __name__ == "__main__":
    main()
