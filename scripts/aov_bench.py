"""Cost of the denoiser feature buffers (vk_render_aov) next to the render of the same frame.

    python scripts/aov_bench.py [--reps 9] [--out FILE.json]

Workloads: cornell_box 600x600 and final_scene 800x800, each with aov_spp 16 and 64, against vk_render of the same
camera and size at the spp bench.py renders (cornell 1000; final_scene the 64 of bench.py's short run), depth 100.  The
calls alternate, each is repeated --reps times after a warm-up, and the median and spread are reported: `kernel_ms` is the
CUDA-event kernel time the call reports, `total_ms` its time with the copy back of the planes (or the image).  The device
name, power limit and SM clocks are read in the same run and stored with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import vecchio_b200 as vb  # noqa: E402

WORKLOADS = [("cornell", "cornell_box", 600, 1000), ("final_scene", "final_scene", 800, 64)]  # label, scene, width, render spp
AOV_SPP = (16, 64)


def device_record():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    fields = [x.strip() for x in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(q.split(","), fields)) if len(fields) == 4 else {"error": r.stderr.strip() or "nvidia-smi failed"}


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = vb.Context(0)
    record = {"device": ctx.device_info(), "smi_before": device_record(), "reps": args.reps, "results": []}
    for label, name, width, spp in WORKLOADS:
        scene = vb.Scene(name, seed=1)
        cam = scene.next_camera()
        height = scene.height_for(width)
        ctx.upload(scene)
        p = vb.render_params(width, height, spp, 100, seed=1)
        runs = {"render": ([], [])}
        runs.update({f"aov_{n}": ([], []) for n in AOV_SPP})
        for rep in range(args.reps + 1):  # rep 0 warms every call up
            _, _, st = ctx.render(cam, p)
            if rep:
                runs["render"][0].append(st.ms_kernels)
                runs["render"][1].append(st.ms_total)
            for n in AOV_SPP:
                _, st = ctx.render_aov(cam, p, n)
                assert st.rays == width * height * n
                if rep:
                    runs[f"aov_{n}"][0].append(st.ms_kernels)
                    runs[f"aov_{n}"][1].append(st.ms_total)
        res = {"workload": f"{name} {width}x{height}", "render_spp": spp, "max_depth": 100}
        for k, (kern, tot) in runs.items():
            res[k] = {"kernel_ms": summary(kern), "total_ms": summary(tot)}
        for n in AOV_SPP:
            rays = width * height * n
            res[f"aov_{n}"]["camera_rays"] = rays
            res[f"aov_{n}"]["grays_per_s"] = rays / (res[f"aov_{n}"]["kernel_ms"]["median"] * 1e-3) * 1e-9
            res[f"aov_{n}"]["share_of_render_kernel"] = res[f"aov_{n}"]["kernel_ms"]["median"] / res["render"]["kernel_ms"]["median"]
        record["results"].append(res)
        print(json.dumps(res), flush=True)
    record["smi_after"] = device_record()
    ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(record, f, indent=1)


if __name__ == "__main__":
    main()
