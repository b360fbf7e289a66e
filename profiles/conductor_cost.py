"""Cost of the rough conductor (bsdfType 2, DESIGN.md 3.12) on the benchmark workload: bench.py's one-GPU scene (1920x1080,
1 M triangles, 4 bounces) with its 16 materials all Lambertian, all conductors at roughness 0.3, and mixed (the odd materials
conductors at 0.3), alternating in one process.

    python profiles/conductor_cost.py [--steps 40] [--warmup 4] [--rounds 3] [--out DIR]

Each window: reset the frame, warm up, then time `steps` samples between CUDA events (whole sample), and in a second window
of the same length the shade stage alone (dprt_stage_profile, DPRT_STAGE_SHADE: shade_post_kernel, plus the MainRay trace
where one is launched) and the records it shaded, since the materials change where paths go (a mirror sends more of them to
the sky, where they end).
The device name and power limit are read in the same process. Prints one JSON line per window and a summary line; --out
also writes them to DIR/conductor_cost.jsonl. profiles/plastic_cost.py runs the same windows for the glossy plastic.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def main(bsdf=2, name="conductor"):
    """The three material tables: all Lambertian, all `bsdf` (named `name`) at roughness 0.3, every other one `bsdf`."""
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    fw, fh = bench.frame_for(1)
    cfg = dprt.make_config(fw, fh, spp=1, bounces=4, scene_size=1)
    chunks, mats, lights = bench.build_world_scene(dprt, 1, 1000000)
    R = dprt.Renderer(cfg)
    c = chunks[0]
    R.upload_chunk(c.index, c.desc(False), c.verts, c.normals, c.mats)
    R.set_lights(lights); R.set_camera(dprt.scene.default_camera(fw, fh))
    R.set_material_roughness(np.full(len(mats), 0.3, np.float32))
    tables = {}
    for mode in ("lambert", name, "mixed"):
        m = np.array(mats, copy=True)
        if mode == name:
            m["bsdfType"][:] = bsdf
        elif mode == "mixed":
            m["bsdfType"][1::2] = bsdf
        tables[mode] = m
    lines, first = [], 0
    info = device_info()
    for rnd in range(args.rounds):
        for mode, m in tables.items():
            R.set_materials(m)
            line = {"round": rnd, "mode": mode, "samples": args.steps}
            for profile in (False, True):
                R.stage_profile(profile)
                R.reset_frame()
                for s in range(args.warmup):
                    R.run_sample(first + s)
                first += args.warmup
                R.synchronize()
                R.reset_stats()
                R.timer_start()
                for s in range(args.steps):
                    R.run_sample(first + s)
                first += args.steps
                ms = R.timer_stop()
                if profile:
                    line["shade_ms_per_sample"] = R.stage_times()["shade"][0] / args.steps
                    line["shade_rays_per_sample"] = R.stats()["rays_shade"] / args.steps
                    line["shade_ns_per_ray"] = 1e6 * line["shade_ms_per_sample"] / line["shade_rays_per_sample"]
                else:
                    line["ms_per_sample"] = ms / args.steps
                    line["Mrays_per_s"] = R.stats()["rays_walked"] / (ms * 1e-3) / 1e6
            R.stage_profile(False)
            print(json.dumps(line), flush=True)
            lines.append(line)
    summary = {"summary": True, "device": info, "frame": [fw, fh]}
    for mode in tables:
        summary[mode] = {k: statistics.median(ln[k] for ln in lines if ln["mode"] == mode)
                         for k in ("ms_per_sample", "shade_ms_per_sample", "shade_rays_per_sample", "shade_ns_per_ray", "Mrays_per_s")}
    print(json.dumps(summary), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"{name}_cost.jsonl"), "w") as f:
            for ln in lines + [summary]:
                f.write(json.dumps(ln) + "\n")
    R.close()


if __name__ == "__main__":
    main()
