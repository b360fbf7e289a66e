"""Cost of the GPU BVH8 build (DESIGN.md 3.10) on one GPU, and how its tree renders against the host builder's.

    python profiles/gpu_build_cost.py [--calls 10] [--warmup 2] [--samples 6] [--out DIR]

1. Build time: dprt_build_chunk_device on terrain chunks of 1 M and 12.5 M triangles and on the garden (flattened, with normals,
   texture coordinates and materials resident on the device): one CUDA-event pair on the context's stream per call (a call
   synchronises its stream several times: the validation read-back and one count per clustering iteration and per level),
   averaged after warm-up. Wall time (host clock around whole calls) of dprt_build_chunk with its host-to-device copies and of
   dprt_upload_chunk (host build + upload) of the same arrays, in the same run.
2. Render: one context, the 1 M-triangle chunk, 1920x1080, bounces 4, spc 4, one sample at a time: ms per sample and the
   instrumented traversal's BVH8 nodes visited and triangles tested per TraRay ray (dprt_enable_counters, a separate sample:
   the counting variant is slower), for the host-built chunk, the GPU-built chunk and the GPU build of the permuted vertices a
   permutation refit leaves behind (the same triangles under other ids).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return name, float(power), float(clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--samples", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    from refit_cases import garden_flat, terrain, upload_desc

    name, power, clock_mhz = card()
    lines = [f"# {name}, power limit {power:.0f} W, max SM clock {clock_mhz:.0f} MHz"]
    inputs = [("terrain_1M", lambda: (*terrain(1000000), None, None)), ("terrain_12.5M", lambda: (*terrain(12500000), None, None))]
    g = garden_flat()
    inputs.append(("garden", lambda: (g[0], g[1], g[3], g[2], g[4]["objects"][0].desc(False))))
    for label, make in inputs:
        v, n, m, uv, desc = make()
        desc = desc if desc is not None else upload_desc(v)
        nt = v.shape[0]
        R = dprt.Renderer(dprt.make_config(16, 16, scene_size=1, proxy_mode=0))
        dev = [None if a is None else R.device_alloc(a.nbytes) for a in (v, n, uv, m)]
        for d, a in zip(dev, (v, n, uv, m)):
            if d is not None:
                R.h2d(d, np.ascontiguousarray(a))
        calls = args.calls if nt <= 1000000 else max(3, args.calls // 3)
        for _ in range(args.warmup):
            R.build_chunk_device(0, desc, *dev, nt)
        tot = 0.0
        for _ in range(calls):
            R.timer_start()
            R.build_chunk_device(0, desc, *dev, nt)
            tot += R.timer_stop()
        nodes, _ = R.chunk_bvh8(0)
        t0 = time.perf_counter()
        for _ in range(calls):
            R.build_chunk(0, desc, v, n, uv, m)
        build_wall = (time.perf_counter() - t0) * 1e3 / calls
        up_calls = max(1, calls // 3)
        t0 = time.perf_counter()
        for _ in range(up_calls):
            R.upload_chunk_uv(0, desc, v, n, uv, m)
        upload_wall = (time.perf_counter() - t0) * 1e3 / up_calls
        host_nodes, _ = R.chunk_bvh8(0)
        for d in dev:
            if d is not None:
                R.device_free(d)
        R.close()
        lines.append(json.dumps({"input": label, "triangles": nt, "gpu_nodes": int(nodes.shape[0]), "host_nodes": int(host_nodes.shape[0]),
                                 "build_chunk_device_ms": round(tot / calls, 3), "build_chunk_wall_ms": round(build_wall, 2),
                                 "upload_chunk_wall_ms": round(upload_wall, 1)}))
        print(lines[-1], flush=True)
        del v, n, m, uv

    w, h = 1920, 1080
    v, n, m = terrain(1000000)
    perm = np.random.default_rng(1).permutation(v.shape[0])
    cfg = dprt.make_config(w, h, spp=1, bounces=4, spc=4, scene_size=1, proxy_mode=0)
    R = dprt.Renderer(cfg)
    R.set_materials(dprt.scene.make_materials(16)); R.set_lights(dprt.scene.make_lights()); R.set_camera(dprt.scene.default_camera(w, h))
    runs = (("host_upload", lambda: R.upload_chunk(0, upload_desc(v), v, n, m)),
            ("gpu_build", lambda: R.build_chunk(0, upload_desc(v), v, n, None, m)),
            ("gpu_build_of_permuted_vertices", lambda: R.build_chunk(0, upload_desc(v), v[perm], n[perm], None, m[perm])))
    for label, make in runs:
        make()
        R.reset_frame()
        for s in range(2):
            R.run_sample(s)
        R.synchronize()
        t0 = time.perf_counter()
        for s in range(args.samples):
            R.run_sample(2 + s)
        R.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.samples
        R.enable_counters(True); R.reset_stats()
        R.run_sample(100)
        R.synchronize()
        c = R.counters()["traverse"]
        walked = R.stats()["walked_traverse"]
        R.enable_counters(False)
        lines.append(json.dumps({"render": label, "triangles": 1000000, "width": w, "height": h, "bounces": 4, "spc": 4,
                                 "ms_per_sample": round(ms, 3), "traray_nodes_per_ray": round(c[0] / max(walked, 1), 3),
                                 "traray_tris_per_ray": round(c[1] / max(walked, 1), 3)}))
        print(lines[-1], flush=True)
    R.close()
    text = "\n".join(lines)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_gpu_build_cost.txt"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
