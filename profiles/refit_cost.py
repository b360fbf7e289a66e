"""Cost of the BVH8 refit (DESIGN.md 3.9) on one GPU, and what a refit does to the render.

    python profiles/refit_cost.py [--calls 30] [--warmup 5] [--out DIR]

1. Refit device time: dprt_refit_chunk_device on a terrain chunk of 1 M triangles (blob and vertices fit the 126 MB L2) and of
   12.5 M (they do not), moderate z-wave vertices resident on the device. A call synchronises its stream (the validation
   read-back and the end), so every call gets its own CUDA-event pair on the context's stream and the pairs are averaged.
2. Wall time (host clock around whole calls): dprt_refit_chunk with its host-to-device copies, and dprt_upload_chunk (host
   BVH8 rebuild + upload) of the same vertices, at both sizes.
3. Render after a refit: one context, 1 M triangles, 1920x1080, bounces 4, spc 4, one sample at a time: ms per sample and
   walked rays per second (dprt_stats.rays_walked) after a fresh upload, after the z-wave refit and after the permutation
   refit, and the instrumented traversal's BVH8 nodes visited and triangles tested per TraRay ray (dprt_enable_counters,
   a separate sample: the counting variant is slower).
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
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--samples", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    from refit_cases import deform, terrain, upload_desc

    name, power, clock_mhz = card()
    lines = [f"# {name}, power limit {power:.0f} W, max SM clock {clock_mhz:.0f} MHz"]
    for ntris in (1000000, 12500000):
        v, n, m = terrain(ntris)
        v2 = deform(v, "zwave")
        R = dprt.Renderer(dprt.make_config(16, 16, scene_size=1, proxy_mode=0))
        t0 = time.perf_counter()
        R.upload_chunk(0, upload_desc(v), v, n, m)
        upload_s = time.perf_counter() - t0
        dv, dn = R.device_alloc(v2.nbytes), R.device_alloc(n.nbytes)
        R.h2d(dv, v2); R.h2d(dn, n)
        nt = v2.shape[0]
        calls = args.calls if ntris <= 1000000 else max(5, args.calls // 3)
        res = {}
        for label, normals in (("verts_only", None), ("verts_and_normals", dn)):
            if normals is None:     # a chunk without normals: re-upload so that dprt_refit_chunk_device accepts normals = NULL
                R.upload_chunk(0, upload_desc(v), v, None, m)
            else:
                R.upload_chunk(0, upload_desc(v), v, n, m)
            for _ in range(args.warmup):
                R.refit_chunk_device(0, dv, normals, nt)
            tot = 0.0
            for _ in range(calls):
                R.timer_start()
                R.refit_chunk_device(0, dv, normals, nt)
                tot += R.timer_stop()
            res[label] = tot / calls
        host_calls = max(3, calls // 3)
        R.refit_chunk(0, v2, n)
        t0 = time.perf_counter()
        for _ in range(host_calls):
            R.refit_chunk(0, v2, n)
        host_ms = (time.perf_counter() - t0) * 1e3 / host_calls
        nodes, _ = R.chunk_bvh8(0)
        R.device_free(dv); R.device_free(dn)
        R.close()
        lines.append(json.dumps({"triangles": nt, "nodes": int(nodes.shape[0]), "refit_device_ms_verts_only": round(res["verts_only"], 4),
                                 "refit_device_ms_with_normals": round(res["verts_and_normals"], 4),
                                 "refit_host_variant_wall_ms": round(host_ms, 3), "upload_chunk_wall_ms": round(upload_s * 1e3, 1),
                                 "blob_bytes": int(nodes.shape[0]) * 80 + nt * 48, "verts_bytes": nt * 36}))
        del v, n, m, v2

    w, h = 1920, 1080
    v, n, m = terrain(1000000)
    cfg = dprt.make_config(w, h, spp=1, bounces=4, spc=4, scene_size=1, proxy_mode=0)
    R = dprt.Renderer(cfg)
    R.upload_chunk(0, upload_desc(v), v, n, m)
    R.set_materials(dprt.scene.make_materials(16)); R.set_lights(dprt.scene.make_lights()); R.set_camera(dprt.scene.default_camera(w, h))
    for label, verts in (("fresh_upload", v), ("zwave_refit", deform(v, "zwave")), ("permutation_refit", deform(v, "permute"))):
        if label != "fresh_upload":
            R.refit_chunk(0, verts, n)
        R.reset_frame()
        for s in range(2):
            R.run_sample(s)
        R.synchronize()
        R.reset_stats()
        t0 = time.perf_counter()
        for s in range(args.samples):
            R.run_sample(2 + s)
        R.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.samples
        st = R.stats()
        R.enable_counters(True); R.reset_stats()
        R.run_sample(100)
        R.synchronize()
        c = R.counters()["traverse"]
        walked = R.stats()["walked_traverse"]
        R.enable_counters(False)
        lines.append(json.dumps({"render": label, "triangles": 1000000, "width": w, "height": h, "bounces": 4, "spc": 4,
                                 "ms_per_sample": round(ms, 3), "walked_mrays_per_s": round(st["rays_walked"] / args.samples / ms / 1e3, 1),
                                 "traray_nodes_per_ray": round(c[0] / max(walked, 1), 2), "traray_tris_per_ray": round(c[1] / max(walked, 1), 2)}))
    R.close()
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_refit_cost.txt"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
