"""Cost of building and moving instanced scene objects on the GPU (DESIGN.md 3.11) on one GPU, against the host path.

    python profiles/instanced_build_cost.py [--calls 5] [--warmup 1] [--samples 6] [--out DIR]

Inputs: the garden's scene object at its test size (4 810 flattened triangles) and the 10.9 M-triangle object of 2 001
instances of tests/instance_cases.py (case_10m). Every figure is a host clock around whole calls, each of which ends in a
device synchronise, averaged after warm-up:
1. Build: dprt_upload_instanced_chunk (host flatten, host BVH8 build, upload) against dprt_build_instanced_chunk (indexed
   arrays and instance table copied, device flatten, GPU build).
2. Move: host flatten of the moved instances plus dprt_refit_chunk against dprt_update_instances; a third of the instances
   turned and shrunk, alternating with the original placement.
3. Render: ms per 1920x1080 sample (bounces 4, spc 4) of the host-uploaded and of the GPU-built chunk.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return name, float(power), float(clock)


def wall_ms(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    return (time.perf_counter() - t0) * 1e3 / calls


def sample_ms(dprt, R, samples):
    R.reset_frame()
    for s in range(2):
        R.run_sample(s)
    R.synchronize()
    t0 = time.perf_counter()
    for s in range(samples):
        R.run_sample(2 + s)
    R.synchronize()
    return (time.perf_counter() - t0) * 1e3 / samples


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--samples", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    from instance_cases import CASES, case_10m, moved, object_desc

    name, power, clock_mhz = card()
    lines = [f"# {name}, power limit {power:.0f} W, max SM clock {clock_mhz:.0f} MHz"]
    w, h = 1920, 1080
    for label, make in (("garden", CASES["garden"]), ("instances_10M", case_10m)):
        meshes, inst = make()
        m1 = moved(inst)
        desc = object_desc(meshes, inst, m1)
        cfg = dprt.make_config(w, h, spp=1, bounces=4, spc=4, scene_size=1, proxy_mode=0)
        R = dprt.Renderer(cfg)
        R.set_materials(dprt.scene.make_materials(16)); R.set_lights(dprt.scene.make_lights()); R.set_camera(dprt.scene.default_camera(w, h))
        nt = dprt.flatten_instances(meshes, inst)[0].shape[0]
        row = {"input": label, "instances": len(inst), "meshes": len(meshes), "triangles": nt}
        row["upload_instanced_chunk_ms"] = round(wall_ms(lambda: R.upload_instanced_chunk(0, desc, meshes, inst), args.calls, args.warmup), 2)
        row["sample_ms_host_uploaded"] = round(sample_ms(dprt, R, args.samples), 3)
        row["build_instanced_chunk_ms"] = round(wall_ms(lambda: R.build_instanced_chunk(0, desc, meshes, inst), args.calls, args.warmup), 2)
        row["sample_ms_gpu_built"] = round(sample_ms(dprt, R, args.samples), 3)
        flip = [0]

        def host_move():
            flip[0] ^= 1
            v, n, _, _ = dprt.flatten_instances(meshes, m1 if flip[0] else inst)
            R.refit_chunk(0, v, n)

        def device_move():
            flip[0] ^= 1
            R.update_instances(0, m1 if flip[0] else inst)

        row["host_flatten_plus_refit_chunk_ms"] = round(wall_ms(host_move, 2 * args.calls, 2 * args.warmup), 3)
        row["update_instances_ms"] = round(wall_ms(device_move, 2 * args.calls, 2 * args.warmup), 3)
        R.close()
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)
    text = "\n".join(lines)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_instanced_build_cost.txt"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
