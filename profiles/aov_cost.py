"""Cost of the first-hit guide buffers (AOVs) on the benchmark workload: bench.py's one-GPU scene (1920x1080, 1 M triangles,
4 bounces), six samples in flight, AOVs off and on alternating in one process.

    python profiles/aov_cost.py [--steps 60] [--warmup 3] [--rounds 3] [--out DIR]

Each window: reset the frame, warm up, then time `steps` samples between CUDA events on every context in flight (as bench.py
does). With AOVs on, the first shade of every sample does one 24-byte read-modify-write per hit pixel on top of the shading.
Prints one JSON line per window and a summary line; --out also writes them to DIR/aov_cost.jsonl.
"""
import argparse
import importlib
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=3, help="warm-up samples per context in flight")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--inflight", type=int, default=6)
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
    R.set_materials(mats); R.set_lights(lights); R.set_camera(dprt.scene.default_camera(fw, fh))
    F = dprt.SamplesInFlight(R, args.inflight)
    K = len(F.ctxs)
    lines, first = [], 0
    for rnd in range(args.rounds):
        for aov in (False, True):
            F.enable_aov(aov)
            F.reset_frame()
            F.run_samples(first, args.warmup * K)
            first += args.warmup * K
            for X in F.ctxs:
                X.synchronize()
                X.reset_stats()
            for X in F.ctxs:
                X.timer_start()
            F.run_samples(first, args.steps)
            first += args.steps
            ms = max(X.timer_stop() for X in F.ctxs)
            rays = F.stats()["rays_walked"]
            line = {"round": rnd, "aov": aov, "samples": args.steps, "ms": ms, "ms_per_sample": ms / args.steps,
                    "Mrays_per_s": rays / (ms * 1e-3) / 1e6}
            if aov:
                F.accumulate()
                albedo, _ = F.reduce_aov(0)
                line["hit_pixel_fraction"] = float((albedo.reshape(-1, 3) != 0).any(axis=1).mean())
            print(json.dumps(line), flush=True)
            lines.append(line)
    per = {a: [ln["ms_per_sample"] for ln in lines if ln["aov"] == a] for a in (False, True)}
    off, on = statistics.median(per[False]), statistics.median(per[True])
    hit = statistics.median(ln["hit_pixel_fraction"] for ln in lines if ln["aov"])
    summary = {"summary": True, "frame": [fw, fh], "samples_in_flight": K, "ms_per_sample_off": per[False], "ms_per_sample_on": per[True],
               "median_off": off, "median_on": on, "cost_percent": 100.0 * (on / off - 1.0),
               "aov_bytes_per_sample": int(24 * 2 * hit * fw * fh), "hit_pixel_fraction": hit}
    print(json.dumps(summary), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "aov_cost.jsonl"), "w") as f:
            for ln in lines + [summary]:
                f.write(json.dumps(ln) + "\n")
    F.close()
    R.close()


if __name__ == "__main__":
    main()
