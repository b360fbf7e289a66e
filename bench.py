#!/usr/bin/env python
"""bench.py -- throughput of the per-sample / per-bounce loop (BASELINE.json metric: Mrays/s and samples/s).

    python bench.py --gpus N --steps K --warmup W            # this repo: libdprt.so on N B200s (torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...   # the CPU oracle of the reference's logic, host cores
    python bench.py ... --dump-outputs DIR                    # also writes the frame image of the K timed steps to DIR

One STEP = one pass of the hot path = one `runSample` (renderer.cpp:1457-1574: path_gen, then bounces+1 times
{[secondary-NN], traverse/partition/exchange until quiescent, shade, shadow}) over one frame of camera paths.
Workload (config.workload): BASELINE.json configs[1]'s scene per GPU -- a synthetic 1 M-triangle chunk and
1920x1080 pixels PER GPU (W = N chunks, frame scaled by sqrt(N) per side so pixels/GPU and triangles/GPU stay
fixed: weak scaling), 1 sample per step, bounces=4, spc=4 shadow paths per hit. For N > 1 the chunks are x-slabs of one
continuous terrain, cut where every owner walks the same number of rays over all bounces (scene.CALIBRATED_SLAB_CUTS,
profiles/calibrate_slabs.py), and before anything is timed a small frame goes through the same data plane and is compared
with the oracle bit for bit ("parity" in the JSON line; a mismatch aborts the run). The literal configs[1] case
(closest-hit primary rays only, through host buffers) and the proxy MLP of configs[0] are measured beside it at
N=1 and reported in the same JSON line ("primary_closest_hit", "proxy_mlp").

A ray = one (origin, direction, tmin, tmax) query that actually WALKED one rank's chunk BVH in TraRay / MainRay /
ShadowRay / SecondaryRay (dprt_stats.rays_walked, counted on the device; records that only ride along in a launch and
MainRay queries answered from the hit cache are not rays; the CPU arm counts the same events, and it does re-trace
MainRay). value = rays of all ranks / max-over-ranks device time of the K steps, inputs resident in HBM, --inflight samples
in flight per GPU (one context and host thread each, dprt.h "samples in flight"), no per-stage events inside the timed
region (the stages overlap). Per-stage times, `roofline` (algorithmic node / triangle counts from the ORACLE's walk over
the uploaded BVH8), `reorder`, `image_reduce` and `stages` come from a second, strictly serial single-context pass over
the same samples with CUDA-event pairs around every stage launch. e2e = the same metric through the host-facing call
sequence of Renderer::launch with host buffers (camera, lights and materials uploaded, frame reset, one sample, image
reduced and copied to pinned host memory) per step, inside the timed region.
"""
import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

# before CUDA initialises: one hardware queue per stream. Six samples in flight are twelve streams per GPU, and the peer-memory
# exchange parks waiting kernels in them (libdprt refuses to wire more streams than queues, DESIGN.md 3.4)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mrays/s"
TRAVERSAL_STAGES = ("traverse", "shade", "shadow_trace", "secondary_trace")
# algorithmic path-record bytes per ray of each traversal stage (DESIGN.md "Algorithmic bytes"):
#   traverse / secondary: 64 B record read + 64 B written back; shade: 64 B read + (1+spc) x 64 B written;
#   shadow: 64 B read + 16 B flag word (or a 12 B direct-light add)
RECORD_BYTES = {"traverse": 128, "secondary_trace": 128, "shade": 64 + 5 * 64, "shadow_trace": 64 + 16, "trace_closest": 32 + 8}
NODE_BYTES, TRI_BYTES = 80, 48
MLP_FLOP_PER_QUERY = 573888     # 2 x 286 944 MACs, NeuralVisNetworkWith4Res256SingleOutput (SURVEY.md 8a16)
DUMP_BYTES = 60 << 20           # --dump-outputs: at most this much .npy data in all


def frame_for(world, base_w=1920, base_h=1080):
    """Pixels per GPU fixed: the 16:9 frame grows by sqrt(world) per side (world=4 -> 3840x2160)."""
    if world == 1:
        return base_w, base_h
    w = int(round(base_w * math.sqrt(world) / 16.0)) * 16
    return w, w * 9 // 16


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tensor_burst": d["bf16_tflops"], "tensor_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=f, stderr=subprocess.DEVNULL)
            f.close()
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 8:
                    continue
                try:
                    sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
                except ValueError:
                    continue
                for k, nm in enumerate(names):
                    if c[4 + k].lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def build_world_scene(dprt, world, tris, layout="slabs"):
    """N > 1: the unit cube is cut into load-balanced x-slabs for the benchmark camera (scene.balanced_slab_layout), one
    1 M-triangle height-field chunk per slab; --layout cells gives the 2x2x1 / 2x2x2 cells the parity tests use."""
    fw, fh = frame_for(world)
    chunks, mats, lights = dprt.scene.make_scene(world, tris, layout=layout, camera=dprt.scene.default_camera(fw, fh))
    return chunks, mats, lights


def proxy_blobs(dprt, world, enable):
    """Untrained proxies with spread outputs (SURVEY.md 7 hard part 3): one vis + one depth network per chunk."""
    if not enable or world < 2:
        return {}
    import torch
    out = {}
    for k in range(world):
        torch.manual_seed(19990201 + k)
        vis = dprt.proxy.spread_output_(dprt.proxy.make_proxy(256, 4).eval(), gain=3.0, seed=k)
        torch.manual_seed(29990201 + k)
        dep = dprt.proxy.spread_output_(dprt.proxy.make_proxy(256, 4).eval(), gain=1.0, seed=100 + k)
        out[k] = (dprt.proxy.pack_module(vis), dprt.proxy.pack_module(dep))
    return out


# ------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the CPU restatement of the reference's logic (oracle/liboracle.so, OpenMP over paths),
    same config and metric; each step a bounded sample of the workload = one runSample over a reduced frame
    (1/ref_scale of the pixels per side) of the same scene. No GPU is touched."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    from oracle import oracle as O
    O.lib()
    O.use_all_host_threads()          # rank 0 runs alone (the other ranks exited): torchrun's OMP_NUM_THREADS=1 does not apply
    W = args.gpus
    fw, fh = frame_for(W)
    # bounded sample: the reference's migrate loop handles every path of a rank in every iteration (~9 per bounce at 8
    # chunks), so a sample costs more per pixel as W grows; the frame shrinks with it to keep a step around a second
    scale = 1 if W == 1 else args.ref_scale * (2 if W <= 4 else 3)      # N = 1: the whole 1920x1080 frame (~2 s per step)
    w, h = max(16, fw // scale), max(9, fh // scale)
    chunks, mats, lights = build_world_scene(dprt, W, args.tris, args.layout)
    cfg = dprt.make_config(w, h, spp=1, bounces=args.bounces, scene_size=W, proxy_mode=1 if (args.proxy and W > 1) else 0,
                           path_gen_mode=args.path_gen_mode if W > 1 else 0, mlp_dtype=1)
    world = O.World(cfg, W)
    blobs = proxy_blobs(dprt, W, args.proxy)
    if W == 1 and args.warmup > 1:
        args.warmup = 1                 # a CPU pass has nothing to warm beyond the first touch; keeps the full-frame arm inside the budget
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
        if c.index in blobs:
            world.set_model(c.index, 0, blobs[c.index][0]); world.set_model(c.index, 1, blobs[c.index][1])
    world.set_materials(mats); world.set_lights(lights); world.set_camera(dprt.scene.default_camera(w, h))
    world.reset_frame()
    for s in range(args.warmup):
        world.render_sample(s)
    def rays_total():
        return sum(world.stats(r)["rays_walked"] for r in range(W))
    r0 = rays_total()
    t0 = time.perf_counter()
    for s in range(args.steps):
        world.render_sample(args.warmup + s)
    dt = time.perf_counter() - t0
    rays = rays_total() - r0
    val = rays / dt / 1e6
    cores = O.num_threads()
    sample = (f"{args.steps} x runSample over the full {w}x{h} frame of the same 1-chunk scene" if scale == 1 else
              f"{args.steps} x runSample over a {w}x{h} frame (1/{scale} per side of {fw}x{fh}) of the same {W}-chunk scene")
    cfg_out = workload_config(args, W, fw, fh)          # N = 1: the very same workload, so the very same config
    if scale != 1:
        cfg_out["reference_arm_frame"] = f"{w}x{h}"
        cfg_out["workload"] += f" -- the CPU arm renders a {w}x{h} sub-sampled frame of it (rate metric, same scene and camera)"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mrays/s", "n_gpus": W, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "samples_per_s": w * h * args.steps / dt,
        "config": cfg_out,
        "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(args, W, fw, fh):
    return {"workload": f"configs[1] scene per GPU: synthetic {args.tris}-triangle chunk x {W} chunk(s), {fw}x{fh} frame "
                        f"(1920x1080 pixels per GPU), 1 spp per step, full per-sample loop with bounces={args.bounces}, spc=4, mc=3",
            "chunks": W, "tris_per_chunk": args.tris, "chunk_layout": "single chunk" if W == 1 else
            ("one continuous terrain in load-balanced x-slabs (k/W quantiles of where the primary rays land)" if args.layout == "slabs" else "2x1x1 / 2x2x1 / 2x2x2 cells"), "width": fw, "height": fh, "bounces": args.bounces,
            "proxy": bool(args.proxy and W > 1), "main_ray": "re-trace" if args.retrace else "hit cache",
            "stage_overlap": bool(not args.serial and not (args.proxy and W > 1)), "samples_in_flight_requested": args.inflight, "path_gen": "rank0" if (args.path_gen_mode == 0 or W == 1) else "striped",
            "l2": "inputs larger than L2: 5 x 64 B path records per pixel (663 MB at 1080p) are rewritten every bounce",
            "parallelism": f"scene-chunk x{W}"}


# ------------------------------------------------------------------------------------------------------
def cpu_baseline(dprt, args, seconds_target=15.0):
    """The oracle on this box's host cores over a bounded sample of the N=1 workload (reduced frame, same scene)."""
    from oracle import oracle as O
    O.lib()
    O.use_all_host_threads()
    fw, fh = frame_for(1)
    w, h = fw // args.ref_scale, fh // args.ref_scale
    chunks, mats, lights = build_world_scene(dprt, 1, args.tris)
    cfg = dprt.make_config(w, h, spp=1, bounces=args.bounces, scene_size=1)
    world = O.World(cfg, 1)
    c = chunks[0]
    world.add_object(0, c.desc(False), c.verts, c.normals, c.mats)
    world.set_materials(mats); world.set_lights(lights); world.set_camera(dprt.scene.default_camera(w, h))
    world.reset_frame()
    world.render_sample(0)          # warm-up (also builds the oracle's BVH)
    st0 = world.stats(0)
    t0 = time.perf_counter()
    n = 0
    while True:
        world.render_sample(1 + n)
        n += 1
        if time.perf_counter() - t0 > seconds_target or n >= 64:
            break
    dt = time.perf_counter() - t0
    st = world.stats(0)
    rays = st["rays_walked"] - st0["rays_walked"]
    return {"value": rays / dt / 1e6, "unit": "Mrays/s", "cores": O.num_threads(), "kind": "port",
            "sample": f"{n} x runSample over a {w}x{h} frame (1/{args.ref_scale} per side) of the same 1-chunk scene, {dt:.1f} s",
            "samples_per_s": w * h * n / dt}


def dump_image(out_dir, img, seed=0):
    """--dump-outputs: the frame image [h, w, 3] as out_dir/image.npy (float32). A frame over DUMP_BYTES (N >= 4) is
    replaced by a fixed, seeded sample of its pixels: image_pixels.npy [k, 3] and their row-major indices,
    image_pixel_index.npy [k] (float64, exact)."""
    img = np.ascontiguousarray(img, np.float32)
    if img.nbytes <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "image.npy"), img)
        return
    pix = img.reshape(-1, 3)
    idx = np.sort(np.random.default_rng(seed).choice(pix.shape[0], DUMP_BYTES // (3 * 4 + 8), replace=False))
    np.save(os.path.join(out_dir, "image_pixels.npy"), pix[idx])
    np.save(os.path.join(out_dir, "image_pixel_index.npy"), idx.astype(np.float64))


def pinned_array(shape, dtype):
    import torch
    t = torch.empty(int(np.prod(shape)) * np.dtype(dtype).itemsize, dtype=torch.uint8, pin_memory=True)
    return t, t.numpy().view(dtype).reshape(shape)


def bench_primary(dprt, R, args, pk):
    """BASELINE configs[1] literally: closest-hit primary rays, 1080p, 1 spp, on the 1 M-triangle chunk."""
    D = dprt.ctypes_defs
    cam = dprt.scene.default_camera(1920, 1080)
    rays = dprt.scene.camera_rays(cam)
    n = rays.size
    d_rays, d_hits = R.device_alloc(rays.nbytes), R.device_alloc(n * 8)
    R.h2d(d_rays, rays)
    for _ in range(3):
        R.trace_closest_device(d_rays, n, d_hits)
    R.synchronize()
    times = []
    for _ in range(max(3, args.steps)):
        R.flush_l2()                      # rays + hits (83 MB) fit in L2: flush between timed iterations
        R.timer_start(); R.trace_closest_device(d_rays, n, d_hits); times.append(R.timer_stop())
    ms = float(np.mean(times))
    # algorithmic bytes from the instrumented variant
    R.reset_stats(); R.enable_counters(True)
    R.trace_closest_device(d_rays, n, d_hits); R.synchronize()
    nodes, tris = R.counters()["trace_closest"]
    R.enable_counters(False)
    alg = n * RECORD_BYTES["trace_closest"] + nodes * NODE_BYTES + tris * TRI_BYTES
    # end to end through host buffers (pinned), H2D + trace + D2H
    keep1, hrays = pinned_array((n,), D.RAY_DTYPE)
    keep2, hhits = pinned_array((n,), D.HIT_DTYPE)
    hrays[:] = rays
    lib, h = R.lib, R.h
    for _ in range(2):
        R._ck(lib.dprt_trace_closest(h, hrays.ctypes.data, n, hhits.ctypes.data), "dprt_trace_closest")
    t0 = time.perf_counter()
    k = max(3, args.steps)
    for _ in range(k):
        R._ck(lib.dprt_trace_closest(h, hrays.ctypes.data, n, hhits.ctypes.data), "dprt_trace_closest")
    e2e_ms = (time.perf_counter() - t0) / k * 1e3
    hit_frac = float((hhits["primID"] >= 0).mean())
    R.device_free(d_rays); R.device_free(d_hits)
    return {"workload": "closest-hit primary rays, 1 M-triangle chunk, 1920x1080, 1 spp (BASELINE configs[1])",
            "value": n / ms / 1e3, "unit": "Mrays/s", "ms": ms, "hit_fraction": hit_frac,
            "e2e": {"value": n / e2e_ms / 1e3, "unit": "Mrays/s", "ms": e2e_ms, "h2d_bytes_per_step": int(rays.nbytes), "d2h_bytes_per_step": n * 8},
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / pk["hbm"], "bytes_per_ray": alg / n,
                         "nodes_per_ray": nodes / n, "tris_per_ray": tris / n}}


def bench_mlp(dprt, args, pk, device):
    """BASELINE configs[0] on the GPU: 4Res256 proxy, 1 M synthetic queries, device-resident, fused tcgen05 kernel."""
    import torch
    torch.manual_seed(19990201)
    m = dprt.proxy.make_proxy(256, 4).eval()
    blob = dprt.proxy.pack_module(m)
    out = {}
    n = 1 << 20
    x = np.random.default_rng(0).random((n, 5)).astype(np.float16).view(np.uint16)
    for name, dt in (("bf16", 0), ("fp16", 1)):
        cfg = dprt.make_config(16, 16, scene_size=2, proxy_mode=1, mlp_dtype=dt)
        P = dprt.Renderer(cfg, rank=0, world=2, device=device)
        P.upload_proxy(1, dprt.make_object_desc(1, [0, 0, 0], [1, 1, 1], is_proxy=1), blob, blob)
        dx, dy = P.device_alloc(x.nbytes), P.device_alloc(n * 2)
        P.h2d(dx, x)
        for _ in range(3):
            P.mlp_infer_device(1, 0, dx, n, dy)
        P.synchronize()
        P.timer_start()
        k = 10
        for _ in range(k):
            P.mlp_infer_device(1, 0, dx, n, dy)
        ms = P.timer_stop() / k
        tf = MLP_FLOP_PER_QUERY * n / (ms * 1e-3) / 1e12
        out[name] = {"Mqueries_per_s": n / ms / 1e3, "ms_per_1Mi": ms, "achieved_tflops": tf, "peak_tflops": pk["tensor_burst"],
                     "frac": tf / pk["tensor_burst"]}
        P.close()
    return {"workload": "NeuralVisNetworkWith4Res256SingleOutput, 2^20 queries resident in HBM, one fused tcgen05/TMEM launch",
            "bound": "tensor", **out}


def oracle_bvh8_counts(dprt, args, W, proxy, chunks, mats, lights, blobs):
    """SURVEY.md 8(d): the BVH bytes of the roofline come from the ORACLE -- a scalar walker with an exact tbest over the very
    BVH8 blob the product uploads (dprt_bvh8_build is deterministic) -- not from the kernel's own counters. One sample of the
    same scene, camera and loop over a sub-sampled frame; per stage: nodes fetched and triangles tested per ray that walked."""
    from oracle import oracle as O
    O.lib(); O.use_all_host_threads()
    fw, fh = frame_for(W)
    w, h = max(16, fw // args.count_scale), max(9, fh // args.count_scale)
    cfg = dprt.make_config(w, h, spp=1, bounces=args.bounces, scene_size=W, proxy_mode=proxy, path_gen_mode=args.path_gen_mode if W > 1 else 0, mlp_dtype=1)
    world = O.World(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
        nodes, tris, _ = dprt.build_bvh8(c.verts, c.mats)
        world.set_bvh8(c.index, nodes, tris)
        if c.index in blobs:
            world.set_model(c.index, 0, blobs[c.index][0]); world.set_model(c.index, 1, blobs[c.index][1])
    world.set_materials(mats); world.set_lights(lights); world.set_camera(dprt.scene.default_camera(w, h))
    world.count_bvh8(True)
    world.reset_frame()
    world.render_sample(args.warmup)
    out = {}
    for name in TRAVERSAL_STAGES:
        n = t = r = 0
        for k in range(W):
            cn, ct, cr = world.bvh8_counters(k)[name]
            n += cn; t += ct; r += cr
        if r:
            out[name] = {"nodes_per_ray": n / r, "tris_per_ray": t / r, "rays_sampled": r}
    world.close()
    return out, f"{w}x{h}"


def parity_gate(dprt, R, args, rank, W, dist, torch):
    """N > 1, before anything is timed: a small frame rendered through the SAME data plane the timed runs use -- a second
    context of this rank on the parent's NCCL communicator, peer-memory exchange wired the same way -- and compared with the
    oracle's W-rank world exactly as tests/mgpu_check.py does: every rank its own path / env / direct buffers bit for bit,
    rank 0 the ncclReduce'd image (NCCL chooses the summation order: 1e-6 relative). Proxies off: with them on the GPU and
    the oracle may legitimately disagree at a threshold, which tests/test_gpu_proxy.py bounds separately."""
    from oracle import oracle as O
    O.lib()
    O.lib().orc_set_num_threads(max(1, (os.cpu_count() or 1) // W))
    D = dprt.ctypes_defs
    w, h, spp, bounces, tris = 256, 144, 2, 4, 20000
    cam = dprt.scene.default_camera(w, h)
    chunks, mats, lights = dprt.scene.make_scene(W, tris, layout=args.layout, camera=cam)
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W, proxy_mode=0, path_gen_mode=args.path_gen_mode,
                           main_ray_retrace=args.retrace, serial_stages=args.serial)
    P = dprt.Renderer(cfg, parent=R)
    world = O.World(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
        if c.node_id == rank:
            P.upload_chunk(c.index, c.desc(False), c.verts, c.normals, c.mats)
        else:
            P.upload_proxy(c.index, c.desc(True), None, None)
    for X in (P, world):
        X.set_materials(mats); X.set_lights(lights); X.set_camera(cam)
    img = P.launch()
    img_o = world.launch()
    N, spc = w * h, cfg.shadowPathCount
    problems = []

    def same(a, b, what):
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        if a.shape != b.shape or not np.array_equal(a.view(np.uint8), b.view(np.uint8)):
            problems.append(f"rank {rank}: {what} differs from the oracle")
    n = P.path_size
    if n != world.path_size(rank):
        problems.append(f"rank {rank}: pathSize {n} vs oracle {world.path_size(rank)}")
    else:
        same(P.download(D.BUF_PATHS, n * (1 + spc)), world.download(rank, D.BUF_PATHS, n * (1 + spc)), "path records")
    same(P.download(D.BUF_ENV), world.download(rank, D.BUF_ENV, 3 * N), "envLightingBuffer")
    same(P.download(D.BUF_DIRECT), world.download(rank, D.BUF_DIRECT, 3 * N * spc), "directLightingBuffer")
    sg, so = P.stats(), world.stats(rank)
    for k in ("rays_traverse", "rays_shade", "rays_shadow", "paths_sent_offrank", "exchange_iters"):
        if sg[k] != so[k]:
            problems.append(f"rank {rank}: {k} {sg[k]} vs oracle {so[k]}")
    err = 0.0
    if rank == 0:
        err = float(np.abs(img - img_o).max() / max(1e-30, float(np.abs(img_o).max())))
        if not (np.isfinite(img).all() and err <= 1e-6):
            problems.append(f"reduced image differs from the oracle: rel err {err:.3e}")
    p2p = P.p2p_enabled
    P.close(); world.close()
    t = torch.tensor([len(problems), sg["paths_sent_offrank"]], dtype=torch.int64, device="cuda")
    dist.all_reduce(t)
    every = [None] * W
    dist.all_gather_object(every, problems)
    return {"ok": int(t[0].item()) == 0, "world": W, "migrated_paths": int(t[1].item()), "image_rel_err": err,
            "data_plane": "peer memory over NVLink (CUDA IPC) + ncclReduce" if p2p else "ncclAllGather + ncclSend/ncclRecv + ncclReduce",
            "frame": f"{w}x{h}, {spp} spp, bounces={bounces}, {tris} triangles per chunk, proxies off",
            "checked": "per rank: pathSize, path records, envLightingBuffer, directLightingBuffer, launch sizes, exchange statistics "
                       "bit-exact vs the oracle's W-rank world; rank 0: reduced image <= 1e-6 rel",
            "problems": [q for ps in every for q in ps][:8]}


def run_dprt(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs a torchrun launch with {args.gpus} ranks")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (libdprt has no CPU fallback; use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    D = dprt.ctypes_defs
    pk = peaks()
    W = world
    uid = None
    if W > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        t = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            t = torch.tensor(list(dprt.get_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(t, 0)
        uid = bytes(t.cpu().tolist())

    fw, fh = frame_for(W)
    N = fw * fh
    proxy = 1 if (args.proxy and W > 1) else 0
    cfg = dprt.make_config(fw, fh, spp=1, bounces=args.bounces, scene_size=W, proxy_mode=proxy,
                           path_gen_mode=args.path_gen_mode if W > 1 else 0, mlp_dtype=args.mlp_dtype, main_ray_retrace=args.retrace,
                           serial_stages=args.serial)
    chunks, mats, lights = build_world_scene(dprt, W, args.tris, args.layout)
    blobs = proxy_blobs(dprt, W, proxy)
    cam = dprt.scene.default_camera(fw, fh)
    R = dprt.Renderer(cfg, rank=rank, world=W, device=local, nccl_unique_id=uid)
    for c in chunks:
        if c.node_id == rank:
            R.upload_chunk(c.index, c.desc(False), c.verts, c.normals, c.mats)
        else:
            vb, db = blobs.get(c.index, (None, None))
            R.upload_proxy(c.index, c.desc(True), vb, db)
    R.set_materials(mats); R.set_lights(lights); R.set_camera(cam)
    if rank != 0 or args.skip_oracle_counts:
        del chunks                      # rank 0 keeps the scene for the oracle's counting pass (after the timed region)

    def barrier():
        torch.cuda.synchronize()
        if W > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allreduce(x, op):
        if W == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    # ---- N > 1: parity gate on the same communicator / peer-memory wiring, before anything is timed ---------
    parity = None
    if W > 1 and not args.skip_parity:
        parity = parity_gate(dprt, R, args, rank, W, dist, torch)
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"metric": METRIC, "value": None, "n_gpus": W, "parity": parity, "error": "parity gate failed: nothing was timed"}), flush=True)
            dist.barrier()
            raise SystemExit(3)

    # ---- samples in flight (dprt.h): K contexts of this rank share the uploaded scene and the communicator; context j renders
    # samples j, j + K, ... from its own host thread. Each sample's work is what it is with K = 1; the launches of one sample's
    # late bounces / late migrate iterations (10^4..10^5 rays, as long as their longest ray) overlap the other's big ones.
    F = dprt.SamplesInFlight(R, args.inflight)
    K_inflight = len(F.ctxs)

    # ---- device-resident timing: W warm-up samples, then exactly K samples between two events ----------------
    F.reset_frame()
    F.run_samples(0, args.warmup * K_inflight)
    for X in F.ctxs:
        X.synchronize()
    barrier()
    for X in F.ctxs:
        X.reset_stats()
    clocks = ClockSampler(local if "CUDA_VISIBLE_DEVICES" not in os.environ else os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local])
    if rank == 0:
        clocks.start()
    for X in F.ctxs:
        X.timer_start()                 # all streams are idle here: the start events coincide
    F.run_samples(args.warmup * K_inflight, args.steps)
    ms = max(X.timer_stop() for X in F.ctxs)
    barrier()
    st = F.stats()
    my_rays_walked = st["rays_walked"]
    ms = allreduce(ms, dist.ReduceOp.MAX if W > 1 else None)
    # ---- --dump-outputs: what a caller of the timed path receives after its last step -- the frame image (warm-up and
    # timed samples accumulated over the contexts in flight, averaged, reduced to rank 0), as SamplesInFlight.launch returns
    # it. Taken here, before the passes below add samples to the primary's frame; written after the clock sampler stops.
    dump_img = None
    if args.dump_outputs:
        F.accumulate()
        dump_img = R.reduce_image(0)
    # ---- per-stage pass over the same samples: CUDA-event pairs around every stage launch on the stream it is launched
    # on. Stage profiling forces strictly serial single-stream execution (no shadow/traverse overlap), so each kernel's
    # duration is its own; the step time of this pass is reported beside it (share_of_step refers to it).
    R.reset_stats(); R.stage_profile(True)
    R.timer_start()
    for s in range(args.steps):
        R.run_sample(args.warmup + s)
    ms_serial = R.timer_stop()
    barrier()
    clk = clocks.stop() if rank == 0 else None          # sampled through the timed region and the serial pass right after it
    if dump_img is not None:
        dump_image(args.dump_outputs, dump_img)
    # the per-frame image average + ncclReduce (renderer.cpp:2031-2052), profiled like a stage: 3 times, device events
    keep_r, himg_r = pinned_array((fh, fw, 3), np.float32)
    R.stage_profile(False)
    R._ck(R.lib.dprt_reduce_image(R.h, 0, himg_r.ctypes.data if rank == 0 else None), "dprt_reduce_image")   # untimed: NCCL sets its channels up on first use
    barrier()
    R.stage_profile(True)
    for _ in range(3):
        R._ck(R.lib.dprt_reduce_image(R.h, 0, himg_r.ctypes.data if rank == 0 else None), "dprt_reduce_image")
    barrier()
    stage = R.stage_times()
    sst = R.stats()
    R.stage_profile(False)
    reduce_ms = allreduce(stage["image"][0] / max(1, stage["image"][1]), dist.ReduceOp.MAX if W > 1 else None)
    stage.pop("image")
    # per-rank view of the serial pass: time inside the exchange stage is mostly waiting for the slowest chunk owner
    mine = {"rank": rank, "rays_walked_per_step": my_rays_walked / args.steps,
            "busy_ms_per_step": sum(t for k, (t, _) in stage.items() if k != "exchange") / args.steps,
            "exchange_ms_per_step": stage["exchange"][0] / args.steps,
            "sent_bytes_per_step": sst["bytes_alltoall"] / args.steps,
            # the records leave inside the partition launch when the peer-memory exchange is on, inside ncclSend/ncclRecv otherwise
            "alltoall_GBps": sst["bytes_alltoall"] / max(1e-9, (stage["exchange"][0] + (stage["partition"][0] if R.p2p_enabled else 0.0)) * 1e-3) / 1e9}
    per_rank = [mine]
    if W > 1:
        per_rank = [None] * W
        dist.all_gather_object(per_rank, mine)
    # rays = BVH walks actually performed (dprt_stats.rays_walked, counted on the device): a live record with at least one
    # local object it has not visited yet. Records that only ride along in a TraRay launch (their chunk is already
    # visited) and MainRay queries answered from the hit cache (DESIGN.md 3.1) are NOT counted in `value`.
    my_rays = st["rays_walked"]
    rays = allreduce(float(my_rays), dist.ReduceOp.SUM if W > 1 else None)
    cached = allreduce(float(st["rays_shade_cached"]), dist.ReduceOp.SUM if W > 1 else None)
    launches = allreduce(float(st["kernel_launches"]), dist.ReduceOp.SUM if W > 1 else None)
    sent = allreduce(float(st["bytes_alltoall"]), dist.ReduceOp.SUM if W > 1 else None)
    value = rays / (ms * 1e-3) / 1e6

    # ---- algorithmic bytes of the traversal kernels (SURVEY.md 8d) -------------------------------------------------
    # rays: the records each launch actually traced (dprt_stats.walked_*: riders of a TraRay launch and cache-answered
    # MainRay queries are not billed); nodes / triangles per ray: the ORACLE's scalar exact-tbest walk over the uploaded BVH8.
    # The kernel's own counters (instrumented variant, never timed) are reported beside them as gpu_*_per_ray.
    R.reset_stats(); R.enable_counters(True)
    for s in range(args.steps):
        R.run_sample(args.warmup + s)
    R.synchronize()
    cnt = R.counters(); cst = R.stats()
    R.enable_counters(False)
    oc, oc_frame = ({}, None)
    if rank == 0 and not args.skip_oracle_counts:
        oc, oc_frame = oracle_bvh8_counts(dprt, args, W, proxy, chunks, mats, lights, blobs)
        del chunks
    if W > 1:
        box = [oc, oc_frame]
        dist.broadcast_object_list(box, 0)
        oc, oc_frame = box
    walked = {"traverse": sst["walked_traverse"], "shade": sst["walked_shade"], "shadow_trace": sst["walked_shadow"], "secondary_trace": sst["walked_secondary"]}
    gwalked = {"traverse": cst["walked_traverse"], "shade": cst["walked_shade"], "shadow_trace": cst["walked_shadow"], "secondary_trace": cst["walked_secondary"]}
    stages_out = {}
    for name in TRAVERSAL_STAGES:
        t_ms, ln = stage[name]
        if ln == 0 or walked[name] == 0:
            continue
        gn, gt = cnt[name]
        g_npr, g_tpr = gn / max(1, gwalked[name]), gt / max(1, gwalked[name])
        if name in oc:
            npr, tpr, src = oc[name]["nodes_per_ray"], oc[name]["tris_per_ray"], "oracle"
        else:
            npr, tpr, src = g_npr, g_tpr, "kernel counters (no oracle sample)"
        alg = walked[name] * (RECORD_BYTES[name] + npr * NODE_BYTES + tpr * TRI_BYTES)
        stages_out[name] = {"ms": t_ms, "launches": ln, "rays": walked[name], "Mrays_per_s": walked[name] / t_ms / 1e3,
                            "alg_bytes": alg, "GBps": alg / (t_ms * 1e-3) / 1e9, "bytes_per_ray": alg / walked[name],
                            "nodes_per_ray": npr, "tris_per_ray": tpr, "counts_from": src,
                            "gpu_nodes_per_ray": g_npr, "gpu_tris_per_ray": g_tpr}
    for name, (t_ms, ln) in stage.items():
        if name not in stages_out and ln:
            stages_out[name] = {"ms": t_ms, "launches": ln}
    dom = max((k for k in TRAVERSAL_STAGES if k in stages_out and "GBps" in stages_out[k]), key=lambda k: stages_out[k]["ms"])
    d = stages_out[dom]
    ncu = {}
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if tj.get("n_gpus") == W and args.tris == tj.get("tris_per_chunk", 1000000) and dom in tj.get("kernels", {}):     # captured on this workload
            ncu = tj["kernels"][dom]
    roofline = {"bound": "hbm", "kernel": dom + "_kernel", "achieved": d["GBps"], "peak": pk["hbm"], "unit": "GB/s",
                "frac": d["GBps"] / pk["hbm"], "traffic": ncu.get("dram_bytes_per_launch"), "alg_bytes_per_launch": d["alg_bytes"] / d["launches"],
                "avg_launch_ms": d["ms"] / d["launches"], "share_of_step": d["ms"] / ms_serial, "serial_pass_ms_per_step": ms_serial / args.steps, "peak_source": pk["source"],
                "counts_from": d["counts_from"], "oracle_counting_frame": oc_frame,
                # what actually bounds the kernel (ncu --set full of the same command, profiles/): L2 throughput, issue slots, lanes
                "l2_gbs": ncu.get("l2_gbs"), "issue_active_pct": ncu.get("issue_active_pct"), "lanes_per_inst": ncu.get("lanes_per_inst"),
                "ncu_source": ncu.get("source"),
                "note": "a 1 M-triangle chunk (48 MB triangles + 15 MB BVH8) is L2-resident: `achieved` is bytes the algorithm must touch per "
                        "ray over the launch time, served mostly by L2/L1 -- `traffic` is what reached DRAM; the kernel is issue-bound "
                        "(issue_active_pct x lanes_per_inst / 32), see DESIGN.md 3.1"}
    # reorder (Work_Efficient_Scan): 64 B read + 64 B written per record the partition emits, over the partition launches
    p_ms, p_ln = stage.get("partition", (0.0, 0))
    reorder = None
    if p_ln and sst["paths_partitioned"]:
        rb = 128.0 * sst["paths_partitioned"]
        reorder = {"bound": "hbm", "kernel": "partition_kernel", "records_per_step": sst["paths_partitioned"] / args.steps, "alg_bytes_per_step": rb / args.steps,
                   "ms_per_step": p_ms / args.steps, "launches_per_step": p_ln / args.steps, "achieved": rb / (p_ms * 1e-3) / 1e9, "peak": pk["hbm"],
                   "unit": "GB/s", "frac": rb / (p_ms * 1e-3) / 1e9 / pk["hbm"], "share_of_step": p_ms / ms_serial}

    # ---- end to end: Renderer::launch() call sequence with host buffers -------------------------------------
    h2d = mats.nbytes + lights.nbytes + 56

    # every context in flight renders its own frames through the same public call sequence: K frames at a time, one host
    # thread each; the ncclReduce of the frames is issued from this thread, context by context (one communicator, one order)
    himgs = [pinned_array((fh, fw, 3), np.float32) for _ in F.ctxs]

    def e2e_front(X, s):
        X.set_materials(mats); X.set_lights(lights); X.set_camera(cam)       # host -> device (launch(): :1725-1849, :1990)
        X.reset_frame()
        X.run_sample(s)

    def e2e_run(first, count):
        """Steps first .. first + count - 1, dealt round-robin to the contexts in flight (one host thread each). A frame's
        average + ncclReduce + copy to host is issued by its own thread, in step order on every rank (a turn counter): one
        communicator, one order of collectives -- and it overlaps the other contexts' rendering."""
        import threading
        errs, turn, cv = [], [first], threading.Condition()

        def work(j):
            try:
                X = F.ctxs[j]
                for s in range(first + j, first + count, K_inflight):
                    e2e_front(X, s)
                    with cv:
                        while turn[0] != s and not errs:
                            cv.wait(0.5)
                    if errs:
                        return
                    X._ck(X.lib.dprt_reduce_image(X.h, 0, himgs[j][1].ctypes.data if rank == 0 else None), "dprt_reduce_image")   # device -> host, pinned
                    with cv:
                        turn[0] = s + 1
                        cv.notify_all()
            except Exception as e:      # noqa: BLE001
                errs.append(e)
                with cv:
                    cv.notify_all()
        th = [threading.Thread(target=work, args=(j,)) for j in range(1, K_inflight)]
        for t in th:
            t.start()
        work(0)
        for t in th:
            t.join()
        if errs:
            raise errs[0]
    e2e_run(0, K_inflight)
    barrier()
    st0 = F.stats()
    t0 = time.perf_counter()
    e2e_run(args.warmup, args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    st1 = F.stats()
    e2e_s = allreduce(e2e_s, dist.ReduceOp.MAX if W > 1 else None)
    e_rays = st1["rays_walked"] - st0["rays_walked"]
    e_rays = allreduce(float(e_rays), dist.ReduceOp.SUM if W > 1 else None)
    e2e = {"value": e_rays / e2e_s / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(N * 12),
           "ms_per_step": e2e_s / args.steps * 1e3, "samples_per_s": N * args.steps / e2e_s,
           "call": "set_materials/set_lights/set_camera + reset_frame + dprt_render_sample + dprt_reduce_image -> pinned host image, per step; "
                   f"{K_inflight} such frames in flight (one context and host thread each)"}

    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": W, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "samples_per_s": N * args.steps / (ms * 1e-3), "rays_per_step": rays / args.steps,
                "main_ray_queries_from_hit_cache_per_step": cached / args.steps,
                "config": workload_config(args, W, fw, fh), "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches),
                "samples_in_flight": K_inflight, "clocks": clk, "stages": stages_out, "ranks": per_rank, "reorder": reorder, "parity": parity,
                "exchange_data_plane": ("peer memory over NVLink (CUDA IPC), no host round trip" if R.p2p_enabled else "ncclAllGather + pinned read + ncclSend/ncclRecv") if W > 1 else "single rank",
                "alltoall": {"bytes_per_step": sent / args.steps, "exchange_iters_per_step": st["exchange_iters"] / args.steps,
                             "GBps_per_gpu_max": max(r["alltoall_GBps"] for r in per_rank), "nvlink_peak_GBps_per_direction": 900.0,
                             "exchange_wait_ms_per_step_max": max(r["exchange_ms_per_step"] for r in per_rank)},
                "image_reduce": {"ms": reduce_ms, "bytes": int(N * 12), "what": "image_average_kernel + ncclReduce(fp32 sum, root 0), device events, max over ranks"},
                "load_balance": {"rays_walked_max_over_mean": max(r["rays_walked_per_step"] for r in per_rank) / max(1e-9, sum(r["rays_walked_per_step"] for r in per_rank) / W)}}
    if W == 1:
        if not args.skip_extras:
            line["primary_closest_hit"] = bench_primary(dprt, R, args, pk)
            F.close()
            R.close()
            line["proxy_mlp"] = bench_mlp(dprt, args, pk, local)
        if not args.skip_cpu:
            line["cpu_baseline"] = cpu_baseline(dprt, args)
    else:
        F.close()
        R.close()
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=("dprt", "reference"), default="dprt")
    ap.add_argument("--tris", type=int, default=1000000, help="triangles per chunk")
    ap.add_argument("--bounces", type=int, default=4)
    ap.add_argument("--proxy", type=int, default=0, help="neural proxies for shadow/secondary rays at remote chunks (N>1)")
    ap.add_argument("--path-gen-mode", type=int, default=1, help="N>1: 0 = rank 0 generates all camera paths (reference), 1 = striped")
    ap.add_argument("--ref-scale", type=int, default=4, help="reference/cpu_baseline arm: frame reduced by this factor per side")
    ap.add_argument("--retrace", type=int, default=0, help="1 = MainRay always re-traces (no hit cache), for A/B")
    ap.add_argument("--layout", choices=("slabs", "cells"), default="slabs", help="N>1: how the unit cube is cut into chunks")
    ap.add_argument("--serial", type=int, default=0, help="1 = no shadow/traverse stream overlap inside dprt_render_sample, for A/B")
    ap.add_argument("--mlp-dtype", type=int, default=1, help="proxy MLP operands: 1 = fp16 (reference's NN_Float, meets 1e-3), 0 = bf16 (out of tolerance)")
    ap.add_argument("--inflight", type=int, default=6, help="samples in flight per GPU in the timed region (contexts sharing one scene; 1 = strictly one sample at a time)")
    ap.add_argument("--count-scale", type=int, default=8, help="oracle BVH8 counting pass: frame reduced by this factor per side")
    ap.add_argument("--skip-oracle-counts", action="store_true", help="roofline bytes from the kernel's own counters (A/B runs only)")
    ap.add_argument("--skip-parity", action="store_true", help="N>1: skip the parity gate (A/B runs only)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frame image they produced to DIR/image.npy (float32; a seeded pixel "
                         "sample above 60 MiB) so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "dprt":
            ap.error("--dump-outputs applies to --impl dprt")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.warmup < 3 and args.impl == "dprt":
        args.warmup = 3        # timing rule: at least 3 warm-up steps
    return run_reference(args) if args.impl == "reference" else run_dprt(args)


if __name__ == "__main__":
    sys.exit(main())
