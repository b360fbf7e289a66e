"""Cost of the denoiser (DESIGN.md 3.8) on one GPU: dprt_denoise_device at 1920x1080 and 3840x2160, 1 and 5 iterations, and
the host variant dprt_denoise with its copies.

    python profiles/denoise_cost.py [--calls 200] [--warmup 20] [--out DIR]

Every device call synchronises its stream, so each call gets its own CUDA-event pair (dprt_timer_start / dprt_timer_stop on
the context's stream) and the pairs are summed: one pair around a batch would also time the host gaps between calls. A pair
still holds the call's own launch latency; the per-iteration figure, (t(5) - t(1)) / 4, does not. The host variant is timed
with the host clock around whole calls (three host-to-device copies, the filter, one copy back).

Bounds, from the code's own counts (atrous_pixel in csrc/denoise.cu):
  bytes: per pixel and iteration the algorithm reads the demodulated colour (float4) and the packed guides (float4 + float2)
         once and writes the colour once (float4): 56 B, over 7.7 TB/s. (At 1080p the 116 MB working set fits the 126 MB L2,
         so the kernel may beat this HBM figure.)
  FP32:  per in-image tap 54 FP32-pipe instructions (9 differences; 3 x (3 mul + 2 add) distances; 3 mul + 2 add for the
         exponent argument; det_exp_neg: 7 fma, 6 mul / add, floor, compare, and 2 for ldexpf; 1 mul for the weight; 1 add +
         3 mul + 3 add to accumulate), counted once each (an fma is one instruction), over SMs x 128 lanes x the max SM clock.
  Taps that fall outside the image are skipped; the tap count is exact per size and step.
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

BYTES_PER_PIXEL_ITER = 16 + 16 + 8 + 16
FP32_PER_TAP = 54
HBM_BPS = 7.7e12


def taps(w, h, iterations):
    """In-image taps of `iterations` iterations (what atrous_pixel evaluates)."""
    t = 0
    for i in range(iterations):
        s = 1 << i
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                t += max(0, w - s * abs(dx)) * max(0, h - s * abs(dy))
    return t


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return name, float(power), float(clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    D = dprt.ctypes_defs
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_denoise_cpu import frame

    name, power, clock_mhz = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    fp32_peak = sms * 128 * clock_mhz * 1e6          # FP32 instructions per second
    lines = [f"# {name}, power limit {power:.0f} W, max SM clock {clock_mhz:.0f} MHz, {sms} SMs: FP32 peak {fp32_peak / 1e12:.1f} T instr/s, "
             f"HBM {HBM_BPS / 1e12:.1f} TB/s (data sheet)"]
    R = dprt.Renderer(dprt.make_config(16, 16, scene_size=1, proxy_mode=0))
    for w, h in ((1920, 1080), (3840, 2160)):
        c, a, n = frame(w, h, seed=w + h)
        bufs = [R.device_alloc(c.nbytes) for _ in range(4)]
        for b, x in zip(bufs, (c, a, n)):
            R.h2d(b, x)
        ms = {}
        for it in (1, 5):
            p = D.DenoiseParams(iterations=it, **{k: v for k, v in D.DENOISE_DEFAULTS.items() if k != "iterations"})
            for _ in range(args.warmup):
                R.denoise_device(w, h, bufs[0], bufs[1], bufs[2], bufs[3], p)
            tot = 0.0
            for _ in range(args.calls):
                R.timer_start()
                R.denoise_device(w, h, bufs[0], bufs[1], bufs[2], bufs[3], p)
                tot += R.timer_stop()
            ms[it] = tot / args.calls
        host = {}
        for it in (1, 5):
            for _ in range(3):
                R.denoise(c, a, n, iterations=it)
            t0 = time.perf_counter()
            k = max(5, args.calls // 10)
            for _ in range(k):
                R.denoise(c, a, n, iterations=it)
            host[it] = (time.perf_counter() - t0) * 1e3 / k
        for b in bufs:
            R.device_free(b)
        N = w * h
        per_iter = (ms[5] - ms[1]) / 4
        for it in (1, 5):
            tb = N * BYTES_PER_PIXEL_ITER * it / HBM_BPS * 1e3
            tf = taps(w, h, it) * FP32_PER_TAP / fp32_peak * 1e3
            r = {"width": w, "height": h, "iterations": it, "device_ms_per_call": round(ms[it], 4), "mpix_per_s": round(N / ms[it] / 1e3, 1),
                 "host_variant_ms_per_call": round(host[it], 3), "bound_bytes_ms": round(tb, 4), "bound_fp32_ms": round(tf, 4),
                 "bound": "fp32" if tf > tb else "bytes", "share_of_larger_bound": round(max(tb, tf) / ms[it], 3)}
            lines.append(json.dumps(r))
        tb1 = N * BYTES_PER_PIXEL_ITER / HBM_BPS * 1e3
        tf1 = (taps(w, h, 5) - taps(w, h, 1)) / 4 * FP32_PER_TAP / fp32_peak * 1e3
        lines.append(json.dumps({"width": w, "height": h, "ms_per_iteration": round(per_iter, 4), "bound_bytes_ms": round(tb1, 4),
                                 "bound_fp32_ms": round(tf1, 4), "share_of_fp32_bound": round(tf1 / per_iter, 3) if per_iter > 0 else None}))
    R.close()
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_denoise_cost.txt"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
