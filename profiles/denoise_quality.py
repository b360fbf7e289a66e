"""Image quality of the denoiser (DESIGN.md 3.8) on the CPU: relMSE against a high-spp render, noisy and denoised.

A quality number, not a speed number, so the CPU reference renders (tests/denoise_reference.py: the oracle with the guide
buffers) are valid for it; dprt.spec_denoise gives the GPU's bits. Prints the table of profiles/denoise_quality.txt: the
defaults, each parameter moved one step either side of them, and (--search) the best grid point.

    python profiles/denoise_quality.py [--search] > profiles/denoise_quality.txt
"""
import argparse
import itertools
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import denoise_reference as R  # noqa: E402
import dprt  # noqa: E402

W, H, LOW, HIGH = 128, 72, 4, 256


def median_rel(x, ref):
    """The median pixel's relative squared error: what the mean hides when a few fireflies dominate it."""
    x, ref = np.asarray(x, np.float64), np.asarray(ref, np.float64)
    return float(np.median(((x - ref) ** 2 / (ref ** 2 + 1e-2)).mean(-1)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--search", action="store_true", help="also scan a parameter grid and report its best point")
    args = ap.parse_args()
    t0 = time.time()
    scenes = {}
    for name in ("landscape", "garden"):
        low, high = R.render(name, W, H, LOW), R.render(name, W, H, HIGH)
        scenes[name] = (low, high[0], R.rel_mse(low[0], high[0]))
    print(f"# denoiser quality: {W}x{H}, 2 bounces, {LOW} spp denoised against {HIGH} spp; relMSE = mean (x - ref)^2 / (ref^2 + 0.01)")
    print(f"# CPU reference renders (oracle + guide buffers), dprt.spec_denoise (bit-identical to the GPU); {time.time() - t0:.1f} s to render")

    def score(p):
        out = {}
        for name, (low, ref, noisy) in scenes.items():
            out[name] = R.rel_mse(dprt.spec_denoise(*low, **p), ref) / noisy
        return out

    def median_ratio(p):
        return {name: median_rel(dprt.spec_denoise(*low, **p), ref) / median_rel(low[0], ref) for name, (low, ref, _) in scenes.items()}

    d = dict(R.DEFAULTS)
    rows = [("defaults", d)]
    for k, f in (("sigma_color", 2.0), ("sigma_normal", 2.0), ("sigma_albedo", 2.0)):
        rows += [(f"{k} / {f:g}", {**d, k: d[k] / f}), (f"{k} x {f:g}", {**d, k: d[k] * f})]
    rows += [("iterations - 1", {**d, "iterations": d["iterations"] - 1}), ("iterations + 1", {**d, "iterations": d["iterations"] + 1})]
    print("noisy relMSE: " + ", ".join(f"{n} {s[2]:.4f}" for n, s in scenes.items()))
    print("ratio = denoised / noisy relMSE; median = the same ratio for the median pixel's error")
    print(f"{'variant':<20} {'L':>2} {'s_col':>6} {'s_nrm':>6} {'s_alb':>6} | " + " | ".join(f"{n:>9} relMSE  ratio median" for n in scenes))
    for label, p in rows:
        r, m = score(p), median_ratio(p)
        print(f"{label:<20} {p['iterations']:>2} {p['sigma_color']:>6g} {p['sigma_normal']:>6g} {p['sigma_albedo']:>6g} | " +
              " | ".join(f"{r[n] * scenes[n][2]:>16.4f} {r[n]:>6.3f} {m[n]:>6.3f}" for n in scenes))
    if args.search:
        best = None
        for L, sc, sn, sa in itertools.product((2, 3, 4, 5), (1.0, 2.0, 4.0, 8.0), (0.3, 1.0, 3.0, 10.0), (0.1, 0.3, 1.0, 3.0)):
            p = {"iterations": L, "sigma_color": sc, "sigma_normal": sn, "sigma_albedo": sa}
            r = score(p)
            g = float(np.sqrt(np.prod(list(r.values()))))
            if best is None or g < best[0]:
                best = (g, p, r)
        print(f"grid best (geometric mean of the two ratios {best[0]:.3f}): {best[1]} " + ", ".join(f"{n} {v:.3f}" for n, v in best[2].items()))


if __name__ == "__main__":
    main()
