"""CPU reference of the denoiser for the tests: tests/denoise_reference.cpp compiled once per process with the oracle's flags
into a temporary directory, plus a float64 numpy model of DESIGN.md 3.8 that uses np.exp, and the image-quality metric."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULTS = {"iterations": 3, "sigma_color": 2.0, "sigma_normal": 1.0, "sigma_albedo": 0.3}     # DPRT_DENOISE_DEFAULT_*
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="denoise_reference_"), "libdenoiseref.so")
        cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
        # the flags of oracle/Makefile: no contraction, hardware fmaf, IEEE semantics
        p = subprocess.run([cxx, "-O3", "-std=c++17", "-fPIC", "-fopenmp", "-march=x86-64-v3", "-ffp-contract=off", "-fno-math-errno",
                            "-shared", "-o", out, os.path.join(ROOT, "tests", "denoise_reference.cpp")], capture_output=True, text=True)
        if p.returncode:
            raise RuntimeError("building tests/denoise_reference.cpp failed:\n" + p.stderr[-4000:])
        L = C.CDLL(out)
        L.ref_exp_neg.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        L.ref_denoise.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def exp_neg(x):
    x = np.ascontiguousarray(x, np.float32)
    out = np.zeros_like(x)
    lib().ref_exp_neg(_ptr(x), x.size, _ptr(out))
    return out


def _params(kw):
    p = dict(DEFAULTS)
    p.update({k: v for k, v in kw.items() if v is not None})
    return p


def denoise(color, albedo, normal, **kw):
    """The reference on [H, W, 3] float32 arrays; parameters not given take the defaults."""
    p = _params(kw)
    c, a, n = (np.ascontiguousarray(x, np.float32) for x in (color, albedo, normal))
    out = np.zeros_like(c)
    assert lib().ref_denoise(p["iterations"], p["sigma_color"], p["sigma_normal"], p["sigma_albedo"], c.shape[1], c.shape[0],
                             _ptr(c), _ptr(a), _ptr(n), _ptr(out)) == 0
    return out


def denoise_f64(color, albedo, normal, **kw):
    """DESIGN.md 3.8 in float64 with np.exp: what binary32 approximates (catches a misreading both float32 sides share)."""
    p = _params(kw)
    c, a, n = (np.asarray(x, np.float64) for x in (color, albedo, normal))
    H, W, _ = c.shape
    e = np.where(a > 0, c / np.where(a > 0, a, 1.0), c)
    h = (0.375, 0.25, 0.0625)
    kn, ka = 1.0 / p["sigma_normal"] ** 2, 1.0 / p["sigma_albedo"] ** 2
    for i in range(p["iterations"]):
        s, kc = 1 << i, 4.0 ** i / p["sigma_color"] ** 2
        wsum, esum = np.zeros((H, W)), np.zeros((H, W, 3))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                # q = p + s (dx, dy), where it lies inside the image
                y0, y1 = max(0, -s * dy), min(H, H - s * dy)
                x0, x1 = max(0, -s * dx), min(W, W - s * dx)
                if y0 >= y1 or x0 >= x1:
                    continue
                P = (slice(y0, y1), slice(x0, x1))
                Q = (slice(y0 + s * dy, y1 + s * dy), slice(x0 + s * dx, x1 + s * dx))
                x = (((e[P] - e[Q]) ** 2).sum(-1) * kc + ((n[P] - n[Q]) ** 2).sum(-1) * kn + ((a[P] - a[Q]) ** 2).sum(-1) * ka)
                w = h[abs(dx)] * h[abs(dy)] * np.exp(-x)
                wsum[P] += w
                esum[P] += w[..., None] * e[Q]
        e = esum / wsum[..., None]
    return np.where(a > 0, e * a, e)


def rel_mse(x, ref, eps=1e-2):
    """Relative mean squared error (x - ref)^2 / (ref^2 + eps), averaged over pixels and channels."""
    x, ref = np.asarray(x, np.float64), np.asarray(ref, np.float64)
    return float(np.mean((x - ref) ** 2 / (ref ** 2 + eps)))


def render(scene, w, h, spp, bounces=2):
    """(colour, albedo, normal), each [H, W, 3], of the CPU reference (AovWorld: the oracle with the guide buffers) at spp.
    scene: "landscape" (the synthetic landscape of scene.make_scene, with water) or "garden" (real_scene.make_garden)."""
    from types import SimpleNamespace

    from aov_reference import AovWorld
    from helpers import build_garden_pair, dprt
    if scene == "landscape":
        chunks, mats, lights = dprt.scene.make_scene(1, 20000, water_frac=0.05)
        world = AovWorld(dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=1, proxy_mode=0), 1)
        for c in chunks:
            world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
        world.set_materials(mats); world.set_lights(lights); world.set_camera(dprt.scene.default_camera(w, h))
    else:
        _, world, _ = build_garden_pair(SimpleNamespace(World=AovWorld), 1, w, h, spp=spp, bounces=bounces, gpu=False)
    world.enable_aov()
    img = world.launch()
    a, n = world.aov()
    world.close()
    return img, a, n
