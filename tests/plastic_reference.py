"""CPU reference of the glossy plastic (bsdfType 3, DESIGN.md 3.13) for the tests: tests/plastic_reference.cpp compiled once per
process with the oracle's flags into a temporary directory. The library carries the whole conductor reference (and through it
the oracle and the AOV reference, all included unchanged) plus the plastic, so PlasticWorld is a CondWorld whose launch() /
render_sample() also shade plastics, and sample() / evaluate() are the BSDF on its own."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from conductor_reference import CondWorld
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="plastic_reference_"), "libplasref.so")
        cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
        # the flags of oracle/Makefile: no contraction, hardware fmaf, IEEE semantics
        p = subprocess.run([cxx, "-O3", "-std=c++17", "-fPIC", "-fopenmp", "-march=x86-64-v3", "-ffp-contract=off", "-fno-math-errno",
                            "-I" + os.path.join(ROOT, "include"), "-shared", "-o", out,
                            os.path.join(ROOT, "tests", "plastic_reference.cpp")], capture_output=True, text=True)
        if p.returncode:
            raise RuntimeError("building tests/plastic_reference.cpp failed:\n" + p.stderr[-4000:])
        saved = O._lib, O.LIB_PATH
        try:                                   # the oracle binding's prototypes, bound to this library
            O._lib, O.LIB_PATH = None, out
            L = O.lib()
        finally:
            O._lib, O.LIB_PATH = saved
        L.aov_enable.argtypes = [C.c_void_p, C.c_int]
        L.aov_forget.argtypes = [C.c_void_p]
        L.aov_buffer.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.aov_reduce.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.cond_set_roughness.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.cond_forget.argtypes = [C.c_void_p]
        L.plas_render_sample.argtypes = [C.c_void_p, C.c_int]
        L.plas_launch.argtypes = [C.c_void_p]
        L.plas_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.plas_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _args(albedo, roughness, wo):
    wo = np.ascontiguousarray(wo, np.float32).reshape(-1, 3)
    n = wo.shape[0]
    albedo = np.ascontiguousarray(np.broadcast_to(np.asarray(albedo, np.float32), (n, 3)))
    r = np.ascontiguousarray(np.broadcast_to(np.asarray(roughness, np.float32), (n,)))
    return albedo, r, wo, n


def sample(albedo, roughness, wo, xi):
    """(wi [n, 3], weight [n, 3]) of the plastic's next path for uniforms xi [n, 3]; both 0 where the path ends."""
    albedo, r, wo, n = _args(albedo, roughness, wo)
    x = np.ascontiguousarray(np.broadcast_to(np.asarray(xi, np.float32), (n, 3)))
    wi, wt = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
    assert lib().plas_sample(_p(albedo), _p(r), _p(wo), _p(x), n, _p(wi), _p(wt)) == 0
    return wi, wt


def evaluate(albedo, roughness, wo, wi):
    """f(wi, wo) [n, 3] of the plastic."""
    albedo, r, wo, n = _args(albedo, roughness, wo)
    w = np.ascontiguousarray(np.broadcast_to(np.asarray(wi, np.float32).reshape(-1, 3), (n, 3)))
    out = np.zeros((n, 3), np.float32)
    assert lib().plas_eval(_p(albedo), _p(r), _p(wo), _p(w), n, _p(out)) == 0
    return out


class PlasticWorld(CondWorld):
    """oracle.World with the conductor, the plastic and the AOV reference's guide buffers: set_material_roughness(), then
    launch() / render_sample() shade bsdfType 2 materials by DESIGN.md 3.12 and bsdfType 3 materials by 3.13."""

    def __init__(self, cfg, W=1):
        self.L = lib()
        self.cfg, self.W = cfg, W
        self.N = cfg.width * cfg.height
        self.h = C.c_void_p(self.L.orc_world_create(C.byref(cfg), W))

    def render_sample(self, s):
        assert self.L.plas_render_sample(self.h, s) == 0

    def launch(self):
        assert self.L.plas_launch(self.h) == 0
        return self.image()
