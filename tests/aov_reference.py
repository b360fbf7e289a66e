"""CPU reference of the first-hit guide buffers (AOVs) for the tests: tests/aov_reference.cpp compiled once per process
with the oracle's flags into a temporary directory. The library carries the whole oracle (oracle/oracle.cpp, included
unchanged) plus the AOV rule, so AovWorld is an oracle World whose launch() also fills the guide buffers."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="aov_reference_"), "libaovref.so")
        cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
        # the flags of oracle/Makefile: no contraction, hardware fmaf, IEEE semantics
        p = subprocess.run([cxx, "-O3", "-std=c++17", "-fPIC", "-fopenmp", "-march=x86-64-v3", "-ffp-contract=off", "-fno-math-errno",
                            "-I" + os.path.join(ROOT, "include"), "-shared", "-o", out, os.path.join(ROOT, "tests", "aov_reference.cpp")],
                           capture_output=True, text=True)
        if p.returncode:
            raise RuntimeError("building tests/aov_reference.cpp failed:\n" + p.stderr[-4000:])
        saved = O._lib, O.LIB_PATH
        try:                                   # the oracle binding's prototypes, bound to this library
            O._lib, O.LIB_PATH = None, out
            L = O.lib()
        finally:
            O._lib, O.LIB_PATH = saved
        L.aov_enable.argtypes = [C.c_void_p, C.c_int]
        L.aov_forget.argtypes = [C.c_void_p]
        L.aov_render_sample.argtypes = [C.c_void_p, C.c_int]
        L.aov_launch.argtypes = [C.c_void_p]
        L.aov_buffer.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.aov_reduce.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class AovWorld(O.World):
    """oracle.World with the guide buffers: enable_aov(), then launch() / render_sample() add the first hits."""

    def __init__(self, cfg, W=1):
        self.L = lib()
        self.cfg, self.W = cfg, W
        self.N = cfg.width * cfg.height
        self.h = C.c_void_p(self.L.orc_world_create(C.byref(cfg), W))

    def close(self):
        if self.h:
            self.L.aov_forget(self.h)
        super().close()

    def enable_aov(self, enable=True):
        assert self.L.aov_enable(self.h, int(enable)) == 0

    def render_sample(self, s):
        assert self.L.aov_render_sample(self.h, s) == 0

    def launch(self):
        assert self.L.aov_launch(self.h) == 0
        return self.image()

    def aov_buffer(self, rank=0):
        """rank's 6N sums, the layout of DPRT_BUF_AOV."""
        out = np.zeros(6 * self.N, np.float32)
        assert self.L.aov_buffer(self.h, rank, out.ctypes.data_as(C.c_void_p)) == 0, "AOVs are not enabled"
        return out

    def aov(self):
        """(albedo, normal), each [H, W, 3]: per rank sum / spp, summed over the ranks in rank order."""
        a = np.zeros((self.cfg.height, self.cfg.width, 3), np.float32)
        n = np.zeros((self.cfg.height, self.cfg.width, 3), np.float32)
        assert self.L.aov_reduce(self.h, a.ctypes.data_as(C.c_void_p), n.ctypes.data_as(C.c_void_p)) == 0, "AOVs are not enabled"
        return a, n
