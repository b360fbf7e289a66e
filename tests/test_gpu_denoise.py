"""The denoiser on the GPU (-m gpu): bit for bit what the specification's host compile computes (dprt.spec_denoise), and
end to end on the reduced frame and guide buffers against the CPU reference (tests/denoise_reference.cpp applied to the
oracle's image and AOVs).

The reduced frames are compared by value, as in test_gpu_aov.py: the reference sums the ranks starting from +0, so a -0 of a
single rank may come back as +0 on one side.
"""
import os
import subprocess

import numpy as np
import pytest

import denoise_reference as DR
from aov_reference import AovWorld
from helpers import D, assert_bits_equal, build_pair, dprt
from test_denoise_cpu import frame
from test_gpu_aov import REF, _assert_value_equal

pytestmark = pytest.mark.gpu
BIN = os.path.join(os.path.dirname(dprt.host.LIB_PATH), "dprt_render")
DPRT_ERR_INVALID = -1


@pytest.fixture(scope="module")
def renderer(gpu_required):
    R = dprt.Renderer(dprt.make_config(16, 16, scene_size=1, proxy_mode=0))
    yield R
    R.close()


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160), (1, 1), (7, 3), (333, 177)])
def test_gpu_equals_spec_bitwise(renderer, w, h):
    """Tile edges (32 x 8 tiles) and image borders: the odd sizes leave partial tiles on both axes."""
    c, a, n = frame(w, h, seed=w * 7919 + h)
    for it in (1, 5, 10):
        assert_bits_equal(renderer.denoise(c, a, n, iterations=it), dprt.spec_denoise(c, a, n, iterations=it), f"{w}x{h}, {it} iterations")
    p = {"iterations": 4, "sigma_color": 8.0, "sigma_normal": 3.0, "sigma_albedo": 1.0}
    assert_bits_equal(renderer.denoise(c, a, n, **p), dprt.spec_denoise(c, a, n, **p), f"{w}x{h}, wide sigmas")


def test_device_variant_and_aliased_output(renderer):
    R = renderer
    w, h = 333, 177
    c, a, n = frame(w, h, seed=3)
    want = R.denoise(c, a, n)
    nbytes = c.nbytes
    bufs = [R.device_alloc(nbytes) for _ in range(4)]
    try:
        for b, x in zip(bufs, (c, a, n)):
            R.h2d(b, x)
        R.denoise_device(w, h, bufs[0], bufs[1], bufs[2], bufs[3])
        got = np.zeros_like(c)
        R.d2h(got, bufs[3])
        assert_bits_equal(got, want, "dprt_denoise_device")
        R.denoise_device(w, h, bufs[0], bufs[1], bufs[2], bufs[0])          # the output over the colour input
        R.d2h(got, bufs[0])
        assert_bits_equal(got, want, "dprt_denoise_device, output aliasing the colour")
        p = D.DenoiseParams(iterations=10, sigma_color=0.5, sigma_normal=0.25, sigma_albedo=0.05)
        R.h2d(bufs[0], c)
        R.denoise_device(w, h, bufs[0], bufs[1], bufs[2], bufs[3], p)
        R.d2h(got, bufs[3])
        assert_bits_equal(got, dprt.spec_denoise(c, a, n, iterations=10, sigma_color=0.5, sigma_normal=0.25, sigma_albedo=0.05), "params")
    finally:
        for b in bufs:
            R.device_free(b)


def test_end_to_end_single_rank(gpu_required, oracle):
    rs, world, _ = build_pair(REF, 1, 20000, 128, 72, spp=4, bounces=2, water_frac=0.05)
    R = rs[0]
    R.enable_aov(); world.enable_aov()
    img = R.launch()
    a, n = R.reduce_aov(0)
    img_o = world.launch()
    a_o, n_o = world.aov()
    _assert_value_equal(img, img_o, "image")
    got = R.denoise(img, a, n)
    want = DR.denoise(img_o, a_o, n_o)
    _assert_value_equal(got, want, "denoised frame")
    assert DR.rel_mse(got, img) > 0, "the denoiser changed nothing"


def test_end_to_end_rank_group(gpu_required, oracle):
    rs, world, _ = build_pair(REF, 2, 6000, 128, 72, spp=2, bounces=2)
    G = dprt.RankGroup(rs)
    G.enable_aov(); world.enable_aov()
    img = G.launch()
    a, n = G.reduce_aov(0)
    img_o = world.launch()
    a_o, n_o = world.aov()
    _assert_value_equal(img, img_o, "image")
    _assert_value_equal(rs[0].denoise(img, a, n), DR.denoise(img_o, a_o, n_o), "denoised frame, two ranks")


def test_no_side_effects(gpu_required, oracle):
    rs, _, _ = build_pair(REF, 1, 20000, 96, 54, spp=2, bounces=2)
    R = rs[0]
    R.enable_aov()
    img1 = R.launch()
    buf1 = R.download(D.BUF_AOV, 6 * R.N)
    a, n = R.reduce_aov(0)
    keep = [x.copy() for x in (img1, a, n)]
    R.denoise(img1, a, n)
    R.denoise(img1, a, n, iterations=10)
    for x, k, what in zip((img1, a, n), keep, ("colour", "albedo", "normal")):
        assert_bits_equal(x, k, f"{what} input after denoise")
    img2 = R.launch()
    assert_bits_equal(img2, img1, "image of a launch after denoise")
    assert_bits_equal(R.download(D.BUF_AOV, 6 * R.N), buf1, "AOV buffer of a launch after denoise")


@pytest.mark.parametrize("W", [1, 2])
def test_dprt_render_denoise(gpu_required, oracle, tmp_path, W):
    tris, w, h, spp, bounces = 8000, 160, 90, 2, 2
    chunks, mats, lights = dprt.scene.make_scene(W, tris, water_frac=0.02)
    cam = dprt.scene.default_camera(w, h)
    scene = str(tmp_path / "scene.dprt")
    dprt.scene.save_scene(scene, chunks, mats, lights, cam)
    cmd = [BIN, "--scene", scene, "--spp", str(spp), "--bounces", str(bounces), "--frames", "2", "--world", str(W)]
    p = subprocess.run(cmd + ["--out", str(tmp_path / "img.exr"), "--denoise", "1"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    p = subprocess.run(cmd + ["--out", str(tmp_path / "plain.exr")], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W, path_gen_mode=1 if W > 1 else 0)
    world = AovWorld(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
    world.set_materials(mats); world.set_lights(lights); world.set_camera(cam)
    world.enable_aov()
    img_o = world.launch()
    want = DR.denoise(img_o, *world.aov())
    files = sorted(os.listdir(tmp_path))
    for f in range(2):
        _assert_value_equal(dprt.scene.load_exr(str(tmp_path / f"{f}img.exr")), img_o, f"frame {f} image")
        _assert_value_equal(dprt.scene.load_exr(str(tmp_path / f"{f}img.denoised.exr")), want, f"frame {f} denoised")
        assert f"{f}img.albedo.exr" not in files, "guide buffers written without --aov 1"
        assert (tmp_path / f"{f}plain.exr").read_bytes() == (tmp_path / f"{f}img.exr").read_bytes()
    assert not [x for x in files if "plain" in x and x.endswith(".denoised.exr")], "a .denoised file without --denoise"


def test_rejected_arguments(renderer):
    R = renderer
    lib = R.lib
    c, a, n = frame(8, 4, 1)
    o = np.zeros_like(c)
    ptr = lambda x: None if x is None else x.ctypes.data_as(dprt.host.C.c_void_p)
    P = lambda **kw: dprt.host.C.byref(D.DenoiseParams(**{**D.DENOISE_DEFAULTS, **kw}))
    assert lib.dprt_denoise(None, None, 8, 4, ptr(c), ptr(a), ptr(n), ptr(o)) == DPRT_ERR_INVALID
    cases = [(None, 0, 4, (c, a, n, o)), (None, 8, -2, (c, a, n, o)), (None, 1 << 15, 1 << 14, (c, a, n, o)),
             (P(iterations=0), 8, 4, (c, a, n, o)), (P(iterations=11), 8, 4, (c, a, n, o)), (P(sigma_color=0.0), 8, 4, (c, a, n, o)),
             (P(sigma_albedo=float("nan")), 8, 4, (c, a, n, o)), (P(sigma_color=1e-17, iterations=10), 8, 4, (c, a, n, o)),
             (None, 8, 4, (c, None, n, o)), (None, 8, 4, (c, a, n, None))]
    for p, w, h, arrs in cases:
        assert lib.dprt_denoise(R.h, p, w, h, *[ptr(x) for x in arrs]) == DPRT_ERR_INVALID, (w, h, arrs is None)
        assert lib.dprt_last_error(R.h).startswith(b"dprt_denoise")
        assert lib.dprt_denoise_device(R.h, p, w, h, *[ptr(x) for x in arrs]) == DPRT_ERR_INVALID
    with pytest.raises(dprt.DprtError):
        R.denoise(c, a, n, sigma_normal=-1.0)
    assert_bits_equal(R.denoise(c, a, n), dprt.spec_denoise(c, a, n), "a valid call after the rejected ones")
