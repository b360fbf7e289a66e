"""First-hit guide buffers (AOVs: albedo and shading normal of the camera paths' first hits) on the GPU against the oracle (-m gpu).

Per rank the buffer must carry the oracle's bits: the albedo and normal come from the same binary32 arithmetic as the
shading program, and each pixel's sum over samples is taken in sample order. The reduced frame result is compared by
value: the reference sums the ranks starting from +0, so a -0 of a single rank comes back as +0. The reference is the oracle
with the AOV rule on top (tests/aov_reference.cpp).
"""
import ctypes as C
import os
import socket
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from aov_reference import AovWorld
from helpers import D, assert_bits_equal, assert_records_equal, build_garden_pair, build_pair, dprt

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(os.path.dirname(dprt.host.LIB_PATH), "dprt_render")
DPRT_ERR_STATE = -5
SPP, BOUNCES = 2, 2
REF = SimpleNamespace(World=AovWorld)      # what build_pair / build_garden_pair need of an oracle module


def _aov_buf(R):
    return R.download(D.BUF_AOV, 6 * R.N)


def _assert_value_equal(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    bad = np.nonzero(a.reshape(-1) != b.reshape(-1))[0]
    assert bad.size == 0, f"{what}: {bad.size} values differ; first at {bad[0]}: gpu={a.reshape(-1)[bad[0]]!r} oracle={b.reshape(-1)[bad[0]]!r}"


def _check_reduced(got, world, what):
    a_o, n_o = world.aov()
    _assert_value_equal(got[0], a_o, f"{what}: reduced albedo")
    _assert_value_equal(got[1], n_o, f"{what}: reduced normal")
    assert a_o.max() > 0 and np.abs(n_o).max() > 0, f"{what}: empty AOVs"


@pytest.mark.parametrize("shortcut,water", [("1", 0.0), ("0", 0.0), ("1", 0.05)])
def test_single_rank_aov_bit_exact(gpu_required, oracle, monkeypatch, shortcut, water):
    """Single-rank bounce (shade from the partition output with cached hits) on and off, and water materials."""
    monkeypatch.setenv("DPRT_SINGLE_RANK_SHORTCUT", shortcut)
    rs, world, _ = build_pair(REF, 1, 20000, 128, 72, spp=SPP, bounces=BOUNCES, water_frac=water)
    R = rs[0]
    R.enable_aov(); world.enable_aov()
    img_g, img_o = R.launch(), world.launch()
    assert_bits_equal(img_g, img_o, "image")
    assert_bits_equal(_aov_buf(R), world.aov_buffer(0), f"AOV buffer, shortcut={shortcut} water={water}")
    _check_reduced(R.reduce_aov(0), world, f"shortcut={shortcut} water={water}")
    if shortcut == "1":
        assert R.stats()["rays_shade_cached"] > 0, "the single-rank bounce did not run"


@pytest.mark.parametrize("proxy,path_gen_mode", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_rank_group_aov_bit_exact(gpu_required, oracle, proxy, path_gen_mode):
    """W = 2 in one process: the first hit of a camera path may be shaded on either rank, after migrating there."""
    W = 2
    models = None
    if proxy:
        from test_gpu_proxy import _models
        models = _models(W, False)
    rs, world, _ = build_pair(REF, W, 6000, 128, 72, spp=SPP, bounces=BOUNCES, proxy_mode=proxy, path_gen_mode=path_gen_mode,
                              models=models, mlp_dtype=1)
    G = dprt.RankGroup(rs)
    G.enable_aov(); world.enable_aov()
    img_g, img_o = G.launch(), world.launch()
    assert_bits_equal(img_g, img_o, "image")
    for r, R in enumerate(rs):
        g = _aov_buf(R)
        assert_bits_equal(g, world.aov_buffer(r), f"rank {r} AOV buffer, proxy={proxy} pathGen={path_gen_mode}")
        assert g.any(), f"rank {r} shaded no first hit: the scene does not split the view"
    _check_reduced(G.reduce_aov(0), world, f"group proxy={proxy} pathGen={path_gen_mode}")


def test_garden_aov_albedo_from_textures(gpu_required, oracle):
    rs, world, g = build_garden_pair(REF, 1, 96, 54, spp=1, bounces=1)
    R = rs[0]
    R.enable_aov(); world.enable_aov()
    R.launch(); world.launch()
    assert_bits_equal(_aov_buf(R), world.aov_buffer(0), "garden AOV buffer")
    got = R.reduce_aov(0)
    _check_reduced(got, world, "garden")
    albedo = got[0]
    base = {tuple(c) for c in np.asarray(g["materials"]["baseColor"], np.float32).tolist()} | {(0.0, 0.0, 0.0)}
    texel = [tuple(c) not in base for c in albedo.reshape(-1, 3).tolist()]
    assert sum(texel) > albedo.shape[0] * albedo.shape[1] // 10, "albedo does not come from the textures"


def test_samples_in_flight_aov(gpu_required, oracle):
    spp = 6
    rs, world, _ = build_pair(REF, 1, 20000, 128, 72, spp=spp, bounces=BOUNCES)
    R = rs[0]
    R.enable_aov(); world.enable_aov()
    R.launch(); world.launch()
    a1, n1 = R.reduce_aov(0)
    _check_reduced((a1, n1), world, "K = 1")
    F = dprt.SamplesInFlight(R, 3)
    try:
        F.enable_aov()
        F.launch()
        a3, n3 = F.reduce_aov(0)
        for x3, x1, what in ((a3, a1, "albedo"), (n3, n1, "normal")):
            err = np.abs(x3 - x1).max() / max(1e-30, float(np.abs(x1).max()))
            assert err <= 1e-6, f"{what} with three samples in flight: {err}"     # the sum over samples in another order
        F.ctxs[1].enable_aov(False)
        assert R.lib.dprt_accumulate_from(R.h, F.ctxs[1].h) == DPRT_ERR_STATE
        assert b"only one" in R.lib.dprt_last_error(R.h)
        assert F.ctxs[1].lib.dprt_accumulate_from(F.ctxs[1].h, R.h) == DPRT_ERR_STATE
    finally:
        F.close()


def test_aov_off_by_default_and_colour_unchanged(gpu_required, oracle):
    rs, world, _ = build_pair(REF, 1, 20000, 128, 72, spp=SPP, bounces=BOUNCES, water_frac=0.05)
    R = rs[0]
    nbytes = C.c_size_t(1)
    assert R.lib.dprt_buffer_bytes(R.h, D.BUF_AOV, C.byref(nbytes)) == 0 and nbytes.value == 0
    with pytest.raises(dprt.DprtError):
        R.reduce_aov(0)
    grp = dprt.RankGroup(rs)
    with pytest.raises(dprt.DprtError):
        grp.reduce_aov(0)
    tot = R.N * (1 + R.cfg.shadowPathCount)
    img_off = R.launch()
    paths_off = R.download(D.BUF_PATHS, tot)
    R.enable_aov()
    img_on = R.launch()
    assert_bits_equal(img_on, img_off, "image, AOVs on vs off")
    assert_records_equal(R.download(D.BUF_PATHS, tot), paths_off, "path records after the frame, AOVs on vs off")
    world.enable_aov()
    world.launch()
    _check_reduced(R.reduce_aov(0), world, "second frame (reset_frame cleared the sums)")


def test_dprt_render_aov_exr(gpu_required, oracle, tmp_path):
    W, tris, w, h, spp, bounces = 1, 8000, 160, 90, 2, 2
    chunks, mats, lights = dprt.scene.make_scene(W, tris, water_frac=0.02)
    cam = dprt.scene.default_camera(w, h)
    scene = str(tmp_path / "scene.dprt")
    dprt.scene.save_scene(scene, chunks, mats, lights, cam)
    out = str(tmp_path / "img.exr")
    p = subprocess.run([BIN, "--scene", scene, "--out", out, "--spp", str(spp), "--bounces", str(bounces), "--frames", "2", "--aov", "1"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W)
    world = AovWorld(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
    world.set_materials(mats); world.set_lights(lights); world.set_camera(cam)
    world.enable_aov()
    img_o = world.launch()
    a_o, n_o = world.aov()
    for f in range(2):
        _assert_value_equal(dprt.scene.load_exr(str(tmp_path / f"{f}img.exr")), img_o, f"frame {f} image")
        _assert_value_equal(dprt.scene.load_exr(str(tmp_path / f"{f}img.albedo.exr")), a_o, f"frame {f} albedo")
        _assert_value_equal(dprt.scene.load_exr(str(tmp_path / f"{f}img.normal.exr")), n_o, f"frame {f} normal")


def test_nccl_reduce_aov_two_processes(gpu_required):
    """The ncclReduce branch of dprt_reduce_aov: one process per GPU (tests/mgpu_aov_check.py)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, {torch.cuda.device_count()} visible")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_aov_check.py")]
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "MGPU_AOV_CHECK_OK" in p.stdout, p.stdout[-2000:] + p.stderr[-4000:]
