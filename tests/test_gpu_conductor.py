"""The rough conductor (bsdfType 2, DESIGN.md 3.12) on the GPU against the oracle (-m gpu): every path record and the image
bit for bit on scenes whose material table mixes Lambertian, water and conductors of several roughnesses, through every way
a sample is rendered (single-rank bounce, MainRay re-trace, rank groups with and without proxies, samples in flight, AOVs,
the C++ host's DPRTSCN3 scene file)."""
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from conductor_reference import CondWorld
from helpers import D, assert_bits_equal, assert_records_equal, build_garden_pair, build_pair, dprt

pytestmark = pytest.mark.gpu
BIN = os.path.join(os.path.dirname(dprt.host.LIB_PATH), "dprt_render")
# material k of the terrain's 16: odd k are conductors of these roughnesses, even k stay Lambertian, 15 is water
COND_ROUGH = {1: 0.0, 3: 1e-4, 5: 0.05, 7: 0.2, 9: 0.3, 11: 0.6, 13: 1.0}
REF = SimpleNamespace(World=CondWorld)     # the oracle with the conductor (and the guide buffers) on top, tests/conductor_reference.cpp


def _mixed(mats):
    """(materials, roughness table): conductors on the odd materials; the Lambertian ones get a roughness too, unused."""
    m = np.array(mats, copy=True)
    rough = np.full(len(m), 0.5, np.float32)
    for k, r in COND_ROUGH.items():
        if k < len(m) and m["bsdfType"][k] == 0:
            m["bsdfType"][k] = 2
            m["baseColor"][k] = [0.95, 0.64, 0.54] if k % 4 == 1 else m["baseColor"][k]
            rough[k] = r
    return m, rough


def _apply(targets, mats, rough):
    for t in targets:
        t.set_materials(mats)
        t.set_material_roughness(rough)


def _terrain(W, tris, w, h, *, spp=2, bounces=3, water=0.03, **kw):
    rs, world, _ = build_pair(REF, W, tris, w, h, spp=spp, bounces=bounces, water_frac=water, **kw)
    m, rough = _mixed(dprt.scene.make_materials(16, water_last=water > 0))      # the table build_pair set
    _apply(rs + [world], m, rough)
    return rs, world, m


def _check_rank(R, world, r, what):
    n = R.path_size
    assert n == world.path_size(r), f"{what}: rank {r} pathSize"
    tot = n * (1 + R.cfg.shadowPathCount)
    assert_records_equal(R.download(D.BUF_PATHS, tot), world.download(r, D.BUF_PATHS, tot), f"{what}: rank {r} paths + shadow paths")
    direct = R.download(D.BUF_DIRECT)
    assert_bits_equal(direct, world.download(r, D.BUF_DIRECT, direct.size), f"{what}: rank {r} direct")
    assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * R.N), f"{what}: rank {r} env")


@pytest.mark.parametrize("shortcut,retrace", [("1", 0), ("0", 0), ("1", 1), ("0", 1)])
def test_single_rank_bit_exact(gpu_required, oracle, monkeypatch, shortcut, retrace):
    monkeypatch.setenv("DPRT_SINGLE_RANK_SHORTCUT", shortcut)
    rs, world, m = _terrain(1, 30000, 256, 144, main_ray_retrace=retrace)
    R = rs[0]
    img_g, img_o = R.launch(), world.launch()
    assert_bits_equal(img_g, img_o, f"image, shortcut={shortcut} retrace={retrace}")
    _check_rank(R, world, 0, f"shortcut={shortcut} retrace={retrace}")
    assert np.isfinite(img_g).all() and img_g.max() > 0
    # the conductors are visible: the same scene all-Lambertian renders differently
    lam = np.array(m, copy=True); lam["bsdfType"][lam["bsdfType"] == 2] = 0
    R.set_materials(lam)
    assert not np.array_equal(R.launch(), img_g)


@pytest.mark.parametrize("proxy,path_gen_mode", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_rank_group_bit_exact(gpu_required, oracle, proxy, path_gen_mode):
    W = 2
    models = None
    if proxy:
        from test_gpu_proxy import _models
        models = _models(W, False)
    rs, world, _ = _terrain(W, 6000, 128, 72, spp=1, bounces=2, proxy_mode=proxy, path_gen_mode=path_gen_mode,
                            models=models, mlp_dtype=1)
    G = dprt.RankGroup(rs)
    for R in rs:
        R.reset_frame()
    world.reset_frame()
    G.run_sample(0)
    world.render_sample(0)
    for r, R in enumerate(rs):
        _check_rank(R, world, r, f"proxy={proxy} pathGen={path_gen_mode}")
    img_g, img_o = G.launch(), world.launch()
    assert_bits_equal(img_g, img_o, f"group image, proxy={proxy} pathGen={path_gen_mode}")


def _garden_conductors(g):
    """Every textured material becomes a conductor (F0 from the texel), plus one untextured mirror."""
    m = np.array(g["materials"], copy=True)
    mt = np.asarray(g["material_textures"])
    rough = np.zeros(len(m), np.float32)
    tex = [k for k in range(len(m)) if k < mt.size and mt[k] >= 0 and m["bsdfType"][k] == 0]
    plain = [k for k in range(len(m)) if k not in tex and m["bsdfType"][k] == 0]
    assert tex and plain
    for k in tex:
        m["bsdfType"][k] = 2; rough[k] = 0.3
    m["bsdfType"][plain[0]] = 2
    return m, rough


def test_textured_garden_bit_exact(gpu_required, oracle):
    rs, world, g = build_garden_pair(REF, 1, 192, 108, spp=2, bounces=3)
    m, rough = _garden_conductors(g)
    _apply(rs + [world], m, rough)
    R = rs[0]
    img_g, img_o = R.launch(), world.launch()
    assert_bits_equal(img_g, img_o, "garden image")
    _check_rank(R, world, 0, "garden")


def test_samples_in_flight_bit_exact(gpu_required, oracle):
    from test_gpu_inflight import _check_contexts, _context_state, predict_inflight
    rs, world, _ = _terrain(1, 20000, 160, 90, spp=5, bounces=3)
    R, K = rs[0], 3
    F = dprt.SamplesInFlight(R, K)                 # the contexts adopt the scene, roughness table included
    try:
        P = predict_inflight(world, K, [(0, 5)])
        before = [X.stats() for X in F.ctxs]
        F.reset_frame()
        F.run_samples(0, 5)
        _check_contexts(_context_state(F), P, 0, before=before)
        F.accumulate()
        R.synchronize()
        assert_bits_equal(R.reduce_image(0), P["image"], "reduce_image after accumulate")
    finally:
        F.close(); R.close(); world.close()


def test_aov_albedo_is_f0(gpu_required, oracle):
    rs, world, _ = _terrain(1, 20000, 128, 72, spp=2, bounces=2)
    R = rs[0]
    R.enable_aov(); world.enable_aov()
    assert_bits_equal(R.launch(), world.launch(), "image")
    assert_bits_equal(R.download(D.BUF_AOV, 6 * R.N), world.aov_buffer(0), "AOV buffer")
    assert world.aov_buffer(0)[:3 * R.N].max() > 0


def test_full_hd_bit_exact(gpu_required, oracle):
    rs, world, _ = _terrain(1, 200000, 1920, 1080, spp=1, bounces=3)
    R = rs[0]
    assert_bits_equal(R.launch(), world.launch(), "1080p image")
    _check_rank(R, world, 0, "1080p")


@pytest.mark.parametrize("W", [1, 2])
def test_dprt_render_scene_file_v3(gpu_required, oracle, tmp_path, W):
    w, h, spp, bounces = 160, 90, 2, 3
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W, path_gen_mode=1 if W > 1 else 0)
    _, _, g = build_garden_pair(REF, W, w, h, spp=spp, bounces=bounces, gpu=False)
    m, rough = _garden_conductors(g)
    world = CondWorld(cfg, W)
    for ob in g["objects"]:
        world.add_instanced_object(ob.index, ob.desc(False), ob.meshes, ob.instances)
    world.set_materials(m); world.set_material_roughness(rough)
    world.set_lights(g["lights"]); world.set_camera(dprt.scene.default_camera(w, h))
    for slot, t in g["textures"].items():
        world.set_texture(slot, t)
    world.set_material_textures(g["material_textures"]); world.set_env_map(g["env_map"], g["env_rotation"])
    img_o = world.launch()
    g = dict(g, materials=m, material_roughness=rough)
    scene, out = str(tmp_path / "garden3.dprt"), str(tmp_path / "garden3.pfm")
    dprt.real_scene.save_scene_v2(scene, g, dprt.scene.default_camera(w, h), dprt.flatten_instances)
    with open(scene, "rb") as f:
        assert f.read(8) == b"DPRTSCN3"
    p = subprocess.run([BIN, "--scene", scene, "--out", out, "--spp", str(spp), "--bounces", str(bounces), "--world", str(W)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    assert_bits_equal(dprt.scene.load_pfm(out).reshape(-1), np.asarray(img_o, np.float32).reshape(-1), f"dprt_render DPRTSCN3, W={W}")


def test_rejected_roughness_changes_nothing(gpu_required, oracle):
    rs, world, _ = _terrain(1, 20000, 128, 72, spp=1, bounces=2)
    R = rs[0]
    img = R.launch()
    assert_bits_equal(img, world.launch(), "image before the rejected calls")
    good = np.full(16, 0.25, np.float32)
    for bad in (np.zeros(0, np.float32), np.zeros(D.MAX_MATERIALS + 1, np.float32),
                np.where(np.arange(16) == 3, np.nan, good).astype(np.float32),
                np.where(np.arange(16) == 5, np.inf, good).astype(np.float32),
                np.where(np.arange(16) == 7, -0.1, good).astype(np.float32),
                np.where(np.arange(16) == 9, 1.5, good).astype(np.float32),
                np.where(np.arange(16) == 0, -np.inf, good).astype(np.float32)):
        with pytest.raises(dprt.DprtError):
            R.set_material_roughness(bad)
        assert_bits_equal(R.launch(), img, f"image after rejecting {bad[:10]}")


def test_roughness_on_lambert_and_water_changes_nothing(gpu_required, oracle):
    rs, world, _ = build_pair(oracle, 1, 20000, 128, 72, spp=2, bounces=3, water_frac=0.05)
    R = rs[0]
    img = R.launch()
    assert_bits_equal(img, world.launch(), "image without a roughness table")
    R.set_material_roughness(np.linspace(0.0, 1.0, D.MAX_MATERIALS, dtype=np.float32))
    assert_bits_equal(R.launch(), img, "image with a roughness table on bsdfType 0 / 1 materials")
