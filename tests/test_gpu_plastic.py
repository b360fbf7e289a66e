"""The glossy plastic (bsdfType 3, DESIGN.md 3.13) on the GPU against the reference (-m gpu): every path record and the image
bit for bit on scenes whose material table mixes Lambertian, water, conductors and plastics of several roughnesses, through
every way a sample is rendered (single-rank bounce, MainRay re-trace, rank groups with and without proxies, samples in
flight, AOVs, the C++ host's DPRTSCN3 scene file, an obj2scene.py --glossy conversion)."""
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from conductor_reference import CondWorld
from helpers import D, assert_bits_equal, assert_records_equal, build_garden_pair, build_pair, dprt
from plastic_reference import PlasticWorld

pytestmark = pytest.mark.gpu
BIN = os.path.join(os.path.dirname(dprt.host.LIB_PATH), "dprt_render")
# material k of the terrain's 16: plastics and conductors of these roughnesses, the rest Lambertian, 15 water
PLASTIC_ROUGH = {2: 1e-4, 3: 0.0, 7: 0.05, 10: 1.0, 11: 0.3}
COND_ROUGH = {1: 0.0, 5: 0.2, 9: 0.6, 13: 1.0}
REF = SimpleNamespace(World=PlasticWorld)  # the oracle with the conductor, the plastic and the guide buffers, tests/plastic_reference.cpp


def _mixed(mats):
    """(materials, roughness table): plastics and conductors on the chosen materials; the Lambertian ones get a roughness too,
    unused."""
    m = np.array(mats, copy=True)
    rough = np.full(len(m), 0.5, np.float32)
    for kind, table in ((3, PLASTIC_ROUGH), (2, COND_ROUGH)):
        for k, r in table.items():
            if k < len(m) and m["bsdfType"][k] == 0:
                m["bsdfType"][k] = kind
                rough[k] = r
    m["baseColor"][3] = [1.3, 0.2, 0.05]               # a diffuse colour with a channel above 1
    return m, rough


def _apply(targets, mats, rough):
    for t in targets:
        t.set_materials(mats)
        t.set_material_roughness(rough)


def _terrain(W, tris, w, h, *, spp=2, bounces=3, water=0.03, **kw):
    rs, world, _ = build_pair(REF, W, tris, w, h, spp=spp, bounces=bounces, water_frac=water, **kw)
    m, rough = _mixed(dprt.scene.make_materials(16, water_last=water > 0))      # the table build_pair set
    assert (m["bsdfType"] == 3).sum() == len(PLASTIC_ROUGH)
    _apply(rs + [world], m, rough)
    return rs, world, m


def _lambert(m):
    lam = np.array(m, copy=True)
    lam["bsdfType"][lam["bsdfType"] == 3] = 0
    return lam


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
    # the plastics are visible: the same scene with them Lambertian renders differently
    R.set_materials(_lambert(m))
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


def _garden_plastics(g):
    """The textured materials become plastics (diffuse colour from the texel) but the last, a conductor (F0 from the texel); an
    untextured one becomes a smooth plastic."""
    m = np.array(g["materials"], copy=True)
    mt = np.asarray(g["material_textures"])
    rough = np.zeros(len(m), np.float32)
    tex = [k for k in range(len(m)) if k < mt.size and mt[k] >= 0 and m["bsdfType"][k] == 0]
    plain = [k for k in range(len(m)) if k not in tex and m["bsdfType"][k] == 0]
    assert len(tex) >= 2 and plain
    for k in tex[:-1]:
        m["bsdfType"][k] = 3; rough[k] = 0.3
    m["bsdfType"][tex[-1]] = 2; rough[tex[-1]] = 0.2
    m["bsdfType"][plain[0]] = 3
    return m, rough


def test_textured_garden_bit_exact(gpu_required, oracle):
    rs, world, g = build_garden_pair(REF, 1, 192, 108, spp=2, bounces=3)
    m, rough = _garden_plastics(g)
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


def test_aov_albedo_is_the_diffuse_colour(gpu_required, oracle):
    rs, world, m = _terrain(1, 20000, 128, 72, spp=2, bounces=2)
    R = rs[0]
    R.enable_aov(); world.enable_aov()
    assert_bits_equal(R.launch(), world.launch(), "image")
    aov = R.download(D.BUF_AOV, 6 * R.N)
    assert_bits_equal(aov, world.aov_buffer(0), "AOV buffer")
    assert world.aov_buffer(0)[:3 * R.N].max() > 0
    # the first hits do not depend on the BSDF: the guides equal those of the scene with its plastics Lambertian
    R.set_materials(_lambert(m))
    R.launch()
    assert_bits_equal(R.download(D.BUF_AOV, 6 * R.N), aov, "AOV buffer, plastics as Lambertian")


def test_full_hd_bit_exact(gpu_required, oracle):
    rs, world, _ = _terrain(1, 200000, 1920, 1080, spp=1, bounces=3)
    R = rs[0]
    assert_bits_equal(R.launch(), world.launch(), "1080p image")
    _check_rank(R, world, 0, "1080p")


def _render(scene, out, spp, bounces, W):
    p = subprocess.run([BIN, "--scene", scene, "--out", out, "--spp", str(spp), "--bounces", str(bounces), "--world", str(W)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    return dprt.scene.load_pfm(out).reshape(-1)


@pytest.mark.parametrize("W", [1, 2])
def test_dprt_render_scene_file_v3(gpu_required, oracle, tmp_path, W):
    w, h, spp, bounces = 160, 90, 2, 3
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W, path_gen_mode=1 if W > 1 else 0)
    _, _, g = build_garden_pair(REF, W, w, h, spp=spp, bounces=bounces, gpu=False)
    m, rough = _garden_plastics(g)
    world = PlasticWorld(cfg, W)
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
    assert_bits_equal(_render(scene, out, spp, bounces, W), np.asarray(img_o, np.float32).reshape(-1), f"dprt_render DPRTSCN3, W={W}")


def test_dprt_render_obj2scene_glossy(gpu_required, oracle, tmp_path, monkeypatch):
    """An OBJ + MTL with metallic, specular, water and plain materials through obj2scene.py --glossy and dprt_render, against
    the reference world built from what the converter wrote."""
    from test_plastic_cpu import obj2scene, write_glossy_obj
    o2s = obj2scene()
    seen, save = {}, o2s.RS.save_scene_v2

    def keep(path, garden, cam, flatten):
        seen.update(garden=garden, cam=cam)
        save(path, garden, cam, flatten)
    monkeypatch.setattr(o2s.RS, "save_scene_v2", keep)
    w, h, spp, bounces, W = 128, 72, 2, 3, 2
    scene, out = str(tmp_path / "glossy.dprt"), str(tmp_path / "glossy.pfm")
    o2s.convert(write_glossy_obj(tmp_path), scene, world=W, width=w, height=h, glossy=True)
    g, cam = seen["garden"], seen["cam"]
    kinds = g["materials"]["bsdfType"].tolist()
    assert 3 in kinds and 2 in kinds and 1 in kinds and 0 in kinds
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W, path_gen_mode=1)
    world = PlasticWorld(cfg, W)
    for ob in g["objects"]:
        v, n, uv, mids = ob.flat
        world.add_object_uv(ob.index, ob.desc(False), v, n, uv, mids)
    world.set_materials(g["materials"]); world.set_material_roughness(g["material_roughness"])
    world.set_lights(g["lights"]); world.set_camera(cam)
    for slot, t in g["textures"].items():
        world.set_texture(slot, t)
    world.set_material_textures(g["material_textures"])
    img_o = np.asarray(world.launch(), np.float32).reshape(-1)
    img_g = _render(scene, out, spp, bounces, W)
    assert_bits_equal(img_g, img_o, "dprt_render on an obj2scene.py --glossy conversion")
    assert np.isfinite(img_g).all() and img_g.max() > 0


def test_scene_without_plastics_unchanged(gpu_required, oracle):
    """A scene with conductors and no plastic renders as the conductor's own reference does, and roughness entries of its
    Lambertian and water materials change nothing."""
    rs, world, _ = build_pair(SimpleNamespace(World=CondWorld), 1, 20000, 128, 72, spp=2, bounces=3, water_frac=0.03)
    m, rough = _mixed(dprt.scene.make_materials(16, water_last=True))
    m = _lambert(m)
    _apply(rs + [world], m, rough)
    R = rs[0]
    img = R.launch()
    assert_bits_equal(img, world.launch(), "image against the conductor reference")
    _check_rank(R, world, 0, "no plastics")
    rough[m["bsdfType"] != 2] = 0.05
    R.set_material_roughness(rough)
    assert_bits_equal(R.launch(), img, "image with other roughness on bsdfType 0 / 1 materials")
