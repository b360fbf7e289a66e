"""Instanced objects flattened, built and moved on the GPU (-m gpu; DESIGN.md 3.11): dprt_build_instanced_chunk against the GPU
build of the host-flattened arrays and its host twin, dprt_update_instances against the host refit of the host-flattened moved
instances, and renders against oracle worlds built from the host-flattened arrays. Everything is bit for bit."""
import ctypes as C

import numpy as np
import pytest

from helpers import D, assert_bits_equal, assert_records_equal, dprt, random_rays
from instance_cases import CASES, case_10m, moved, object_desc
from refit_cases import assert_blob_equal
from test_gpu_refit import _render_equal, _trace_equal

pytestmark = pytest.mark.gpu


def _case(name):
    return case_10m() if name == "10m" else CASES[name]()


def _renderer(w=16, h=16, spp=1, bounces=1):
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=1, proxy_mode=0)
    return dprt.Renderer(cfg)


def _twin_equal(blob, v, uv, m, what):
    nodes, tris = blob
    tris = tris.copy()
    if uv is not None:                       # the texture-coordinate tail's marker: the twin's records carry none
        assert (tris["pad_"] == len(tris)).all(), what
        tris["pad_"] = 0
    assert_blob_equal((nodes, tris), dprt.spec_bvh8_build_gpu(v, m)[:2], what)


@pytest.mark.parametrize("case", sorted(CASES) + ["10m"])
def test_device_flatten_builds_the_host_flattened_chunk(gpu_required, case):
    meshes, inst = _case(case)
    v, n, uv, m = dprt.flatten_instances(meshes, inst)
    desc = object_desc(meshes, inst)
    R = _renderer()
    R.build_instanced_chunk(0, desc, meshes, inst)
    blob = R.chunk_bvh8(0)
    _twin_equal(blob, v, uv, m, f"{case}: instanced build vs twin of the host-flattened arrays")
    R.build_chunk(0, desc, v, n, uv, m)
    assert_blob_equal(R.chunk_bvh8(0), blob, f"{case}: instanced build vs build_chunk of the host-flattened arrays")
    R.close()


def _garden_scene(X, g, cam):
    X.set_materials(g["materials"]); X.set_lights(g["lights"]); X.set_camera(cam)
    for slot, t in g["textures"].items():
        X.set_texture(slot, t)
    X.set_material_textures(g["material_textures"])
    X.set_env_map(g["env_map"], g["env_rotation"])


def _garden_world(oracle, cfg, g, instances=None, desc=None):
    """Oracle world of the garden's objects from the host-flattened arrays; instances: {scene index: instance list} overrides,
    desc: the object description of a one-object garden."""
    world = oracle.World(cfg, len(g["objects"]))
    for ob in g["objects"]:
        inst = (instances or {}).get(ob.index, ob.instances)
        v, n, uv, m = dprt.flatten_instances(ob.meshes, inst)
        world.add_object_uv(ob.index, desc or ob.desc(False), v, n, uv, m)
    _garden_scene(world, g, dprt.scene.default_camera(cfg.width, cfg.height))
    return world


def _garden_renderer(g, w, h, spp=2, bounces=4, desc=None):
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=1, proxy_mode=0)
    R = dprt.Renderer(cfg)
    ob = g["objects"][0]
    R.build_instanced_chunk(0, desc or ob.desc(False), ob.meshes, ob.instances)
    _garden_scene(R, g, dprt.scene.default_camera(w, h))
    return R


def test_textured_garden_renders_like_the_oracle(gpu_required, oracle):
    g = dprt.real_scene.make_garden(1)
    R = _garden_renderer(g, 160, 90)
    world = _garden_world(oracle, R.cfg, g)
    _render_equal(R, world, "textured garden, instanced GPU build")
    _trace_equal(R, world, "textured garden, instanced GPU build")
    R.close()


def test_two_rank_group(gpu_required, oracle):
    g = dprt.real_scene.make_garden(2)
    w, h = 128, 72
    cfg = dprt.make_config(w, h, spp=2, bounces=4, scene_size=2, proxy_mode=0)
    rs = []
    for r in range(2):
        R = dprt.Renderer(cfg, rank=r, world=2)
        for ob in g["objects"]:
            if ob.node_id == r:
                R.build_instanced_chunk(ob.index, ob.desc(False), ob.meshes, ob.instances)
            else:
                R.upload_proxy(ob.index, ob.desc(True), None, None)
        _garden_scene(R, g, dprt.scene.default_camera(w, h))
        rs.append(R)
    world = _garden_world(oracle, cfg, g)
    img_g, img_o = dprt.RankGroup(rs).launch(), world.launch()
    N, spc = w * h, cfg.shadowPathCount
    for r, R in enumerate(rs):
        k = R.path_size
        assert k == world.path_size(r)
        assert_records_equal(R.download(D.BUF_PATHS, k * (1 + spc)), world.download(r, D.BUF_PATHS, k * (1 + spc)), f"rank {r} paths")
        assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * N), f"rank {r} env")
        assert_bits_equal(R.download(D.BUF_DIRECT), world.download(r, D.BUF_DIRECT, 3 * N * spc), f"rank {r} direct")
    assert_bits_equal(img_g, img_o, "two-rank garden, instanced GPU builds")
    assert img_g.max() > 0
    for R in rs:
        R.close()


@pytest.mark.parametrize("case", ["garden", "mixed_uv", "zero_tris", "10m"])
def test_update_equals_host_refit(gpu_required, case):
    """Instances moved, some of them twice, then moved back: every blob is the host refit of the build's blob to the host-flattened
    moved instances, and the one dprt_refit_chunk makes of them."""
    meshes, inst = _case(case)
    m1 = moved(inst, every=3)
    m2 = moved(m1, every=2, angle=-0.2, shrink=0.9)
    desc = object_desc(meshes, inst, m1, m2)
    R, H = _renderer(), _renderer()
    R.build_instanced_chunk(0, desc, meshes, inst)
    H.build_instanced_chunk(0, desc, meshes, inst)
    blob0 = R.chunk_bvh8(0)
    for k, mk in enumerate([m1, m2, inst]):
        v, n, _, _ = dprt.flatten_instances(meshes, mk)
        R.update_instances(0, mk)
        blob = R.chunk_bvh8(0)
        assert_blob_equal(blob, dprt.spec_bvh8_refit(blob0[0], blob0[1], v), f"{case} step {k}: update vs host refit")
        H.refit_chunk(0, v, n)
        assert_blob_equal(blob, H.chunk_bvh8(0), f"{case} step {k}: update vs dprt_refit_chunk")
    assert_blob_equal(R.chunk_bvh8(0), blob0, f"{case}: moved back")
    R.close(); H.close()


def test_moved_garden_renders_like_the_oracle(gpu_required, oracle):
    g = dprt.real_scene.make_garden(1)
    ob = g["objects"][0]
    m1 = moved(ob.instances, every=3)
    m2 = moved(m1, every=2, angle=-0.2, shrink=0.9)
    desc = object_desc(ob.meshes, ob.instances, m1, m2)
    R = _garden_renderer(g, 160, 90, desc=desc)
    img0, blob0 = R.launch(), R.chunk_bvh8(0)
    R.update_instances(0, m1)
    R.update_instances(0, m2)
    world = _garden_world(oracle, R.cfg, g, {0: m2}, desc)
    _render_equal(R, world, "garden, instances moved on the GPU")
    rays = np.concatenate([random_rays(50000, 3, lo=0.0, hi=1.0), dprt.scene.camera_rays(dprt.scene.default_camera(320, 180))])
    hg, ho = R.trace_closest(rays), world.trace_closest(0, rays)
    assert_bits_equal(hg["primID"], ho["primID"], "garden, instances moved on the GPU: primID")
    assert_bits_equal(hg["t"], ho["t"], "garden, instances moved on the GPU: t")
    R.update_instances(0, ob.instances)
    assert_blob_equal(R.chunk_bvh8(0), blob0, "garden moved back: blob")
    assert_bits_equal(R.launch(), img0, "garden moved back: image")
    R.close()


def test_samples_in_flight_see_the_update(gpu_required, oracle):
    g = dprt.real_scene.make_garden(1)
    ob = g["objects"][0]
    m1 = moved(ob.instances, every=2)
    desc = object_desc(ob.meshes, ob.instances, m1)
    R = _garden_renderer(g, 160, 90, spp=6, bounces=3, desc=desc)
    F = dprt.SamplesInFlight(R, 3)
    R.update_instances(0, m1)               # device memory shared with the adopting contexts
    img = F.launch()
    img_o = _garden_world(oracle, R.cfg, g, {0: m1}, desc).launch()
    err = float(np.abs(img - img_o).max() / np.abs(img_o).max())
    assert np.isfinite(img).all() and err <= 1e-6, err
    F.close(); R.close()


def test_rejections_change_nothing(gpu_required):
    g = dprt.real_scene.make_garden(1)
    ob = g["objects"][0]
    meshes, inst = ob.meshes, ob.instances
    desc = object_desc(meshes, inst, moved(inst))
    R = _garden_renderer(g, 64, 36, spp=1, bounces=2, desc=desc)
    img0, blob0 = R.launch(), R.chunk_bvh8(0)

    def with_mesh(k, **kw):
        out = list(meshes)
        out[k] = dict(out[k], **kw)
        return out

    def with_matrix(i, M):
        out = list(inst)
        out[i] = (out[i][0], np.asarray(M, np.float32))
        return out

    def over_cap():                          # a mesh description claiming 2^27 triangles: refused before any array is copied
        md, nm, ins, ni, keep = D.pack_meshes(meshes, inst)
        md[0].ntris = 1 << 27
        rc = R.lib.dprt_build_instanced_chunk(R.h, 0, C.byref(desc), md, nm, ins, ni)
        del keep
        assert rc == -4, rc                  # DPRT_ERR_CAPACITY
        raise dprt.DprtError("over the cap")

    singular = np.zeros((3, 4), np.float32)
    nonfinite = np.array(inst[3][1], np.float32); nonfinite[2, 2] = np.inf
    nan = np.array(inst[3][1], np.float32); nan[0, 1] = np.nan
    far = np.array(inst[3][1], np.float32); far[0, 3] += 10.0
    textured = next(k for k, m in enumerate(meshes) if m["texcoords"] is not None)
    empty = list(meshes) + [dict(meshes[0], indices=np.zeros((0, 3), np.int32), normal_indices=np.zeros((0, 3), np.int32),
                                 texcoords=None, texcoord_indices=None)]
    builds = [
        ("unknown index", lambda: R.build_instanced_chunk(1, desc, meshes, inst)),
        ("negative index", lambda: R.build_instanced_chunk(-1, desc, meshes, inst)),
        ("nodeID outside the world", lambda: R.build_instanced_chunk(0, D.make_object_desc(1, ob.aabb_min, ob.aabb_max), meshes, inst)),
        ("mesh index out of range", lambda: R.build_instanced_chunk(0, desc, meshes, inst + [(len(meshes), np.eye(4)[:3])])),
        ("position index out of range", lambda: R.build_instanced_chunk(0, desc, with_mesh(1, indices=np.asarray(meshes[1]["indices"]) + 10 ** 6), inst)),
        ("negative normal index", lambda: R.build_instanced_chunk(0, desc, with_mesh(2, normal_indices=-np.ones_like(meshes[2]["normal_indices"])), inst)),
        ("texture-coordinate index out of range", lambda: R.build_instanced_chunk(
            0, desc, with_mesh(textured, texcoord_indices=np.asarray(meshes[textured]["texcoord_indices"]) + len(meshes[textured]["texcoords"])), inst)),
        ("index out of range in a mesh no instance uses", lambda: R.build_instanced_chunk(
            0, desc, meshes + [dict(meshes[1], indices=np.asarray(meshes[1]["indices"]) + 10 ** 6)], inst)),
        ("singular transform", lambda: R.build_instanced_chunk(0, desc, meshes, with_matrix(3, singular))),
        ("non-finite transform", lambda: R.build_instanced_chunk(0, desc, meshes, with_matrix(3, nonfinite))),
        ("singular transform of a zero-triangle instance", lambda: R.build_instanced_chunk(0, desc, empty, inst + [(len(meshes), singular)])),
        ("over the triangle cap", over_cap),
    ]
    cfg2 = dprt.make_config(16, 16, scene_size=2, proxy_mode=0)
    P = dprt.Renderer(cfg2, rank=0, world=2)             # index 1 is a proxy there, index 0 an uploaded (host-built) chunk
    P.upload_instanced_chunk(0, desc, meshes, inst)
    P.upload_proxy(1, D.make_object_desc(1, ob.aabb_min, ob.aabb_max, is_proxy=1), None, None)
    other_mesh = list(inst)
    other_mesh[5] = (other_mesh[4][0] if other_mesh[4][0] != other_mesh[5][0] else other_mesh[0][0], other_mesh[5][1])
    assert other_mesh[5][0] != inst[5][0]
    updates = [
        ("update: unknown index", lambda: R.update_instances(1, inst)),
        ("update: proxy", lambda: P.update_instances(1, inst)),
        ("update: chunk made by upload_instanced_chunk", lambda: P.update_instances(0, inst)),
        ("update: fewer instances", lambda: R.update_instances(0, inst[:-1])),
        ("update: more instances", lambda: R.update_instances(0, inst + inst[:1])),
        ("update: another mesh", lambda: R.update_instances(0, other_mesh)),
        ("update: singular transform", lambda: R.update_instances(0, with_matrix(3, singular))),
        ("update: non-finite transform", lambda: R.update_instances(0, with_matrix(3, nonfinite))),
        ("update: NaN in a transform", lambda: R.update_instances(0, with_matrix(3, nan))),
        ("update: outside the object's AABB", lambda: R.update_instances(0, with_matrix(3, far))),
    ]
    for what, call in builds + updates:
        with pytest.raises(dprt.DprtError):
            call()
        assert_blob_equal(R.chunk_bvh8(0), blob0, what)
    assert_bits_equal(R.launch(), img0, "render after the rejected calls")
    R.update_instances(0, moved(inst))       # the chunk still moves after them
    P.close(); R.close()
