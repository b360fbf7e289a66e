"""Shared builders for the parity tests: the same scene goes into libdprt and into the oracle."""
import importlib

import numpy as np

dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
D = dprt.ctypes_defs


def build_pair(O, W, tris_per_chunk, width, height, *, spp=1, bounces=2, proxy_mode=0, path_gen_mode=0, water_frac=0.0,
               group=True, models=None, mlp_dtype=1, device=0, main_ray_retrace=0, serial_stages=0, reference_migrate=0, gpu=True):
    """Returns (renderers[list of W Renderer], oracle World, chunks). models: {scene_index: (vis_blob, depth_blob)}.
    gpu=False builds the oracle world only (no renderers)."""
    chunks, mats, lights = dprt.scene.make_scene(W, tris_per_chunk, water_frac=water_frac)
    cfg = dprt.make_config(width, height, spp=spp, bounces=bounces, scene_size=W, proxy_mode=proxy_mode,
                           path_gen_mode=path_gen_mode, mlp_dtype=mlp_dtype, main_ray_retrace=main_ray_retrace,
                           serial_stages=serial_stages, reference_migrate=reference_migrate)
    cam = dprt.scene.default_camera(width, height)
    world = O.World(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
        if models and c.index in models:
            vb, db = models[c.index]
            if vb is not None:
                world.set_model(c.index, 0, vb)
            if db is not None:
                world.set_model(c.index, 1, db)
    world.set_materials(mats)
    world.set_lights(lights)
    world.set_camera(cam)
    rs = []
    for r in range(W if gpu else 0):
        R = dprt.Renderer(cfg, rank=r, world=W, device=device)
        for c in chunks:
            if c.node_id == r:
                R.upload_chunk(c.index, c.desc(False), c.verts, c.normals, c.mats)
            else:
                vb, db = (models or {}).get(c.index, (None, None))
                R.upload_proxy(c.index, c.desc(True), vb, db)
        R.set_materials(mats)
        R.set_lights(lights)
        R.set_camera(cam)
        rs.append(R)
    return rs, world, chunks


def assert_records_equal(a, b, what):
    """Bitwise comparison of structured record arrays with a readable first-mismatch report."""
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.size == 0:
        return
    ab, bb = a.view(np.uint8).reshape(a.size, -1), b.view(np.uint8).reshape(b.size, -1)
    bad = np.nonzero((ab != bb).any(axis=1))[0]
    if bad.size:
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.size}/{a.size} records differ; first at {i}:\n gpu   ={a[i]}\n oracle={b[i]}")


def assert_bits_equal(a, b, what):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    av, bv = a.view(np.uint8), b.view(np.uint8)
    if not np.array_equal(av, bv):
        idx = np.nonzero(a.reshape(-1) != b.reshape(-1))[0]
        i = int(idx[0]) if idx.size else -1
        raise AssertionError(f"{what}: {idx.size}/{a.size} values differ; first at {i}: gpu={a.reshape(-1)[i]!r} oracle={b.reshape(-1)[i]!r}")


def random_rays(n, seed, lo=-0.2, hi=1.2):
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, D.RAY_DTYPE)
    rays["origin"] = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays["direction"] = d.astype(np.float32)
    rays["tMin"] = D.DPRT_EPSILON
    rays["tMax"] = np.finfo(np.float32).max
    return rays


def build_garden_pair(O, W, width, height, *, spp=1, bounces=2, gpu=True, device=0, textures=True, env_map=True, clusters=18,
                      ground=(40, 40), cluster_scale=0.05, main_ray_retrace=0, serial_stages=0, reference_migrate=0):
    """The real-scene front end (SURVEY.md 8f row 3) on both sides: W instanced, textured scene objects (real_scene.make_garden)
    go through dprt_upload_instanced_chunk / dprt_set_texture / dprt_set_material_textures / dprt_set_env_map and through the
    oracle's own flatten and texture code. gpu=False builds the oracle world only. Returns (renderers, world, garden)."""
    g = dprt.real_scene.make_garden(W, clusters=clusters, ground=ground, cluster_scale=cluster_scale)
    cfg = dprt.make_config(width, height, spp=spp, bounces=bounces, scene_size=W, proxy_mode=0, main_ray_retrace=main_ray_retrace,
                           serial_stages=serial_stages, reference_migrate=reference_migrate)
    cam = dprt.scene.default_camera(width, height)
    world = O.World(cfg, W)
    for ob in g["objects"]:
        world.add_instanced_object(ob.index, ob.desc(False), ob.meshes, ob.instances)
    world.set_materials(g["materials"]); world.set_lights(g["lights"]); world.set_camera(cam)
    if textures:
        for slot, t in g["textures"].items():
            world.set_texture(slot, t)
        world.set_material_textures(g["material_textures"])
    if env_map:
        world.set_env_map(g["env_map"], g["env_rotation"])
    rs = []
    for r in range(W if gpu else 0):
        R = dprt.Renderer(cfg, rank=r, world=W, device=device)
        for ob in g["objects"]:
            if ob.node_id == r:
                R.upload_instanced_chunk(ob.index, ob.desc(False), ob.meshes, ob.instances)
            else:
                R.upload_proxy(ob.index, ob.desc(True), None, None)
        R.set_materials(g["materials"]); R.set_lights(g["lights"]); R.set_camera(cam)
        if textures:
            for slot, t in g["textures"].items():
                R.set_texture(slot, t)
            R.set_material_textures(g["material_textures"])
        if env_map:
            R.set_env_map(g["env_map"], g["env_rotation"])
        rs.append(R)
    return rs, world, g
