"""First-hit guide buffers (AOVs) of the CPU reference, checked against independent facts (no GPU).

The albedo and normal the first shade of a sample adds per pixel are this project's own specification (DESIGN.md 3.7): the
albedo the shading program uses, and the interpolated, normalised, face-forwarded shading normal. Here the camera records
are traced on their own and the reference's AOVs (the oracle with the AOV rule, tests/aov_reference.cpp) must say what
those hits say.
"""
import numpy as np

from aov_reference import AovWorld
from helpers import D, dprt


def _world(W=1, water_frac=0.05, w=64, h=36, spp=1, bounces=2):
    chunks, mats, lights = dprt.scene.make_scene(W, 4000, water_frac=water_frac)
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=W, proxy_mode=0)
    world = AovWorld(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
    world.set_materials(mats); world.set_lights(lights); world.set_camera(dprt.scene.default_camera(w, h))
    return world, chunks, mats, lights


def test_oracle_aov_matches_first_hit_of_camera_rays():
    world, chunks, mats, _ = _world()
    N = world.N
    world.begin_sample(0)
    world.path_gen(0)
    recs = world.download(0, D.BUF_PATHS, N)
    world.enable_aov()
    world.launch()                                       # spp = 1: sample 0 regenerates the same camera records
    albedo, normal = (x.reshape(-1, 3) for x in world.aov())
    assert np.array_equal(world.aov_buffer(0), np.concatenate([albedo.reshape(-1), normal.reshape(-1)]))

    rays = np.zeros(N, D.RAY_DTYPE)
    rays["origin"], rays["direction"] = recs["origin"], recs["direction"]
    rays["tMin"], rays["tMax"] = D.DPRT_EPSILON, np.finfo(np.float32).max
    hits = world.trace_closest(0, rays)
    px = recs["pixelIndex"]
    hit = hits["primID"] >= 0
    assert hit.sum() > N // 4 and (~hit).sum() > 0, "the view must show both geometry and sky"

    base = mats["baseColor"][chunks[0].mats[hits["primID"][hit]]]
    assert np.array_equal(albedo[px[hit]], base.astype(np.float32)), "albedo is the hit material's baseColor"
    assert (mats["bsdfType"][chunks[0].mats[hits["primID"][hit]]] == 1).any(), "no water hit: the test does not cover it"
    assert not albedo[px[~hit]].any() and not normal[px[~hit]].any(), "a miss adds +0"

    n = normal[px[hit]].astype(np.float64)
    assert np.abs(np.linalg.norm(n, axis=1) - 1.0).max() <= 1e-6, "shading normal has unit length"
    assert (np.einsum("ij,ij->i", n, rays["direction"][hit].astype(np.float64)) <= 0).all(), "normal faces the incoming ray"


def test_oracle_aov_only_first_shade_of_each_sample():
    """Two samples, two bounces: each pixel's normal sum is at most spp long (one first hit per sample), never more."""
    world, _, _, _ = _world(spp=2)
    world.enable_aov()
    world.launch()
    _, normal = world.aov()
    assert np.linalg.norm(normal.reshape(-1, 3).astype(np.float64), axis=1).max() <= 1.0 + 1e-6


def test_oracle_image_unchanged_by_aov(oracle):
    """The reference's render loop with AOVs on gives the oracle's own image, bit for bit."""
    world, chunks, mats, lights = _world(spp=2)
    world.enable_aov()
    on = world.launch()
    plain = oracle.World(world.cfg, 1)
    c = chunks[0]
    plain.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
    plain.set_materials(mats); plain.set_lights(lights); plain.set_camera(dprt.scene.default_camera(64, 36))
    off = plain.launch()
    assert off.max() > 0
    assert np.array_equal(off.view(np.uint32), on.view(np.uint32)), "enabling the AOVs changes the colour image"
