"""BVH8 build on the GPU (-m gpu; DESIGN.md 3.10): dprt_build_chunk / dprt_build_chunk_device against the host twin
dprt_spec_bvh8_build_gpu bit for bit, and renders of GPU-built chunks against the oracle. Hits do not depend on the tree
(watertight test, fixed tie-break), so everything is bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import D, assert_bits_equal, assert_records_equal, build_pair, dprt
from refit_cases import assert_blob_equal, deform, garden_flat, terrain, upload_desc
from test_bvh_gpu_build_cpu import CASES
from test_gpu_refit import _render_equal, _trace_equal, _world

pytestmark = pytest.mark.gpu
BIN = os.path.join(os.path.dirname(dprt.host.LIB_PATH), "dprt_render")


def _renderer(w=160, h=90, spp=2, bounces=4):
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=1, proxy_mode=0)
    R = dprt.Renderer(cfg)
    R.set_materials(dprt.scene.make_materials(16)); R.set_lights(dprt.scene.make_lights()); R.set_camera(dprt.scene.default_camera(w, h))
    return R


def _to_device(R, *arrays):
    out = []
    for a in arrays:
        if a is None:
            out.append(None)
            continue
        a = np.ascontiguousarray(a)
        d = R.device_alloc(max(a.nbytes, 4))
        R.h2d(d, a)
        out.append(d)
    return out


def _build_device(R, si, desc, v, n, uv, m):
    ptrs = _to_device(R, v, n, uv, m)
    try:
        R.build_chunk_device(si, desc, *ptrs, v.shape[0])
    finally:
        for p in ptrs:
            if p is not None:
                R.device_free(p)


def _twin_blob(v, m):
    return dprt.spec_bvh8_build_gpu(v, m)[:2]


@pytest.mark.parametrize("case", sorted(CASES) + ["terrain_100k", "terrain_1m"])
def test_device_build_equals_twin(gpu_required, case):
    if case == "terrain_100k":
        v = terrain(100000)[0]
    elif case == "terrain_1m":
        v = terrain(1000000)[0]
    else:
        v = CASES[case]()
    m = (np.arange(v.shape[0]) % 7).astype(np.int32)
    twin = _twin_blob(v, m)
    R = _renderer(16, 16)
    R.build_chunk(0, upload_desc(v), v, None, None, m)
    assert_blob_equal(R.chunk_bvh8(0), twin, f"{case}: host-array variant vs twin")
    _build_device(R, 0, upload_desc(v), v, None, None, m)
    assert_blob_equal(R.chunk_bvh8(0), twin, f"{case}: device-array variant vs twin")
    R.close()


@pytest.mark.parametrize("device", [False, True])
def test_single_rank_render_after_build(gpu_required, oracle, device):
    v, n, m = terrain(20000)
    R = _renderer()
    if device:
        _build_device(R, 0, upload_desc(v), v, n, None, m)
    else:
        R.build_chunk(0, upload_desc(v), v, n, None, m)
    world = _world(oracle, R.cfg, [(upload_desc(v), v, n, m)])
    _render_equal(R, world, "GPU-built chunk")
    _trace_equal(R, world, "GPU-built chunk")
    R.close()


def test_full_size_1m_1080p(gpu_required, oracle):
    oracle.use_all_host_threads()
    v, n, m = terrain(1000000)
    R = _renderer(1920, 1080)
    R.build_chunk(0, upload_desc(v), v, n, None, m)
    world = _world(oracle, R.cfg, [(upload_desc(v), v, n, m)])
    _render_equal(R, world, "1 M triangles, 1080p, GPU-built")
    _trace_equal(R, world, "1 M triangles, GPU-built")
    R.close()


def test_textured_garden_with_cutouts(gpu_required, oracle):
    """The leaf-order texture-coordinate tail: the garden's albedo / opacity maps and cut-outs read it on every hit."""
    v, n, uv, m, g, inst = garden_flat()
    ob = g["objects"][0]
    w, h = 160, 90
    cfg = dprt.make_config(w, h, spp=2, bounces=4, scene_size=1, proxy_mode=0)
    cam = dprt.scene.default_camera(w, h)
    R = dprt.Renderer(cfg)
    world = oracle.World(cfg, 1)
    R.build_chunk(0, ob.desc(False), v, n, uv, m)
    world.add_instanced_object(0, ob.desc(False), ob.meshes, inst)
    for X in (R, world):
        X.set_materials(g["materials"]); X.set_lights(g["lights"]); X.set_camera(cam)
        for slot, t in g["textures"].items():
            X.set_texture(slot, t)
        X.set_material_textures(g["material_textures"])
        X.set_env_map(g["env_map"], g["env_rotation"])
    nodes, tris = R.chunk_bvh8(0)
    assert (tris["pad_"] == len(tris)).all()
    twin = _twin_blob(v, m)
    tris["pad_"] = 0
    assert_blob_equal((nodes, tris), twin, "garden vs twin")
    _render_equal(R, world, "textured garden, GPU-built")
    _trace_equal(R, world, "textured garden, GPU-built")
    R.close()


def test_two_rank_group_one_gpu_built(gpu_required, oracle):
    rs, world, chunks = build_pair(oracle, 2, 6000, 128, 72, spp=2, bounces=4, proxy_mode=0)
    c0 = chunks[0]
    rs[0].build_chunk(0, c0.desc(False), c0.verts, c0.normals, None, c0.mats)      # rank 1 keeps its host-built chunk
    G = dprt.RankGroup(rs)
    img_g, img_o = G.launch(), world.launch()
    N, spc = 128 * 72, rs[0].cfg.shadowPathCount
    for r, R in enumerate(rs):
        k = R.path_size
        assert k == world.path_size(r)
        assert_records_equal(R.download(D.BUF_PATHS, k * (1 + spc)), world.download(r, D.BUF_PATHS, k * (1 + spc)), f"rank {r} paths")
        assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * N), f"rank {r} env")
        assert_bits_equal(R.download(D.BUF_DIRECT), world.download(r, D.BUF_DIRECT, 3 * N * spc), f"rank {r} direct")
    assert_bits_equal(img_g, img_o, "two-rank image, one chunk GPU-built")
    for R in rs:
        R.close()


@pytest.mark.parametrize("kind", ["zscale", "permute"])
def test_refit_of_gpu_built_chunk(gpu_required, kind):
    v, n, m = terrain(100000)
    R = _renderer(16, 16)
    R.build_chunk(0, upload_desc(v), v, n, None, m)
    blob0 = R.chunk_bvh8(0)
    assert_blob_equal(blob0, _twin_blob(v, m), "build vs twin")
    v2 = deform(v, kind)
    R.refit_chunk(0, v2, n)
    assert_blob_equal(R.chunk_bvh8(0), dprt.spec_bvh8_refit(blob0[0], blob0[1], v2), f"{kind} refit vs spec")
    R.refit_chunk(0, v, n)
    assert_blob_equal(R.chunk_bvh8(0), blob0, f"{kind}: refit back to V")
    R.close()


def _traray_per_ray(R, sample):
    R.enable_counters(True); R.reset_stats(); R.reset_frame()
    R.run_sample(sample)
    R.synchronize()
    c, walked = R.counters()["traverse"], R.stats()["walked_traverse"]
    R.enable_counters(False)
    return c[0] / walked, c[1] / walked


def test_rebuild_after_permutation(gpu_required, oracle):
    """A permutation refit keeps the old grouping, so every box spans the chunk (DESIGN.md 3.9); a GPU rebuild of the permuted
    vertices (the same triangles under other ids) brings the per-ray work back to that of a build of the original ones."""
    v, n, m = terrain(20000)
    R = _renderer()
    R.build_chunk(0, upload_desc(v), v, n, None, m)
    base = _traray_per_ray(R, 0)
    perm = np.random.default_rng(1).permutation(v.shape[0])
    vp, n_p, mp = v[perm], n[perm], m[perm]
    R.refit_chunk(0, vp, n)
    refit = _traray_per_ray(R, 0)
    R.build_chunk(0, upload_desc(v), vp, n_p, None, mp)
    rebuilt = _traray_per_ray(R, 0)
    print(f"TraRay nodes, triangles per ray: GPU build {base}, permutation refit {refit}, GPU rebuild {rebuilt}")
    assert refit[0] > 10 * base[0]
    assert rebuilt[0] <= 1.05 * base[0] and rebuilt[1] <= 1.05 * base[1], (rebuilt, base)
    world = _world(oracle, R.cfg, [(upload_desc(v), vp, n_p, mp)])
    _render_equal(R, world, "rebuilt from permuted vertices")
    R.close()


def test_samples_in_flight_share_the_built_chunk(gpu_required, oracle):
    v, n, m = terrain(20000)
    R = _renderer(spp=6, bounces=3)
    R.build_chunk(0, upload_desc(v), v, n, None, m)
    F = dprt.SamplesInFlight(R, 3)
    img = F.launch()
    img_o = _world(oracle, R.cfg, [(upload_desc(v), v, n, m)]).launch()
    err = float(np.abs(img - img_o).max() / np.abs(img_o).max())
    assert np.isfinite(img).all() and err <= 1e-6, err
    F.close(); R.close()


@pytest.mark.parametrize("device", [False, True])
def test_rejections_change_nothing(gpu_required, device):
    v, n, m = terrain(20000)
    R = _renderer(64, 36, spp=1, bounces=2)
    R.upload_chunk(0, upload_desc(v), v, n, m)
    img0, blob0 = R.launch(), R.chunk_bvh8(0)
    v2 = deform(v, "zscale")
    nan, inf, badm, negm = v2.copy(), v2.copy(), m.copy(), m.copy()
    nan[5, 2] = np.nan
    inf[7, 0] = -np.inf
    badm[11] = 256                                           # DPRT_MAX_MATERIALS
    negm[3] = -1
    desc = upload_desc(v2)
    outside = upload_desc(v2, node_id=1)                     # a nodeID outside this one-rank world

    def build(si, d, vv, mm, ntris=None):
        if ntris is not None:                                # over the triangle cap: refused before any array is read
            if device:
                dv, = _to_device(R, vv)
                try:
                    return R.build_chunk_device(si, d, dv, None, None, None, ntris)
                finally:
                    R.device_free(dv)
            p = vv.ctypes.data_as(C.c_void_p)
            return R._ck(R.lib.dprt_build_chunk(R.h, si, C.byref(d), p, None, None, None, ntris), "dprt_build_chunk")
        if device:
            return _build_device(R, si, d, vv, n, None, mm)
        return R.build_chunk(si, d, vv, n, None, mm)

    cases = [("unknown index", 1, desc, v2, m, None), ("negative index", -1, desc, v2, m, None),
             ("nodeID outside the world", 0, outside, v2, m, None), ("nan", 0, desc, nan, m, None), ("inf", 0, desc, inf, m, None),
             ("material too large", 0, desc, v2, badm, None), ("negative material", 0, desc, v2, negm, None),
             ("over the triangle cap", 0, desc, v2, m, 1 << 27)]
    for what, si, d, vv, mm, nt in cases:
        with pytest.raises(dprt.DprtError):
            build(si, d, vv, mm, nt)
        assert_blob_equal(R.chunk_bvh8(0), blob0, what)
    assert_bits_equal(R.launch(), img0, "render after the rejected builds")
    R.close()


def test_dprt_render_gpu_build_same_image(gpu_required, tmp_path):
    chunks, mats, lights = dprt.scene.make_scene(1, 8000, water_frac=0.02)
    scene = str(tmp_path / "scene.dprt")
    dprt.scene.save_scene(scene, chunks, mats, lights, dprt.scene.default_camera(160, 90))
    imgs = []
    for flag in ("0", "1"):
        out = str(tmp_path / f"img{flag}.pfm")
        p = subprocess.run([BIN, "--scene", scene, "--out", out, "--spp", "2", "--bounces", "3", "--gpu-build", flag],
                           capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr[-2000:]
        imgs.append(dprt.scene.load_pfm(out))
    assert imgs[0].max() > 0
    assert_bits_equal(imgs[1], imgs[0], "dprt_render --gpu-build 1 vs 0")
