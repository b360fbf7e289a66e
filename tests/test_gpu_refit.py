"""BVH8 refit on the GPU (-m gpu; DESIGN.md 3.9): dprt_refit_chunk / dprt_refit_chunk_device against the host specification
dprt_spec_bvh8_refit, and renders after a refit against an oracle world built directly from the moved vertices. Hits do not
depend on the tree (watertight test, fixed tie-break), so everything is bit for bit."""
import numpy as np
import pytest

from helpers import D, assert_bits_equal, assert_records_equal, build_pair, dprt, random_rays
from refit_cases import assert_blob_equal, deform, garden_flat, terrain, upload_desc

pytestmark = pytest.mark.gpu


def _renderer(v, n, m, w=160, h=90, spp=2, bounces=4):
    cfg = dprt.make_config(w, h, spp=spp, bounces=bounces, scene_size=1, proxy_mode=0)
    R = dprt.Renderer(cfg)
    R.upload_chunk(0, upload_desc(v), v, n, m)
    R.set_materials(dprt.scene.make_materials(16)); R.set_lights(dprt.scene.make_lights()); R.set_camera(dprt.scene.default_camera(w, h))
    return R


def _world(oracle, cfg, chunks):
    """Oracle world of W = len(chunks) objects; chunks: (desc, verts9, normals9, mat_ids) per scene index."""
    world = oracle.World(cfg, len(chunks))
    for k, (desc, v, n, m) in enumerate(chunks):
        world.add_object(k, desc, v, n, m)
    world.set_materials(dprt.scene.make_materials(16)); world.set_lights(dprt.scene.make_lights())
    world.set_camera(dprt.scene.default_camera(cfg.width, cfg.height))
    return world


def _render_equal(R, world, what):
    """launch on both sides; image, path records, env and direct buffers of the last sample bit for bit."""
    img_g, img_o = R.launch(), world.launch()
    n, spc, N = R.path_size, R.cfg.shadowPathCount, R.N
    assert n == world.path_size(0), what
    assert_records_equal(R.download(D.BUF_PATHS, n * (1 + spc)), world.download(0, D.BUF_PATHS, n * (1 + spc)), f"{what}: paths")
    assert_bits_equal(R.download(D.BUF_ENV), world.download(0, D.BUF_ENV, 3 * N), f"{what}: env")
    assert_bits_equal(R.download(D.BUF_DIRECT), world.download(0, D.BUF_DIRECT, 3 * N * spc), f"{what}: direct")
    assert_bits_equal(img_g, img_o, f"{what}: image")
    assert np.isfinite(img_g).all() and img_g.max() > 0
    return img_g


def _trace_equal(R, world, what):
    rays = np.concatenate([random_rays(50000, 3, lo=0.0, hi=1.0), dprt.scene.camera_rays(dprt.scene.default_camera(320, 180))])
    hg, ho = R.trace_closest(rays), world.trace_closest(0, rays)
    assert_bits_equal(hg["primID"], ho["primID"], f"{what}: primID")
    assert_bits_equal(hg["t"], ho["t"], f"{what}: t")
    assert (hg["primID"] >= 0).mean() > 0.3


@pytest.mark.parametrize("ntris,kind", [(100000, "identity"), (100000, "zscale"), (100000, "permute"), (1000000, "permute")])
def test_device_refit_equals_spec(gpu_required, ntris, kind):
    v, n, m = terrain(ntris)
    R = _renderer(v, n, m, 16, 16)
    blob0 = R.chunk_bvh8(0)
    assert_blob_equal(blob0, dprt.build_bvh8(v, m)[:2], "upload vs host build")
    v2 = v if kind == "identity" else deform(v, kind)
    R.refit_chunk(0, v2, n)
    assert_blob_equal(R.chunk_bvh8(0), dprt.spec_bvh8_refit(blob0[0], blob0[1], v2), f"{kind}: device vs spec")
    R.refit_chunk(0, v, n)
    assert_blob_equal(R.chunk_bvh8(0), blob0, f"{kind}: refit back to V")
    R.close()


def test_device_variant_equals_host_variant(gpu_required):
    v, n, m = terrain(50000)
    v2 = deform(v, "zjitter")
    A, B = _renderer(v, n, m, 16, 16), _renderer(v, n, m, 16, 16)
    A.refit_chunk(0, v2, n)
    dv, dn = B.device_alloc(v2.nbytes), B.device_alloc(n.nbytes)
    B.h2d(dv, v2); B.h2d(dn, n)
    B.refit_chunk_device(0, dv, dn, v2.shape[0])
    assert_blob_equal(B.chunk_bvh8(0), A.chunk_bvh8(0), "device variant vs host variant")
    B.device_free(dv); B.device_free(dn)
    A.close(); B.close()


@pytest.mark.parametrize("kind", ["zscale", "zjitter", "permute"])
def test_single_rank_render_after_refit(gpu_required, oracle, kind):
    v, n, m = terrain(20000)
    R = _renderer(v, n, m)
    img_before = R.launch()
    v2 = deform(v, kind)
    R.refit_chunk(0, v2, n)
    world = _world(oracle, R.cfg, [(upload_desc(v), v2, n, m)])
    _render_equal(R, world, f"after {kind} refit")
    _trace_equal(R, world, f"after {kind} refit")
    # back to V: the original blob and the original render
    blob0 = dprt.build_bvh8(v, m)[:2]
    R.refit_chunk(0, v, n)
    assert_blob_equal(R.chunk_bvh8(0), blob0, "refit back to V")
    assert_bits_equal(R.launch(), img_before, "render after the refit back to V")
    R.close()


def test_full_size_1m_1080p_after_permutation(gpu_required, oracle):
    oracle.use_all_host_threads()
    v, n, m = terrain(1000000)
    R = _renderer(v, n, m, 1920, 1080, spp=2, bounces=4)
    v2 = deform(v, "permute")
    R.refit_chunk(0, v2, n)
    world = _world(oracle, R.cfg, [(upload_desc(v), v2, n, m)])
    _render_equal(R, world, "1 M triangles, 1080p, permutation refit")
    _trace_equal(R, world, "1 M triangles, permutation refit")
    R.close()


def test_two_rank_group_after_refit(gpu_required, oracle):
    rs, _, chunks = build_pair(oracle, 2, 6000, 128, 72, spp=2, bounces=4, proxy_mode=0)
    c0, c1 = chunks
    v2 = deform(c0.verts, "zscale")
    rs[0].refit_chunk(0, v2, c0.normals)
    world = _world(oracle, rs[0].cfg, [(c0.desc(False), v2, c0.normals, c0.mats), (c1.desc(False), c1.verts, c1.normals, c1.mats)])
    G = dprt.RankGroup(rs)
    img_g, img_o = G.launch(), world.launch()
    N, spc = 128 * 72, rs[0].cfg.shadowPathCount
    for r, R in enumerate(rs):
        k = R.path_size
        assert k == world.path_size(r)
        assert_records_equal(R.download(D.BUF_PATHS, k * (1 + spc)), world.download(r, D.BUF_PATHS, k * (1 + spc)), f"rank {r} paths")
        assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * N), f"rank {r} env")
        assert_bits_equal(R.download(D.BUF_DIRECT), world.download(r, D.BUF_DIRECT, 3 * N * spc), f"rank {r} direct")
    assert_bits_equal(img_g, img_o, "two-rank reduced image after refit")
    for R in rs:
        R.close()


def test_samples_in_flight_share_the_refit(gpu_required, oracle):
    v, n, m = terrain(20000)
    R = _renderer(v, n, m, spp=6, bounces=3)
    F = dprt.SamplesInFlight(R, 3)
    v2 = deform(v, "zscale")
    R.refit_chunk(0, v2, n)                 # device memory shared with the adopting contexts
    img = F.launch()
    img_o = _world(oracle, R.cfg, [(upload_desc(v), v2, n, m)]).launch()
    err = float(np.abs(img - img_o).max() / np.abs(img_o).max())
    assert np.isfinite(img).all() and err <= 1e-6, err
    F.close(); R.close()


def test_garden_moved_instances(gpu_required, oracle):
    v, n, uv, m, g, _ = garden_flat()
    vm, nm, uvm, mm, _, moved = garden_flat(moved=True)
    assert np.array_equal(uv, uvm) and np.array_equal(m, mm)
    ob = g["objects"][0]
    w, h = 160, 90
    cfg = dprt.make_config(w, h, spp=2, bounces=4, scene_size=1, proxy_mode=0)
    cam = dprt.scene.default_camera(w, h)
    R = dprt.Renderer(cfg)
    world = oracle.World(cfg, 1)
    R.upload_instanced_chunk(0, ob.desc(False), ob.meshes, ob.instances)
    world.add_instanced_object(0, ob.desc(False), ob.meshes, moved)
    for X in (R, world):
        X.set_materials(g["materials"]); X.set_lights(g["lights"]); X.set_camera(cam)
        for slot, t in g["textures"].items():
            X.set_texture(slot, t)
        X.set_material_textures(g["material_textures"])
        X.set_env_map(g["env_map"], g["env_rotation"])
    R.refit_chunk(0, vm, nm)
    _render_equal(R, world, "garden with moved instances")
    _trace_equal(R, world, "garden with moved instances")
    R.close()


@pytest.mark.parametrize("device", [False, True])
def test_rejections_change_nothing(gpu_required, device):
    v, n, m = terrain(20000)
    R = _renderer(v, n, m, 64, 36, spp=1, bounces=2)
    R2 = _renderer(v, None, m, 16, 16)                      # uploaded without normals
    cfg = dprt.make_config(16, 16, scene_size=2, proxy_mode=0)
    P = dprt.Renderer(cfg, rank=0, world=2)                 # index 1 is a proxy there
    P.upload_chunk(0, upload_desc(v), v, n, m)
    P.upload_proxy(1, upload_desc(v, 1), None, None)
    img0, blob0, blob2 = R.launch(), R.chunk_bvh8(0), R2.chunk_bvh8(0)
    lo, hi = v.reshape(-1, 3).min(0), v.reshape(-1, 3).max(0)
    nan, inf, out = v.copy(), v.copy(), v.copy()
    nan[5, 2] = np.nan
    inf[7, 0] = -np.inf
    out[9, 1] = hi[1] + 0.01

    def refit(X, si, vv, nn):
        if not device:
            return X.refit_chunk(si, vv, nn)
        dv = X.device_alloc(max(vv.nbytes, 4)); X.h2d(dv, np.ascontiguousarray(vv))
        dn = None
        if nn is not None:
            dn = X.device_alloc(nn.nbytes); X.h2d(dn, nn)
        try:
            X.refit_chunk_device(si, dv, dn, vv.shape[0])
        finally:
            X.device_free(dv)
            if dn is not None:
                X.device_free(dn)

    cases = [("unknown index", R, 1, v, n), ("negative index", R, -1, v, n), ("proxy object", P, 1, v, n),
             ("fewer triangles", R, 0, v[:-1], n[:-1]), ("nan", R, 0, nan, n), ("inf", R, 0, inf, n), ("outside aabb", R, 0, out, n),
             ("normals missing", R, 0, deform(v, "zscale"), None), ("normals given", R2, 0, deform(v, "zscale"), n)]
    for what, X, si, vv, nn in cases:
        with pytest.raises(dprt.DprtError):
            refit(X, si, vv, nn)
        assert_blob_equal(R.chunk_bvh8(0), blob0, what)
        assert_blob_equal(R2.chunk_bvh8(0), blob2, what)
    assert_bits_equal(R.launch(), img0, "render after the rejected refits (blob and normals unchanged)")
    for X in (R, R2, P):
        X.close()
