"""GPU parity tests (-m gpu): every stage of the per-bounce loop, called through the C ABI of libdprt.so, is
compared with the oracle on the same seeded inputs.

Thresholds (fixed before any GPU number was taken, BASELINE.json north_star): hit primitive ids, routing
decisions, partition order: bit-exact. Path records, lighting buffers: bit-exact as well, because kernels and
oracle implement one arithmetic specification (DESIGN.md); where a test allows a tolerance it says so.
"""
import numpy as np
import pytest

from helpers import D, assert_bits_equal, assert_records_equal, build_pair, dprt, random_rays

pytestmark = pytest.mark.gpu


def _stagewise_bounce(R, world, rank, N, spc):
    """One bounce of stages on rank `rank` of a W=1 world, comparing buffers after every stage."""
    R.traverse(); world.traverse(rank)
    n = R.path_size
    assert n == world.path_size(rank)
    assert_records_equal(R.download(D.BUF_PATHS, n), world.download(rank, D.BUF_PATHS, n), "paths after traverse")
    assert_bits_equal(R.download(D.BUF_HIT_PRIM, n), world.download(rank, D.BUF_HIT_PRIM, n), "hit primitive ids (traverse)")
    assert_bits_equal(R.download(D.BUF_ENV), world.download(rank, D.BUF_ENV, 3 * N), "env after traverse")
    R.partition(); world.partition(rank)
    off_g, off_o = R.download(D.BUF_TRANSFER_OFFSET, 2), world.download(rank, D.BUF_TRANSFER_OFFSET, 2)
    assert_bits_equal(off_g, off_o, "transferOffset")
    assert_records_equal(R.download(D.BUF_TRANSFER, int(off_g[1])), world.download(rank, D.BUF_TRANSFER, int(off_o[1])), "transfer buffer")
    assert R.exchange() is True and world.exchange() is True
    n = R.path_size
    assert n == world.path_size(rank) == int(off_g[1])
    R.shade(); world.shade(rank)
    tot = n * (1 + spc)
    assert_records_equal(R.download(D.BUF_PATHS, tot), world.download(rank, D.BUF_PATHS, tot), "paths after shade")
    assert_bits_equal(R.download(D.BUF_HIT_PRIM, n), world.download(rank, D.BUF_HIT_PRIM, n), "hit primitive ids (shade)")
    R.reset_nn(); world.reset_nn(rank)
    R.shadow_trace(); world.shadow_trace(rank)
    assert_records_equal(R.download(D.BUF_PATHS, tot), world.download(rank, D.BUF_PATHS, tot), "paths after shadow trace")
    assert_bits_equal(R.download(D.BUF_DIRECT), world.download(rank, D.BUF_DIRECT, 3 * N * spc), "direct planes after shadow trace")
    R.frame_buffer_update(); world.frame_buffer_update(rank)
    assert_bits_equal(R.download(D.BUF_DIRECT), world.download(rank, D.BUF_DIRECT, 3 * N * spc), "direct after frame buffer update")


@pytest.mark.parametrize("tris,w,h,water", [(2000, 96, 54, 0.0), (60000, 320, 180, 0.05)])
def test_single_rank_stagewise_bit_exact(gpu_required, oracle, tris, w, h, water):
    rs, world, _ = build_pair(oracle, 1, tris, w, h, bounces=2, proxy_mode=0, water_frac=water)
    R = rs[0]
    N, spc = w * h, R.cfg.shadowPathCount
    R.enable_hit_prim(True); world.enable_hit_prim(True)
    R.reset_frame(); world.reset_frame()
    R.begin_sample(0); world.begin_sample(0)
    R.path_gen(); world.path_gen(0)
    assert_records_equal(R.download(D.BUF_PATHS, N), world.download(0, D.BUF_PATHS, N), "paths after path_gen")
    for _ in range(3):
        _stagewise_bounce(R, world, 0, N, spc)
    hit = world.download(0, D.BUF_HIT_PRIM, N)
    assert (hit >= 0).sum() > 0


def test_single_rank_image_bit_exact(gpu_required, oracle):
    rs, world, _ = build_pair(oracle, 1, 20000, 160, 90, spp=2, bounces=3, proxy_mode=0)
    img_g = rs[0].launch()
    img_o = world.launch()
    assert np.isfinite(img_g).all() and img_g.max() > 0
    assert_bits_equal(img_g, img_o, "final image, 1 rank, proxies off")
    sg, so = rs[0].stats(), world.stats(0)
    for k in ("rays_traverse", "rays_shade", "rays_shadow"):
        assert sg[k] == so[k], k
    # BVH walks: the oracle re-traces every MainRay query, libdprt answers them from the hit cache
    assert sg["rays_walked"] + sg["rays_shade_cached"] == so["rays_walked"]
    assert 0 < sg["rays_walked"] < so["rays_walked"]


@pytest.mark.parametrize("serial", [0, 1])
def test_stage_overlap_same_bits(gpu_required, oracle, serial):
    """dprt_render_sample with the ShadowRay module of bounce b on the aux stream beside the TraRay loop of bounce b+1
    (serialStages=0, default) and strictly serial (serialStages=1): same image and path records as the oracle."""
    rs, world, _ = build_pair(oracle, 1, 30000, 256, 144, spp=3, bounces=4, proxy_mode=0, water_frac=0.03, serial_stages=serial)
    R = rs[0]
    img_g, img_o = R.launch(), world.launch()
    assert_bits_equal(img_g, img_o, f"image, serialStages={serial}")
    n = R.path_size
    assert n == world.path_size(0)
    tot = n * (1 + R.cfg.shadowPathCount)
    assert_records_equal(R.download(D.BUF_PATHS, tot), world.download(0, D.BUF_PATHS, tot), "paths + shadow paths after the last bounce")
    assert_bits_equal(R.download(D.BUF_DIRECT), world.download(0, D.BUF_DIRECT, 3 * 256 * 144 * R.cfg.shadowPathCount), "direct planes")


@pytest.mark.parametrize("W,proxy", [(1, 0), (4, 0)])
def test_hit_cache_equals_retrace(gpu_required, oracle, W, proxy):
    """MainRay answered from the hit cache (default) and MainRay re-traced like kernel.cu:382-413 (mainRayRetrace=1)
    give the same bits as the oracle, which always re-traces; the cache must actually be exercised."""
    imgs = []
    for retrace in (0, 1):
        rs, world, _ = build_pair(oracle, W, 8000, 128, 72, spp=2, bounces=3, proxy_mode=proxy, main_ray_retrace=retrace)
        G = dprt.RankGroup(rs)
        imgs.append(G.launch())
        cached = sum(R.stats()["rays_shade_cached"] for R in rs)
        shaded = sum(R.stats()["rays_shade"] for R in rs)
        assert shaded > 0
        if retrace:
            assert cached == 0
        else:
            assert 0 < cached <= shaded
            if W == 1:
                assert cached == shaded      # one rank: every path that reaches MainRay was traced here in the same bounce
        if not retrace:
            img_o = world.launch()
    assert_bits_equal(imgs[0], img_o, "image with hit cache vs oracle")
    assert_bits_equal(imgs[1], img_o, "image with re-trace vs oracle")


@pytest.mark.parametrize("W,refmig", [(2, 0), (4, 0), (8, 0), (4, 1), (3, 0)])
def test_multi_rank_group_migration_bit_exact(gpu_required, oracle, W, refmig):
    """W chunk owners emulated as W contexts on one GPU; exchange through dprt_exchange_group. refmig=0: migrate loop with
    the settled deque (only travelling paths are traced / partitioned / sent); refmig=1: every iteration over every path."""
    rs, world, _ = build_pair(oracle, W, 6000, 128, 72, spp=1, bounces=2, proxy_mode=0, reference_migrate=refmig)
    G = dprt.RankGroup(rs)
    for R in rs:
        R.reset_frame()
    world.reset_frame()
    G.run_sample(0)
    world.render_sample(0)
    N, spc = 128 * 72, rs[0].cfg.shadowPathCount
    sent = 0
    for r, R in enumerate(rs):
        n = R.path_size
        assert n == world.path_size(r), f"rank {r} pathSize"
        assert_records_equal(R.download(D.BUF_PATHS, n * (1 + spc)), world.download(r, D.BUF_PATHS, n * (1 + spc)), f"rank {r} paths")
        assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * N), f"rank {r} env")
        assert_bits_equal(R.download(D.BUF_DIRECT), world.download(r, D.BUF_DIRECT, 3 * N * spc), f"rank {r} direct")
        sg, so = R.stats(), world.stats(r)
        assert sg["paths_sent_offrank"] == so["paths_sent_offrank"] and sg["exchange_iters"] == so["exchange_iters"]
        assert sg["rays_traverse"] == so["rays_traverse"] and sg["rays_walked"] + sg["rays_shade_cached"] == so["rays_walked"]
        sent += sg["paths_sent_offrank"]
    assert sent > 0, "no path migrated: the scene does not exercise the exchange"
    assert_bits_equal(G.reduce_image(0), world.image(), "reduced image")


@pytest.mark.parametrize("staged", [0, 1])
@pytest.mark.parametrize("W,spp,pgm", [(2, 1, 0), (3, 2, 1), (4, 2, 0)])
def test_multi_rank_group_peer_memory_exchange_bit_exact(gpu_required, oracle, monkeypatch, W, spp, pgm, staged):
    """The peer-memory exchange (p2p_exchange.cuh: counts kernel -> partition scattering straight into the owners' receive
    buffers -> flag barrier, no host round trip) driven for W contexts on one device: same kernels and protocol as one
    process per GPU, with plain device pointers where those use CUDA IPC mappings. Every buffer bit-exact against the oracle,
    with the per-thread and with the TMA-staged partition (DPRT_PARTITION_STAGED)."""
    monkeypatch.setenv("DPRT_P2P_GROUP", "1")
    monkeypatch.setenv("DPRT_PARTITION_STAGED", str(staged))
    rs, world, _ = build_pair(oracle, W, 6000, 128, 72, spp=spp, bounces=3, proxy_mode=0, path_gen_mode=pgm, serial_stages=1)
    G = dprt.RankGroup(rs)
    img_g, img_o = G.launch(), world.launch()
    assert all(R.p2p_enabled for R in rs), "the group did not switch to the peer-memory exchange"
    N, spc = 128 * 72, rs[0].cfg.shadowPathCount
    sent = 0
    for r, R in enumerate(rs):
        n = R.path_size
        assert n == world.path_size(r), f"rank {r} pathSize"
        assert_records_equal(R.download(D.BUF_PATHS, n * (1 + spc)), world.download(r, D.BUF_PATHS, n * (1 + spc)), f"rank {r} paths")
        assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * N), f"rank {r} env")
        assert_bits_equal(R.download(D.BUF_DIRECT), world.download(r, D.BUF_DIRECT, 3 * N * spc), f"rank {r} direct")
        sg, so = R.stats(), world.stats(r)
        assert sg["paths_sent_offrank"] == so["paths_sent_offrank"] and sg["exchange_iters"] == so["exchange_iters"]
        sent += sg["paths_sent_offrank"]
    assert sent > 0
    assert_bits_equal(img_g, img_o, "reduced image")


def test_striped_path_generation_same_image(gpu_required, oracle):
    rs, world, _ = build_pair(oracle, 2, 6000, 96, 54, bounces=1, proxy_mode=0, path_gen_mode=1)
    img_g = dprt.RankGroup(rs).launch()
    img_o = world.launch()
    assert_bits_equal(img_g, img_o, "striped path generation image")


def test_partition_random_keys_against_oracle(gpu_required, oracle, monkeypatch):
    """Work_Efficient_Scan drop-in on arbitrary uploaded paths (histogram fallback path), W = 8, ragged sizes: empty, partial
    and multi-tile launches, with the per-thread and then the TMA-staged partition (DPRT_PARTITION_STAGED, read on every
    launch) on the same context, so the staged kernel also picks up the tile state the per-thread one left."""
    W, w, h = 8, 256, 128
    cfg = dprt.make_config(w, h, scene_size=1)
    world = oracle.World(cfg, W)
    R = dprt.Renderer(cfg, rank=3, world=W)
    rng = np.random.default_rng(11)
    for staged in (0, 1):
        monkeypatch.setenv("DPRT_PARTITION_STAGED", str(staged))
        for n in (0, 1, 31, 1024, 1025, 5000, w * h):
            p = np.zeros(n, D.PATH_DTYPE)
            p["pixelIndex"] = np.arange(n)
            p["origin"] = rng.random((n, 3), dtype=np.float32)
            p["isValid"] = rng.random(n) < 0.8
            p["targetNode"] = rng.integers(-1, W + 1, n)
            R.upload(D.BUF_PATHS, p); world.upload(3, D.BUF_PATHS, p)
            R.set_path_size(n); world.set_path_size(3, n)
            R.partition(); world.partition(3)
            off_g, off_o = R.download(D.BUF_TRANSFER_OFFSET, W + 1), world.download(3, D.BUF_TRANSFER_OFFSET, W + 1)
            assert_bits_equal(off_g, off_o, f"offsets n={n} staged={staged}")
            assert_records_equal(R.download(D.BUF_TRANSFER, int(off_g[W])), world.download(3, D.BUF_TRANSFER, int(off_o[W])),
                                 f"transfer n={n} staged={staged}")


@pytest.mark.parametrize("tris,nrays", [(1, 4096), (5000, 200000), (200000, 400000)])
def test_trace_closest_operator(gpu_required, oracle, tris, nrays):
    """The optixTrace closest-hit equivalent through host buffers: primitive ids bit-exact, t bit-exact."""
    rs, world, chunks = build_pair(oracle, 1, tris, 64, 36)
    cam = dprt.scene.default_camera(640, 360)
    rays = np.concatenate([dprt.scene.camera_rays(cam)[: nrays // 2], random_rays(nrays - nrays // 2, 5)])
    hg = rs[0].trace_closest(rays)
    ho = world.trace_closest(0, rays)
    assert_bits_equal(hg["primID"], ho["primID"], "primitive ids")
    assert_bits_equal(hg["t"], ho["t"], "hit distance")
    assert rs[0].trace_closest(rays[:0]).size == 0


def test_trace_closest_full_size_properties(gpu_required, oracle):
    """BASELINE config 2 at full size (1 M triangles, 1080p primary rays): sampled oracle comparison plus
    size-independent properties over all rays."""
    rs, world, chunks = build_pair(oracle, 1, 1000000, 64, 36)
    c = chunks[0]
    cam = dprt.scene.default_camera(1920, 1080)
    rays = dprt.scene.camera_rays(cam)
    hg = rs[0].trace_closest(rays)
    hit = hg["primID"] >= 0
    assert 0.8 < hit.mean() < 1.0
    # (1) the reported hit point lies on the reported triangle's plane
    idx = np.nonzero(hit)[0]
    v = c.verts[hg["primID"][idx]].astype(np.float64).reshape(-1, 3, 3)
    nrm = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    P = rays["origin"][idx].astype(np.float64) + hg["t"][idx, None].astype(np.float64) * rays["direction"][idx].astype(np.float64)
    assert np.abs(((P - v[:, 0]) * nrm).sum(1)).max() < 1e-5
    # (2) idempotence: tracing again with tMax = t + ulp finds the same primitive; with tMax = t finds nothing closer
    again = rays.copy()
    again["tMax"] = np.where(hit, np.nextafter(hg["t"], np.float32(np.inf)), rays["tMax"])
    h2 = rs[0].trace_closest(again)
    assert_bits_equal(h2["primID"], hg["primID"], "re-trace with tMax just beyond the hit")
    # (3) oracle agreement on a bounded sample (every 16th ray)
    sub = rays[::16]
    ho = world.trace_closest(0, sub)
    assert_bits_equal(hg[::16]["primID"], ho["primID"], "sampled primitive ids at full size")
    assert_bits_equal(hg[::16]["t"], ho["t"], "sampled t at full size")


def test_traversal_counters_against_oracle_bvh8_walker(gpu_required, oracle):
    """bench.py's roofline bills BVH bytes from the ORACLE's scalar exact-tbest walk over the uploaded BVH8 (SURVEY.md 8d),
    not from the kernel's own counters. Here both are taken on the same rays: the kernel culls with a lagging tbest and expands
    nodes ahead of its triangle tests, so in the closest-hit stages it fetches at least (to within a handful of triangles met in
    another order) what the scalar walker does -- and it must stay within a small factor of it; rays walked per stage must
    agree exactly."""
    W, w, h = 2, 160, 90
    rs, world, chunks = build_pair(oracle, W, 20000, w, h, spp=1, bounces=2, proxy_mode=0, main_ray_retrace=1)
    for c in chunks:
        nodes, tris, _ = dprt.build_bvh8(c.verts, c.mats)
        world.set_bvh8(c.index, nodes, tris)
    world.count_bvh8(True)
    for R in rs:
        R.enable_counters(True); R.reset_stats()
    G = dprt.RankGroup(rs)
    img_g, img_o = G.launch(), world.launch()
    assert_bits_equal(img_g, img_o, "image with counters on")
    for r, R in enumerate(rs):
        cg, co, sg, so = R.counters(), world.bvh8_counters(r), R.stats(), world.stats(r)
        for stage, key in (("traverse", "walked_traverse"), ("shade", "walked_shade"), ("shadow_trace", "walked_shadow")):
            assert sg[key] == so[key] == co[stage][2], (r, stage, sg[key], so[key], co[stage][2])
            gn, gt = cg[stage]; on, ot, _ = co[stage]
            print(f"rank {r} {stage}: nodes gpu/oracle = {gn}/{on} = {gn / max(on, 1):.3f}, tris {gt}/{ot} = {gt / max(ot, 1):.3f}")
            if stage != "shadow_trace":       # any-hit: whichever occluder is found first ends the walk, no ordering between the two
                # (nearly) never fewer: the warp walks two nodes per step and tests triangles 32 at a time, so now and then it meets
                # the closest hit before a triangle the scalar near-first walker tests first -- a handful per 10^5
                assert gn >= 0.99 * on - 16 and gt >= 0.99 * ot - 16, (r, stage)
            assert gn <= 2.0 * on + 64 and gt <= 2.5 * ot + 64, (r, stage)
        R.close()


def test_config3_full_size_two_chunks_1080p_four_bounces(gpu_required, oracle):
    """BASELINE configs[2] at full size: 2 chunk owners x 1 M triangles, 1920x1080, bounces = 4 (5 loop iterations), ray
    migration through the exchange -- every pixel of the frame, every record of both ranks, bit-exact against the oracle
    (which needs a few seconds for it on the box's host cores). Two contexts on one device stand in for the two GPUs; the
    NCCL / peer-memory data planes are covered by test_gpu_multi.py and by bench.py's parity gate."""
    oracle.use_all_host_threads()
    W, w, h = 2, 1920, 1080
    rs, world, _ = build_pair(oracle, W, 1000000, w, h, spp=1, bounces=4, proxy_mode=0)
    G = dprt.RankGroup(rs)
    img_g, img_o = G.launch(), world.launch()
    N, spc = w * h, rs[0].cfg.shadowPathCount
    sent = 0
    for r, R in enumerate(rs):
        n = R.path_size
        assert n == world.path_size(r), f"rank {r} pathSize"
        assert_records_equal(R.download(D.BUF_PATHS, n * (1 + spc)), world.download(r, D.BUF_PATHS, n * (1 + spc)), f"rank {r} paths")
        assert_bits_equal(R.download(D.BUF_ENV), world.download(r, D.BUF_ENV, 3 * N), f"rank {r} env")
        assert_bits_equal(R.download(D.BUF_DIRECT), world.download(r, D.BUF_DIRECT, 3 * N * spc), f"rank {r} direct")
        sg, so = R.stats(), world.stats(r)
        for k in ("rays_traverse", "rays_shade", "rays_shadow", "paths_sent_offrank", "exchange_iters"):
            assert sg[k] == so[k], (r, k, sg[k], so[k])
        sent += sg["paths_sent_offrank"]
        R.close()
    assert sent > 100000, "config 3 is about migration: expected many paths to cross ranks"
    assert_bits_equal(img_g, img_o, "1080p image")
    assert np.isfinite(img_g).all() and img_g.max() > 0


@pytest.mark.parametrize("k", [2, 3])
def test_samples_in_flight_same_image(gpu_required, oracle, k):
    """K samples in flight (K contexts sharing one uploaded scene, one host thread each): every sample is computed exactly as
    before, only the per-pixel sum over samples is formed in another order -- image within 1e-6 relative of the oracle's, and
    the launch sizes / walked-ray statistics add up to the oracle's exactly."""
    rs, world, _ = build_pair(oracle, 1, 20000, 160, 90, spp=6, bounces=3, proxy_mode=0)
    R = rs[0]
    F = dprt.SamplesInFlight(R, k)
    assert len(F.ctxs) == k
    img = F.launch()
    img_o = world.launch()
    err = float(np.abs(img - img_o).max() / np.abs(img_o).max())
    assert np.isfinite(img).all() and err <= 1e-6, err
    st, so = F.stats(), world.stats(0)
    assert st["rays_traverse"] == so["rays_traverse"] and st["rays_shadow"] == so["rays_shadow"]
    assert st["rays_walked"] + st["rays_shade_cached"] == so["rays_walked"]
    F.close(); R.close()
