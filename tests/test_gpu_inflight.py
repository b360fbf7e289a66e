"""What bench.py times, held to exact predictions: samples in flight per context, and the device-resident trace and MLP operators.

Samples in flight (host.SamplesInFlight, DESIGN.md 3.5): context j starts from reset_frame and renders samples j, j + K,
j + 2K, ... in that order, so its colour sums (BUF_DIRECT plane 0, BUF_ENV) are the oracle's after the same reset_frame and
the same samples, bit for bit, however the K contexts overlap on the device. accumulate() adds contexts 1 .. K-1 into
context 0 in index order with a plain fp32 add (accumulate_kernel), and dprt_reduce_image at one rank is
(direct + env) / (float)spp (image_average_kernel, compiled without contraction). The same float32 operations in numpy
therefore predict the frame image bit for bit (`predict_inflight`); the AOV sums and reduce_aov follow the same rule.

The GPU tests carry their own gpu mark; the last test needs no GPU: it shows that the prediction differs from the serial
image, so the exact checks can tell the in-flight summation order from the one-sample-at-a-time one.
"""
from collections import namedtuple
from types import SimpleNamespace

import numpy as np
import pytest

from helpers import D, assert_bits_equal, build_garden_pair, build_pair, dprt

STAT_KEYS = ("rays_traverse", "rays_shade", "rays_shadow")


# ---- prediction ------------------------------------------------------------------------------------------------------

def deal(k, first, count):
    """The samples each of k contexts renders in SamplesInFlight.run_samples(first, count), in the order it renders them."""
    return [list(range(first + j, first + count, k)) for j in range(k)]


def predict_inflight(world, k, calls, timed_from=0, aov=False):
    """What k samples in flight on one rank compute, from the oracle world (one world, reused context by context).

    calls: the (first, count) arguments of the run_samples calls after one reset_frame. Statistics are those of the calls from
    index timed_from on (reset_stats on every context between calls timed_from - 1 and timed_from); the oracle has no
    reset_stats, so they are the difference of world.stats(0) around those calls. aov: world is an AovWorld.
    Returns a dict of per-context lists -- samples[j], direct[j] (plane 0, 3N), env[j] (3N), aov[j] (6N), stats[j] --
    and the frame: direct_sum, env_sum, aov_sum (context 0 after accumulate()), image (reduce_image(0), [H, W, 3]),
    albedo and normal (reduce_aov(0))."""
    N, spp = world.N, np.float32(world.cfg.spp)
    P = {"samples": [], "direct": [], "env": [], "aov": [], "stats": []}
    for j in range(k):
        world.reset_frame()
        if aov:
            world.enable_aov()            # a zeroed guide buffer: the oracle's reset_frame leaves it alone
        mine, before = [], world.stats(0)
        for i, (first, count) in enumerate(calls):
            if i == timed_from:
                before = world.stats(0)
            for s in deal(k, first, count)[j]:
                world.render_sample(s)
                mine.append(s)
        after = world.stats(0)
        P["stats"].append({key: after[key] - before[key] for key in after})
        P["samples"].append(mine)
        P["direct"].append(world.download(0, D.BUF_DIRECT, 3 * N))
        P["env"].append(world.download(0, D.BUF_ENV, 3 * N))
        if aov:
            P["aov"].append(world.aov_buffer(0))
    d, e = P["direct"][0].copy(), P["env"][0].copy()
    a = P["aov"][0].copy() if aov else None
    for j in range(1, k):                 # accumulate(): into context 0, in index order
        d += P["direct"][j]
        e += P["env"][j]
        if aov:
            a += P["aov"][j]
    P["direct_sum"], P["env_sum"], P["aov_sum"] = d, e, a
    shape = (world.cfg.height, world.cfg.width, 3)
    P["image"] = ((d + e) / spp).reshape(shape)
    if aov:
        P["albedo"], P["normal"] = (a[:3 * N] / spp).reshape(shape), (a[3 * N:] / spp).reshape(shape)
    return P


def _context_state(F, aov=False):
    """Per context after its samples: (direct plane 0, env, AOV sums or None, statistics)."""
    for X in F.ctxs:
        X.synchronize()
    return [(X.download(D.BUF_DIRECT, 3 * X.N), X.download(D.BUF_ENV, 3 * X.N), X.download(D.BUF_AOV, 6 * X.N) if aov else None,
             X.stats()) for X in F.ctxs]


def _check_contexts(got, P, retrace, before=None, what=""):
    """Every context's buffers bit for bit and its statistics exactly against the prediction. before: statistics of every
    context taken before the samples (None: they were reset)."""
    for j, (d, e, a, sg) in enumerate(got):
        if before is not None:
            sg = {key: sg[key] - before[j][key] for key in sg}
        tag = f"{what}context {j} (samples {P['samples'][j]})"
        assert_bits_equal(d, P["direct"][j], f"{tag}: direct plane 0")
        assert_bits_equal(e, P["env"][j], f"{tag}: env")
        if a is not None:
            assert_bits_equal(a, P["aov"][j], f"{tag}: AOV sums")
        so = P["stats"][j]
        for key in STAT_KEYS:
            assert sg[key] == so[key], (tag, key, sg[key], so[key])
        # the oracle re-traces every MainRay query; libdprt answers them from the hit cache unless mainRayRetrace is on
        assert sg["rays_walked"] + sg["rays_shade_cached"] == so["rays_walked"], (tag, sg["rays_walked"], sg["rays_shade_cached"], so["rays_walked"])
        if retrace:
            assert sg["rays_shade_cached"] == 0, tag
        elif so["rays_shade"] > 0:
            assert sg["rays_shade_cached"] > 0, f"{tag}: the hit cache answered nothing"


# ---- bench.py's N = 1 sequence at full size ----------------------------------------------------------------------------

FULL_W, FULL_H = 1920, 1080


@pytest.fixture(scope="module")
def bench_scene():
    """bench.py's N = 1 scene (build_world_scene with the default --tris and --layout): one 1 M-triangle chunk."""
    cam = dprt.scene.default_camera(FULL_W, FULL_H)
    chunks, mats, lights = dprt.scene.make_scene(1, 1_000_000, layout="slabs", camera=cam)
    return chunks, mats, lights, cam


def _bench_renderer(O, scene, cfg, with_world=True):
    chunks, mats, lights, cam = scene
    R = dprt.Renderer(cfg, rank=0, world=1)
    world = O.World(cfg, 1) if with_world else None
    for c in chunks:
        R.upload_chunk(c.index, c.desc(False), c.verts, c.normals, c.mats)
        if world is not None:
            world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
    for X in (R, world) if world is not None else (R,):
        X.set_materials(mats); X.set_lights(lights); X.set_camera(cam)
    return R, world


def _bench_config():
    """bench.py's N = 1 config at its defaults (run_dprt: --bounces 4 --mlp-dtype 1 --retrace 0 --serial 0, no proxies)."""
    return dprt.make_config(FULL_W, FULL_H, spp=1, bounces=4, scene_size=1, proxy_mode=0, path_gen_mode=0, mlp_dtype=1,
                            main_ray_retrace=0, serial_stages=0)


@pytest.mark.gpu
def test_bench_n1_six_samples_in_flight_bit_exact(gpu_required, oracle, bench_scene):
    """The timed region of bench.py's N = 1 line at its defaults (--warmup 3 --steps 8 --inflight 6), as run_dprt drives it
    (bench.py lines 519-547): SamplesInFlight(R, 6); F.reset_frame(); F.run_samples(0, warmup * K); synchronize and
    reset_stats every context; timer_start on every context; F.run_samples(warmup * K, steps); timer_stop; the Mrays/s
    numerator is rays_walked summed over the contexts; --dump-outputs then takes F.accumulate() and R.reduce_image(0).
    Contexts 0-1 render 5 samples, contexts 2-5 render 4; each one's buffers and timed statistics are the oracle's, and the
    frame image is the predicted composition bit for bit."""
    oracle.use_all_host_threads()
    K, warmup, steps = 6, 3, 8
    cfg = _bench_config()
    R, world = _bench_renderer(oracle, bench_scene, cfg)
    F = dprt.SamplesInFlight(R, K)
    try:
        assert len(F.ctxs) == K
        F.reset_frame()
        F.run_samples(0, warmup * K)
        for X in F.ctxs:
            X.synchronize()
        for X in F.ctxs:
            X.reset_stats()
        for X in F.ctxs:
            X.timer_start()
        F.run_samples(warmup * K, steps)
        ms = max(X.timer_stop() for X in F.ctxs)
        assert ms > 0
        got = _context_state(F)
        calls = [(0, warmup * K), (warmup * K, steps)]
        P = predict_inflight(world, K, calls, timed_from=1)
        assert [len(s) for s in P["samples"]] == [5, 5, 4, 4, 4, 4]
        _check_contexts(got, P, retrace=0)
        assert F.stats()["rays_walked"] == sum(g[3]["rays_walked"] for g in got) > 0      # bench.py's Mrays/s numerator
        F.accumulate()
        img = R.reduce_image(0)
        assert np.isfinite(img).all() and img.max() > 0
        assert_bits_equal(img, P["image"], "frame image after accumulate + reduce_image (26 samples, 6 in flight)")
    finally:
        F.close(); R.close(); world.close()


# ---- a small grid ------------------------------------------------------------------------------------------------------

Case = namedtuple("Case", "k spp serial retrace water scene aov w h tris bounces")


def _case(k, spp, serial=0, retrace=0, water=0.0, scene="terrain", aov=False, w=160, h=90, tris=20000, bounces=3):
    return Case(k, spp, serial, retrace, water, scene, aov, w, h, tris, bounces)


# spp in {1, K - 1, K + 1, 2K + 1} for every K: idle contexts (spp < K), unequal counts, non-power-of-two averages
GRID = [
    _case(2, 1), _case(2, 3, serial=1), _case(2, 5, retrace=1),
    _case(3, 1, retrace=1), _case(3, 2, serial=1), _case(3, 4), _case(3, 7, serial=1, retrace=1),
    _case(6, 1, serial=1), _case(6, 5, retrace=1), _case(6, 7, water=0.03),
    _case(6, 13, serial=1, retrace=1, w=256, h=144, tris=30000, bounces=4),
    _case(3, 4, scene="garden", bounces=2),
    _case(3, 5, aov=True, bounces=2),
]


def _case_id(c):
    return (f"K{c.k}-spp{c.spp}-serial{c.serial}-retrace{c.retrace}" + (f"-water{c.water}" if c.water else "")
            + ("" if c.scene == "terrain" else f"-{c.scene}") + ("-aov" if c.aov else "") + f"-{c.w}x{c.h}")


def _build(O, c, gpu):
    """(renderer or None, oracle world) of a grid case; the world is an AovWorld for the AOV case."""
    if c.aov:
        from aov_reference import AovWorld
        O = SimpleNamespace(World=AovWorld)
    if c.scene == "garden":
        rs, world, _ = build_garden_pair(O, 1, c.w, c.h, spp=c.spp, bounces=c.bounces, gpu=gpu, main_ray_retrace=c.retrace,
                                         serial_stages=c.serial)
    else:
        rs, world, _ = build_pair(O, 1, c.tris, c.w, c.h, spp=c.spp, bounces=c.bounces, water_frac=c.water, main_ray_retrace=c.retrace,
                                  serial_stages=c.serial, gpu=gpu)
    return (rs[0] if rs else None), world


@pytest.mark.gpu
@pytest.mark.parametrize("c", GRID, ids=_case_id)
def test_samples_in_flight_grid_bit_exact(gpu_required, oracle, c):
    """Per context: buffers bit for bit and statistics exactly as the oracle's over that context's samples; context 0's sums
    after accumulate(), the image of reduce_image(0) (and the AOVs of reduce_aov(0)) as predicted; then two F.launch() in a
    row give the same bits (nothing carried across frames: tickets, queue heads, hit caches)."""
    R, world = _build(oracle, c, gpu=True)
    F = dprt.SamplesInFlight(R, c.k)
    try:
        assert len(F.ctxs) == c.k
        if c.aov:
            F.enable_aov()
        P = predict_inflight(world, c.k, [(0, c.spp)], aov=c.aov)
        before = [X.stats() for X in F.ctxs]
        F.reset_frame()
        F.run_samples(0, c.spp)
        _check_contexts(_context_state(F, c.aov), P, c.retrace, before=before)
        F.accumulate()
        R.synchronize()
        assert_bits_equal(R.download(D.BUF_DIRECT, 3 * R.N), P["direct_sum"], "context 0 direct plane 0 after accumulate")
        assert_bits_equal(R.download(D.BUF_ENV, 3 * R.N), P["env_sum"], "context 0 env after accumulate")
        img = R.reduce_image(0)
        assert np.isfinite(img).all() and img.max() > 0
        assert_bits_equal(img, P["image"], "reduce_image after accumulate")
        if c.aov:
            assert_bits_equal(R.download(D.BUF_AOV, 6 * R.N), P["aov_sum"], "context 0 AOV sums after accumulate")
            a, n = F.reduce_aov(0)
            assert_bits_equal(a, P["albedo"], "reduce_aov albedo"); assert_bits_equal(n, P["normal"], "reduce_aov normal")
            assert P["albedo"].max() > 0 and np.abs(P["normal"]).max() > 0
        for rep in (1, 2):
            assert_bits_equal(F.launch(), P["image"], f"F.launch() #{rep}")
            if c.aov:
                a, n = F.reduce_aov(0)
                assert_bits_equal(a, P["albedo"], f"albedo after F.launch() #{rep}")
                assert_bits_equal(n, P["normal"], f"normal after F.launch() #{rep}")
    finally:
        F.close(); R.close(); world.close()


# ---- device-resident closest hit as bench_primary calls it -------------------------------------------------------------

SENTINEL = 64


def _pattern(nbytes):
    return np.full(nbytes + SENTINEL, 0xA5, np.uint8)


def _hits_and_tail(R, dev, n):
    raw = np.zeros(n * D.HIT_DTYPE.itemsize + SENTINEL, np.uint8)
    R.d2h(raw, dev)
    return raw[:-SENTINEL].view(D.HIT_DTYPE), raw[-SENTINEL:]


@pytest.mark.gpu
def test_trace_closest_device_as_bench_primary(gpu_required, oracle, bench_scene):
    """bench_primary (bench.py lines 276-296): 1080p camera rays on the 1 M-triangle chunk, three trace_closest_device launches
    back to back with no sync, flush_l2 before a fourth; every hit buffer equals the host trace_closest bit for bit (and the
    oracle on every 16th ray) and the 64 bytes behind it stay untouched. Then the counters-instrumented instantiation:
    same hits, and its node / triangle counts within the bounds test_traversal_counters_against_oracle_bvh8_walker allows
    against the oracle's scalar walk over the product's BVH8 blob (whose primitive ids agree too). n = 0 writes nothing."""
    oracle.use_all_host_threads()
    R, world = _bench_renderer(oracle, bench_scene, _bench_config())
    rays = dprt.scene.camera_rays(bench_scene[3])
    n = rays.size
    hb = n * D.HIT_DTYPE.itemsize
    d_rays = R.device_alloc(rays.nbytes)
    bufs = [R.device_alloc(hb + SENTINEL) for _ in range(4)]
    try:
        R.h2d(d_rays, rays)
        for b in bufs:
            R.h2d(b, _pattern(hb))
        R.synchronize()
        for b in bufs[:3]:
            R.trace_closest_device(d_rays, n, b)
        R.flush_l2()
        R.trace_closest_device(d_rays, n, bufs[3])
        R.synchronize()
        ref = R.trace_closest(rays)
        assert 0.8 < (ref["primID"] >= 0).mean() < 1.0
        ho = world.trace_closest(0, rays[::16])
        assert_bits_equal(ref[::16]["primID"], ho["primID"], "host trace_closest primitive ids vs oracle (every 16th ray)")
        assert_bits_equal(ref[::16]["t"], ho["t"], "host trace_closest t vs oracle (every 16th ray)")
        for i, b in enumerate(bufs):
            hits, tail = _hits_and_tail(R, b, n)
            assert_bits_equal(hits, ref, f"device hits, launch {i + 1}")
            assert (tail == 0xA5).all(), f"launch {i + 1} wrote past the hits"

        # the instrumented instantiation (bench_primary's roofline bytes)
        R.h2d(bufs[0], _pattern(hb))
        R.reset_stats(); R.enable_counters(True)
        R.trace_closest_device(d_rays, n, bufs[0]); R.synchronize()
        gn, gt = R.counters()["trace_closest"]
        R.enable_counters(False)
        hits, tail = _hits_and_tail(R, bufs[0], n)
        assert_bits_equal(hits, ref, "device hits, counters on")
        assert (tail == 0xA5).all(), "the instrumented launch wrote past the hits"
        c = bench_scene[0][0]
        nodes, tris, _ = dprt.build_bvh8(c.verts, c.mats)
        hw, on, ot = oracle.bvh8_trace(nodes, tris, rays)
        assert_bits_equal(hw["primID"], ref["primID"], "oracle BVH8 walk primitive ids")
        print(f"trace_closest: nodes gpu/oracle = {gn}/{on} = {gn / max(on, 1):.3f}, tris {gt}/{ot} = {gt / max(ot, 1):.3f}")
        assert 0.99 * on - 16 <= gn <= 2.0 * on + 64, (gn, on)
        assert 0.99 * ot - 16 <= gt <= 2.5 * ot + 64, (gt, ot)

        # n = 0: nothing written
        R.h2d(bufs[1], _pattern(hb))
        R.trace_closest_device(d_rays, 0, bufs[1]); R.synchronize()
        raw = np.zeros(hb + SENTINEL, np.uint8)
        R.d2h(raw, bufs[1])
        assert (raw == 0xA5).all(), "n = 0 wrote to the hit buffer"
    finally:
        for b in bufs:
            R.device_free(b)
        R.device_free(d_rays)
        R.close(); world.close()


# ---- device-resident MLP as bench_mlp calls it -------------------------------------------------------------------------

def _module_float64(m, x16, rows=1 << 16):
    import torch
    m64 = m.double()
    x = torch.from_numpy(x16.view(np.float16).astype(np.float64))
    with torch.no_grad():
        return np.concatenate([m64(x[i:i + rows]).numpy().reshape(-1) for i in range(0, x.shape[0], rows)])


@pytest.mark.gpu
def test_mlp_infer_device_as_bench_mlp(gpu_required, oracle):
    """bench_mlp (bench.py lines 320-346): the 4Res256 proxy, 2^20 fp16 queries from default_rng(0), bf16 and fp16 operands,
    3 launches of mlp_infer_device then 10 back to back. The last output equals host mlp_infer bit for bit, is within 1e-3
    (fp16) / 4e-3 (bf16) of the float64 PyTorch module (and, fp16, of oracle.mlp_forward), and the bytes behind y stay
    untouched."""
    import torch
    torch.manual_seed(19990201)
    m = dprt.proxy.make_proxy(256, 4).eval()
    blob = dprt.proxy.pack_module(m)
    n = 1 << 20
    x = np.random.default_rng(0).random((n, 5)).astype(np.float16).view(np.uint16)
    y64 = _module_float64(m, x)
    yo, _ = oracle.mlp_forward(blob, x)
    for name, dt, tol in (("bf16", 0, 4e-3), ("fp16", 1, 1e-3)):
        cfg = dprt.make_config(16, 16, scene_size=2, proxy_mode=1, mlp_dtype=dt)
        P = dprt.Renderer(cfg, rank=0, world=2)
        P.upload_proxy(1, dprt.make_object_desc(1, [0, 0, 0], [1, 1, 1], is_proxy=1), blob, blob)
        dx, dy = P.device_alloc(x.nbytes), P.device_alloc(n * 2 + SENTINEL)
        try:
            P.h2d(dx, x)
            P.h2d(dy, _pattern(n * 2))
            for _ in range(3):
                P.mlp_infer_device(1, 0, dx, n, dy)
            P.synchronize()
            for _ in range(10):
                P.mlp_infer_device(1, 0, dx, n, dy)
            P.synchronize()
            raw = np.zeros(n * 2 + SENTINEL, np.uint8)
            P.d2h(raw, dy)
            assert (raw[-SENTINEL:] == 0xA5).all(), f"{name}: wrote past y"
            y = raw[:-SENTINEL].view(np.uint16)
            assert_bits_equal(y, P.mlp_infer(1, 0, x), f"{name}: device-resident vs host mlp_infer")
            yf = y.view(np.float16).astype(np.float64)
            err = float(np.abs(yf - y64).max())
            print(f"{name}: max |gpu - float64 module| = {err:.3e}")
            assert np.isfinite(yf).all() and err <= tol, (name, err)
            if dt == 1:
                assert float(np.abs(yf - yo).max()) <= tol
        finally:
            P.device_free(dx); P.device_free(dy)
            P.close()


# ---- the exact checks can tell the orders apart (no GPU) ----------------------------------------------------------------

def test_inflight_dealing_is_run_samples_rule():
    """deal() is the rule SamplesInFlight.run_samples applies, for the calls the tests above make."""
    class Recorder:
        def __init__(self):
            self.seen = []

        def run_sample(self, s):
            self.seen.append(s)

    for k, calls in ((6, [(0, 18), (18, 8)]), *((c.k, [(0, c.spp)]) for c in GRID)):
        F = object.__new__(dprt.SamplesInFlight)
        F.ctxs = [Recorder() for _ in range(k)]
        for first, count in calls:
            F.run_samples(first, count)
        want = [sum((deal(k, first, count)[j] for first, count in calls), []) for j in range(k)]
        assert [X.seen for X in F.ctxs] == want, (k, calls)


def test_inflight_prediction_differs_from_serial_image(oracle):
    """For every grid case in which some context renders two or more samples, the predicted in-flight image differs from the
    one-sample-at-a-time image (world.launch()) in at least one pixel's bits: the exact comparison would catch a GPU that
    summed the samples in the serial order (or any other)."""
    checked = 0
    for c in GRID:
        if c.k < 2 or c.spp <= c.k:
            continue
        _, world = _build(oracle, c, gpu=False)
        P = predict_inflight(world, c.k, [(0, c.spp)], aov=c.aov)
        serial = world.launch()
        diff = int((P["image"].view(np.uint32) != serial.view(np.uint32)).sum())
        print(f"{_case_id(c)}: {diff} of {serial.size} values differ from the serial image")
        assert diff > 0, _case_id(c)
        world.close()
        checked += 1
    assert checked >= 5
