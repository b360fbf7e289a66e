"""The glue around the trace kernels (-m gpu).

- With proxies off the any-hit trace adds the unoccluded shadow terms to directLightingBuffer itself; no post kernel runs.
- At W = 1 dprt_render_sample shades straight from the partition output with the hits of the hit cache: no copy back to
  the path buffer, no MainRay trace launch. DPRT_SINGLE_RANK_SHORTCUT=0 turns that off.

Both must leave every buffer, the image and the statistics exactly as the oracle computes them.
"""
import numpy as np
import pytest

from helpers import D, assert_bits_equal, assert_records_equal, build_pair, dprt

pytestmark = pytest.mark.gpu

SPP, BOUNCES = 2, 3


def _render(oracle, monkeypatch, shortcut, *, serial=0, lights=None):
    monkeypatch.setenv("DPRT_SINGLE_RANK_SHORTCUT", shortcut)
    rs, world, _ = build_pair(oracle, 1, 30000, 256, 144, spp=SPP, bounces=BOUNCES, proxy_mode=0, water_frac=0.03,
                              serial_stages=serial)
    R = rs[0]
    if lights is not None:
        R.set_lights(lights); world.set_lights(lights)
    img = R.launch()
    tot = R.path_size * (1 + R.cfg.shadowPathCount)
    out = {"image": img, "paths": R.download(D.BUF_PATHS, tot), "direct": R.download(D.BUF_DIRECT),
           "env": R.download(D.BUF_ENV), "stats": R.stats(), "n": R.path_size}
    return out, world


def _check_against_oracle(g, world, what):
    img_o = world.launch()
    assert g["n"] == world.path_size(0)
    assert_bits_equal(g["image"], img_o, f"{what}: image")
    tot = g["paths"].shape[0]
    assert_records_equal(g["paths"], world.download(0, D.BUF_PATHS, tot), f"{what}: paths + shadow paths after the last bounce")
    assert_bits_equal(g["direct"], world.download(0, D.BUF_DIRECT, g["direct"].size), f"{what}: direct planes")
    assert_bits_equal(g["env"], world.download(0, D.BUF_ENV, g["env"].size), f"{what}: env")
    sg, so = g["stats"], world.stats(0)
    for k in ("rays_traverse", "rays_shade", "rays_shadow"):
        assert sg[k] == so[k], (what, k, sg[k], so[k])
    assert sg["rays_walked"] + sg["rays_shade_cached"] == so["rays_walked"], what
    assert sg["shade_cache_stale"] == 0, what


@pytest.mark.parametrize("serial", [0, 1])
def test_single_rank_shortcut_same_bits(gpu_required, oracle, monkeypatch, serial):
    """dprt_render_sample with the single-rank bounce on and off: the same bits, as the oracle's; the shortcut answers every
    MainRay query from the hit cache and saves the MainRay trace launch of each bounce."""
    on, world = _render(oracle, monkeypatch, "1", serial=serial)
    off, _ = _render(oracle, monkeypatch, "0", serial=serial)
    _check_against_oracle(on, world, f"shortcut on, serialStages={serial}")
    for k in ("image", "direct", "env"):
        assert_bits_equal(on[k], off[k], f"{k}, shortcut on vs off")
    assert_records_equal(on["paths"], off["paths"], "paths, shortcut on vs off")
    s_on, s_off = on["stats"], off["stats"]
    for k in ("rays_traverse", "rays_shade", "rays_shadow", "rays_walked", "rays_shade_cached", "walked_traverse",
              "walked_shade", "walked_shadow", "paths_partitioned", "shade_cache_stale"):
        assert s_on[k] == s_off[k], (k, s_on[k], s_off[k])
    assert s_on["rays_shade_cached"] == s_on["rays_shade"] > 0      # W = 1: every MainRay query is a hit-cache hit
    saved = s_off["kernel_launches"] - s_on["kernel_launches"]
    assert 0 < saved <= SPP * (BOUNCES + 1), saved                 # one per bounce that shaded anything


def test_subnormal_direct_terms_bit_exact(gpu_required, oracle, monkeypatch):
    """Light emission scaled by 1e-40: most direct-light terms are subnormal. The trace kernel adds them with a plain
    IEEE add (a float atomic would flush them to zero), bit-exact against the oracle."""
    lights = dprt.scene.make_lights(scale=1e-40)
    g, world = _render(oracle, monkeypatch, "1", lights=lights)
    _check_against_oracle(g, world, "subnormal lights")
    d = world.download(0, D.BUF_DIRECT, g["direct"].size)
    tiny = np.finfo(np.float32).tiny
    assert ((d != 0) & (np.abs(d) < tiny)).sum() > 0, "no subnormal direct terms: the test does not exercise them"


def test_proxy_shadow_post_unchanged(gpu_required, oracle):
    """Proxies on at W = 2: shadow rays still go through the post kernel's proxy march; image and direct planes of both
    ranks are the oracle's."""
    from test_gpu_proxy import _models
    W = 2
    rs, world, _ = build_pair(oracle, W, 6000, 128, 72, spp=2, bounces=2, proxy_mode=1, models=_models(W, False), mlp_dtype=1)
    img_g = dprt.RankGroup(rs).launch()
    img_o = world.launch()
    assert np.isfinite(img_g).all() and img_g.max() > 0
    assert_bits_equal(img_g, img_o, "proxy-on image")
    for r, R in enumerate(rs):
        d = R.download(D.BUF_DIRECT)
        assert_bits_equal(d, world.download(r, D.BUF_DIRECT, d.size), f"rank {r} direct planes")
        sg, so = R.stats(), world.stats(r)
        for k in ("rays_shadow", "nn_queries"):
            assert sg[k] == so[k], (r, k, sg[k], so[k])
    assert sum(R.stats()["nn_queries"] for R in rs) > 0
