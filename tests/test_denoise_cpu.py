"""The denoiser's arithmetic specification (DESIGN.md 3.8) on the CPU (no GPU).

dprt_spec_denoise runs the kernels' own source on the host; tests/denoise_reference.cpp restates the specification
independently. The two must agree bit for bit, and both must agree with a float64 model that uses np.exp. The image-quality
test renders with the CPU reference (the oracle with the guide buffers) and holds the defaults to profiles/denoise_quality.txt.
"""
import ctypes as C

import numpy as np
import pytest

import denoise_reference as R
from helpers import D, dprt

DPRT_ERR_INVALID = -1
SIZES = [(1, 1), (2, 3), (5, 1), (37, 19), (256, 144)]          # (width, height)
PARAMS = [{}, {"sigma_color": 0.5, "sigma_normal": 0.25, "sigma_albedo": 0.05}, {"sigma_color": 8.0, "sigma_normal": 3.0, "sigma_albedo": 1.0}]


def frame(w, h, seed):
    """Colour up to ~1e3 (HDR) on a smooth field, albedo in blocks with zeros (whole pixels and single channels), unit
    normals in blocks with a little jitter, zero normals (and albedo) where the camera ray would have missed."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = 1.0 + 0.5 * np.sin(xx / 7.0)[..., None] * np.cos(yy / 5.0)[..., None] + np.zeros((h, w, 3), np.float32)
    color = (base * rng.gamma(2.0, 0.5, (h, w, 3))).astype(np.float32)
    hot = rng.random((h, w)) < 0.01
    color[hot] *= rng.uniform(100.0, 1000.0, (int(hot.sum()), 1)).astype(np.float32)
    bx, by = (xx // 6).astype(int), (yy // 5).astype(int)
    pal = rng.uniform(0.05, 0.9, (64, 3)).astype(np.float32)
    albedo = pal[(bx * 7 + by * 3) % 64]
    albedo[rng.random((h, w, 3)) < 0.03] = 0.0
    nrm = rng.normal(size=(64, 3))
    normal = nrm[(bx * 5 + by * 11) % 64] + 0.05 * rng.normal(size=(h, w, 3))
    normal = (normal / np.linalg.norm(normal, axis=-1, keepdims=True)).astype(np.float32)
    miss = rng.random((h, w)) < 0.05
    albedo[miss] = 0.0
    normal[miss] = 0.0
    return color.astype(np.float32), albedo.astype(np.float32), normal


@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("iterations", [1, 5, 10])
@pytest.mark.parametrize("pi", range(len(PARAMS)))
def test_product_equals_reference_bitwise(w, h, iterations, pi):
    c, a, n = frame(w, h, seed=1000 * w + h)
    p = dict(PARAMS[pi], iterations=iterations)
    got = dprt.spec_denoise(c, a, n, **p)
    ref = R.denoise(c, a, n, **p)
    assert np.isfinite(got).all()
    bad = np.nonzero(got.view(np.uint32) != ref.view(np.uint32))
    assert bad[0].size == 0, f"{bad[0].size} values differ; first {tuple(b[0] for b in bad)}: {got[bad][0]!r} vs {ref[bad][0]!r}"


def test_defaults_are_the_stated_ones():
    c, a, n = frame(37, 19, 5)
    assert np.array_equal(dprt.spec_denoise(c, a, n).view(np.uint32), dprt.spec_denoise(c, a, n, **D.DENOISE_DEFAULTS).view(np.uint32))
    assert D.DENOISE_DEFAULTS == R.DEFAULTS


@pytest.mark.parametrize("w,h", [(37, 19), (256, 144)])
@pytest.mark.parametrize("iterations", [1, 5, 10])
@pytest.mark.parametrize("pi", range(len(PARAMS)))
def test_float64_model(w, h, iterations, pi):
    """Binary32 against float64 with np.exp: |f32 - f64| <= 1e-4 (|f64| + 1e-3), i.e. a relative 1e-4 with an absolute floor
    for the near-zero outputs of zero-albedo channels."""
    c, a, n = frame(w, h, seed=7 * w + h)
    p = dict(PARAMS[pi], iterations=iterations)
    got = dprt.spec_denoise(c, a, n, **p).astype(np.float64)
    model = R.denoise_f64(c, a, n, **p)
    err = np.abs(got - model) / (np.abs(model) + 1e-3)
    assert err.max() <= 1e-4, f"max scaled error {err.max():.3g} at {np.unravel_index(err.argmax(), err.shape)}"


def test_exp_neg_endpoints():
    x = np.array([0.0, -0.0, 88.0, 88.5, 1e30, np.inf, np.nan], np.float32)
    y = R.exp_neg(x)
    assert y[0] == 1.0 and y[1] == 1.0
    assert (y[2:] == 0.0).all()
    assert R.exp_neg(np.array([np.nextafter(np.float32(88.0), np.float32(0.0))], np.float32))[0] > 0.0


def test_exp_neg_monotone_and_accurate():
    """Every 61st binary32 in [0, 88): non-increasing; relative error <= 1e-7 against exp while the result is normal,
    at most one subnormal ulp (2^-149) beyond."""
    top = int(np.float32(88.0).view(np.uint32))
    bits = np.arange(0, top, 61, dtype=np.uint32)
    x = bits.view(np.float32)
    y = R.exp_neg(x)
    assert (np.diff(y) <= 0).all(), "det_exp_neg is not non-increasing"
    e = np.exp(-x.astype(np.float64))
    normal = e >= np.finfo(np.float32).tiny
    rel = np.abs(y[normal] - e[normal]) / e[normal]
    assert rel.max() <= 1e-7, rel.max()
    assert (np.abs(y[~normal] - e[~normal]) <= 2.0 ** -149).all()


def test_constant_image_is_a_fixed_point():
    h, w = 24, 40
    c = np.full((h, w, 3), [0.7, 1.9, 3.1], np.float32)
    a = np.full((h, w, 3), [0.25, 0.5, 0.8], np.float32)
    n = np.full((h, w, 3), [0.0, 0.6, 0.8], np.float32)
    for it in (1, 5, 10):
        out = dprt.spec_denoise(c, a, n, iterations=it)
        ulp = np.spacing(c)
        assert (np.abs(out - c) <= 4 * ulp).all(), (it, np.abs(out - c).max())


@pytest.mark.parametrize("guide", ["albedo", "normal"])
def test_step_edge_in_a_guide_is_kept(guide):
    """Left and right halves differ in one guide and in colour; pixels two or more columns from the edge keep their side's
    value within 1e-3 (relative) at the defaults."""
    h, w, edge = 16, 32, 16
    c = np.zeros((h, w, 3), np.float32)
    a = np.full((h, w, 3), 0.5, np.float32)
    n = np.zeros((h, w, 3), np.float32)
    n[..., 2] = 1.0
    c[:, :edge] = 0.2
    c[:, edge:] = 2.0
    if guide == "albedo":
        a[:, edge:] = 0.8
    else:
        n[:, edge:] = [1.0, 0.0, 0.0]
    out = dprt.spec_denoise(c, a, n)
    keep = np.r_[0:edge - 2, edge + 2:w]
    err = np.abs(out[:, keep] - c[:, keep]) / c[:, keep]
    assert err.max() <= 1e-3, f"{guide} edge: {err.max():.3g}"


def test_quality_against_high_spp():
    """4 spp denoised at the defaults against 256 spp (CPU reference renders, 128 x 72, 2 bounces). The bounds are the
    measured ratios of profiles/denoise_quality.txt (0.965 and 0.525) with a little room: the landscape's guides are noisy
    at 4 spp (random sub-pixel triangles) and half its relMSE sits in 1 % of the pixels, which the filter keeps apart."""
    bound = {"landscape": 0.98, "garden": 0.6}
    for scene, b in bound.items():
        low, high = R.render(scene, 128, 72, 4), R.render(scene, 128, 72, 256)
        noisy = R.rel_mse(low[0], high[0])
        den = R.rel_mse(dprt.spec_denoise(*low), high[0])
        assert den <= b * noisy, f"{scene}: denoised relMSE {den:.4f}, noisy {noisy:.4f}, ratio {den / noisy:.3f} > {b}"


def test_rejected_parameters():
    lib = dprt.load_library()
    c, a, n = frame(8, 4, 3)
    o = np.zeros_like(c)
    P = lambda **kw: C.byref(D.DenoiseParams(**{**D.DENOISE_DEFAULTS, **kw}))
    ptr = lambda x: x.ctypes.data_as(C.c_void_p)
    call = lambda p, w=8, h=4, arrs=(c, a, n, o): lib.dprt_spec_denoise(p, w, h, *[None if x is None else ptr(x) for x in arrs])
    assert call(None) == 0 and call(P()) == 0
    for kw in ({"iterations": 0}, {"iterations": 11}, {"iterations": -3}, {"sigma_color": 0.0}, {"sigma_normal": -1.0},
               {"sigma_albedo": float("nan")}, {"sigma_color": float("inf")}, {"sigma_normal": 1e-20}, {"sigma_albedo": 1e30},
               {"sigma_color": 1e-17, "iterations": 10}):
        assert call(P(**kw)) == DPRT_ERR_INVALID, kw
    assert call(P(sigma_color=1e-17, iterations=1)) == 0       # Kc_0 is finite; only 4^9 Kc_0 overflows
    for w, h in ((0, 4), (8, 0), (-1, 4), (1 << 15, 1 << 14)):  # the last is 2^29 pixels: rejected before the arrays are read
        assert call(None, w, h) == DPRT_ERR_INVALID, (w, h)
    for i in range(4):
        arrs = [c, a, n, o]
        arrs[i] = None
        assert call(None, arrs=arrs) == DPRT_ERR_INVALID, i
    with pytest.raises(dprt.DprtError):
        dprt.spec_denoise(c, a, n, iterations=11)
