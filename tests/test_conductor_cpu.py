"""CPU tests of the rough conductor (bsdfType 2, DESIGN.md 3.12): the product's host compile of conductor.cuh
(dprt_spec_conductor_sample / _eval) against the restatement of tests/conductor_reference.cpp bit for bit, sampling against evaluation through a
float64 model, physical sanity, and the DPRTSCN3 scene file. No GPU needed; tests/test_gpu_conductor.py renders it."""
import hashlib

import numpy as np
import pytest

import conductor_reference as ref
from helpers import dprt

ROUGH = [0.0, 1e-4, 0.05, 0.3, 1.0]
XI_MAX = np.float32(1.0 - 2.0 ** -24)            # the largest value rnd() returns


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _wo_grid():
    """Local outgoing directions: near-normal, generic, grazing, down to the smallest positive binary32 cosines."""
    out = []
    for z in [1.0, 0.999999, 0.9, 0.5, 0.1, 1e-3, 1e-6, 1e-20, 1e-38, 1e-45]:
        for phi in [0.0, 0.7, 2.0, 3.9, 5.5]:
            s = np.sqrt(max(0.0, 1.0 - z * z))
            w = np.array([s * np.cos(phi), s * np.sin(phi), 0.0], np.float32)
            w[2] = np.float32(z)                     # keep the tiny cosine exactly (the float64 normalise would not)
            out.append(w)
    out.append(np.array([0.0, 0.0, 1.0], np.float32))
    out.append(np.array([1.0, 0.0, 0.0], np.float32))                  # wo.z = 0: the rough lobe ends the path
    out.append(np.array([0.6, 0.0, -0.8], np.float32))                 # below the surface
    return np.array(out, np.float32)


def _grid():
    wo = _wo_grid()
    f0s = np.array([[0, 0, 0], [1, 1, 1], [0.95, 0.64, 0.54], [0.1, 0.5, 0.9]], np.float32)
    xis = np.array([[0, 0], [0, XI_MAX], [XI_MAX, 0], [XI_MAX, XI_MAX], [0.5, 0.5], [0.25, 0.9], [0.999, 0.001]], np.float32)
    W, F, R, X = np.meshgrid(np.arange(len(wo)), np.arange(len(f0s)), np.arange(len(ROUGH)), np.arange(len(xis)), indexing="ij")
    return f0s[F.ravel()], np.array(ROUGH, np.float32)[R.ravel()], wo[W.ravel()], xis[X.ravel()]


def test_host_compile_equals_reference():
    f0, r, wo, xi = _grid()
    wi, wt = dprt.spec_conductor_sample(f0, r, wo, xi)
    wio, wto = ref.sample(f0, r, wo, xi)
    assert np.array_equal(_bits(wi), _bits(wio)) and np.array_equal(_bits(wt), _bits(wto))
    assert np.isfinite(wi).all() and np.isfinite(wt).all()
    live = (wt != 0).any(axis=1)
    assert live.sum() > 0.5 * live.size
    # light directions: the sampled ones, every grid direction, and random ones of both hemispheres
    rng = np.random.default_rng(7)
    wl = np.concatenate([wi, _wo_grid()[rng.integers(0, len(_wo_grid()), len(wi))], _unit(rng.normal(size=(len(wi), 3)))]).astype(np.float32)
    f0e, re, woe = np.tile(f0, (3, 1)), np.tile(r, 3), np.tile(wo, (3, 1))
    f = dprt.spec_conductor_eval(f0e, re, woe, wl)
    assert np.array_equal(_bits(f), _bits(ref.evaluate(f0e, re, woe, wl)))
    assert np.isfinite(f).all() and (f >= 0).all()
    assert not f[re == 0].any()                                         # the mirror is a delta: no light sample reaches it


def test_mirror_and_dead_paths():
    wo = _wo_grid()
    f0 = np.array([0.9, 0.5, 0.1], np.float32)
    wi, wt = dprt.spec_conductor_sample(f0, 0.0, wo, [0.3, 0.6])
    assert np.array_equal(wi, wo * np.array([-1, -1, 1], np.float32))
    m = 1.0 - np.clip(wo[:, 2:3].astype(np.float64), 0, 1)
    assert np.allclose(wt, f0 + (1 - f0) * m ** 5, rtol=1e-6, atol=1e-7)
    wi, wt = dprt.spec_conductor_sample(f0, 0.3, wo, [0.3, 0.6])
    dead = wo[:, 2] <= 0
    assert not wi[dead].any() and not wt[dead].any()
    assert (wi[(wt != 0).any(axis=1), 2] > 0).all()


# ---- float64 model of the lobe ----
def _f_model(alpha, wo, wi):
    """f(wi, wo) with F0 = 1: D G2 / (4 wo.z wi.z), in float64, from the textbook formulas."""
    h = _unit(wo + wi)
    a2 = alpha * alpha
    D_ = a2 / (np.pi * ((a2 - 1.0) * h[..., 2] ** 2 + 1.0) ** 2)
    L = lambda w: (np.sqrt(1.0 + a2 * (w[..., 0] ** 2 + w[..., 1] ** 2) / w[..., 2] ** 2) - 1.0) / 2.0
    G2 = 1.0 / (1.0 + L(wo) + L(wi))
    return np.where((wi[..., 2] > 0) & (wo[..., 2] > 0), D_ * G2 / (4.0 * wo[..., 2] * wi[..., 2]), 0.0)


def test_eval_matches_float64_model():
    rng = np.random.default_rng(3)
    n = 20000
    wo = _unit(rng.normal(size=(n, 3)) * [1, 1, 0.5] + [0, 0, 0.6]).astype(np.float32)
    wi = _unit(rng.normal(size=(n, 3)) * [1, 1, 0.5] + [0, 0, 0.6]).astype(np.float32)
    for r in [0.05, 0.3, 0.7, 1.0]:
        alpha = max(np.float64(np.float32(r) * np.float32(r)), 1e-3)
        f = dprt.spec_conductor_eval([1, 1, 1], r, wo, wi)[:, 0].astype(np.float64)
        ref = _f_model(alpha, wo.astype(np.float64), wi.astype(np.float64))
        ok = (wo[:, 2] > 1e-3) & (wi[:, 2] > 1e-3)
        assert np.allclose(f[ok], ref[ok], rtol=2e-5, atol=1e-30), r
        assert not f[(wo[:, 2] <= 0) | (wi[:, 2] <= 0)].any()


def _hemisphere_quadrature(nt=2048, npf=2048):
    th = (np.arange(nt) + 0.5) * (np.pi / 2 / nt)
    ph = (np.arange(npf) + 0.5) * (2 * np.pi / npf)
    T, P = np.meshgrid(th, ph, indexing="ij")
    w = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], -1).reshape(-1, 3)
    dw = (np.sin(T) * (np.pi / 2 / nt) * (2 * np.pi / npf)).ravel()
    return w, dw


HALF_SPACES = [None, (1, 0, 0), (0, 1, 0), (1, 1, -1), (-1, 0.5, 0.2), (0.3, -1, 0.5)]


def _g(wi, k):
    n = HALF_SPACES[k]
    return np.ones(len(wi)) if n is None else (wi @ np.asarray(n, np.float64) > 0).astype(np.float64)


def test_sampling_matches_evaluation():
    """E[weight g(wi)] over the sampler (2^20 uniforms) = integral of f cos g over the hemisphere (float64 model): the next
    path and the light samples describe the same lobe, in total and in shape (g = indicators of half-spaces)."""
    wq, dw = _hemisphere_quadrature()
    rng = np.random.default_rng(11)
    xi = rng.random((1 << 20, 2)).astype(np.float32)
    for wo in [_unit([0, 0, 1]), _unit([0.3, 0.1, 0.9]), _unit([0.8, -0.3, 0.5]), _unit([0.95, 0.2, 0.1])]:
        wo32 = wo.astype(np.float32)
        for r in [0.2236, 0.5, 1.0]:                           # alpha = 0.05, 0.25, 1
            alpha = max(np.float64(np.float32(r) * np.float32(r)), 1e-3)
            wi, wt = dprt.spec_conductor_sample([1, 1, 1], r, np.broadcast_to(wo32, (len(xi), 3)), xi)
            wt = wt[:, 0].astype(np.float64)
            fq = _f_model(alpha, np.broadcast_to(wo, wq.shape), wq) * wq[:, 2] * dw
            for k in range(len(HALF_SPACES)):
                x = wt * _g(wi.astype(np.float64), k)
                mc, err = x.mean(), x.std() / np.sqrt(len(x))
                quad = float((fq * _g(wq, k)).sum())
                assert abs(mc - quad) < 5 * err + 2e-3 * max(quad, 1e-3), (wo, r, k, mc, quad, err)


def test_physical_sanity():
    rng = np.random.default_rng(5)
    n = 200000
    wo = np.concatenate([_wo_grid(), _unit(rng.normal(size=(n, 3)) * [1, 1, 0.3] + [0, 0, 0.3]).astype(np.float32)])
    wo = wo[wo[:, 2] > 0]
    xi = rng.random((len(wo), 2)).astype(np.float32)
    for r in ROUGH[1:] + [0.01, 0.5, 0.8]:
        # F0 = 1: the weight is G2 / G1 exactly, which never exceeds 1, so neither does the directional albedo E[weight]
        wi, wt = dprt.spec_conductor_sample([1, 1, 1], r, wo, xi)
        assert (wt <= 1.0).all() and (wt >= 0.0).all(), r
        assert wt[:, 0].mean() <= 1.0
        # reciprocity of eval: h = normalize(wo + wi) and the Smith term are symmetric; only F(wi.h) vs F(wo.h) rounds, by a
        # few ulps, more where wo and wi are nearly opposite and wo + wi cancels
        wl = _unit(rng.normal(size=(len(wo), 3)) * [1, 1, 0.5] + [0, 0, 0.5]).astype(np.float32)
        f0 = rng.random((len(wo), 3)).astype(np.float32)
        a = dprt.spec_conductor_eval(f0, r, wo, wl)
        b = dprt.spec_conductor_eval(f0, r, wl, wo)
        assert np.allclose(a, b, rtol=5e-5, atol=0), r
    # white furnace by quadrature of the product's eval: the directional albedo with F0 = 1 stays <= 1
    wq, dw = _hemisphere_quadrature(1024, 1024)
    for wo in [_unit([0, 0, 1]), _unit([0.7, 0.1, 0.7]), _unit([0.99, 0, 0.14])]:
        for r in [0.3, 0.6, 1.0]:
            f = dprt.spec_conductor_eval([1, 1, 1], r, np.broadcast_to(wo.astype(np.float32), wq.shape), wq.astype(np.float32))
            assert float((f[:, 0] * wq[:, 2] * dw).sum()) <= 1.0 + 1e-3, (wo, r)


# ---- scene files ----
V2_SHA256 = "d5670775ef30544ef9d3a30ffd5d7dafd22245a2e8eef899de9c5ac7c3cfebe8"     # recorded before DPRTSCN3 existed


def _write(tmp_path, g, name):
    p = tmp_path / name
    dprt.real_scene.save_scene_v2(str(p), g, dprt.scene.default_camera(64, 48), dprt.flatten_instances)
    return p.read_bytes()


def test_scene_file_v2_unchanged_and_v3_layout(tmp_path):
    g = dprt.real_scene.make_garden(2, clusters=6)
    v2 = _write(tmp_path, g, "v2.bin")
    assert v2[:8] == b"DPRTSCN2" and hashlib.sha256(v2).hexdigest() == V2_SHA256
    rough = np.linspace(0.0, 1.0, len(g["materials"]), dtype=np.float32)
    g["material_roughness"] = rough
    v3 = _write(tmp_path, g, "v3.bin")
    assert v3[:8] == b"DPRTSCN3" and v3[8:-4 * rough.size] == v2[8:]
    assert np.array_equal(np.frombuffer(v3[-4 * rough.size:], np.float32), rough)
    g["material_roughness"] = rough[:-1]
    with pytest.raises(ValueError):
        _write(tmp_path, g, "bad.bin")
