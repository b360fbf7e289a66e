"""CPU tests of the glossy plastic (bsdfType 3, DESIGN.md 3.13): the product's host compile of plastic.cuh
(dprt_spec_plastic_sample / _eval) against the restatement of tests/plastic_reference.cpp bit for bit, sampling against
evaluation through a float64 model, physical sanity, and obj2scene.py's --glossy MTL mapping. No GPU needed;
tests/test_gpu_plastic.py renders it."""
import ctypes as C
import hashlib
import importlib.util
import os

import numpy as np
import pytest

import plastic_reference as ref
from helpers import D, dprt
from test_conductor_cpu import HALF_SPACES, ROUGH, XI_MAX, _bits, _g, _hemisphere_quadrature, _unit, _wo_grid

ALBEDOS = np.array([[0, 0, 0], [1, 1, 1], [0.8, 0.3, 0.1], [1.5, 0.2, 0.4]], np.float32)
XI12 = np.array([[0, 0], [0, XI_MAX], [XI_MAX, 0], [XI_MAX, XI_MAX], [0.5, 0.5], [0.25, 0.9], [0.999, 0.001]], np.float32)
F32 = np.float32


def _fresnel32(c):
    """The coat's Schlick Fresnel at F0 = 0.04 in binary32, in the specification's order (numpy does not contract)."""
    m = F32(1) - np.clip(np.asarray(c, F32), F32(0), F32(1))
    m2 = m * m
    return F32(0.04) + (F32(1) - F32(0.04)) * ((m2 * m2) * m)


def _ps32(albedo, woz):
    """ps = Fs / (Fs + (1 - Fs) max(0, Y)) in binary32: where xi3 switches from the specular to the diffuse lobe."""
    a = np.asarray(albedo, F32)
    y = np.maximum(F32(0), (F32(0.2126) * a[..., 0] + F32(0.7152) * a[..., 1]) + F32(0.0722) * a[..., 2])
    fs = _fresnel32(woz)
    return fs / (fs + (F32(1) - fs) * y)


def _grid():
    """(albedo, roughness, wo, xi [n, 3]): every albedo, roughness, wo and (xi1, xi2) corner, with xi3 at 0, just below ps,
    at ps (where ps < 1; a uniform never reaches 1) and at XI_MAX."""
    wo = _wo_grid()
    W, A, R, X = np.meshgrid(np.arange(len(wo)), np.arange(len(ALBEDOS)), np.arange(len(ROUGH)), np.arange(len(XI12)), indexing="ij")
    a, r, w, x = ALBEDOS[A.ravel()], np.array(ROUGH, F32)[R.ravel()], wo[W.ravel()], XI12[X.ravel()]
    ps = _ps32(a, w[:, 2])
    below = np.nextafter(ps, F32(0))
    at = np.where(ps <= XI_MAX, ps, XI_MAX)
    xi3 = np.concatenate([np.zeros_like(ps), below, at, np.full_like(ps, XI_MAX)])
    k = 4
    return np.tile(a, (k, 1)), np.tile(r, k), np.tile(w, (k, 1)), np.column_stack([np.tile(x, (k, 1)), xi3]).astype(F32)


def test_host_compile_equals_reference():
    a, r, wo, xi = _grid()
    wi, wt = dprt.spec_plastic_sample(a, r, wo, xi)
    wio, wto = ref.sample(a, r, wo, xi)
    assert np.array_equal(_bits(wi), _bits(wio)) and np.array_equal(_bits(wt), _bits(wto))
    assert np.isfinite(wi).all() and np.isfinite(wt).all() and (wt >= 0).all()
    dead = wo[:, 2] <= 0
    assert not wi[dead].any() and not wt[dead].any()
    # the third uniform chooses the lobe: below ps the conductor's sample at F0 = 0.04, from ps on Lambert's hemisphere sample
    ps = _ps32(a, wo[:, 2])
    spec = ~dead & (xi[:, 2] < ps)
    cwi, cwt = dprt.spec_conductor_sample([0.04, 0.04, 0.04], r[spec], wo[spec], xi[spec, :2])
    assert np.array_equal(wi[spec], cwi)
    assert np.array_equal(wt[spec], (cwt / ps[spec, None]).astype(F32))
    diff = ~dead & ~spec
    assert diff.sum() > 0.2 * diff.size and np.array_equal(wi[diff, 2], xi[diff, 0])
    # light directions: the sampled ones, every grid direction, and random ones of both hemispheres
    rng = np.random.default_rng(7)
    wl = np.concatenate([wi, _wo_grid()[rng.integers(0, len(_wo_grid()), len(wi))], _unit(rng.normal(size=(len(wi), 3)))]).astype(F32)
    ae, re, woe = np.tile(a, (3, 1)), np.tile(r, 3), np.tile(wo, (3, 1))
    f = dprt.spec_plastic_eval(ae, re, woe, wl)
    assert np.array_equal(_bits(f), _bits(ref.evaluate(ae, re, woe, wl)))
    assert np.isfinite(f).all() and (f >= 0).all()
    assert not f[(woe[:, 2] <= 0) | (wl[:, 2] <= 0)].any()
    # never a delta: at r == 0 the diffuse base still takes light
    assert f[(re == 0) & (ae[:, 0] > 0) & (woe[:, 2] > 1e-3) & (wl[:, 2] > 1e-3)].all()


def test_eval_without_albedo_is_the_conductor_lobe():
    a, r, wo, _ = _grid()
    rng = np.random.default_rng(9)
    wl = np.concatenate([_wo_grid()[rng.integers(0, len(_wo_grid()), len(wo))], _unit(rng.normal(size=(len(wo), 3)))]).astype(F32)
    r2, wo2 = np.tile(r, 2), np.tile(wo, (2, 1))
    f = dprt.spec_plastic_eval([0, 0, 0], r2, wo2, wl)
    assert np.array_equal(_bits(f), _bits(dprt.spec_conductor_eval([0.04, 0.04, 0.04], r2, wo2, wl)))


# ---- float64 model of the BSDF ----
def _fresnel64(c):
    m = 1.0 - np.clip(c, 0.0, 1.0)
    return 0.04 + 0.96 * m ** 5


def _spec_model(alpha, wo, wi):
    """The coat's GGX lobe at F0 = 0.04, from the textbook formulas: F(wi.h) D G2 / (4 wo.z wi.z)."""
    h = _unit(wo + wi)
    a2 = alpha * alpha
    D_ = a2 / (np.pi * ((a2 - 1.0) * h[..., 2] ** 2 + 1.0) ** 2)
    L = lambda w: (np.sqrt(1.0 + a2 * (w[..., 0] ** 2 + w[..., 1] ** 2) / w[..., 2] ** 2) - 1.0) / 2.0
    G2 = 1.0 / (1.0 + L(wo) + L(wi))
    F = _fresnel64(np.sum(wi * h, -1))
    return np.where((wi[..., 2] > 0) & (wo[..., 2] > 0), F * D_ * G2 / (4.0 * wo[..., 2] * wi[..., 2]), 0.0)


def _diffuse_model(albedo, wo, wi):
    k = (1.0 - _fresnel64(wo[..., 2])) * (1.0 - _fresnel64(wi[..., 2])) / np.pi
    return np.where((wi[..., 2] > 0) & (wo[..., 2] > 0), k, 0.0)[..., None] * np.asarray(albedo, np.float64)


def test_eval_matches_float64_model():
    rng = np.random.default_rng(3)
    n = 20000
    wo = _unit(rng.normal(size=(n, 3)) * [1, 1, 0.5] + [0, 0, 0.6]).astype(F32)
    wi = _unit(rng.normal(size=(n, 3)) * [1, 1, 0.5] + [0, 0, 0.6]).astype(F32)
    albedo = np.array([0.8, 0.3, 0.1])
    # below cosines of 1e-2, 1 - F(c) = 0.96 (1 - m^5) loses bits to cancellation in binary32 (4e-5 relative at c = 1e-3)
    ok = (wo[:, 2] > 1e-2) & (wi[:, 2] > 1e-2)
    for r in [0.0, 0.05, 0.3, 1.0]:
        alpha = max(np.float64(F32(r) * F32(r)), 1e-3)
        f = dprt.spec_plastic_eval(albedo, r, wo, wi).astype(np.float64)
        m = _diffuse_model(albedo, wo.astype(np.float64), wi.astype(np.float64))
        if r > 0:
            m = m + _spec_model(alpha, wo.astype(np.float64), wi.astype(np.float64))[:, None]
        assert np.allclose(f[ok], m[ok], rtol=2e-5, atol=1e-30), r


WOS = [_unit([0, 0, 1]), _unit([0.3, 0.1, 0.9]), _unit([0.8, -0.3, 0.5]), _unit([0.95, 0.2, 0.1])]


def test_sampling_matches_evaluation():
    """E[weight g(wi)] over the sampler (2^20 uniforms) = integral of f cos g over the hemisphere (float64 model), per channel:
    the next path and the light samples describe the same BSDF, in total and in shape (g = indicators of half-spaces)."""
    wq, dw = _hemisphere_quadrature()
    rng = np.random.default_rng(11)
    xi = rng.random((1 << 20, 3)).astype(F32)
    albedo = np.array([0.8, 0.3, 0.1], F32)
    for wo in WOS:
        wo32 = wo.astype(F32)
        wob = np.broadcast_to(wo, wq.shape)
        fd = _diffuse_model(albedo, wob, wq) * (wq[:, 2] * dw)[:, None]
        for r in [0.2236, 0.5, 1.0]:                           # alpha = 0.05, 0.25, 1
            alpha = max(np.float64(F32(r) * F32(r)), 1e-3)
            wi, wt = dprt.spec_plastic_sample(albedo, r, np.broadcast_to(wo32, (len(xi), 3)), xi)
            fq = fd + (_spec_model(alpha, wob, wq) * wq[:, 2] * dw)[:, None]
            for k in range(len(HALF_SPACES)):
                gm, gq = _g(wi.astype(np.float64), k), _g(wq, k)
                for c in range(3):
                    x = wt[:, c].astype(np.float64) * gm
                    mc, err = x.mean(), x.std() / np.sqrt(len(x))
                    quad = float((fq[:, c] * gq).sum())
                    assert abs(mc - quad) < 5 * err + 2e-3 * max(quad, 1e-3), (wo, r, k, c, mc, quad, err)


def test_smooth_coat_delta_and_diffuse_parts():
    """r == 0: the specular branch is the delta mirror, whose expected weight is F(wo.z); the diffuse branch matches the
    diffuse term's integral, in total and over half-spaces."""
    wq, dw = _hemisphere_quadrature()
    rng = np.random.default_rng(13)
    xi = rng.random((1 << 20, 3)).astype(F32)
    albedo = np.array([0.8, 0.3, 0.1], F32)
    for wo in WOS:
        wo32 = wo.astype(F32)
        wi, wt = dprt.spec_plastic_sample(albedo, 0.0, np.broadcast_to(wo32, (len(xi), 3)), xi)
        spec = xi[:, 2] < _ps32(albedo, wo32[2])
        assert np.array_equal(wi[spec], np.broadcast_to(wo32 * np.array([-1, -1, 1], F32), (int(spec.sum()), 3)))
        x = np.where(spec, wt[:, 0].astype(np.float64), 0.0)
        mc, err = x.mean(), x.std() / np.sqrt(len(x))
        assert abs(mc - _fresnel64(float(wo32[2]))) < 5 * err + 1e-6, (wo, mc, err)
        fd = _diffuse_model(albedo, np.broadcast_to(wo, wq.shape), wq) * (wq[:, 2] * dw)[:, None]
        for k in range(len(HALF_SPACES)):
            gm, gq = _g(wi.astype(np.float64), k), _g(wq, k)
            for c in range(3):
                x = np.where(spec, 0.0, wt[:, c].astype(np.float64)) * gm
                mc, err = x.mean(), x.std() / np.sqrt(len(x))
                quad = float((fd[:, c] * gq).sum())
                assert abs(mc - quad) < 5 * err + 2e-3 * max(quad, 1e-3), (wo, k, c, mc, quad, err)


def test_reciprocity_and_positivity():
    rng = np.random.default_rng(5)
    n = 200000
    wo = np.concatenate([_wo_grid(), _unit(rng.normal(size=(n, 3)) * [1, 1, 0.3] + [0, 0, 0.3]).astype(F32)])
    wl = _unit(rng.normal(size=(len(wo), 3)) * [1, 1, 0.5] + [0, 0, 0.5]).astype(F32)
    albedo = rng.random((len(wo), 3)).astype(F32) * F32(1.2)
    for r in ROUGH + [0.01, 0.5, 0.8]:
        a = dprt.spec_plastic_eval(albedo, r, wo, wl)
        b = dprt.spec_plastic_eval(albedo, r, wl, wo)
        assert np.isfinite(a).all() and (a >= 0).all(), r
        # the diffuse term is symmetric to the bit; the specular one rounds F(wi.h) vs F(wo.h) by a few ulps
        assert np.allclose(a, b, rtol=5e-5, atol=0), r


@pytest.mark.parametrize("r", ROUGH)
def test_directional_albedo_at_most_one(r):
    """White diffuse colour: E[weight] over 2^20 samples is the directional albedo, at most 1 up to the Monte Carlo error."""
    rng = np.random.default_rng(17)
    xi = rng.random((1 << 20, 3)).astype(F32)
    for z in [1.0, 0.7, 0.3, 0.1, 0.02]:
        wo = np.array([np.sqrt(1 - z * z), 0.0, z], F32)
        _, wt = dprt.spec_plastic_sample([1, 1, 1], r, np.broadcast_to(wo, (len(xi), 3)), xi)
        x = wt[:, 0].astype(np.float64)
        assert x.mean() <= 1.0 + 5 * x.std() / np.sqrt(len(x)), (r, z, x.mean())


# ---- obj2scene.py --glossy ----
GLOSSY_MTL = ("newmtl ground\nKd 0.5 0.5 0.5\nKs 0.5 0.5 0.5\nNs 100\nillum 2\nmap_Kd checker.pfm\n"
              "newmtl leaf\nKd 0.1 0.6 0.1\nKs 0.04 0.04 0.04\nPr 0.3\nillum 2\n"
              "newmtl rock\nKd 0.9 0.6 0.5\nKs 1 1 1\nPm 1\nPr 0.2\nillum 3\n"
              "newmtl water\nNi 1.33\nKs 1 1 1\nNs 900\nillum 7\n"
              "newmtl leaf2\nKd 0.2 0.7 0.2\nKs 0 0 0\nNs 50\nillum 2\n")
# material order of the file (first use in the OBJ), and what --glossy makes of each: (bsdfType, baseColor, roughness)
GLOSSY_EXPECT = {"ground": (3, (0.5, 0.5, 0.5), (2.0 / 102.0) ** 0.25), "leaf": (3, (0.1, 0.6, 0.1), 0.3),
                 "leaf2": (0, (0.2, 0.7, 0.2), 0.0), "rock": (2, (0.9, 0.6, 0.5), 0.2), "water": (1, (1.0, 1.0, 1.0), 0.0)}
# a conversion of that OBJ / MTL without --glossy, recorded before the flag existed: Ks / Ns / Pr / Pm change nothing
FLAGLESS_SHA256 = "dcaa0fb2060e9a07dc87629edc83b2d89246d8ab9aec76c7e19b2bf1ff4f20f4"


def obj2scene():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("obj2scene", os.path.join(root, "pg2024-data-parallel-ray-tracing_b200", "obj2scene.py"))
    o2s = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(o2s)
    return o2s


def write_glossy_obj(tmp_path, mtl=GLOSSY_MTL):
    """The small procedural garden as OBJ + MTL (+ a checker texture) under tmp_path; returns the OBJ's path."""
    g = dprt.real_scene.make_garden(W=1, clusters=3, ground=(12, 12))
    obj = tmp_path / "glossy.obj"
    dprt.real_scene.save_obj(str(obj), g["objects"][0].meshes, ["ground", "leaf", "rock", "water", "leaf2"])
    obj.write_text("mtllib glossy.mtl\n" + obj.read_text())
    (tmp_path / "glossy.mtl").write_text(mtl)
    dprt.scene.save_pfm(str(tmp_path / "checker.pfm"), dprt.real_scene.checker_texture(8)[..., :3])
    return str(obj)


def _materials_of(b):
    """(materials, texture slot per material) of a DPRTSCN2 / DPRTSCN3 file (layout: csrc/dprt_render.cpp)."""
    nmat = int(np.frombuffer(b, "<i4", 1, 12)[0])
    o = 24 + C.sizeof(D.Camera)
    return np.frombuffer(b, D.MATERIAL_DTYPE, nmat, o), np.frombuffer(b, "<i4", nmat, o + nmat * D.MATERIAL_DTYPE.itemsize)


def test_obj2scene_glossy_mapping(tmp_path):
    o2s = obj2scene()
    obj = write_glossy_obj(tmp_path)
    plain, glossy = str(tmp_path / "plain.dprt"), str(tmp_path / "glossy.dprt")
    info = o2s.convert(obj, plain, world=2, width=64, height=36)
    b0 = open(plain, "rb").read()
    assert b0[:8] == b"DPRTSCN2" and hashlib.sha256(b0).hexdigest() == FLAGLESS_SHA256
    assert o2s.convert(obj, glossy, world=2, width=64, height=36, glossy=True) == info
    b1 = open(glossy, "rb").read()
    names = info["materials"]
    assert b1[:8] == b"DPRTSCN3" and len(b1) == len(b0) + 4 * len(names)
    mats, mat_tex = _materials_of(b1)
    rough = np.frombuffer(b1[-4 * len(names):], np.float32)
    for i, nm in enumerate(names):
        kind, color, r = GLOSSY_EXPECT[nm]
        assert mats["bsdfType"][i] == kind and np.allclose(mats["baseColor"][i], color) and rough[i] == F32(r), nm
    assert mat_tex.tolist() == _materials_of(b0)[1].tolist() == [0, -1, -1, -1, -1]    # the plastic ground keeps its texture
    # only the material table and the roughness table differ from the flag-less file
    start = 24 + C.sizeof(D.Camera)
    end = start + mats.nbytes
    assert b1[8:start] == b0[8:start] and b1[end:-4 * len(names)] == b0[end:]
    # --glossy on an MTL without metallic or specular materials: byte-identical to the flag-less DPRTSCN2 file
    write_glossy_obj(tmp_path, "newmtl ground\nKd 0.5 0.5 0.5\nmap_Kd checker.pfm\nnewmtl rock\nKs 0.5 0.5 0.5\nillum 1\n")
    o2s.convert(obj, plain, world=1, width=32, height=18)
    o2s.convert(obj, glossy, world=1, width=32, height=18, glossy=True)
    assert open(glossy, "rb").read() == open(plain, "rb").read()


def test_glossy_material_rules():
    o2s = obj2scene()
    m = lambda **kw: dict(o2s._mtl_default(), **kw)
    g = o2s.glossy_material
    assert g(m()) is None                                                      # plain Lambertian
    assert g(m(Ks=(0.5, 0.5, 0.5))) is None                                    # no illum: no specular highlight asked for
    assert g(m(Ks=(0.5, 0.5, 0.5), illum=1)) is None
    assert g(m(Ks=(0.5, 0.5, 0.5), illum=4, water=True)) is None               # water stays water
    assert g(m(Ks=(0.0, 0.0, 0.1), illum=2, Ns=0.0)) == (3, 1.0)
    assert g(m(Ks=(1, 1, 1), illum=2)) == (3, 1.0)                             # a missing Ns counts as 0
    assert g(m(Ks=(1, 1, 1), illum=2, Ns=1e9))[1] < 0.01
    assert g(m(Ks=(1, 1, 1), illum=2, Ns=-5.0)) == (3, 1.0)                    # clipped to [0, 1]
    assert g(m(Ks=(1, 1, 1), illum=2, Pr=1.7)) == (3, 1.0)
    assert g(m(Ks=(1, 1, 1), illum=2, Pr=-0.2)) == (3, 0.0)
    assert g(m(Pm=0.3, Ks=(1, 1, 1), illum=2, Pr=0.4)) == (3, 0.4)             # below the metallic threshold: plastic
    kind, r = g(m(Pm=0.5, Ns=30.0))                                            # metallic: the conductor, (2 / 32)^(1/4)
    assert kind == 2 and abs(r - 0.5) < 1e-12
