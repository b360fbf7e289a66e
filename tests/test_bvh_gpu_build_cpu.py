"""GPU BVH8 builder specification (DESIGN.md 3.10) on the CPU (no GPU), through its host twin dprt_spec_bvh8_build_gpu.

The twin runs the device kernels' functions one element after the other, so what holds here holds for the device blob, which
tests/test_gpu_bvh_build.py compares with the twin bit for bit: the structure the traversal and the refit rely on, conservative
slot boxes, determinism, the node encoding of the refit, and a tree quality close to the host builder's.
"""
import ctypes as C

import numpy as np
import pytest

from refit_cases import assert_blob_equal, dprt, terrain, upload_desc
from test_bvh_refit_cpu import IDENTITY, assert_conservative

DPRT_ERR_INVALID = -1


def _same_centroid():
    """Triangles of every size and orientation whose boxes are all centred on the origin: one Morton code for all of them."""
    rng = np.random.default_rng(11)
    d = (rng.normal(size=(400, 3)) * rng.uniform(0.01, 2.0, (400, 1))).astype(np.float32)
    return np.concatenate([d, -d, np.zeros_like(d)], 1)


def _coincident(kind, count, base=20000):
    """A terrain chunk (base > 0) with `count` coincident triangles: all corners on one point, or one non-degenerate triangle
    repeated. Every pair of them is at the same PLOC distance."""
    if kind == "zero_area":
        t = np.full((1, 9), 0.5, np.float32)
    else:
        t = np.array([[0.3, 0.3, 0.2, 0.35, 0.3, 0.2, 0.3, 0.36, 0.25]], np.float32)
    c = np.repeat(t, count, 0)
    return np.concatenate([terrain(base)[0], c]) if base else c


COINCIDENT = {"terrain_300_zero_area": lambda: _coincident("zero_area", 300), "terrain_300_identical": lambda: _coincident("identical", 300),
              "5000_zero_area": lambda: _coincident("zero_area", 5000, 0), "300_identical": lambda: _coincident("identical", 300, 0)}
CASES = {**IDENTITY, "same_centroid": _same_centroid, **COINCIDENT}


def build(v, m=None):
    return dprt.spec_bvh8_build_gpu(v, m)


def assert_structure(nodes, tris, depth, v, m):
    n = len(tris)
    assert sorted(tris["primID"].tolist()) == list(range(n)), "every primID exactly once"
    g = v[tris["primID"]]
    assert np.array_equal(tris["v0"], g[:, 0:3]) and np.array_equal(tris["v1"], g[:, 3:6]) and np.array_equal(tris["v2"], g[:, 6:9])
    assert np.array_equal(tris["matID"], m[tris["primID"]]) and not tris["pad_"].any()
    assert not (nodes["tmask"] >> 24).any()
    children, leaves = [], []
    for i, nd in enumerate(nodes):
        imask, tmask = int(nd["imask"]), int(nd["tmask"])
        for s in range(8):
            grp = (tmask >> (3 * s)) & 7
            assert grp in (0, 1, 3, 7), (i, s, grp)
            assert not (grp and (imask >> s) & 1), (i, s)
        ni, nt = bin(imask).count("1"), bin(tmask).count("1")
        children += range(int(nd["childBase"]), int(nd["childBase"]) + ni)
        leaves += range(int(nd["triBase"]), int(nd["triBase"]) + nt)
    # BFS: the internal children of the nodes in index order are exactly nodes 1, 2, ..., and so come after their parent
    assert children == list(range(1, len(nodes))), "children in contiguous BFS levels after their parents"
    assert leaves == list(range(n)), "leaf slots cover the triangle records in order"
    levels, first, last = 0, 0, 1
    while first < last:
        levels += 1
        nxt = max([last] + [int(nodes[i]["childBase"]) + bin(int(nodes[i]["imask"])).count("1") for i in range(first, last) if nodes[i]["imask"]])
        first, last = last, nxt
    assert levels == depth <= 36


@pytest.mark.parametrize("case", sorted(CASES))
def test_gpu_build_spec(case):
    v = CASES[case]()
    m = (np.arange(v.shape[0]) % 7).astype(np.int32)
    nodes, tris, depth = build(v, m)
    assert_structure(nodes, tris, depth, v, m)
    assert_conservative(nodes, tris, v)
    again = build(v, m)
    assert_blob_equal(again[:2], (nodes, tris), f"{case}: second build")
    assert again[2] == depth
    # the node encoding is the refit's (and the host builder's): refitting to the same vertices changes nothing
    assert_blob_equal(dprt.spec_bvh8_refit(nodes, tris, v), (nodes, tris), f"{case}: refit(build(V), V)")


@pytest.mark.parametrize("case", sorted(COINCIDENT))
def test_coincident_triangles_build_balanced(case):
    """Runs of equal PLOC distances merge in parallel (DESIGN.md 3.10 step 3): the depth stays that of a balanced tree, as close
    to the host builder's as on ordinary input, instead of growing with the number of coincident triangles."""
    v = COINCIDENT[case]()
    depth, host_depth = build(v)[2], dprt.build_bvh8(v)[2]
    assert depth <= min(36, host_depth + 2), (depth, host_depth)


def test_coincident_run_length_does_not_set_the_depth():
    """Ten times more coincident zero-area triangles add at most the ceil(log2(10)) = 4 levels of a balanced binary subtree
    (every cost there is 0, so the collapse keeps 2-wide nodes), not a level per triangle."""
    d300, d3000 = build(_coincident("zero_area", 300))[2], build(_coincident("zero_area", 3000))[2]
    assert d3000 - d300 <= 4, (d300, d3000)


def _overflowing():
    """Finite coordinates near FLT_MAX / 2: box extents, half areas and SAH costs overflow to +inf (and 0 x inf to NaN)."""
    rng = np.random.default_rng(5)
    c = rng.uniform(-1.6e38, 1.6e38, (600, 1, 3))
    return np.clip(c + rng.normal(0.0, 2e37, (600, 3, 3)), -3.3e38, 3.3e38).astype(np.float32).reshape(-1, 9)


@pytest.mark.parametrize("builder", ["gpu_twin", "host"])
def test_overflowing_costs_still_give_a_valid_tree(builder):
    """With overflowing costs the collapse never makes a leaf slot of more than 3 triangles and the slot assignment still
    places every child (bvh_node.cuh): both builders give a well-formed blob."""
    v = _overflowing()
    assert np.isfinite(v).all()
    m = (np.arange(v.shape[0]) % 7).astype(np.int32)
    nodes, tris, depth = build(v, m) if builder == "gpu_twin" else dprt.build_bvh8(v, m)
    assert_structure(nodes, tris, depth, v, m)


def test_gpu_build_materials_do_not_steer_the_tree():
    v = terrain(2000)[0]
    a, b = build(v), build(v, np.full(len(v), 5, np.int32))
    assert not a[1]["matID"].any() and (b[1]["matID"] == 5).all()
    b[1]["matID"] = 0
    assert_blob_equal(a[:2], b[:2], "with and without materials")


def _cost_per_ray(oracle, blob, v, n, m, w=240, h=135):
    """4 x nodes + triangles per TraRay and shadow ray of the oracle's BVH8 walker over `blob` (profiles/bvh_quality.py)."""
    cfg = dprt.make_config(w, h, spp=1, bounces=4, scene_size=1, proxy_mode=0)
    world = oracle.World(cfg, 1)
    world.add_object(0, upload_desc(v), v, n, m)
    world.set_bvh8(0, blob[0], blob[1])
    world.set_materials(dprt.scene.make_materials(16)); world.set_lights(dprt.scene.make_lights())
    world.set_camera(dprt.scene.default_camera(w, h))
    world.count_bvh8(True); world.reset_frame(); world.render_sample(0)
    tn = tt = tr = 0
    for name in ("traverse", "shadow_trace"):
        a, b, r = world.bvh8_counters(0)[name]
        tn, tt, tr = tn + a, tt + b, tr + r
    return (4 * tn + tt) / tr


# DESIGN.md 3.10: on this chunk and frame the GPU tree costs 1.125 x the host tree per ray (kPlocRadius 4; 1.140 at 8, 1.162 at 16)
QUALITY_BOUND = 1.20


def test_gpu_build_quality_against_host_build(oracle):
    oracle.use_all_host_threads()
    v, n, m = terrain(200000, seed=2)
    host = _cost_per_ray(oracle, dprt.build_bvh8(v, m), v, n, m)
    gpu = _cost_per_ray(oracle, build(v, m), v, n, m)
    print(f"cost per ray: host build {host:.3f}, GPU build {gpu:.3f}, ratio {gpu / host:.4f}")
    assert gpu <= QUALITY_BOUND * host, (gpu, host)


def _raw(v, ntris, out=True, m=None):
    lib = dprt.load_library()
    h = C.c_void_p()
    p = None if v is None else v.ctypes.data_as(C.c_void_p)
    rc = lib.dprt_spec_bvh8_build_gpu(p, None if m is None else m.ctypes.data_as(C.c_void_p), ntris, C.byref(h) if out else None)
    if rc == 0:
        lib.dprt_bvh8_free(h)
    else:
        assert not h.value
    return rc


@pytest.mark.parametrize("what", ["null_vertices", "null_out", "zero", "negative", "nan", "inf", "over_cap"])
def test_gpu_build_spec_rejects(what):
    v = terrain(2000)[0]
    ntris, out = len(v), True
    if what == "null_vertices":
        v = None
    elif what == "null_out":
        out = False
    elif what == "zero":
        ntris = 0
    elif what == "negative":
        ntris = -5
    elif what == "nan":
        v[17, 4] = np.nan
    elif what == "inf":
        v[3, 8] = -np.inf
    elif what == "over_cap":
        ntris = 1 << 27                      # refused before the array is read
    assert _raw(v, ntris, out) == DPRT_ERR_INVALID
    with pytest.raises(dprt.DprtError):
        if what in ("nan", "inf"):
            dprt.spec_bvh8_build_gpu(v)
        else:
            dprt.spec_bvh8_build_gpu(np.zeros((0, 9), np.float32))
