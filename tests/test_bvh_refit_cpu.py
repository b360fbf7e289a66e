"""BVH8 refit specification (DESIGN.md 3.9) on the CPU (no GPU).

dprt_spec_bvh8_refit is the host compile of the refit kernels' source, and the node encoding it runs is the builder's own
(bvh_node.cuh). A refit with the build's vertices must therefore give the build back bit for bit; with moved vertices it must
keep the topology, carry the new corners by primID and leave every slot box conservative by the traversal's margin.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

from refit_cases import D, DEFORMATIONS, assert_blob_equal, deform, dprt, garden_flat, random_tris, terrain

DPRT_ERR_INVALID = -1
TOPOLOGY = ("imask", "childBase", "triBase", "tmask", "reserved_")


def refit(blob, v):
    return dprt.spec_bvh8_refit(blob[0], blob[1], v)


def build(v, m=None):
    nodes, tris, _ = dprt.build_bvh8(v, m)
    return nodes, tris


# ---- identity: refit(build(V), V) == build(V) --------------------------------------------------------------------------------
def _degenerate():
    rng = np.random.default_rng(3)
    p = rng.uniform(0.0, 1.0, (64, 3)).astype(np.float32)
    zero_area = np.repeat(p[:32], 3, 0).reshape(-1, 9)                       # all three corners on one point
    d = rng.normal(size=(32, 3)).astype(np.float32)
    t = np.array([0.0, 0.5, 1.0], np.float32)
    collinear = (p[32:, None, :] + t[None, :, None] * d[:, None, :]).reshape(-1, 9)  # corners on one line
    return np.concatenate([zero_area, collinear, random_tris(16, 4)]).astype(np.float32)


def _flat():
    v = random_tris(500, 5).reshape(-1, 3)
    v[:, 2] = np.float32(0.25)
    return v.reshape(-1, 9)


IDENTITY = {
    "terrain_20k": lambda: terrain(20000)[0],
    "terrain_200k": lambda: terrain(200000, seed=2)[0],
    "garden": lambda: garden_flat()[0],
    **{f"tris_{n}": (lambda n=n: random_tris(n, 10 + n)) for n in (1, 2, 3, 4, 5, 9, 17)},
    "degenerate": _degenerate,
    "flat_z": _flat,
    "near_1e4": lambda: random_tris(3000, 6, centre=1.0e4, scale=3.0),
}


@pytest.mark.parametrize("case", sorted(IDENTITY))
def test_refit_identity(case):
    v = IDENTITY[case]()
    mats = (np.arange(v.shape[0]) % 7).astype(np.int32)
    blob = build(v, mats)
    assert_blob_equal(refit(blob, v), blob, case)


# ---- the builder's output is pinned: sha256 of dprt_bvh8_build recorded before the node rule moved to bvh_node.cuh ---------
def _hash_scenes():
    chunks, _, _ = dprt.scene.make_scene(1, 20000)
    yield "terrain20k", chunks[0].verts, chunks[0].mats
    g = dprt.real_scene.make_garden(1)
    ob = g["objects"][0]
    v, _, _, m = dprt.flatten_instances(ob.meshes, ob.instances)
    yield "garden", v, m
    rng = np.random.default_rng(7)
    c = rng.uniform(-3.0, 5.0, (1000, 1, 3))
    v = (c + rng.normal(0.0, 0.2, (1000, 3, 3))).astype(np.float32).reshape(-1, 9)
    yield "random1000", v, rng.integers(0, 16, 1000).astype(np.int32)


BUILD_SHA256 = {
    "terrain20k": "14d4fb50c2dc801e2baf3069ec5324216330a9b2d1d95280eb619148ef8468f5",
    "garden": "998a2095c61ae925e86d8653a3a554193bfe2eec68bafe244860a99d08a9030a",
    "random1000": "60c44a7ca4c02b6642a63a0f85b467d0988af83066db3a1656044fd3e25f2360",
}


def test_builder_output_unchanged():
    for name, v, m in _hash_scenes():
        nodes, tris, depth = dprt.build_bvh8(v, m)
        h = hashlib.sha256(nodes.tobytes() + tris.tobytes() + np.int32(depth).tobytes()).hexdigest()
        assert h == BUILD_SHA256[name], name


# ---- deformed vertices ---------------------------------------------------------------------------------------------------------
def exact_boxes(nodes, tris):
    """float64 exact AABB of every node's subtree and of every used slot: {(node, slot): (lo, hi)}."""
    corners = np.stack([tris["v0"], tris["v1"], tris["v2"]], 1).astype(np.float64)     # [ntris, 3, 3]
    tlo, thi = corners.min(1), corners.max(1)
    node_box = [None] * len(nodes)
    slots = {}
    for i in range(len(nodes) - 1, -1, -1):
        n = nodes[i]
        imask, tmask = int(n["imask"]), int(n["tmask"])
        irank = 0
        for s in range(8):
            if (imask >> s) & 1:
                slots[(i, s)] = node_box[int(n["childBase"]) + irank]
                irank += 1
                continue
            k = bin((tmask >> (3 * s)) & 7).count("1")
            if k:
                t0 = int(n["triBase"]) + bin(tmask & ((1 << (3 * s)) - 1)).count("1")
                slots[(i, s)] = (tlo[t0:t0 + k].min(0), thi[t0:t0 + k].max(0))
        used = [slots[(i, s)] for s in range(8) if (i, s) in slots]
        node_box[i] = (np.min([u[0] for u in used], 0), np.max([u[1] for u in used], 0))
    return slots


def assert_conservative(nodes, tris, v):
    """Every used slot's dequantised box (float64) holds the exact AABB of the triangles below it widened by pad + 2^-7 of the
    node's quantisation step; unused slots hold the empty box."""
    pad = np.float64(np.ldexp(np.float32(max(float(np.abs(v).max()), 1.0)), -16).astype(np.float32))
    for (i, s), (lo, hi) in exact_boxes(nodes, tris).items():
        n = nodes[i]
        for a, (ql, qh) in enumerate((("qlox", "qhix"), ("qloy", "qhiy"), ("qloz", "qhiz"))):
            sc = np.ldexp(1.0, int(n["e"][a]) - 127)
            cpad = pad + sc * (1.0 / 128.0)
            p0 = np.float64(n["p"][a])
            assert p0 + int(n[ql][s]) * sc <= lo[a] - cpad, (i, s, a)
            assert p0 + int(n[qh][s]) * sc >= hi[a] + cpad, (i, s, a)
    for i, n in enumerate(nodes):
        for s in range(8):
            if not ((int(n["imask"]) >> s) & 1) and not ((int(n["tmask"]) >> (3 * s)) & 7):
                assert n["qlox"][s] == 255 and n["qhix"][s] == 0, (i, s)


@pytest.mark.parametrize("kind", DEFORMATIONS)
@pytest.mark.parametrize("case", ["terrain", "garden"])
def test_refit_deformed(case, kind):
    v = terrain(20000)[0] if case == "terrain" else garden_flat()[0]
    blob = build(v)
    v2 = deform(v, kind)
    nodes, tris = refit(blob, v2)
    for f in TOPOLOGY:
        assert np.array_equal(nodes[f], blob[0][f]), f
    for f in ("primID", "matID", "pad_"):
        assert np.array_equal(tris[f], blob[1][f]), f
    g = v2[tris["primID"]]
    assert np.array_equal(tris["v0"], g[:, 0:3]) and np.array_equal(tris["v1"], g[:, 3:6]) and np.array_equal(tris["v2"], g[:, 6:9])
    assert_conservative(nodes, tris, v2)
    assert_blob_equal(refit((nodes, tris), v), blob, f"{case} {kind} round trip")


def test_refit_garden_moved_instances_conservative():
    v, _, _, _, _, _ = garden_flat()
    vm = garden_flat(moved=True)[0]
    nodes, tris = refit(build(v), vm)
    assert_conservative(nodes, tris, vm)


# ---- rejections leave the arrays unchanged --------------------------------------------------------------------------------------
def _spec_raw(nodes, tris, v, nnodes=None, ntris=None):
    lib = dprt.load_library()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    return lib.dprt_spec_bvh8_refit(p(nodes), len(nodes) if nnodes is None else nnodes, p(tris), len(tris) if ntris is None else ntris, p(v))


def _malformed():
    def child_out(n, t):
        i = int(np.nonzero(n["imask"])[0][-1]); n["childBase"][i] = len(n)
    def child_before(n, t):
        i = int(np.nonzero(n["imask"])[0][-1]); n["childBase"][i] = i
    def tri_out(n, t):
        i = int(np.nonzero(n["tmask"])[0][-1]); n["triBase"][i] = len(t) - 1
    def prim_out(n, t):
        t["primID"][5] = len(t)
    def prim_negative(n, t):
        t["primID"][0] = -1
    def tmask_high(n, t):
        n["tmask"][0] |= np.uint32(1 << 24)
    def tmask_gap(n, t):
        i = int(np.nonzero(n["tmask"])[0][0]); n["tmask"][i] = (int(n["tmask"][i]) & ~7) | 5
    def slot_both(n, t):
        i = int(np.nonzero(n["imask"])[0][0]); s = int(np.log2(int(n["imask"][i]) & -int(n["imask"][i]))); n["tmask"][i] |= np.uint32(1 << (3 * s))
    return {f.__name__: f for f in (child_out, child_before, tri_out, prim_out, prim_negative, tmask_high, tmask_gap, slot_both)}


MALFORMED = _malformed()


@pytest.mark.parametrize("what", sorted(MALFORMED) + ["nan_vertex", "inf_vertex", "fewer_tris", "zero_nodes"])
def test_refit_rejects(what):
    v = terrain(2000)[0]
    nodes, tris = build(v)
    v2 = deform(v, "zscale")
    kw = {}
    if what in MALFORMED:
        MALFORMED[what](nodes, tris)
    elif what == "nan_vertex":
        v2[17, 4] = np.nan
    elif what == "inf_vertex":
        v2[3, 8] = np.inf
    elif what == "fewer_tris":
        kw["ntris"] = len(tris) - 1
    elif what == "zero_nodes":
        kw["nnodes"] = 0
    n0, t0 = nodes.copy(), tris.copy()
    assert _spec_raw(nodes, tris, v2, **kw) == DPRT_ERR_INVALID
    assert_blob_equal((nodes, tris), (n0, t0), what)


def test_refit_python_size_mismatch():
    v = terrain(2000)[0]
    blob = build(v)
    with pytest.raises(dprt.DprtError):
        dprt.spec_bvh8_refit(blob[0], blob[1], v[:-1])
