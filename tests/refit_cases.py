"""Chunks and vertex deformations shared by the BVH8 refit tests (test_bvh_refit_cpu.py, test_gpu_refit.py).

Every deformation keeps the vertices inside the bounding box of the input, so a chunk uploaded with its own box (scene.Chunk:
the vertex bounds widened by 1e-4) accepts them."""
import numpy as np

from helpers import D, dprt


def terrain(ntris, seed=0):
    """A heightfield chunk of ~ntris triangles over the unit square: (verts9, normals9, mat_ids)."""
    q = max(1, ntris // 2)
    nx = max(2, int(round(np.sqrt(q))))
    ny = max(2, int(round(q / nx)))
    return dprt.scene.make_heightfield_chunk((0.0, 0.0, 0.0), (1.0, 1.0, 0.5), nx, ny, seed)


def garden_flat(moved=False):
    """The garden's single scene object flattened (verts9, normals9, uv6, mat_ids); moved=True: every element instance (all but
    the ground and the pond) shrunk by 0.8 around its own origin and turned by 0.3 rad about its own vertical axis."""
    g = dprt.real_scene.make_garden(1)
    ob = g["objects"][0]
    inst = ob.instances
    if moved:
        c, s = np.cos(0.3), np.sin(0.3)
        R = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]]) * 0.8
        inst = [(mi, M) if k < 2 else (mi, np.concatenate([np.asarray(M, np.float64)[:, :3] @ R, np.asarray(M, np.float64)[:, 3:]], 1)
                                                 .astype(np.float32)) for k, (mi, M) in enumerate(ob.instances)]
    v, n, uv, m = dprt.flatten_instances(ob.meshes, inst)
    return v, n, uv, m, g, inst


def random_tris(n, seed, centre=0.0, scale=1.0):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-1.0, 1.0, (n, 1, 3))
    v = centre + scale * (c + rng.normal(0.0, 0.15, (n, 3, 3)))
    return v.astype(np.float32).reshape(-1, 9)


def deform(v, kind, seed=1):
    """One of DEFORMATIONS applied to verts9 [n, 9] (float32); the result stays inside the input's bounding box."""
    P = v.reshape(-1, 3).astype(np.float64)
    lo, hi = P.min(0), P.max(0)
    rng = np.random.default_rng(seed)
    if kind == "zscale":            # heights scaled towards the middle
        mid = 0.5 * (lo[2] + hi[2])
        P[:, 2] = mid + 0.5 * (P[:, 2] - mid)
    elif kind == "zwave":           # a moderate travelling wave on the heights
        mid = 0.5 * (lo[2] + hi[2])
        P[:, 2] = mid + (P[:, 2] - mid) * (0.75 + 0.25 * np.sin(9.0 * P[:, 0] + 4.0 * P[:, 1]))
    elif kind == "zjitter":         # random z jitter, clipped to the input's z range
        P[:, 2] = np.clip(P[:, 2] + rng.normal(0.0, 0.02 * (hi[2] - lo[2]), P.shape[0]), lo[2], hi[2])
    elif kind == "permute":         # whole triangles trade places: triangle p gets the corners of triangle perm[p]
        return np.ascontiguousarray(v.reshape(-1, 9)[rng.permutation(v.shape[0])])
    elif kind == "collapse":        # every vertex on one point
        P[:] = 0.5 * (lo + hi)
    elif kind == "faces":           # every vertex pushed out to the face of the box it is nearest to (in box-relative units)
        half = np.maximum(0.5 * (hi - lo), 1e-30)
        r = (P - 0.5 * (lo + hi)) / half
        a = np.argmax(np.abs(r), 1)
        idx = np.arange(P.shape[0])
        P[idx, a] = np.where(r[idx, a] >= 0.0, hi[a], lo[a])
    else:
        raise ValueError(kind)
    out = P.astype(np.float32)
    return np.clip(out, lo.astype(np.float32), hi.astype(np.float32)).reshape(v.shape)


DEFORMATIONS = ("zscale", "zjitter", "permute", "collapse", "faces")


def assert_blob_equal(a, b, what):
    na, ta = a
    nb, tb = b
    assert na.shape == nb.shape and ta.shape == tb.shape, f"{what}: sizes {na.shape}/{ta.shape} vs {nb.shape}/{tb.shape}"
    for name, x, y in (("nodes", na, nb), ("tris", ta, tb)):
        xb, yb = x.view(np.uint8).reshape(x.size, -1), y.view(np.uint8).reshape(y.size, -1)
        bad = np.nonzero((xb != yb).any(1))[0]
        assert bad.size == 0, f"{what}: {bad.size}/{x.size} {name} records differ; first at {int(bad[0])}:\n {x[bad[0]]}\n {y[bad[0]]}"


def upload_desc(v, node_id=0):
    """The object description scene.Chunk gives these vertices (their bounds widened by 1e-4)."""
    return dprt.scene.Chunk(0, node_id, v, None, None).desc(False)


__all__ = ["D", "dprt", "terrain", "garden_flat", "random_tris", "deform", "DEFORMATIONS", "assert_blob_equal", "upload_desc"]
