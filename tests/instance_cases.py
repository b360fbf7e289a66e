"""Instanced scene objects shared by the flatten tests (test_instance_flatten_cpu.py) and the GPU instanced-build tests
(test_gpu_instanced_build.py): indexed meshes plus (mesh, 3x4 matrix) instances, as ctypes_defs.pack_meshes takes them."""
import hashlib

import numpy as np

from helpers import dprt


def random_mesh(ntris, seed, textured=True, material=0):
    """Indices drawn at random over small attribute arrays: every corner gathers through its own three index streams."""
    rng = np.random.default_rng(seed)
    npos, nnrm, ntc = max(1, ntris // 2 + 3), max(1, ntris // 3 + 2), max(1, ntris // 4 + 2)
    nrm = rng.normal(size=(nnrm, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    m = {"positions": rng.uniform(-1.0, 1.0, (npos, 3)).astype(np.float32), "indices": rng.integers(0, npos, (ntris, 3), dtype=np.int32),
         "normals": nrm.astype(np.float32), "normal_indices": rng.integers(0, nnrm, (ntris, 3), dtype=np.int32),
         "texcoords": None, "texcoord_indices": None, "material": material}
    if textured:
        m["texcoords"] = rng.uniform(-2.0, 3.0, (ntc, 2)).astype(np.float32)
        m["texcoord_indices"] = rng.integers(0, ntc, (ntris, 3), dtype=np.int32)
    return m


def grid_mesh(nx, ny, seed, textured=True, material=0):
    """A bumpy sheet of 2 nx ny triangles over [-1, 1]^2: neighbouring triangles are neighbours in space."""
    rng = np.random.default_rng(seed)
    x, y = np.meshgrid(np.linspace(-1.0, 1.0, nx + 1), np.linspace(-1.0, 1.0, ny + 1), indexing="ij")
    z = 0.1 * np.sin(3.0 * x + rng.uniform(0, 6)) * np.cos(2.0 * y)
    P = np.stack([x, y, z], -1).reshape(-1, 3)
    k = np.arange((nx + 1) * (ny + 1)).reshape(nx + 1, ny + 1)
    a, b, c, d = k[:-1, :-1].ravel(), k[1:, :-1].ravel(), k[1:, 1:].ravel(), k[:-1, 1:].ravel()
    idx = np.concatenate([np.stack([a, b, c], 1), np.stack([a, c, d], 1)]).astype(np.int32)
    nrm = np.stack([-0.3 * np.cos(3.0 * x), 0.2 * np.sin(2.0 * y), np.ones_like(x)], -1).reshape(-1, 3)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    m = {"positions": P.astype(np.float32), "indices": idx, "normals": nrm.astype(np.float32), "normal_indices": idx.copy(),
         "texcoords": None, "texcoord_indices": None, "material": material}
    if textured:
        m["texcoords"] = (0.5 * (P[:, :2] + 1.0)).astype(np.float32)
        m["texcoord_indices"] = idx.copy()
    return m


def one_triangle(seed, textured, material=0):
    rng = np.random.default_rng(seed)
    n = rng.normal(size=(1, 3))
    m = {"positions": rng.uniform(-1, 1, (3, 3)).astype(np.float32), "indices": np.array([[0, 1, 2]], np.int32),
         "normals": (n / np.linalg.norm(n)).astype(np.float32), "normal_indices": np.zeros((1, 3), np.int32),
         "texcoords": None, "texcoord_indices": None, "material": material}
    if textured:
        m["texcoords"] = rng.uniform(0, 1, (3, 2)).astype(np.float32)
        m["texcoord_indices"] = np.array([[2, 0, 1]], np.int32)
    return m


def empty_mesh(textured, material=0):
    m = {"positions": np.zeros((0, 3), np.float32), "indices": np.zeros((0, 3), np.int32), "normals": np.zeros((0, 3), np.float32),
         "normal_indices": np.zeros((0, 3), np.int32), "texcoords": None, "texcoord_indices": None, "material": material}
    if textured:
        m["texcoords"], m["texcoord_indices"] = np.zeros((0, 2), np.float32), np.zeros((0, 3), np.int32)
    return m


def placement(rng, mirror=None, scale=0.08):
    """A 3x4 float32 matrix: turned about z, tilted, scaled, placed in the unit cube; mirror = axis to negate (det < 0)."""
    s = scale * rng.uniform(0.5, 1.5, 3)
    if mirror is not None:
        s[mirror] = -s[mirror]
    t, tilt = rng.uniform(0, 2 * np.pi), rng.uniform(-0.4, 0.4)
    c, sn, ct, st = np.cos(t), np.sin(t), np.cos(tilt), np.sin(tilt)
    A = np.array([[c, -sn, 0], [sn, c, 0], [0, 0, 1.0]]) @ np.array([[1.0, 0, 0], [0, ct, -st], [0, st, ct]]) @ np.diag(s)
    return np.concatenate([A, rng.uniform(0.1, 0.9, (3, 1))], 1).astype(np.float32)


def case_garden():
    ob = dprt.real_scene.make_garden(1)["objects"][0]
    return ob.meshes, ob.instances


def case_mirrored():
    rng = np.random.default_rng(11)
    meshes = [random_mesh(40, 1), grid_mesh(6, 5, 2, textured=False, material=3)]
    return meshes, [(k % 2, placement(rng, mirror=k % 3)) for k in range(9)]


def case_mixed_uv():
    rng = np.random.default_rng(12)
    meshes = [random_mesh(30, 3, textured=True, material=1), random_mesh(25, 4, textured=False, material=2),
              grid_mesh(4, 4, 5, textured=True, material=4), grid_mesh(3, 7, 6, textured=False)]
    return meshes, [(k % 4, placement(rng)) for k in range(14)]


def case_zero_tris():
    rng = np.random.default_rng(13)
    meshes = [empty_mesh(False), random_mesh(20, 7), empty_mesh(True, 5), grid_mesh(3, 3, 8, textured=False), empty_mesh(False)]
    order = [0, 1, 2, 2, 3, 4, 1, 0, 3, 4]                # zero-triangle instances first, last, in runs and between others
    return meshes, [(mi, placement(rng)) for mi in order]


def case_one_tri():
    rng = np.random.default_rng(14)
    meshes = [one_triangle(20 + k, textured=k % 2 == 0, material=k) for k in range(5)]
    return meshes, [(int(rng.integers(0, 5)), placement(rng, mirror=0 if k % 7 == 0 else None)) for k in range(300)]


CASES = {"garden": case_garden, "mirrored": case_mirrored, "mixed_uv": case_mixed_uv, "zero_tris": case_zero_tris, "one_tri": case_one_tri}


def case_10m():
    """About 2 000 instances, 10.9 M flattened triangles: one instance of a 1.5 M-triangle mesh, thousands of smaller ones down to
    single triangles."""
    rng = np.random.default_rng(15)
    meshes = [grid_mesh(750, 1000, 30, material=1), grid_mesh(60, 75, 31, textured=False, material=2), grid_mesh(20, 25, 32, material=3),
              one_triangle(33, True, 4), random_mesh(37, 34, textured=False, material=5)]
    inst = [(0, placement(rng, scale=0.3))]
    inst += [(1, placement(rng, mirror=0 if k % 9 == 4 else None, scale=0.02)) for k in range(950)]
    inst += [(2, placement(rng, scale=0.01)) for _ in range(900)]
    inst += [(3, placement(rng, scale=0.01)) for _ in range(100)]
    inst += [(4, placement(rng, scale=0.01)) for _ in range(50)]
    order = rng.permutation(len(inst))
    return meshes, [inst[k] for k in order]


def moved(instances, every=3, angle=0.3, shrink=0.8):
    """Every `every`-th instance turned by `angle` about its own vertical axis and shrunk around its own origin."""
    c, s = np.cos(angle), np.sin(angle)
    Rz = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]]) * shrink
    return [(mi, np.concatenate([np.asarray(M, np.float64)[:, :3] @ Rz, np.asarray(M, np.float64)[:, 3:]], 1).astype(np.float32))
            if k % every == 0 else (mi, M) for k, (mi, M) in enumerate(instances)]


def object_desc(meshes, *instance_lists):
    """An object description whose AABB holds every listed placement of the instances."""
    inst = [x for lst in instance_lists for x in lst if len(meshes[x[0]]["positions"])]
    return dprt.real_scene.InstancedObject(0, 0, meshes, inst).desc(False)


def flatten_digest(v, n, uv, m):
    h = hashlib.sha256()
    for a in (v, n, uv, m):
        h.update(b"none" if a is None else np.ascontiguousarray(a).tobytes())
    return h.hexdigest()
