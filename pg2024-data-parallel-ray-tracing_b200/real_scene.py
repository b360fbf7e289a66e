"""A small "real-scene" generator for the front end of SURVEY.md 8f row 3: indexed meshes, three levels of instancing,
albedo + opacity textures with alpha cut-outs, an environment map, a water surface.

The reference's scene loaders (Moana island, Bistro, San Miguel: OBJ / ptex / EXR readers) are not in its tree and the
scenes themselves are not redistributable, so the parity cases use this procedural garden, which exercises the same data
paths: a ground mesh with shared vertices / normals / tiled texture coordinates (HitGroupData in indexed form,
pipeline_helper.cpp:182-193), "bush" details made of leaf cards whose texture has transparent texels (the __anyhit__ah
cut-out of kernel.cu:311-359), untextured rocks, a water quad (bsdfs/water.hpp) -- details instanced into elements,
elements instanced into the scene object (pipeline_helper.cpp:268-272), one instance mirrored so that the normal transform's
determinant sign matters -- and a lat-long HDR sky (kernel.cu:28-48). Everything here is plain input data for both libdprt
and the oracle; nothing is computed on behalf of either.
"""
import numpy as np

from . import ctypes_defs as D
from .scene import make_lights, rnd_np, tea4_np

MAT_GROUND, MAT_LEAF, MAT_ROCK, MAT_WATER, MAT_LEAF2 = 0, 1, 2, 3, 4
TEX_CHECKER, TEX_LEAF = 0, 5          # a gap in the slot table on purpose


def _rand(n, key):
    """n reference-RNG floats in [0, 1) (tea<4> + one LCG step), reproducible everywhere."""
    v, _ = rnd_np(tea4_np(np.arange(n, dtype=np.uint32), np.uint32(key)))
    return v.astype(np.float64)


def checker_texture(n=32):
    y, x = np.mgrid[0:n, 0:n]
    c = ((x // 4 + y // 4) & 1).astype(np.float32)
    t = np.zeros((n, n, 4), np.float32)
    t[..., 0] = 0.25 + 0.55 * c
    t[..., 1] = 0.45 + 0.25 * (1.0 - c)
    t[..., 2] = 0.20 + 0.15 * c + 0.2 * (x / n)
    t[..., 3] = 1.0
    return t


def leaf_texture(n=32):
    """Opaque green ellipse on a fully transparent background, one texel of soft edge (bilinear alpha crosses 0.05 inside a texel)."""
    y, x = np.mgrid[0:n, 0:n]
    u, v = (x + 0.5) / n - 0.5, (y + 0.5) / n - 0.5
    r = np.sqrt((u / 0.42) ** 2 + (v / 0.30) ** 2)
    t = np.zeros((n, n, 4), np.float32)
    t[..., 0] = 0.10 + 0.25 * (u + 0.5)
    t[..., 1] = 0.45 + 0.40 * (v + 0.5)
    t[..., 2] = 0.08
    t[..., 3] = np.clip((1.0 - r) * 6.0, 0.0, 1.0)
    return t


def sky_env_map(w=64, h=32):
    """Lat-long RGBA radiance: row = theta / pi (0 = +z), column = phi / 2pi; horizon glow + a soft sun."""
    th = (np.arange(h) + 0.5) / h * np.pi
    ph = (np.arange(w) + 0.5) / w * 2.0 * np.pi
    T, P = np.meshgrid(th, ph, indexing="ij")
    up = np.cos(T)
    sun_dir = np.array([np.cos(1.1) * np.sin(0.9), np.sin(1.1) * np.sin(0.9), np.cos(0.9)])
    d = np.stack([np.cos(P) * np.sin(T), np.sin(P) * np.sin(T), np.cos(T)], -1)
    sun = np.exp(-((1.0 - d @ sun_dir) / 0.02))
    e = np.zeros((h, w, 4), np.float32)
    e[..., 0] = 0.35 + 0.25 * (1.0 - np.abs(up)) + 6.0 * sun
    e[..., 1] = 0.45 + 0.30 * np.clip(up, 0, 1) + 5.0 * sun
    e[..., 2] = 0.60 + 0.35 * np.clip(up, 0, 1) + 3.0 * sun
    e[..., :3] *= np.where(up[..., None] < 0, 0.35, 1.0)
    e[..., 3] = 1.0
    return e


def ground_height(x, y):
    return 0.30 + 0.05 * np.sin(5.0 * x + 0.4) * np.cos(4.0 * y - 0.2) + 0.02 * np.sin(17.0 * x * y)


def ground_mesh(x0, x1, nx, ny, uv_tiles=6.0):
    """Indexed grid: shared positions, per-vertex normals (same indices), per-vertex texture coordinates that tile (values > 1)."""
    gx, gy = np.meshgrid(np.linspace(x0, x1, nx + 1), np.linspace(0.0, 1.0, ny + 1), indexing="ij")
    z = ground_height(gx, gy)
    P = np.stack([gx, gy, z], -1)
    nrm = np.cross(np.gradient(P, axis=0), np.gradient(P, axis=1))
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    vid = (np.arange(nx + 1)[:, None] * (ny + 1) + np.arange(ny + 1)[None, :])
    a, b, c, d = vid[:-1, :-1], vid[1:, :-1], vid[1:, 1:], vid[:-1, 1:]
    idx = np.stack([np.stack([a, b, c], -1), np.stack([a, c, d], -1)], 2).reshape(-1, 3)
    uv = np.stack([gx * uv_tiles, gy * uv_tiles - 1.5], -1)      # negative and > 1 coordinates: wrap addressing
    return {"positions": P.reshape(-1, 3), "indices": idx, "normals": nrm.reshape(-1, 3), "normal_indices": idx,
            "texcoords": uv.reshape(-1, 2), "texcoord_indices": idx, "material": MAT_GROUND}


def bush_mesh(cards=14, key=0xB05, material=MAT_LEAF):
    """Leaf cards: 4 positions per card, ONE normal per card, and 4 texture coordinates shared by all cards -- three index
    arrays that really differ (what normalIndices / texCoordsIndices exist for)."""
    r = _rand(cards * 8, key).reshape(cards, 8)
    pos, idx, nrm, nidx, tidx = [], [], [], [], []
    for k in range(cards):
        c = (r[k, 0:3] - 0.5) * np.array([0.8, 0.8, 0.6]) + np.array([0.0, 0.0, 0.45])
        az, el, roll = 2 * np.pi * r[k, 3], (r[k, 4] - 0.5) * 1.6, 2 * np.pi * r[k, 5]
        n = np.array([np.cos(az) * np.cos(el), np.sin(az) * np.cos(el), np.sin(el)])
        t = np.cross(n, [0.0, 0.0, 1.0]); t /= np.linalg.norm(t)
        b = np.cross(n, t)
        t, b = np.cos(roll) * t + np.sin(roll) * b, -np.sin(roll) * t + np.cos(roll) * b
        s = 0.22 + 0.18 * r[k, 6]
        q = [c - s * t - s * b, c + s * t - s * b, c + s * t + s * b, c - s * t + s * b]
        base = 4 * k
        pos += q
        idx += [[base, base + 1, base + 2], [base, base + 2, base + 3]]
        nrm.append(n)
        nidx += [[k, k, k], [k, k, k]]
        tidx += [[0, 1, 2], [0, 2, 3]]
    uv = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], np.float32)
    return {"positions": np.array(pos), "indices": np.array(idx), "normals": np.array(nrm), "normal_indices": np.array(nidx),
            "texcoords": uv, "texcoord_indices": np.array(tidx), "material": material}


def rock_mesh(key=0x70C):
    """Once-subdivided octahedron pushed onto a jittered sphere; smooth normals; no texture coordinates."""
    v = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    f = [(0, 2, 4), (2, 1, 4), (1, 3, 4), (3, 0, 4), (2, 0, 5), (1, 2, 5), (3, 1, 5), (0, 3, 5)]
    verts, cache, faces = [np.array(p, np.float64) for p in v], {}, []

    def mid(a, b):
        k = (min(a, b), max(a, b))
        if k not in cache:
            m = verts[a] + verts[b]
            verts.append(m / np.linalg.norm(m))
            cache[k] = len(verts) - 1
        return cache[k]
    for a, b, c in f:
        ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
        faces += [(a, ab, ca), (ab, b, bc), (ca, bc, c), (ab, bc, ca)]
    V = np.array(verts)
    jit = 0.8 + 0.4 * _rand(len(V), key)
    P = V * jit[:, None] * np.array([0.35, 0.30, 0.22]) + np.array([0.0, 0.0, 0.15])
    N = V / np.array([0.35, 0.30, 0.22])
    N /= np.linalg.norm(N, axis=1, keepdims=True)
    idx = np.array(faces)
    return {"positions": P, "indices": idx, "normals": N, "normal_indices": idx, "texcoords": None, "texcoord_indices": None,
            "material": MAT_ROCK}


def pond_mesh(x0, x1):
    cx = 0.5 * (x0 + x1)
    hw = 0.18 * (x1 - x0)
    P = np.array([[cx - hw, 0.30, 0.335], [cx + hw, 0.30, 0.335], [cx + hw, 0.55, 0.335], [cx - hw, 0.55, 0.335]])
    idx = np.array([[0, 1, 2], [0, 2, 3]])
    return {"positions": P, "indices": idx, "normals": np.array([[0.0, 0.0, 1.0]]), "normal_indices": np.zeros((2, 3), np.int32),
            "texcoords": None, "texcoord_indices": None, "material": MAT_WATER}


def _affine(scale=(1, 1, 1), rot_z=0.0, translate=(0, 0, 0), tilt=0.0):
    c, s = np.cos(rot_z), np.sin(rot_z)
    Rz = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])
    ct, st = np.cos(tilt), np.sin(tilt)
    Rx = np.array([[1.0, 0, 0], [0, ct, -st], [0, st, ct]])
    M = np.eye(4)
    M[:3, :3] = Rz @ Rx @ np.diag(scale)
    M[:3, 3] = translate
    return M


def flatten_hierarchy(scene_instances, elements):
    """Three traversable levels -> the flat (mesh, 3x4 matrix) list the C ABI takes. scene_instances: list of
    ("mesh", mesh_index, M4) | ("element", element_name, M4); elements: {name: [(mesh_index, M4), ...]}. Matrices are composed in
    float64 and rounded once (the reference hands OptiX per-level matrices and lets it compose them per ray)."""
    out = []
    for kind, what, M in scene_instances:
        if kind == "mesh":
            out.append((what, M[:3].astype(np.float32)))
        else:
            for mi, Md in elements[what]:
                out.append((mi, (M @ Md)[:3].astype(np.float32)))
    return out


class InstancedObject:
    """One scene object (chunk) in front-end form: meshes + flat instance list + its object-space AABB."""

    def __init__(self, index, node_id, meshes, instances):
        self.index, self.node_id, self.meshes, self.instances = index, node_id, meshes, instances
        lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
        for mi, M in instances:
            P = np.asarray(meshes[mi]["positions"], np.float64).reshape(-1, 3)
            Q = P @ np.asarray(M, np.float64)[:, :3].T + np.asarray(M, np.float64)[:, 3]
            lo, hi = np.minimum(lo, Q.min(0)), np.maximum(hi, Q.max(0))
        self.aabb_min, self.aabb_max = (lo - 1e-3).astype(np.float32), (hi + 1e-3).astype(np.float32)

    def desc(self, is_proxy):
        return D.make_object_desc(self.node_id, self.aabb_min, self.aabb_max, is_proxy=int(is_proxy))

    @property
    def ntris(self):
        return int(sum(np.asarray(self.meshes[mi]["indices"]).reshape(-1, 3).shape[0] for mi, _ in self.instances))


def make_garden(W=1, clusters=18, ground=(40, 40), seed=0, cluster_scale=0.05):
    """W scene objects (x-slabs of the unit square, one per rank). Returns a dict: objects [InstancedObject], materials,
    material_textures [int32 per material], textures {slot: rgba}, env_map, env_rotation, lights. cluster_scale: size of an
    element instance (between cluster_scale and 2 cluster_scale): shrink it when asking for thousands of clusters."""
    mats = np.zeros(5, D.MATERIAL_DTYPE)
    mats["baseColor"][MAT_GROUND] = (0.9, 0.1, 0.9)     # never seen: the checker map replaces it
    mats["baseColor"][MAT_LEAF] = (0.9, 0.1, 0.9)
    mats["baseColor"][MAT_LEAF2] = (0.9, 0.1, 0.9)
    mats["baseColor"][MAT_ROCK] = (0.55, 0.5, 0.45)
    mats["baseColor"][MAT_WATER] = (1.0, 1.0, 1.0)
    mats["bsdfType"][MAT_WATER] = 1
    mat_tex = np.array([TEX_CHECKER, TEX_LEAF, -1, -1, TEX_LEAF], np.int32)
    objects = []
    for k in range(W):
        x0, x1 = k / W, (k + 1) / W
        meshes = [ground_mesh(x0, x1, max(2, ground[0] // W), ground[1]), bush_mesh(14, 0xB05 + seed), bush_mesh(9, 0xB06 + seed, MAT_LEAF2),
                  rock_mesh(0x70C + seed), pond_mesh(x0, x1)]
        G, BUSH_A, BUSH_B, ROCK, POND = range(5)
        # level 2: an element = a rock with bushes around it (details instanced into an element)
        elements = {
            "cluster": [(ROCK, _affine()), (BUSH_A, _affine((0.9, 0.9, 1.1), 0.3, (0.55, 0.1, 0.0))),
                        (BUSH_B, _affine((0.7, 0.7, 0.8), 1.9, (-0.45, 0.35, 0.0))), (BUSH_A, _affine((0.6, 0.8, 0.7), 4.0, (0.05, -0.6, 0.0), tilt=0.25))],
            "thicket": [(BUSH_A, _affine((1.2, 1.2, 1.4), 0.0)), (BUSH_B, _affine((1.0, 1.0, 1.0), 2.2, (0.3, 0.3, 0.1)))],
        }
        # level 3: the scene object = ground + pond + instanced elements
        inst = [("mesh", G, np.eye(4)), ("mesh", POND, np.eye(4))]
        n = max(1, clusters // W)
        r = _rand(n * 6, 0xC1A + 97 * k + seed).reshape(n, 6)
        for j in range(n):
            cx = x0 + (0.08 + 0.84 * r[j, 0]) * (x1 - x0)
            cy = 0.06 + 0.88 * r[j, 1]
            s = cluster_scale * (1.0 + r[j, 2])
            mirror = -1.0 if j % 5 == 3 else 1.0                    # a mirrored instance: det < 0
            M = _affine((s * mirror, s * (0.8 + 0.4 * r[j, 3]), s), 2 * np.pi * r[j, 4], (cx, cy, float(ground_height(cx, cy)) - 0.2 * s))
            inst.append(("element", "cluster" if r[j, 5] < 0.7 else "thicket", M))
        objects.append(InstancedObject(k, k, meshes, flatten_hierarchy(inst, elements)))
    return {"objects": objects, "materials": mats, "material_textures": mat_tex,
            "textures": {TEX_CHECKER: checker_texture(), TEX_LEAF: leaf_texture()},
            "env_map": sky_env_map(), "env_rotation": 0.7, "lights": make_lights()}


# ---- Wavefront OBJ / MTL: the mesh format behind the reference's scene objects ("obj for small details", pipeline_helper.cpp:268) ----
def load_obj(path, material_ids=None):
    """Reads a Wavefront OBJ into the front end's mesh dicts, one per `usemtl` group (= one SBT record of the reference:
    its own materialID, normals / normalIndices / texCoords / texCoordsIndices, pipeline_helper.cpp:182-193). The three index
    streams of `f v/vt/vn` stay separate, exactly as HitGroupData keeps them; polygons are fanned into triangles; negative
    (relative) indices are resolved; a face without normals gets its geometric normal as a new shared entry.
    material_ids: {material name: index into the material table}; unknown / absent names get running indices.
    Returns (meshes, material_names) with material_names[i] = name of material index i."""
    pos, nrm, tex = [], [], []
    groups, order = {}, []
    names = dict(material_ids or {})
    cur = None

    def group(name):
        if name not in names:
            names[name] = max(names.values(), default=-1) + 1
        if name not in groups:
            groups[name] = {"v": [], "n": [], "t": [], "has_t": True}
            order.append(name)
        return groups[name]

    def fix(i, n):
        i = int(i)
        return i - 1 if i > 0 else n + i

    with open(path) as f:
        for line in f:
            p = line.split("#", 1)[0].split()
            if not p:
                continue
            if p[0] == "v":
                pos.append([float(x) for x in p[1:4]])
            elif p[0] == "vn":
                nrm.append([float(x) for x in p[1:4]])
            elif p[0] == "vt":
                tex.append([float(p[1]), float(p[2]) if len(p) > 2 else 0.0])
            elif p[0] == "usemtl":
                cur = group(p[1] if len(p) > 1 else "default")
            elif p[0] == "f":
                if cur is None:
                    cur = group("default")
                corners = []
                for c in p[1:]:
                    q = (c.split("/") + ["", ""])[:3]
                    corners.append((fix(q[0], len(pos)), fix(q[1], len(tex)) if q[1] else None, fix(q[2], len(nrm)) if q[2] else None))
                for k in range(1, len(corners) - 1):
                    tri = (corners[0], corners[k], corners[k + 1])
                    if any(c[2] is None for c in tri):
                        a, b, c3 = (np.asarray(pos[c[0]], np.float64) for c in tri)
                        n = np.cross(b - a, c3 - a)
                        ln = np.linalg.norm(n)
                        nrm.append((n / ln if ln > 0 else np.array([0.0, 0.0, 1.0])).tolist())
                        tri = tuple((c[0], c[1], len(nrm) - 1) for c in tri)
                    cur["v"].append([c[0] for c in tri]); cur["n"].append([c[2] for c in tri])
                    if any(c[1] is None for c in tri):
                        cur["has_t"] = False
                    cur["t"].append([c[1] if c[1] is not None else 0 for c in tri])
    P, N, T = np.asarray(pos, np.float32).reshape(-1, 3), np.asarray(nrm, np.float32).reshape(-1, 3), np.asarray(tex, np.float32).reshape(-1, 2)
    meshes = []
    for name in order:
        g = groups[name]
        if not g["v"]:
            continue
        has_t = g["has_t"] and T.shape[0] > 0
        meshes.append({"positions": P, "indices": np.asarray(g["v"], np.int32), "normals": N, "normal_indices": np.asarray(g["n"], np.int32),
                       "texcoords": T if has_t else None, "texcoord_indices": np.asarray(g["t"], np.int32) if has_t else None,
                       "material": names[name], "name": name})
    inv = sorted(names, key=lambda k: names[k])
    return meshes, inv


def save_obj(path, meshes, material_names=None):
    """Writes mesh dicts as one OBJ (one `usemtl` group per mesh, separate v / vt / vn index streams). For tests and for handing
    the procedural garden to other tools."""
    with open(path, "w") as f:
        vo = to = no = 0
        for k, m in enumerate(meshes):
            P = np.asarray(m["positions"], np.float32).reshape(-1, 3)
            N = np.asarray(m["normals"], np.float32).reshape(-1, 3)
            T = None if m.get("texcoords") is None else np.asarray(m["texcoords"], np.float32).reshape(-1, 2)
            for v in P:
                f.write("v %.9g %.9g %.9g\n" % tuple(v))
            for v in N:
                f.write("vn %.9g %.9g %.9g\n" % tuple(v))
            if T is not None:
                for v in T:
                    f.write("vt %.9g %.9g\n" % tuple(v))
            f.write("usemtl %s\n" % (material_names[m["material"]] if material_names else "mat%d" % m["material"]))
            I, NI = np.asarray(m["indices"]).reshape(-1, 3), np.asarray(m["normal_indices"]).reshape(-1, 3)
            TI = None if T is None else np.asarray(m["texcoord_indices"]).reshape(-1, 3)
            for t in range(I.shape[0]):
                if TI is None:
                    f.write("f " + " ".join("%d//%d" % (I[t, c] + 1 + vo, NI[t, c] + 1 + no) for c in range(3)) + "\n")
                else:
                    f.write("f " + " ".join("%d/%d/%d" % (I[t, c] + 1 + vo, TI[t, c] + 1 + to, NI[t, c] + 1 + no) for c in range(3)) + "\n")
            vo += P.shape[0]; no += N.shape[0]; to += 0 if T is None else T.shape[0]


def load_texture(path):
    """Image file -> [h, w, 4] float32 RGBA, row 0 = v 0 (the reference loads with stbi_loadf after
    stbi_set_flip_vertically_on_load(1), renderer.cpp:1636-1647: bottom row first, 4 components, alpha 1 when absent).
    .pfm / .exr through this package's own readers (RGB), anything else through OpenCV when it is installed."""
    low = path.lower()
    if low.endswith(".pfm") or low.endswith(".exr"):
        from .scene import load_exr, load_pfm
        rgb = load_pfm(path) if low.endswith(".pfm") else load_exr(path)
        img = np.concatenate([rgb, np.ones(rgb.shape[:2] + (1,), np.float32)], -1)
    else:
        import cv2
        raw = cv2.imread(path, cv2.IMREAD_UNCHANGED)
        if raw is None:
            raise FileNotFoundError(path)
        scale = 1.0 if raw.dtype.kind == "f" else 1.0 / np.iinfo(raw.dtype).max
        raw = raw.astype(np.float32) * np.float32(scale)
        if raw.ndim == 2:
            raw = np.repeat(raw[..., None], 3, -1)
        rgb = raw[..., 2::-1]
        a = raw[..., 3:4] if raw.shape[2] > 3 else np.ones(raw.shape[:2] + (1,), np.float32)
        img = np.concatenate([rgb, a], -1)
    return np.ascontiguousarray(img[::-1], np.float32)


def save_scene_v2(path, garden, cam, flatten):
    """Scene file of the C++ host in its real-scene variant (csrc/dprt_render.cpp documents the layout): the dict of make_garden
    (or the same keys filled from load_obj / load_texture) with every object flattened by `flatten` = host.flatten_instances
    (dprt_flatten_instances: what dprt_upload_instanced_chunk would do); an object that already carries its flat streams
    as `.flat = (verts9, normals9, uv6 or None, mat_ids)` is written as is (obj2scene.py cuts one flattened scene into chunks).
    A scene with a "material_roughness" table (one float per material, dprt_set_material_roughness) is written as DPRTSCN3:
    the same bytes after the magic, then the table."""
    import ctypes as C
    mats, mat_tex = np.ascontiguousarray(garden["materials"], D.MATERIAL_DTYPE), np.full(len(garden["materials"]), -1, np.int32)
    mt = np.asarray(garden.get("material_textures", []), np.int32)
    mat_tex[:mt.size] = mt
    textures = garden.get("textures") or {}
    rough = garden.get("material_roughness")
    if rough is not None:
        rough = np.ascontiguousarray(rough, np.float32)
        if rough.shape != (len(mats),):
            raise ValueError(f"material_roughness has shape {rough.shape}, the scene has {len(mats)} materials")
    with open(path, "wb") as f:
        f.write(b"DPRTSCN2" if rough is None else b"DPRTSCN3")
        f.write(np.array([len(garden["objects"]), len(mats), len(garden["lights"]), len(textures)], np.int32).tobytes())
        f.write(bytes(C.string_at(C.addressof(cam), C.sizeof(cam))))
        f.write(mats.tobytes()); f.write(mat_tex.tobytes())
        f.write(np.ascontiguousarray(garden["lights"], D.LIGHT_DTYPE).tobytes())
        for slot in sorted(textures):
            t = np.ascontiguousarray(textures[slot], np.float32)
            f.write(np.array([slot, t.shape[1], t.shape[0]], np.int32).tobytes()); f.write(t.tobytes())
        env = garden.get("env_map")
        if env is None:
            f.write(np.array([0, 0], np.int32).tobytes()); f.write(np.float32(0.0).tobytes())
        else:
            e = np.ascontiguousarray(env, np.float32)
            f.write(np.array([e.shape[1], e.shape[0]], np.int32).tobytes()); f.write(np.float32(garden.get("env_rotation", 0.0)).tobytes())
            f.write(e.tobytes())
        for ob in garden["objects"]:
            v, n, uv, m = ob.flat if getattr(ob, "flat", None) is not None else flatten(ob.meshes, ob.instances)
            d = ob.desc(False)
            f.write(bytes(C.string_at(C.addressof(d), C.sizeof(d))))
            f.write(np.array([v.shape[0]], np.int64).tobytes())
            f.write(np.array([0 if uv is None else 1], np.int32).tobytes())
            f.write(np.ascontiguousarray(v, np.float32).tobytes()); f.write(np.ascontiguousarray(n, np.float32).tobytes())
            if uv is not None:
                f.write(np.ascontiguousarray(uv, np.float32).tobytes())
            f.write(np.ascontiguousarray(m, np.int32).tobytes())
            f.write(np.array([0], np.int64).tobytes()); f.write(np.array([0], np.int64).tobytes())      # no proxy networks
        if rough is not None:
            f.write(rough.tobytes())
