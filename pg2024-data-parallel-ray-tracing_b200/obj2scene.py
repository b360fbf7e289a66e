#!/usr/bin/env python
"""Wavefront OBJ (+ MTL, + texture images) -> scene file of the C++ host (`dprt_render --scene`, DPRTSCN2 layout).

The reference renders OBJ-based scenes (Bistro, San Miguel; "obj for small details", pipeline_helper.cpp:268) whose loaders
are not in its tree. This is the equivalent path here, host only (no GPU): the OBJ's `usemtl` groups become meshes with their
own v / vt / vn index streams (HitGroupData, pipeline_helper.cpp:182-193), the MTL gives base colour (`Kd`), albedo / opacity
map (`map_Kd`, loaded bottom row first like stbi_loadf after stbi_set_flip_vertically_on_load(1), renderer.cpp:1636-1647) and
the BSDF (a dielectric `illum` 4 / 6 / 7 / 9 or `Ni` within 0.05 of 1.33 -> Water, everything else Lambertian: the two BSDFs the
reference has; with --glossy, metallic and specular materials become the rough conductor and the glossy plastic, see
glossy_material), the geometry is flattened by dprt_flatten_instances and cut into W x-slabs by triangle centroid (one scene
object per chunk owner), and everything is written with real_scene.save_scene_v2.

    python pg2024-data-parallel-ray-tracing_b200/obj2scene.py scene.obj --out scene.dprt [--world 2] [--width 1920 --height 1080]
           [--eye x,y,z --look-at x,y,z --up 0,0,1 --vfov 40] [--env sky.pfm|sky.exr --env-rotation 2.0] [--lights default|bistro|...]
           [--glossy]
    dprt_render --scene scene.dprt --out image.exr --spp 64 --world 2
"""
import argparse
import importlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
D = dprt.ctypes_defs
RS = dprt.real_scene


def _mtl_default():
    return {"Kd": (0.8, 0.8, 0.8), "map_Kd": None, "water": False, "Ks": (0.0, 0.0, 0.0), "Ns": None, "illum": None, "Pr": None,
            "Pm": None}


def load_mtl(path):
    """{name: {"Kd": (r, g, b), "map_Kd": file or None, "water": bool, "Ks": (r, g, b), "Ns", "illum", "Pr", "Pm": number or
    None when absent}} from a Wavefront MTL file (Pr / Pm: roughness and metallic of the PBR extension)."""
    mats, cur = {}, None
    with open(path) as f:
        for line in f:
            p = line.split("#", 1)[0].split()
            if not p:
                continue
            if p[0] == "newmtl":
                cur = mats.setdefault(p[1] if len(p) > 1 else "default", _mtl_default())
            elif cur is None:
                continue
            elif p[0] == "Kd" and len(p) >= 4:
                cur["Kd"] = tuple(float(x) for x in p[1:4])
            elif p[0] == "map_Kd" and len(p) >= 2:
                cur["map_Kd"] = p[-1]
            elif p[0] == "illum" and len(p) >= 2:
                cur["illum"] = int(float(p[1]))
                if cur["illum"] in (4, 6, 7, 9):
                    cur["water"] = True
            elif p[0] == "Ni" and len(p) >= 2 and abs(float(p[1]) - 1.33) < 0.05:
                cur["water"] = True
            elif p[0] == "Ks" and len(p) >= 4:
                cur["Ks"] = tuple(float(x) for x in p[1:4])
            elif p[0] in ("Ns", "Pr", "Pm") and len(p) >= 2:
                cur[p[0]] = float(p[1])
    return mats


def glossy_material(m):
    """(bsdfType, roughness) of an MTL material under --glossy, or None when it stays as without the flag:
    - `Pm` >= 0.5 (metallic): the rough conductor (bsdfType 2), F0 = `Kd` (or the `map_Kd` texel);
    - otherwise a non-water material with a non-zero `Ks` and `illum` >= 2: the glossy plastic (bsdfType 3), diffuse colour `Kd`
      (or the `map_Kd` texel). `Ks`'s colour is not used: the plastic's coat has the fixed F0 0.04 (DESIGN.md 3.13).
    Roughness: `Pr` when given, else (2 / (Ns + 2))^(1/4) (Walter et al. 2007's Phong-exponent match alpha = sqrt(2 / (Ns + 2))
    with alpha = r^2; a missing `Ns` counts as 0), clipped to [0, 1]."""
    if m["Pm"] is not None and m["Pm"] >= 0.5:
        kind = 2
    elif not m["water"] and any(k != 0.0 for k in m["Ks"]) and m["illum"] is not None and m["illum"] >= 2:
        kind = 3
    else:
        return None
    r = m["Pr"] if m["Pr"] is not None else (2.0 / (max(m["Ns"] or 0.0, 0.0) + 2.0)) ** 0.25
    return kind, float(np.clip(r, 0.0, 1.0))


def mtllibs_of(obj_path):
    libs = []
    with open(obj_path) as f:
        for line in f:
            p = line.split()
            if p and p[0] == "mtllib":
                libs += p[1:]
    return libs


class FlatObject:
    """One chunk owner's share of the flattened scene, in the shape real_scene.save_scene_v2 expects of an object."""

    def __init__(self, index, v, n, uv, m):
        self.index, self.node_id = index, index
        self.flat = (v, n, uv, m)
        self.meshes, self.instances = None, None
        P = v.reshape(-1, 3)
        self.aabb_min, self.aabb_max = P.min(0).astype(np.float32) - np.float32(1e-3), P.max(0).astype(np.float32) + np.float32(1e-3)

    def desc(self, is_proxy):
        return D.make_object_desc(self.node_id, self.aabb_min, self.aabb_max, is_proxy=int(is_proxy))


def convert(obj_path, out_path, world=1, width=1920, height=1080, eye=None, look_at=None, up=(0, 0, 1), vfov=40.0, env=None,
            env_rotation=0.0, lights="fit", light_scale=1.0, glossy=False):
    """Writes the scene file; glossy: map metallic and specular MTL materials to bsdfType 2 / 3 (glossy_material) and write
    their roughness table (DPRTSCN3) when any material was mapped. Without it the file does not depend on Ks / Ns / Pr / Pm."""
    base = os.path.dirname(os.path.abspath(obj_path))
    mtl = {}
    for lib in mtllibs_of(obj_path):
        p = os.path.join(base, lib)
        if os.path.exists(p):
            mtl.update(load_mtl(p))
    meshes, names = RS.load_obj(obj_path)
    if not meshes:
        raise SystemExit(f"{obj_path}: no faces")
    if len(names) > D.MAX_MATERIALS:
        raise SystemExit(f"{len(names)} materials: the material table holds {D.MAX_MATERIALS}")
    mats = np.zeros(len(names), D.MATERIAL_DTYPE)
    mat_tex = np.full(len(names), -1, np.int32)
    textures, slot_of = {}, {}
    rough, mapped = np.zeros(len(names), np.float32), False
    for i, nm in enumerate(names):
        m = mtl.get(nm, _mtl_default())
        mats["baseColor"][i] = (1.0, 1.0, 1.0) if m["water"] else m["Kd"]
        mats["bsdfType"][i] = 1 if m["water"] else 0
        g = glossy_material(m) if glossy else None
        if g is not None:
            mats["baseColor"][i] = m["Kd"]
            mats["bsdfType"][i], rough[i], mapped = g[0], g[1], True
        if m["map_Kd"]:
            f = os.path.join(base, m["map_Kd"].replace("\\", "/"))
            if f not in slot_of:
                if len(slot_of) >= D.MAX_TEXTURES:
                    raise SystemExit(f"more than {D.MAX_TEXTURES} distinct textures")
                slot_of[f] = len(slot_of)
                textures[slot_of[f]] = RS.load_texture(f)
            mat_tex[i] = slot_of[f]
    ident = [(k, np.eye(4, dtype=np.float32)[:3]) for k in range(len(meshes))]
    v, n, uv, m = dprt.flatten_instances(meshes, ident)
    # W x-slabs with equal triangle counts, by centroid: one scene object per chunk owner (renderer.cpp:1812-1842)
    cx = v.reshape(-1, 3, 3)[:, :, 0].mean(1)
    order = np.argsort(cx, kind="stable")
    objects = []
    for k in range(world):
        sel = np.sort(order[len(order) * k // world: len(order) * (k + 1) // world])
        if sel.size == 0:
            raise SystemExit(f"chunk {k} of {world} would be empty")
        objects.append(FlatObject(k, v[sel], n[sel], None if uv is None else uv[sel], m[sel]))
    lo, hi = v.reshape(-1, 3).min(0), v.reshape(-1, 3).max(0)
    ctr, ext = 0.5 * (lo + hi), float(np.linalg.norm(hi - lo))
    up = np.asarray(up, np.float64)
    if look_at is None:
        look_at = ctr
    if eye is None:      # three quarters of a diagonal away, above the horizon along `up`
        side = np.cross(up, [1.0, 0.0, 0.0]) if abs(up[0]) < 0.9 else np.cross(up, [0.0, 1.0, 0.0])
        eye = np.asarray(look_at, np.float64) - 0.75 * ext * side / np.linalg.norm(side) + 0.45 * ext * up / np.linalg.norm(up)
    cam = D.make_camera(eye, look_at, up, vfov, width, height)
    if lights == "fit":  # the benchmark's two downward-facing area-light triangles, scaled with the scene (area / distance^2 is scale-free)
        L = dprt.scene.make_lights(light_scale)
        upn = up / np.linalg.norm(up)
        a = np.cross(upn, [1.0, 0.0, 0.0]) if abs(upn[0]) < 0.9 else np.cross(upn, [0.0, 1.0, 0.0])
        a /= np.linalg.norm(a)
        b = np.cross(upn, a)
        for key in ("p0", "p1", "p2"):
            q = L[key].astype(np.float64) - np.array([0.5, 0.5, 2.0])          # make_lights: a 0.5 square at height 2 over the unit square
            L[key] = (ctr + 0.5 * ext * (q[:, 0:1] * a + q[:, 1:2] * b) + (0.5 * float(np.dot(hi - lo, np.abs(upn))) + 0.75 * ext) * upn).astype(np.float32)
        # the light normal must face the scene: swap two corners if it points along +up
        for i in range(L.size):
            nrm = np.cross(L["p1"][i] - L["p0"][i], L["p2"][i] - L["p0"][i])
            if np.dot(nrm, upn) > 0:
                L["p1"][i], L["p2"][i] = L["p2"][i].copy(), L["p1"][i].copy()
    else:
        L = dprt.scene.reference_lights(lights)
    garden = {"objects": objects, "materials": mats, "material_textures": mat_tex, "textures": textures, "lights": L,
              "env_map": None if env is None else RS.load_texture(env), "env_rotation": env_rotation}
    if mapped:
        garden["material_roughness"] = rough
    RS.save_scene_v2(out_path, garden, cam, dprt.flatten_instances)
    return {"triangles": int(v.shape[0]), "materials": names, "textures": {s: list(t.shape) for s, t in textures.items()},
            "chunks": [int(o.flat[0].shape[0]) for o in objects], "bounds": [lo.tolist(), hi.tolist()]}


def _vec(s):
    return tuple(float(x) for x in s.split(","))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("obj")
    ap.add_argument("--out", required=True)
    ap.add_argument("--world", type=int, default=1, help="chunk owners (ranks / GPUs): the scene is cut into this many x-slabs")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--eye", type=_vec); ap.add_argument("--look-at", type=_vec); ap.add_argument("--up", type=_vec, default=(0.0, 0.0, 1.0))
    ap.add_argument("--vfov", type=float, default=40.0)
    ap.add_argument("--env"); ap.add_argument("--env-rotation", type=float, default=0.0)
    ap.add_argument("--lights", default="fit", help='"fit" (two area lights over the scene) or a table of scene.reference_lights: default, san_miguel, air_drome, bistro')
    ap.add_argument("--light-scale", type=float, default=1.0)
    ap.add_argument("--glossy", action="store_true", help="metallic (Pm >= 0.5) -> rough conductor, specular (Ks != 0, illum >= 2) -> "
                    "glossy plastic, roughness from Pr or Ns; writes DPRTSCN3 when any material maps")
    a = ap.parse_args()
    import json
    print(json.dumps(convert(a.obj, a.out, a.world, a.width, a.height, a.eye, a.look_at, a.up, a.vfov, a.env, a.env_rotation, a.lights, a.light_scale,
                             a.glossy)))


if __name__ == "__main__":
    main()
