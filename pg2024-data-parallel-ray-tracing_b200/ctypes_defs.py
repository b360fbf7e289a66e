"""ctypes / numpy mirrors of include/dprt_types.h (shared by the libdprt binding and the oracle binding).

Every structure here restates one POD of ``include/dprt_types.h``; sizes are asserted at import.
"""
import ctypes as C

import numpy as np

DPRT_EPSILON = 1e-3
MAX_WORLD = 32


class Config(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("bounces", C.c_int32),
                ("shadowPathCount", C.c_int32), ("maxCount", C.c_int32), ("sceneSize", C.c_int32),
                ("proxyMode", C.c_int32), ("pathGenMode", C.c_int32), ("mlpDtype", C.c_int32),
                ("envColor", C.c_float * 3), ("mainRayRetrace", C.c_int32), ("serialStages", C.c_int32),
                ("referenceMigrate", C.c_int32)]


class ObjectDesc(C.Structure):
    _fields_ = [("nodeID", C.c_int32), ("isProxy", C.c_int32), ("aabbMin", C.c_float * 3), ("aabbMax", C.c_float * 3),
                ("maxLength", C.c_float), ("worldToObject", C.c_float * 12)]


class Camera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("U", C.c_float * 3), ("V", C.c_float * 3), ("W", C.c_float * 3),
                ("width", C.c_int32), ("height", C.c_int32)]


class MeshDesc(C.Structure):
    """dprt_mesh_desc: one GAS + its HitGroupData in indexed form (pipeline_helper.cpp:182-193)."""
    _fields_ = [("positions", C.c_void_p), ("nPositions", C.c_int64), ("indices", C.c_void_p), ("ntris", C.c_int64),
                ("normals", C.c_void_p), ("nNormals", C.c_int64), ("normalIndices", C.c_void_p),
                ("texCoords", C.c_void_p), ("nTexCoords", C.c_int64), ("texCoordIndices", C.c_void_p),
                ("materialID", C.c_int32), ("pad_", C.c_int32)]


class InstanceDesc(C.Structure):
    """dprt_instance_desc: mesh index + row-major 3x4 object-to-world matrix."""
    _fields_ = [("mesh", C.c_int32), ("pad_", C.c_int32), ("objectToWorld", C.c_float * 12)]


class DenoiseParams(C.Structure):
    """dprt_denoise_params (DESIGN.md 3.8)."""
    _fields_ = [("iterations", C.c_int32), ("sigma_color", C.c_float), ("sigma_normal", C.c_float), ("sigma_albedo", C.c_float)]


# DPRT_DENOISE_DEFAULT_*: what a NULL dprt_denoise_params selects
DENOISE_DEFAULTS = {"iterations": 3, "sigma_color": 2.0, "sigma_normal": 1.0, "sigma_albedo": 0.3}


MAX_TEXTURES = 64
MAX_MATERIALS = 256


def pack_meshes(meshes, instances):
    """meshes: list of dicts {positions [nP,3], indices [nT,3], normals [nN,3], normal_indices [nT,3], texcoords [nU,2] | None,
    texcoord_indices [nT,3] | None, material int}; instances: list of (mesh index, 3x4 float matrix).
    Returns (MeshDesc array, n_meshes, InstanceDesc array, n_instances, keepalive list of the numpy arrays behind the pointers)."""
    keep = []

    def arr(a, dt, cols):
        a = np.ascontiguousarray(a, dt).reshape(-1, cols)
        keep.append(a)
        return a

    md = (MeshDesc * len(meshes))()
    for k, m in enumerate(meshes):
        pos, idx = arr(m["positions"], np.float32, 3), arr(m["indices"], np.int32, 3)
        nrm, nidx = arr(m["normals"], np.float32, 3), arr(m["normal_indices"], np.int32, 3)
        assert nidx.shape == idx.shape
        md[k].positions, md[k].nPositions = pos.ctypes.data, pos.shape[0]
        md[k].indices, md[k].ntris = idx.ctypes.data, idx.shape[0]
        md[k].normals, md[k].nNormals = nrm.ctypes.data, nrm.shape[0]
        md[k].normalIndices = nidx.ctypes.data
        if m.get("texcoords") is not None:
            tc, tidx = arr(m["texcoords"], np.float32, 2), arr(m["texcoord_indices"], np.int32, 3)
            assert tidx.shape == idx.shape
            md[k].texCoords, md[k].nTexCoords, md[k].texCoordIndices = tc.ctypes.data, tc.shape[0], tidx.ctypes.data
        else:
            md[k].texCoords, md[k].nTexCoords, md[k].texCoordIndices = None, 0, None
        md[k].materialID = int(m["material"])
    ins = (InstanceDesc * len(instances))()
    for k, (mi, M) in enumerate(instances):
        ins[k].mesh = int(mi)
        ins[k].objectToWorld[:] = np.asarray(M, np.float32).reshape(12).tolist()
    return md, len(meshes), ins, len(instances), keep


class Stats(C.Structure):
    _fields_ = [("rays_traverse", C.c_int64), ("rays_shade", C.c_int64), ("rays_shadow", C.c_int64),
                ("rays_secondary", C.c_int64), ("nn_queries", C.c_int64), ("paths_sent_offrank", C.c_int64),
                ("exchange_iters", C.c_int64), ("kernel_launches", C.c_int64), ("bytes_alltoall", C.c_int64),
                ("rays_shade_cached", C.c_int64), ("rays_walked", C.c_int64), ("walked_traverse", C.c_int64),
                ("walked_shade", C.c_int64), ("walked_shadow", C.c_int64), ("walked_secondary", C.c_int64), ("paths_partitioned", C.c_int64),
                ("shade_cache_stale", C.c_int64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_ if k != "reserved_"}


PATH_DTYPE = np.dtype([("origin", "<f4", 3), ("direction", "<f4", 3), ("tMax", "<f4"), ("throughput", "<f4", 3),
                       ("pixelIndex", "<i4"), ("shadowPathID", "<i4"), ("visitedMask", "<u4"), ("currentNode", "<i4"),
                       ("targetNode", "<i4"), ("isShadowRay", "u1"), ("isDelta", "u1"), ("isValid", "u1"), ("isHit", "u1")])
QUERY_DTYPE = np.dtype([("throughput", "<f4", 3), ("pixelIndex", "<i4"), ("hitSequence", "<i4"), ("hitAABBID", "<i4"),
                        ("shadowPathID", "<i4"), ("instanceID", "<i4"), ("pathIndex", "<i4"), ("normalizedT", "<f4"),
                        ("isValid", "u1"), ("isInside", "u1"), ("pad_", "u1", 2), ("reserved_", "<i4")])
RAY_DTYPE = np.dtype([("origin", "<f4", 3), ("tMin", "<f4"), ("direction", "<f4", 3), ("tMax", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("primID", "<i4")])
MATERIAL_DTYPE = np.dtype([("baseColor", "<f4", 3), ("bsdfType", "<i4")])
LIGHT_DTYPE = np.dtype([("p0", "<f4", 3), ("p1", "<f4", 3), ("p2", "<f4", 3), ("Le", "<f4", 3)])
NODE_DTYPE = np.dtype([("p", "<f4", 3), ("e", "u1", 3), ("imask", "u1"), ("childBase", "<u4"), ("triBase", "<u4"),
                       ("tmask", "<u4"), ("reserved_", "<u4"), ("qlox", "u1", 8), ("qloy", "u1", 8), ("qloz", "u1", 8),
                       ("qhix", "u1", 8), ("qhiy", "u1", 8), ("qhiz", "u1", 8)])
TRI_DTYPE = np.dtype([("v0", "<f4", 3), ("primID", "<i4"), ("v1", "<f4", 3), ("matID", "<i4"), ("v2", "<f4", 3), ("pad_", "<i4")])

assert PATH_DTYPE.itemsize == 64 and QUERY_DTYPE.itemsize == 48 and RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 8
assert NODE_DTYPE.itemsize == 80 and TRI_DTYPE.itemsize == 48 and MATERIAL_DTYPE.itemsize == 16 and LIGHT_DTYPE.itemsize == 48
assert C.sizeof(Config) == 64 and C.sizeof(ObjectDesc) == 84 and C.sizeof(Camera) == 56 and C.sizeof(Stats) == 136
assert C.sizeof(MeshDesc) == 88 and C.sizeof(InstanceDesc) == 56

P2P_HANDLE_BYTES = 208     # DPRT_P2P_HANDLE_BYTES

# dprt_buffer_id
BUF_PATHS, BUF_TRANSFER, BUF_TRANSFER_OFFSET, BUF_DIRECT, BUF_ENV, BUF_NN_INPUT, BUF_NN_QUERY, BUF_NN_PACKED_INPUT, \
    BUF_NN_PACKED_QUERY, BUF_SCENE_OFFSET, BUF_PRED, BUF_OCCLUSION, BUF_CONTRIBUTION, BUF_HIT_PRIM, BUF_AOV = range(15)

# dprt_stage_id
STAGE_NAMES = ("path_gen", "traverse", "partition", "exchange", "shade", "shadow_trace", "secondary_trace", "bucket",
               "proxy_mlp", "frame_update", "depth_update", "target_update", "image", "trace_closest")
STAGE_COUNT = len(STAGE_NAMES)

BUFFER_DTYPES = {
    BUF_PATHS: PATH_DTYPE, BUF_TRANSFER: PATH_DTYPE, BUF_TRANSFER_OFFSET: np.dtype("<i4"), BUF_DIRECT: np.dtype("<f4"),
    BUF_ENV: np.dtype("<f4"), BUF_NN_INPUT: np.dtype("<u2"), BUF_NN_QUERY: QUERY_DTYPE, BUF_NN_PACKED_INPUT: np.dtype("<u2"),
    BUF_NN_PACKED_QUERY: QUERY_DTYPE, BUF_SCENE_OFFSET: np.dtype("<i4"), BUF_PRED: np.dtype("<u2"),
    BUF_OCCLUSION: np.dtype("<f4"), BUF_CONTRIBUTION: np.dtype("<f4"), BUF_HIT_PRIM: np.dtype("<i4"), BUF_AOV: np.dtype("<f4"),
}


def make_config(width, height, spp=1, bounces=4, spc=4, mc=3, scene_size=1, proxy_mode=0, path_gen_mode=0,
                mlp_dtype=1, env_color=(0.6, 0.7, 0.9), main_ray_retrace=0, serial_stages=0, reference_migrate=0):
    cfg = Config()
    cfg.mainRayRetrace, cfg.serialStages, cfg.referenceMigrate = int(main_ray_retrace), int(serial_stages), int(reference_migrate)
    cfg.width, cfg.height, cfg.spp, cfg.bounces = width, height, spp, bounces
    cfg.shadowPathCount, cfg.maxCount, cfg.sceneSize = spc, mc, scene_size
    cfg.proxyMode, cfg.pathGenMode, cfg.mlpDtype = proxy_mode, path_gen_mode, mlp_dtype
    cfg.envColor[:] = [float(c) for c in env_color]
    return cfg


def make_object_desc(node_id, aabb_min, aabb_max, is_proxy=0, world_to_object=None):
    d = ObjectDesc()
    d.nodeID, d.isProxy = int(node_id), int(is_proxy)
    mn = np.asarray(aabb_min, np.float32)
    mx = np.asarray(aabb_max, np.float32)
    d.aabbMin[:] = mn.tolist()
    d.aabbMax[:] = mx.tolist()
    diff = (mx - mn).astype(np.float32)
    # (aabb.m_max - aabb.m_min).length() in fp32, renderer.cpp:1830: fma(z,z,fma(y,y,x*x)) then sqrt
    acc = np.float32(diff[0] * diff[0])
    acc = np.float32(np.float64(diff[1]) * np.float64(diff[1]) + np.float64(acc))
    acc = np.float32(np.float64(diff[2]) * np.float64(diff[2]) + np.float64(acc))
    d.maxLength = float(np.sqrt(acc, dtype=np.float32))
    m = np.eye(4, dtype=np.float32)[:3] if world_to_object is None else np.asarray(world_to_object, np.float32).reshape(3, 4)
    d.worldToObject[:] = m.reshape(-1).tolist()
    return d


def make_camera(origin, look_at, up, vfov_deg, width, height):
    """Pinhole camera basis, pre-scaled like dprt_camera documents (computed in float64, stored float32)."""
    o = np.asarray(origin, np.float64)
    w = np.asarray(look_at, np.float64) - o
    w /= np.linalg.norm(w)
    u = np.cross(w, np.asarray(up, np.float64))
    u /= np.linalg.norm(u)
    v = np.cross(u, w)
    th = np.tan(np.radians(vfov_deg) / 2.0)
    cam = Camera()
    cam.origin[:] = o.astype(np.float32).tolist()
    cam.U[:] = (u * th * (width / height)).astype(np.float32).tolist()
    cam.V[:] = (v * th).astype(np.float32).tolist()
    cam.W[:] = w.astype(np.float32).tolist()
    cam.width, cam.height = int(width), int(height)
    return cam
