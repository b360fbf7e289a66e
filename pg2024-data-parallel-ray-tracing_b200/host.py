"""ctypes binding of libdprt.so -- the reference-side stub a maintainer would write (INTEGRATION.md).

``Renderer`` mirrors ``moana::Renderer`` of the reference (src/render/renderer.cpp): ``launch`` ->
:meth:`Renderer.launch`, ``runSample`` -> :meth:`Renderer.run_sample`, and one method per stage helper
(``primaryRayModule`` :1212, ``generateSecondaryAndShadowRay`` :1320, ``shadowRayModuleBasedNN`` :1349,
``secondaryRayModuleBasedNN`` :1407) plus the free functions of src/cuda (``Work_Efficient_Scan`` ->
:meth:`partition`, ``Frame_Buffer_Update`` -> :meth:`frame_buffer_update`, ...). There is no CPU fallback:
a missing library or a box without a GPU raises.
"""
import ctypes as C
import os

import numpy as np

from . import ctypes_defs as D

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdprt.so")

_PROTOTYPES = {
    # name: (restype, argtypes)
    "dprt_get_unique_id": (C.c_int, [C.c_void_p]),
    "dprt_create": (C.c_int, [C.POINTER(D.Config), C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "dprt_create_shared": (C.c_int, [C.POINTER(D.Config), C.c_void_p, C.POINTER(C.c_void_p)]),
    "dprt_destroy": (None, [C.c_void_p]),
    "dprt_last_error": (C.c_char_p, [C.c_void_p]),
    "dprt_synchronize": (C.c_int, [C.c_void_p]),
    "dprt_get_stats": (C.c_int, [C.c_void_p, C.POINTER(D.Stats)]),
    "dprt_reset_stats": (C.c_int, [C.c_void_p]),
    "dprt_bvh8_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.POINTER(C.c_void_p)]),
    "dprt_bvh8_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "dprt_bvh8_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "dprt_bvh8_free": (None, [C.c_void_p]),
    "dprt_upload_chunk": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(D.ObjectDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "dprt_refit_chunk": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]),
    "dprt_refit_chunk_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]),
    "dprt_spec_bvh8_refit": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "dprt_chunk_bvh8_copy": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]),
    "dprt_upload_proxy": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(D.ObjectDesc), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    "dprt_flatten_count": (C.c_int64, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "dprt_flatten_instances": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_int)]),
    "dprt_upload_chunk_uv": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(D.ObjectDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "dprt_upload_instanced_chunk": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(D.ObjectDesc), C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "dprt_set_texture": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "dprt_set_material_textures": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "dprt_set_env_map": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float]),
    "dprt_spec_texture_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "dprt_spec_env_lookup": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int64, C.c_void_p]),
    "dprt_set_materials": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "dprt_set_lights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "dprt_set_camera": (C.c_int, [C.c_void_p, C.POINTER(D.Camera)]),
    "dprt_reset_frame": (C.c_int, [C.c_void_p]),
    "dprt_begin_sample": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_path_gen": (C.c_int, [C.c_void_p]),
    "dprt_traverse": (C.c_int, [C.c_void_p]),
    "dprt_partition": (C.c_int, [C.c_void_p]),
    "dprt_exchange": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "dprt_plan_exchange": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64),
                                    C.POINTER(C.c_int)]),
    "dprt_plan_exchange_deque": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32),
                                           C.POINTER(C.c_int32), C.POINTER(C.c_int)]),
    "dprt_shade": (C.c_int, [C.c_void_p]),
    "dprt_reset_nn": (C.c_int, [C.c_void_p]),
    "dprt_shadow_trace": (C.c_int, [C.c_void_p]),
    "dprt_secondary_trace": (C.c_int, [C.c_void_p]),
    "dprt_bucket_queries": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "dprt_proxy_infer": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "dprt_frame_buffer_update": (C.c_int, [C.c_void_p]),
    "dprt_depth_buffer_update": (C.c_int, [C.c_void_p]),
    "dprt_target_node_update": (C.c_int, [C.c_void_p]),
    "dprt_primary_ray_module": (C.c_int, [C.c_void_p]),
    "dprt_shadow_ray_module": (C.c_int, [C.c_void_p]),
    "dprt_secondary_ray_module": (C.c_int, [C.c_void_p]),
    "dprt_render_sample": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_reduce_image": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "dprt_enable_aov": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_reduce_aov": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "dprt_reduce_aov_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "dprt_denoise": (C.c_int, [C.c_void_p, C.POINTER(D.DenoiseParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dprt_denoise_device": (C.c_int, [C.c_void_p, C.POINTER(D.DenoiseParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "dprt_spec_denoise": (C.c_int, [C.POINTER(D.DenoiseParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dprt_adopt_scene": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dprt_accumulate_from": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dprt_p2p_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dprt_p2p_connect": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "dprt_p2p_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_p2p_enabled": (C.c_int, [C.c_void_p]),
    "dprt_exchange_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_int)]),
    "dprt_render_sample_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    "dprt_reduce_image_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p]),
    "dprt_get_path_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "dprt_set_path_size": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_buffer_bytes": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "dprt_download": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "dprt_upload": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "dprt_enable_hit_prim": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_trace_closest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "dprt_trace_closest_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "dprt_gen_train_data": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "dprt_gen_precom_data": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dprt_mlp_infer": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "dprt_mlp_infer_device": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "dprt_device_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "dprt_device_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dprt_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "dprt_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "dprt_timer_start": (C.c_int, [C.c_void_p]),
    "dprt_timer_stop": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "dprt_flush_l2": (C.c_int, [C.c_void_p]),
    "dprt_stage_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_get_stage_times": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "dprt_enable_counters": (C.c_int, [C.c_void_p, C.c_int]),
    "dprt_get_counters": (C.c_int, [C.c_void_p, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOTYPES)

_lib = None


class DprtError(RuntimeError):
    pass


def load_library(path=None):
    """dlopen libdprt.so and bind every prototype of include/dprt.h. Raises if the library is absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("DPRT_LIB") or LIB_PATH      # DPRT_LIB: A/B builds of the same ABI (profiles/)
    if not os.path.exists(p):
        raise DprtError(f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(p)
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if path is None:
        _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def get_unique_id():
    buf = (C.c_char * 128)()
    rc = load_library().dprt_get_unique_id(buf)
    if rc:
        raise DprtError(f"dprt_get_unique_id failed: {rc}")
    return bytes(buf)


def build_bvh8(verts9, mat_ids=None, pad=-1.0):
    """Host BVH8 build -> (nodes[NODE_DTYPE], tris[TRI_DTYPE], max_depth). No GPU needed."""
    lib = load_library()
    v = np.ascontiguousarray(verts9, np.float32).reshape(-1, 9)
    m = None if mat_ids is None else np.ascontiguousarray(mat_ids, np.int32)
    h = C.c_void_p()
    rc = lib.dprt_bvh8_build(_ptr(v), _ptr(m), v.shape[0], float(pad), C.byref(h))
    if rc:
        raise DprtError(f"dprt_bvh8_build failed: {rc}")
    try:
        nn, nt, md = C.c_int64(), C.c_int64(), C.c_int32()
        lib.dprt_bvh8_info(h, C.byref(nn), C.byref(nt), C.byref(md))
        nodes = np.zeros(nn.value, D.NODE_DTYPE)
        tris = np.zeros(nt.value, D.TRI_DTYPE)
        lib.dprt_bvh8_copy(h, _ptr(nodes), _ptr(tris))
    finally:
        lib.dprt_bvh8_free(h)
    return nodes, tris, int(md.value)


def spec_bvh8_refit(nodes, tris, verts9):
    """dprt_spec_bvh8_refit (host only, no GPU): the BVH8 (nodes[NODE_DTYPE], tris[TRI_DTYPE], e.g. from build_bvh8) refitted to
    new corners verts9 [ntris, 9] indexed by primID, exactly as dprt_refit_chunk does it on the device. Returns refitted
    copies; the inputs are left alone. Raises on a malformed blob, a size mismatch or a non-finite vertex."""
    n = np.array(nodes, D.NODE_DTYPE, copy=True)
    t = np.array(tris, D.TRI_DTYPE, copy=True)
    v = np.ascontiguousarray(verts9, np.float32).reshape(-1, 9)
    if v.shape[0] != t.shape[0]:
        raise DprtError(f"spec_bvh8_refit: {v.shape[0]} vertex triples for {t.shape[0]} triangle records")
    rc = load_library().dprt_spec_bvh8_refit(_ptr(n), n.shape[0], _ptr(t), t.shape[0], _ptr(v))
    if rc:
        raise DprtError(f"dprt_spec_bvh8_refit failed ({rc})")
    return n, t


def flatten_instances(meshes, instances):
    """dprt_flatten_instances (host only, no GPU): indexed meshes + instance transforms -> (verts9 [n,9], normals9 [n,9],
    uv6 [n,6] or None, mat_ids [n]); primitive id = running index over (instance, triangle). See ctypes_defs.pack_meshes."""
    lib = load_library()
    md, nm, ins, ni, keep = D.pack_meshes(meshes, instances)
    n = lib.dprt_flatten_count(md, nm, ins, ni)
    if n <= 0:
        raise DprtError(f"dprt_flatten_count: invalid mesh / instance description ({n})")
    v, nr, uv, mats = np.zeros((n, 9), np.float32), np.zeros((n, 9), np.float32), np.zeros((n, 6), np.float32), np.zeros(n, np.int32)
    has = C.c_int(0)
    rc = lib.dprt_flatten_instances(md, nm, ins, ni, _ptr(v), _ptr(nr), _ptr(uv), _ptr(mats), C.byref(has))
    del keep
    if rc:
        raise DprtError(f"dprt_flatten_instances failed ({rc})")
    return v, nr, (uv if has.value else None), mats


def spec_texture_sample(rgba, u, v, clamp_v=False):
    """dprt_spec_texture_sample (host only): bilinear look-up of an [h, w, 4] float texture at (u, v) from the kernels' source."""
    t = np.ascontiguousarray(rgba, np.float32)
    uu, vv = np.ascontiguousarray(u, np.float32), np.ascontiguousarray(v, np.float32)
    out = np.zeros((uu.size, 4), np.float32)
    rc = load_library().dprt_spec_texture_sample(_ptr(t), t.shape[1], t.shape[0], _ptr(uu), _ptr(vv), uu.size, int(clamp_v), _ptr(out))
    if rc:
        raise DprtError(f"dprt_spec_texture_sample failed ({rc})")
    return out


def spec_env_lookup(rgba, rotation, dirs):
    """dprt_spec_env_lookup (host only): environment-map radiance of unit directions [n, 3]."""
    t = np.ascontiguousarray(rgba, np.float32)
    d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
    out = np.zeros((d.shape[0], 3), np.float32)
    rc = load_library().dprt_spec_env_lookup(_ptr(t), t.shape[1], t.shape[0], float(rotation), _ptr(d), d.shape[0], _ptr(out))
    if rc:
        raise DprtError(f"dprt_spec_env_lookup failed ({rc})")
    return out


def denoise_params(iterations=None, sigma_color=None, sigma_normal=None, sigma_albedo=None):
    """dprt_denoise_params with the DPRT_DENOISE_DEFAULT_* values for the arguments left at None; None when all are."""
    given = {"iterations": iterations, "sigma_color": sigma_color, "sigma_normal": sigma_normal, "sigma_albedo": sigma_albedo}
    if all(v is None for v in given.values()):
        return None
    return D.DenoiseParams(**{k: D.DENOISE_DEFAULTS[k] if v is None else v for k, v in given.items()})


def _denoise_inputs(color, albedo, normal):
    c = np.ascontiguousarray(color, np.float32)
    if c.ndim != 3 or c.shape[2] != 3:
        raise DprtError(f"denoise: colour must be [H, W, 3], got {c.shape}")
    a, n = np.ascontiguousarray(albedo, np.float32), np.ascontiguousarray(normal, np.float32)
    if a.shape != c.shape or n.shape != c.shape:
        raise DprtError(f"denoise: albedo {a.shape} and normal {n.shape} must match the colour {c.shape}")
    return c, a, n


def spec_denoise(color, albedo, normal, iterations=None, sigma_color=None, sigma_normal=None, sigma_albedo=None):
    """dprt_spec_denoise (host only): the denoiser of dprt_denoise on [H, W, 3] float32 arrays, bit for bit what the GPU
    computes. Parameters left at None take the DPRT_DENOISE_DEFAULT_* values."""
    c, a, n = _denoise_inputs(color, albedo, normal)
    out = np.zeros_like(c)
    p = denoise_params(iterations, sigma_color, sigma_normal, sigma_albedo)
    rc = load_library().dprt_spec_denoise(None if p is None else C.byref(p), c.shape[1], c.shape[0], _ptr(c), _ptr(a), _ptr(n), _ptr(out))
    if rc:
        raise DprtError(f"dprt_spec_denoise failed ({rc})")
    return out


def plan_exchange(gathered_offsets, rank):
    """dprt_plan_exchange: gathered [W, W+1] int32 offset matrix -> (send_count[W], recv_offset[W+1], recv_count[W],
    recv_total, all_local). Host only; this is the plan dprt_exchange executes with ncclSend/ncclRecv."""
    M = np.ascontiguousarray(gathered_offsets, np.int32)
    W = M.shape[0]
    if M.shape != (W, W + 1):
        raise DprtError(f"offset matrix must be [W, W+1], got {M.shape}")
    sc, ro, rc = np.zeros(W, np.int32), np.zeros(W + 1, np.int32), np.zeros(W, np.int32)
    tot, loc = C.c_int64(0), C.c_int(0)
    r = load_library().dprt_plan_exchange(_ptr(M), W, int(rank), _ptr(sc), _ptr(ro), _ptr(rc), C.byref(tot), C.byref(loc))
    if r:
        raise DprtError(f"dprt_plan_exchange failed ({r})")
    return sc, ro, rc, int(tot.value), bool(loc.value)


def plan_exchange_deque(rows, rank):
    """dprt_plan_exchange_deque: rows [W, W+2] int32 (W+1-bucket partition offsets of every rank's travelling paths) ->
    dict(send_count, recv_count, dst_offset, piece=(offL, cL, offR, cR), new_nl, new_active, all_local). Host only."""
    M = np.ascontiguousarray(rows, np.int32)
    W = M.shape[0]
    if M.shape != (W, W + 2):
        raise DprtError(f"offset rows must be [W, W+2], got {M.shape}")
    sc, rc, do, piece = np.zeros(W, np.int32), np.zeros(W, np.int32), np.zeros(W, np.int32), np.zeros(4, np.int32)
    nl, na, loc = C.c_int32(0), C.c_int32(0), C.c_int(0)
    r = load_library().dprt_plan_exchange_deque(_ptr(M), W, int(rank), _ptr(sc), _ptr(rc), _ptr(do), _ptr(piece), C.byref(nl), C.byref(na), C.byref(loc))
    if r:
        raise DprtError(f"dprt_plan_exchange_deque failed ({r})")
    return {"send_count": sc, "recv_count": rc, "dst_offset": do, "piece": tuple(int(x) for x in piece), "new_nl": int(nl.value),
            "new_active": int(na.value), "all_local": bool(loc.value)}


def exchange_host_records(transfer, offsets, rank, world, dist):
    """The exchange protocol of dprt_exchange on HOST record arrays over a torch.distributed process group
    (any backend: this is how the protocol is exercised with gloo on CPU-only machines; the product path moves
    device buffers with NCCL inside libdprt). transfer: bucket-major PATH_DTYPE records of this rank, offsets:
    its transferOffset row [W+1]. Returns (received records in source-rank order, done)."""
    import torch
    row = torch.from_numpy(np.ascontiguousarray(offsets[: world + 1], np.int32).copy())
    rows = [torch.zeros(world + 1, dtype=torch.int32) for _ in range(world)]
    dist.all_gather(rows, row)                                            # MPI_Alltoall(counts), renderer.cpp:1272
    M = torch.stack(rows).numpy()
    sc, ro, rc, total, all_local = plan_exchange(M, rank)
    out = np.zeros(total, D.PATH_DTYPE)
    R = D.PATH_DTYPE.itemsize
    reqs, keep = [], []
    for peer in range(world):                                             # MPI_Alltoallv, renderer.cpp:1280
        if peer == rank:
            continue
        if sc[peer] > 0:
            seg = np.ascontiguousarray(transfer[offsets[peer]:offsets[peer] + sc[peer]]).view(np.uint8).copy()
            t = torch.from_numpy(seg); keep.append(t)
            reqs.append(dist.isend(t, peer))
        if rc[peer] > 0:
            t = torch.zeros(int(rc[peer]) * R, dtype=torch.uint8); keep.append((peer, t))
            reqs.append(dist.irecv(t, peer))
    for q in reqs:
        q.wait()
    for k in keep:
        if isinstance(k, tuple):
            peer, t = k
            out[ro[peer]:ro[peer] + rc[peer]] = t.numpy().view(D.PATH_DTYPE)
    if sc[rank] > 0:
        out[ro[rank]:ro[rank] + sc[rank]] = transfer[offsets[rank]:offsets[rank] + sc[rank]]
    return out, all_local


def partition_host_records_deque(paths, rank, world, n_lower):
    """The W+1-bucket stable partition of the settled-deque migrate loop on HOST records (what partition_kernel<PathOps>
    does on the device with B = W + 1): bucket = targetNode, except that records which stay on this rank and sit at index
    >= n_lower (they came from higher ranks) go to bucket W. Returns (bucket-major records, offsets row [W+2])."""
    p = np.ascontiguousarray(paths, D.PATH_DTYPE)
    t = p["targetNode"].astype(np.int64)
    valid = (p["isValid"] != 0) & (t >= 0) & (t < world)
    key = np.where((t == rank) & (np.arange(p.size) >= n_lower), world, t)
    idx = np.nonzero(valid)[0]
    order = idx[np.argsort(key[idx], kind="stable")]
    row = np.zeros(world + 2, np.int32)
    row[1:] = np.cumsum(np.bincount(key[idx], minlength=world + 1)[: world + 1])
    return p[order], row


def exchange_host_records_deque(buckets, row, rank, world, dist):
    """The settled-deque exchange of dprt_primary_ray_module on HOST record arrays over a torch.distributed process group
    (gloo on CPU-only machines; the product moves device buffers with NCCL): all-gather of the W+2 offsets, plan from
    dprt_plan_exchange_deque, send/recv of the travelling buckets. Returns (new active records: arrivals from lower ranks,
    then from higher ranks; n_lower; first self piece; second self piece; done)."""
    import torch
    rows = [torch.zeros(world + 2, dtype=torch.int32) for _ in range(world)]
    dist.all_gather(rows, torch.from_numpy(np.ascontiguousarray(row, np.int32).copy()))
    plan = plan_exchange_deque(torch.stack(rows).numpy(), rank)
    sc, rc = plan["send_count"], plan["recv_count"]
    R = D.PATH_DTYPE.itemsize
    reqs, keep, got = [], [], {}
    for peer in range(world):
        if peer == rank:
            continue
        if sc[peer] > 0:
            t = torch.from_numpy(np.ascontiguousarray(buckets[row[peer]:row[peer] + sc[peer]]).view(np.uint8).copy()); keep.append(t)
            reqs.append(dist.isend(t, peer))
        if rc[peer] > 0:
            t = torch.zeros(int(rc[peer]) * R, dtype=torch.uint8); got[peer] = t
            reqs.append(dist.irecv(t, peer))
    for q in reqs:
        q.wait()
    parts = [got[peer].numpy().view(D.PATH_DTYPE) for peer in range(world) if peer in got]     # source-rank order: lower ranks first
    active = np.concatenate(parts) if parts else np.zeros(0, D.PATH_DTYPE)
    oL, cL, oR, cR = plan["piece"]
    return active, plan["new_nl"], buckets[oL:oL + cL], buckets[oR:oR + cR], plan["all_local"]


class Renderer:
    """One rank of the data-parallel renderer (one GPU, one scene-chunk owner)."""

    def __init__(self, cfg, rank=0, world=1, device=0, nccl_unique_id=None, parent=None):
        """parent: another Renderer of the same rank whose NCCL communicator this one borrows (dprt_create_shared)."""
        self.lib = load_library()
        self.cfg = cfg
        self.N = cfg.width * cfg.height
        h = C.c_void_p()
        if parent is not None:
            rank, world = parent.rank, parent.world
            rc = self.lib.dprt_create_shared(C.byref(cfg), parent.h, C.byref(h))
        else:
            idbuf = None
            if nccl_unique_id is not None:
                idbuf = C.create_string_buffer(bytes(nccl_unique_id), 128)
            rc = self.lib.dprt_create(C.byref(cfg), rank, world, device, idbuf, C.byref(h))
        self.rank, self.world = rank, world
        if rc:
            raise DprtError(f"dprt_create failed ({rc}): {self.lib.dprt_last_error(None).decode()}")
        self.h = h

    # -- peer-memory exchange wiring for hosts without NCCL (dprt.h: export -> all-gather -> connect -> agree -> enable)
    @property
    def p2p_enabled(self):
        return bool(self.lib.dprt_p2p_enabled(self.h))

    def p2p_export(self):
        buf = C.create_string_buffer(D.P2P_HANDLE_BYTES)
        self._ck(self.lib.dprt_p2p_export(self.h, buf), "dprt_p2p_export")
        return bytes(buf.raw)

    def p2p_connect(self, all_handles):
        blob = b"".join(all_handles)
        ok = C.c_int(0)
        self._ck(self.lib.dprt_p2p_connect(self.h, blob, C.byref(ok)), "dprt_p2p_connect")
        return bool(ok.value)

    def p2p_enable(self, enable):
        self._ck(self.lib.dprt_p2p_enable(self.h, 1 if enable else 0), "dprt_p2p_enable")

    # -- plumbing ---------------------------------------------------------------------------------
    def _ck(self, rc, what):
        if rc:
            raise DprtError(f"{what} failed ({rc}): {self.lib.dprt_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.dprt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        self._ck(self.lib.dprt_synchronize(self.h), "dprt_synchronize")

    def stats(self):
        s = D.Stats()
        self._ck(self.lib.dprt_get_stats(self.h, C.byref(s)), "dprt_get_stats")
        return s.as_dict()

    def reset_stats(self):
        self._ck(self.lib.dprt_reset_stats(self.h), "dprt_reset_stats")

    # -- scene ------------------------------------------------------------------------------------
    def upload_chunk(self, scene_index, desc, verts9, normals9, mat_ids):
        v = np.ascontiguousarray(verts9, np.float32).reshape(-1, 9)
        n = None if normals9 is None else np.ascontiguousarray(normals9, np.float32).reshape(-1, 9)
        m = None if mat_ids is None else np.ascontiguousarray(mat_ids, np.int32)
        self._ck(self.lib.dprt_upload_chunk(self.h, scene_index, C.byref(desc), _ptr(v), _ptr(n), _ptr(m), v.shape[0]),
                 "dprt_upload_chunk")

    def upload_chunk_uv(self, scene_index, desc, verts9, normals9, uv6, mat_ids):
        """dprt_upload_chunk_uv: flat triangles with per-corner texture coordinates (uv6 [n,6] or None)."""
        v = np.ascontiguousarray(verts9, np.float32).reshape(-1, 9)
        n = None if normals9 is None else np.ascontiguousarray(normals9, np.float32).reshape(-1, 9)
        u = None if uv6 is None else np.ascontiguousarray(uv6, np.float32).reshape(-1, 6)
        m = None if mat_ids is None else np.ascontiguousarray(mat_ids, np.int32)
        self._ck(self.lib.dprt_upload_chunk_uv(self.h, scene_index, C.byref(desc), _ptr(v), _ptr(n), _ptr(u), _ptr(m), v.shape[0]),
                 "dprt_upload_chunk_uv")

    def refit_chunk(self, scene_index, verts9, normals9=None):
        """dprt_refit_chunk: moved corners (and normals, when the chunk has them) of local chunk scene_index, same triangles.
        Instanced objects: flatten_instances with the moved instances, then this."""
        v = np.ascontiguousarray(verts9, np.float32).reshape(-1, 9)
        n = None if normals9 is None else np.ascontiguousarray(normals9, np.float32).reshape(-1, 9)
        self._ck(self.lib.dprt_refit_chunk(self.h, scene_index, _ptr(v), _ptr(n), v.shape[0]), "dprt_refit_chunk")

    def refit_chunk_device(self, scene_index, verts9_dev, normals9_dev, ntris):
        """dprt_refit_chunk_device on device buffers of ntris * 9 floats (normals9_dev may be None)."""
        self._ck(self.lib.dprt_refit_chunk_device(self.h, scene_index, verts9_dev, normals9_dev, ntris), "dprt_refit_chunk_device")

    def chunk_bvh8(self, scene_index):
        """dprt_chunk_bvh8_copy: the device BVH8 of local chunk scene_index -> (nodes[NODE_DTYPE], tris[TRI_DTYPE])."""
        nn, nt = C.c_int64(), C.c_int64()
        self._ck(self.lib.dprt_chunk_bvh8_copy(self.h, scene_index, C.byref(nn), C.byref(nt), None, None), "dprt_chunk_bvh8_copy")
        nodes, tris = np.zeros(nn.value, D.NODE_DTYPE), np.zeros(nt.value, D.TRI_DTYPE)
        self._ck(self.lib.dprt_chunk_bvh8_copy(self.h, scene_index, None, None, _ptr(nodes), _ptr(tris)), "dprt_chunk_bvh8_copy")
        return nodes, tris

    def upload_instanced_chunk(self, scene_index, desc, meshes, instances):
        """dprt_upload_instanced_chunk: indexed meshes (ctypes_defs.pack_meshes dicts) placed by (mesh, 3x4 matrix) instances."""
        md, nm, ins, ni, keep = D.pack_meshes(meshes, instances)
        self._ck(self.lib.dprt_upload_instanced_chunk(self.h, scene_index, C.byref(desc), md, nm, ins, ni), "dprt_upload_instanced_chunk")
        del keep

    def set_texture(self, texture_index, rgba):
        """params.albedoTextures[texture_index]: [h, w, 4] float RGBA (alpha = opacity), or None to remove it."""
        if rgba is None:
            self._ck(self.lib.dprt_set_texture(self.h, texture_index, None, 0, 0), "dprt_set_texture")
            return
        t = np.ascontiguousarray(rgba, np.float32)
        assert t.ndim == 3 and t.shape[2] == 4
        self._ck(self.lib.dprt_set_texture(self.h, texture_index, _ptr(t), t.shape[1], t.shape[0]), "dprt_set_texture")

    def set_material_textures(self, texture_index):
        t = np.ascontiguousarray(texture_index, np.int32)
        self._ck(self.lib.dprt_set_material_textures(self.h, _ptr(t), t.size), "dprt_set_material_textures")

    def set_env_map(self, rgba, rotation_offset=0.0):
        """params.envLightTexture: [h, w, 4] float lat-long map, or None for the analytic sky."""
        if rgba is None:
            self._ck(self.lib.dprt_set_env_map(self.h, None, 0, 0, 0.0), "dprt_set_env_map")
            return
        t = np.ascontiguousarray(rgba, np.float32)
        assert t.ndim == 3 and t.shape[2] == 4
        self._ck(self.lib.dprt_set_env_map(self.h, _ptr(t), t.shape[1], t.shape[0], float(rotation_offset)), "dprt_set_env_map")

    def upload_proxy(self, scene_index, desc, vis_blob=None, depth_blob=None):
        vb = None if vis_blob is None else np.frombuffer(vis_blob, np.uint8)
        db = None if depth_blob is None else np.frombuffer(depth_blob, np.uint8)
        self._ck(self.lib.dprt_upload_proxy(self.h, scene_index, C.byref(desc), _ptr(vb), 0 if vb is None else vb.size,
                                            _ptr(db), 0 if db is None else db.size), "dprt_upload_proxy")

    def set_materials(self, mats):
        m = np.ascontiguousarray(mats, D.MATERIAL_DTYPE)
        self._ck(self.lib.dprt_set_materials(self.h, _ptr(m), m.size), "dprt_set_materials")

    def set_lights(self, lights):
        l = np.ascontiguousarray(lights, D.LIGHT_DTYPE)
        self._ck(self.lib.dprt_set_lights(self.h, _ptr(l), l.size), "dprt_set_lights")

    def set_camera(self, cam):
        self._ck(self.lib.dprt_set_camera(self.h, C.byref(cam)), "dprt_set_camera")

    # -- stages (reference call sites in include/dprt.h) ----------------------------------------------
    def reset_frame(self):
        self._ck(self.lib.dprt_reset_frame(self.h), "dprt_reset_frame")

    def begin_sample(self, sample):
        self._ck(self.lib.dprt_begin_sample(self.h, sample), "dprt_begin_sample")

    def path_gen(self):
        self._ck(self.lib.dprt_path_gen(self.h), "dprt_path_gen")

    def traverse(self):
        self._ck(self.lib.dprt_traverse(self.h), "dprt_traverse")

    def partition(self):
        self._ck(self.lib.dprt_partition(self.h), "dprt_partition")

    def exchange(self):
        done = C.c_int(0)
        self._ck(self.lib.dprt_exchange(self.h, C.byref(done)), "dprt_exchange")
        return bool(done.value)

    def shade(self):
        self._ck(self.lib.dprt_shade(self.h), "dprt_shade")

    def reset_nn(self):
        self._ck(self.lib.dprt_reset_nn(self.h), "dprt_reset_nn")

    def shadow_trace(self):
        self._ck(self.lib.dprt_shadow_trace(self.h), "dprt_shadow_trace")

    def secondary_trace(self):
        self._ck(self.lib.dprt_secondary_trace(self.h), "dprt_secondary_trace")

    def bucket_queries(self, which, inside_only):
        total = C.c_int(0)
        self._ck(self.lib.dprt_bucket_queries(self.h, which, int(inside_only), C.byref(total)), "dprt_bucket_queries")
        return int(total.value)

    def proxy_infer(self, kind, pred_offset=0):
        self._ck(self.lib.dprt_proxy_infer(self.h, kind, pred_offset), "dprt_proxy_infer")

    def frame_buffer_update(self):
        self._ck(self.lib.dprt_frame_buffer_update(self.h), "dprt_frame_buffer_update")

    def depth_buffer_update(self):
        self._ck(self.lib.dprt_depth_buffer_update(self.h), "dprt_depth_buffer_update")

    def target_node_update(self):
        self._ck(self.lib.dprt_target_node_update(self.h), "dprt_target_node_update")

    def primary_ray_module(self):
        self._ck(self.lib.dprt_primary_ray_module(self.h), "dprt_primary_ray_module")

    def shadow_ray_module(self):
        self._ck(self.lib.dprt_shadow_ray_module(self.h), "dprt_shadow_ray_module")

    def secondary_ray_module(self):
        self._ck(self.lib.dprt_secondary_ray_module(self.h), "dprt_secondary_ray_module")

    def run_sample(self, sample):
        self._ck(self.lib.dprt_render_sample(self.h, sample), "dprt_render_sample")

    def reduce_image(self, root=0):
        out = np.zeros((self.cfg.height, self.cfg.width, 3), np.float32) if self.rank == root else None
        self._ck(self.lib.dprt_reduce_image(self.h, root, _ptr(out)), "dprt_reduce_image")
        return out

    def enable_aov(self, enable=True):
        """dprt_enable_aov: accumulate the first-hit albedo and shading normal of every sample (the guide buffers a denoiser
        takes beside the colour; dprt.h has the rule). Off by default; the first enable allocates the buffer."""
        self._ck(self.lib.dprt_enable_aov(self.h, int(enable)), "dprt_enable_aov")

    def reduce_aov(self, root=0):
        """dprt_reduce_aov (collective): (albedo, normal), each [H, W, 3] float32 = sum / spp over the ranks, on root; None
        elsewhere. The averaged normal is not renormalised."""
        shape = (self.cfg.height, self.cfg.width, 3)
        a, n = (np.zeros(shape, np.float32), np.zeros(shape, np.float32)) if self.rank == root else (None, None)
        self._ck(self.lib.dprt_reduce_aov(self.h, root, _ptr(a), _ptr(n)), "dprt_reduce_aov")
        return (a, n) if self.rank == root else None

    def denoise(self, color, albedo, normal, iterations=None, sigma_color=None, sigma_normal=None, sigma_albedo=None):
        """dprt_denoise on this context's GPU: the [H, W, 3] colour filtered with its albedo and normal guides (e.g. reduce_image
        and reduce_aov of the same frame; any size). Returns [H, W, 3] float32. Parameters left at None take the defaults."""
        c, a, n = _denoise_inputs(color, albedo, normal)
        out = np.zeros_like(c)
        p = denoise_params(iterations, sigma_color, sigma_normal, sigma_albedo)
        self._ck(self.lib.dprt_denoise(self.h, None if p is None else C.byref(p), c.shape[1], c.shape[0], _ptr(c), _ptr(a), _ptr(n),
                                       _ptr(out)), "dprt_denoise")
        return out

    def denoise_device(self, width, height, color_dev, albedo_dev, normal_dev, out_dev, params=None):
        """dprt_denoise_device on device buffers of 3 * width * height floats (params: D.DenoiseParams or None)."""
        self._ck(self.lib.dprt_denoise_device(self.h, None if params is None else C.byref(params), width, height, color_dev, albedo_dev,
                                              normal_dev, out_dev), "dprt_denoise_device")

    def launch(self):
        """Renderer::launch (renderer.cpp:1576): reset, spp x runSample, average + reduce to rank 0."""
        self.reset_frame()
        for s in range(self.cfg.spp):
            self.run_sample(s)
        return self.reduce_image(0)

    # -- state access -----------------------------------------------------------------------------------
    @property
    def path_size(self):
        a, b = C.c_int(), C.c_int()
        self._ck(self.lib.dprt_get_path_size(self.h, C.byref(a), C.byref(b)), "dprt_get_path_size")
        return int(a.value)

    @property
    def shadow_path_size(self):
        a, b = C.c_int(), C.c_int()
        self._ck(self.lib.dprt_get_path_size(self.h, C.byref(a), C.byref(b)), "dprt_get_path_size")
        return int(b.value)

    def set_path_size(self, n):
        self._ck(self.lib.dprt_set_path_size(self.h, int(n)), "dprt_set_path_size")

    def download(self, buf, count=None, offset=0):
        dt = D.BUFFER_DTYPES[buf]
        if count is None:
            nbytes = C.c_size_t()
            self._ck(self.lib.dprt_buffer_bytes(self.h, buf, C.byref(nbytes)), "dprt_buffer_bytes")
            count = nbytes.value // dt.itemsize - offset
        out = np.zeros(count, dt)
        if count:
            self._ck(self.lib.dprt_download(self.h, buf, offset * dt.itemsize, _ptr(out), out.nbytes), "dprt_download")
        return out

    def upload(self, buf, array, offset=0):
        dt = D.BUFFER_DTYPES[buf]
        a = np.ascontiguousarray(array, dt)
        if a.size:
            self._ck(self.lib.dprt_upload(self.h, buf, offset * dt.itemsize, _ptr(a), a.nbytes), "dprt_upload")

    def enable_hit_prim(self, enable=True):
        self._ck(self.lib.dprt_enable_hit_prim(self.h, int(enable)), "dprt_enable_hit_prim")

    # -- standalone operators ------------------------------------------------------------------------------
    def trace_closest(self, rays):
        r = np.ascontiguousarray(rays, D.RAY_DTYPE)
        hits = np.zeros(r.size, D.HIT_DTYPE)
        self._ck(self.lib.dprt_trace_closest(self.h, _ptr(r), r.size, _ptr(hits)), "dprt_trace_closest")
        return hits

    def gen_train_data(self, scene_index, rays):
        """Vis pipeline (vis_ray_kernel.cu:98-161): (features [n,5] f32, labels [n] f32; 1.0 = miss) for a local object."""
        r = np.ascontiguousarray(rays, D.RAY_DTYPE)
        feat, lab = np.zeros((r.size, 5), np.float32), np.zeros(r.size, np.float32)
        self._ck(self.lib.dprt_gen_train_data(self.h, scene_index, _ptr(r), r.size, _ptr(feat), _ptr(lab)), "dprt_gen_train_data")
        return feat, lab

    def gen_precom_data(self, scene_index, rays):
        """Precom pipeline (precom_ray_kernel.cu:193-299): (features [n,5] at the proxy-AABB hit, labels [n] = depth of the
        geometry behind the AABB surface / maxLength, 1.0 = geometry missed; valid [n] u8 = the ray met the AABB)."""
        r = np.ascontiguousarray(rays, D.RAY_DTYPE)
        feat, lab, valid = np.zeros((r.size, 5), np.float32), np.zeros(r.size, np.float32), np.zeros(r.size, np.uint8)
        self._ck(self.lib.dprt_gen_precom_data(self.h, scene_index, _ptr(r), r.size, _ptr(feat), _ptr(lab), _ptr(valid)), "dprt_gen_precom_data")
        return feat, lab, valid

    def mlp_infer(self, scene_index, kind, x_half):
        x = np.ascontiguousarray(x_half, np.uint16).reshape(-1, 5)
        y = np.zeros(x.shape[0], np.uint16)
        self._ck(self.lib.dprt_mlp_infer(self.h, scene_index, kind, _ptr(x), x.shape[0], _ptr(y)), "dprt_mlp_infer")
        return y

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.lib.dprt_device_alloc(self.h, nbytes, C.byref(p)), "dprt_device_alloc")
        return p

    def device_free(self, p):
        self._ck(self.lib.dprt_device_free(self.h, p), "dprt_device_free")

    def h2d(self, dev, array):
        a = np.ascontiguousarray(array)
        self._ck(self.lib.dprt_memcpy_h2d(self.h, dev, _ptr(a), a.nbytes), "dprt_memcpy_h2d")

    def d2h(self, array, dev):
        self._ck(self.lib.dprt_memcpy_d2h(self.h, _ptr(array), dev, array.nbytes), "dprt_memcpy_d2h")

    def trace_closest_device(self, rays_dev, n, hits_dev):
        self._ck(self.lib.dprt_trace_closest_device(self.h, rays_dev, n, hits_dev), "dprt_trace_closest_device")

    def mlp_infer_device(self, scene_index, kind, x_dev, n, y_dev):
        self._ck(self.lib.dprt_mlp_infer_device(self.h, scene_index, kind, x_dev, n, y_dev), "dprt_mlp_infer_device")

    def timer_start(self):
        self._ck(self.lib.dprt_timer_start(self.h), "dprt_timer_start")

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self.lib.dprt_timer_stop(self.h, C.byref(ms)), "dprt_timer_stop")
        return float(ms.value)

    def flush_l2(self):
        self._ck(self.lib.dprt_flush_l2(self.h), "dprt_flush_l2")

    def stage_profile(self, enable=True):
        self._ck(self.lib.dprt_stage_profile(self.h, int(enable)), "dprt_stage_profile")

    def stage_times(self):
        """{stage name: (device ms, launches)} accumulated since the last reset_stats()."""
        ms = np.zeros(D.STAGE_COUNT, np.float64)
        ln = np.zeros(D.STAGE_COUNT, np.int64)
        self._ck(self.lib.dprt_get_stage_times(self.h, _ptr(ms), _ptr(ln)), "dprt_get_stage_times")
        return {D.STAGE_NAMES[i]: (float(ms[i]), int(ln[i])) for i in range(D.STAGE_COUNT)}

    def enable_counters(self, enable=True):
        self._ck(self.lib.dprt_enable_counters(self.h, int(enable)), "dprt_enable_counters")

    def counters(self):
        """{stage name: (bvh8 nodes visited, triangles tested)} of the instrumented traversal variants."""
        c = np.zeros(2 * D.STAGE_COUNT, np.uint64)
        self._ck(self.lib.dprt_get_counters(self.h, _ptr(c)), "dprt_get_counters")
        return {D.STAGE_NAMES[i]: (int(c[2 * i]), int(c[2 * i + 1])) for i in range(D.STAGE_COUNT)}


class SamplesInFlight:
    """K samples of a frame in flight on one rank (dprt.h "samples in flight"): K contexts sharing one uploaded scene and
    the NCCL communicator, one host thread each; context j renders samples j, j + K, ... The frame is the primary's.
    With W > 1 every context brings up to two streams that may hold a waiting kernel: the process needs
    CUDA_DEVICE_MAX_CONNECTIONS >= 2 K in its environment before CUDA initialises (libdprt refuses otherwise)."""

    def __init__(self, primary, k=2):
        self.primary = primary
        self.ctxs = [primary]
        if primary.world > 1 and not primary.p2p_enabled:
            k = 1        # the NCCL fallback exchange issues collectives from the sampling thread: one context per communicator
        for _ in range(max(1, int(k)) - 1):
            R = Renderer(primary.cfg, parent=primary)
            R._ck(R.lib.dprt_adopt_scene(R.h, primary.h), "dprt_adopt_scene")
            self.ctxs.append(R)

    def adopt(self):
        """Call again after the primary's scene, lights or camera changed."""
        for R in self.ctxs[1:]:
            R._ck(R.lib.dprt_adopt_scene(R.h, self.primary.h), "dprt_adopt_scene")

    def reset_frame(self):
        for R in self.ctxs:
            R.reset_frame()

    def run_samples(self, first, count):
        """Samples first .. first + count - 1, dealt round-robin to the contexts; returns when all are enqueued and the
        host side of every migrate loop is through (device work may still be running: synchronize / accumulate next)."""
        import threading
        k = len(self.ctxs)
        errs = []

        def work(j):
            try:
                for s in range(first + j, first + count, k):
                    self.ctxs[j].run_sample(s)
            except Exception as e:       # noqa: BLE001 -- re-raised on the calling thread
                errs.append(e)
        th = [threading.Thread(target=work, args=(j,)) for j in range(1, k)]
        for t in th:
            t.start()
        work(0)
        for t in th:
            t.join()
        if errs:
            raise errs[0]

    def accumulate(self):
        """Adds every other context's sums into the primary's: colour, and the AOVs when they are on."""
        for R in self.ctxs[1:]:
            self.primary._ck(self.primary.lib.dprt_accumulate_from(self.primary.h, R.h), "dprt_accumulate_from")

    def enable_aov(self, enable=True):
        for R in self.ctxs:
            R.enable_aov(enable)

    def reduce_aov(self, root=0):
        """The frame's AOVs after launch() (whose accumulate() brought every context's sums to the primary)."""
        return self.primary.reduce_aov(root)

    def launch(self):
        """Renderer.launch with the samples in flight: reset, spp samples, accumulate, average + reduce."""
        self.reset_frame()
        self.run_samples(0, self.primary.cfg.spp)
        self.accumulate()
        return self.primary.reduce_image(0)

    def stats(self):
        out = None
        for R in self.ctxs:
            st = R.stats()
            out = st if out is None else {k: out[k] + st[k] for k in out}
        return out

    def close(self):
        for R in self.ctxs[1:]:
            R.close()
        self.ctxs = [self.primary]


class RankGroup:
    """W contexts driven by one thread (dprt_*_group): multi-chunk runs on fewer GPUs than ranks."""

    def __init__(self, renderers):
        self.rs = list(renderers)
        self.lib = self.rs[0].lib
        self.arr = (C.c_void_p * len(self.rs))(*[r.h for r in self.rs])

    def exchange(self):
        done = C.c_int(0)
        self.rs[0]._ck(self.lib.dprt_exchange_group(self.arr, len(self.rs), C.byref(done)), "dprt_exchange_group")
        return bool(done.value)

    def run_sample(self, sample):
        self.rs[0]._ck(self.lib.dprt_render_sample_group(self.arr, len(self.rs), sample), "dprt_render_sample_group")

    def reduce_image(self, root=0):
        cfg = self.rs[0].cfg
        out = np.zeros((cfg.height, cfg.width, 3), np.float32)
        self.rs[0]._ck(self.lib.dprt_reduce_image_group(self.arr, len(self.rs), root, _ptr(out)), "dprt_reduce_image_group")
        return out

    def enable_aov(self, enable=True):
        for r in self.rs:
            r.enable_aov(enable)

    def reduce_aov(self, root=0):
        """(albedo, normal), each [H, W, 3]: per rank sum / spp, summed over the ranks in rank order."""
        cfg = self.rs[0].cfg
        a, n = np.zeros((cfg.height, cfg.width, 3), np.float32), np.zeros((cfg.height, cfg.width, 3), np.float32)
        self.rs[0]._ck(self.lib.dprt_reduce_aov_group(self.arr, len(self.rs), root, _ptr(a), _ptr(n)), "dprt_reduce_aov_group")
        return a, n

    def launch(self):
        for r in self.rs:
            r.reset_frame()
        for s in range(self.rs[0].cfg.spp):
            self.run_sample(s)
        return self.reduce_image(0)
