"""Multi-process, multi-GPU check of the first-hit guide buffers (dprt_reduce_aov over NCCL).

Launched by tests/test_gpu_aov.py (or by hand) as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P tests/mgpu_aov_check.py
One process per GPU. Every rank renders its share with AOVs on and compares its own AOV buffer with the CPU reference's W-rank
world (the oracle with the AOV rule, tests/aov_reference.cpp) bit for bit; rank 0 compares the AOVs that ncclReduce
brought to it with the reference's rank-ordered sum: by value at W = 2 (a two-term sum does not depend on the order; the
reference's starts from +0, so a -0 comes back as +0), else at 1e-6 relative.
"""
import importlib
import os
import sys

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist
    rank, W, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")
    D = dprt.ctypes_defs
    from aov_reference import AovWorld
    from helpers import assert_bits_equal

    t = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        t = torch.tensor(list(dprt.get_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(t, 0)
    uid = bytes(t.cpu().tolist())

    w, h = 128, 72
    chunks, mats, lights = dprt.scene.make_scene(W, 6000, water_frac=0.03)
    cfg = dprt.make_config(w, h, spp=2, bounces=2, scene_size=W, proxy_mode=0, path_gen_mode=1)
    cam = dprt.scene.default_camera(w, h)
    R = dprt.Renderer(cfg, rank=rank, world=W, device=local, nccl_unique_id=uid)
    world = AovWorld(cfg, W)
    for c in chunks:
        world.add_object(c.index, c.desc(False), c.verts, c.normals, c.mats)
        if c.node_id == rank:
            R.upload_chunk(c.index, c.desc(False), c.verts, c.normals, c.mats)
        else:
            R.upload_proxy(c.index, c.desc(True), None, None)
    for X in (R, world):
        X.set_materials(mats); X.set_lights(lights); X.set_camera(cam); X.enable_aov()

    R.launch()
    got = R.reduce_aov(0)
    world.launch()
    N = w * h
    assert_bits_equal(R.download(D.BUF_AOV, 6 * N), world.aov_buffer(rank), f"rank {rank} AOV buffer")
    if rank == 0:
        for g, o, what in zip(got, world.aov(), ("albedo", "normal")):
            assert np.abs(o).max() > 0, what
            if W == 2:
                assert np.array_equal(g, o), f"2-rank reduced {what} differs"
            else:
                err = np.abs(g - o).max() / max(1e-30, float(np.abs(o).max()))
                assert err <= 1e-6, f"reduced {what} differs: {err}"
        print(f"MGPU_AOV_CHECK_OK world={W}", flush=True)
    else:
        assert got is None
    R.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
