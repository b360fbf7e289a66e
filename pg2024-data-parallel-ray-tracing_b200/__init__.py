"""dprt -- B200-native per-sample / per-bounce inner loop of the PG2024 data-parallel ray tracer.

The product is ``libdprt.so`` (hand-written sm_100a CUDA behind the C ABI of ``include/dprt.h``); this package
holds its sources (``csrc/``), the ctypes binding that mirrors the reference's host interface (``host.py``),
the synthetic-scene generators of the benchmark configs (``scene.py``) and the PyTorch proxy definition +
weight export of the training side (``proxy.py``), and the proxy training pipeline around ``dprt_gen_train_data``
(``proxy_train.py``). Import it as::

    import importlib; dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")

(or ``import dprt`` via the alias module at the repository root).
"""
from . import ctypes_defs, host, proxy, proxy_train, real_scene, scene  # noqa: F401
from .ctypes_defs import make_camera, make_config, make_object_desc  # noqa: F401
from .host import (DprtError, RankGroup, Renderer, SamplesInFlight, build_bvh8, flatten_instances, get_unique_id, load_library,  # noqa: F401
                   plan_exchange, plan_exchange_deque, spec_bvh8_build_gpu, spec_bvh8_refit, spec_conductor_eval, spec_conductor_sample, spec_denoise,
                   spec_env_lookup, spec_plastic_eval, spec_plastic_sample, spec_texture_sample)

__all__ = ["ctypes_defs", "host", "proxy", "proxy_train", "real_scene", "scene", "make_camera", "make_config", "make_object_desc", "DprtError",
           "RankGroup", "Renderer", "SamplesInFlight", "build_bvh8", "flatten_instances", "get_unique_id", "load_library", "spec_bvh8_build_gpu", "spec_bvh8_refit", "spec_conductor_eval", "spec_conductor_sample", "spec_denoise",
           "spec_env_lookup", "spec_plastic_eval", "spec_plastic_sample", "spec_texture_sample"]
