"""Generates the committed golden fixtures from the REFERENCE itself (run in the build container only).

  rng_kat.json   tea<4>/rnd known answers from /root/reference/optix/random.hpp compiled into
                 oracle/_ref/librefrng.so (make -C oracle ref REF=<reference tree>)
  mlp_golden.npz forward outputs of /root/reference/trainingcode/module.py classes on PyTorch-CPU fp32 under
                 torch.manual_seed(19990201) (the reference's seed, trainingcode/main.py:76), for fp16-rounded
                 inputs x ~ U[0,1)^5 from torch.Generator().manual_seed(0); plus a check that
                 proxy.make_proxy() re-creates the very same parameters from the same seed, so the weights
                 themselves need not be committed.

Nothing under tests/ reads /root/reference at test time; only this script does.
"""
import importlib
import importlib.util
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"

from oracle import oracle as O  # noqa: E402

dprt = importlib.import_module("pg2024-data-parallel-ray-tracing_b200")


def rng_kat():
    R = O.ref_rng()
    assert R is not None, "run `make -C oracle ref REF=<reference tree>` first"
    cases = [(0, 0), (1, 0), (1920, 1), (2073599, 15), (123456789, 987654321), (0xFFFFFFFF, 0xFFFFFFFF), (8294399, 63)]
    out = []
    for a, b in cases:
        seed = int(R.ref_tea4(a, b))
        seq = np.zeros(8, np.float32)
        R.ref_rnd_sequence(seed, 8, seq.ctypes.data)
        out.append({"val0": a, "val1": b, "tea4": seed, "rnd": [float(v) for v in seq], "rnd_hex": [int(v) for v in seq.view(np.uint32)]})
    json.dump({"source": "optix/random.hpp via oracle/_ref/librefrng.so", "cases": out}, open(os.path.join(HERE, "rng_kat.json"), "w"), indent=1)
    print("rng_kat.json", len(out), "cases")


def mlp_golden():
    spec = importlib.util.spec_from_file_location("ref_module", os.path.join(REF, "trainingcode", "module.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    g = torch.Generator().manual_seed(0)
    x = torch.rand(512, 5, generator=g).half().float()          # the renderer feeds fp16 features
    out = {"x_f16": x.half().numpy().view(np.uint16)}
    for name, width, nres, sig in (("NeuralVisNetworkWith4Res256SingleOutput", 256, 4, False), ("NeuralVisNetworkWith6Res256SingleOutput", 256, 6, False),
                                   ("NeuralVisNetworkWith4Res128SingleOutput", 128, 4, False), ("NeuralVisNetworkWith4Res128SingleOutputSigmoid", 128, 4, True),
                                   ("NeuralVisNetworkWith4Res256SingleOutputSigmoid", 256, 4, True)):
        torch.manual_seed(19990201)
        m_ref = getattr(ref, name)().eval()
        torch.manual_seed(19990201)
        m_own = dprt.proxy.make_proxy(width, nres, sigmoid=sig).eval()
        sd_ref, sd_own = m_ref.state_dict(), m_own.state_dict()
        assert list(sd_ref.keys()) == list(sd_own.keys()), "parameter names differ from the reference"
        for k in sd_ref:
            assert torch.equal(sd_ref[k], sd_own[k]), k
        with torch.no_grad():
            y = m_ref(x)
            assert torch.equal(y, m_own(x))
        tag = f"{nres}res{width}" + ("_sigmoid" if sig else "")
        out[f"y_{tag}"] = y.numpy().reshape(-1).astype(np.float32)
        if sig:
            print(name, "y range", float(y.min()), float(y.max()))
            continue
        # decision-test variant: outputs spread around 0.5 (same transform applied to both)
        dprt.proxy.spread_output_(m_own, gain=3.0, seed=1)
        m_ref.load_state_dict(m_own.state_dict())
        with torch.no_grad():
            ys = m_ref(x)
        out[f"y_{tag}_spread"] = ys.numpy().reshape(-1).astype(np.float32)
        print(name, "y range", float(y.min()), float(y.max()), "spread range", float(ys.min()), float(ys.max()))
    np.savez_compressed(os.path.join(HERE, "mlp_golden.npz"), **out)
    print("mlp_golden.npz written")


if __name__ == "__main__":
    rng_kat()
    mlp_golden()
