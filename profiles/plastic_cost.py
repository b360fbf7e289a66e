"""Cost of the glossy plastic (bsdfType 3, DESIGN.md 3.13) on the benchmark workload: conductor_cost.py's windows (bench.py's
one-GPU scene, 1920x1080, 1 M triangles, 4 bounces) with its 16 materials all Lambertian, all plastics at roughness 0.3, and
mixed (the odd materials plastics at 0.3), alternating in one process. The device name and power limit are read in the same
process.

    python profiles/plastic_cost.py [--steps 40] [--warmup 4] [--rounds 3] [--out DIR]     (--out: DIR/plastic_cost.jsonl)
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import conductor_cost  # noqa: E402

if __name__ == "__main__":
    conductor_cost.main(bsdf=3, name="plastic")
