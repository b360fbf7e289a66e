"""The host flatten of instanced, indexed meshes (dprt_flatten_instances) pinned bit for bit. Its instance arithmetic lives in
csrc/instance_xform.cuh, shared with the device flatten of dprt_build_instanced_chunk / dprt_update_instances; the digests
below were recorded from the host flatten before that arithmetic moved into the shared header. No GPU needed."""
import numpy as np
import pytest

from helpers import dprt
from instance_cases import CASES, flatten_digest

PINNED = {
    "garden": "d62eba8d90c72f76e511c7a74c405364c5742634a7c6693fcd2be960f2d9c825",
    "mirrored": "823be8e7006528d919973ae592e31bc4d81c35c7898447e3e0853239a96079ee",
    "mixed_uv": "ab2bbf761edeb509ec67826e45ece23d1d34381ea6ac6143b77eea3e94baa134",
    "zero_tris": "35e34c4d7091c7ec381fb58210e0f634e7c6626720ded9596f8bc5a004712e18",
    "one_tri": "5fc3093bf7cb7378ccb6d7c9f7632d0605723b499f51530012f664d26512984e",
}


@pytest.mark.parametrize("case", sorted(PINNED))
def test_flatten_output_is_pinned(case):
    meshes, instances = CASES[case]()
    assert flatten_digest(*dprt.flatten_instances(meshes, instances)) == PINNED[case]


def test_cases_cover_what_they_name():
    meshes, inst = CASES["mirrored"]()
    assert all(np.linalg.det(np.asarray(M, np.float64)[:, :3]) < 0 for _, M in inst)
    meshes, _ = CASES["mixed_uv"]()
    assert {m["texcoords"] is None for m in meshes} == {True, False}
    meshes, inst = CASES["zero_tris"]()
    empty = [len(meshes[mi]["indices"]) == 0 for mi, _ in inst]
    assert empty[0] and empty[-1] and any(not e for e in empty)
    meshes, _ = CASES["one_tri"]()
    assert all(len(m["indices"]) == 1 for m in meshes)


def test_singular_transform_of_an_empty_instance_is_rejected():
    """A zero-triangle instance contributes no triangle, but its transform is still checked (as the device flatten does)."""
    meshes, inst = CASES["zero_tris"]()
    dprt.flatten_instances(meshes, inst)
    bad = list(inst)
    bad[0] = (bad[0][0], np.zeros((3, 4), np.float32))
    with pytest.raises(dprt.DprtError):
        dprt.flatten_instances(meshes, bad)
    nonfinite = list(inst)
    M = np.array(inst[0][1], np.float32)
    M[1, 1] = np.inf
    nonfinite[0] = (inst[0][0], M)
    with pytest.raises(dprt.DprtError):
        dprt.flatten_instances(meshes, nonfinite)
