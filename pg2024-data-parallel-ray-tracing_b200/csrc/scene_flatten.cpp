// scene_flatten.cpp -- host side of the real-scene front end (SURVEY.md 8f row 3): indexed, instanced meshes -> the flat
// per-corner streams the kernels read.
//
// The reference keeps a scene object as up to three levels of OptiX traversables (pipeline_helper.cpp:268-272) whose leaf
// GASes carry an SBT record with INDEXED shading attributes (HitGroupData, pipeline_helper.cpp:182-193); its closest-hit
// program transforms the hit triangle's corners and normals to world space per hit (kernel.cu:205-240:
// optixTransformPointFromObjectToWorldSpace / optixTransformNormalFromObjectToWorldSpace) and gathers normals and texture
// coordinates through two index arrays. Here that work is done ONCE at upload: every (instance, triangle) becomes a
// world-space triangle with three world-space normals and three texture coordinates, stored contiguously per primitive.
// B200 has 180 GB of HBM; the per-hit cost drops to 36 + 24 contiguous bytes and the BVH is a single level.
//
// The instance arithmetic (corners M p, normals A^-T n) is instance_xform.cuh, shared with the device flatten of
// instance_flatten.cu. Built with -ffp-contract=off.
#include <cmath>
#include <cstring>

#include "scene_flatten.h"
#include "instance_xform.cuh"

namespace dprt {

namespace {

bool mesh_ok(const dprt_mesh_desc& m) {
    if (m.ntris < 0 || m.nPositions < 0 || m.nNormals < 0 || m.nTexCoords < 0) return false;
    if (m.ntris == 0) return true;
    if (!m.positions || !m.indices || !m.normals || !m.normalIndices) return false;
    if ((m.texCoords == nullptr) != (m.texCoordIndices == nullptr)) return false;
    if (m.materialID < 0 || m.materialID >= DPRT_MAX_MATERIALS) return false;
    return true;
}

}  // namespace

int64_t flatten_count(const dprt_mesh_desc* meshes, int nMeshes, const dprt_instance_desc* instances, int64_t nInstances) {
    if (!meshes || !instances || nMeshes <= 0 || nInstances <= 0) return -1;
    for (int m = 0; m < nMeshes; m++) if (!mesh_ok(meshes[m])) return -1;
    int64_t total = 0;
    for (int64_t i = 0; i < nInstances; i++) {
        const int mi = instances[i].mesh;
        if (mi < 0 || mi >= nMeshes) return -1;
        total += meshes[mi].ntris;
    }
    return total;
}

int flatten_instances(const dprt_mesh_desc* meshes, int nMeshes, const dprt_instance_desc* instances, int64_t nInstances,
                      float* verts9, float* normals9, float* uv6, int32_t* matIds, int* hasUv) {
    const int64_t total = flatten_count(meshes, nMeshes, instances, nInstances);
    if (total <= 0 || !verts9 || !normals9) return -1;
    bool anyUv = false;
    for (int m = 0; m < nMeshes; m++) anyUv = anyUv || (meshes[m].ntris > 0 && meshes[m].texCoords != nullptr);
    if (hasUv) *hasUv = anyUv ? 1 : 0;
    // index ranges, once per mesh
    for (int m = 0; m < nMeshes; m++) {
        const dprt_mesh_desc& me = meshes[m];
        for (int64_t k = 0; k < 3 * me.ntris; k++) {
            if (me.indices[k] < 0 || me.indices[k] >= me.nPositions) return -1;
            if (me.normalIndices[k] < 0 || me.normalIndices[k] >= me.nNormals) return -1;
            if (me.texCoordIndices && (me.texCoordIndices[k] < 0 || me.texCoordIndices[k] >= me.nTexCoords)) return -1;
        }
    }
    int64_t base = 0;
    for (int64_t i = 0; i < nInstances; i++) {
        const dprt_mesh_desc& me = meshes[instances[i].mesh];
        const float* M = instances[i].objectToWorld;
        float g[9];
        if (!instance_normal_matrix(M, g)) return -1;
#pragma omp parallel for schedule(static) if (me.ntris > 4096)
        for (int64_t t = 0; t < me.ntris; t++) {
            const int64_t p = base + t;
            for (int c = 0; c < 3; c++) {
                instance_corner(M, me.positions + 3 * (int64_t)me.indices[3 * t + c], verts9 + 9 * p + 3 * c);
                instance_normal(g, me.normals + 3 * (int64_t)me.normalIndices[3 * t + c], normals9 + 9 * p + 3 * c);
                if (uv6) {
                    float* u = uv6 + 6 * p + 2 * c;
                    if (me.texCoords) {
                        const float* tc = me.texCoords + 2 * (int64_t)me.texCoordIndices[3 * t + c];
                        u[0] = tc[0]; u[1] = tc[1];
                    } else { u[0] = 0.0f; u[1] = 0.0f; }
                }
            }
            if (matIds) matIds[p] = me.materialID;
        }
        base += me.ntris;
    }
    return 0;
}

}  // namespace dprt
