// instance_flatten.cu -- the flatten of instanced, indexed meshes on the device (DESIGN.md 3.11): what scene_flatten.cpp does
// on the host, with the same arithmetic (instance_xform.cuh) and the same output, bit for bit, written straight into the
// buffers the GPU BVH8 build or the refit reads. Compiled with --fmad=false.
//
// One launch per instance: the normal matrix, the singular / non-finite transform flag and the instance's triangle count,
// followed by CUB's exclusive scan of the counts. One launch per flattened triangle p (primID: the running index over
// (instance, triangle), as on the host): an upper-bound search in the scan finds the instance, so instances of one triangle
// and of millions balance alike. A third launch checks every index of every mesh against the mesh's counts; the gathers of the
// flatten stay inside the arrays whatever the indices hold, and the caller rejects the result on the flag.
#include <cub/device/device_scan.cuh>

#include "dprt_internal.cuh"
#include "instance_xform.cuh"

namespace dprt {
namespace {

constexpr int kThreads = 256;
unsigned blocks(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

// one past the last entry of scan[0, n) that is <= p
__device__ __forceinline__ int64_t upper_bound(const int64_t* __restrict__ scan, int64_t n, int64_t p) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (scan[mid] <= p) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kThreads) instance_prep_kernel(const DevMesh* __restrict__ meshes, const dprt_instance_desc* __restrict__ inst,
                                                                 int64_t n, int64_t* __restrict__ count, float* __restrict__ G,
                                                                 uint32_t* __restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i > n) return;
    if (i == n) { count[n] = 0; return; }         // the scan's extra entry: its output is the total
    count[i] = meshes[inst[i].mesh].ntris;
    if (!instance_normal_matrix(inst[i].objectToWorld, G + 9 * i)) atomicOr(flags, kFlattenSingular);
}

__global__ void __launch_bounds__(kThreads) mesh_index_check_kernel(const DevMesh* __restrict__ meshes, const int64_t* __restrict__ meshTriBase,
                                                                    int nMeshes, int64_t total, uint32_t* __restrict__ flags) {
    const int64_t k = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (k >= total) return;
    const DevMesh& me = meshes[upper_bound(meshTriBase, nMeshes, k) - 1];
    const int64_t t = k - meshTriBase[&me - meshes];
    bool bad = false;
    for (int c = 0; c < 3; c++) {
        const int32_t a = me.indices[3 * t + c], b = me.normalIndices[3 * t + c];
        bad = bad || a < 0 || a >= me.nPositions || b < 0 || b >= me.nNormals;
        if (me.texCoordIndices) {
            const int32_t u = me.texCoordIndices[3 * t + c];
            bad = bad || u < 0 || u >= me.nTexCoords;
        }
    }
    if (bad) atomicOr(flags, kFlattenBadIndex);
}

__global__ void __launch_bounds__(kThreads) instance_flatten_kernel(const DevMesh* __restrict__ meshes, const dprt_instance_desc* __restrict__ inst,
                                                                    int64_t n, const int64_t* __restrict__ scan, const float* __restrict__ G,
                                                                    int64_t ntris, float* __restrict__ verts9, float* __restrict__ normals9,
                                                                    float* __restrict__ uv6, int32_t* __restrict__ mats) {
    const int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= ntris) return;
    const int64_t i = upper_bound(scan, n, p) - 1;
    const DevMesh& me = meshes[inst[i].mesh];
    const int64_t t = p - scan[i];
    float M[12], g[9];
    for (int k = 0; k < 12; k++) M[k] = inst[i].objectToWorld[k];
    for (int k = 0; k < 9; k++) g[k] = G[9 * i + k];
    const float zero[3] = {0.f, 0.f, 0.f};
    for (int c = 0; c < 3; c++) {
        const int32_t a = me.indices[3 * t + c], b = me.normalIndices[3 * t + c];
        instance_corner(M, a >= 0 && a < me.nPositions ? me.positions + 3 * (int64_t)a : zero, verts9 + 9 * p + 3 * c);
        instance_normal(g, b >= 0 && b < me.nNormals ? me.normals + 3 * (int64_t)b : zero, normals9 + 9 * p + 3 * c);
        if (uv6) {
            float* u = uv6 + 6 * p + 2 * c;
            const int32_t x = me.texCoordIndices ? me.texCoordIndices[3 * t + c] : -1;
            if (x >= 0 && x < me.nTexCoords) { u[0] = me.texCoords[2 * (int64_t)x]; u[1] = me.texCoords[2 * (int64_t)x + 1]; }
            else { u[0] = 0.0f; u[1] = 0.0f; }
        }
    }
    if (mats) mats[p] = me.materialID;
}

struct FlattenScratch { int64_t* count; int64_t* scan; float* G; void* temp; size_t tempBytes; size_t total; };

FlattenScratch carve(void* base, int64_t n) {
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    FlattenScratch s{};
    cub::DeviceScan::ExclusiveSum(nullptr, s.tempBytes, (const int64_t*)nullptr, (int64_t*)nullptr, (int)(n + 1));
    const size_t oScan = up((size_t)(n + 1) * sizeof(int64_t)), oG = oScan + up((size_t)(n + 1) * sizeof(int64_t));
    const size_t oTemp = oG + up((size_t)n * 9 * sizeof(float));
    s.total = oTemp + up(s.tempBytes);
    char* b = (char*)base;
    s.count = (int64_t*)b; s.scan = (int64_t*)(b + oScan); s.G = (float*)(b + oG); s.temp = b + oTemp;
    return s;
}

}  // namespace

size_t instance_flatten_scratch_bytes(int64_t nInstances) { return carve(nullptr, nInstances).total; }

cudaError_t launch_mesh_index_check(const DevMesh* meshes, const int64_t* meshTriBase, int nMeshes, int64_t meshTris, uint32_t* flags,
                                    cudaStream_t stream) {
    if (meshTris > 0) mesh_index_check_kernel<<<blocks(meshTris), kThreads, 0, stream>>>(meshes, meshTriBase, nMeshes, meshTris, flags);
    return cudaGetLastError();
}

cudaError_t launch_instance_flatten(const DevMesh* meshes, const dprt_instance_desc* instances, int64_t nInstances, int64_t ntris,
                                    void* scratch, float* verts9, float* normals9, float* uv6, int32_t* mats, uint32_t* flags,
                                    cudaStream_t stream) {
    FlattenScratch s = carve(scratch, nInstances);
    instance_prep_kernel<<<blocks(nInstances + 1), kThreads, 0, stream>>>(meshes, instances, nInstances, s.count, s.G, flags);
    cudaError_t e = cub::DeviceScan::ExclusiveSum(s.temp, s.tempBytes, s.count, s.scan, (int)(nInstances + 1), stream);
    if (e != cudaSuccess) return e;
    instance_flatten_kernel<<<blocks(ntris), kThreads, 0, stream>>>(meshes, instances, nInstances, s.scan, s.G, ntris, verts9, normals9,
                                                                     uv6, mats);
    return cudaGetLastError();
}

}  // namespace dprt
