// bvh_build.h -- host-side BVH8 build for one scene chunk (see bvh_build.cpp).
#pragma once
#include <cstdint>
#include <vector>
#include "dprt_types.h"

namespace dprt {

struct Bvh8 {
    std::vector<dprt_bvh8_node> nodes;
    std::vector<dprt_bvh8_tri> tris;   // leaf order; primID = caller's triangle index
    int max_depth = 0;
    float bounds[6] = {0, 0, 0, 0, 0, 0};
};

// verts: ntris*9 floats; mat_ids: ntris ints or nullptr; pad < 0 selects 2^-16 * max|coordinate|.
int bvh8_build(const float* verts, const int32_t* mat_ids, int64_t ntris, float pad, Bvh8& out);

// Host twin of the GPU builder (bvh_gpu_build.cu, DESIGN.md 3.10): the blob dprt_build_chunk_device makes of these triangles, bit
// for bit (triangle records without texture coordinates). DPRT_ERR_INVALID with the reason in *why: null vertices, ntris <= 0 or
// >= 2^27, a non-finite coordinate.
int spec_bvh8_build_gpu(const float* verts, const int32_t* mat_ids, int64_t ntris, Bvh8& out, const char** why);

}  // namespace dprt
