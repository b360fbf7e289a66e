// refit.cu -- BVH8 refit: new vertex positions into an uploaded chunk's BVH8, same topology (DESIGN.md 3.9 is the
// specification). Compiled with --fmad=false on the device and -ffp-contract=off on the host: the kernels and
// dprt_spec_bvh8_refit run the same functions, and the node encoding is the builder's own (bvh_node.cuh), so a refit with
// the vertices of the build reproduces the build bit for bit.
//
// One refit = one triangle launch (corners gathered by primID) + one node launch per depth level, deepest level first. The
// builder writes nodes in BFS order, so every level is one contiguous index range (ObjMem::levels, derived at upload) and
// a node's internal children sit in the next level; each node leaves its exact box (24 bytes) in the scratch for its parent.
#include <cmath>
#include <vector>

#include "dprt_internal.cuh"
#include "bvh_node.cuh"

namespace dprt {
namespace {

#ifdef __CUDA_ARCH__
#define RF_POPC(x) __popc(x)
#else
#define RF_POPC(x) __builtin_popcount(x)
#endif

constexpr int kStatThreads = 256, kStatBlocks = 296;   // 2 blocks per SM on a B200
constexpr size_t kPartOffset = 256;                     // scratch: final RefitStats | kStatBlocks partials | node boxes
size_t boxes_offset() { return kPartOffset + ((kStatBlocks * sizeof(RefitStats) + 255) & ~(size_t)255); }

// leaf record t <- the corners of its triangle; primID, matID and pad_ stay
DPRT_NODE_HD void refit_tri(dprt_bvh8_tri& t, const float* verts9) {
    const float* v = verts9 + 9 * (size_t)t.primID;
    for (int a = 0; a < 3; a++) { t.v0[a] = v[a]; t.v1[a] = v[3 + a]; t.v2[a] = v[6 + a]; }
}

// node i from the (refitted) triangles of its leaf slots and the exact boxes of its internal children (6 floats per node in
// `boxes`); leaves node i's own exact box there
DPRT_NODE_HD void refit_node(dprt_bvh8_node* nodes, uint32_t i, const dprt_bvh8_tri* tris, float* boxes, float pad) {
    dprt_bvh8_node n = nodes[i];
    float lo[8][3], hi[8][3];
    uint32_t used = 0, irank = 0;
    for (int s = 0; s < 8; s++) {
        if ((n.imask >> s) & 1u) {
            const float* b = boxes + 6 * (size_t)(n.childBase + irank++);
            for (int a = 0; a < 3; a++) { lo[s][a] = b[a]; hi[s][a] = b[3 + a]; }
            used |= 1u << s;
            continue;
        }
        const uint32_t k = RF_POPC((n.tmask >> (3 * s)) & 7u);
        if (!k) continue;
        const dprt_bvh8_tri* t = tris + n.triBase + RF_POPC(n.tmask & ((1u << (3 * s)) - 1u));
        for (int a = 0; a < 3; a++) { lo[s][a] = FLT_MAX; hi[s][a] = -FLT_MAX; }
        for (uint32_t j = 0; j < k; j++) {
            const float* c[3] = {t[j].v0, t[j].v1, t[j].v2};
            for (int q = 0; q < 3; q++)
                for (int a = 0; a < 3; a++) {
                    lo[s][a] = c[q][a] < lo[s][a] ? c[q][a] : lo[s][a];
                    hi[s][a] = c[q][a] > hi[s][a] ? c[q][a] : hi[s][a];
                }
        }
        used |= 1u << s;
    }
    float blo[3], bhi[3];
    bvh8_encode_node(n, lo, hi, used, pad, blo, bhi);
    nodes[i] = n;
    for (int a = 0; a < 3; a++) { boxes[6 * (size_t)i + a] = blo[a]; boxes[6 * (size_t)i + 3 + a] = bhi[a]; }
}

__global__ void __launch_bounds__(256) refit_tris_kernel(dprt_bvh8_tri* __restrict__ tris, int64_t ntris, const float* __restrict__ verts9) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ntris) refit_tri(tris[t], verts9);
}

__global__ void __launch_bounds__(128) refit_nodes_kernel(dprt_bvh8_node* __restrict__ nodes, int64_t first, int64_t last,
                                                          const dprt_bvh8_tri* __restrict__ tris, float* __restrict__ boxes, float pad) {
    const int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < last) refit_node(nodes, (uint32_t)i, tris, boxes, pad);
}

// min / max of the finite coordinates per axis and the count of non-finite ones, reduced over the block into out
__device__ void stats_block_reduce(float lo[3], float hi[3], uint32_t bad, RefitStats* out) {
    __shared__ float slo[kStatThreads / 32][3], shi[kStatThreads / 32][3];
    __shared__ uint32_t sbad[kStatThreads / 32];
    for (int o = 16; o > 0; o >>= 1) {
        for (int a = 0; a < 3; a++) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        for (int a = 0; a < 3; a++) { slo[w][a] = lo[a]; shi[w][a] = hi[a]; }
        sbad[w] = bad;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        RefitStats r;
        for (int a = 0; a < 3; a++) { r.lo[a] = FLT_MAX; r.hi[a] = -FLT_MAX; }
        r.nonfinite = 0; r.pad_ = 0;
        for (int k = 0; k < kStatThreads / 32; k++) {
            for (int a = 0; a < 3; a++) { r.lo[a] = fminf(r.lo[a], slo[k][a]); r.hi[a] = fmaxf(r.hi[a], shi[k][a]); }
            r.nonfinite += sbad[k];
        }
        *out = r;
    }
}

__global__ void __launch_bounds__(kStatThreads) refit_stats_kernel(const float* __restrict__ verts, int64_t nverts, RefitStats* __restrict__ part) {
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    uint32_t bad = 0;
    for (int64_t i = (int64_t)blockIdx.x * kStatThreads + threadIdx.x; i < nverts; i += (int64_t)gridDim.x * kStatThreads)
        for (int a = 0; a < 3; a++) {
            const float x = verts[3 * i + a];
            if (isfinite(x)) { lo[a] = fminf(lo[a], x); hi[a] = fmaxf(hi[a], x); } else bad++;
        }
    stats_block_reduce(lo, hi, bad, part + blockIdx.x);
}

__global__ void __launch_bounds__(kStatThreads) refit_stats_final_kernel(const RefitStats* __restrict__ part, int n, RefitStats* __restrict__ out) {
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    uint32_t bad = 0;
    for (int k = threadIdx.x; k < n; k += kStatThreads) {
        for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], part[k].lo[a]); hi[a] = fmaxf(hi[a], part[k].hi[a]); }
        bad += part[k].nonfinite;
    }
    stats_block_reduce(lo, hi, bad, out);
}

}  // namespace

size_t refit_scratch_bytes(int64_t nnodes) { return boxes_offset() + 6 * sizeof(float) * (size_t)nnodes; }

void launch_refit_stats(const float* verts9, int64_t ntris, void* scratch, cudaStream_t stream) {
    RefitStats* part = (RefitStats*)((char*)scratch + kPartOffset);
    refit_stats_kernel<<<kStatBlocks, kStatThreads, 0, stream>>>(verts9, 3 * ntris, part);
    refit_stats_final_kernel<<<1, kStatThreads, 0, stream>>>(part, kStatBlocks, (RefitStats*)scratch);
}

void launch_refit(dprt_bvh8_node* nodes, dprt_bvh8_tri* tris, int64_t ntris, const float* verts9, const int64_t* levels, int nlevels,
                  float pad, void* scratch, cudaStream_t stream) {
    refit_tris_kernel<<<(unsigned)((ntris + 255) / 256), 256, 0, stream>>>(tris, ntris, verts9);
    float* boxes = (float*)((char*)scratch + boxes_offset());
    for (int d = nlevels - 1; d >= 0; d--) {
        const int64_t n = levels[d + 1] - levels[d];
        refit_nodes_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(nodes, levels[d], levels[d + 1], tris, boxes, pad);
    }
}

int spec_bvh8_refit(dprt_bvh8_node* nodes, int64_t nnodes, dprt_bvh8_tri* tris, int64_t ntris, const float* verts9, const char** why) {
    *why = "";
    if (!nodes || !tris || !verts9 || nnodes < 1 || ntris < 1 || nnodes > 0xffffffffLL || ntris > 0x7fffffffLL) {
        *why = "null array or size out of range"; return DPRT_ERR_INVALID;
    }
    // the blob comes from outside the library: every index it holds is checked before anything is written
    for (int64_t i = 0; i < nnodes; i++) {
        const dprt_bvh8_node& n = nodes[i];
        if (n.tmask >> 24) { *why = "tmask bits above 23"; return DPRT_ERR_INVALID; }
        for (int s = 0; s < 8; s++) {
            const uint32_t g = (n.tmask >> (3 * s)) & 7u;
            if (g != 0 && g != 1 && g != 3 && g != 7) { *why = "slot triangle bits not of the form 1, 11, 111"; return DPRT_ERR_INVALID; }
            if (g && ((n.imask >> s) & 1u)) { *why = "slot both internal and leaf"; return DPRT_ERR_INVALID; }
        }
        if (n.imask && ((int64_t)n.childBase <= i || (int64_t)n.childBase + RF_POPC(n.imask) > nnodes)) {
            *why = "childBase outside the node array (or not after its parent)"; return DPRT_ERR_INVALID;
        }
        if (n.tmask && (int64_t)n.triBase + RF_POPC(n.tmask) > ntris) { *why = "triBase outside the triangle array"; return DPRT_ERR_INVALID; }
    }
    for (int64_t t = 0; t < ntris; t++)
        if (tris[t].primID < 0 || tris[t].primID >= ntris) { *why = "primID outside the vertex array"; return DPRT_ERR_INVALID; }
    float m = 0.f;
    for (int64_t k = 0; k < 9 * ntris; k++) {
        if (!std::isfinite(verts9[k])) { *why = "non-finite coordinate"; return DPRT_ERR_INVALID; }
        m = std::fmax(m, std::fabs(verts9[k]));
    }
    const float pad = bvh8_chunk_pad(m);
    for (int64_t t = 0; t < ntris; t++) refit_tri(tris[t], verts9);
    std::vector<float> boxes(6 * (size_t)nnodes);
    for (int64_t i = nnodes - 1; i >= 0; i--) refit_node(nodes, (uint32_t)i, tris, boxes.data(), pad);
    return 0;
}

}  // namespace dprt
