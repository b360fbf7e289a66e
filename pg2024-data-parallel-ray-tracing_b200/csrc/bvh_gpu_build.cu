// bvh_gpu_build.cu -- BVH8 build on the GPU from device-resident triangles (DESIGN.md 3.10 is the specification), and its host
// twin spec_bvh8_build_gpu. Both run the per-element functions below, in the same order of dependent steps, and the collapse,
// slot assignment and node encoding are the host builder's own (bvh_node.cuh), so the device blob equals the twin's bit for
// bit. It is a different binary tree from bvh8_build's (PLOC instead of binned SAH), so it is not that builder's blob.
// Compiled with --fmad=false on the device and -ffp-contract=off on the host: every float step is one binary32 operation.
//
// Steps: triangle boxes and centroids -> 63-bit Morton codes in the centroid bounds -> stable radix sort -> PLOC binary tree
// (Meister & Bittner 2018), each new node's SAH cost row computed when it is created -> breadth-first emission, one level at a
// time (count, scan, write). The host reads back one 64-bit count per PLOC iteration and per level, never nodes or triangles.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>
#include <vector>

#include "dprt_internal.cuh"
#include "bvh_build.h"
#include "bvh_node.cuh"

namespace dprt {
namespace {

// Search radius of the nearest-neighbour step: each cluster looks at the kPlocRadius clusters on either side of it in the
// Morton-ordered cluster array. Chosen from the CPU quality measurement in DESIGN.md 3.10.
constexpr int kPlocRadius = 4;
constexpr uint32_t kSlotEmpty = 0xffffffffu, kSlotLeaf = 0x80000000u;

// The arrays of one build. Binary node ids: leaves 0..n-1 in sorted (Morton) order, internal nodes n..2n-2 in creation order,
// so children always have lower ids than their parents; the root is the last one created.
struct GbView {
    int32_t n;
    const float* verts;        // 9 per triangle
    float* cen;                // 3 per triangle, padded to whole triples with copies of centroid 0
    uint64_t* keys;            // Morton code per triangle (input order)
    int32_t* idx;              // sorted position -> triangle index
    float* box;                // 6 per binary node: lo, hi
    int32_t* child;            // 2 per internal node (index id - n)
    int32_t* pcount;           // triangles below each binary node
    float* C; uint8_t* K; uint8_t* K8;   // SAH cost rows (bvh_node.cuh): 8 + 8 + 1 per binary node
    int32_t* cl; int32_t* cl2; int32_t* nn;   // clusters (node ids) by position, the compacted next array, nearest neighbour
    uint64_t* flag; uint64_t* flagEx;         // n + 1: (kept << 32 | merged) per position and its exclusive scan
    int32_t* wbin;             // wide node -> its binary node (wide nodes in BFS order)
    uint32_t* wslot;           // 8 per wide node: child binary id per slot, | kSlotLeaf for a leaf slot, kSlotEmpty
    uint64_t* wcnt; uint64_t* wscan;          // n + 1: (internal children << 32 | triangles) per wide node and its scan
};

struct GbTree {
    const GbView& v;
    DPRT_NODE_HD bool is_leaf(int m) const { return m < v.n; }
    DPRT_NODE_HD int left(int m) const { return v.child[2 * (m - v.n)]; }
    DPRT_NODE_HD int right(int m) const { return v.child[2 * (m - v.n) + 1]; }
    DPRT_NODE_HD const uint8_t* k(int m) const { return v.K + 8 * (size_t)m; }
};

// the exact box of triangle p, grown corner by corner as bvh_build.cpp's Box::grow does it
DPRT_NODE_HD void gb_tri_box(const float* verts, int p, float* lo, float* hi) {
    const float* v = verts + 9 * (size_t)p;
    for (int a = 0; a < 3; a++) { lo[a] = FLT_MAX; hi[a] = -FLT_MAX; }
    for (int q = 0; q < 3; q++)
        for (int a = 0; a < 3; a++) {
            const float x = v[3 * q + a];
            lo[a] = x < lo[a] ? x : lo[a];
            hi[a] = hi[a] < x ? x : hi[a];
        }
}

DPRT_NODE_HD void gb_centroid(const GbView& v, int i) {
    float lo[3], hi[3];
    gb_tri_box(v.verts, i, lo, hi);
    for (int a = 0; a < 3; a++) v.cen[3 * (size_t)i + a] = 0.5f * (lo[a] + hi[a]);
}

DPRT_NODE_HD uint64_t gb_expand21(uint32_t x) {
    uint64_t e = x & 0x1fffffu;
    e = (e | e << 32) & 0x1f00000000ffffull;
    e = (e | e << 16) & 0x1f0000ff0000ffull;
    e = (e | e << 8) & 0x100f00f00f00f00full;
    e = (e | e << 4) & 0x10c30c30c30c30c3ull;
    e = (e | e << 2) & 0x1249249249249249ull;
    return e;
}

// Morton code of centroid i in the centroid bounds clo / chi: per axis q = trunc((c - lo) * (2^21 / (hi - lo))) clamped to
// [0, 2^21 - 1] (0 on an axis of no extent); x in bit 3k + 2, y in 3k + 1, z in 3k
DPRT_NODE_HD void gb_morton(const GbView& v, int i, const float* clo, const float* chi) {
    uint64_t code = 0;
    for (int a = 0; a < 3; a++) {
        const float ext = chi[a] - clo[a];
        uint32_t q = 0;
        if (ext > 0.f) {
            const float s = 2097152.0f / ext;
            const float f = (v.cen[3 * (size_t)i + a] - clo[a]) * s;
            q = f >= 2097151.0f ? 2097151u : (f > 0.f ? (uint32_t)f : 0u);
        }
        code |= gb_expand21(q) << (2 - a);
    }
    v.keys[i] = code;
    v.idx[i] = i;
}

// binary leaf b: triangle idx[b] (after the sort), one cluster
DPRT_NODE_HD void gb_leaf(const GbView& v, int b) {
    float* bx = v.box + 6 * (size_t)b;
    gb_tri_box(v.verts, v.idx[b], bx, bx + 3);
    v.pcount[b] = 1;
    bvh8_dp_leaf(bvh8_half_area(bx, bx + 3), 1, v.C + 8 * (size_t)b, v.K + 8 * (size_t)b);
    v.cl[b] = b;
}

// PLOC distance: half area of the union box, as Box::half_area; NaN (an overflowing extent times 0) counts as +inf so that
// the distances are totally ordered and every iteration has a mutual pair
DPRT_NODE_HD float gb_dist(const float* a, const float* b) {
    float lo[3], hi[3];
    for (int k = 0; k < 3; k++) { lo[k] = b[k] < a[k] ? b[k] : a[k]; hi[k] = a[3 + k] < b[3 + k] ? b[3 + k] : a[3 + k]; }
    const float d = bvh8_half_area(lo, hi);
    return d == d ? d : INFINITY;
}

// Order of the candidate pairs {i, j} at equal distance: nearer positions first, then pairs whose lower position is even, then
// the lower position. The key is symmetric in i and j, so (distance, key) orders the unordered pairs totally: the least pair
// of all is mutual and every iteration merges. In a run of equal boxes (coincident triangles) it pairs 2k with 2k + 1, so the
// whole run merges in parallel and builds a balanced subtree, instead of one pair per iteration at the run's lowest position.
DPRT_NODE_HD uint64_t gb_tie_key(int i, int j) {
    const uint32_t lo = (uint32_t)(i < j ? i : j), gap = (uint32_t)(i < j ? j - i : i - j);
    return ((uint64_t)gap << 33) | ((uint64_t)(lo & 1u) << 32) | lo;
}

// nearest neighbour of the cluster at position i among positions i - r .. i + r (nc clusters); ties by gb_tie_key
DPRT_NODE_HD void gb_nearest(const GbView& v, int i, int nc) {
    const float* bi = v.box + 6 * (size_t)v.cl[i];
    const int lo = i - kPlocRadius < 0 ? 0 : i - kPlocRadius, hi = i + kPlocRadius > nc - 1 ? nc - 1 : i + kPlocRadius;
    float best = INFINITY; uint64_t bkey = 0; int bj = -1;
    for (int j = lo; j <= hi; j++) {
        if (j == i) continue;
        const float d = gb_dist(bi, v.box + 6 * (size_t)v.cl[j]);
        const uint64_t key = gb_tie_key(i, j);
        if (bj < 0 || d < best || (d == best && key < bkey)) { best = d; bkey = key; bj = j; }
    }
    v.nn[i] = bj;
}

// position i: kept (not the higher of a mutual pair) in the high word, merged (the lower of a mutual pair) in the low word
DPRT_NODE_HD void gb_flag(const GbView& v, int i, int nc) {
    const int j = v.nn[i];
    const bool mutual = v.nn[j] == i;
    v.flag[i] = ((uint64_t)!(mutual && j < i) << 32) | (uint64_t)(mutual && i < j);
    if (i == nc - 1) v.flag[nc] = 0;
}

// compaction: a kept position moves to its scanned place; a mutual pair becomes new node next_id + (merges before it), at the
// place of its lower position, with its cost row computed from its children's
DPRT_NODE_HD void gb_merge(const GbView& v, int i, int next_id) {
    const int j = v.nn[i];
    const bool mutual = v.nn[j] == i;
    if (mutual && j < i) return;
    const uint64_t ex = v.flagEx[i];
    const int pos = (int)(ex >> 32);
    if (!mutual) { v.cl2[pos] = v.cl[i]; return; }
    const int id = next_id + (int)(uint32_t)ex, l = v.cl[i], r = v.cl[j];
    float* b = v.box + 6 * (size_t)id;
    const float* bl = v.box + 6 * (size_t)l; const float* br = v.box + 6 * (size_t)r;
    for (int a = 0; a < 3; a++) { b[a] = br[a] < bl[a] ? br[a] : bl[a]; b[3 + a] = bl[3 + a] < br[3 + a] ? br[3 + a] : bl[3 + a]; }
    v.child[2 * (size_t)(id - v.n)] = l; v.child[2 * (size_t)(id - v.n) + 1] = r;
    const int pc = v.pcount[l] + v.pcount[r];
    v.pcount[id] = pc;
    v.K8[id] = bvh8_dp_node(bvh8_half_area(b, b + 3), pc, v.C + 8 * (size_t)l, v.C + 8 * (size_t)r, v.C + 8 * (size_t)id,
                            v.K + 8 * (size_t)id);
    v.cl2[pos] = id;
}

// wide node g: its children (collapse), their slots, and its counts of internal children and triangles
DPRT_NODE_HD void gb_emit_count(const GbView& v, int64_t g, int root) {
    const int b = v.wbin[g];
    Bvh8Child ch[8]; int nch = 0;
    const GbTree t{v};
    if (b < v.n || (b == root && v.K[8 * (size_t)root] == 1)) ch[nch++] = Bvh8Child{b, true};     // a root that is itself a leaf
    else { bvh8_collect(t, t.left(b), v.K8[b], ch, nch); bvh8_collect(t, t.right(b), 8 - v.K8[b], ch, nch); }
    float clo[8][3], chi[8][3]; int slot_of[8];
    for (int c = 0; c < nch; c++)
        for (int a = 0; a < 3; a++) { clo[c][a] = v.box[6 * (size_t)ch[c].n + a]; chi[c][a] = v.box[6 * (size_t)ch[c].n + 3 + a]; }
    bvh8_assign_slots(clo, chi, nch, slot_of);
    uint32_t* ws = v.wslot + 8 * g;
    for (int s = 0; s < 8; s++) ws[s] = kSlotEmpty;
    uint32_t ni = 0, nt = 0;
    for (int c = 0; c < nch; c++) {
        ws[slot_of[c]] = (uint32_t)ch[c].n | (ch[c].leaf ? kSlotLeaf : 0u);
        if (ch[c].leaf) nt += (uint32_t)v.pcount[ch[c].n]; else ni++;
    }
    v.wcnt[g] = ((uint64_t)ni << 32) | nt;
}

// the internal children of wide node g become the wide nodes next + (scanned count) .. of the next level, in slot order
DPRT_NODE_HD void gb_emit_items(const GbView& v, int64_t g, int64_t next) {
    int64_t o = next + (int64_t)(v.wscan[g] >> 32);
    for (int s = 0; s < 8; s++) {
        const uint32_t x = v.wslot[8 * g + s];
        if (x != kSlotEmpty && !(x & kSlotLeaf)) v.wbin[o++] = (int)x;
    }
}

// wide node g (level starting at triangle record tri0, next level at node next): triangle records of its leaf slots, each
// slot's triangles from left to right, then the node itself
DPRT_NODE_HD void gb_emit_write(const GbView& v, int64_t g, int64_t next, int64_t tri0, const int32_t* mats, const float* uv6,
                                int32_t uvCount, float pad, dprt_bvh8_node* nodes, dprt_bvh8_tri* tris, float* uvTail) {
    const uint64_t ex = v.wscan[g];
    dprt_bvh8_node node;
    memset(&node, 0, sizeof(node));
    node.childBase = (uint32_t)(next + (int64_t)(ex >> 32));
    node.triBase = (uint32_t)(tri0 + (int64_t)(uint32_t)ex);
    float slo[8][3], shi[8][3];
    uint32_t used = 0, t = node.triBase;
    for (int s = 0; s < 8; s++) {
        const uint32_t x = v.wslot[8 * g + s];
        if (x == kSlotEmpty) continue;
        const int c = (int)(x & ~kSlotLeaf);
        if (!(x & kSlotLeaf)) {
            node.imask |= (uint8_t)(1u << s);
        } else {
            const int lcount = v.pcount[c];         // <= 3
            node.tmask |= (uint32_t)(lcount == 1 ? 1 : (lcount == 2 ? 3 : 7)) << (3 * s);
            int st[4], sp = 0;
            st[sp++] = c;
            while (sp) {                            // the subtree's leaves, left to right
                const int m = st[--sp];
                if (m >= v.n) { st[sp++] = v.child[2 * (size_t)(m - v.n) + 1]; st[sp++] = v.child[2 * (size_t)(m - v.n)]; continue; }
                const int p = v.idx[m];
                dprt_bvh8_tri& r = tris[t];
                const float* src = v.verts + 9 * (size_t)p;
                for (int a = 0; a < 3; a++) { r.v0[a] = src[a]; r.v1[a] = src[3 + a]; r.v2[a] = src[6 + a]; }
                r.primID = p; r.matID = mats ? mats[p] : 0; r.pad_ = uvCount;
                if (uvTail) {
                    for (int k = 0; k < 6; k++) uvTail[8 * (size_t)t + k] = uv6[6 * (size_t)p + k];
                    uvTail[8 * (size_t)t + 6] = 0.0f; uvTail[8 * (size_t)t + 7] = 0.0f;
                }
                t++;
            }
        }
        used |= 1u << s;
        for (int a = 0; a < 3; a++) { slo[s][a] = v.box[6 * (size_t)c + a]; shi[s][a] = v.box[6 * (size_t)c + 3 + a]; }
    }
    float nlo[3], nhi[3];
    bvh8_encode_node(node, slo, shi, used, pad, nlo, nhi);
    nodes[g] = node;
}

// ---- device ------------------------------------------------------------------------------------------------------------
constexpr int kThreads = 256;
unsigned blocks(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

__global__ void __launch_bounds__(kThreads) gb_centroid_kernel(GbView v) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= v.n) return;
    gb_centroid(v, i);
    if (i == 0)                                     // pad to whole triples with copies of centroid 0: the bounds reduction reads triangles
        for (int k = v.n; k % 3; k++)
            for (int a = 0; a < 3; a++) v.cen[3 * (size_t)k + a] = v.cen[a];
}

__global__ void __launch_bounds__(kThreads) gb_material_check_kernel(const int32_t* __restrict__ mats, int64_t n, uint32_t* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i < n && (mats[i] < 0 || mats[i] >= DPRT_MAX_MATERIALS)) *bad = 1;     // every writer stores the same value
}

__global__ void __launch_bounds__(kThreads) gb_morton_kernel(GbView v, const RefitStats* __restrict__ cb) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < v.n) gb_morton(v, i, cb->lo, cb->hi);
}

__global__ void __launch_bounds__(kThreads) gb_leaf_kernel(GbView v) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < v.n) gb_leaf(v, i);
}

__global__ void __launch_bounds__(kThreads) gb_nearest_kernel(GbView v, int nc) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < nc) gb_nearest(v, i, nc);
}

__global__ void __launch_bounds__(kThreads) gb_flag_kernel(GbView v, int nc) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < nc) gb_flag(v, i, nc);
}

__global__ void __launch_bounds__(kThreads) gb_merge_kernel(GbView v, int nc, int next_id) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < nc) gb_merge(v, i, next_id);
}

__global__ void __launch_bounds__(kThreads) gb_emit_count_kernel(GbView v, int64_t first, int64_t last, int root) {
    const int64_t g = first + (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (g < last) gb_emit_count(v, g, root);
    if (g == last) v.wcnt[g] = 0;                   // the scan's extra entry: its output is the level's total
}

__global__ void __launch_bounds__(kThreads) gb_emit_items_kernel(GbView v, int64_t first, int64_t last) {
    const int64_t g = first + (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (g < last) gb_emit_items(v, g, last);
}

__global__ void __launch_bounds__(kThreads) gb_emit_write_kernel(GbView v, int64_t first, int64_t last, int64_t tri0, const int32_t* mats,
                                                                 const float* uv6, int32_t uvCount, float pad, dprt_bvh8_node* nodes,
                                                                 dprt_bvh8_tri* tris, float* uvTail) {
    const int64_t g = first + (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (g < last) gb_emit_write(v, g, last, tri0, mats, uv6, uvCount, pad, nodes, tris, uvTail);
}

// Scratch layout of a build of n triangles. base == nullptr only measures it.
struct Carve {
    char* base; size_t off = 0;
    template <class T> T* take(size_t count) {
        off = (off + 255) & ~(size_t)255;
        T* p = base ? (T*)(base + off) : nullptr;
        off += count * sizeof(T);
        return p;
    }
};

struct GbDevice {
    GbView v;
    uint64_t* keysAlt; int32_t* idxAlt;     // the radix sort's second buffers
    void* vstats; void* cstats;             // launch_refit_stats scratch: vertices, centroids
    uint32_t* badMat;
    void* temp; size_t tempBytes;           // cub temporary storage (sort or scan)
};

size_t cub_temp_bytes(int64_t n) {
    size_t sortBytes = 0, scanBytes = 0;
    cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
    cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, dk, dv, (int)n, 0, 63);
    cub::DeviceScan::ExclusiveSum(nullptr, scanBytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (int)n + 1);
    return std::max(sortBytes, scanBytes);
}

GbDevice carve(void* scratch, int64_t n, size_t tempBytes, size_t* total = nullptr) {
    Carve c{(char*)scratch};
    GbDevice d{};
    const size_t nb = 2 * (size_t)n - 1, ni = n > 1 ? (size_t)n - 1 : 1;
    d.vstats = c.take<char>(refit_scratch_bytes(0));
    d.cstats = c.take<char>(refit_scratch_bytes(0));
    d.badMat = c.take<uint32_t>(1);
    GbView& v = d.v;
    v.n = (int32_t)n;
    v.cen = c.take<float>(9 * (size_t)((n + 2) / 3));
    v.keys = c.take<uint64_t>(n); d.keysAlt = c.take<uint64_t>(n);
    v.idx = c.take<int32_t>(n); d.idxAlt = c.take<int32_t>(n);
    v.box = c.take<float>(6 * nb);
    v.child = c.take<int32_t>(2 * ni);
    v.pcount = c.take<int32_t>(nb);
    v.C = c.take<float>(8 * nb);
    v.K = c.take<uint8_t>(8 * nb);
    v.K8 = c.take<uint8_t>(nb);
    v.cl = c.take<int32_t>(n); v.cl2 = c.take<int32_t>(n); v.nn = c.take<int32_t>(n);
    v.flag = c.take<uint64_t>(n + 1); v.flagEx = c.take<uint64_t>(n + 1);
    v.wbin = c.take<int32_t>(n + 1);              // at most max(1, n - 1) wide nodes: each has >= 2 children unless it is the only one
    v.wslot = c.take<uint32_t>(8 * ((size_t)n + 1));
    v.wcnt = c.take<uint64_t>(n + 1); v.wscan = c.take<uint64_t>(n + 1);
    d.temp = c.take<char>(tempBytes); d.tempBytes = tempBytes;
    if (total) *total = c.off;
    return d;
}

// one 64-bit count back to the host
cudaError_t read_count(const uint64_t* src, uint64_t* out, cudaStream_t stream) {
    cudaError_t e = cudaMemcpyAsync(out, src, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream);
    return e != cudaSuccess ? e : cudaStreamSynchronize(stream);
}

}  // namespace

size_t gpu_build_scratch_bytes(int64_t ntris) {
    size_t total = 0;
    carve(nullptr, ntris, cub_temp_bytes(ntris), &total);
    return total;
}

cudaError_t gpu_build_check(const float* verts9, const int32_t* mats, int64_t ntris, void* scratch, cudaStream_t stream, RefitStats* st,
                            uint32_t* badMat, const uint32_t* flags, uint32_t* flagsOut) {
    GbDevice d = carve(scratch, ntris, 0);
    cudaError_t e;
    if ((e = cudaMemsetAsync(d.badMat, 0, sizeof(uint32_t), stream)) != cudaSuccess) return e;
    launch_refit_stats(verts9, ntris, d.vstats, stream);
    if (mats) gb_material_check_kernel<<<blocks(ntris), kThreads, 0, stream>>>(mats, ntris, d.badMat);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(st, d.vstats, sizeof(RefitStats), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(badMat, d.badMat, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    if (flags && (e = cudaMemcpyAsync(flagsOut, flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    return cudaStreamSynchronize(stream);
}

cudaError_t gpu_build_tree(const float* verts9, int64_t ntris, void* scratch, cudaStream_t stream, int maxDepth, std::vector<int64_t>& levels,
                           std::vector<int64_t>& triBase, const char** why) {
    *why = nullptr;
    GbDevice d = carve(scratch, ntris, cub_temp_bytes(ntris));
    GbView v = d.v;
    v.verts = verts9;
    const int n = (int)ntris;
    cudaError_t e;
    // Morton order
    gb_centroid_kernel<<<blocks(n), kThreads, 0, stream>>>(v);
    launch_refit_stats(v.cen, (n + 2) / 3, d.cstats, stream);
    gb_morton_kernel<<<blocks(n), kThreads, 0, stream>>>(v, (const RefitStats*)d.cstats);
    cub::DoubleBuffer<uint64_t> dk(v.keys, d.keysAlt);
    cub::DoubleBuffer<int32_t> dv(v.idx, d.idxAlt);
    size_t tb = d.tempBytes;
    if ((e = cub::DeviceRadixSort::SortPairs(d.temp, tb, dk, dv, n, 0, 63, stream)) != cudaSuccess) return e;
    if (dv.Current() != v.idx &&      // the sorted order lives in v.idx from here on
        (e = cudaMemcpyAsync(v.idx, dv.Current(), sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToDevice, stream)) != cudaSuccess) return e;
    gb_leaf_kernel<<<blocks(n), kThreads, 0, stream>>>(v);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    // PLOC
    int nc = n, next = n;
    while (nc > 1) {
        gb_nearest_kernel<<<blocks(nc), kThreads, 0, stream>>>(v, nc);
        gb_flag_kernel<<<blocks(nc), kThreads, 0, stream>>>(v, nc);
        tb = d.tempBytes;
        if ((e = cub::DeviceScan::ExclusiveSum(d.temp, tb, v.flag, v.flagEx, nc + 1, stream)) != cudaSuccess) return e;
        gb_merge_kernel<<<blocks(nc), kThreads, 0, stream>>>(v, nc, next);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        uint64_t tot = 0;
        if ((e = read_count(v.flagEx + nc, &tot, stream)) != cudaSuccess) return e;
        const int merged = (int)(uint32_t)tot;
        if (merged == 0) { *why = "no mutual nearest neighbours (cannot happen with totally ordered distances)"; return cudaSuccess; }
        nc = (int)(tot >> 32); next += merged;
        std::swap(v.cl, v.cl2);
    }
    const int root = n == 1 ? 0 : next - 1;
    // emission, pass 1: per level the wide nodes' children and slots, the scan of their counts, the next level's items
    if ((e = cudaMemcpyAsync(v.wbin, &root, sizeof(int), cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    levels.assign(1, 0); triBase.assign(1, 0);
    int64_t first = 0, last = 1;
    while (first < last) {
        if ((int)levels.size() - 1 >= maxDepth) { levels.push_back(last); return cudaSuccess; }     // one level too many: depth > maxDepth
        levels.push_back(last);
        gb_emit_count_kernel<<<blocks(last - first + 1), kThreads, 0, stream>>>(v, first, last, root);
        tb = d.tempBytes;
        if ((e = cub::DeviceScan::ExclusiveSum(d.temp, tb, v.wcnt + first, v.wscan + first, (int)(last - first + 1), stream)) != cudaSuccess)
            return e;
        gb_emit_items_kernel<<<blocks(last - first), kThreads, 0, stream>>>(v, first, last);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        uint64_t tot = 0;
        if ((e = read_count(v.wscan + last, &tot, stream)) != cudaSuccess) return e;
        triBase.push_back(triBase.back() + (int64_t)(uint32_t)tot);
        first = last; last += (int64_t)(tot >> 32);
    }
    return cudaSuccess;
}

void launch_gpu_build_write(const float* verts9, const int32_t* mats, const float* uv6, int64_t ntris, float pad, void* scratch,
                            const std::vector<int64_t>& levels, const std::vector<int64_t>& triBase, dprt_bvh8_node* nodes,
                            dprt_bvh8_tri* tris, cudaStream_t stream) {
    GbDevice d = carve(scratch, ntris, 0);
    GbView v = d.v;
    v.verts = verts9;
    float* uvTail = uv6 ? (float*)(tris + ntris) : nullptr;
    for (size_t k = 0; k + 1 < levels.size(); k++)
        gb_emit_write_kernel<<<blocks(levels[k + 1] - levels[k]), kThreads, 0, stream>>>(
            v, levels[k], levels[k + 1], triBase[k], mats, uv6, uv6 ? (int32_t)ntris : 0, pad, nodes, tris, uvTail);
}

// ---- host twin: the same functions, one element after the other ------------------------------------------------------------
int spec_bvh8_build_gpu(const float* verts9, const int32_t* mat_ids, int64_t ntris, Bvh8& out, const char** why) {
    out.nodes.clear(); out.tris.clear(); out.max_depth = 0;
    *why = "";
    if (!verts9 || ntris <= 0) { *why = "null vertex array or ntris <= 0"; return DPRT_ERR_INVALID; }
    if (ntris >= ((int64_t)1 << 27)) { *why = "more than 2^27 triangles"; return DPRT_ERR_INVALID; }
    float m = 0.f;
    for (int64_t k = 0; k < 9 * ntris; k++) {
        if (!std::isfinite(verts9[k])) { *why = "non-finite coordinate"; return DPRT_ERR_INVALID; }
        m = std::fmax(m, std::fabs(verts9[k]));
    }
    const float pad = bvh8_chunk_pad(m);
    const int n = (int)ntris;
    const size_t nb = 2 * (size_t)n - 1;
    std::vector<float> cen(3 * (size_t)n), box(6 * nb), C(8 * nb);
    std::vector<uint64_t> keys(n), flag(n + 1), flagEx(n + 1), wcnt(n + 1), wscan(n + 1);
    std::vector<int32_t> idx(n), child(n > 1 ? 2 * (size_t)(n - 1) : 2), pcount(nb), cl(n), cl2(n), nn(n), wbin(n + 1);
    std::vector<uint8_t> K(8 * nb), K8(nb);
    std::vector<uint32_t> wslot(8 * ((size_t)n + 1));
    GbView v{n, verts9, cen.data(), keys.data(), idx.data(), box.data(), child.data(), pcount.data(), C.data(), K.data(), K8.data(),
             cl.data(), cl2.data(), nn.data(), flag.data(), flagEx.data(), wbin.data(), wslot.data(), wcnt.data(), wscan.data()};
    auto exclusive = [](const uint64_t* in, uint64_t* o, int64_t count) {
        uint64_t s = 0;
        for (int64_t k = 0; k < count; k++) { o[k] = s; s += in[k]; }
    };
    // Morton order: the bounds of the finite centroid coordinates, as the device's bounds reduction takes them
    for (int i = 0; i < n; i++) gb_centroid(v, i);
    float clo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, chi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int i = 0; i < n; i++)
        for (int a = 0; a < 3; a++) {
            const float x = cen[3 * (size_t)i + a];
            if (!std::isfinite(x)) continue;
            clo[a] = x < clo[a] ? x : clo[a];
            chi[a] = chi[a] < x ? x : chi[a];
        }
    for (int i = 0; i < n; i++) gb_morton(v, i, clo, chi);
    std::stable_sort(idx.begin(), idx.end(), [&](int32_t a, int32_t b) { return keys[a] < keys[b]; });
    for (int b = 0; b < n; b++) gb_leaf(v, b);
    // PLOC
    int nc = n, next = n;
    while (nc > 1) {
        for (int i = 0; i < nc; i++) gb_nearest(v, i, nc);
        for (int i = 0; i < nc; i++) gb_flag(v, i, nc);
        exclusive(v.flag, v.flagEx, nc + 1);
        for (int i = 0; i < nc; i++) gb_merge(v, i, next);
        const uint64_t tot = v.flagEx[nc];
        if ((uint32_t)tot == 0) { *why = "no mutual nearest neighbours"; return DPRT_ERR_STATE; }
        nc = (int)(tot >> 32); next += (int)(uint32_t)tot;
        std::swap(v.cl, v.cl2);
    }
    const int root = n == 1 ? 0 : next - 1;
    // emission
    std::vector<int64_t> levels(1, 0), triBase(1, 0);
    v.wbin[0] = root;
    for (int64_t first = 0, last = 1; first < last;) {
        levels.push_back(last);
        for (int64_t g = first; g < last; g++) gb_emit_count(v, g, root);
        v.wcnt[last] = 0;
        exclusive(v.wcnt + first, v.wscan + first, last - first + 1);
        for (int64_t g = first; g < last; g++) gb_emit_items(v, g, last);
        const uint64_t tot = v.wscan[last];
        triBase.push_back(triBase.back() + (int64_t)(uint32_t)tot);
        first = last; last += (int64_t)(tot >> 32);
    }
    out.nodes.resize(levels.back());
    out.tris.resize(n);
    for (size_t k = 0; k + 1 < levels.size(); k++)
        for (int64_t g = levels[k]; g < levels[k + 1]; g++)
            gb_emit_write(v, g, levels[k + 1], triBase[k], mat_ids, nullptr, 0, pad, out.nodes.data(), out.tris.data(), nullptr);
    out.max_depth = (int)levels.size() - 1;
    for (int a = 0; a < 3; a++) { out.bounds[a] = FLT_MAX; out.bounds[3 + a] = -FLT_MAX; }
    for (int64_t k = 0; k < 3 * ntris; k++)
        for (int a = 0; a < 3; a++) {
            const float x = verts9[3 * k + a];
            out.bounds[a] = x < out.bounds[a] ? x : out.bounds[a];
            out.bounds[3 + a] = out.bounds[3 + a] < x ? x : out.bounds[3 + a];
        }
    return 0;
}

}  // namespace dprt
