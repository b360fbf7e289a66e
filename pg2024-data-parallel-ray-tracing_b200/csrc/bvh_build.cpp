// bvh_build.cpp -- host-side acceleration-structure build for one scene chunk.
//
// Replaces the OptiX GAS build the reference delegates to the driver (AccelerationStructure.handle,
// renderer.cpp:1832; the build itself is in the missing scene loader, SURVEY.md section 0 "L0").
// Binned-SAH binary BVH (leaves <= 3 triangles) -> SAH-optimal collapse to 8-wide nodes (dynamic programme) -> octant-ordered
// slot assignment -> conservative 8-bit quantisation into the 80-byte compressed wide BVH node
// (Ylitie, Karras, Laine 2017). The result of a closest-hit query does not depend on this structure
// (tie-break on primitive id, see DESIGN.md), so the oracle is free to use its own.
#include "bvh_build.h"
#include "bvh_node.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>

namespace dprt {

namespace {

struct Box {
    float lo[3], hi[3];
    void reset() {
        for (int a = 0; a < 3; a++) { lo[a] = std::numeric_limits<float>::max(); hi[a] = -std::numeric_limits<float>::max(); }
    }
    void grow(const Box& b) {
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], b.lo[a]); hi[a] = std::max(hi[a], b.hi[a]); }
    }
    void grow(const float* p) {
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p[a]); hi[a] = std::max(hi[a], p[a]); }
    }
    float half_area() const { return bvh8_half_area(lo, hi); }
};

struct Node2 {
    Box box;
    int left = -1, right = -1;   // children (internal)
    int first = 0, count = 0;    // primitive range (leaf when count > 0)
    int pfirst = 0, pcount = 0;  // primitive range of the whole subtree (every node)
};

struct Builder2 {
    const std::vector<Box>& pbox;
    const std::vector<float>& pcen;  // 3 per prim
    std::vector<int>& idx;
    std::vector<Node2>& nodes;
    std::atomic<int> nnodes{0};

    Builder2(const std::vector<Box>& b, const std::vector<float>& c, std::vector<int>& i, std::vector<Node2>& n)
        : pbox(b), pcen(c), idx(i), nodes(n) {}

    int alloc() { return nnodes.fetch_add(1); }

    void build(int ni, int first, int count, int depth) {
        Node2& node = nodes[ni];
        Box bb, cb; bb.reset(); cb.reset();
        for (int i = first; i < first + count; i++) {
            int p = idx[i];
            bb.grow(pbox[p]);
            cb.grow(&pcen[3 * (size_t)p]);
        }
        node.box = bb;
        node.pfirst = first; node.pcount = count;
        if (count <= 3) { node.first = first; node.count = count; return; }

        constexpr int NB = 16, NBMAX = NB;
        int best_axis = -1, best_split = -1; float best_cost = std::numeric_limits<float>::max();
        for (int a = 0; a < 3; a++) {
            float ext = cb.hi[a] - cb.lo[a];
            if (!(ext > 0.f)) continue;
            Box bins[NBMAX]; int cnt[NBMAX];
            for (int b = 0; b < NB; b++) { bins[b].reset(); cnt[b] = 0; }
            float scale = NB / ext;
            for (int i = first; i < first + count; i++) {
                int p = idx[i];
                int b = (int)((pcen[3 * (size_t)p + a] - cb.lo[a]) * scale);
                b = std::min(NB - 1, std::max(0, b));
                bins[b].grow(pbox[p]); cnt[b]++;
            }
            float rarea[NBMAX]; int rcnt[NBMAX];
            Box acc; acc.reset(); int c = 0;
            for (int b = NB - 1; b > 0; b--) { acc.grow(bins[b]); c += cnt[b]; rarea[b] = acc.half_area(); rcnt[b] = c; }
            acc.reset(); c = 0;
            for (int b = 0; b < NB - 1; b++) {
                acc.grow(bins[b]); c += cnt[b];
                if (c == 0 || rcnt[b + 1] == 0) continue;
                float cost = acc.half_area() * c + rarea[b + 1] * rcnt[b + 1];
                if (cost < best_cost) { best_cost = cost; best_axis = a; best_split = b; }
            }
        }
        int mid;
        if (best_axis >= 0) {
            float ext = cb.hi[best_axis] - cb.lo[best_axis];
            float scale = NB / ext, lo = cb.lo[best_axis];
            int a = best_axis, sp = best_split;
            auto it = std::partition(idx.begin() + first, idx.begin() + first + count, [&](int p) {
                int b = (int)((pcen[3 * (size_t)p + a] - lo) * scale);
                b = std::min(NB - 1, std::max(0, b));
                return b <= sp;
            });
            mid = (int)(it - idx.begin());
        } else {
            mid = first + count / 2;
        }
        if (mid == first || mid == first + count) mid = first + count / 2;

        int l = alloc(), r = alloc();
        node.left = l; node.right = r; node.count = 0;
        int lc = mid - first, rc = first + count - mid;
        if (count > 32768) {
#pragma omp task shared(nodes) firstprivate(l, first, lc, depth)
            build(l, first, lc, depth + 1);
#pragma omp task shared(nodes) firstprivate(r, mid, rc, depth)
            build(r, mid, rc, depth + 1);
#pragma omp taskwait
        } else {
            build(l, first, lc, depth + 1);
            build(r, mid, rc, depth + 1);
        }
    }
};

}  // namespace

int bvh8_build(const float* verts, const int32_t* mat_ids, int64_t ntris64, float pad, Bvh8& out) {
    out.nodes.clear(); out.tris.clear(); out.max_depth = 0;
    if (ntris64 <= 0 || ntris64 > (int64_t)0x3fffffff || !verts) return -1;
    const int ntris = (int)ntris64;

    std::vector<Box> pbox(ntris);
    std::vector<float> pcen(3 * (size_t)ntris);
    Box scene; scene.reset();
#pragma omp parallel for schedule(static)
    for (int i = 0; i < ntris; i++) {
        Box b; b.reset();
        const float* v = verts + 9 * (size_t)i;
        b.grow(v); b.grow(v + 3); b.grow(v + 6);
        pbox[i] = b;
        for (int a = 0; a < 3; a++) pcen[3 * (size_t)i + a] = 0.5f * (b.lo[a] + b.hi[a]);
    }
    for (int i = 0; i < ntris; i++) scene.grow(pbox[i]);
    if (pad < 0.f) {
        float m = 0.f;
        for (int a = 0; a < 3; a++) m = std::max(m, std::max(std::fabs(scene.lo[a]), std::fabs(scene.hi[a])));
        pad = bvh8_chunk_pad(m);
    }
    for (int a = 0; a < 3; a++) { out.bounds[a] = scene.lo[a]; out.bounds[3 + a] = scene.hi[a]; }

    std::vector<int> idx(ntris);
    for (int i = 0; i < ntris; i++) idx[i] = i;
    std::vector<Node2> n2(2 * (size_t)ntris + 1);
    Builder2 b2(pbox, pcen, idx, n2);
    int root = b2.alloc();
#pragma omp parallel
    {
#pragma omp single
        b2.build(root, 0, ntris, 0);
    }

    // ---- collapse to 8-wide: the SAH-optimal choice by dynamic programming (bvh_node.cuh) ----
    const int nn = b2.nnodes.load();
    std::vector<float> C((size_t)nn * 8);          // C[n * 8 + i - 1]
    std::vector<uint8_t> K((size_t)nn * 8);        // i = 1: 1 = leaf, 2 = wide node; i >= 2: roots given to the left child, 0 = as for i - 1
    std::vector<uint8_t> K8((size_t)nn);           // wide node rooted at n: roots given to its left child
    for (int n = nn - 1; n >= 0; n--) {            // children are allocated after their parent: decreasing index = bottom-up
        const Node2& nd = n2[n];
        const float A = nd.box.half_area();
        float* c = &C[(size_t)n * 8]; uint8_t* k = &K[(size_t)n * 8];
        if (nd.count > 0) { bvh8_dp_leaf(A, nd.count, c, k); continue; }
        K8[n] = bvh8_dp_node(A, nd.pcount, &C[(size_t)nd.left * 8], &C[(size_t)nd.right * 8], c, k);
    }
    struct Tree {
        const std::vector<Node2>& n2; const std::vector<uint8_t>& K;
        bool is_leaf(int n) const { return n2[n].count > 0; }
        int left(int n) const { return n2[n].left; }
        int right(int n) const { return n2[n].right; }
        const uint8_t* k(int n) const { return &K[(size_t)n * 8]; }
    } tree{n2, K};

    // BFS so that the internal children of a node are contiguous
    struct Item { int n2; int out; int depth; };
    std::vector<Item> queue;
    out.nodes.resize(1);
    queue.push_back({root, 0, 1});
    out.tris.reserve(ntris);
    size_t qh = 0;
    while (qh < queue.size()) {
        Item it = queue[qh++];
        out.max_depth = std::max(out.max_depth, it.depth);
        const Node2& nd = n2[it.n2];
        Bvh8Child ch[8]; int nch = 0;
        if (nd.count > 0 || (it.n2 == root && K[(size_t)root * 8] == 1)) ch[nch++] = Bvh8Child{it.n2, true};     // a root that is itself a leaf
        else { bvh8_collect(tree, nd.left, K8[it.n2], ch, nch); bvh8_collect(tree, nd.right, 8 - K8[it.n2], ch, nch); }
        float clo[8][3], chi[8][3]; int slot_of[8];
        for (int c = 0; c < nch; c++)
            for (int a = 0; a < 3; a++) { clo[c][a] = n2[ch[c].n].box.lo[a]; chi[c][a] = n2[ch[c].n].box.hi[a]; }
        bvh8_assign_slots(clo, chi, nch, slot_of);
        int child_in_slot[8]; bool leaf_in_slot[8];
        for (int s = 0; s < 8; s++) { child_in_slot[s] = -1; leaf_in_slot[s] = false; }
        for (int c = 0; c < nch; c++) { child_in_slot[slot_of[c]] = ch[c].n; leaf_in_slot[slot_of[c]] = ch[c].leaf; }

        dprt_bvh8_node node;
        std::memset(&node, 0, sizeof(node));
        float slo[8][3], shi[8][3];
        uint32_t used = 0;
        node.triBase = (uint32_t)out.tris.size();
        int ninternal = 0;
        for (int s = 0; s < 8; s++)
            if (child_in_slot[s] >= 0 && !leaf_in_slot[s]) ninternal++;
        node.childBase = (uint32_t)out.nodes.size();
        if (ninternal) out.nodes.resize(out.nodes.size() + ninternal);
        int irank = 0, toff = 0;
        for (int s = 0; s < 8; s++) {
            int c = child_in_slot[s];
            if (c < 0) continue;
            const Node2& cn = n2[c];
            if (!leaf_in_slot[s]) {
                node.imask |= (uint8_t)(1u << s);
                queue.push_back({c, (int)node.childBase + irank, it.depth + 1});
                irank++;
            } else {
                const int lcount = cn.pcount;            // <= 3: a binary leaf, or a subtree the collapse turned into one leaf slot
                uint8_t unary = lcount == 1 ? 1 : (lcount == 2 ? 3 : 7);
                node.tmask |= (uint32_t)unary << (3 * s);
                for (int k = 0; k < lcount; k++) {
                    int p = idx[cn.pfirst + k];
                    dprt_bvh8_tri t;
                    const float* v = verts + 9 * (size_t)p;
                    std::memcpy(t.v0, v, 12); std::memcpy(t.v1, v + 3, 12); std::memcpy(t.v2, v + 6, 12);
                    t.primID = p; t.matID = mat_ids ? mat_ids[p] : 0; t.pad_ = 0;
                    out.tris.push_back(t);
                }
                toff += lcount;
            }
            used |= 1u << s;
            for (int a = 0; a < 3; a++) { slo[s][a] = cn.box.lo[a]; shi[s][a] = cn.box.hi[a]; }
        }
        float nlo[3], nhi[3];
        bvh8_encode_node(node, slo, shi, used, pad, nlo, nhi);
        out.nodes[it.out] = node;
    }
    return 0;
}

}  // namespace dprt
