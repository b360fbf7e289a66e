// bvh_node.cuh -- the rule that turns the exact boxes of a BVH8 node's children into the node's stored frame, exponents and
// quantised slot boxes. One definition for the host builder (bvh_build.cpp, plain g++) and for the refit (refit.cu: device
// kernels and the host specification dprt_spec_bvh8_refit), so that a refit of an unchanged chunk reproduces the build bit
// for bit (DESIGN.md 3.9). Below it, the SAH-optimal collapse to 8 wide and the slot assignment, shared by the host builder
// and the GPU builder (bvh_gpu_build.cu, DESIGN.md 3.10). Every step is exact or a single IEEE-rounded operation: compile
// without FMA contraction.
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>
#include "dprt_types.h"

#ifdef __CUDACC__
#define DPRT_NODE_HD __host__ __device__ __forceinline__
#else
#define DPRT_NODE_HD inline
#endif

namespace dprt {

// Smallest e with 255 * 2^e >= extent, clamped to [-126, 127], stored biased like an IEEE exponent (e + 127). Exact:
// extent = f 2^x with f in [0.5, 1) (frexp), and 255 2^(x-9) < 2^(x-1) <= extent < 255 2^(x-7), so e is x - 8 or x - 7.
DPRT_NODE_HD uint8_t bvh8_exponent(float extent) {
    if (!(extent > 0.f)) return 1;                 // 2^-126: degenerate axis
    if (!(extent <= FLT_MAX)) return 254;          // 2^127: clamped
    int x;
    frexp((double)extent, &x);
    int e = x - 8;
    if (ldexp(255.0, e) < (double)extent) e++;
    e = e < -126 ? -126 : (e > 127 ? 127 : e);
    return (uint8_t)(e + 127);
}

// Writes p, e and the six quantised bounds of every slot of `node` from the exact boxes lo[s], hi[s] of the slots in `used`
// (bit s); unused slots get the empty box. imask, tmask, childBase, triBase are left alone. box_lo / box_hi receive the
// exact box of the whole node (the union of the slot boxes): what its parent's slot needs.
//  - frame: the union padded by pad * 1.01 + extent / 8192 per axis, a little more than any slot is padded below, so that
//    no slot bound clamps;
//  - slot s: its box padded by pad + 2^-7 of a quantisation step (the slack of the traversal kernel's folded dequantisation,
//    bvh_traverse.cuh), rounded outwards to the 8-bit grid p + q 2^e, checked in double.
DPRT_NODE_HD void bvh8_encode_node(dprt_bvh8_node& node, const float (*lo)[3], const float (*hi)[3], uint32_t used, float pad,
                                   float* box_lo, float* box_hi) {
    float nlo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, nhi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int s = 0; s < 8; s++) {
        if (!((used >> s) & 1u)) continue;
        for (int a = 0; a < 3; a++) {
            nlo[a] = lo[s][a] < nlo[a] ? lo[s][a] : nlo[a];
            nhi[a] = hi[s][a] > nhi[a] ? hi[s][a] : nhi[a];
        }
    }
    for (int a = 0; a < 3; a++) {
        const float fp = pad * 1.01f + (nhi[a] - nlo[a]) * (1.0f / 8192.0f);
        const float plo = nlo[a] - fp, phi = nhi[a] + fp;
        node.p[a] = plo;
        node.e[a] = bvh8_exponent(phi - plo);
        box_lo[a] = nlo[a]; box_hi[a] = nhi[a];
    }
    uint8_t* qlo[3] = {node.qlox, node.qloy, node.qloz};
    uint8_t* qhi[3] = {node.qhix, node.qhiy, node.qhiz};
    for (int s = 0; s < 8; s++) {
        if (!((used >> s) & 1u)) {
            for (int a = 0; a < 3; a++) { qlo[a][s] = 255; qhi[a][s] = 0; }
            continue;
        }
        for (int a = 0; a < 3; a++) {
            const double sc = ldexp(1.0, (int)node.e[a] - 127);
            const double cpad = (double)pad + sc * (1.0 / 128.0);
            const double l = (double)lo[s][a] - cpad, h = (double)hi[s][a] + cpad;
            const double p0 = (double)node.p[a];
            int ql = (int)floor((l - p0) / sc);
            int qh = (int)ceil((h - p0) / sc);
            ql = ql < 0 ? 0 : (ql > 255 ? 255 : ql);
            qh = qh < 0 ? 0 : (qh > 255 ? 255 : qh);
            while (ql > 0 && p0 + ql * sc > l) ql--;
            while (qh < 255 && p0 + qh * sc < h) qh++;
            qlo[a][s] = (uint8_t)ql; qhi[a][s] = (uint8_t)qh;
        }
    }
}

// The padding of a chunk: 2^-16 of its largest absolute coordinate, at least 2^-16 (bvh8_build with pad < 0).
DPRT_NODE_HD float bvh8_chunk_pad(float max_abs) { return ldexpf(max_abs > 1.0f ? max_abs : 1.0f, -16); }

// ---- the SAH-optimal collapse of a binary tree to 8-wide nodes (Ylitie, Karras, Laine 2017, section 3.1) ------------------
// Shared by the host builder (bvh_build.cpp) and the GPU builder and its host twin (bvh_gpu_build.cu), so that both collapse
// by the same recurrence, the same float operations and the same slot assignment.
// C(n, i) = least SAH cost of representing the subtree of binary node n by at most i wide-BVH roots, a root being a wide
// internal node (cost cNode x area, its <= 8 children are roots of n's two subtrees) or a leaf slot with <= 3 triangles
// (cost cPrim x triangles x area):
//   C(n, 1) = min(leaf(n), cNode A_n + min_k C(left, k) + C(right, 8 - k))
//   C(n, i) = min(C(n, i - 1), min_k C(left, k) + C(right, i - k))
// Why the optimum: a wide node costs a ray a full node step however few of its eight slots it uses, and a collapse decided
// one node at a time leaves many nodes with two or three leaf children at the bottom of the tree. Minimising the cost over
// the whole subtree avoids them.
// cNode : cPrim = 4 : 1 is the trace kernel's issue-slot ratio of a node step to a triangle test (profiles/bvh_quality.py).
constexpr float kBvh8CostNode = 4.0f;
constexpr float kBvh8CostPrim = 1.0f;

// the half surface area of a box; 0 for an inverted (empty) box
DPRT_NODE_HD float bvh8_half_area(const float* lo, const float* hi) {
    float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    if (dx < 0 || dy < 0 || dz < 0) return 0.f;
    return dx * dy + dy * dz + dz * dx;
}

// Cost row of a binary leaf of `count` triangles and half area A: c[i - 1] = C(n, i), k[i - 1] = 1.
DPRT_NODE_HD void bvh8_dp_leaf(float A, int count, float* c, uint8_t* k) {
    for (int i = 0; i < 8; i++) { c[i] = A * (float)count * kBvh8CostPrim; k[i] = 1; }
}

// Cost row of an internal binary node of half area A with `pcount` triangles below it, from its children's rows cl, cr.
// k[0]: 1 = the subtree becomes one leaf slot, 2 = a wide node; k[i - 1], i >= 2: roots given to the left child, 0 = as for
// i - 1. Returns the roots a wide node rooted here gives its left child (the other 8 - K8 go to the right).
DPRT_NODE_HD uint8_t bvh8_dp_node(float A, int pcount, const float* cl, const float* cr, float* c, uint8_t* k) {
    float dist[9]; uint8_t dk[9];
    for (int j = 2; j <= 8; j++) {
        float best = FLT_MAX; int bk = 1;
        for (int x = 1; x < j; x++) { const float v = cl[x - 1] + cr[j - x - 1]; if (v < best) { best = v; bk = x; } }
        dist[j] = best; dk[j] = (uint8_t)bk;
    }
    const float cLeaf = pcount <= 3 ? A * (float)pcount * kBvh8CostPrim : FLT_MAX;
    const float cInt = dist[8] + A * kBvh8CostNode;
    c[0] = cInt < cLeaf ? cInt : cLeaf; k[0] = pcount <= 3 && cLeaf <= cInt ? 1 : 2;   // never a leaf slot of > 3, even when cInt overflows
    for (int i = 2; i <= 8; i++) {
        if (dist[i] < c[i - 2]) { c[i - 1] = dist[i]; k[i - 1] = dk[i]; } else { c[i - 1] = c[i - 2]; k[i - 1] = 0; }
    }
    return dk[8];
}

// A child of a wide node: binary node n, as a leaf slot (its <= 3 triangles) or as a wide node of its own.
struct Bvh8Child { int n; bool leaf; };

// The <= i roots that represent binary node n's subtree, left to right, appended to out[cnt..]. Tree: is_leaf(n), left(n),
// right(n) and k(n) (the 8 entries of n's k row).
template <class Tree>
DPRT_NODE_HD void bvh8_collect(const Tree& t, int n, int i, Bvh8Child* out, int& cnt) {
    int sn[16], si[16], sp = 0;                        // depth-first, left first; at most one entry per root still to emit
    sn[sp] = n; si[sp] = i; sp++;
    while (sp) {
        sp--;
        const int m = sn[sp], j = si[sp];
        if (t.is_leaf(m)) { out[cnt++] = Bvh8Child{m, true}; continue; }
        const uint8_t* K = t.k(m);
        if (j == 1) { out[cnt++] = Bvh8Child{m, K[0] == 1}; continue; }
        const int kk = K[j - 1];
        if (kk == 0) { sn[sp] = m; si[sp] = j - 1; sp++; continue; }
        sn[sp] = t.right(m); si[sp] = j - kk; sp++;
        sn[sp] = t.left(m); si[sp] = kk; sp++;
    }
}

// Greedy octant slot assignment of nch <= 8 children with exact boxes lo[c], hi[c]: slot_of[c] in 0..7. The node frame is
// the union of the children; each child goes to the free slot that best matches the direction from the frame's centre to
// its own (the traversal visits slots in an order derived from the ray's octant).
DPRT_NODE_HD void bvh8_assign_slots(const float (*lo)[3], const float (*hi)[3], int nch, int* slot_of) {
    float nlo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, nhi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int c = 0; c < nch; c++)
        for (int a = 0; a < 3; a++) { nlo[a] = lo[c][a] < nlo[a] ? lo[c][a] : nlo[a]; nhi[a] = nhi[a] < hi[c][a] ? hi[c][a] : nhi[a]; }
    float cost[8][8]; bool slot_used[8] = {false, false, false, false, false, false, false, false};
    bool child_done[8] = {false, false, false, false, false, false, false, false};
    float ncx[3];
    for (int a = 0; a < 3; a++) ncx[a] = 0.5f * (nlo[a] + nhi[a]);
    for (int c = 0; c < nch; c++) {
        float d[3];
        for (int a = 0; a < 3; a++) d[a] = 0.5f * (lo[c][a] + hi[c][a]) - ncx[a];
        for (int s = 0; s < 8; s++) {
            float sx = (s & 1) ? -1.f : 1.f, sy = (s & 2) ? -1.f : 1.f, sz = (s & 4) ? -1.f : 1.f;
            cost[c][s] = d[0] * sx + d[1] * sy + d[2] * sz;
        }
    }
    for (int k = 0; k < nch; k++) {
        int bc = -1, bs = -1; float bv = FLT_MAX;
        for (int c = 0; c < nch; c++) {
            if (child_done[c]) continue;
            for (int s = 0; s < 8; s++) {
                if (slot_used[s]) continue;
                if (cost[c][s] < bv) { bv = cost[c][s]; bc = c; bs = s; }
            }
        }
        if (bc < 0) {                                  // only non-finite or overflowing costs left: first child, first slot
            for (bc = 0; child_done[bc]; bc++) {}
            for (bs = 0; slot_used[bs]; bs++) {}
        }
        child_done[bc] = true; slot_used[bs] = true; slot_of[bc] = bs;
    }
}

}  // namespace dprt
