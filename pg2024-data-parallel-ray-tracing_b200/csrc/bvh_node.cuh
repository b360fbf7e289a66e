// bvh_node.cuh -- the rule that turns the exact boxes of a BVH8 node's children into the node's stored frame, exponents and
// quantised slot boxes. One definition for the host builder (bvh_build.cpp, plain g++) and for the refit (refit.cu: device
// kernels and the host specification dprt_spec_bvh8_refit), so that a refit of an unchanged chunk reproduces the build bit
// for bit (DESIGN.md 3.9). Every step is exact or a single IEEE-rounded operation: compile without FMA contraction.
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

}  // namespace dprt
