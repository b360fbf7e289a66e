// bvh_traverse.cuh -- traversal of the 80-byte compressed 8-wide BVH as a resumable per-lane state machine.
//
// This is what replaces optixTrace() (call sites: optix/kernel.cu:394, distributed_traversal_kernel.cu:245,
// shadow_ray_kernel.cu:177, secondary_ray_kernel.cu:200). Closest-hit results are independent of the BVH and
// of the traversal order: every candidate triangle goes through the watertight test of dprt_math.cuh and ties
// in t resolve to the lower primitive id. That freedom is what lets kernels.cu run the traversal as a
// persistent wavefront in which a lane that finishes its ray immediately picks up the next one.
#pragma once
#include "dprt_math.cuh"

namespace dprt {

// Byte j of a packed plane word -> the float 32768 + q, exactly: the byte lands in mantissa bits 8..15 of 2^15
// (ulp 2^-8). One PRMT with an immediate selector; `magic` = 0x47000000 arrives as a kernel argument so that ptxas
// cannot fold it: PRMT takes one immediate, and it has to be the selector -- with the constant in that slot the
// compiler spends a move per PRMT fetching the four selectors from uniform registers (48 moves per node).
template <int J>
DPRT_D float qbias(uint32_t w, uint32_t magic) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(magic), "n"(0x7604 | (J << 4)));
    return __uint_as_float(r);
}

#define DPRT_STACK 40

// instrumentation (dprt_enable_counters): BVH8 nodes fetched and triangles tested by one thread
struct TraceCount { uint32_t nodes, tris; };

struct Trav {
    // ray
    V3 o, d; float tmin;
    float idx, idy, idz;            // reciprocal direction (zero components nudged to +-1e-20)
    uint32_t octinv;                // 7 - octant
    // result so far (over all objects traced for this ray)
    float tbest;                    // closest accepted t; starts at the ray's tmax
    int   hitPrim, hitTri, hitObj;  // hitTri < 0: nothing yet
    float ha, hb;                   // barycentrics of the best hit (weights of v1, v2)
    // current object
    float tlimit;                   // strict upper bound for this object = tbest when the object was entered
    int   tiePrim;                  // lowest primitive id among this object's hits at tbest
    const uint4* nodes; const float4* tris;
    uint2 ng;                       // node group: child base, hit bits of internal children | imask
    uint2 tg;                       // pending triangle group: triangle base, leaf-triangle bits
    int sp;
};   // the traversal stack (uint2[DPRT_STACK]) is a separate local array so that this struct stays in registers

DPRT_D void trav_init_ray(Trav& s, V3 o, V3 d, float tmin, float tmax) {
    s.o = o; s.d = d; s.tmin = tmin;
    const float dxs = fabsf(d.x) > 1e-20f ? d.x : copysignf(1e-20f, d.x);
    const float dys = fabsf(d.y) > 1e-20f ? d.y : copysignf(1e-20f, d.y);
    const float dzs = fabsf(d.z) > 1e-20f ? d.z : copysignf(1e-20f, d.z);
    s.idx = 1.0f / dxs; s.idy = 1.0f / dys; s.idz = 1.0f / dzs;
    s.octinv = 7u - ((dxs < 0.0f ? 1u : 0u) | (dys < 0.0f ? 2u : 0u) | (dzs < 0.0f ? 4u : 0u));
    s.tbest = tmax; s.hitPrim = -1; s.hitTri = -1; s.hitObj = -1; s.ha = 0.f; s.hb = 0.f;
    s.ng = make_uint2(0u, 0u); s.tg = make_uint2(0u, 0u); s.sp = 0;      // no object entered yet: no work of either kind
}

DPRT_D void trav_enter_object(Trav& s, const uint4* nodes, const float4* tris) {
    s.nodes = nodes; s.tris = tris;
    s.tlimit = s.tbest; s.tiePrim = 0x7fffffff;
    s.ng = make_uint2(0u, 0x80000000u); s.tg = make_uint2(0u, 0u); s.sp = 0;
}

// The traversal is split in two phases. trav_node expands one node (8 child slabs) for the calling lane and
// leaves the leaf triangles it found in s.tg. Triangles are NOT tested by the lane that found them: the lanes of
// a warp append their (owner lane, triangle) pairs to a warp-wide queue in shared memory and, once 32 pairs are
// waiting, the whole warp tests 32 of them at once (tri_round), whichever rays they belong to. Node expansion
// runs with nearly all lanes busy and triangle tests run 32 wide, instead of 3-4 lanes wide when every lane
// tests its own leaf. tbest of a lane lags by the queueing delay, which only makes node culling conservative.
// Slab test of the 8 children of node `ni` against one ray: returns the node's child base / triangle base and the
// hit bits of its internal children (bits 24..31, octant order: higher bit = nearer) and of its leaf triangles (0..23).
// bit s -> bit s ^ o of an 8-bit mask (o = 7 - octant): three conditional swaps
DPRT_D uint32_t xor_permute8(uint32_t m, uint32_t o) {
    if (o & 1u) m = ((m & 0x55u) << 1) | ((m >> 1) & 0x55u);
    if (o & 2u) m = ((m & 0x33u) << 2) | ((m >> 2) & 0x33u);
    if (o & 4u) m = ((m & 0x0fu) << 4) | (m >> 4);
    return m;
}

// Slab test of the 8 children of node `ni` against one ray. Every child slot s owns a fixed pattern of bits -- 3 s .. 3 s + 2
// for its (at most three) leaf triangles, 24 + s for "internal child" -- so the per-child work after the slab test is one
// select of an immediate; the node's tmask / imask then keep the bits that exist, and the internal bits are moved to
// octant order (higher bit = nearer) for the whole node at once. Returns the child base / triangle base with those bits,
// and tmask: the triangle behind bit b is triBase + popc(tmask & ((1 << b) - 1)).
DPRT_D void expand_node(const uint4* __restrict__ nodes, uint32_t ni, float ox, float oy, float oz, float idx, float idy, float idz,
                        uint32_t octinv, float tmin, float tbest, uint32_t magic, uint2& ng, uint2& tg, uint32_t& tmask) {
    const uint4* np = nodes + 5 * (size_t)ni;
    const uint4 n0 = __ldg(np + 0), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
    const bool nx = !(octinv & 1u), ny = !(octinv & 2u), nz = !(octinv & 4u);

    const float adjx = __uint_as_float((n0.w & 0xffu) << 23) * idx;
    const float adjy = __uint_as_float(((n0.w >> 8) & 0xffu) << 23) * idy;
    const float adjz = __uint_as_float(((n0.w >> 16) & 0xffu) << 23) * idz;
    // plane distance t = (p + q 2^e - o) / d = q adj + org. The byte is dequantised as F = 32768 + q (qbias), so the
    // constant term carries the bias: t = F adj + (org - 32768 adj), one FFMA per plane. The folded constant is
    // rounded at magnitude 2^15 |adj|, i.e. to 2^-9 of a quantisation step: the builder pads every child box by
    // 2^-7 of a step for it (bvh_build.cpp), so the slab test stays conservative. Culling only -- accepted hits go
    // through the exact triangle test, results do not depend on this arithmetic.
    const float orgx = fmaf(-32768.0f, adjx, (__uint_as_float(n0.x) - ox) * idx);
    const float orgy = fmaf(-32768.0f, adjy, (__uint_as_float(n0.y) - oy) * idy);
    const float orgz = fmaf(-32768.0f, adjz, (__uint_as_float(n0.z) - oz) * idz);

    uint32_t acc = 0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const uint32_t lox = h ? (nx ? n3.w : n2.y) : (nx ? n3.z : n2.x);
        const uint32_t hix = h ? (nx ? n2.y : n3.w) : (nx ? n2.x : n3.z);
        const uint32_t loy = h ? (ny ? n4.y : n2.w) : (ny ? n4.x : n2.z);
        const uint32_t hiy = h ? (ny ? n2.w : n4.y) : (ny ? n2.z : n4.x);
        const uint32_t loz = h ? (nz ? n4.w : n3.y) : (nz ? n4.z : n3.x);
        const uint32_t hiz = h ? (nz ? n3.y : n4.w) : (nz ? n3.x : n4.z);
#define DPRT_CHILD(J)                                                                                   \
        {                                                                                               \
            const float tnx = fmaf(qbias<J>(lox, magic), adjx, orgx);                                   \
            const float tny = fmaf(qbias<J>(loy, magic), adjy, orgy);                                   \
            const float tnz = fmaf(qbias<J>(loz, magic), adjz, orgz);                                   \
            const float tfx = fmaf(qbias<J>(hix, magic), adjx, orgx);                                   \
            const float tfy = fmaf(qbias<J>(hiy, magic), adjy, orgy);                                   \
            const float tfz = fmaf(qbias<J>(hiz, magic), adjz, orgz);                                   \
            const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmin));                                  \
            const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tbest));                                 \
            constexpr uint32_t kSlot = 4u * h_ + J;                                                     \
            acc |= (tn <= tf) ? ((7u << (3u * kSlot)) | (1u << (24u + kSlot))) : 0u;                     \
        }
        if (h == 0) { constexpr uint32_t h_ = 0; DPRT_CHILD(0) DPRT_CHILD(1) DPRT_CHILD(2) DPRT_CHILD(3) }
        else        { constexpr uint32_t h_ = 1; DPRT_CHILD(0) DPRT_CHILD(1) DPRT_CHILD(2) DPRT_CHILD(3) }
#undef DPRT_CHILD
    }
    const uint32_t imask = n0.w >> 24;
    tmask = n1.z;
    ng = make_uint2(n1.x, (xor_permute8((acc >> 24) & imask, octinv) << 24) | imask);
    tg = make_uint2(n1.y, acc & tmask);
}

// index of the node that bit `bit` (24..31) of node group g stands for
DPRT_D uint32_t group_node(uint2 g, uint32_t bit, uint32_t octinv) {
    const uint32_t slot = (bit - 24u) ^ octinv;
    return g.x + __popc(g.y & 0xffu & ((1u << slot) - 1u));
}

// expands the nearest pending node of the lane; returns the node's tmask (the caller parks it in WarpQueue::tmask while
// the lane's triangle group s.tg is pending)
template <bool COUNT>
DPRT_D uint32_t trav_node(Trav& s, uint2* stack, TraceCount& cnt, const uint32_t magic) {
    const uint32_t bit = 31u - __clz(s.ng.y);
    const uint32_t ni = group_node(s.ng, bit, s.octinv);
    s.ng.y &= ~(1u << bit);
    if (s.ng.y & 0xff000000u) { if (s.sp < DPRT_STACK) stack[s.sp++] = s.ng; }
    if (COUNT) cnt.nodes++;
    uint32_t tmask;
    expand_node(s.nodes, ni, s.o.x, s.o.y, s.o.z, s.idx, s.idy, s.idz, s.octinv, s.tmin, s.tbest, magic, s.ng, s.tg, tmask);
    return tmask;
}

// ---- alpha cut-out (the __anyhit__ah program of every pipeline: kernel.cu:311-359, distributed_traversal_kernel.cu:110-158,
// shadow_ray_kernel.cu:42-90, secondary_ray_kernel.cu:66-114, vis / precom :33-81) ------------------------------------------
// A candidate intersection with a triangle whose material has a texture is dropped when the texture's opacity at the hit's
// texture coordinate is below 0.05 (optixIgnoreIntersection). Chunks uploaded with texture coordinates carry their triangle
// count in the w word of every triangle's third vector (0 otherwise: the test below is one compare on a register the
// intersection already loaded) and their per-corner coordinates behind the triangle array, 32 bytes per triangle.
struct TexCtx { const DevTexture* textures; const int32_t* matTex; };

__device__ __noinline__ bool alpha_cutout_ignored(const DevTexture* __restrict__ textures, const int32_t* __restrict__ matTex,
                                                   const float4* __restrict__ tris, int ntris, uint32_t ti, int matID, float al, float be) {
    const int tex = __ldg(matTex + matID);
    if (tex < 0) return false;
    const DevTexture T = textures[tex];
    if (T.texels == nullptr) return false;
    const float4* uv = tris + 3 * (size_t)ntris + 2 * (size_t)ti;
    const float4 a = __ldg(uv), b = __ldg(uv + 1);
    const float u = tex_interp(a.x, a.z, b.x, al, be), v = tex_interp(a.y, a.w, b.y, al, be);
    return tex_bilinear_alpha(T, u, v) < 0.05f;
}

// ---- warp-wide triangle queue -----------------------------------------------------------------------
#define DPRT_QCAP 128                      // queue capacity per warp (pairs)
#define DPRT_TRI_BITS 27                   // queue entry = owner lane << 27 | triangle index
#define DPRT_POOLCAP 1024                  // cooperative-mode node pool per warp (global scratch: shared memory is L1 capacity)
#define DPRT_POOLLIM 760                   // wide steps keep the pool below this; above it one node per step (DFS), which adds
                                           // at most 7 entries per tree level: 760 + 7 * 36 (deepest BVH accepted at upload) < 1024

struct WarpQueue {
    float4 rayA[32];                       // per owner lane: origin.xyz, tmin
    float4 rayB[32];                       // Sx, Sy, Sz, bits(kx | ky << 2 | kz << 4)
    float4 aux[32];                        // winner of a round: bits(tri index), alpha, beta, -
    unsigned long long key[32];            // min over a round of (bits(t) << 32 | prim); ~0 = no hit
    const float4* tris[32];                // triangle array of the owner's current object
    float  tlimit[32];                     // strict upper bound for the owner's current object
    int    cnt[32];                        // pairs of this owner tested in the round
    uint32_t tmask[32];                    // tmask of the node whose leaf triangles the lane's s.tg refers to
    uint32_t q[DPRT_QCAP];
    int    plen;                           // cooperative tail mode: pool length hand-over
};

DPRT_D void wq_set_ray(WarpQueue& w, int lane, const Trav& s) {
    w.rayA[lane] = make_float4(s.o.x, s.o.y, s.o.z, s.tmin);
    const RayShear rs = ray_shear(s.d);
    w.rayB[lane] = make_float4(rs.Sx, rs.Sy, rs.Sz, __uint_as_float((uint32_t)(rs.kx | (rs.ky << 2) | (rs.kz << 4))));
    w.key[lane] = ~0ull; w.cnt[lane] = 0;
}
DPRT_D void wq_set_object(WarpQueue& w, int lane, const Trav& s) { w.tris[lane] = s.tris; w.tlimit[lane] = s.tlimit; }

// Appends the pending triangles of all lanes (s.tg) to the queue, as far as they fit. Warp-synchronous.
DPRT_D void wq_append(WarpQueue& w, int& qlen, int lane, bool busy, Trav& s, int& pend) {
    const unsigned FULL = 0xffffffffu;
    const int c = busy ? __popc(s.tg.y) : 0;
    if (__ballot_sync(FULL, c > 0) == 0u) return;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
    const int total = __shfl_sync(FULL, incl, 31);
    int pos = qlen + incl - c;
    const uint32_t tm = w.tmask[lane];
    while (s.tg.y != 0u && busy && pos < DPRT_QCAP) {
        const uint32_t k = __ffs(s.tg.y) - 1u;
        s.tg.y &= s.tg.y - 1u;
        const uint32_t ti = s.tg.x + __popc(tm & ((1u << k) - 1u));
        w.q[pos++] = ((uint32_t)lane << DPRT_TRI_BITS) | ti;
        pend++;
    }
    qlen = min(DPRT_QCAP, qlen + total);
}

// Tests the last min(32, qlen) pairs of the queue with all lanes and hands the closest accepted hit of each owner
// back to it. ANY: the owner keeps the first accepted hit. Warp-synchronous; every lane of the warp must call it.
template <bool ANY, bool COUNT>
DPRT_D void tri_round(WarpQueue& w, int& qlen, int lane, Trav& s, int obj, int& pend, TraceCount& cnt, const TexCtx& tc) {
    __syncwarp();
    const int n = min(32, qlen);
    const bool valid = lane < n;
    const int e = qlen - n + lane;
    qlen -= n;
    unsigned long long key = ~0ull; int owner = 0; uint32_t ti = 0u; float al = 0.f, be = 0.f;
    if (valid) {
        const uint32_t ent = w.q[e];
        owner = (int)(ent >> DPRT_TRI_BITS); ti = ent & ((1u << DPRT_TRI_BITS) - 1u);
        const float4 ra = w.rayA[owner], rb = w.rayB[owner];
        const float4* tp = w.tris[owner] + 3 * (size_t)ti;
        const float4 a = __ldg(tp + 0), b = __ldg(tp + 1), c = __ldg(tp + 2);
        RayShear rs; const uint32_t kp = __float_as_uint(rb.w);
        rs.kx = (int)(kp & 3u); rs.ky = (int)((kp >> 2) & 3u); rs.kz = (int)((kp >> 4) & 3u); rs.Sx = rb.x; rs.Sy = rb.y; rs.Sz = rb.z;
        if (COUNT) cnt.tris++;
        float t;
        if (tri_intersect(rs, v3(ra.x, ra.y, ra.z), v3(a.x, a.y, a.z), v3(b.x, b.y, b.z), v3(c.x, c.y, c.z), ra.w, w.tlimit[owner], &t, &al, &be)) {
            const int nuv = __float_as_int(c.w);       // != 0: the chunk has texture coordinates (alpha cut-outs possible)
            if (nuv == 0 || !alpha_cutout_ignored(tc.textures, tc.matTex, w.tris[owner], nuv, ti, __float_as_int(b.w), al, be)) {
                key = ((unsigned long long)__float_as_uint(t) << 32) | (unsigned long long)(uint32_t)__float_as_int(a.w);
                atomicMin(&w.key[owner], key);
            }
        }
        atomicAdd(&w.cnt[owner], 1);
    }
    __syncwarp();
    if (valid && key != ~0ull && w.key[owner] == key) w.aux[owner] = make_float4(__uint_as_float(ti), al, be, 0.f);
    __syncwarp();
    const int mine = w.cnt[lane];
    if (mine) {
        pend -= mine; w.cnt[lane] = 0;
        const unsigned long long k = w.key[lane];
        if (k != ~0ull) {
            w.key[lane] = ~0ull;
            const float t = __uint_as_float((uint32_t)(k >> 32)); const int prim = (int)(uint32_t)k;
            const bool take = ANY ? (s.hitTri < 0) : (t < s.tbest || (t == s.tbest && prim < s.tiePrim));
            if (take) {
                const float4 x = w.aux[lane];
                s.tbest = t; s.tiePrim = prim; s.hitPrim = prim; s.hitTri = (int)__float_as_uint(x.x); s.hitObj = obj; s.ha = x.y; s.hb = x.z;
            }
        }
    }
    __syncwarp();
}


// ---- cooperative tail mode ----------------------------------------------------------------------------
// Once the ray queue is exhausted a warp is left with a few rays, and its running time is the node count of the
// longest one at one node per loop iteration (a grazing ray over the height field visits hundreds of nodes while 31
// lanes idle). coop_run() finishes the current object of ONE ray (owner lane L) with all 32 lanes: the owner's
// traversal stack becomes a shared pool of node indices, every lane expands one node per step, hit children go back
// to the pool, leaf triangles to the warp triangle queue (owner L), whose rounds feed the shrinking tbest back.
// Valid because the closest hit is the minimum over all accepted triangle tests in (t, primitive id) order and the
// any-hit answer is a flag: neither depends on the order in which nodes are visited.

// appends the pending triangles of all lanes (tg) to the queue on behalf of `owner`, as far as they fit; returns the
// number appended (warp-uniform)
DPRT_D int coop_append(WarpQueue& w, int& qlen, int lane, int owner, uint2& tg, uint32_t tm) {
    const unsigned FULL = 0xffffffffu;
    const int c = __popc(tg.y);
    if (__ballot_sync(FULL, c > 0) == 0u) return 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
    const int total = __shfl_sync(FULL, incl, 31);
    int pos = qlen + incl - c;
    while (tg.y != 0u && pos < DPRT_QCAP) {
        const uint32_t k = __ffs(tg.y) - 1u;
        tg.y &= tg.y - 1u;
        w.q[pos++] = ((uint32_t)owner << DPRT_TRI_BITS) | (tg.x + __popc(tm & ((1u << k) - 1u)));
    }
    const int before = qlen;
    qlen = min(DPRT_QCAP, qlen + total);
    return qlen - before;
}

template <bool ANY, bool COUNT>
DPRT_D void coop_run(WarpQueue& w, uint32_t* __restrict__ pool, int& qlen, int lane, int L, Trav& s, uint2* stack, int obj, int& pend,
                     bool& exh, TraceCount& cnt, const uint32_t magic, const TexCtx& tc) {
    const unsigned FULL = 0xffffffffu;
    while (qlen > 0) tri_round<ANY, COUNT>(w, qlen, lane, s, obj, pend, cnt, tc);     // every owner's queued pairs first
    // the owner's ray, in every lane's registers
    const float ox = __shfl_sync(FULL, s.o.x, L), oy = __shfl_sync(FULL, s.o.y, L), oz = __shfl_sync(FULL, s.o.z, L);
    const float idx = __shfl_sync(FULL, s.idx, L), idy = __shfl_sync(FULL, s.idy, L), idz = __shfl_sync(FULL, s.idz, L);
    const float tmin = __shfl_sync(FULL, s.tmin, L);
    const uint32_t octinv = __shfl_sync(FULL, s.octinv, L);
    const uint4* nodes = (const uint4*)(uintptr_t)__shfl_sync(FULL, (unsigned long long)(uintptr_t)s.nodes, L);
    float ct = __shfl_sync(FULL, s.tbest, L);
    uint2 ctg = make_uint2(0u, 0u);
    uint32_t ctm = 0u;                  // tmask of the node behind this lane's ctg
    if (lane == L) {
        int n = 0;
        for (int i = 0; i <= s.sp; i++) {                 // bottom of the stack first, the current group last (on top)
            const uint2 g = i < s.sp ? stack[i] : s.ng;
            uint32_t m = g.y & 0xff000000u;
            while (m) { const uint32_t bit = __ffs(m) - 1u; m &= m - 1u; pool[n++] = group_node(g, bit, octinv); }   // far first
        }
        w.plen = n;
        ctg = s.tg; ctm = w.tmask[lane];
        s.ng = make_uint2(0u, 0u); s.tg = make_uint2(0u, 0u); s.sp = 0;
    }
    __syncwarp();
    int plen = w.plen;
    for (;;) {
        const int added = coop_append(w, qlen, lane, L, ctg, ctm);
        if (lane == L) pend += added;
        const bool more = __ballot_sync(FULL, ctg.y != 0u) != 0u;
        if (qlen > 0 && (qlen >= 32 || more || plen == 0)) {
            tri_round<ANY, COUNT>(w, qlen, lane, s, obj, pend, cnt, tc);
            ct = __shfl_sync(FULL, s.tbest, L);
            if (ANY && __shfl_sync(FULL, (int)(s.hitTri >= 0), L)) {          // accepted: drop what is left of this ray
                qlen = 0; plen = 0; ctg.y = 0u;
                if (lane == L) pend = 0;
                break;
            }
            continue;
        }
        if (plen == 0) break;                                                  // pool, queue and pending groups are empty
        // every lane takes one node off the top of the pool (lane 0 the nearest), as many as are sure to fit back
        const int np = max(1, min(min(32, plen), (DPRT_POOLLIM - plen) >> 3));
        uint2 cg = make_uint2(0u, 0u);
        if (lane < np) {
            const uint32_t ni = pool[plen - 1 - lane];
            if (COUNT) cnt.nodes++;
            expand_node(nodes, ni, ox, oy, oz, idx, idy, idz, octinv, tmin, ct, magic, cg, ctg, ctm);
        }
        plen -= np;
        __syncwarp();
        const int c = __popc(cg.y >> 24);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
        const int total = __shfl_sync(FULL, incl, 31);
        int pos = plen + total - incl;                                          // lane 0's children end up on top
        uint32_t m = cg.y & 0xff000000u;
        while (m) { const uint32_t bit = __ffs(m) - 1u; m &= m - 1u; pool[pos++] = group_node(cg, bit, octinv); }
        plen += total;
        __syncwarp();
    }
    if (lane == L) exh = true;          // object exhausted: the caller's step (2) moves on to the next object / completes the ray
}

}  // namespace dprt
