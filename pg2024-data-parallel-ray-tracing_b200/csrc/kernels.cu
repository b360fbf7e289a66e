// kernels.cu -- the ray-tracing stage kernels of the per-bounce loop (sm_100a).
//
//   path_gen_kernel                 <- optix/path_gen_kernel.cu:46-105              (PathGen raygen)
//   trace_kernel<TM_TRAVERSE>  + traverse_post_kernel   <- optix/distributed_traversal_kernel.cu:215-340 (TraRay)
//   trace_kernel<TM_SHADE>     + shade_post_kernel      <- optix/kernel.cu:362-466 + closest hit :171-300 (MainRay)
//   trace_kernel<TM_SHADOW>   [+ shadow_post_kernel]    <- optix/shadow_ray_kernel.cu:150-355            (ShadowRay; post kernel with proxies only)
//   trace_kernel<TM_SECONDARY> + secondary_post_kernel  <- optix/secondary_ray_kernel.cu:172-369         (SecondaryRay)
//   trace_kernel<TM_RAYS>           <- a bare optixTrace closest-hit launch (BASELINE config 2)
//
// Every stage is split the way the hardware wants it: the optixTrace part runs in ONE persistent wavefront
// kernel (trace_kernel) whose warps pull rays from a global queue and refill lanes as soon as their ray is done
// (rays of very different length share a warp without idling it), and the per-path program around the trace
// (routing, shading, proxy march) runs as a fully coherent one-thread-per-path kernel over the same records.
// Compiled with --fmad=false: the arithmetic is the specification in dprt_math.cuh.
#include "dprt_internal.cuh"
#include <algorithm>
#include <cstdlib>
#include "bvh_traverse.cuh"
#include "plastic.cuh"

namespace dprt {

namespace {

constexpr int kBlock = 128;

struct PathRegs {
    V3 origin, direction; float tMax; V3 throughput;
    int pixelIndex, shadowPathID; uint32_t visitedMask; int currentNode, targetNode; uint32_t flags;
};
// flag bytes: isShadowRay | isDelta<<8 | isValid<<16 | isHit<<24
constexpr uint32_t F_SHADOW = 1u, F_DELTA = 1u << 8, F_VALID = 1u << 16, F_HIT = 1u << 24;

DPRT_D PathRegs load_path(const dprt_path_record* p) {
    const float4* q = reinterpret_cast<const float4*>(p);
    float4 a = q[0], b = q[1], c = q[2], d = q[3];
    PathRegs r;
    r.origin = v3(a.x, a.y, a.z); r.direction = v3(a.w, b.x, b.y); r.tMax = b.z;
    r.throughput = v3(b.w, c.x, c.y);
    r.pixelIndex = __float_as_int(c.z); r.shadowPathID = __float_as_int(c.w);
    r.visitedMask = __float_as_uint(d.x); r.currentNode = __float_as_int(d.y);
    r.targetNode = __float_as_int(d.z); r.flags = __float_as_uint(d.w);
    return r;
}
DPRT_D void store_path(dprt_path_record* p, const PathRegs& r) {
    float4* q = reinterpret_cast<float4*>(p);
    q[0] = make_float4(r.origin.x, r.origin.y, r.origin.z, r.direction.x);
    q[1] = make_float4(r.direction.y, r.direction.z, r.tMax, r.throughput.x);
    q[2] = make_float4(r.throughput.y, r.throughput.z, __int_as_float(r.pixelIndex), __int_as_float(r.shadowPathID));
    q[3] = make_float4(__uint_as_float(r.visitedMask), __int_as_float(r.currentNode), __int_as_float(r.targetNode),
                       __uint_as_float(r.flags));
}
DPRT_D void store_zero_path(dprt_path_record* p) {
    float4* q = reinterpret_cast<float4*>(p);
    float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    q[0] = z; q[1] = z; q[2] = z; q[3] = z;
}

// calculateEnvironmentLighting (distributed_traversal_kernel.cu:82-103, kernel.cu:28-48): the reference looks a lat-long
// texture up at (phi/2pi, theta/pi) -- env_map_lookup when dprt_set_env_map installed one; the synthetic benchmark scenes
// have none and use the analytic sky Le = envColor*(0.5+0.5*d.z).
DPRT_D V3 env_radiance(const DevParams& p, V3 d) {
    if (p.envMap.texels) {           // dprt_set_env_map: params.envLightTexture
        const float4 e = env_map_lookup(p.envMap, p.envRotation, d);
        return v3(e.x, e.y, e.z);
    }
    float w = fmaf(0.5f, d.z, 0.5f);
    return v3(p.envColor[0] * w, p.envColor[1] * w, p.envColor[2] * w);
}
DPRT_D void add_env(const DevParams& p, PathRegs& path) {
    path.throughput = v3mul(path.throughput, env_radiance(p, path.direction));
    const int px = path.pixelIndex * 3;
    p.env[px + 0] += path.throughput.x;   // one live path per pixel per rank: non-atomic like the reference (:332-334)
    p.env[px + 1] += path.throughput.y;
    p.env[px + 2] += path.throughput.z;
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) path_gen_kernel(DevParams p, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int width = p.camera.width;
    const int pixel = p.pathGenMode == 1 ? i * p.worldSize + p.worldID : i;
    const int row = pixel / width, col = pixel - row * width;
    uint32_t seed = tea4((uint32_t)pixel, (uint32_t)p.sampleCount);
    const float xi1 = rnd(seed), xi2 = rnd(seed);
    // Camera::generateRay(row, col, xi): pinhole through the jittered pixel position
    const float a = fmaf(2.0f, ((float)col + xi1) / (float)width, -1.0f);
    const float b = fmaf(-2.0f, ((float)row + xi2) / (float)p.camera.height, 1.0f);
    const dprt_camera& c = p.camera;
    V3 dir = v3(fmaf(c.U[0], a, fmaf(c.V[0], b, c.W[0])), fmaf(c.U[1], a, fmaf(c.V[1], b, c.W[1])),
                fmaf(c.U[2], a, fmaf(c.V[2], b, c.W[2])));
    PathRegs r;
    r.origin = v3(c.origin[0], c.origin[1], c.origin[2]);
    r.direction = v3normalized(dir);
    r.tMax = FLT_MAX;
    r.throughput = v3(1.f, 1.f, 1.f);
    r.pixelIndex = pixel; r.shadowPathID = -1; r.visitedMask = 0u; r.currentNode = -1; r.targetNode = -1;
    r.flags = F_VALID;
    store_path(p.paths + i, r);
}

// ------------------------------------------------------------------------------------------------
// ================================================================================================
// Persistent wavefront trace.
//
// begin(i): read what the ray needs from record i (48 of its 64 bytes) and enter the first local object.
// step:     bvh_traverse.cuh, until the last local object is exhausted (closest hit) or a triangle is accepted (any hit).
// end(i):   write the few words the stage needs (tMax/currentNode/isHit, or a 32-byte hit record for shading).
// A warp refills its idle lanes from the queue whenever at least kRefill of them are idle.
enum TraceMode { TM_TRAVERSE = 0, TM_SHADE = 1, TM_SHADOW = 2, TM_SECONDARY = 3, TM_RAYS = 4 };

constexpr int kTraceBlock = 128;
#ifndef DPRT_TRACE_MINBLOCKS
#define DPRT_TRACE_MINBLOCKS 6
#endif
constexpr int kTraceBlocksPerSM = DPRT_TRACE_MINBLOCKS;
constexpr int kNodesPerStepDefault = 2;
constexpr int kRefillDefault = 12;
constexpr int kTriVoteDefault = 8;
constexpr int kCoopDefault = 8;
constexpr int kRaysPerLaneDefault = 1;

template <int MODE> struct StageOf;
template <> struct StageOf<TM_TRAVERSE> { static constexpr int id = DPRT_STAGE_TRAVERSE; };
template <> struct StageOf<TM_SHADE> { static constexpr int id = DPRT_STAGE_SHADE; };
template <> struct StageOf<TM_SHADOW> { static constexpr int id = DPRT_STAGE_SHADOW_TRACE; };
template <> struct StageOf<TM_SECONDARY> { static constexpr int id = DPRT_STAGE_SECONDARY_TRACE; };
template <> struct StageOf<TM_RAYS> { static constexpr int id = DPRT_STAGE_TRACE_CLOSEST; };

struct TraceArgs {
    const DevObject* objects; int sceneSize; int worldID;
    dprt_path_record* recs;          // first record of the launch (paths, or paths + pathSize for shadow rays)
    HitRec* hits;                    // TM_SHADE
    const dprt_ray* rays; dprt_hit* rayHits;   // TM_RAYS
    int32_t* hitPrim;                // parity aid (may be null)
    int32_t* queue;                  // ray queue head
    unsigned long long* counters;
    int refill;                      // refill a warp when at least this many lanes are idle
    int triVote;                     // force a triangle round when at least this many busy lanes cannot expand a node
    uint32_t prmtMagic;              // 0x47000000 (bvh_traverse.cuh qbias): a run-time value on purpose
    uint32_t* coopPool;              // DPRT_POOLCAP words per resident warp
    int coop;                        // tail: a warp left with at most this many rays finishes them one at a time, 32 lanes per ray
    int nodesPerStep;                // a lane expands up to this many nodes per warp step while it finds no leaf triangles
    HitRec* hitCache; uint32_t epoch; unsigned long long* cacheHits;   // DevParams::hitCache (null = off)
    const DevTexture* textures; const int32_t* matTex;      // alpha cut-outs (bvh_traverse.cuh: alpha_cutout_ignored)
    // TM_SHADOW with proxies off: an unoccluded ray adds its term to directLightingBuffer here (shadow_add_direct); null = the
    // post kernel does it
    float* direct; int frameBufferSize; int spc;
};

// next local object at or after `from` that the ray still has to visit; sceneSize when none
DPRT_D int next_object(const TraceArgs& a, int from, uint32_t skipMask) {
    for (int k = from; k < a.sceneSize; k++) {
        const DevObject& ob = a.objects[k];
        if (ob.isProxy) continue;
        if ((skipMask >> ob.nodeID) & 1u) continue;
        return k;
    }
    return a.sceneSize;
}


// end(idx): what the stage keeps of a finished ray
template <int MODE>
DPRT_D void trace_end(const TraceArgs& a, int idx, const Trav& s, uint32_t flags) {
    const bool hit = s.hitTri >= 0;
    if (MODE == TM_TRAVERSE || MODE == TM_SECONDARY || MODE == TM_SHADE) {
        // TraRay / SecondaryRay: the result goes to hits[idx] (32 coalesced bytes); the post kernel, which rewrites the whole
        // record anyway, folds it in (tMax / currentNode / isHit) and files it in the hit cache under the pixel -- no
        // dependent record read and no scattered 4-byte stores in here. MainRay: hits[idx] is what the shading program reads.
        float4* h = reinterpret_cast<float4*>(a.hits + idx);
        h[0] = make_float4(s.tbest, __int_as_float(hit ? s.hitPrim : -1), __int_as_float(s.hitTri), __int_as_float(s.hitObj));
        h[1] = make_float4(s.ha, s.hb, 0.f, 0.f);
    } else if (MODE == TM_SHADOW) {
        if (hit) {    // any local occluder kills the shadow path (shadow_ray_kernel.cu:169-195)
            flags = (flags | F_HIT) & ~F_VALID;
            reinterpret_cast<uint32_t*>(a.recs + idx)[15] = flags;
        }
    } else {
        reinterpret_cast<float2*>(a.rayHits)[idx] = make_float2(s.tbest, __int_as_float(hit ? s.hitPrim : -1));
    }
}

// ShadowRay with proxies off (shadow_ray_kernel.cu:344-349): remote chunks are transparent to shadow rays, so a ray the
// any-hit trace left unoccluded adds its contribution. Plain load-add-store, not a float atomic: red.add.f32 flushes
// subnormal terms to zero. Each (pixel, plane) has exactly one shadow record per launch, so there is one writer.
DPRT_D void shadow_add_direct(const TraceArgs& a, int rec) {
    const float4* q = reinterpret_cast<const float4*>(a.recs + rec);
    const float tx = q[1].w;
    const float4 q2 = q[2];
    const size_t px = ((size_t)a.frameBufferSize * __float_as_int(q2.w) + __float_as_int(q2.z)) * 3;
    const float inv = (float)a.spc;
    a.direct[px + 0] += tx / inv;
    a.direct[px + 1] += q2.x / inv;
    a.direct[px + 2] += q2.y / inv;
}

// The unoccluded records a warp finished, queued in shared memory (lits[0..nlit)) so that their record and directLighting
// loads happen together, one record per lane, instead of stalling the warp each time one lane finishes a ray. Warp-uniform.
DPRT_D void shadow_flush(const TraceArgs& a, const int32_t* lits, int nlit, int lane) {
    __syncwarp();
    for (int k = lane; k < nlit; k += 32) shadow_add_direct(a, lits[k]);
    __syncwarp();
}

// Resident blocks per SM = register budget. The any-hit (shadow) trace has the shortest dependency chains per ray and gains
// from a seventh block (72 registers, ~70 bytes of spills); the closest-hit modes lose more to the spills than they gain
// (profiles/ab_r1d_regs.txt).
template <int MODE> constexpr int trace_min_blocks() { return MODE == 2 ? (kTraceBlocksPerSM == 6 ? 7 : kTraceBlocksPerSM) : kTraceBlocksPerSM; }

template <int MODE, bool COUNT>
__global__ void __launch_bounds__(kTraceBlock, trace_min_blocks<MODE>()) trace_kernel(TraceArgs a, int n) {
    constexpr bool ANY = MODE == TM_SHADOW;
    const unsigned FULL = 0xffffffffu;
    __shared__ WarpQueue s_wq[kTraceBlock / 32];
    __shared__ int32_t s_lits[ANY ? kTraceBlock / 32 * 64 : 1];      // TM_SHADOW: unoccluded records not yet added (shadow_flush)
    WarpQueue& w = s_wq[threadIdx.x >> 5];
    int32_t* lits = s_lits + (ANY ? (threadIdx.x >> 5) * 64 : 0);
    int nlit = 0;                    // warp-uniform: entries of lits (< 32 between steps; a step adds at most 32)
    const int lane = threadIdx.x & 31;
    const TexCtx tc = {a.textures, a.matTex};
    Trav s;
    uint2 stack[DPRT_STACK];
    int idx = -1, obj = 0, pend = 0;
    bool exh = false;                // the current object has no node work left (triangles may still be queued)
    uint32_t skipMask = 0u, flags = 0u;
    bool retry = false;              // TM_SHADE: the bounded trace may be repeated unbounded
    uint32_t cached = 0u;            // TM_SHADE: queries answered from the hit cache
    uint32_t walked = 0u;            // rays of this lane that entered at least one local object
    TraceCount cnt = {0u, 0u};
    bool exhausted = false;          // warp-uniform: the ray queue has no more rays
    int qlen = 0;                    // warp-uniform: pairs waiting in the triangle queue
    const int kRefill = a.refill;

    for (;;) {
        // ---- refill idle lanes: one atomic per refill reserves exactly the rays the idle lanes need ----
        const unsigned idle = __ballot_sync(FULL, idx < 0);
        if (!exhausted && __popc(idle) >= kRefill) {
            const int leader = __ffs(idle) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(a.queue, __popc(idle));
            base = __shfl_sync(FULL, base, leader);
            if (base + __popc(idle) >= n) exhausted = true;
            const int my = base + __popc(idle & ((1u << lane) - 1u));
            if (idx < 0 && my < n) {
                V3 o, d; float tmin = DPRT_EPSILON, tmax; bool live = true;
                skipMask = 0u; retry = false;
                if (MODE == TM_RAYS) {
                    const float4 r0 = __ldg(reinterpret_cast<const float4*>(a.rays) + 2 * (size_t)my);
                    const float4 r1 = __ldg(reinterpret_cast<const float4*>(a.rays) + 2 * (size_t)my + 1);
                    o = v3(r0.x, r0.y, r0.z); tmin = r0.w; d = v3(r1.x, r1.y, r1.z); tmax = r1.w;
                } else {
                    const float4* q = reinterpret_cast<const float4*>(a.recs + my);
                    const float4 q0 = q[0], q1 = q[1], q3 = q[3];
                    o = v3(q0.x, q0.y, q0.z); d = v3(q0.w, q1.x, q1.y); tmax = q1.z;
                    flags = __float_as_uint(q3.w);
                    live = (flags & F_VALID) != 0u;
                    if (MODE == TM_TRAVERSE) skipMask = __float_as_uint(q3.x);
                    if (MODE == TM_SHADE && live && a.hitCache) {
                        // Hit cache: when TraRay / SecondaryRay already found the closest hit of this very ray (same pixel,
                        // same bounce of the same sample = same epoch) on this rank's geometry, the re-trace of kernel.cu:382-413
                        // would return exactly that record (same candidates, same arithmetic, same tie rule): reuse it.
                        const int pixel = __float_as_int(q[2].z);
                        const float4* c = reinterpret_cast<const float4*>(a.hitCache + pixel);
                        const float4 c1 = c[1];
                        if (__float_as_uint(c1.z) == a.epoch) {
                            float4* h = reinterpret_cast<float4*>(a.hits + my);
                            h[0] = c[0]; h[1] = c1;
                            live = false; cached++;
                        }
                    }
                    if (MODE == TM_SHADE) {
                        // The reference re-traces with tMax = infinity (kernel.cu:382-413). When the record says "hit on
                        // this rank at tMax", the closest local hit is at t <= tMax: a trace bounded by the next float
                        // above tMax returns the very same (t, prim, barycentrics) while culling part of the BVH.
                        // A bounded trace that finds nothing is repeated unbounded, so the hint never changes a result.
                        const int currentNode = __float_as_int(q3.y);
                        if ((flags & F_HIT) && currentNode == a.worldID && tmax > 0.0f && tmax < FLT_MAX) {
                            tmax = __uint_as_float(__float_as_uint(tmax) + 1u); retry = true;
                        } else {
                            tmax = FLT_MAX;
                        }
                    }
                }
                if (live) {
                    idx = my; pend = 0; exh = false;
                    trav_init_ray(s, o, d, tmin, tmax);
                    wq_set_ray(w, lane, s);
                    obj = next_object(a, 0, skipMask);
                    if (obj < a.sceneSize) { trav_enter_object(s, a.objects[obj].nodes, a.objects[obj].tris); wq_set_object(w, lane, s); walked++; }
                }
            }
        }
        const unsigned act = __ballot_sync(FULL, idx >= 0);
        if (act == 0u) { if (exhausted) break; continue; }

        // ---- traverse until too few lanes are busy ----
        const int minBusy = exhausted ? 1 : (32 - kRefill + 1);
        do {
            // (1) leaf triangles found by the last node phase go to the warp queue
            wq_append(w, qlen, lane, idx >= 0, s, pend);
            // (2) pop / object switch / ray completion
            int lit = -1;                // TM_SHADOW: record of an unoccluded ray that finished in this step
            if (idx >= 0) {
                bool done = false;
                if (obj >= a.sceneSize) {
                    done = pend == 0;
                } else {
                    if (!exh && s.tg.y == 0u && (s.ng.y & 0xff000000u) == 0u) {
                        if (s.sp == 0) exh = true; else s.ng = stack[--s.sp];
                    }
                    if (ANY && s.hitTri >= 0) { exh = true; s.tg.y = 0u; }      // accepted: only wait for queued pairs
                    if (exh && s.tg.y == 0u && pend == 0) {
                        if (ANY && s.hitTri >= 0) done = true;
                        else {
                            obj = next_object(a, obj + 1, skipMask);
                            if (obj < a.sceneSize) {
                                trav_enter_object(s, a.objects[obj].nodes, a.objects[obj].tris); wq_set_object(w, lane, s); exh = false;
                            } else done = true;
                        }
                    }
                }
                if (done && MODE == TM_SHADE && retry && s.hitTri < 0) {
                    retry = false; done = false;
                    s.tbest = FLT_MAX;
                    obj = next_object(a, 0, 0u);
                    if (obj < a.sceneSize) {
                        trav_enter_object(s, a.objects[obj].nodes, a.objects[obj].tris); wq_set_object(w, lane, s); exh = false;
                    } else done = true;
                }
                if (done) {
                    trace_end<MODE>(a, idx, s, flags);
                    if (ANY && s.hitTri < 0) lit = idx;
                    idx = -1;
                }
            }
            if (ANY && a.direct) {
                const unsigned lm = __ballot_sync(FULL, lit >= 0);
                if (lm != 0u) {
                    if (lit >= 0) lits[nlit + __popc(lm & ((1u << lane) - 1u))] = lit;
                    nlit += __popc(lm);
                    if (nlit >= 32) { shadow_flush(a, lits, nlit, lane); nlit = 0; }
                }
            }
            // (2.5) tail of the launch: few rays left in this warp -> all lanes work on one of them (bvh_traverse.cuh)
            if (exhausted && a.coop > 0) {
                const unsigned workM = __ballot_sync(FULL, idx >= 0 && obj < a.sceneSize && !exh);
                if (workM != 0u && __popc(__ballot_sync(FULL, idx >= 0)) <= a.coop) {
                    coop_run<ANY, COUNT>(w, a.coopPool + (size_t)(blockIdx.x * (kTraceBlock / 32) + (threadIdx.x >> 5)) * DPRT_POOLCAP, qlen, lane,
                                         __ffs(workM) - 1, s, stack, obj, pend, exh, cnt, a.prmtMagic, tc);
                    continue;
                }
            }
            // (3) the warp votes: a full (or forced) triangle round, else one node per lane
            const bool busy = idx >= 0;
            const bool canNode = busy && obj < a.sceneSize && !exh && s.tg.y == 0u;
            const unsigned nodeM = __ballot_sync(FULL, canNode);
            const unsigned waitM = __ballot_sync(FULL, busy && !canNode);
            if (qlen > 0 && (qlen >= 32 || nodeM == 0u || __popc(waitM) >= a.triVote)) tri_round<ANY, COUNT>(w, qlen, lane, s, obj, pend, cnt, tc);
            else if (canNode) {
                // Up to nodesPerStep nodes per warp step: most nodes yield no leaf triangles, and the warp-level bookkeeping
                // around a step costs as much as the slab tests of a node. A lane stops early when it has triangles to queue.
                int left = a.nodesPerStep;
#pragma unroll 1
                for (;;) {
                    const uint32_t tm = trav_node<COUNT>(s, stack, cnt, a.prmtMagic);
                    if (s.tg.y != 0u) { w.tmask[lane] = tm; break; }
                    if (--left == 0) break;
                    if ((s.ng.y & 0xff000000u) == 0u) { if (s.sp == 0) break; s.ng = stack[--s.sp]; }
                }
            }
        } while (__popc(__ballot_sync(FULL, idx >= 0)) >= minBusy);
    }
    if (ANY && nlit > 0) shadow_flush(a, lits, nlit, lane);
    if (a.cacheHits) {               // device-side statistics: [0] MainRay queries answered from the cache, [1] rays that walked a BVH, [2 + stage] the same per stage
        if (MODE == TM_SHADE) {
            cached = __reduce_add_sync(FULL, cached);
            if (lane == 0 && cached) atomicAdd(a.cacheHits, (unsigned long long)cached);
        }
        walked = __reduce_add_sync(FULL, walked);
        if (lane == 0 && walked) { atomicAdd(a.cacheHits + 1, (unsigned long long)walked); atomicAdd(a.cacheHits + 2 + StageOf<MODE>::id, (unsigned long long)walked); }
    }
    if (COUNT) {
        if (cnt.nodes) atomicAdd(a.counters + 2 * StageOf<MODE>::id, (unsigned long long)cnt.nodes);
        if (cnt.tris) atomicAdd(a.counters + 2 * StageOf<MODE>::id + 1, (unsigned long long)cnt.tris);
    }
}

// What the closest-hit trace of TraRay / SecondaryRay found for record i (hits[i], written by trace_kernel for every valid
// record of the launch): distributed_traversal_kernel.cu:256-263 / secondary_ray_kernel.cu:211-218, plus the hit cache entry
// MainRay will look up under the path's pixel.
DPRT_D void merge_trace_result(const DevParams& p, int i, PathRegs& path) {
    const float4 h0 = reinterpret_cast<const float4*>(p.hits + i)[0];
    const int prim = __float_as_int(h0.y);
    if (prim < 0) return;
    path.tMax = h0.x; path.currentNode = p.worldID; path.flags |= F_HIT;
    if (p.hitPrim) p.hitPrim[i] = prim;
    if (p.hitCache) {
        const float4 h1 = reinterpret_cast<const float4*>(p.hits + i)[1];
        float4* c = reinterpret_cast<float4*>(p.hitCache + path.pixelIndex);
        c[0] = h0;
        c[1] = make_float4(h1.x, h1.y, __uint_as_float(p.hitEpoch), __int_as_float(path.pixelIndex));
    }
}

// ================================================================================================
// TraRay program after the trace (distributed_traversal_kernel.cu:266-339): own bit, nearest unvisited proxy AABB
// within tMax decides the next owner, environment light on a total miss; histogram by-product for the partition.
__global__ void __launch_bounds__(kBlock) traverse_post_kernel(DevParams p, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) p.traceQueue[0] = 0;     // ray-queue head for the next trace launch on this stream (launch_trace)
    bool outValid = false; int target = -1;
    if (i < n) {
        PathRegs path = load_path(p.paths + i);
        if (p.hitPrim) p.hitPrim[i] = -1;
        if (path.flags & F_VALID) {
            merge_trace_result(p, i, path);
            const V3 o = path.origin, d = path.direction;
            path.visitedMask |= (1u << p.worldID);
            float tProxy = path.tMax; bool proxyHit = false;
            for (int k = 0; k < p.sceneSize; k++) {
                const DevObject& ob = p.objects[k];
                if (ob.isProxy != 1) continue;
                if ((path.visitedMask >> ob.nodeID) & 1u) continue;
                const V3 ol = xform_point(ob.w2o, o), dl = xform_vector(ob.w2o, d);
                float t; bool inside;
                if (aabb_intersect(ol, dl, ob.aabbMin, ob.aabbMax, DPRT_EPSILON, tProxy, &t, &inside)) {
                    tProxy = t; proxyHit = true; path.targetNode = ob.nodeID;
                }
            }
            if (!proxyHit) path.targetNode = path.currentNode;
            if (!proxyHit && !(path.flags & F_HIT)) {
                add_env(p, path);
                path.flags &= ~F_VALID;
            }
            store_path(p.paths + i, path);
            outValid = (path.flags & F_VALID) != 0;
            target = path.targetNode;
        }
    }
    // by-product for the partition stage: valid paths per destination (warp-aggregated)
    outValid = outValid && target >= 0 && target < p.worldSize;
    if (target == p.worldID && i >= p.splitL) target = p.worldSize;      // settled-deque mode: second piece of the self segment
    const unsigned m = __ballot_sync(0xffffffffu, outValid);
    if (outValid) {
        const unsigned peers = __match_any_sync(m, target);
        if ((threadIdx.x & 31) == (__ffs(peers) - 1)) atomicAdd(p.pathHist + target, __popc(peers));
    }
}

// ------------------------------------------------------------------------------------------------
struct BsdfSample { V3 wiLocal; float weight; bool isDelta; };

DPRT_D BsdfSample sample_lambertian(float xi1, float xi2) {           // bsdfs/lambertian.hpp:10-32
    BsdfSample s; s.wiLocal = uniform_hemisphere(xi1, xi2); s.weight = 2.0f; s.isDelta = false; return s;
}
DPRT_D float fresnel_dielectric(float cosI, float etaI, float etaT) { // moana Fresnel::dielectricReflectance (PBRT)
    const float eta = etaI / etaT;
    const float sin2t = (eta * eta) * fmaxf(0.0f, fmaf(-cosI, cosI, 1.0f));
    if (sin2t >= 1.0f) return 1.0f;
    const float cosT = sqrtf(1.0f - sin2t);
    const float rParl = (etaT * cosI - etaI * cosT) / (etaT * cosI + etaI * cosT);
    const float rPerp = (etaI * cosI - etaT * cosT) / (etaI * cosI + etaT * cosT);
    return 0.5f * (rParl * rParl + rPerp * rPerp);
}
DPRT_D BsdfSample sample_water(float xi1, V3 normal, V3 woWorld, bool isInside) {   // bsdfs/water.hpp:12-94
    const V3 wo = frame_to_local(normal, woWorld);
    float etaI = 1.0f, etaT = 1.33f;
    if (isInside) { float t = etaI; etaI = etaT; etaT = t; }
    V3 wi = v3(0.f, 0.f, 0.f);
    {   // Snell::refract about the local +z normal
        const float eta = etaI / etaT;
        const float sin2t = (eta * eta) * fmaxf(0.0f, fmaf(-wo.z, wo.z, 1.0f));
        if (sin2t < 1.0f) { const float cosT = sqrtf(1.0f - sin2t); wi = v3(-(eta * wo.x), -(eta * wo.y), -cosT); }
    }
    const float fr = fresnel_dielectric(fabsf(wo.z), etaI, etaT);
    BsdfSample s; s.isDelta = true;
    if (xi1 < fr) {
        wi = v3(-wo.x, -wo.y, wo.z);                                   // wo.reflect((0,0,1))
        const float cosTheta = fabsf(wi.z);
        const float thr = cosTheta == 0.0f ? 0.0f : fr / cosTheta;
        s.wiLocal = wi; s.weight = thr / fr;
    } else {
        const float ft = 1.0f - fr;
        const float cosTheta = fabsf(wi.z);
        const float thr = cosTheta == 0.0f ? 0.0f : ft / cosTheta;
        const float corr = (etaI / etaT) * (etaI / etaT);
        s.wiLocal = wi; s.weight = thr * corr / ft;
    }
    return s;
}

// MainRay program after the trace: closest-hit program (kernel.cu:171-300), createSamplingRecord (:50-64),
// generateNextNewPath (:134-162), generateShadowPath x spc (:66-132, :442-465).
// src: the records to shade (paths, or the partition output when the single-rank bounce skips the copy back). fromCache: the
// hit comes from the hit cache under the record's pixel instead of hits[i] (the MainRay trace was not launched).
// aov: the first-hit guide buffers (albedo sums 3N, normal sums 3N) when this is the sample's first shade with AOVs on, else
// null. A kernel argument rather than a DevParams field, so that no other kernel's parameters move. At most one record per
// pixel reaches the first shade of a sample on a rank, and only the rank that owns the hit shades it: plain adds, no race.
// roughness: DPRT_MAX_MATERIALS entries, read for bsdfType 2 and 3 only (conductor.cuh, plastic.cuh); a kernel argument for
// the same reason.
__global__ void __launch_bounds__(kBlock) shade_post_kernel(DevParams p, int n, const dprt_path_record* src, bool fromCache,
                                                            float* aov, const float* roughness) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) p.traceQueue[0] = 0;
    if (i >= n) return;
    PathRegs path = load_path(src + i);
    if (!(path.flags & F_VALID)) { if (p.livePixel) p.livePixel[i] = -1; return; }
    const V3 o = path.origin, d = path.direction;
    const float4* hr = reinterpret_cast<const float4*>(fromCache ? p.hitCache + path.pixelIndex : p.hits + i);
    const float4 h0 = hr[0], h1 = hr[1];
    if (fromCache) {
        // every record that survives the single-rank partition was filed in this epoch by traverse_post_kernel; an entry of
        // another epoch would be a broken invariant, counted in cacheHits[2 + DPRT_STAGE_COUNT]
        const unsigned m = __activemask();
        const unsigned stale = __ballot_sync(m, __float_as_uint(h1.z) != p.hitEpoch);
        if ((threadIdx.x & 31) == __ffs(m) - 1) {
            if (m != stale) atomicAdd(p.cacheHits, (unsigned long long)__popc(m & ~stale));
            if (stale) atomicAdd(p.cacheHits + 2 + DPRT_STAGE_COUNT, (unsigned long long)__popc(stale));
        }
    }
    const float ht = h0.x; const int hprim = __float_as_int(h0.y), htri = __float_as_int(h0.z), hobj = __float_as_int(h0.w);
    const bool isHit = htri >= 0;
    if (p.hitPrim) p.hitPrim[i] = isHit ? hprim : -1;
    if (p.livePixel) p.livePixel[i] = isHit ? path.pixelIndex : -1;     // pixels whose shadow planes this bounce can touch
    if (!isHit) {
        // kernel.cu:416-423: environment light, path dies. The reference then writes an invalid record built
        // from an uninitialised sampling record; the defined behaviour here is the all-zero (invalid) record.
        add_env(p, path);
        store_zero_path(p.paths + i);
        for (int s = 0; s < p.spc; s++) store_zero_path(p.paths + (size_t)i * p.spc + s + p.pathSize);
        return;
    }
    const DevObject& ob = p.objects[hobj];
    // closest-hit program (kernel.cu:171-300): interpolated vertex normal, base colour, face-forward
    const float4 tb = __ldg(ob.tris + 3 * (size_t)htri + 1);
    const int matID = __float_as_int(tb.w);
    const dprt_material mat = p.materials[matID];
    V3 albedo = v3(mat.baseColor[0], mat.baseColor[1], mat.baseColor[2]);
    {   // kernel.cu:251-281: a textured material takes its base colour from the albedo map at the interpolated coordinate
        const int nuv = __float_as_int(__ldg(ob.tris + 3 * (size_t)htri + 2).w);
        const int tex = nuv != 0 ? p.matTex[matID] : -1;
        if (tex >= 0 && p.textures[tex].texels) {
            const float4* uv = ob.tris + 3 * (size_t)nuv + 2 * (size_t)htri;
            const float4 ua = __ldg(uv), ub = __ldg(uv + 1);
            const float4 c = tex_bilinear(p.textures[tex], tex_interp(ua.x, ua.z, ub.x, h1.x, h1.y), tex_interp(ua.y, ua.w, ub.y, h1.x, h1.y), false);
            albedo = v3(c.x, c.y, c.z);
        }
    }
    const V3 point = v3at(o, d, ht);
    const V3 woWorld = v3neg(d);
    V3 normal;
    {
        const float* nn = ob.normals + 9 * (size_t)hprim;
        const V3 n0 = v3normalized(v3(nn[0], nn[1], nn[2]));
        const V3 n1 = v3normalized(v3(nn[3], nn[4], nn[5]));
        const V3 n2 = v3normalized(v3(nn[6], nn[7], nn[8]));
        const float alpha = h1.x, beta = h1.y, gamma = 1.0f - alpha - beta;
        normal = v3(fmaf(beta, n2.x, fmaf(alpha, n1.x, gamma * n0.x)), fmaf(beta, n2.y, fmaf(alpha, n1.y, gamma * n0.y)),
                    fmaf(beta, n2.z, fmaf(alpha, n1.z, gamma * n0.z)));
        normal = v3normalized(normal);
    }
    bool isInside = false;
    if (v3dot(normal, woWorld) < 0.0f) { normal = v3neg(normal); isInside = true; }
    if (aov) {
        float* a = aov + 3 * (size_t)path.pixelIndex;
        float* nrm = a + 3 * (size_t)p.frameBufferSize;
        a[0] += albedo.x; a[1] += albedo.y; a[2] += albedo.z;
        nrm[0] += normal.x; nrm[1] += normal.y; nrm[2] += normal.z;
    }
    // createSamplingRecord (kernel.cu:50-64): the seed ignores the bounce, as in the reference
    uint32_t seed = tea4((uint32_t)path.pixelIndex, (uint32_t)p.sampleCount);
    const float xi1 = rnd(seed), xi2 = rnd(seed);
    // bsdfType 2, the conductor (DESIGN.md 3.12; albedo is its F0), and 3, the plastic (DESIGN.md 3.13; albedo is its diffuse
    // colour, and it draws a third uniform to choose its lobe): their throughput factor replaces weight * cos * albedo
    const bool isCond = mat.bsdfType == 2, isGlossy = isCond || mat.bsdfType == 3;
    BsdfSample bs; CondSample cs; V3 woLocal; float rough = 0.0f;
    if (isGlossy) {
        woLocal = frame_to_local(normal, woWorld);
        rough = roughness[matID];
        cs = isCond ? cond_sample(albedo, rough, woLocal, xi1, xi2) : plastic_sample(albedo, rough, woLocal, xi1, xi2, rnd(seed));
        bs.wiLocal = cs.wi; bs.weight = 0.0f; bs.isDelta = isCond && rough == 0.0f;      // the plastic's diffuse lobe takes light
    } else {
        bs = mat.bsdfType == 1 ? sample_water(xi1, normal, woWorld, isInside) : sample_lambertian(xi1, xi2);
    }

    // generateNextNewPath (kernel.cu:134-162)
    PathRegs next;
    next.origin = point;
    next.direction = v3normalized(frame_to_world(normal, bs.wiLocal));
    next.tMax = FLT_MAX;
    const float cosThetaWi = fabsf(bs.wiLocal.z);
    next.throughput = isGlossy ? v3mul(path.throughput, cs.weight) : v3mul(v3scale(v3scale(path.throughput, bs.weight), cosThetaWi), albedo);
    next.pixelIndex = path.pixelIndex; next.shadowPathID = -1; next.visitedMask = 0u;
    next.currentNode = -1; next.targetNode = -1; next.flags = F_VALID;
    if (isGlossy && !cs.valid) store_zero_path(p.paths + i);            // a lobe sampled below the surface: the path ends
    else store_path(p.paths + i, next);

    // generateShadowPath x spc (kernel.cu:66-132, 442-465)
    for (int s = 0; s < p.spc; s++) {
        dprt_path_record* slot = p.paths + (size_t)i * p.spc + s + p.pathSize;
        if (bs.isDelta) { store_zero_path(slot); continue; }      // reference leaves the reset (zero) slot
        uint32_t sseed = tea4((uint32_t)(path.pixelIndex * p.spc + s), (uint32_t)p.sampleCount);
        const float x1 = rnd(sseed), x2 = rnd(sseed), x3 = rnd(sseed);
        int li = (int)floorf(x1 * (float)p.lightCount);
        const dprt_light_tri L = p.lights[li];
        // Triangle::sample(xi2, xi3): uniform area sampling, areaPDF = 1/area
        const V3 p0 = v3(L.p0[0], L.p0[1], L.p0[2]), p1 = v3(L.p1[0], L.p1[1], L.p1[2]), p2 = v3(L.p2[0], L.p2[1], L.p2[2]);
        const float su = sqrtf(x2);
        const float b0 = 1.0f - su, b1 = x3 * su, b2 = 1.0f - b0 - b1;
        const V3 lp = v3(fmaf(b2, p2.x, fmaf(b1, p1.x, b0 * p0.x)), fmaf(b2, p2.y, fmaf(b1, p1.y, b0 * p0.y)),
                         fmaf(b2, p2.z, fmaf(b1, p1.z, b0 * p0.z)));
        const V3 cr = v3cross(v3sub(p1, p0), v3sub(p2, p0));
        const float crl = v3length(cr);
        const V3 ln = v3scale(cr, 1.0f / crl);
        float areaPDF = 1.0f / (0.5f * crl);
        areaPDF = areaPDF * (1.0f / (float)p.lightCount);
        const V3 ldir = v3sub(lp, point);
        const V3 wi = v3normalized(ldir);
        const float stMax = v3length(ldir);
        const float f1 = fmaxf(0.0f, v3dot(ln, v3neg(wi)));
        const float f2 = fmaxf(0.0f, v3dot(wi, normal));
        // the conductor's or the plastic's f(wi, wo) takes the place of Lambert's albedo * 1/pi
        const V3 fr = isGlossy ? (isCond ? cond_eval(albedo, rough, woLocal, frame_to_local(normal, wi))
                                         : plastic_eval(albedo, rough, woLocal, frame_to_local(normal, wi)))
                               : albedo;
        V3 c = v3mul(v3mul(v3(L.Le[0], L.Le[1], L.Le[2]), path.throughput), fr);
        c = v3scale(v3scale(c, f1), f2);
        const float tt = stMax * stMax;
        c = v3(c.x / areaPDF / tt, c.y / areaPDF / tt, c.z / areaPDF / tt);
        if (!isGlossy) c = v3scale(c, 0.318309886183790671538f);
        PathRegs sh;
        sh.origin = point; sh.direction = wi; sh.tMax = stMax; sh.throughput = c;
        sh.pixelIndex = path.pixelIndex; sh.shadowPathID = s; sh.visitedMask = 0u; sh.currentNode = -1; sh.targetNode = -1;
        sh.flags = F_SHADOW | F_VALID;
        store_path(slot, sh);
    }
}

// Proxy-AABB march shared by the shadow and secondary stages (shadow_ray_kernel.cu:198-350,
// secondary_ray_kernel.cu:226-362). Emits <= mc queries into slot base `q0 = threadIndex*mc`.
struct MarchOut { int count; bool envMiss; };

DPRT_D void clear_query_slots(const DevParams& p, int threadIndex, int from) {
    if (!p.proxyMode) return;                     // no query buffers exist when proxies are off
    for (int q = from; q < p.mc; q++) {                                                          // reset by count, not memset
        p.nnQuery[(size_t)threadIndex * p.mc + q].hitAABBID = 0;
        p.nnKey[(size_t)threadIndex * p.mc + q] = 0;
    }
}

template <bool SECONDARY>
DPRT_D int proxy_march(const DevParams& p, const PathRegs& path, int threadIndex, float tMaxPath, int* shHist) {
    const V3 o = path.origin, d = path.direction;
    const int mc = p.mc;
    bool isHit = true; bool isInside = false; float tMin = 0.0f; int count = 0; int hitIdx = -1;
    bool addedDirect = false;
    while (isHit && count < mc) {
        isHit = false;
        float tMax = tMaxPath;
        V3 pl = v3(0, 0, 0), oloc = v3(0, 0, 0), dloc = v3(0, 0, 0);
        for (int k = 0; k < p.sceneSize; k++) {
            const DevObject& ob = p.objects[k];
            if (ob.isProxy != 1) continue;
            const V3 ol = xform_point(ob.w2o, o), dl = xform_vector(ob.w2o, d);
            float t; bool ins;
            if (aabb_intersect(ol, dl, ob.aabbMin, ob.aabbMax, tMin + DPRT_EPSILON, tMax, &t, &ins)) {
                tMax = t; isHit = true; hitIdx = k; isInside = ins;
                oloc = ol; dloc = dl;
                pl = xform_point(ob.w2o, v3at(o, d, t));   // optixTransformPointFromWorldToObjectSpace(getHitPoint())
            }
        }
        if (isHit) tMin = tMax;
        if (isHit) {
            const DevObject& ob = p.objects[hitIdx];
            if (isInside) {
                bool skip = false;
                for (int q = 0; q < count; q++) {
                    const dprt_nn_query& e = p.nnQuery[(size_t)threadIndex * mc + q];
                    if (e.hitAABBID == hitIdx + 1 && e.instanceID == hitIdx) skip = true;
                }
                if (skip && count) continue;
            }
            V3 dirL = isInside ? v3neg(dloc) : dloc;
            float phi, theta;
            det_cartesian_to_spherical(v3normalized(dirL), &phi, &theta);
            dprt_half* in = p.nnInput + ((size_t)threadIndex * mc + count) * 5;
            in[0] = f32_to_f16_bits((pl.x - ob.aabbMin[0]) / (ob.aabbMax[0] - ob.aabbMin[0]));
            in[1] = f32_to_f16_bits((pl.y - ob.aabbMin[1]) / (ob.aabbMax[1] - ob.aabbMin[1]));
            in[2] = f32_to_f16_bits((pl.z - ob.aabbMin[2]) / (ob.aabbMax[2] - ob.aabbMin[2]));
            in[3] = f32_to_f16_bits(phi / 6.28318530717958647692f);
            in[4] = f32_to_f16_bits(theta / 3.14159265358979323846f);
            dprt_nn_query e;
            e.pixelIndex = path.pixelIndex; e.hitSequence = count; e.hitAABBID = hitIdx + 1;
            e.isValid = 1; e.instanceID = hitIdx; e.isInside = isInside ? 1 : 0; e.pad_[0] = e.pad_[1] = 0; e.reserved_ = 0;
            const float dist = v3length(v3sub(oloc, pl));
            if (SECONDARY) {
                e.throughput[0] = tMax; e.throughput[1] = ob.maxLength; e.throughput[2] = tMax / dist;
                e.shadowPathID = 0; e.pathIndex = ob.nodeID;
                e.normalizedT = isInside ? tMax / ob.maxLength : 0.0f;
            } else {
                e.throughput[0] = path.throughput.x; e.throughput[1] = path.throughput.y; e.throughput[2] = path.throughput.z;
                e.shadowPathID = path.shadowPathID;
                e.pathIndex = isInside ? threadIndex * mc + count : 0;
                e.normalizedT = isInside ? dist / ob.maxLength : 0.0f;
            }
            p.nnQuery[(size_t)threadIndex * mc + count] = e;
            p.nnKey[(size_t)threadIndex * mc + count] = (uint8_t)((hitIdx + 1) | (isInside ? 0x80 : 0));
            // histogram by-product for the bucketing stage: all queries, and inside-only
            atomicAdd(shHist + hitIdx, 1);
            if (isInside) atomicAdd(shHist + 32 + hitIdx, 1);
            count++;
        } else if (count == 0) {
            addedDirect = true;
        }
    }
    clear_query_slots(p, threadIndex, count);
    return addedDirect ? -1 : count;   // -1: nothing in the way at all
}

DPRT_D void flush_query_hist(const DevParams& p, const int* shHist) {
    const int t = threadIdx.x;
    if (t < p.sceneSize) { if (shHist[t]) atomicAdd(p.queryHist + t, shHist[t]); }
    else if (t >= 32 && t < 32 + p.sceneSize) { if (shHist[t]) atomicAdd(p.queryHist + p.sceneSize + (t - 32), shHist[t]); }
}

// ShadowRay program after the any-hit trace with proxies on (shadow_ray_kernel.cu:198-350): occluded paths were marked by
// the trace; the others march through the proxy AABBs or, with nothing in the way, add their contribution. With proxies off
// the trace kernel adds the contributions itself and this kernel is not launched.
__global__ void __launch_bounds__(kBlock) shadow_post_kernel(DevParams p, int nShadow) {
    __shared__ int shHist[64];
    if (threadIdx.x < 64) shHist[threadIdx.x] = 0;
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) p.traceQueue[0] = 0;
    if (i < nShadow) {
        const PathRegs path = load_path(p.paths + (size_t)p.pathSize + i);
        if (!(path.flags & F_VALID)) {
            clear_query_slots(p, i, 0);
        } else {
            const int r = proxy_march<false>(p, path, i, path.tMax, shHist);
            if (r < 0) {
                const size_t px = ((size_t)p.frameBufferSize * path.shadowPathID + path.pixelIndex) * 3;
                const float inv = (float)p.spc;
                p.direct[px + 0] += path.throughput.x / inv;
                p.direct[px + 1] += path.throughput.y / inv;
                p.direct[px + 2] += path.throughput.z / inv;
            }
        }
    }
    __syncthreads();
    flush_query_hist(p, shHist);
}

// SecondaryRay program after the trace (secondary_ray_kernel.cu:192, :226-362).
__global__ void __launch_bounds__(kBlock) secondary_post_kernel(DevParams p, int n) {
    __shared__ int shHist[64];
    if (threadIdx.x < 64) shHist[threadIdx.x] = 0;
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) p.traceQueue[0] = 0;
    if (i < n) {
        PathRegs path = load_path(p.paths + i);
        if (p.hitPrim) p.hitPrim[i] = -1;
        if (!(path.flags & F_VALID)) {
            clear_query_slots(p, i, 0);
        } else {
            merge_trace_result(p, i, path);
            for (int k = 0; k < p.sceneSize; k++) if (p.objects[k].isProxy != 2) path.visitedMask |= (1u << p.objects[k].nodeID);
            const int r = proxy_march<true>(p, path, i, path.tMax, shHist);
            if (r < 0 && !(path.flags & F_HIT)) {
                add_env(p, path);
                path.flags &= ~F_VALID;
            }
            store_path(p.paths + i, path);
        }
    }
    __syncthreads();
    flush_query_hist(p, shHist);
}

// Vis pipeline after its trace (vis_ray_kernel.cu:145-160): the encoding the proxy MLPs are trained on, the same one the
// ShadowRay / SecondaryRay programs feed them with (proxy_march above).
__global__ void __launch_bounds__(kBlock) train_features_kernel(const DevObject* __restrict__ obj, const dprt_ray* __restrict__ rays,
                                                                 const dprt_hit* __restrict__ hits, int64_t n, float* __restrict__ feat,
                                                                 float* __restrict__ label) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const DevObject& ob = *obj;
    const float4 r0 = __ldg(reinterpret_cast<const float4*>(rays) + 2 * i), r1 = __ldg(reinterpret_cast<const float4*>(rays) + 2 * i + 1);
    const V3 ol = xform_point(ob.w2o, v3(r0.x, r0.y, r0.z)), dl = xform_vector(ob.w2o, v3(r1.x, r1.y, r1.z));
    float phi, theta;
    det_cartesian_to_spherical(v3normalized(dl), &phi, &theta);
    float* f = feat + 5 * i;
    f[0] = (ol.x - ob.aabbMin[0]) / (ob.aabbMax[0] - ob.aabbMin[0]);
    f[1] = (ol.y - ob.aabbMin[1]) / (ob.aabbMax[1] - ob.aabbMin[1]);
    f[2] = (ol.z - ob.aabbMin[2]) / (ob.aabbMax[2] - ob.aabbMin[2]);
    f[3] = phi / 6.28318530717958647692f;
    f[4] = theta / 3.14159265358979323846f;
    const float2 h = reinterpret_cast<const float2*>(hits)[i];
    label[i] = __float_as_int(h.y) >= 0 ? h.x / ob.maxLength : 1.0f;
}

// Precom pipeline (precom_ray_kernel.cu:193-299): a camera path meets the proxied object's AABB (front face, or back face when
// the origin is inside) -> the MLP input encoding at the AABB hit; the object's ORIGINAL geometry is then traced with
// tMax = inf and the label is the depth behind the AABB surface, (t_geo - t_aabb) / maxLength. This kernel does the AABB
// stage and rewrites the staged ray for the geometry stage (tMax = inf); precom_label_kernel finishes after the trace.
__global__ void __launch_bounds__(kBlock) precom_features_kernel(const DevObject* __restrict__ obj, dprt_ray* __restrict__ rays, int64_t n,
                                                                  float* __restrict__ feat, float* __restrict__ tAabb) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const DevObject& ob = *obj;
    float4* rp = reinterpret_cast<float4*>(rays) + 2 * i;
    const float4 r0 = rp[0], r1 = rp[1];
    const V3 o = v3(r0.x, r0.y, r0.z), d = v3(r1.x, r1.y, r1.z);
    const V3 ol = xform_point(ob.w2o, o), dl = xform_vector(ob.w2o, d);
    float* f = feat + 5 * i;
    float t; bool inside;
    if (aabb_intersect(ol, dl, ob.aabbMin, ob.aabbMax, r0.w, r1.w, &t, &inside)) {
        const V3 pl = xform_point(ob.w2o, v3at(o, d, t));
        const V3 dirL = inside ? v3neg(dl) : dl;
        float phi, theta;
        det_cartesian_to_spherical(v3normalized(dirL), &phi, &theta);
        f[0] = (pl.x - ob.aabbMin[0]) / (ob.aabbMax[0] - ob.aabbMin[0]);
        f[1] = (pl.y - ob.aabbMin[1]) / (ob.aabbMax[1] - ob.aabbMin[1]);
        f[2] = (pl.z - ob.aabbMin[2]) / (ob.aabbMax[2] - ob.aabbMin[2]);
        f[3] = phi / 6.28318530717958647692f;
        f[4] = theta / 3.14159265358979323846f;
        tAabb[i] = t;
    } else {
        f[0] = f[1] = f[2] = f[3] = f[4] = 0.0f;     // the reference leaves its (zeroed) buffers untouched
        tAabb[i] = -1.0f;
    }
    rp[1] = make_float4(r1.x, r1.y, r1.z, FLT_MAX);  // geometry stage: path.tMax = __FLT_MAX__ (precom_ray_kernel.cu:262)
}
// label: (t_geo - t_aabb) / maxLength when AABB and geometry are both hit; 1.0 -- the loaders' "miss" value
// (trainingcode/datasets.py:166-170) -- when the AABB is hit and the geometry is not; valid = 0 when the AABB is missed
__global__ void __launch_bounds__(kBlock) precom_label_kernel(const DevObject* __restrict__ obj, const dprt_hit* __restrict__ hits, const float* __restrict__ tAabb,
                                                               int64_t n, float* __restrict__ label, uint8_t* __restrict__ valid) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float ta = tAabb[i];
    const float2 h = reinterpret_cast<const float2*>(hits)[i];
    const bool aabb = ta >= 0.0f, geo = __float_as_int(h.y) >= 0;
    label[i] = aabb ? (geo ? (h.x - ta) / obj->maxLength : 1.0f) : 1.0f;
    valid[i] = aabb ? 1 : 0;
}

inline int blocks_for(int64_t n) { return (int)((n + kBlock - 1) / kBlock); }

int num_sms() {
    static int cached[64] = {0};
    int dev = 0; cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    if (!cached[dev]) cudaDeviceGetAttribute(&cached[dev], cudaDevAttrMultiProcessorCount, dev);
    return cached[dev] > 0 ? cached[dev] : 148;
}

// tuning knobs (defaults measured on B200, see profiles/): environment overrides are for experiments only
int env_int(const char* name, int dflt, int lo, int hi) {
    const char* v = getenv(name);
    if (!v) return dflt;
    const int x = atoi(v);
    return x < lo ? lo : (x > hi ? hi : x);
}
int tune_refill() { static int v = env_int("DPRT_TRACE_REFILL", kRefillDefault, 1, 32); return v; }
int tune_trivote() { static int v = env_int("DPRT_TRACE_TRIVOTE", kTriVoteDefault, 1, 32); return v; }
int tune_coop() { static int v = env_int("DPRT_TRACE_COOP", kCoopDefault, 0, 32); return v; }
int tune_rpl() { static int v = env_int("DPRT_TRACE_RPL", kRaysPerLaneDefault, 1, 64); return v; }
int tune_nodes() { static int v = env_int("DPRT_TRACE_NODES", kNodesPerStepDefault, 1, 16); return v; }
int tune_blocks() { static int v = env_int("DPRT_TRACE_BLOCKS_PER_SM", 0, 0, 16); return v; }     // 0 = the launch bound of the mode

template <int MODE>
void launch_trace(TraceArgs a, int64_t n, cudaStream_t s) {
    // the queue head is zero here: cleared at allocation and again after every launch -- by the post kernel that follows each
    // stage's trace launch on the same stream (one cudaMemsetAsync less per launch), by a memset after the bare TM_RAYS launch
    // and after a TM_SHADOW launch that has no post kernel (proxies off)
    // the context's trace scratch: the 64-byte queue head, then the cooperative-mode node pools
    a.coopPool = reinterpret_cast<uint32_t*>(a.queue + 16);
    // Grid: never more warps than keep every lane supplied with ~tune_rpl() rays. A warp runs until its longest ray is
    // done, so with one ray per lane its efficiency is mean/max ray length; with a few rays per lane the refill evens it out.
    const int64_t want = (n + (int64_t)kTraceBlock * tune_rpl() - 1) / ((int64_t)kTraceBlock * tune_rpl());
    const int perSM = tune_blocks() > 0 ? tune_blocks() : trace_min_blocks<MODE>();
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)num_sms() * perSM));
    if (a.counters) trace_kernel<MODE, true><<<blocks, kTraceBlock, 0, s>>>(a, (int)n);
    else trace_kernel<MODE, false><<<blocks, kTraceBlock, 0, s>>>(a, (int)n);
    if (MODE == TM_RAYS) cudaMemsetAsync(a.queue, 0, sizeof(int32_t), s);
}

TraceArgs trace_args(const DevParams& p, dprt_path_record* recs) {
    TraceArgs a;
    a.objects = p.objects; a.sceneSize = p.sceneSize; a.worldID = p.worldID; a.recs = recs; a.hits = p.hits;
    a.rays = nullptr; a.rayHits = nullptr; a.hitPrim = p.hitPrim; a.queue = p.traceQueue; a.counters = p.counters;
    a.refill = tune_refill(); a.triVote = tune_trivote(); a.prmtMagic = 0x47000000u; a.coop = tune_coop(); a.nodesPerStep = tune_nodes();
    a.hitCache = p.hitCache; a.epoch = p.hitEpoch; a.cacheHits = p.cacheHits;
    a.textures = p.textures; a.matTex = p.matTex;
    a.direct = nullptr; a.frameBufferSize = p.frameBufferSize; a.spc = p.spc;
    return a;
}

}  // namespace

// dprt_spec_texture_sample / dprt_spec_env_lookup: host loops over the DPRT_HD functions of dprt_math.cuh
int spec_texture_sample(const float* rgba, int width, int height, const float* u, const float* v, int64_t n, int clampV, float* out4) {
    if (!rgba || !u || !v || !out4 || width < 1 || height < 1 || n < 0) return DPRT_ERR_INVALID;
    const DevTexture T = {reinterpret_cast<const float4*>(rgba), width, height};
    for (int64_t i = 0; i < n; i++) {
        const float4 c = tex_bilinear(T, u[i], v[i], clampV != 0);
        out4[4 * i + 0] = c.x; out4[4 * i + 1] = c.y; out4[4 * i + 2] = c.z; out4[4 * i + 3] = c.w;
    }
    return 0;
}
int spec_env_lookup(const float* rgba, int width, int height, float rotationOffset, const float* dirs3, int64_t n, float* out3) {
    if (!rgba || !dirs3 || !out3 || width < 1 || height < 1 || n < 0) return DPRT_ERR_INVALID;
    const DevTexture T = {reinterpret_cast<const float4*>(rgba), width, height};
    for (int64_t i = 0; i < n; i++) {
        const float4 c = env_map_lookup(T, rotationOffset, v3(dirs3[3 * i], dirs3[3 * i + 1], dirs3[3 * i + 2]));
        out3[3 * i + 0] = c.x; out3[3 * i + 1] = c.y; out3[3 * i + 2] = c.z;
    }
    return 0;
}

// dprt_spec_conductor_sample / dprt_spec_conductor_eval: host loops over conductor.cuh
int spec_conductor_sample(const float* f0, const float* r, const float* wo, const float* xi, int64_t n, float* wi, float* weight) {
    if (!f0 || !r || !wo || !xi || !wi || !weight || n < 0) return DPRT_ERR_INVALID;
    for (int64_t i = 0; i < n; i++) {
        const CondSample s = cond_sample(v3(f0[3 * i], f0[3 * i + 1], f0[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                                         xi[2 * i], xi[2 * i + 1]);
        wi[3 * i] = s.wi.x; wi[3 * i + 1] = s.wi.y; wi[3 * i + 2] = s.wi.z;
        weight[3 * i] = s.weight.x; weight[3 * i + 1] = s.weight.y; weight[3 * i + 2] = s.weight.z;
    }
    return 0;
}
int spec_conductor_eval(const float* f0, const float* r, const float* wo, const float* wi, int64_t n, float* f) {
    if (!f0 || !r || !wo || !wi || !f || n < 0) return DPRT_ERR_INVALID;
    for (int64_t i = 0; i < n; i++) {
        const V3 v = cond_eval(v3(f0[3 * i], f0[3 * i + 1], f0[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                               v3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]));
        f[3 * i] = v.x; f[3 * i + 1] = v.y; f[3 * i + 2] = v.z;
    }
    return 0;
}

// dprt_spec_plastic_sample / dprt_spec_plastic_eval: host loops over plastic.cuh
int spec_plastic_sample(const float* albedo, const float* r, const float* wo, const float* xi, int64_t n, float* wi, float* weight) {
    if (!albedo || !r || !wo || !xi || !wi || !weight || n < 0) return DPRT_ERR_INVALID;
    for (int64_t i = 0; i < n; i++) {
        const CondSample s = plastic_sample(v3(albedo[3 * i], albedo[3 * i + 1], albedo[3 * i + 2]), r[i],
                                            v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]), xi[3 * i], xi[3 * i + 1], xi[3 * i + 2]);
        wi[3 * i] = s.wi.x; wi[3 * i + 1] = s.wi.y; wi[3 * i + 2] = s.wi.z;
        weight[3 * i] = s.weight.x; weight[3 * i + 1] = s.weight.y; weight[3 * i + 2] = s.weight.z;
    }
    return 0;
}
int spec_plastic_eval(const float* albedo, const float* r, const float* wo, const float* wi, int64_t n, float* f) {
    if (!albedo || !r || !wo || !wi || !f || n < 0) return DPRT_ERR_INVALID;
    for (int64_t i = 0; i < n; i++) {
        const V3 v = plastic_eval(v3(albedo[3 * i], albedo[3 * i + 1], albedo[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                                  v3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]));
        f[3 * i] = v.x; f[3 * i + 1] = v.y; f[3 * i + 2] = v.z;
    }
    return 0;
}

size_t trace_scratch_bytes() {
    // 64 B for the ray-queue head + one cooperative-mode node pool per warp that can be resident
    return 64 + (size_t)num_sms() * std::max(tune_blocks(), 8) * (kTraceBlock / 32) * DPRT_POOLCAP * sizeof(uint32_t);
}

// forces the module load of the kernels of the migrate loop (p2p_exchange.cuh: never a first launch beside a spinning kernel)
cudaError_t trace_preload_kernels() {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, trace_kernel<TM_TRAVERSE, false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, trace_kernel<TM_TRAVERSE, true>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, traverse_post_kernel);
    return e;
}

void launch_path_gen(const DevParams& p, int n, cudaStream_t s) {
    if (n > 0) path_gen_kernel<<<blocks_for(n), kBlock, 0, s>>>(p, n);
}
void launch_traverse(const DevParams& p, int n, cudaStream_t s) {
    if (n <= 0) return;
    launch_trace<TM_TRAVERSE>(trace_args(p, p.paths), n, s);
    traverse_post_kernel<<<blocks_for(n), kBlock, 0, s>>>(p, n);
}
void launch_shade(const DevParams& p, int n, float* aov, const float* roughness, cudaStream_t s) {
    if (n <= 0) return;
    launch_trace<TM_SHADE>(trace_args(p, p.paths), n, s);
    shade_post_kernel<<<blocks_for(n), kBlock, 0, s>>>(p, n, p.paths, false, aov, roughness);
}
void launch_shade_cached(const DevParams& p, int n, float* aov, const float* roughness, cudaStream_t s) {
    if (n > 0) shade_post_kernel<<<blocks_for(n), kBlock, 0, s>>>(p, n, p.transfer, true, aov, roughness);
}
void launch_shadow_trace(const DevParams& p, int nShadow, cudaStream_t s) {
    if (nShadow <= 0) return;
    TraceArgs a = trace_args(p, p.paths + p.pathSize);
    if (!p.proxyMode) a.direct = p.direct;
    launch_trace<TM_SHADOW>(a, nShadow, s);
    if (p.proxyMode) shadow_post_kernel<<<blocks_for(nShadow), kBlock, 0, s>>>(p, nShadow);
    else cudaMemsetAsync(p.traceQueue, 0, sizeof(int32_t), s);     // the queue reset the post kernel would have done
}
void launch_secondary_trace(const DevParams& p, int n, cudaStream_t s) {
    if (n <= 0) return;
    launch_trace<TM_SECONDARY>(trace_args(p, p.paths), n, s);
    secondary_post_kernel<<<blocks_for(n), kBlock, 0, s>>>(p, n);
}
void launch_train_features(const DevObject* obj, const dprt_ray* rays, const dprt_hit* hits, int64_t n, float* features,
                           float* labels, cudaStream_t s) {
    if (n > 0) train_features_kernel<<<blocks_for(n), kBlock, 0, s>>>(obj, rays, hits, n, features, labels);
}
void launch_precom_features(const DevObject* obj, dprt_ray* rays, int64_t n, float* features, float* t_aabb, cudaStream_t s) {
    if (n > 0) precom_features_kernel<<<blocks_for(n), kBlock, 0, s>>>(obj, rays, n, features, t_aabb);
}
void launch_precom_labels(const DevObject* obj, const dprt_hit* hits, const float* t_aabb, int64_t n, float* labels, uint8_t* valid, cudaStream_t s) {
    if (n > 0) precom_label_kernel<<<blocks_for(n), kBlock, 0, s>>>(obj, hits, t_aabb, n, labels, valid);
}
void launch_trace_closest(const DevObject* objects, int sceneSize, const DevTexture* textures, const int32_t* matTex, const dprt_ray* rays,
                          dprt_hit* hits, int64_t n, int32_t* queue, unsigned long long* counters, cudaStream_t s) {
    if (n <= 0) return;
    TraceArgs a;
    a.objects = objects; a.sceneSize = sceneSize; a.worldID = 0; a.recs = nullptr; a.hits = nullptr;
    a.rays = rays; a.rayHits = hits; a.hitPrim = nullptr; a.queue = queue; a.counters = counters;
    a.refill = tune_refill(); a.triVote = tune_trivote(); a.prmtMagic = 0x47000000u; a.coop = tune_coop(); a.nodesPerStep = tune_nodes();
    a.hitCache = nullptr; a.epoch = 0u; a.cacheHits = nullptr;
    a.textures = textures; a.matTex = matTex;
    launch_trace<TM_RAYS>(a, n, s);
}

}  // namespace dprt
