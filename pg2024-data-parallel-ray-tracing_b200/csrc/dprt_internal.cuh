// dprt_internal.cuh -- device-side parameter block and launch prototypes shared by the .cu files.
// DevParams is the equivalent of the reference's Renderer::Params (SURVEY.md section 2.4), passed by value.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "dprt_types.h"
#include "dprt_math.cuh"

namespace dprt {

struct DevObject {                 // AccelerationStructure (renderer.cpp:1812-1842) as the kernels see it
    int32_t nodeID;
    int32_t isProxy;
    float   aabbMin[3];
    float   aabbMax[3];
    float   maxLength;
    float   w2o[12];
    const uint4*  nodes;           // BVH8 nodes, 5 x uint4 each (local objects only)
    const float4* tris;            // leaf-ordered triangles, 3 x float4 each
    const float*  normals;         // 9 floats per original triangle (vertex normals), may be null
};

struct HitRec {                    // closest-hit result handed from the trace to the shading program (32 bytes)
    float   t;
    int32_t prim;                  // original primitive id, -1 = miss
    int32_t tri;                   // index into the leaf-ordered triangle array, -1 = miss
    int32_t obj;                   // scene index of the object that was hit
    float   alpha, beta;           // barycentric weights of v1, v2
    uint32_t epoch;                // hit cache only: trace epoch the entry was written in (0 = never)
    int32_t pixel;                 // hit cache only: pixelIndex of the path
};

struct DevParams {
    int32_t pathSize;
    int32_t shadowPathSize;
    int32_t spc;                   // shadowPathCount
    int32_t mc;                    // maxCount
    int32_t sceneSize;
    int32_t worldID;
    int32_t worldSize;
    int32_t sampleCount;
    int32_t frameBufferSize;       // N = width*height
    int32_t lightCount;
    int32_t proxyMode;
    int32_t pathGenMode;
    float   envColor[3];
    dprt_camera camera;

    const DevObject*      objects;
    const dprt_material*  materials;
    const dprt_light_tri* lights;

    dprt_path_record* paths;       // pathDataBuffer: slot 0 live paths, pathSize + i*spc + s shadow paths
    dprt_path_record* transfer;    // transferPathDataBuffer
    int32_t* transferOffset;       // W+1
    int32_t* pathHist;             // W counters: valid paths per targetNode (by-product of traverse)
    float*   direct;               // directLightingBuffer, spc planes of 3N
    float*   env;                  // envLightingBuffer 3N
    float*   contribution;         // 3N*spc
    float*   occlusion;            // shadowOcclusionFloatTypeBuffer N*mc*spc
    dprt_half*     nnInput;        // inputDataBuffer
    dprt_half*     nnPackedInput;
    dprt_nn_query* nnQuery;        // NNPathDataBuffer
    dprt_nn_query* nnPackedQuery;
    uint8_t* nnKey;                // per query slot: hitAABBID | isInside << 7 (0 = empty): what the bucketing reads instead of
                                   // the 48-byte records, most of which are empty
    int32_t* sceneOffset;          // sceneSize+1
    int32_t* queryHist;            // sceneSize counters (all queries), then sceneSize (inside only)
    dprt_half* pred;               // predBuffer
    int32_t* hitPrim;              // parity aid, may be null
    unsigned long long* counters;  // instrumentation: {nodes, tris} per dprt_stage_id, null = off
    HitRec*  hits;                 // N closest-hit records (MainRay trace -> shading program)
    int32_t* traceQueue;           // head of the persistent trace kernel's ray queue
    HitRec*  hitCache;             // per pixel: closest local hit of the pixel's path in the current epoch (null = off)
    uint32_t hitEpoch;             // one epoch per bounce of a sample: entries of older epochs are stale
    unsigned long long* cacheHits; // device statistics (dprt_api.cu kDevStats): [0] MainRay queries answered from the cache
    int32_t  splitL;               // settled-deque mode of the migrate loop: records at index >= splitL that stay on this
                                   // rank are counted in bucket worldSize instead of bucket worldID (INT_MAX: reference)
    int32_t* secLive;              // per path slot of the last Target_Node_Update: pixel whose tMax scratch it used, or -1
    int32_t* livePixel;            // per path slot of the last MainRay launch: pixel that got shadow paths, or -1
    // real-scene front end (dprt.h): albedo / opacity maps, texture index per material (-1 = none), environment map
    const DevTexture* textures;    // DPRT_MAX_TEXTURES slots, texels == null: slot empty
    const int32_t*    matTex;      // DPRT_MAX_MATERIALS entries
    DevTexture        envMap;      // texels == null: analytic sky of envColor
    float             envRotation;
};

// stage launches (all asynchronous on `stream`)
void launch_path_gen(const DevParams& p, int n, cudaStream_t stream);
void launch_traverse(const DevParams& p, int n, cudaStream_t stream);
// aov: first-hit guide buffers (6N floats) to add to, or null (AOVs off, or not the sample's first shade)
void launch_shade(const DevParams& p, int n, float* aov, cudaStream_t stream);
// MainRay without its trace: shades the partition output p.transfer[0..n) with the hits of the hit cache (single rank only)
void launch_shade_cached(const DevParams& p, int n, float* aov, cudaStream_t stream);
// proxies off: the any-hit trace also adds the unoccluded terms to directLightingBuffer and no post kernel follows
void launch_shadow_trace(const DevParams& p, int nShadow, cudaStream_t stream);
void launch_secondary_trace(const DevParams& p, int n, cudaStream_t stream);
size_t trace_scratch_bytes();   // per-context scratch of the persistent trace kernel (queue head + cooperative-mode pools)
void launch_trace_closest(const DevObject* objects, int sceneSize, const DevTexture* textures, const int32_t* matTex, const dprt_ray* rays,
                          dprt_hit* hits, int64_t n, int32_t* queue, unsigned long long* counters, cudaStream_t stream);

// Vis pipeline epilogue (vis_ray_kernel.cu:145-160): features and label of every traced training ray of object `obj`
void launch_train_features(const DevObject* obj, const dprt_ray* rays, const dprt_hit* hits, int64_t n, float* features,
                           float* labels, cudaStream_t stream);

// Precom pipeline (precom_ray_kernel.cu:193-299): AABB stage (features, t_aabb; rewrites the staged rays' tMax to inf for the
// geometry trace that follows), then the label from the geometry hit
void launch_precom_features(const DevObject* obj, dprt_ray* rays, int64_t n, float* features, float* t_aabb, cudaStream_t stream);
void launch_precom_labels(const DevObject* obj, const dprt_hit* hits, const float* t_aabb, int64_t n, float* labels, uint8_t* valid,
                          cudaStream_t stream);

// dprt_spec_*: the texture / environment look-ups of dprt_math.cuh on host arrays (kernels.cu: same source, host compile)
int spec_texture_sample(const float* rgba, int width, int height, const float* u, const float* v, int64_t n, int clampV, float* out4);
int spec_env_lookup(const float* rgba, int width, int height, float rotationOffset, const float* dirs3, int64_t n, float* out3);

// denoiser (denoise.cu, DESIGN.md 3.8). denoise_check resolves p (NULL: the defaults) into *out and checks the frame size and
// parameters: DPRT_ERR_INVALID with the reason in *why. launch_denoise enqueues the pack launch and one launch per iteration on
// `stream` (scratch: denoise_scratch_bytes(width * height)); out may alias any input. spec_denoise: the same on the host.
int denoise_check(const dprt_denoise_params* p, int width, int height, dprt_denoise_params* out, const char** why);
size_t denoise_scratch_bytes(int64_t pixels);
void launch_denoise(const dprt_denoise_params& p, int width, int height, const float* color, const float* albedo, const float* normal,
                    float* out, void* scratch, cudaStream_t stream);
int spec_denoise(const dprt_denoise_params& p, int width, int height, const float* color, const float* albedo, const float* normal, float* out);

// BVH8 refit (refit.cu, DESIGN.md 3.9). launch_refit_stats reduces ntris * 9 coordinates into the RefitStats at the start of
// the scratch (refit_scratch_bytes(nnodes)). launch_refit rewrites the triangle records from verts9 (by primID) and then the
// nodes, one launch per depth level: levels holds nlevels + 1 node-index boundaries, level d = [levels[d], levels[d + 1]).
// spec_bvh8_refit: the same on host arrays, after checking every index of the blob (DPRT_ERR_INVALID with the reason in *why).
struct RefitStats { float lo[3], hi[3]; uint32_t nonfinite, pad_; };   // over the finite coordinates; count of the others
size_t refit_scratch_bytes(int64_t nnodes);
void launch_refit_stats(const float* verts9, int64_t ntris, void* scratch, cudaStream_t stream);
void launch_refit(dprt_bvh8_node* nodes, dprt_bvh8_tri* tris, int64_t ntris, const float* verts9, const int64_t* levels, int nlevels,
                  float pad, void* scratch, cudaStream_t stream);
int spec_bvh8_refit(dprt_bvh8_node* nodes, int64_t nnodes, dprt_bvh8_tri* tris, int64_t ntris, const float* verts9, const char** why);

// partition / bucketing (partition.cu)
struct PartitionScratch {
    unsigned long long* tileState; // tiles * 32 words {generation, status | value}; zeroed once at allocation, never cleared
    uint32_t* tileCounter;         // running ticket counter (dynamic tile ids); zeroed once, never cleared
    int32_t   maxTiles;
    uint32_t  tickets;             // host mirror: tickets taken by all earlier launches on this scratch
    uint32_t  generation;          // host mirror: launches so far (0 = the zeroed state array matches no launch)
};
void launch_path_histogram(const dprt_path_record* paths, int n, int W, int32_t* hist, cudaStream_t stream);
// B buckets. B == W: bucket = targetNode (reference). B == W + 1 (settled-deque mode): records that stay on rank `me` and
// sit at index >= splitL go to bucket W, so that the self segment comes out in two pieces (before / after the old own block).
void launch_partition_paths(const dprt_path_record* paths, int n, int W, int B, int me, int splitL, const int32_t* hist,
                            dprt_path_record* out, int32_t* offsets, PartitionScratch& s, cudaStream_t stream);
// peer-memory exchange: W + 1 buckets, bucket b's records go to plan->dst[b] + (index inside the bucket); no offsets output
struct P2PPlan;
void launch_partition_paths_peer(const dprt_path_record* paths, int n, int W, int me, int splitL, const P2PPlan* plan,
                                 PartitionScratch& s, cudaStream_t stream);
cudaError_t partition_preload_kernels();
cudaError_t trace_preload_kernels();
void launch_query_histogram(const dprt_nn_query* q, int n, int S, int insideOnly, int32_t* hist, cudaStream_t stream);
// keys: DevParams::nnKey when it is known to mirror q (written by the same launch that wrote q), else null
void launch_partition_queries(const dprt_nn_query* q, const uint8_t* keys, const dprt_half* in, int n, int S, int insideOnly,
                              const int32_t* hist, dprt_nn_query* outQ, dprt_half* outIn, int32_t* offsets,
                              PartitionScratch& s, cudaStream_t stream);

// NN epilogues (epilogue.cu): frame_buffer_update.cu equivalents
void launch_shadow_occlusion(const DevParams& p, int size, cudaStream_t stream);
// live != null: only the `liveCount` pixels listed there can hold non-zero terms (the others fold to a bitwise no-op)
void launch_contribution(const DevParams& p, const int32_t* live, int liveCount, cudaStream_t stream);
// zero the shadow planes 1..spc-1 of directLightingBuffer for the listed pixels (resetNNBuffers by count); nn != 0: also
// their shadowOcclusion / contribution entries (what Frame_Buffer_Update read for them)
void launch_reset_planes(const DevParams& p, const int32_t* live, int liveCount, int nn, cudaStream_t stream);
// zero the tMax scratch Target_Node_Update used for the listed pixels (2*mc floats each in the occlusion buffer)
void launch_reset_sec(const DevParams& p, const int32_t* live, int liveCount, cudaStream_t stream);
void launch_depth_update(const DevParams& p, int size, cudaStream_t stream);
void launch_tmax(const DevParams& p, int size, cudaStream_t stream);
void launch_target_node(const DevParams& p, int n, cudaStream_t stream);
void launch_accumulate(float* direct, float* env, const float* direct2, const float* env2, int n3, cudaStream_t stream);
void launch_image_average(const float* direct, const float* env, float* out, int n3, float invSpp, cudaStream_t stream);
// out = sum / spp: one plane of the first-hit guide buffers
void launch_aov_average(const float* sum, float* out, int n3, float spp, cudaStream_t stream);

}  // namespace dprt
