/*
 * dprt_types.h -- plain-old-data contract of the data-parallel path-tracing hot path.
 *
 * One header, compiled by gcc (oracle, C/C++ hosts), g++ and nvcc. No CUDA, torch or C++ types.
 * Every struct restates a type of the reference that is only knowable from its use sites
 * (SURVEY.md section 2.4); the citation beside each field group is the reference use site
 * (paths relative to the reference tree).
 */
#ifndef DPRT_TYPES_H
#define DPRT_TYPES_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Reference constants: renderer.cpp:1602-1603 (maxCount=3, shadowPathCount=4), util.hpp:10 (Epsilon). */
#define DPRT_DEFAULT_MAX_COUNT 3
#define DPRT_DEFAULT_SHADOW_PATH_COUNT 4
#define DPRT_EPSILON 1e-3f
#define DPRT_MAX_WORLD 32          /* visitedMask is a 32-bit set: distributed_traversal_kernel.cu:29-31 */
#define DPRT_MAX_SCENE_OBJECTS 64
#define DPRT_MAX_LIGHTS 64
#define DPRT_MAX_MATERIALS 256

/* WavefrontPathData: field order from the designated initialiser at optix/kernel.cu:115-129.
 * 64 bytes; all-zero bytes == invalid path (renderer.cpp:354-358 relies on that). This is also the
 * wire format of the path all-to-all (renderer.cpp:1267-1280). */
typedef struct dprt_path_record {
    float    origin[3];
    float    direction[3];
    float    tMax;
    float    throughput[3];
    int32_t  pixelIndex;
    int32_t  shadowPathID;
    uint32_t visitedMask;
    int32_t  currentNode;
    int32_t  targetNode;
    uint8_t  isShadowRay;
    uint8_t  isDelta;
    uint8_t  isValid;
    uint8_t  isHit;
} dprt_path_record;

/* NNPathData: fields from shadow_ray_kernel.cu:284-299,321-341 and secondary_ray_kernel.cu:289-304.
 * 48 bytes; all-zero == empty slot (hitAABBID 0, isValid 0). */
typedef struct dprt_nn_query {
    float    throughput[3];   /* shadow: path contribution; secondary: {t_aabb, maxLength, t_aabb/|oL-pL|} */
    int32_t  pixelIndex;
    int32_t  hitSequence;     /* "hitScequnce" in the reference: 0..maxCount-1 */
    int32_t  hitAABBID;       /* scene index + 1; 0 = empty */
    int32_t  shadowPathID;
    int32_t  instanceID;
    int32_t  pathIndex;       /* shadow/inside: unpacked slot index; secondary: proxy owner nodeID */
    float    normalizedT;
    uint8_t  isValid;
    uint8_t  isInside;
    uint8_t  pad_[2];
    int32_t  reserved_;       /* pads the record to 48 bytes (three 16-byte words) */
} dprt_nn_query;

/* NN_Float == IEEE binary16 (shadow_ray_kernel.cu:279, renderer.cpp:801). Features are 5 halves per query. */
typedef uint16_t dprt_half;
#define DPRT_NN_FEATURES 5

/* aabbRecord + AccelerationStructure (renderer.cpp:1812-1842): one entry per scene object as seen from
 * one rank. isProxy != 0: this rank holds only the object's AABB and its proxy MLPs. */
typedef struct dprt_object_desc {
    int32_t nodeID;           /* owner rank */
    int32_t isProxy;
    float   aabbMin[3];       /* object-space AABB (m_minX.. m_maxZ) */
    float   aabbMax[3];
    float   maxLength;        /* AABB diagonal, renderer.cpp:1830 */
    float   worldToObject[12];/* row-major 3x4; identity for the synthetic scenes */
} dprt_object_desc;

/* HitGroupData subset (pipeline_helper.cpp:182-193): per-mesh base colour and BSDF type. */
typedef struct dprt_material {
    float   baseColor[3];
    int32_t bsdfType;         /* 0 = Diffuse (Lambertian), 1 = Water, 2 = rough conductor (baseColor is F0; roughness from
                                 dprt_set_material_roughness, DESIGN.md 3.12), 3 = glossy plastic (baseColor is the diffuse
                                 colour under a GGX coat of F0 0.04 and the same roughness, DESIGN.md 3.13); any other value
                                 shades as 0 */
} dprt_material;

/* ---- real-scene front end (SURVEY.md 8f row 3) ------------------------------------------------------------------------
 * One triangle mesh of a scene object with its shading attributes in the reference's INDEXED form: a GAS plus the
 * HitGroupData of its SBT record (pipeline_helper.cpp:182-193: normals / normalIndices / texCoords / texCoordsIndices /
 * materialID; kernel.cu:205-262 reads them per hit). All pointers are caller-owned host memory. */
typedef struct dprt_mesh_desc {
    const float*   positions;        /* nPositions * 3, object space */
    int64_t        nPositions;
    const int32_t* indices;          /* ntris * 3 vertex indices */
    int64_t        ntris;
    const float*   normals;          /* nNormals * 3 */
    int64_t        nNormals;
    const int32_t* normalIndices;    /* ntris * 3 */
    const float*   texCoords;        /* nTexCoords * 2; NULL = the mesh has no texture coordinates */
    int64_t        nTexCoords;
    const int32_t* texCoordIndices;  /* ntris * 3; NULL with texCoords */
    int32_t        materialID;       /* HitGroupData.materialID: one material (base colour, BSDF, texture) per mesh record */
    int32_t        pad_;
} dprt_mesh_desc;

/* One instance of a mesh inside a scene object: the reference nests up to three traversable levels ("obj for small
 * details / instanced details yields element / instanced element yields scene object", pipeline_helper.cpp:268-272);
 * the host composes the levels into one object-to-world matrix per leaf instance (row-major 3x4). */
typedef struct dprt_instance_desc {
    int32_t mesh;                    /* index into the mesh array */
    int32_t pad_;
    float   objectToWorld[12];
} dprt_instance_desc;

#define DPRT_MAX_TEXTURES 64         /* albedoTextures[] slots (renderer.cpp:1621-1721) */

/* moana Triangle light + radiance (renderer.cpp:1725-1808, kernel.cu:95-99). */
typedef struct dprt_light_tri {
    float p0[3], p1[3], p2[3];
    float Le[3];
} dprt_light_tri;

/* Pinhole camera. The reference Camera class is not in the tree (path_gen_kernel.cu:58-61 is the only
 * use); the basis vectors are pre-scaled by the host: U = right*aspect*tan(vfov/2), V = up*tan(vfov/2). */
typedef struct dprt_camera {
    float origin[3];
    float U[3];
    float V[3];
    float W[3];
    int32_t width;
    int32_t height;
} dprt_camera;

/* RenderRequest + Params scalars (renderer.cpp:1599-1605). */
typedef struct dprt_config {
    int32_t width;
    int32_t height;
    int32_t spp;
    int32_t bounces;          /* the sample loop runs bounces+1 iterations: renderer.cpp:1530 */
    int32_t shadowPathCount;  /* spc */
    int32_t maxCount;         /* mc */
    int32_t sceneSize;        /* number of scene objects (local + proxy) */
    int32_t proxyMode;        /* 1 = reference behaviour (neural proxies), 0 = sequential visiting only */
    int32_t pathGenMode;      /* 0 = rank 0 generates all camera paths (renderer.cpp:1514), 1 = striped */
    int32_t mlpDtype;         /* 1 = fp16 operands (the reference's NN_Float; meets the 1e-3 proxy tolerance; what every host here defaults to), 0 = bf16 operands (opt-in, ~3e-3); fp32 accumulate either way */
    float   envColor[3];      /* analytic environment: Le = envColor * (0.5 + 0.5*dir.z) */
    int32_t mainRayRetrace;   /* 0 = MainRay reuses the closest hit TraRay / SecondaryRay found for the same ray on this rank
                                 (identical result, see DESIGN.md "hit cache"); 1 = always re-trace like kernel.cu:382-413 */
    int32_t serialStages;     /* 0 = dprt_render_sample may run the ShadowRay module of bounce b on a second CUDA stream beside
                                 the TraRay loop of bounce b+1 (independent data, same results; proxyMode 0 only);
                                 1 = every stage strictly in order on one stream */
    int32_t referenceMigrate; /* 0 = the migrate loop of dprt_primary_ray_module keeps paths that have reached their final rank in
                                 a double-ended buffer and only traces / partitions / sends the ones still travelling (same
                                 final buffers, DESIGN.md "settled deque"); 1 = every iteration handles every path, as
                                 Work_Efficient_Scan + MPI_Alltoallv do (renderer.cpp:1212-1318) */
} dprt_config;

/* Standalone closest-hit query (the optixTrace equivalent used by BASELINE config 2). */
typedef struct dprt_ray {
    float origin[3];
    float tMin;
    float direction[3];
    float tMax;
} dprt_ray;

typedef struct dprt_hit {
    float   t;                /* FLT_MAX-initialised tMax when no hit */
    int32_t primID;           /* original triangle index, -1 = miss */
} dprt_hit;

/* Edge-avoiding a-trous denoiser (dprt_denoise, DESIGN.md 3.8). NULL parameters select the defaults below. */
typedef struct dprt_denoise_params {
    int32_t iterations;       /* L in 1..DPRT_DENOISE_MAX_ITERATIONS; iteration i reads taps 2^i pixels apart */
    float sigma_color;        /* colour (albedo-demodulated) edge-stopping sigma of iteration 0; halves every iteration */
    float sigma_normal;
    float sigma_albedo;
} dprt_denoise_params;
#define DPRT_DENOISE_MAX_ITERATIONS 10
#define DPRT_DENOISE_MAX_PIXELS (1 << 28)
#define DPRT_DENOISE_DEFAULT_ITERATIONS 3        /* defaults: the CPU quality study of profiles/denoise_quality.txt */
#define DPRT_DENOISE_DEFAULT_SIGMA_COLOR 2.0f
#define DPRT_DENOISE_DEFAULT_SIGMA_NORMAL 1.0f
#define DPRT_DENOISE_DEFAULT_SIGMA_ALBEDO 0.3f

/* Compressed wide BVH node, 80 bytes (Ylitie, Karras, Laine 2017 layout). */
typedef struct dprt_bvh8_node {
    float    p[3];
    uint8_t  e[3];
    uint8_t  imask;
    uint32_t childBase;       /* first internal child; child in slot s is childBase + popcount(imask & ((1 << s) - 1)) */
    uint32_t triBase;         /* first leaf triangle; the triangle behind tmask bit b is triBase + popcount(tmask & ((1 << b) - 1)) */
    uint32_t tmask;           /* bit 3 s + k: the leaf child in slot s has a k-th triangle (leaves hold <= 3) */
    uint32_t reserved_;
    uint8_t  qlox[8], qloy[8], qloz[8];
    uint8_t  qhix[8], qhiy[8], qhiz[8];
} dprt_bvh8_node;

/* Leaf-ordered triangle, 48 bytes. pad_ is 0 for a chunk without texture coordinates; for a chunk uploaded with them it
 * holds the chunk's triangle count in every record: the per-corner texture coordinates (32 bytes per triangle, leaf order:
 * u0 v0 u1 v1 | u2 v2 0 0) follow the triangle array in the same allocation, so a kernel that holds a triangle pointer finds
 * them without another table (bvh_traverse.cuh: alpha cut-out any-hit). */
typedef struct dprt_bvh8_tri {
    float    v0[3]; int32_t primID;
    float    v1[3]; int32_t matID;
    float    v2[3]; int32_t pad_;
} dprt_bvh8_tri;

/* Per-stage counters (the std::cout counters of renderer.cpp:1269,1283,1008,1156,1317 as data). */
typedef struct dprt_stats {
    int64_t rays_traverse;    /* paths traced by TraRay launches */
    int64_t rays_shade;
    int64_t rays_shadow;
    int64_t rays_secondary;
    int64_t nn_queries;       /* MLP rows evaluated (vis + depth) */
    int64_t paths_sent_offrank;
    int64_t exchange_iters;
    int64_t kernel_launches;
    int64_t bytes_alltoall;
    int64_t rays_shade_cached; /* subset of rays_shade answered from the hit cache instead of a second BVH walk */
    int64_t rays_walked;       /* rays of all four stages that actually walked a local BVH: live record, at least one local
                                  object not yet visited, not answered from the hit cache (rays_* count launch sizes, like
                                  the reference's optixLaunch dimensions) */
    int64_t walked_traverse;   /* rays_walked split by stage (TraRay / MainRay / ShadowRay / SecondaryRay): the rays whose records */
    int64_t walked_shade;      /* a launch actually traced -- what bench.py bills record bytes for (riders of a TraRay launch  */
    int64_t walked_shadow;     /* and cache-answered MainRay queries are in rays_* but not here)                               */
    int64_t walked_secondary;
    int64_t paths_partitioned; /* records written by the path partition (Work_Efficient_Scan): the reorder roofline's unit */
    int64_t shade_cache_stale; /* single-rank bounce of dprt_render_sample: MainRay queries whose hit-cache entry was of another
                                  epoch (an invariant says never; shaded with the stale entry, so any non-zero count is a bug) */
} dprt_stats;

/* Buffer identifiers for dprt_download/dprt_upload (parity harness access to Params buffers). */
enum dprt_buffer_id {
    DPRT_BUF_PATHS = 0,        /* pathDataBuffer: (1+spc)*N records */
    DPRT_BUF_TRANSFER = 1,     /* transferPathDataBuffer: N records */
    DPRT_BUF_TRANSFER_OFFSET = 2, /* W+1 ints */
    DPRT_BUF_DIRECT = 3,       /* directLightingBuffer: spc planes of 3N floats */
    DPRT_BUF_ENV = 4,          /* envLightingBuffer: 3N floats */
    DPRT_BUF_NN_INPUT = 5,     /* inputDataBuffer: 5 halves per slot */
    DPRT_BUF_NN_QUERY = 6,     /* NNPathDataBuffer */
    DPRT_BUF_NN_PACKED_INPUT = 7,
    DPRT_BUF_NN_PACKED_QUERY = 8,
    DPRT_BUF_SCENE_OFFSET = 9, /* sceneSize+1 ints */
    DPRT_BUF_PRED = 10,        /* predBuffer halves */
    DPRT_BUF_OCCLUSION = 11,   /* shadowOcclusionFloatTypeBuffer */
    DPRT_BUF_CONTRIBUTION = 12,
    DPRT_BUF_HIT_PRIM = 13,    /* parity aid: per path slot hit primitive id of the last trace */
    DPRT_BUF_AOV = 14,         /* first-hit guide buffers (dprt_enable_aov): albedo sums 3N floats, then normal sums 3N floats */
    DPRT_BUF_COUNT = 15
};

/* Stage identifiers for dprt_get_stage_times / dprt_get_counters: one per reference call site of runSample. */
enum dprt_stage_id {
    DPRT_STAGE_PATH_GEN = 0,
    DPRT_STAGE_TRAVERSE = 1,
    DPRT_STAGE_PARTITION = 2,
    DPRT_STAGE_EXCHANGE = 3,
    DPRT_STAGE_SHADE = 4,
    DPRT_STAGE_SHADOW_TRACE = 5,
    DPRT_STAGE_SECONDARY_TRACE = 6,
    DPRT_STAGE_BUCKET = 7,
    DPRT_STAGE_PROXY_MLP = 8,
    DPRT_STAGE_FRAME_UPDATE = 9,
    DPRT_STAGE_DEPTH_UPDATE = 10,
    DPRT_STAGE_TARGET_UPDATE = 11,
    DPRT_STAGE_IMAGE = 12,
    DPRT_STAGE_TRACE_CLOSEST = 13,
    DPRT_STAGE_COUNT = 14
};

/* bytes one rank exports for the peer-memory exchange (dprt_p2p_export): three CUDA IPC handles + a status word */
#define DPRT_P2P_HANDLE_BYTES 208

enum dprt_error {
    DPRT_OK = 0,
    DPRT_ERR_INVALID = -1,
    DPRT_ERR_CUDA = -2,
    DPRT_ERR_NCCL = -3,
    DPRT_ERR_CAPACITY = -4,
    DPRT_ERR_STATE = -5
};

#ifdef __cplusplus
}
#endif
#endif /* DPRT_TYPES_H */

#ifdef __cplusplus
static_assert(sizeof(dprt_path_record) == 64, "dprt_path_record must be 64 bytes");
static_assert(sizeof(dprt_nn_query) == 48, "dprt_nn_query must be 48 bytes");
static_assert(sizeof(dprt_bvh8_node) == 80, "dprt_bvh8_node must be 80 bytes");
static_assert(sizeof(dprt_bvh8_tri) == 48, "dprt_bvh8_tri must be 48 bytes");
static_assert(sizeof(dprt_ray) == 32 && sizeof(dprt_hit) == 8, "ray/hit layout");
static_assert(sizeof(dprt_config) == 64 && sizeof(dprt_object_desc) == 84 && sizeof(dprt_camera) == 56, "config layout");
static_assert(sizeof(dprt_mesh_desc) == 88 && sizeof(dprt_instance_desc) == 56, "mesh / instance layout");
#endif
