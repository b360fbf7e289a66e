// dprt_api.cu -- context, buffer ownership, stage sequencing and the C ABI of libdprt.so.
//
// Host-side restatement of src/render/renderer.cpp: mallocBuffers/deferredMallocBuffers (:547-741), the reset
// helpers (:336-514), primaryRayModule (:1212-1318), generateSecondaryAndShadowRay (:1320-1347),
// shadowRayModuleBasedNN (:1349-1405), secondaryRayModuleBasedNN (:1407-1452), runSample (:1457-1574) and the
// image average + reduce of launch() (:2031-2052). OptiX launches become the kernels of kernels.cu, the
// Work_Efficient_Scan* loops the single-pass partition of partition.cu, torch::jit forward the fused MLP of
// mlp.cu, and host-staged MPI becomes NCCL on device buffers. There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types only: the library is bound at run time (see NcclApi)

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "dprt.h"
#include "dprt_internal.cuh"
#include "bvh_build.h"
#include "bvh_node.cuh"
#include "scene_flatten.h"
#include "mlp.cuh"
#include "p2p_exchange.cuh"

using namespace dprt;

struct dprt_bvh8 { Bvh8 b; };

constexpr int kDevStats = 3 + DPRT_STAGE_COUNT;     // words of dprt_ctx::d_cacheHits

namespace {

std::string g_create_error;

// Streams this library has created per device. The peer-memory exchange parks a waiting kernel in a context's stream;
// when two streams share a hardware queue (CUDA_DEVICE_MAX_CONNECTIONS, 8 by default) whatever is queued behind that kernel
// waits with it, and with several contexts per rank (samples in flight) that can close a cycle across ranks. The waits are
// bounded, so it would end in DPRT_ERR_STATE rather than a hang -- but it is refused up front instead (create_impl).
std::atomic<int> g_streams[64];
int max_connections() {
    const char* e = getenv("CUDA_DEVICE_MAX_CONNECTIONS");
    const int v = e ? atoi(e) : 8;
    return v < 1 ? 1 : (v > 32 ? 32 : v);
}

// NCCL is resolved with dlopen("libnccl.so.2") on first use instead of a link-time dependency: when the
// process already holds a copy (torch bundles its own, newer one) glibc hands back that very library, and a
// single-rank user of libdprt never needs NCCL at all.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
    bool load() {
        if (handle) return true;
        handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!handle) { error = std::string("dlopen(libnccl.so.2): ") + dlerror(); return false; }
        auto sym = [&](const char* n) { void* p = dlsym(handle, n); if (!p) error = std::string("dlsym ") + n; return p; };
        GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
        AllGather = (decltype(AllGather))sym("ncclAllGather");
        Send = (decltype(Send))sym("ncclSend");
        Recv = (decltype(Recv))sym("ncclRecv");
        Reduce = (decltype(Reduce))sym("ncclReduce");
        GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
        GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
        if (!error.empty()) { dlclose(handle); handle = nullptr; return false; }
        return true;
    }
};
NcclApi g_nccl;

// Device memory of one scene object (chunk geometry or the two proxy networks). Shared, not copied, between the contexts of a
// rank that render samples of the same scene (dprt_adopt_scene): freed when the last of them lets go, in whatever order
// the contexts are destroyed.
struct ObjMem {
    int device = 0;
    void* d_nodes = nullptr; void* d_tris = nullptr; void* d_normals = nullptr;
    MlpModel* vis = nullptr; MlpModel* depth = nullptr;
    std::vector<int64_t> levels;     // chunk BVH8: node-index boundaries of the depth levels (dprt_refit_chunk), levels.size() - 1 levels
    ~ObjMem() {
        cudaSetDevice(device);
        if (d_nodes) cudaFree(d_nodes);
        if (d_tris) cudaFree(d_tris);
        if (d_normals) cudaFree(d_normals);
        if (vis) mlp_destroy(vis);
        if (depth) mlp_destroy(depth);
    }
};

// Texels of one albedo / opacity map or of the environment map; shared between the contexts of a rank like ObjMem.
struct TexMem {
    int device = 0; void* d = nullptr; int w = 0, h = 0;
    ~TexMem() { cudaSetDevice(device); if (d) cudaFree(d); }
};

struct ObjectHost {
    bool present = false;
    dprt_object_desc desc{};
    std::shared_ptr<ObjMem> mem;     // owner of everything below
    void* d_nodes = nullptr; void* d_tris = nullptr; void* d_normals = nullptr;
    int64_t nnodes = 0, ntris = 0;
    MlpModel* vis = nullptr; MlpModel* depth = nullptr;
    void release() { mem.reset(); d_nodes = d_tris = d_normals = nullptr; vis = depth = nullptr; nnodes = ntris = 0; }
};

}  // namespace

struct dprt_ctx {
    dprt_config cfg{};
    int rank = 0, world = 1, device = 0;
    int N = 0;
    cudaStream_t stream = nullptr;
    ncclComm_t comm = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    DevParams hp{};
    std::vector<ObjectHost> objects;
    DevObject* d_objects = nullptr;
    dprt_material* d_materials = nullptr;
    dprt_light_tri* d_lights = nullptr;
    // real-scene front end: texture table (DPRT_MAX_TEXTURES slots), texture index per material (-1 = none), environment map
    DevTexture* d_textures = nullptr;
    int32_t* d_matTex = nullptr;
    std::shared_ptr<TexMem> tex[DPRT_MAX_TEXTURES];
    std::shared_ptr<TexMem> envTex;
    size_t buf_bytes[DPRT_BUF_COUNT] = {0};
    void* buf_ptr[DPRT_BUF_COUNT] = {nullptr};
    MlpGroupEntry* d_mlpTable = nullptr; // [2][32]: per kind (vis, depth) the proxy network of every scene object (grouped MLP launch)
    int32_t* d_hist = nullptr;          // 32 path + 64 query counters
    PartitionScratch scratch{};
    uint8_t* d_nnKey = nullptr;         // one key byte per NN query slot
    HitRec* d_hits = nullptr;           // N closest-hit records (MainRay)
    HitRec* d_hitCache = nullptr;       // N per-pixel closest hits of the current epoch (null when cfg.mainRayRetrace)
    unsigned long long* d_cacheHits = nullptr;   // kDevStats words: [0] MainRay queries answered from the cache, [1] rays that walked a BVH, [2 + stage] per stage,
                                                 // [2 + DPRT_STAGE_COUNT] stale hit-cache entries met by launch_shade_cached (since reset_stats)
    // "reset by count" of the shadow planes of directLightingBuffer: MainRay records which pixels get shadow paths
    // (two lists, ping-pong: one describes the planes that are dirty now, the other is free for the next MainRay)
    int32_t* d_live[2] = {nullptr, nullptr};
    int liveCount[2] = {0, 0};
    int shadeIdx = -1;                  // list written by the last dprt_shade whose shadow paths are still in place; -1 = none
    int dirtyIdx = -1;                  // which list covers the dirty planes; -1 = planes are clean, -2 = unknown (full memset)
    // settled deque of the migrate loop (cfg.referenceMigrate == 0, W > 1): paths that have reached their final rank
    dprt_path_record* d_settled = nullptr;   // 2N records; the block [front, back) grows at both ends from the middle
    int front = 0, back = 0;
    int nL = 0;                         // active records [0, nL) came from lower ranks, [nL, pathSize) from higher ones
    // peer-memory exchange (p2p_exchange.cuh; DPRT_P2P=0 forces the NCCL fallback)
    bool p2p = false;                   // tables connected: the deque exchange runs over peer memory
    bool p2pGroup = false;              // connected as an in-process group (dprt_*_group only)
    bool p2pGroupActive = false;        // the group driver is running the peer-memory exchange right now
    std::shared_ptr<void> commKeep;     // the communicator's owner handle, shared with the contexts created from this one (dprt_create_shared)
    int countedStreams = 0;             // this context's share of g_streams[device]
    P2PMailbox* d_mailbox = nullptr;
    dprt_path_record* d_active[2] = {nullptr, nullptr};    // arrivals land here (never in `paths`)
    P2PPeers* d_peers = nullptr;
    P2PPlan* d_plan = nullptr;
    P2PHostPlan* h_plan = nullptr;      // mapped pinned memory the host polls
    P2PHostPlan* d_hplan = nullptr;     // device address of h_plan
    uint32_t p2pSeq = 0;                // one per migrate iteration, never reset
    std::vector<void*> ipcOpened;       // peer mappings to close
    int32_t* d_secLive = nullptr;       // pixels whose tMax scratch the last Target_Node_Update used
    int secDirty = 0;                   // entries of d_secLive to clear at the next resetNNBuffers
    bool nnScratchDirty = false;        // occlusion / contribution may hold non-zero data
    uint32_t epoch = 1;                 // bumped whenever the rays behind the path records change (new bounce, new paths)
    int32_t* d_queue = nullptr;         // ray queue head of the persistent trace kernel
    // second stream for the ShadowRay module of dprt_render_sample (cfg.serialStages == 0, proxies off)
    cudaStream_t aux = nullptr;
    cudaEvent_t evShade = nullptr, evAux = nullptr;
    int32_t* d_queue_aux = nullptr;     // trace scratch of launches on the aux stream
    bool auxPending = false;            // aux work not yet joined into `stream`
    int auxGuardBase = 0;               // first path slot the pending aux work reads (its shadow paths start there)
    // single-rank bounce inside dprt_render_sample (single_rank_shortcut): the exchange leaves the partition output in
    // `transfer` and MainRay shades it from there with the hits of the hit cache
    bool shortcut = false;
    bool recsInTransfer = false;        // set by such an exchange, consumed by the dprt_shade that follows
    // first-hit guide buffers (dprt_enable_aov): buf_ptr[DPRT_BUF_AOV] while enabled, else null
    float* d_aov = nullptr;
    bool aovPending = false;            // armed by dprt_begin_sample, consumed by the dprt_shade that follows
    float* d_image = nullptr;           // averaged image, 3N
    float* d_image_sum = nullptr;       // reduce target, 3N
    int32_t* d_gather = nullptr;        // W*(W+1) offsets of all ranks
    int32_t* h_pinned = nullptr;        // pinned staging for counts/offsets
    void* d_flush = nullptr; size_t flush_bytes = 0;
    void* d_io = nullptr; size_t io_bytes = 0;   // staging for the standalone host-buffer operators
    void* d_denoise = nullptr; size_t denoise_bytes = 0;   // denoiser scratch (dprt_denoise_device): grown to the largest frame
    void* d_refit = nullptr; size_t refit_bytes = 0;       // refit scratch (dprt_refit_chunk_device): grown to the largest chunk
    int pathSize = 0, shadowPathSize = 0;
    int sample = 0;
    int queryTotal = 0;                 // rows of the last bucketing
    int queryWhich = 0;
    std::vector<int> h_sceneOffset;
    bool histFresh = false;             // pathHist holds the histogram of the current paths
    bool qhistFresh = false;            // queryHist holds the histograms of the current queries
    std::vector<int> h_offsets;         // last transferOffset (W+1)
    dprt_stats stats{};
    std::string err;
    std::vector<void*> user_allocs;
    // per-stage device timing (dprt_stage_profile): event pairs recorded around each stage, resolved lazily
    bool profile = false;
    std::vector<cudaEvent_t> evPool;
    struct Pending { int stage; cudaEvent_t a, b; };
    std::vector<Pending> pending;
    double stageMs[DPRT_STAGE_COUNT] = {0};
    int64_t stageLaunches[DPRT_STAGE_COUNT] = {0};
    unsigned long long* d_counters = nullptr;   // 2*DPRT_STAGE_COUNT, allocated on first dprt_enable_counters
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
            return DPRT_ERR_CUDA;                                                                  \
        }                                                                                          \
    } while (0)

#define NK(call)                                                                                   \
    do {                                                                                           \
        ncclResult_t e_ = (call);                                                                  \
        if (e_ != ncclSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + g_nccl.GetErrorString(e_);                         \
            return DPRT_ERR_NCCL;                                                                  \
        }                                                                                          \
    } while (0)

int fail(dprt_ctx* ctx, int code, const std::string& msg) { ctx->err = msg; return code; }

// peer-memory exchange, defined further down (inside the extern "C" part of this file)
extern "C" {
bool p2p_requested();
int p2p_connect_nccl(dprt_ctx* ctx);
void p2p_free(dprt_ctx* ctx);
}

// makes `stream` wait for the ShadowRay module that dprt_render_sample left running on the aux stream
int join_aux(dprt_ctx* ctx) {
    if (ctx->auxPending) {
        ctx->auxPending = false;
        CK(cudaStreamWaitEvent(ctx->stream, ctx->evAux, 0));
    }
    return 0;
}

void resolve_pending(dprt_ctx* ctx) {
    for (auto& pd : ctx->pending) {
        float ms = 0.f;
        if (cudaEventSynchronize(pd.b) == cudaSuccess && cudaEventElapsedTime(&ms, pd.a, pd.b) == cudaSuccess) {
            ctx->stageMs[pd.stage] += ms; ctx->stageLaunches[pd.stage] += 1;
        }
        ctx->evPool.push_back(pd.a); ctx->evPool.push_back(pd.b);
    }
    ctx->pending.clear();
}

// Brackets one stage with an event pair on the context's stream when profiling is on (a no-op otherwise).
struct StageScope {
    dprt_ctx* ctx; int stage; cudaEvent_t a = nullptr, b = nullptr;
    StageScope(dprt_ctx* c, int st, bool active = true) : ctx(c), stage(st) {
        if (!ctx->profile || !active) return;
        if (ctx->pending.size() >= 8192) resolve_pending(ctx);
        auto get = [&]() {
            cudaEvent_t e = nullptr;
            if (!ctx->evPool.empty()) { e = ctx->evPool.back(); ctx->evPool.pop_back(); } else cudaEventCreate(&e);
            return e;
        };
        a = get(); b = get();
        cudaEventRecord(a, ctx->stream);
    }
    ~StageScope() {
        if (!a) return;
        cudaEventRecord(b, ctx->stream);
        ctx->pending.push_back({stage, a, b});
    }
};

int alloc_buf(dprt_ctx* ctx, int id, size_t bytes) {
    bytes = std::max<size_t>(bytes, 256);
    CK(cudaMalloc(&ctx->buf_ptr[id], bytes));
    CK(cudaMemsetAsync(ctx->buf_ptr[id], 0, bytes, ctx->stream));
    ctx->buf_bytes[id] = bytes;
    return 0;
}

void sync_params(dprt_ctx* ctx) {
    DevParams& p = ctx->hp;
    p.pathSize = ctx->pathSize; p.shadowPathSize = ctx->shadowPathSize;
    p.spc = ctx->cfg.shadowPathCount; p.mc = ctx->cfg.maxCount; p.sceneSize = ctx->cfg.sceneSize;
    p.worldID = ctx->rank; p.worldSize = ctx->world; p.sampleCount = ctx->sample;
    p.frameBufferSize = ctx->N; p.proxyMode = ctx->cfg.proxyMode; p.pathGenMode = ctx->cfg.pathGenMode;
    for (int k = 0; k < 3; k++) p.envColor[k] = ctx->cfg.envColor[k];
    p.splitL = 0x7fffffff;
    p.hitCache = ctx->d_hitCache; p.hitEpoch = ctx->epoch; p.cacheHits = ctx->d_cacheHits;
}

int upload_objects(dprt_ctx* ctx) {
    std::vector<DevObject> h(ctx->cfg.sceneSize);
    for (int i = 0; i < ctx->cfg.sceneSize; i++) {
        const ObjectHost& o = ctx->objects[i];
        DevObject d{};
        d.nodeID = o.present ? o.desc.nodeID : 0; d.isProxy = o.present ? (o.desc.isProxy ? 1 : 0) : 2;   // 2 = slot not uploaded: skipped everywhere
        if (!o.present) {   // never hit: inverted box
            for (int a = 0; a < 3; a++) { d.aabbMin[a] = 1.f; d.aabbMax[a] = -1.f; }
            d.w2o[0] = d.w2o[5] = d.w2o[10] = 1.f;
        } else {
            std::memcpy(d.aabbMin, o.desc.aabbMin, 12); std::memcpy(d.aabbMax, o.desc.aabbMax, 12);
            d.maxLength = o.desc.maxLength; std::memcpy(d.w2o, o.desc.worldToObject, 48);
        }
        d.nodes = (const uint4*)o.d_nodes; d.tris = (const float4*)o.d_tris; d.normals = (const float*)o.d_normals;
        h[i] = d;
    }
    CK(cudaMemcpyAsync(ctx->d_objects, h.data(), h.size() * sizeof(DevObject), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int ensure_io(dprt_ctx* ctx, size_t bytes) {
    if (ctx->io_bytes >= bytes) return 0;
    if (ctx->d_io) cudaFree(ctx->d_io);
    ctx->d_io = nullptr; ctx->io_bytes = 0;
    CK(cudaMalloc(&ctx->d_io, bytes));
    ctx->io_bytes = bytes;
    return 0;
}

// reads transferOffset (W+1 ints) to the host
int read_offsets(dprt_ctx* ctx) {
    const int W = ctx->world;
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->hp.transferOffset, (W + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->h_offsets.assign(ctx->h_pinned, ctx->h_pinned + W + 1);
    return 0;
}

}  // namespace

// ================================================================================================
extern "C" {

int dprt_get_unique_id(void* out128) {
    if (!out128) return DPRT_ERR_INVALID;
    ncclUniqueId id;
    if (!g_nccl.load()) { g_create_error = g_nccl.error; return DPRT_ERR_NCCL; }
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) return DPRT_ERR_NCCL;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    std::memcpy(out128, &id, 128);
    return 0;
}

const char* dprt_last_error(const dprt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

static int create_impl(const dprt_config* cfg, int rank, int world, int device, const void* nccl_unique_id, dprt_ctx* parent, dprt_ctx** out) {
    if (!cfg || !out) { g_create_error = "null argument"; return DPRT_ERR_INVALID; }
    *out = nullptr;
    if (world < 1 || world > DPRT_MAX_WORLD || rank < 0 || rank >= world || cfg->width <= 0 || cfg->height <= 0 ||
        cfg->sceneSize < 1 || cfg->sceneSize > 32 || cfg->shadowPathCount < 1 || cfg->maxCount < 1 || cfg->maxCount > 8 ||
        cfg->shadowPathCount > 16 || cfg->spp < 1 || cfg->bounces < 0 || (int64_t)cfg->width * cfg->height > (int64_t)0x7fffffff / 64) {
        g_create_error = "invalid configuration"; return DPRT_ERR_INVALID;
    }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(ce) + " (libdprt has no CPU fallback)";
        return DPRT_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { g_create_error = "device index out of range"; return DPRT_ERR_INVALID; }
    dprt_ctx* ctx = new dprt_ctx();
    ctx->cfg = *cfg; ctx->rank = rank; ctx->world = world; ctx->device = device;
    ctx->N = cfg->width * cfg->height;
    auto bail = [&](int code) { g_create_error = ctx->err; dprt_destroy(ctx); return code; };
    auto body = [&]() -> int {
        CK(cudaSetDevice(device));
        CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        if (device < 64) { g_streams[device]++; ctx->countedStreams++; }
        CK(cudaEventCreate(&ctx->ev0)); CK(cudaEventCreate(&ctx->ev1));
        const size_t N = ctx->N, spc = cfg->shadowPathCount, mc = cfg->maxCount;
        ctx->objects.resize(cfg->sceneSize);
        CK(cudaMalloc(&ctx->d_objects, sizeof(DevObject) * cfg->sceneSize));
        CK(cudaMalloc(&ctx->d_materials, sizeof(dprt_material) * DPRT_MAX_MATERIALS));
        CK(cudaMemsetAsync(ctx->d_materials, 0, sizeof(dprt_material) * DPRT_MAX_MATERIALS, ctx->stream));
        CK(cudaMalloc(&ctx->d_lights, sizeof(dprt_light_tri) * DPRT_MAX_LIGHTS));
        CK(cudaMalloc(&ctx->d_textures, sizeof(DevTexture) * DPRT_MAX_TEXTURES));
        CK(cudaMemsetAsync(ctx->d_textures, 0, sizeof(DevTexture) * DPRT_MAX_TEXTURES, ctx->stream));      // texels == null: empty slot
        CK(cudaMalloc(&ctx->d_matTex, sizeof(int32_t) * DPRT_MAX_MATERIALS));
        CK(cudaMemsetAsync(ctx->d_matTex, 0xff, sizeof(int32_t) * DPRT_MAX_MATERIALS, ctx->stream));        // -1: untextured
        int r;
        if ((r = alloc_buf(ctx, DPRT_BUF_PATHS, (1 + spc) * N * sizeof(dprt_path_record)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_TRANSFER, N * sizeof(dprt_path_record)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_TRANSFER_OFFSET, 64 * sizeof(int32_t)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_DIRECT, spc * 3 * N * sizeof(float)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_ENV, 3 * N * sizeof(float)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_SCENE_OFFSET, 64 * sizeof(int32_t)))) return r;
        // N*mc*spc floats (renderer.cpp:709-711); Target_Node_Update reuses the buffer as a [pixel][mc][2] scratch
        // (frame_buffer_update.cu:239-248 -- the reference hard-codes spc = 4), so never fewer than 2 floats per (pixel, mc)
        if ((r = alloc_buf(ctx, DPRT_BUF_OCCLUSION, N * mc * std::max<size_t>(spc, 2) * sizeof(float)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_CONTRIBUTION, 3 * N * spc * sizeof(float)))) return r;
        const size_t Q = cfg->proxyMode ? N * mc * spc : 1;
        if ((r = alloc_buf(ctx, DPRT_BUF_NN_INPUT, Q * 5 * sizeof(dprt_half)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_NN_PACKED_INPUT, Q * 5 * sizeof(dprt_half) + 64))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_NN_QUERY, Q * sizeof(dprt_nn_query)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_NN_PACKED_QUERY, Q * sizeof(dprt_nn_query)))) return r;
        if ((r = alloc_buf(ctx, DPRT_BUF_PRED, Q * 4 * sizeof(dprt_half)))) return r;
        CK(cudaMalloc(&ctx->d_mlpTable, 2 * 32 * sizeof(MlpGroupEntry)));
        CK(cudaMemsetAsync(ctx->d_mlpTable, 0, 2 * 32 * sizeof(MlpGroupEntry), ctx->stream));
        CK(cudaMalloc(&ctx->d_hist, 128 * sizeof(int32_t)));
        CK(cudaMemsetAsync(ctx->d_hist, 0, 128 * sizeof(int32_t), ctx->stream));
        ctx->scratch.maxTiles = (int)((std::max(Q, N) + 1023) / 1024) + 1;     // the smallest tile any partition kernel uses
        CK(cudaMalloc(&ctx->scratch.tileState, (size_t)ctx->scratch.maxTiles * 32 * sizeof(unsigned long long)));
        CK(cudaMemsetAsync(ctx->scratch.tileState, 0, (size_t)ctx->scratch.maxTiles * 32 * sizeof(unsigned long long), ctx->stream));
        CK(cudaMalloc(&ctx->scratch.tileCounter, sizeof(uint32_t)));
        CK(cudaMemsetAsync(ctx->scratch.tileCounter, 0, sizeof(uint32_t), ctx->stream));
        ctx->scratch.tickets = 0u; ctx->scratch.generation = 0u;
        CK(cudaMalloc(&ctx->d_hits, N * sizeof(HitRec)));
        for (int k = 0; k < 2; k++) CK(cudaMalloc(&ctx->d_live[k], N * sizeof(int32_t)));
        if (cfg->proxyMode) CK(cudaMalloc(&ctx->d_secLive, N * sizeof(int32_t)));
        if (!cfg->mainRayRetrace) {
            CK(cudaMalloc(&ctx->d_hitCache, N * sizeof(HitRec)));
            CK(cudaMemsetAsync(ctx->d_hitCache, 0, N * sizeof(HitRec), ctx->stream));      // epoch 0 = never written
        }
        CK(cudaMalloc(&ctx->d_cacheHits, kDevStats * sizeof(unsigned long long)));
        CK(cudaMemsetAsync(ctx->d_cacheHits, 0, kDevStats * sizeof(unsigned long long), ctx->stream));
        CK(cudaMalloc(&ctx->d_queue, trace_scratch_bytes()));
        CK(cudaMemsetAsync(ctx->d_queue, 0, 64, ctx->stream));
        if (!cfg->serialStages && !cfg->proxyMode) {
            int lo = 0, hi = 0;
            CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));          // the main stream carries the critical path: aux gets the lowest priority
            CK(cudaStreamCreateWithPriority(&ctx->aux, cudaStreamNonBlocking, lo));
            if (device < 64) { g_streams[device]++; ctx->countedStreams++; }
            CK(cudaEventCreateWithFlags(&ctx->evShade, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->evAux, cudaEventDisableTiming));
            CK(cudaMalloc(&ctx->d_queue_aux, trace_scratch_bytes()));
            CK(cudaMemsetAsync(ctx->d_queue_aux, 0, 64, ctx->stream));
        }
        CK(cudaMalloc(&ctx->d_image, 3 * N * sizeof(float)));
        CK(cudaMalloc(&ctx->d_image_sum, 3 * N * sizeof(float)));
        CK(cudaMalloc(&ctx->d_gather, sizeof(int32_t) * (size_t)world * (world + 2)));
        CK(cudaMallocHost(&ctx->h_pinned, sizeof(int32_t) * std::max<size_t>(256, (size_t)world * (world + 2))));
        if (world > 1 && world < 32 && !cfg->referenceMigrate) CK(cudaMalloc(&ctx->d_settled, 2 * N * sizeof(dprt_path_record)));

        DevParams& p = ctx->hp;
        p.objects = ctx->d_objects; p.materials = ctx->d_materials; p.lights = ctx->d_lights;
        p.textures = ctx->d_textures; p.matTex = ctx->d_matTex; p.envMap = DevTexture{nullptr, 0, 0}; p.envRotation = 0.0f;
        p.paths = (dprt_path_record*)ctx->buf_ptr[DPRT_BUF_PATHS];
        p.transfer = (dprt_path_record*)ctx->buf_ptr[DPRT_BUF_TRANSFER];
        p.transferOffset = (int32_t*)ctx->buf_ptr[DPRT_BUF_TRANSFER_OFFSET];
        p.pathHist = ctx->d_hist; p.queryHist = ctx->d_hist + 32;
        p.direct = (float*)ctx->buf_ptr[DPRT_BUF_DIRECT]; p.env = (float*)ctx->buf_ptr[DPRT_BUF_ENV];
        p.contribution = (float*)ctx->buf_ptr[DPRT_BUF_CONTRIBUTION]; p.occlusion = (float*)ctx->buf_ptr[DPRT_BUF_OCCLUSION];
        p.nnInput = (dprt_half*)ctx->buf_ptr[DPRT_BUF_NN_INPUT]; p.nnPackedInput = (dprt_half*)ctx->buf_ptr[DPRT_BUF_NN_PACKED_INPUT];
        CK(cudaMalloc(&ctx->d_nnKey, Q));
        p.nnKey = ctx->d_nnKey;
        p.nnQuery = (dprt_nn_query*)ctx->buf_ptr[DPRT_BUF_NN_QUERY]; p.nnPackedQuery = (dprt_nn_query*)ctx->buf_ptr[DPRT_BUF_NN_PACKED_QUERY];
        p.sceneOffset = (int32_t*)ctx->buf_ptr[DPRT_BUF_SCENE_OFFSET];
        p.pred = (dprt_half*)ctx->buf_ptr[DPRT_BUF_PRED];
        p.hitPrim = nullptr; p.counters = nullptr;
        p.hits = ctx->d_hits; p.traceQueue = ctx->d_queue;
        p.camera.width = cfg->width; p.camera.height = cfg->height;
        p.lightCount = 0;
        sync_params(ctx);
        ctx->h_sceneOffset.assign(cfg->sceneSize + 1, 0);
        ctx->h_offsets.assign(world + 1, 0);
        for (int i = 0; i < cfg->sceneSize; i++) { ctx->objects[i].desc.nodeID = 0; ctx->objects[i].desc.isProxy = 1; }
        if ((r = upload_objects(ctx))) return r;
        if (parent && parent->comm && world > 1) {
            ctx->comm = parent->comm; ctx->commKeep = parent->commKeep;   // collectives of the two contexts must not interleave
        } else if (nccl_unique_id && world > 1) {
            ncclUniqueId id; std::memcpy(&id, nccl_unique_id, 128);
            if (!g_nccl.load()) { ctx->err = g_nccl.error; return DPRT_ERR_NCCL; }
            NK(g_nccl.CommInitRank(&ctx->comm, world, id, rank));
            ctx->commKeep = std::shared_ptr<void>((void*)ctx->comm, [](void* c) { if (c) g_nccl.CommDestroy((ncclComm_t)c); });
        }
        // peer-memory exchange: a collective decision over the communicator (all ranks or none, p2p_connect_nccl)
        if (ctx->comm) { int pr = p2p_connect_nccl(ctx); if (pr) return pr; }
        if (ctx->p2p && device < 64 && g_streams[device] > max_connections()) {
            ctx->err = "the contexts of this process hold " + std::to_string((int)g_streams[device]) + " CUDA streams on this device but only " +
                       std::to_string(max_connections()) + " hardware queues (CUDA_DEVICE_MAX_CONNECTIONS): the peer-memory exchange needs a queue per stream. "
                       "Set CUDA_DEVICE_MAX_CONNECTIONS=32 before the first CUDA call, or keep fewer samples in flight";
            return DPRT_ERR_STATE;
        }
        CK(cudaStreamSynchronize(ctx->stream));
        return 0;
    };
    int r = body();
    if (r) return bail(r);
    *out = ctx;
    return 0;
}

int dprt_create(const dprt_config* cfg, int rank, int world, int device, const void* nccl_unique_id, dprt_ctx** out) {
    return create_impl(cfg, rank, world, device, nccl_unique_id, nullptr, out);
}

int dprt_create_shared(const dprt_config* cfg, dprt_ctx* parent, dprt_ctx** out) {
    if (!parent) { g_create_error = "null parent"; return DPRT_ERR_INVALID; }
    return create_impl(cfg, parent->rank, parent->world, parent->device, nullptr, parent, out);
}

void dprt_destroy(dprt_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->device >= 0 && ctx->device < 64) g_streams[ctx->device] -= ctx->countedStreams;
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    ctx->comm = nullptr; ctx->commKeep.reset();          // ncclCommDestroy when the last context on this communicator goes
    for (auto& o : ctx->objects) o.release();
    for (int i = 0; i < DPRT_BUF_COUNT; i++) if (ctx->buf_ptr[i]) cudaFree(ctx->buf_ptr[i]);
    for (void* p : ctx->user_allocs) cudaFree(p);
    if (ctx->d_objects) cudaFree(ctx->d_objects);
    if (ctx->d_materials) cudaFree(ctx->d_materials);
    if (ctx->d_lights) cudaFree(ctx->d_lights);
    if (ctx->d_textures) cudaFree(ctx->d_textures);
    if (ctx->d_matTex) cudaFree(ctx->d_matTex);
    for (auto& t : ctx->tex) t.reset();
    ctx->envTex.reset();
    if (ctx->d_hist) cudaFree(ctx->d_hist);
    if (ctx->d_mlpTable) cudaFree(ctx->d_mlpTable);
    if (ctx->scratch.tileState) cudaFree(ctx->scratch.tileState);
    if (ctx->scratch.tileCounter) cudaFree(ctx->scratch.tileCounter);
    if (ctx->d_hits) cudaFree(ctx->d_hits);
    if (ctx->d_nnKey) cudaFree(ctx->d_nnKey);
    for (int k = 0; k < 2; k++) if (ctx->d_live[k]) cudaFree(ctx->d_live[k]);
    if (ctx->d_secLive) cudaFree(ctx->d_secLive);
    p2p_free(ctx);
    if (ctx->aux) cudaStreamDestroy(ctx->aux);
    if (ctx->evShade) cudaEventDestroy(ctx->evShade);
    if (ctx->evAux) cudaEventDestroy(ctx->evAux);
    if (ctx->d_queue_aux) cudaFree(ctx->d_queue_aux);
    if (ctx->d_hitCache) cudaFree(ctx->d_hitCache);
    if (ctx->d_cacheHits) cudaFree(ctx->d_cacheHits);
    if (ctx->d_queue) cudaFree(ctx->d_queue);
    if (ctx->d_image) cudaFree(ctx->d_image);
    if (ctx->d_image_sum) cudaFree(ctx->d_image_sum);
    if (ctx->d_gather) cudaFree(ctx->d_gather);
    if (ctx->d_settled) cudaFree(ctx->d_settled);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    resolve_pending(ctx);
    for (cudaEvent_t e : ctx->evPool) cudaEventDestroy(e);
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    if (ctx->d_flush) cudaFree(ctx->d_flush);
    if (ctx->d_io) cudaFree(ctx->d_io);
    if (ctx->d_denoise) cudaFree(ctx->d_denoise);
    if (ctx->d_refit) cudaFree(ctx->d_refit);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int dprt_synchronize(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    return 0;
}
int dprt_get_stats(const dprt_ctx* ctx, dprt_stats* out) {
    if (!ctx || !out) return DPRT_ERR_INVALID;
    *out = ctx->stats;
    if (ctx->d_cacheHits) {            // the one statistic that is only known on the device
        unsigned long long v[kDevStats] = {0};
        if (cudaSetDevice(ctx->device) != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess ||
            cudaMemcpy(v, ctx->d_cacheHits, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return DPRT_ERR_CUDA;
        out->rays_shade_cached = (int64_t)v[0]; out->rays_walked = (int64_t)v[1];
        out->walked_traverse = (int64_t)v[2 + DPRT_STAGE_TRAVERSE]; out->walked_shade = (int64_t)v[2 + DPRT_STAGE_SHADE];
        out->walked_shadow = (int64_t)v[2 + DPRT_STAGE_SHADOW_TRACE]; out->walked_secondary = (int64_t)v[2 + DPRT_STAGE_SECONDARY_TRACE];
        out->shade_cache_stale = (int64_t)v[2 + DPRT_STAGE_COUNT];
    }
    return 0;
}
int dprt_reset_stats(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    ctx->stats = dprt_stats{};
    cudaSetDevice(ctx->device);
    resolve_pending(ctx);
    for (int i = 0; i < DPRT_STAGE_COUNT; i++) { ctx->stageMs[i] = 0.0; ctx->stageLaunches[i] = 0; }
    if (ctx->d_counters) CK(cudaMemsetAsync(ctx->d_counters, 0, 2 * DPRT_STAGE_COUNT * sizeof(unsigned long long), ctx->stream));
    if (ctx->d_cacheHits) CK(cudaMemsetAsync(ctx->d_cacheHits, 0, kDevStats * sizeof(unsigned long long), ctx->stream));
    return 0;
}

int dprt_stage_profile(dprt_ctx* ctx, int enable) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    resolve_pending(ctx);
    ctx->profile = enable != 0;
    return 0;
}
int dprt_get_stage_times(dprt_ctx* ctx, double* ms_out, int64_t* launches_out) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    resolve_pending(ctx);
    for (int i = 0; i < DPRT_STAGE_COUNT; i++) {
        if (ms_out) ms_out[i] = ctx->stageMs[i];
        if (launches_out) launches_out[i] = ctx->stageLaunches[i];
    }
    return 0;
}
int dprt_enable_counters(dprt_ctx* ctx, int enable) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (enable && !ctx->d_counters) {
        CK(cudaMalloc(&ctx->d_counters, 2 * DPRT_STAGE_COUNT * sizeof(unsigned long long)));
        CK(cudaMemsetAsync(ctx->d_counters, 0, 2 * DPRT_STAGE_COUNT * sizeof(unsigned long long), ctx->stream));
    }
    ctx->hp.counters = enable ? ctx->d_counters : nullptr;
    return 0;
}
int dprt_get_counters(dprt_ctx* ctx, uint64_t* counts_out) {
    if (!ctx || !counts_out) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->d_counters) { std::memset(counts_out, 0, 2 * DPRT_STAGE_COUNT * sizeof(uint64_t)); return 0; }
    CK(cudaMemcpyAsync(counts_out, ctx->d_counters, 2 * DPRT_STAGE_COUNT * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---- scene -------------------------------------------------------------------------------------
int dprt_bvh8_build(const float* verts9, const int32_t* mat_ids, int64_t ntris, float pad, dprt_bvh8** out) {
    if (!out) return DPRT_ERR_INVALID;
    dprt_bvh8* b = new dprt_bvh8();
    if (bvh8_build(verts9, mat_ids, ntris, pad, b->b)) { delete b; *out = nullptr; return DPRT_ERR_INVALID; }
    *out = b; return 0;
}
int dprt_bvh8_info(const dprt_bvh8* b, int64_t* nnodes, int64_t* ntris, int32_t* max_depth) {
    if (!b) return DPRT_ERR_INVALID;
    if (nnodes) *nnodes = (int64_t)b->b.nodes.size();
    if (ntris) *ntris = (int64_t)b->b.tris.size();
    if (max_depth) *max_depth = b->b.max_depth;
    return 0;
}
int dprt_bvh8_copy(const dprt_bvh8* b, dprt_bvh8_node* nodes_out, dprt_bvh8_tri* tris_out) {
    if (!b) return DPRT_ERR_INVALID;
    if (nodes_out) std::memcpy(nodes_out, b->b.nodes.data(), b->b.nodes.size() * sizeof(dprt_bvh8_node));
    if (tris_out) std::memcpy(tris_out, b->b.tris.data(), b->b.tris.size() * sizeof(dprt_bvh8_tri));
    return 0;
}
void dprt_bvh8_free(dprt_bvh8* b) { delete b; }

int dprt_upload_chunk_uv(dprt_ctx* ctx, int si, const dprt_object_desc* desc, const float* verts9, const float* normals9,
                         const float* uv6, const int32_t* mat_ids, int64_t ntris) {
    if (!ctx || !desc || !verts9 || si < 0 || si >= ctx->cfg.sceneSize || ntris <= 0) return DPRT_ERR_INVALID;
    if (desc->nodeID < 0 || desc->nodeID >= ctx->world) return fail(ctx, DPRT_ERR_INVALID, "nodeID out of range");
    if (ntris >= ((int64_t)1 << 27)) return fail(ctx, DPRT_ERR_CAPACITY, "more than 2^27 triangles in one chunk (bvh_traverse.cuh: DPRT_TRI_BITS)");
    if (mat_ids)
        for (int64_t i = 0; i < ntris; i++)
            if (mat_ids[i] < 0 || mat_ids[i] >= DPRT_MAX_MATERIALS) return fail(ctx, DPRT_ERR_INVALID, "material id out of range");
    CK(cudaSetDevice(ctx->device));
    Bvh8 b;
    if (bvh8_build(verts9, mat_ids, ntris, -1.f, b)) return fail(ctx, DPRT_ERR_INVALID, "bvh8_build failed");
    if (b.max_depth > 36) return fail(ctx, DPRT_ERR_CAPACITY, "BVH8 deeper than the traversal stack");
    ObjectHost& o = ctx->objects[si];
    CK(cudaStreamSynchronize(ctx->stream));            // nothing in flight reads the old geometry
    o.release();
    auto mem = std::make_shared<ObjMem>();
    mem->device = ctx->device;
    o.desc = *desc; o.desc.isProxy = 0; o.present = true;
    const size_t nt = b.tris.size();
    // texture coordinates: 32 bytes per triangle in leaf order behind the triangle array (dprt_bvh8_tri.pad_ = triangle count)
    std::vector<float> uvLeaf;
    if (uv6) {
        uvLeaf.assign(nt * 8, 0.0f);
        for (size_t t = 0; t < nt; t++) {
            b.tris[t].pad_ = (int32_t)nt;
            const float* u = uv6 + 6 * (size_t)b.tris[t].primID;
            for (int k = 0; k < 6; k++) uvLeaf[8 * t + k] = u[k];
        }
    }
    CK(cudaMalloc(&mem->d_nodes, b.nodes.size() * sizeof(dprt_bvh8_node)));
    CK(cudaMalloc(&mem->d_tris, nt * sizeof(dprt_bvh8_tri) + uvLeaf.size() * sizeof(float)));
    CK(cudaMemcpy(mem->d_nodes, b.nodes.data(), b.nodes.size() * sizeof(dprt_bvh8_node), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(mem->d_tris, b.tris.data(), nt * sizeof(dprt_bvh8_tri), cudaMemcpyHostToDevice));
    if (uv6) CK(cudaMemcpy((char*)mem->d_tris + nt * sizeof(dprt_bvh8_tri), uvLeaf.data(), uvLeaf.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (normals9) {
        CK(cudaMalloc(&mem->d_normals, (size_t)ntris * 9 * sizeof(float)));
        CK(cudaMemcpy(mem->d_normals, normals9, (size_t)ntris * 9 * sizeof(float), cudaMemcpyHostToDevice));
    }
    // BFS order: level 0 is the root, and the internal children of level d are exactly level d + 1
    mem->levels.assign(1, 0);
    for (int64_t first = 0, last = 1; first < last;) {
        mem->levels.push_back(last);
        int64_t next = last;
        for (int64_t i = first; i < last; i++)
            if (b.nodes[i].imask) next = std::max<int64_t>(next, (int64_t)b.nodes[i].childBase + __builtin_popcount(b.nodes[i].imask));
        first = last; last = next;
    }
    o.mem = mem; o.d_nodes = mem->d_nodes; o.d_tris = mem->d_tris; o.d_normals = mem->d_normals;
    o.nnodes = (int64_t)b.nodes.size(); o.ntris = (int64_t)nt;
    return upload_objects(ctx);
}

int dprt_upload_chunk(dprt_ctx* ctx, int si, const dprt_object_desc* desc, const float* verts9, const float* normals9,
                      const int32_t* mat_ids, int64_t ntris) {
    return dprt_upload_chunk_uv(ctx, si, desc, verts9, normals9, nullptr, mat_ids, ntris);
}

int64_t dprt_flatten_count(const dprt_mesh_desc* meshes, int n_meshes, const dprt_instance_desc* instances, int64_t n_instances) {
    return flatten_count(meshes, n_meshes, instances, n_instances);
}
int dprt_flatten_instances(const dprt_mesh_desc* meshes, int n_meshes, const dprt_instance_desc* instances, int64_t n_instances,
                           float* verts9, float* normals9, float* uv6, int32_t* mat_ids, int* has_uv) {
    return flatten_instances(meshes, n_meshes, instances, n_instances, verts9, normals9, uv6, mat_ids, has_uv) ? DPRT_ERR_INVALID : 0;
}

int dprt_upload_instanced_chunk(dprt_ctx* ctx, int si, const dprt_object_desc* desc, const dprt_mesh_desc* meshes, int n_meshes,
                                const dprt_instance_desc* instances, int64_t n_instances) {
    if (!ctx || !desc) return DPRT_ERR_INVALID;
    const int64_t nt = flatten_count(meshes, n_meshes, instances, n_instances);
    if (nt <= 0) return fail(ctx, DPRT_ERR_INVALID, "dprt_upload_instanced_chunk: invalid mesh / instance description");
    std::vector<float> verts((size_t)nt * 9), normals((size_t)nt * 9), uv((size_t)nt * 6);
    std::vector<int32_t> mats((size_t)nt);
    int hasUv = 0;
    if (flatten_instances(meshes, n_meshes, instances, n_instances, verts.data(), normals.data(), uv.data(), mats.data(), &hasUv))
        return fail(ctx, DPRT_ERR_INVALID, "dprt_upload_instanced_chunk: index out of range or singular instance transform");
    return dprt_upload_chunk_uv(ctx, si, desc, verts.data(), normals.data(), hasUv ? uv.data() : nullptr, mats.data(), nt);
}

// ---- textures, environment map (renderer.cpp:1621-1721, :1851) ------------------------------------
namespace {
int upload_texels(dprt_ctx* ctx, const float* rgba, int width, int height, std::shared_ptr<TexMem>& out) {
    auto m = std::make_shared<TexMem>();
    m->device = ctx->device; m->w = width; m->h = height;
    const size_t bytes = (size_t)width * height * 4 * sizeof(float);
    CK(cudaMalloc(&m->d, bytes));
    CK(cudaMemcpy(m->d, rgba, bytes, cudaMemcpyHostToDevice));
    out = m;
    return 0;
}
int upload_texture_table(dprt_ctx* ctx) {
    DevTexture h[DPRT_MAX_TEXTURES];
    for (int i = 0; i < DPRT_MAX_TEXTURES; i++)
        h[i] = ctx->tex[i] ? DevTexture{(const float4*)ctx->tex[i]->d, ctx->tex[i]->w, ctx->tex[i]->h} : DevTexture{nullptr, 0, 0};
    CK(cudaMemcpy(ctx->d_textures, h, sizeof(h), cudaMemcpyHostToDevice));
    return 0;
}
}  // namespace

int dprt_set_texture(dprt_ctx* ctx, int ti, const float* rgba, int width, int height) {
    if (!ctx || ti < 0 || ti >= DPRT_MAX_TEXTURES) return DPRT_ERR_INVALID;
    if (rgba && (width < 1 || height < 1 || (int64_t)width * height > ((int64_t)1 << 28))) return fail(ctx, DPRT_ERR_INVALID, "texture size");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));            // nothing in flight samples the old texels
    if (ctx->aux) CK(cudaStreamSynchronize(ctx->aux));
    std::shared_ptr<TexMem> m;
    if (rgba) { int r = upload_texels(ctx, rgba, width, height, m); if (r) return r; }
    ctx->tex[ti] = m;
    return upload_texture_table(ctx);
}

int dprt_set_material_textures(dprt_ctx* ctx, const int32_t* texture_index, int n) {
    if (!ctx || !texture_index || n < 1 || n > DPRT_MAX_MATERIALS) return DPRT_ERR_INVALID;
    for (int i = 0; i < n; i++)
        if (texture_index[i] < -1 || texture_index[i] >= DPRT_MAX_TEXTURES) return fail(ctx, DPRT_ERR_INVALID, "texture index out of range");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->aux) CK(cudaStreamSynchronize(ctx->aux));
    CK(cudaMemcpy(ctx->d_matTex, texture_index, sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    return 0;
}

int dprt_set_env_map(dprt_ctx* ctx, const float* rgba, int width, int height, float rotation_offset) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (rgba && (width < 1 || height < 1 || (int64_t)width * height > ((int64_t)1 << 28))) return fail(ctx, DPRT_ERR_INVALID, "environment map size");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->aux) CK(cudaStreamSynchronize(ctx->aux));
    std::shared_ptr<TexMem> m;
    if (rgba) { int r = upload_texels(ctx, rgba, width, height, m); if (r) return r; }
    ctx->envTex = m;
    ctx->hp.envMap = m ? DevTexture{(const float4*)m->d, m->w, m->h} : DevTexture{nullptr, 0, 0};
    ctx->hp.envRotation = rotation_offset;
    return 0;
}

// the same two look-ups on host arrays, from the source the kernels compile (dprt_math.cuh); no device involved
int dprt_spec_texture_sample(const float* rgba, int width, int height, const float* u, const float* v, int64_t n, int clamp_v, float* out4) {
    return spec_texture_sample(rgba, width, height, u, v, n, clamp_v, out4);
}
int dprt_spec_env_lookup(const float* rgba, int width, int height, float rotation_offset, const float* dirs3, int64_t n, float* out3) {
    return spec_env_lookup(rgba, width, height, rotation_offset, dirs3, n, out3);
}

int dprt_upload_proxy(dprt_ctx* ctx, int si, const dprt_object_desc* desc, const void* vis_blob, size_t vis_bytes,
                      const void* depth_blob, size_t depth_bytes) {
    if (!ctx || !desc || si < 0 || si >= ctx->cfg.sceneSize) return DPRT_ERR_INVALID;
    if (desc->nodeID < 0 || desc->nodeID >= ctx->world) return fail(ctx, DPRT_ERR_INVALID, "nodeID out of range");
    CK(cudaSetDevice(ctx->device));
    ObjectHost& o = ctx->objects[si];
    CK(cudaStreamSynchronize(ctx->stream));            // a launch in flight may still read the old networks / table rows
    o.release();
    auto mem = std::make_shared<ObjMem>();
    mem->device = ctx->device;
    o.desc = *desc; o.desc.isProxy = 1; o.present = true;
    if (vis_blob && mlp_create(vis_blob, vis_bytes, ctx->cfg.mlpDtype, &mem->vis, ctx->err)) return DPRT_ERR_INVALID;
    if (depth_blob && mlp_create(depth_blob, depth_bytes, ctx->cfg.mlpDtype, &mem->depth, ctx->err)) return DPRT_ERR_INVALID;
    o.mem = mem; o.vis = mem->vis; o.depth = mem->depth;
    const MlpGroupEntry ev = mlp_group_entry(o.vis), ed = mlp_group_entry(o.depth);
    CK(cudaMemcpy(ctx->d_mlpTable + si, &ev, sizeof(ev), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->d_mlpTable + 32 + si, &ed, sizeof(ed), cudaMemcpyHostToDevice));
    return upload_objects(ctx);
}

int dprt_adopt_scene(dprt_ctx* ctx, dprt_ctx* from) {
    if (!ctx || !from || ctx == from) return DPRT_ERR_INVALID;
    if (ctx->device != from->device || ctx->rank != from->rank || ctx->world != from->world || ctx->cfg.sceneSize != from->cfg.sceneSize ||
        ctx->cfg.mlpDtype != from->cfg.mlpDtype)
        return fail(ctx, DPRT_ERR_INVALID, "dprt_adopt_scene: the two contexts must be the same rank, device, scene size and proxy operand type");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream)); CK(cudaStreamSynchronize(from->stream));
    for (int i = 0; i < ctx->cfg.sceneSize; i++) ctx->objects[i] = from->objects[i];      // shares the device memory (ObjMem)
    CK(cudaMemcpy(ctx->d_materials, from->d_materials, sizeof(dprt_material) * DPRT_MAX_MATERIALS, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(ctx->d_lights, from->d_lights, sizeof(dprt_light_tri) * DPRT_MAX_LIGHTS, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(ctx->d_mlpTable, from->d_mlpTable, 2 * 32 * sizeof(MlpGroupEntry), cudaMemcpyDeviceToDevice));
    for (int i = 0; i < DPRT_MAX_TEXTURES; i++) ctx->tex[i] = from->tex[i];                 // shares the texels (TexMem)
    CK(cudaMemcpy(ctx->d_textures, from->d_textures, sizeof(DevTexture) * DPRT_MAX_TEXTURES, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(ctx->d_matTex, from->d_matTex, sizeof(int32_t) * DPRT_MAX_MATERIALS, cudaMemcpyDeviceToDevice));
    ctx->envTex = from->envTex; ctx->hp.envMap = from->hp.envMap; ctx->hp.envRotation = from->hp.envRotation;
    ctx->hp.lightCount = from->hp.lightCount;
    if (from->hp.camera.width == ctx->cfg.width && from->hp.camera.height == ctx->cfg.height) ctx->hp.camera = from->hp.camera;
    return upload_objects(ctx);
}

int dprt_accumulate_from(dprt_ctx* ctx, dprt_ctx* other) {
    if (!ctx || !other || ctx == other) return DPRT_ERR_INVALID;
    if (ctx->device != other->device || ctx->N != other->N) return fail(ctx, DPRT_ERR_INVALID, "dprt_accumulate_from: same device and frame size required");
    if (!ctx->d_aov != !other->d_aov) return fail(ctx, DPRT_ERR_STATE, "dprt_accumulate_from: AOVs are enabled on only one of the two contexts");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(other->stream));              // other's samples are complete
    launch_accumulate(ctx->hp.direct, ctx->hp.env, other->hp.direct, other->hp.env, ctx->N * 3, ctx->stream);
    ctx->stats.kernel_launches += 1;
    if (ctx->d_aov) {                                      // the albedo and normal planes, as one pair of planes
        launch_accumulate(ctx->d_aov, ctx->d_aov + 3 * (size_t)ctx->N, other->d_aov, other->d_aov + 3 * (size_t)ctx->N, ctx->N * 3, ctx->stream);
        ctx->stats.kernel_launches += 1;
    }
    CK(cudaGetLastError());
    return 0;
}

int dprt_set_materials(dprt_ctx* ctx, const dprt_material* mats, int n) {
    if (!ctx || !mats || n < 1 || n > DPRT_MAX_MATERIALS) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(ctx->d_materials, mats, sizeof(dprt_material) * n, cudaMemcpyHostToDevice));
    return 0;
}
int dprt_set_lights(dprt_ctx* ctx, const dprt_light_tri* lights, int n) {
    if (!ctx || !lights || n < 1 || n > DPRT_MAX_LIGHTS) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(ctx->d_lights, lights, sizeof(dprt_light_tri) * n, cudaMemcpyHostToDevice));
    ctx->hp.lightCount = n;
    return 0;
}
int dprt_set_camera(dprt_ctx* ctx, const dprt_camera* cam) {
    if (!ctx || !cam) return DPRT_ERR_INVALID;
    if (cam->width != ctx->cfg.width || cam->height != ctx->cfg.height) return fail(ctx, DPRT_ERR_INVALID, "camera resolution != config");
    ctx->hp.camera = *cam;
    return 0;
}

// ---- stages ------------------------------------------------------------------------------------
int dprt_reset_frame(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->hp.direct, 0, ctx->buf_bytes[DPRT_BUF_DIRECT], ctx->stream));
    CK(cudaMemsetAsync(ctx->hp.env, 0, ctx->buf_bytes[DPRT_BUF_ENV], ctx->stream));
    if (ctx->buf_ptr[DPRT_BUF_AOV]) CK(cudaMemsetAsync(ctx->buf_ptr[DPRT_BUF_AOV], 0, ctx->buf_bytes[DPRT_BUF_AOV], ctx->stream));
    // contribution / occlusion are only ever written by the proxy epilogues (and by dprt_upload, which raises nnScratchDirty):
    // with proxies off they are still the zeros of the allocation -- 1.6 GB of memset per frame at 5424x3056 not issued
    if (ctx->cfg.proxyMode || ctx->nnScratchDirty) {
        CK(cudaMemsetAsync(ctx->hp.contribution, 0, ctx->buf_bytes[DPRT_BUF_CONTRIBUTION], ctx->stream));
        CK(cudaMemsetAsync(ctx->hp.occlusion, 0, ctx->buf_bytes[DPRT_BUF_OCCLUSION], ctx->stream));
    }
    ctx->dirtyIdx = -1; ctx->nnScratchDirty = false; ctx->secDirty = 0;
    return 0;
}

int dprt_begin_sample(dprt_ctx* ctx, int sample) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    ctx->sample = sample;
    ctx->epoch++;
    ctx->aovPending = true;
    // resetSampleBuffers: offsets to zero. Path buffers are reset by count (slots >= pathSize are never read).
    CK(cudaMemsetAsync(ctx->hp.transferOffset, 0, 64 * sizeof(int32_t), ctx->stream));
    CK(cudaMemsetAsync(ctx->hp.sceneOffset, 0, 64 * sizeof(int32_t), ctx->stream));
    const int N = ctx->N, W = ctx->world;
    if (ctx->cfg.pathGenMode == 1) ctx->pathSize = (N - ctx->rank + W - 1) / W;
    else ctx->pathSize = ctx->rank == 0 ? N : 0;      // renderer.cpp:1514: only rank 0 generates camera paths
    ctx->shadowPathSize = 0;
    ctx->histFresh = false; ctx->qhistFresh = false;
    sync_params(ctx);
    return 0;
}

int dprt_path_gen(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    ctx->epoch++;
    sync_params(ctx);
    StageScope sc_(ctx, DPRT_STAGE_PATH_GEN, ctx->pathSize > 0);
    launch_path_gen(ctx->hp, ctx->pathSize, ctx->stream);
    ctx->stats.kernel_launches += ctx->pathSize > 0;
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

int dprt_traverse(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    CK(cudaMemsetAsync(ctx->hp.pathHist, 0, 32 * sizeof(int32_t), ctx->stream));
    StageScope sc_(ctx, DPRT_STAGE_TRAVERSE, ctx->pathSize > 0);
    launch_traverse(ctx->hp, ctx->pathSize, ctx->stream);
    ctx->stats.kernel_launches += 2 * (ctx->pathSize > 0);                  // trace + post
    ctx->stats.rays_traverse += ctx->pathSize;
    ctx->histFresh = true;
    CK(cudaGetLastError());
    return 0;
}

int dprt_partition(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    StageScope sc_(ctx, DPRT_STAGE_PARTITION);
    if (!ctx->histFresh) {
        launch_path_histogram(ctx->hp.paths, ctx->pathSize, ctx->world, ctx->hp.pathHist, ctx->stream);
        ctx->stats.kernel_launches += ctx->pathSize > 0;
    }
    launch_partition_paths(ctx->hp.paths, ctx->pathSize, ctx->world, ctx->world, ctx->rank, 0x7fffffff, ctx->hp.pathHist, ctx->hp.transfer,
                           ctx->hp.transferOffset, ctx->scratch, ctx->stream);
    ctx->stats.kernel_launches += 1;
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

int dprt_plan_exchange(const int32_t* M, int W, int me, int32_t* send_count, int32_t* recv_offset, int32_t* recv_count,
                       int64_t* recv_total, int* all_local) {
    if (!M || W < 1 || W > DPRT_MAX_WORLD || me < 0 || me >= W) return DPRT_ERR_INVALID;
    int64_t offdiag = 0, roff = 0;
    for (int s = 0; s < W; s++) {
        if (M[s * (W + 1)] != 0) return DPRT_ERR_INVALID;
        for (int d = 0; d < W; d++) {
            const int64_t c = (int64_t)M[s * (W + 1) + d + 1] - M[s * (W + 1) + d];
            if (c < 0) return DPRT_ERR_INVALID;
            if (s != d) offdiag += c;
            if (s == me && send_count) send_count[d] = (int32_t)c;
            if (d == me) {
                if (recv_offset) recv_offset[s] = (int32_t)roff;
                if (recv_count) recv_count[s] = (int32_t)c;
                roff += c;
            }
        }
    }
    if (roff > 0x7fffffff) return DPRT_ERR_CAPACITY;
    if (recv_offset) recv_offset[W] = (int32_t)roff;
    if (recv_total) *recv_total = roff;
    if (all_local) *all_local = offdiag == 0;
    return 0;
}

int dprt_exchange(dprt_ctx* ctx, int* done) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int W = ctx->world, me = ctx->rank;
    const size_t R = sizeof(dprt_path_record);
    StageScope sc_(ctx, DPRT_STAGE_EXCHANGE);
    if (W == 1) {
        int r = read_offsets(ctx); if (r) return r;
        const int cnt = ctx->h_offsets[1];
        if (ctx->shortcut) ctx->recsInTransfer = true;     // dprt_shade reads the records where the partition left them
        else if (cnt > 0) CK(cudaMemcpyAsync(ctx->hp.paths, ctx->hp.transfer, cnt * R, cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->pathSize = cnt; ctx->stats.paths_partitioned += cnt;
        if (done) *done = 1;
        ctx->stats.exchange_iters++;
        return 0;
    }
    if (!ctx->comm) return fail(ctx, DPRT_ERR_STATE, "dprt_exchange on a multi-rank context without an NCCL communicator");
    // MPI_Alltoall(counts): every rank learns the whole W x (W+1) offset matrix in one all-gather
    NK(g_nccl.AllGather(ctx->hp.transferOffset, ctx->d_gather, W + 1, ncclInt32, ctx->comm, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->d_gather, sizeof(int32_t) * W * (W + 1), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t* M = ctx->h_pinned;     // M[s*(W+1)+d] = offset of rank s's segment for destination d
    ctx->h_offsets.assign(M + me * (W + 1), M + (me + 1) * (W + 1));
    ctx->stats.paths_partitioned += ctx->h_offsets[W];
    std::vector<int32_t> sendCnt(W), recvOff(W + 1, 0), recvCnt(W);
    int64_t recvTotal64 = 0; int allLocal = 0;
    if (dprt_plan_exchange(M, W, me, sendCnt.data(), recvOff.data(), recvCnt.data(), &recvTotal64, &allLocal))
        return fail(ctx, DPRT_ERR_INVALID, "inconsistent offset matrix in the exchange");
    const int recvTotal = (int)recvTotal64;
    const long offdiag = allLocal ? 0 : 1;
    if ((size_t)recvTotal > (size_t)ctx->N) return fail(ctx, DPRT_ERR_CAPACITY, "received more paths than the frame holds");
    if (ctx->auxPending && recvTotal > ctx->auxGuardBase) { int jr = join_aux(ctx); if (jr) return jr; }   // would land on shadow paths still in use
    // MPI_Alltoallv: grouped send/recv straight from the partitioned device buffer
    NK(g_nccl.GroupStart());
    for (int peer = 0; peer < W; peer++) {
        if (peer == me) continue;
        const int sc = sendCnt[peer];
        const int rc = recvCnt[peer];
        if (sc > 0) NK(g_nccl.Send(ctx->hp.transfer + ctx->h_offsets[peer], (size_t)sc * R, ncclUint8, peer, ctx->comm, ctx->stream));
        if (rc > 0) NK(g_nccl.Recv(ctx->hp.paths + recvOff[peer], (size_t)rc * R, ncclUint8, peer, ctx->comm, ctx->stream));
        ctx->stats.paths_sent_offrank += sc; ctx->stats.bytes_alltoall += (int64_t)sc * R;
    }
    NK(g_nccl.GroupEnd());
    const int selfc = ctx->h_offsets[me + 1] - ctx->h_offsets[me];
    if (selfc > 0)
        CK(cudaMemcpyAsync(ctx->hp.paths + recvOff[me], ctx->hp.transfer + ctx->h_offsets[me], (size_t)selfc * R,
                           cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->pathSize = recvTotal;
    if (done) *done = offdiag == 0;     // MPI_Allreduce(LAND) of "nothing crossed ranks" (renderer.cpp:1292-1298)
    ctx->stats.exchange_iters++;
    return 0;
}

int dprt_exchange_group(dprt_ctx** ctxs, int W, int* done) {
    if (!ctxs || W < 1) return DPRT_ERR_INVALID;
    const size_t R = sizeof(dprt_path_record);
    for (int s = 0; s < W; s++) {
        if (!ctxs[s] || ctxs[s]->world != W || ctxs[s]->rank != s) return DPRT_ERR_INVALID;
        dprt_ctx* ctx = ctxs[s];
        CK(cudaSetDevice(ctx->device));
        int r = read_offsets(ctx); if (r) return r;
        ctx->stats.paths_partitioned += ctx->h_offsets[W];
    }
    long offdiag = 0;
    for (int d = 0; d < W; d++) {
        dprt_ctx* ctx = ctxs[d];
        CK(cudaSetDevice(ctx->device));
        int roff = 0;
        for (int s = 0; s < W; s++) {
            const int c = ctxs[s]->h_offsets[d + 1] - ctxs[s]->h_offsets[d];
            if (s != d) { offdiag += c; ctxs[s]->stats.paths_sent_offrank += c; ctxs[s]->stats.bytes_alltoall += (int64_t)c * R; }
            if (roff + c > ctx->N) return fail(ctx, DPRT_ERR_CAPACITY, "received more paths than the frame holds");
            if (c > 0) {
                if (ctxs[s]->device == ctx->device)
                    CK(cudaMemcpyAsync(ctx->hp.paths + roff, ctxs[s]->hp.transfer + ctxs[s]->h_offsets[d], c * R,
                                       cudaMemcpyDeviceToDevice, ctx->stream));
                else
                    CK(cudaMemcpyPeerAsync(ctx->hp.paths + roff, ctx->device, ctxs[s]->hp.transfer + ctxs[s]->h_offsets[d],
                                           ctxs[s]->device, c * R, ctx->stream));
            }
            roff += c;
        }
        CK(cudaStreamSynchronize(ctx->stream));   // sources may be re-partitioned next iteration
        ctx->pathSize = roff;
        ctx->stats.exchange_iters++;
    }
    if (done) *done = offdiag == 0;
    return 0;
}

int dprt_shade(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (ctx->hp.lightCount < 1) return fail(ctx, DPRT_ERR_STATE, "no lights set");
    ctx->shadowPathSize = ctx->cfg.shadowPathCount * ctx->pathSize;     // renderer.cpp:1328
    const int w = ctx->dirtyIdx == 0 ? 1 : 0;                           // the list that does not describe dirty planes
    ctx->hp.livePixel = ctx->d_live[w]; ctx->liveCount[w] = ctx->pathSize; ctx->shadeIdx = w;
    sync_params(ctx);
    StageScope sc_(ctx, DPRT_STAGE_SHADE, ctx->pathSize > 0);
    const bool cached = ctx->recsInTransfer;
    ctx->recsInTransfer = false;
    float* aov = ctx->aovPending ? ctx->d_aov : nullptr;     // the sample's first shade: the camera paths' first hits
    ctx->aovPending = false;
    if (cached) launch_shade_cached(ctx->hp, ctx->pathSize, aov, ctx->stream);
    else launch_shade(ctx->hp, ctx->pathSize, aov, ctx->stream);
    ctx->stats.kernel_launches += (cached ? 1 : 2) * (ctx->pathSize > 0);   // [trace +] post
    ctx->stats.rays_shade += ctx->pathSize;
    ctx->epoch++;                       // the records now hold the next bounce's rays: cached hits are stale
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

int dprt_reset_nn(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    // resetNNBuffers (renderer.cpp:367-414), by count instead of by capacity. Query/feature/prediction buffers are
    // reset inside the producing kernels. occlusion / contribution are only ever written by the proxy epilogues.
    // The shadow planes 1..spc-1 of directLightingBuffer are only written by the ShadowRay program, for pixels of the
    // paths the preceding MainRay shaded: those pixels are zeroed, the rest of the planes is zero already.
    const bool nnAll = ctx->nnScratchDirty || (ctx->cfg.proxyMode && ctx->dirtyIdx == -2);   // contents unknown: clear everything
    if (nnAll) {
        CK(cudaMemsetAsync(ctx->hp.occlusion, 0, ctx->buf_bytes[DPRT_BUF_OCCLUSION], ctx->stream));
        CK(cudaMemsetAsync(ctx->hp.contribution, 0, ctx->buf_bytes[DPRT_BUF_CONTRIBUTION], ctx->stream));
        ctx->nnScratchDirty = false;
    } else if (ctx->cfg.proxyMode && ctx->secDirty > 0) {
        sync_params(ctx);
        launch_reset_sec(ctx->hp, ctx->d_secLive, ctx->secDirty, ctx->stream);     // what Target_Node_Update left behind
        ctx->stats.kernel_launches += 1;
    }
    ctx->secDirty = 0;
    if (ctx->dirtyIdx == -2) {
        if (ctx->cfg.shadowPathCount > 1)
            CK(cudaMemsetAsync(ctx->hp.direct + (size_t)ctx->N * 3, 0, (size_t)ctx->N * 3 * sizeof(float) * (ctx->cfg.shadowPathCount - 1),
                               ctx->stream));
    } else if (ctx->dirtyIdx >= 0) {
        sync_params(ctx);
        launch_reset_planes(ctx->hp, ctx->d_live[ctx->dirtyIdx], ctx->liveCount[ctx->dirtyIdx], ctx->cfg.proxyMode && !nnAll, ctx->stream);
        ctx->stats.kernel_launches += ctx->liveCount[ctx->dirtyIdx] > 0;
    }
    ctx->dirtyIdx = -1;
    CK(cudaMemsetAsync(ctx->hp.queryHist, 0, 64 * sizeof(int32_t), ctx->stream));
    ctx->qhistFresh = false;
    return 0;
}

int dprt_shadow_trace(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    CK(cudaMemsetAsync(ctx->hp.queryHist, 0, 64 * sizeof(int32_t), ctx->stream));
    StageScope sc_(ctx, DPRT_STAGE_SHADOW_TRACE, ctx->shadowPathSize > 0);
    launch_shadow_trace(ctx->hp, ctx->shadowPathSize, ctx->stream);
    ctx->stats.kernel_launches += (ctx->hp.proxyMode ? 2 : 1) * (ctx->shadowPathSize > 0);   // trace [+ post with proxies]
    ctx->stats.rays_shadow += ctx->shadowPathSize;
    // planes now hold this bounce's terms: covered by the MainRay list if nothing else was dirty, else unknown
    if (ctx->shadowPathSize > 0)
        ctx->dirtyIdx = (ctx->shadeIdx >= 0 && (ctx->dirtyIdx == -1 || ctx->dirtyIdx == ctx->shadeIdx)) ? ctx->shadeIdx : -2;
    ctx->qhistFresh = true; ctx->queryWhich = 0;
    CK(cudaGetLastError());
    return 0;
}

int dprt_secondary_trace(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->cfg.proxyMode) return fail(ctx, DPRT_ERR_STATE, "secondary stage needs proxyMode=1");
    sync_params(ctx);
    CK(cudaMemsetAsync(ctx->hp.queryHist, 0, 64 * sizeof(int32_t), ctx->stream));
    StageScope sc_(ctx, DPRT_STAGE_SECONDARY_TRACE, ctx->pathSize > 0);
    launch_secondary_trace(ctx->hp, ctx->pathSize, ctx->stream);
    ctx->stats.kernel_launches += 2 * (ctx->pathSize > 0);                  // trace + post
    ctx->stats.rays_secondary += ctx->pathSize;
    ctx->qhistFresh = true; ctx->queryWhich = 1;
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

int dprt_bucket_queries(dprt_ctx* ctx, int which, int inside_only, int* total) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->cfg.proxyMode) return fail(ctx, DPRT_ERR_STATE, "query bucketing needs proxyMode=1");
    sync_params(ctx);
    const int S = ctx->cfg.sceneSize;
    const int n = ctx->cfg.maxCount * (which == 0 ? ctx->shadowPathSize : ctx->pathSize);
    int32_t* hist = ctx->hp.queryHist + (inside_only ? S : 0);
    StageScope sc_(ctx, DPRT_STAGE_BUCKET);
    if (!ctx->qhistFresh || ctx->queryWhich != which) {
        hist = ctx->d_hist + 96;
        launch_query_histogram(ctx->hp.nnQuery, n, S, inside_only ? 1 : 0, hist, ctx->stream);
        ctx->stats.kernel_launches += n > 0;
    }
    const bool keysFresh = ctx->qhistFresh && ctx->queryWhich == which;      // same launch wrote records, histogram and keys
    launch_partition_queries(ctx->hp.nnQuery, keysFresh ? ctx->hp.nnKey : nullptr, ctx->hp.nnInput, n, S, inside_only ? 1 : 0, hist, ctx->hp.nnPackedQuery,
                             ctx->hp.nnPackedInput, ctx->hp.sceneOffset, ctx->scratch, ctx->stream);
    ctx->stats.kernel_launches += 1;
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->hp.sceneOffset, (S + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));      // renderer.cpp:781-787: sceneOffset is read back before the forward loop
    ctx->h_sceneOffset.assign(ctx->h_pinned, ctx->h_pinned + S + 1);
    ctx->queryTotal = ctx->h_sceneOffset[S];
    if (total) *total = ctx->queryTotal;
    CK(cudaGetLastError());
    return 0;
}

int dprt_proxy_infer(dprt_ctx* ctx, int kind, int pred_offset) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int S = ctx->cfg.sceneSize;
    if (pred_offset < 0 || (size_t)(pred_offset + ctx->queryTotal) * sizeof(dprt_half) > ctx->buf_bytes[DPRT_BUF_PRED])
        return fail(ctx, DPRT_ERR_CAPACITY, "prediction range outside predBuffer");
    StageScope sc_(ctx, DPRT_STAGE_PROXY_MLP, ctx->queryTotal > 0);
    if (ctx->queryTotal > 0)
        CK(cudaMemsetAsync(ctx->hp.pred + pred_offset, 0, (size_t)ctx->queryTotal * sizeof(dprt_half), ctx->stream));
    // ONE launch for every proxy (the per-object forward loops of renderer.cpp:879-969, 1040-1120): object i owns rows
    // [sceneOffset[i], sceneOffset[i+1]) of the packed queries; the kernel reads the offsets and the model table on the device
    int64_t pairs = 0, rows = 0;
    for (int i = 0; i < S; i++) {
        const int cnt = ctx->h_sceneOffset[i + 1] - ctx->h_sceneOffset[i];
        const MlpModel* m = kind == 0 ? ctx->objects[i].vis : ctx->objects[i].depth;
        if (cnt <= 0 || !m) continue;                        // "padding" model slot (renderer.cpp:791): predictions stay 0
        pairs += ((cnt + 127) / 128 + 1) / 2; rows += cnt;
    }
    if (pairs > 0) {
        if (mlp_forward_group(ctx->d_mlpTable + (kind ? 32 : 0), ctx->hp.sceneOffset, S, pairs, ctx->cfg.mlpDtype, ctx->hp.nnPackedInput,
                              ctx->hp.pred + pred_offset, ctx->stream, ctx->err)) return DPRT_ERR_CUDA;
        ctx->stats.kernel_launches += 1;
        ctx->stats.nn_queries += rows;
    }
    CK(cudaGetLastError());
    return 0;
}

int dprt_frame_buffer_update(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    StageScope sc_(ctx, DPRT_STAGE_FRAME_UPDATE);
    launch_shadow_occlusion(ctx->hp, ctx->cfg.proxyMode ? ctx->queryTotal : 0, ctx->stream);
    const bool sparse = ctx->dirtyIdx >= 0 && ctx->dirtyIdx == ctx->shadeIdx;     // else: every pixel (reference behaviour)
    if (!sparse && ctx->cfg.proxyMode && ctx->queryTotal > 0) ctx->nnScratchDirty = true;   // entries outside any pixel list
    if (ctx->dirtyIdx != -1)
        launch_contribution(ctx->hp, sparse ? ctx->d_live[ctx->dirtyIdx] : nullptr, sparse ? ctx->liveCount[ctx->dirtyIdx] : 0, ctx->stream);
    ctx->stats.kernel_launches += (ctx->dirtyIdx != -1) + (ctx->queryTotal > 0);
    CK(cudaGetLastError());
    return 0;
}
int dprt_depth_buffer_update(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    StageScope sc_(ctx, DPRT_STAGE_DEPTH_UPDATE, ctx->queryTotal > 0);
    launch_depth_update(ctx->hp, ctx->queryTotal, ctx->stream);
    ctx->stats.kernel_launches += ctx->queryTotal > 0;
    ctx->qhistFresh = ctx->qhistFresh;   // normalizedT changes, keys do not
    CK(cudaGetLastError());
    return 0;
}
int dprt_target_node_update(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    StageScope sc_(ctx, DPRT_STAGE_TARGET_UPDATE);
    ctx->hp.secLive = ctx->d_secLive;
    launch_tmax(ctx->hp, ctx->queryTotal, ctx->stream);
    launch_target_node(ctx->hp, ctx->pathSize, ctx->stream);
    if (ctx->secDirty > 0 || !ctx->d_secLive) ctx->nnScratchDirty = true;       // two updates without a reset in between: unknown
    else ctx->secDirty = ctx->pathSize;
    ctx->stats.kernel_launches += (ctx->queryTotal > 0) + (ctx->pathSize > 0);
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

// ---- settled deque: the migrate loop without the riders ---------------------------------------------
// In the reference every iteration of primaryRayModule runs TraRay, Work_Efficient_Scan and MPI_Alltoallv over ALL paths
// of the rank, although a path that has reached the rank of its closest hit (targetNode == rank, own bit visited) comes
// out of each of those steps unchanged. The buffer of rank r after an iteration is  L ++ M ++ R : records received from
// lower ranks, the rank's own segment, records received from higher ranks; the own segment of the NEXT iteration is
// stay(L) ++ M ++ stay(R), because the partition is stable and nothing in M moves or dies. So M is kept in the middle of
// a 2N-record buffer and grows at both ends, and only L ++ R (what arrived in the last exchange) is traced, partitioned
// (W + 1 buckets: the self bucket in its two pieces) and sent on. When the loop ends the active set is empty and M is
// the rank's path buffer, record for record what the reference would hold.
namespace {

bool deque_enabled(const dprt_ctx* ctx) { return ctx->d_settled && !ctx->hp.hitPrim; }

bool deque_p2p(const dprt_ctx* ctx) { return ctx->p2p && (ctx->p2pGroup ? ctx->p2pGroupActive : true); }

int deque_begin(dprt_ctx* ctx) {
    ctx->front = ctx->back = ctx->N; ctx->nL = 0;
    if (deque_p2p(ctx)) {          // inside the loop the counts kernel leaves the histogram zeroed for the next TraRay launch
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemsetAsync(ctx->hp.pathHist, 0, 32 * sizeof(int32_t), ctx->stream));
    }
    return 0;
}

int deque_traverse(dprt_ctx* ctx) {
    CK(cudaSetDevice(ctx->device));
    sync_params(ctx);
    ctx->hp.splitL = ctx->nL;
    if (!deque_p2p(ctx)) CK(cudaMemsetAsync(ctx->hp.pathHist, 0, 32 * sizeof(int32_t), ctx->stream));   // W + 1 <= 32 buckets
    {
        StageScope sc_(ctx, DPRT_STAGE_TRAVERSE, ctx->pathSize > 0);
        launch_traverse(ctx->hp, ctx->pathSize, ctx->stream);
    }
    ctx->hp.splitL = 0x7fffffff;
    ctx->stats.kernel_launches += 2 * (ctx->pathSize > 0);                  // trace + post
    ctx->stats.rays_traverse += ctx->pathSize + (ctx->back - ctx->front);          // the reference launches over the riders too
    CK(cudaGetLastError());
    return 0;
}

int deque_partition(dprt_ctx* ctx) {
    StageScope sc_(ctx, DPRT_STAGE_PARTITION);
    launch_partition_paths(ctx->hp.paths, ctx->pathSize, ctx->world, ctx->world + 1, ctx->rank, ctx->nL, ctx->hp.pathHist,
                           ctx->hp.transfer, ctx->hp.transferOffset, ctx->scratch, ctx->stream);
    ctx->stats.kernel_launches += 1;
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

// rows: W rows of W + 2 offsets (row s = transferOffset of rank s: buckets 0..W-1 by destination, bucket W = second self piece)
struct DequePlan {
    std::vector<int> sendCnt, recvCnt;
    std::vector<int> dstOffset;      // where this rank's bucket d starts among the arrivals of rank d (source-rank order)
    int cL = 0, cR = 0, offL = 0, offR = 0, newNL = 0, newActive = 0; bool allLocal = true;
};
int deque_plan(const int32_t* rows, int W, int me, DequePlan& p) {
    p.sendCnt.assign(W, 0); p.recvCnt.assign(W, 0); p.dstOffset.assign(W, 0);
    for (int s = 0; s < W; s++) {
        const int32_t* r = rows + (size_t)s * (W + 2);
        if (r[0] != 0) return DPRT_ERR_INVALID;
        for (int d = 0; d <= W; d++) if (r[d + 1] < r[d]) return DPRT_ERR_INVALID;
        for (int d = 0; d < W; d++) {
            const int c = r[d + 1] - r[d];
            if (s != d && c > 0) p.allLocal = false;
            if (s == me && d != me) p.sendCnt[d] = c;
            if (d == me && s != me) { p.recvCnt[s] = c; p.newActive += c; if (s < me) p.newNL += c; }
            if (s < me && s != d) p.dstOffset[d] += c;               // lower ranks' records precede mine at every destination
        }
        if (s == me) { p.offL = r[me]; p.cL = r[me + 1] - r[me]; p.offR = r[W]; p.cR = r[W + 1] - r[W]; }
    }
    return 0;
}

// moves the two pieces of the self segment from the transfer buffer to the ends of the settled block
int deque_absorb(dprt_ctx* ctx, const DequePlan& p) {
    const size_t R = sizeof(dprt_path_record);
    if (ctx->front - p.cL < 0 || ctx->back + p.cR > 2 * ctx->N || (ctx->back - ctx->front) + p.cL + p.cR > ctx->N)
        return fail(ctx, DPRT_ERR_CAPACITY, "more settled paths than the frame holds");
    if (p.cL > 0) CK(cudaMemcpyAsync(ctx->d_settled + ctx->front - p.cL, ctx->hp.transfer + p.offL, p.cL * R, cudaMemcpyDeviceToDevice, ctx->stream));
    if (p.cR > 0) CK(cudaMemcpyAsync(ctx->d_settled + ctx->back, ctx->hp.transfer + p.offR, p.cR * R, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->front -= p.cL; ctx->back += p.cR;
    return 0;
}

int deque_exchange(dprt_ctx* ctx, int* done) {
    CK(cudaSetDevice(ctx->device));
    const int W = ctx->world, me = ctx->rank;
    const size_t R = sizeof(dprt_path_record);
    StageScope sc_(ctx, DPRT_STAGE_EXCHANGE);
    if (!ctx->comm) return fail(ctx, DPRT_ERR_STATE, "dprt_exchange on a multi-rank context without an NCCL communicator");
    NK(g_nccl.AllGather(ctx->hp.transferOffset, ctx->d_gather, W + 2, ncclInt32, ctx->comm, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->d_gather, sizeof(int32_t) * W * (W + 2), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    DequePlan p;
    if (deque_plan(ctx->h_pinned, W, me, p)) return fail(ctx, DPRT_ERR_INVALID, "inconsistent offset matrix in the exchange");
    if (p.newActive > ctx->N) return fail(ctx, DPRT_ERR_CAPACITY, "received more paths than the frame holds");
    if (ctx->auxPending && p.newActive > ctx->auxGuardBase) { int jr = join_aux(ctx); if (jr) return jr; }
    const int32_t* row = ctx->h_pinned + (size_t)me * (W + 2);
    ctx->stats.paths_partitioned += row[W + 1];
    NK(g_nccl.GroupStart());
    int roff = 0;
    for (int peer = 0; peer < W; peer++) {
        if (peer == me) continue;
        const int sc = p.sendCnt[peer], rc = p.recvCnt[peer];
        if (sc > 0) NK(g_nccl.Send(ctx->hp.transfer + row[peer], (size_t)sc * R, ncclUint8, peer, ctx->comm, ctx->stream));
        if (rc > 0) NK(g_nccl.Recv(ctx->hp.paths + roff, (size_t)rc * R, ncclUint8, peer, ctx->comm, ctx->stream));
        roff += rc;
        ctx->stats.paths_sent_offrank += sc; ctx->stats.bytes_alltoall += (int64_t)sc * R;
    }
    NK(g_nccl.GroupEnd());
    int r = deque_absorb(ctx, p); if (r) return r;
    ctx->pathSize = p.newActive; ctx->nL = p.newNL;
    if (done) *done = p.allLocal;
    ctx->stats.exchange_iters++;
    return 0;
}

int deque_exchange_group(dprt_ctx** ctxs, int W, int* done) {
    const size_t R = sizeof(dprt_path_record);
    std::vector<int32_t> rows((size_t)W * (W + 2));
    for (int s = 0; s < W; s++) {
        dprt_ctx* ctx = ctxs[s];
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpyAsync(ctx->h_pinned, ctx->hp.transferOffset, (W + 2) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        std::copy(ctx->h_pinned, ctx->h_pinned + W + 2, rows.begin() + (size_t)s * (W + 2));
        ctx->stats.paths_partitioned += ctx->h_pinned[W + 1];
    }
    bool allLocal = true;
    for (int d = 0; d < W; d++) {
        dprt_ctx* ctx = ctxs[d];
        CK(cudaSetDevice(ctx->device));
        DequePlan p;
        if (deque_plan(rows.data(), W, d, p)) return fail(ctx, DPRT_ERR_INVALID, "inconsistent offset matrix in the exchange");
        if (p.newActive > ctx->N) return fail(ctx, DPRT_ERR_CAPACITY, "received more paths than the frame holds");
        allLocal = allLocal && p.allLocal;
        int roff = 0;
        for (int s = 0; s < W; s++) {
            if (s == d) continue;
            const int c = p.recvCnt[s];
            const int32_t* srow = rows.data() + (size_t)s * (W + 2);
            ctxs[s]->stats.paths_sent_offrank += c; ctxs[s]->stats.bytes_alltoall += (int64_t)c * R;
            if (c > 0) {
                if (ctxs[s]->device == ctx->device)
                    CK(cudaMemcpyAsync(ctx->hp.paths + roff, ctxs[s]->hp.transfer + srow[d], c * R, cudaMemcpyDeviceToDevice, ctx->stream));
                else
                    CK(cudaMemcpyPeerAsync(ctx->hp.paths + roff, ctx->device, ctxs[s]->hp.transfer + srow[d], ctxs[s]->device, c * R, ctx->stream));
            }
            roff += c;
        }
        int r = deque_absorb(ctx, p); if (r) return r;
        CK(cudaStreamSynchronize(ctx->stream));   // sources are re-partitioned next iteration
        ctx->pathSize = p.newActive; ctx->nL = p.newNL;
        ctx->stats.exchange_iters++;
    }
    if (done) *done = allLocal;
    return 0;
}

// the active set is empty: the settled block is the path buffer
int deque_finish(dprt_ctx* ctx) {
    CK(cudaSetDevice(ctx->device));
    ctx->hp.paths = (dprt_path_record*)ctx->buf_ptr[DPRT_BUF_PATHS];      // the peer-memory exchange reads arrivals from its own buffers
    const int n = ctx->back - ctx->front;
    if (ctx->auxPending && n > ctx->auxGuardBase) { int jr = join_aux(ctx); if (jr) return jr; }
    StageScope sc_(ctx, DPRT_STAGE_EXCHANGE);
    if (n > 0) CK(cudaMemcpyAsync(ctx->hp.paths, ctx->d_settled + ctx->front, (size_t)n * sizeof(dprt_path_record), cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->pathSize = n; ctx->nL = 0;
    return 0;
}

}  // namespace

int dprt_plan_exchange_deque(const int32_t* rows, int W, int me, int32_t* send_count, int32_t* recv_count, int32_t* dst_offset,
                             int32_t* piece, int32_t* new_nl, int32_t* new_active, int* all_local) {
    if (!rows || W < 1 || W >= DPRT_MAX_WORLD || me < 0 || me >= W) return DPRT_ERR_INVALID;
    DequePlan p;
    if (deque_plan(rows, W, me, p)) return DPRT_ERR_INVALID;
    for (int k = 0; k < W; k++) {
        if (send_count) send_count[k] = p.sendCnt[k];
        if (recv_count) recv_count[k] = p.recvCnt[k];
        if (dst_offset) dst_offset[k] = p.dstOffset[k];
    }
    if (piece) { piece[0] = p.offL; piece[1] = p.cL; piece[2] = p.offR; piece[3] = p.cR; }
    if (new_nl) *new_nl = p.newNL;
    if (new_active) *new_active = p.newActive;
    if (all_local) *all_local = p.allLocal ? 1 : 0;
    return 0;
}

// ---- the deque exchange over peer memory (p2p_exchange.cuh, DESIGN.md 3.4) ------------------------------------------
namespace {

bool p2p_requested() { const char* v = getenv("DPRT_P2P"); return !(v && v[0] == '0'); }     // default on; DPRT_P2P=0 forces NCCL

unsigned long long p2p_timeout_ns() {
    static unsigned long long v = [] { const char* e = getenv("DPRT_P2P_TIMEOUT_MS"); long ms = e ? atol(e) : 20000; return (unsigned long long)(ms < 1 ? 1 : ms) * 1000000ull; }();
    return v;
}

int p2p_alloc(dprt_ctx* ctx) {
    CK(cudaSetDevice(ctx->device));
    if (ctx->d_mailbox) return 0;
    CK(cudaMalloc(&ctx->d_mailbox, sizeof(P2PMailbox)));
    CK(cudaMemset(ctx->d_mailbox, 0, sizeof(P2PMailbox)));
    for (int k = 0; k < 2; k++) CK(cudaMalloc(&ctx->d_active[k], (size_t)ctx->N * sizeof(dprt_path_record)));
    CK(cudaMalloc(&ctx->d_peers, sizeof(P2PPeers)));
    CK(cudaMalloc(&ctx->d_plan, sizeof(P2PPlan)));
    CK(cudaMemset(ctx->d_plan, 0, sizeof(P2PPlan)));
    CK(cudaHostAlloc(&ctx->h_plan, sizeof(P2PHostPlan), cudaHostAllocMapped));
    std::memset(ctx->h_plan, 0, sizeof(P2PHostPlan));
    CK(cudaHostGetDevicePointer((void**)&ctx->d_hplan, ctx->h_plan, 0));
    // every kernel of the migrate loop is loaded NOW: with lazy module loading a first launch may synchronise the context,
    // which deadlocks when it happens beside another rank's waiting kernel (one thread driving several ranks)
    CK(p2p_preload_kernels()); CK(partition_preload_kernels()); CK(trace_preload_kernels());
    return 0;
}

void p2p_free(dprt_ctx* ctx) {
    for (void* q : ctx->ipcOpened) cudaIpcCloseMemHandle(q);
    ctx->ipcOpened.clear();
    if (ctx->d_mailbox) cudaFree(ctx->d_mailbox);
    for (int k = 0; k < 2; k++) if (ctx->d_active[k]) cudaFree(ctx->d_active[k]);
    if (ctx->d_peers) cudaFree(ctx->d_peers);
    if (ctx->d_plan) cudaFree(ctx->d_plan);
    if (ctx->h_plan) cudaFreeHost(ctx->h_plan);
    ctx->d_mailbox = nullptr; ctx->d_active[0] = ctx->d_active[1] = nullptr; ctx->d_peers = nullptr; ctx->d_plan = nullptr; ctx->h_plan = nullptr;
    ctx->p2p = false;
}

struct P2PHandles { cudaIpcMemHandle_t h[3]; int32_t ok; int32_t pad_[3]; };     // mailbox, active[0], active[1]
static_assert(sizeof(P2PHandles) == DPRT_P2P_HANDLE_BYTES, "dprt_p2p_export size");

bool p2p_eligible(const dprt_ctx* ctx) { return ctx->d_settled && ctx->world > 1 && ctx->world <= kP2PMaxWorld; }

// my three IPC handles (ok = 0 when this rank cannot take part: the peers then fall back together)
int p2p_export(dprt_ctx* ctx, P2PHandles* out) {
    std::memset(out, 0, sizeof(*out));
    if (!p2p_eligible(ctx) || !p2p_requested()) return 0;
    if (p2p_alloc(ctx)) return 0;
    if (cudaIpcGetMemHandle(&out->h[0], ctx->d_mailbox) != cudaSuccess || cudaIpcGetMemHandle(&out->h[1], ctx->d_active[0]) != cudaSuccess ||
        cudaIpcGetMemHandle(&out->h[2], ctx->d_active[1]) != cudaSuccess) { cudaGetLastError(); return 0; }
    out->ok = 1;
    return 0;
}

// opens every peer's handles; returns 1 when this rank now holds a complete pointer table (not yet enabled)
int p2p_open(dprt_ctx* ctx, const P2PHandles* all) {
    const int W = ctx->world, me = ctx->rank;
    for (int s = 0; s < W; s++) if (!all[s].ok) return 0;
    P2PPeers tbl; std::memset(&tbl, 0, sizeof(tbl));
    for (int s = 0; s < W; s++) {
        void* ptr[3] = {ctx->d_mailbox, ctx->d_active[0], ctx->d_active[1]};
        if (s != me)
            for (int k = 0; k < 3; k++) {
                if (cudaIpcOpenMemHandle(&ptr[k], all[s].h[k], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return 0; }
                ctx->ipcOpened.push_back(ptr[k]);
            }
        tbl.mailbox[s] = (P2PMailbox*)ptr[0]; tbl.active[s][0] = (dprt_path_record*)ptr[1]; tbl.active[s][1] = (dprt_path_record*)ptr[2];
    }
    if (cudaMemcpy(ctx->d_peers, &tbl, sizeof(tbl), cudaMemcpyHostToDevice) != cudaSuccess) { cudaGetLastError(); return 0; }
    return 1;
}

// one process per GPU: handles all-gathered over the communicator, then a second all-gather agrees on "every rank opened
// every handle" -- either all ranks use peer memory or all use the NCCL exchange (a split decision would deadlock)
int p2p_connect_nccl(dprt_ctx* ctx) {
    const int W = ctx->world;
    if (!ctx->comm || W > kP2PMaxWorld) return 0;
    P2PHandles mine;
    p2p_export(ctx, &mine);
    char* d_all = nullptr;
    CK(cudaMalloc(&d_all, sizeof(P2PHandles) * (size_t)(W + 1)));
    std::vector<P2PHandles> all(W);
    for (int round = 0; round < 2; round++) {
        CK(cudaMemcpyAsync(d_all + sizeof(P2PHandles) * W, &mine, sizeof(P2PHandles), cudaMemcpyHostToDevice, ctx->stream));
        NK(g_nccl.AllGather(d_all + sizeof(P2PHandles) * W, d_all, sizeof(P2PHandles), ncclUint8, ctx->comm, ctx->stream));
        CK(cudaMemcpyAsync(all.data(), d_all, sizeof(P2PHandles) * (size_t)W, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (round == 0) mine.ok = p2p_open(ctx, all.data());         // second round carries "opened everything"
    }
    CK(cudaFree(d_all));
    bool ok = true;
    for (int s = 0; s < W; s++) ok = ok && all[s].ok;
    if (ok) ctx->p2p = true; else p2p_free(ctx);
    return 0;
}

// in-process rank group: the other contexts' pointers are valid as they are (peer access enabled across devices)
int p2p_connect_group(dprt_ctx** ctxs, int W) {
    if (W > kP2PMaxWorld) return 0;
    for (int k = 0; k < W; k++) {
        if (!ctxs[k]->d_settled) return 0;
        int r = p2p_alloc(ctxs[k]); if (r) return r;
    }
    for (int k = 0; k < W; k++) {
        dprt_ctx* ctx = ctxs[k];
        CK(cudaSetDevice(ctx->device));
        P2PPeers tbl; std::memset(&tbl, 0, sizeof(tbl));
        for (int s = 0; s < W; s++) {
            if (ctxs[s]->device != ctx->device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[s]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(ctx, DPRT_ERR_CUDA, "no peer access between the group's devices");
                cudaGetLastError();
            }
            tbl.mailbox[s] = ctxs[s]->d_mailbox; tbl.active[s][0] = ctxs[s]->d_active[0]; tbl.active[s][1] = ctxs[s]->d_active[1];
        }
        CK(cudaMemcpy(ctx->d_peers, &tbl, sizeof(tbl), cudaMemcpyHostToDevice));
        ctx->p2p = true; ctx->p2pGroup = true;
    }
    return 0;
}

// after deque_traverse: counts -> partition (scattering straight into the owners' buffers) -> barrier, all on the rank's
// stream; nothing here waits on the host
int p2p_exchange_enqueue(dprt_ctx* ctx) {
    CK(cudaSetDevice(ctx->device));
    const int W = ctx->world, me = ctx->rank;
    const uint32_t seq = ++ctx->p2pSeq;
    const int parity = (int)((seq - 1u) & 1u);
    {
        StageScope sc_(ctx, DPRT_STAGE_EXCHANGE);
        P2PCountsArgs a;
        a.peers = ctx->d_peers; a.mine = ctx->d_mailbox; a.hist = ctx->hp.pathHist; a.W = W; a.me = me; a.parity = parity; a.seq = seq;
        a.settled = ctx->d_settled; a.front = ctx->front; a.back = ctx->back; a.capacity = ctx->N;
        a.plan = ctx->d_plan; a.hostPlan = ctx->d_hplan; a.timeoutNs = p2p_timeout_ns();
        launch_p2p_counts(a, ctx->stream);
    }
    {
        StageScope sc_(ctx, DPRT_STAGE_PARTITION, ctx->pathSize > 0);
        launch_partition_paths_peer(ctx->hp.paths, ctx->pathSize, W, me, ctx->nL, ctx->d_plan, ctx->scratch, ctx->stream);
    }
    {
        StageScope sc_(ctx, DPRT_STAGE_EXCHANGE);
        launch_p2p_barrier(ctx->d_peers, ctx->d_mailbox, ctx->d_plan, ctx->d_hplan, W, me, parity, seq, p2p_timeout_ns(), ctx->stream);
    }
    ctx->stats.kernel_launches += 2 + (ctx->pathSize > 0);
    ctx->histFresh = false;
    CK(cudaGetLastError());
    return 0;
}

// the host learns the plan from the mapped copy the counts kernel wrote (while partition and barrier are still running),
// extends the settled block by the two self pieces and switches to the buffer the arrivals are landing in
int p2p_exchange_finish(dprt_ctx* ctx, int* done) {
    CK(cudaSetDevice(ctx->device));
    const uint32_t seq = ctx->p2pSeq;
    const int parity = (int)((seq - 1u) & 1u);
    volatile P2PHostPlan* hp = ctx->h_plan;
    for (long spins = 0; hp->seq != seq; spins++) {
        if ((spins & 0x3f) == 0x3f) std::this_thread::yield();      // several contexts of a rank may be polling (samples in flight)
        if ((spins & 0xfff) == 0xfff) {
            cudaError_t e = cudaStreamQuery(ctx->stream);
            if (e != cudaSuccess && e != cudaErrorNotReady) return fail(ctx, DPRT_ERR_CUDA, std::string("peer-memory exchange: ") + cudaGetErrorString(e));
            if (e == cudaSuccess && hp->seq != seq) return fail(ctx, DPRT_ERR_STATE, "peer-memory exchange: the stream drained without a plan");
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    P2PHostPlan plan;
    std::memcpy(&plan, (const void*)ctx->h_plan, sizeof(plan));
    if (plan.error) {
        hp->abort = 1u;
        static const char* what[] = {"", "a peer did not arrive in time", "aborted by a peer", "more paths than a receive buffer or the settled block holds", "inconsistent histogram rows"};
        return fail(ctx, plan.error == P2P_ERR_CAPACITY ? DPRT_ERR_CAPACITY : DPRT_ERR_STATE,
                    std::string("peer-memory exchange: ") + what[plan.error >= 0 && plan.error <= 4 ? plan.error : 0]);
    }
    ctx->stats.paths_sent_offrank += plan.sent; ctx->stats.bytes_alltoall += (int64_t)plan.sent * (int64_t)sizeof(dprt_path_record);
    ctx->stats.paths_partitioned += plan.total;
    ctx->front -= plan.cL; ctx->back += plan.cR;
    ctx->pathSize = plan.newActive; ctx->nL = plan.newNL;
    ctx->hp.paths = ctx->d_active[parity ^ 1];             // restored by deque_finish
    if (done) *done = plan.allLocal;
    ctx->stats.exchange_iters++;
    return 0;
}

}  // namespace

// Peer-memory wiring for hosts that bring their own bootstrap (no NCCL communicator in the context): every rank exports
// DPRT_P2P_HANDLE_BYTES, the host all-gathers them by whatever means it has (MPI, a socket, torch.distributed), every rank
// connects. Collective: call on all ranks or on none. *enabled = 0 when any rank could not take part (the context then
// needs an NCCL communicator for dprt_primary_ray_module).
int dprt_p2p_export(dprt_ctx* ctx, void* handle_out) {
    if (!ctx || !handle_out) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    return p2p_export(ctx, (P2PHandles*)handle_out);
}
int dprt_p2p_connect(dprt_ctx* ctx, const void* all_handles, int* enabled) {
    if (!ctx || !all_handles) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int ok = ctx->d_mailbox ? p2p_open(ctx, (const P2PHandles*)all_handles) : 0;
    if (enabled) *enabled = ok;
    return 0;
}
// second half: the host has agreed (all-reduce of *enabled) on whether every rank connected
int dprt_p2p_enable(dprt_ctx* ctx, int enable) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (enable && ctx->d_mailbox) {
        if (ctx->device < 64 && g_streams[ctx->device] > max_connections()) {
            p2p_free(ctx);
            return fail(ctx, DPRT_ERR_STATE, "more CUDA streams on this device than hardware queues (CUDA_DEVICE_MAX_CONNECTIONS): set it to 32 before the first CUDA call");
        }
        ctx->p2p = true;
    } else p2p_free(ctx);
    return 0;
}
int dprt_p2p_enabled(const dprt_ctx* ctx) { return ctx && ctx->p2p ? 1 : 0; }

// ---- composite modules ---------------------------------------------------------------------------
int dprt_primary_ray_module(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (deque_enabled(ctx)) {
        int r = deque_begin(ctx);
        for (;;) {
            int done = 0;
            if ((r = deque_traverse(ctx))) return r;
            if (deque_p2p(ctx) && !ctx->p2pGroup) { if ((r = p2p_exchange_enqueue(ctx))) return r; r = p2p_exchange_finish(ctx, &done); }
            else { if ((r = deque_partition(ctx))) return r; r = deque_exchange(ctx, &done); }
            if (r) return r;
            if (done) break;
        }
        return deque_finish(ctx);
    }
    for (;;) {
        int r, done = 0;
        if ((r = dprt_traverse(ctx))) return r;
        if ((r = dprt_partition(ctx))) return r;
        if ((r = dprt_exchange(ctx, &done))) return r;
        if (done) break;
    }
    return 0;
}

int dprt_shadow_ray_module(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    int r;
    if ((r = dprt_shadow_trace(ctx))) return r;
    if (ctx->cfg.proxyMode) {
        int total = 0;
        if ((r = dprt_bucket_queries(ctx, 0, 1, &total))) return r;       // Work_Efficient_Scan_For_NN_HIT_INSIDE
        if ((r = dprt_proxy_infer(ctx, 1, 0))) return r;                  // castShadowRaysDepthNN
        if ((r = dprt_depth_buffer_update(ctx))) return r;
        if ((r = dprt_bucket_queries(ctx, 0, 0, &total))) return r;       // Work_Efficient_Scan_For_NN
        if ((r = dprt_proxy_infer(ctx, 0, 0))) return r;                  // castShadowRaysNN
    } else {
        ctx->queryTotal = 0;
    }
    return dprt_frame_buffer_update(ctx);
}

int dprt_secondary_ray_module(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    int r, total = 0;
    if ((r = dprt_secondary_trace(ctx))) return r;
    if ((r = dprt_bucket_queries(ctx, 1, 0, &total))) return r;
    if ((r = dprt_proxy_infer(ctx, 0, 0))) return r;                      // vis -> pred[0..total)
    if ((r = dprt_proxy_infer(ctx, 1, total))) return r;                  // depth -> pred[total..2 total) (renderer.cpp:956)
    return dprt_target_node_update(ctx);
}

namespace {
// one bounce of runSample for one rank, split at the exchange so that a group can interleave ranks
int bounce_pre(dprt_ctx* ctx, int bounce) {
    int r;
    if (bounce > 0 && ctx->cfg.proxyMode) {
        if ((r = dprt_reset_nn(ctx))) return r;
        if ((r = dprt_secondary_ray_module(ctx))) return r;
    }
    return 0;
}
int bounce_post(dprt_ctx* ctx) {
    int r;
    if ((r = dprt_shade(ctx))) return r;
    if ((r = dprt_reset_nn(ctx))) return r;
    return dprt_shadow_ray_module(ctx);
}
}  // namespace

namespace {
// Single-rank bounce: at W = 1 with proxies off every path the partition keeps was hit on this rank, and traverse_post_kernel
// filed that hit in the hit cache in the current epoch -- the MainRay trace would only copy it from there. So the exchange
// skips the copy of the partition output back to `paths`, and dprt_shade shades straight from `transfer` with the cached
// hits (launch_shade_cached), one launch instead of two plus a D2D copy. The buffers after the bounce are the same: the
// shading program writes every path slot the copy wrote. The parity aid needs hitPrim from the MainRay trace, and an
// uploaded proxy can retarget a path that was not hit. DPRT_SINGLE_RANK_SHORTCUT=0 turns it off (A/B, tests).
bool single_rank_shortcut(const dprt_ctx* ctx) {
    if (ctx->world != 1 || ctx->cfg.proxyMode || !ctx->d_hitCache || ctx->hp.hitPrim) return false;
    for (const ObjectHost& o : ctx->objects) if (o.present && o.desc.isProxy) return false;
    const char* v = getenv("DPRT_SINGLE_RANK_SHORTCUT");
    return !(v && std::strcmp(v, "0") == 0);
}

int render_sample(dprt_ctx* ctx, int sample) {
    int r;
    if ((r = dprt_begin_sample(ctx, sample))) return r;
    if ((r = dprt_path_gen(ctx))) return r;
    // The ShadowRay module of bounce b only reads the shadow paths MainRay(b) wrote (slots >= pathSize) and only writes
    // directLightingBuffer; the TraRay loop of bounce b+1 works on slots < pathSize, the transfer buffer and
    // envLightingBuffer. With proxies off (no shared NN buffers, no host round trip in the shadow module) the two run
    // side by side: shadow(b) on the low-priority aux stream fills the SMs that the tail of the migrate loop leaves idle.
    const bool overlap = ctx->aux && !ctx->profile;
    for (int bounce = 0; bounce <= ctx->cfg.bounces; bounce++) {          // inclusive: renderer.cpp:1530
        if ((r = bounce_pre(ctx, bounce))) return r;
        if ((r = dprt_primary_ray_module(ctx))) return r;
        if (!overlap) { if ((r = bounce_post(ctx))) return r; continue; }
        if ((r = join_aux(ctx))) return r;                                // MainRay rewrites the shadow slots and the pixel lists
        if ((r = dprt_shade(ctx))) return r;
        CK(cudaEventRecord(ctx->evShade, ctx->stream));
        cudaStream_t mainStream = ctx->stream; int32_t* mainQueue = ctx->hp.traceQueue;
        ctx->stream = ctx->aux; ctx->hp.traceQueue = ctx->d_queue_aux;
        cudaError_t ce = cudaStreamWaitEvent(ctx->aux, ctx->evShade, 0);
        r = ce != cudaSuccess ? DPRT_ERR_CUDA : dprt_reset_nn(ctx);
        if (!r) r = dprt_shadow_ray_module(ctx);
        if (!r && cudaEventRecord(ctx->evAux, ctx->aux) != cudaSuccess) r = DPRT_ERR_CUDA;
        ctx->stream = mainStream; ctx->hp.traceQueue = mainQueue;
        if (r) return r;
        ctx->auxPending = true; ctx->auxGuardBase = ctx->pathSize;
    }
    return join_aux(ctx);
}
}  // namespace

int dprt_render_sample(dprt_ctx* ctx, int sample) {
    if (!ctx) return DPRT_ERR_INVALID;
    ctx->shortcut = single_rank_shortcut(ctx);
    const int r = render_sample(ctx, sample);
    ctx->shortcut = false; ctx->recsInTransfer = false;
    return r;
}

int dprt_render_sample_group(dprt_ctx** ctxs, int W, int sample) {
    if (!ctxs || W < 1) return DPRT_ERR_INVALID;
    int r;
    for (int k = 0; k < W; k++) {
        if ((r = dprt_begin_sample(ctxs[k], sample))) return r;
        if ((r = dprt_path_gen(ctxs[k]))) return r;
    }
    const int bounces = ctxs[0]->cfg.bounces;
    bool deque = true;
    for (int k = 0; k < W; k++) deque = deque && ctxs[k] && deque_enabled(ctxs[k]) && ctxs[k]->world == W && ctxs[k]->rank == k;
    // one thread driving W ranks on shared devices: the waiting kernels of all ranks must be able to run side by side, which
    // needs a hardware queue per stream (8 by default, CUDA_DEVICE_MAX_CONNECTIONS); small groups only, opt-in (the
    // group's default exchange is plain peer copies driven by the host)
    const char* pg = getenv("DPRT_P2P_GROUP");
    bool p2p = deque && W > 1 && W <= 8 && pg && pg[0] == '1';
    if (p2p && !ctxs[0]->p2pGroup) { if ((r = p2p_connect_group(ctxs, W))) return r; }
    for (int k = 0; k < W; k++) p2p = p2p && ctxs[k]->p2p && ctxs[k]->p2pGroup;
    for (int k = 0; k < W; k++) ctxs[k]->p2pGroupActive = p2p;
    for (int bounce = 0; bounce <= bounces; bounce++) {
        for (int k = 0; k < W; k++) if ((r = bounce_pre(ctxs[k], bounce))) return r;
        if (deque) for (int k = 0; k < W; k++) deque_begin(ctxs[k]);
        for (;;) {
            int done = 0;
            for (int k = 0; k < W; k++) {
                if ((r = deque ? deque_traverse(ctxs[k]) : dprt_traverse(ctxs[k]))) return r;
                if (!p2p && (r = deque ? deque_partition(ctxs[k]) : dprt_partition(ctxs[k]))) return r;
            }
            if (p2p) {
                for (int k = 0; k < W; k++) if ((r = p2p_exchange_enqueue(ctxs[k]))) return r;      // every rank's kernels are in flight ...
                for (int k = 0; k < W; k++) { int dk = 0; if ((r = p2p_exchange_finish(ctxs[k], &dk))) return r; done = dk; }   // ... before any is waited for
            } else if ((r = deque ? deque_exchange_group(ctxs, W, &done) : dprt_exchange_group(ctxs, W, &done))) return r;
            if (done) break;
        }
        if (deque) for (int k = 0; k < W; k++) if ((r = deque_finish(ctxs[k]))) return r;
        for (int k = 0; k < W; k++) if ((r = bounce_post(ctxs[k]))) return r;
    }
    return 0;
}

int dprt_reduce_image(dprt_ctx* ctx, int root, float* out_host) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int n3 = ctx->N * 3;
    const float* src = ctx->d_image;
    {
        StageScope sc_(ctx, DPRT_STAGE_IMAGE);
        launch_image_average(ctx->hp.direct, ctx->hp.env, ctx->d_image, n3, (float)ctx->cfg.spp, ctx->stream);
        ctx->stats.kernel_launches += 1;
        if (ctx->world > 1) {
            if (!ctx->comm) return fail(ctx, DPRT_ERR_STATE, "dprt_reduce_image on a multi-rank context without an NCCL communicator");
            NK(g_nccl.Reduce(ctx->d_image, ctx->d_image_sum, n3, ncclFloat32, ncclSum, root, ctx->comm, ctx->stream));
            src = ctx->d_image_sum;
        }
    }
    if (ctx->rank == root && out_host)
        CK(cudaMemcpyAsync(out_host, src, sizeof(float) * n3, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int dprt_reduce_image_group(dprt_ctx** ctxs, int W, int root, float* out_host) {
    if (!ctxs || W < 1 || root < 0 || root >= W || !out_host) return DPRT_ERR_INVALID;
    // rank-ordered fp32 sum on the host side of the harness; the NCCL path is dprt_reduce_image
    dprt_ctx* ctx = ctxs[0];
    const int n3 = ctx->N * 3;
    std::vector<float> tmp(n3);
    std::fill(out_host, out_host + n3, 0.f);
    for (int k = 0; k < W; k++) {
        ctx = ctxs[k];
        CK(cudaSetDevice(ctx->device));
        launch_image_average(ctx->hp.direct, ctx->hp.env, ctx->d_image, n3, (float)ctx->cfg.spp, ctx->stream);
        CK(cudaMemcpyAsync(tmp.data(), ctx->d_image, sizeof(float) * n3, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < n3; i++) out_host[i] += tmp[i];
    }
    return 0;
}

// The guide buffers go through the image's scratch (d_image, d_image_sum) one plane at a time: albedo, then normal.
int dprt_reduce_aov(dprt_ctx* ctx, int root, float* albedo_host, float* normal_host) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (!ctx->buf_ptr[DPRT_BUF_AOV]) return fail(ctx, DPRT_ERR_STATE, "dprt_reduce_aov: AOVs were never enabled (dprt_enable_aov)");
    if (ctx->world > 1 && !ctx->comm) return fail(ctx, DPRT_ERR_STATE, "dprt_reduce_aov on a multi-rank context without an NCCL communicator");
    CK(cudaSetDevice(ctx->device));
    const int n3 = ctx->N * 3;
    float* out[2] = {albedo_host, normal_host};
    for (int plane = 0; plane < 2; plane++) {
        const float* src = ctx->d_image;
        {
            StageScope sc_(ctx, DPRT_STAGE_IMAGE);
            launch_aov_average((const float*)ctx->buf_ptr[DPRT_BUF_AOV] + (size_t)plane * n3, ctx->d_image, n3, (float)ctx->cfg.spp, ctx->stream);
            ctx->stats.kernel_launches += 1;
            if (ctx->world > 1) {
                NK(g_nccl.Reduce(ctx->d_image, ctx->d_image_sum, n3, ncclFloat32, ncclSum, root, ctx->comm, ctx->stream));
                src = ctx->d_image_sum;
            }
        }
        if (ctx->rank == root && out[plane])
            CK(cudaMemcpyAsync(out[plane], src, sizeof(float) * n3, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));       // the next plane reuses the scratch
    }
    return 0;
}

int dprt_reduce_aov_group(dprt_ctx** ctxs, int W, int root, float* albedo_host, float* normal_host) {
    if (!ctxs || W < 1 || root < 0 || root >= W || !albedo_host || !normal_host) return DPRT_ERR_INVALID;
    for (int k = 0; k < W; k++)
        if (!ctxs[k]->buf_ptr[DPRT_BUF_AOV]) return fail(ctxs[k], DPRT_ERR_STATE, "dprt_reduce_aov_group: AOVs were never enabled (dprt_enable_aov)");
    // rank-ordered fp32 sum on the host, like dprt_reduce_image_group
    const int n3 = ctxs[0]->N * 3;
    std::vector<float> tmp(n3);
    float* out[2] = {albedo_host, normal_host};
    for (int plane = 0; plane < 2; plane++) {
        std::fill(out[plane], out[plane] + n3, 0.f);
        for (int k = 0; k < W; k++) {
            dprt_ctx* ctx = ctxs[k];
            CK(cudaSetDevice(ctx->device));
            launch_aov_average((const float*)ctx->buf_ptr[DPRT_BUF_AOV] + (size_t)plane * n3, ctx->d_image, n3, (float)ctx->cfg.spp, ctx->stream);
            CK(cudaMemcpyAsync(tmp.data(), ctx->d_image, sizeof(float) * n3, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            for (int i = 0; i < n3; i++) out[plane][i] += tmp[i];
        }
    }
    return 0;
}

// ---- state access ----------------------------------------------------------------------------------
int dprt_get_path_size(const dprt_ctx* ctx, int* ps, int* sps) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (ps) *ps = ctx->pathSize;
    if (sps) *sps = ctx->shadowPathSize;
    return 0;
}
int dprt_set_path_size(dprt_ctx* ctx, int ps) {
    if (!ctx || ps < 0 || ps > ctx->N) return DPRT_ERR_INVALID;
    ctx->pathSize = ps; ctx->histFresh = false; ctx->qhistFresh = false;
    ctx->epoch++;                       // the harness is about to install its own paths
    ctx->shadeIdx = -1;
    return 0;
}
int dprt_buffer_bytes(const dprt_ctx* ctx, int id, size_t* bytes) {
    if (!ctx || id < 0 || id >= DPRT_BUF_COUNT || !bytes) return DPRT_ERR_INVALID;
    *bytes = ctx->buf_bytes[id]; return 0;
}
int dprt_download(dprt_ctx* ctx, int id, size_t off, void* host, size_t bytes) {
    if (!ctx || id < 0 || id >= DPRT_BUF_COUNT || !host) return DPRT_ERR_INVALID;
    if (!ctx->buf_ptr[id] || off + bytes > ctx->buf_bytes[id]) return fail(ctx, DPRT_ERR_CAPACITY, "download range outside buffer");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(host, (const char*)ctx->buf_ptr[id] + off, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
int dprt_upload(dprt_ctx* ctx, int id, size_t off, const void* host, size_t bytes) {
    if (!ctx || id < 0 || id >= DPRT_BUF_COUNT || !host) return DPRT_ERR_INVALID;
    if (!ctx->buf_ptr[id] || off + bytes > ctx->buf_bytes[id]) return fail(ctx, DPRT_ERR_CAPACITY, "upload range outside buffer");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync((char*)ctx->buf_ptr[id] + off, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->histFresh = false; ctx->qhistFresh = false;
    if (id == DPRT_BUF_PATHS) { ctx->epoch++; ctx->shadeIdx = -1; }
    if (id == DPRT_BUF_DIRECT) ctx->dirtyIdx = -2;
    if (id == DPRT_BUF_OCCLUSION || id == DPRT_BUF_CONTRIBUTION) { ctx->nnScratchDirty = true; ctx->dirtyIdx = -2; }
    return 0;
}
int dprt_enable_hit_prim(dprt_ctx* ctx, int enable) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (enable && !ctx->buf_ptr[DPRT_BUF_HIT_PRIM]) {
        int r = alloc_buf(ctx, DPRT_BUF_HIT_PRIM, (size_t)(1 + ctx->cfg.shadowPathCount) * ctx->N * sizeof(int32_t));
        if (r) return r;
    }
    ctx->hp.hitPrim = enable ? (int32_t*)ctx->buf_ptr[DPRT_BUF_HIT_PRIM] : nullptr;
    return 0;
}
int dprt_enable_aov(dprt_ctx* ctx, int enable) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (enable && !ctx->buf_ptr[DPRT_BUF_AOV]) {
        int r = alloc_buf(ctx, DPRT_BUF_AOV, 6 * (size_t)ctx->N * sizeof(float));
        if (r) return r;
    }
    ctx->d_aov = enable ? (float*)ctx->buf_ptr[DPRT_BUF_AOV] : nullptr;
    return 0;
}

// ---- standalone operators ----------------------------------------------------------------------------
// the ray queue head of the persistent trace kernel is a 32-bit counter that every resident warp may bump by 32 past n
static const int64_t kMaxTraceRays = (int64_t)0x7fffffff - (int64_t)(1 << 20);

int dprt_trace_closest_device(dprt_ctx* ctx, const void* rays_dev, int64_t n, void* hits_dev) {
    if (!ctx || !rays_dev || !hits_dev || n < 0) return DPRT_ERR_INVALID;
    if (n > kMaxTraceRays) return fail(ctx, DPRT_ERR_INVALID, "more rays than one launch can index (split the batch)");
    CK(cudaSetDevice(ctx->device));
    StageScope sc_(ctx, DPRT_STAGE_TRACE_CLOSEST, n > 0);
    launch_trace_closest(ctx->d_objects, ctx->cfg.sceneSize, ctx->d_textures, ctx->d_matTex, (const dprt_ray*)rays_dev, (dprt_hit*)hits_dev, n, ctx->d_queue,
                         ctx->hp.counters, ctx->stream);
    ctx->stats.kernel_launches += n > 0;
    ctx->stats.rays_traverse += n;
    CK(cudaGetLastError());
    return 0;
}

int dprt_trace_closest(dprt_ctx* ctx, const dprt_ray* rays_host, int64_t n, dprt_hit* hits_host) {
    if (!ctx || !rays_host || !hits_host || n < 0) return DPRT_ERR_INVALID;
    if (n > kMaxTraceRays) return fail(ctx, DPRT_ERR_INVALID, "more rays than one launch can index (split the batch)");
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const size_t rb = (size_t)n * sizeof(dprt_ray), hb = (size_t)n * sizeof(dprt_hit);
    int r = ensure_io(ctx, rb + hb); if (r) return r;
    char* d = (char*)ctx->d_io;
    CK(cudaMemcpyAsync(d, rays_host, rb, cudaMemcpyHostToDevice, ctx->stream));
    if ((r = dprt_trace_closest_device(ctx, d, n, d + rb))) return r;
    CK(cudaMemcpyAsync(hits_host, d + rb, hb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int dprt_gen_train_data(dprt_ctx* ctx, int si, const dprt_ray* rays_host, int64_t n, float* features_host, float* labels_host) {
    if (!ctx || !rays_host || !features_host || !labels_host || n < 0) return DPRT_ERR_INVALID;
    if (si < 0 || si >= ctx->cfg.sceneSize || !ctx->objects[si].present || ctx->objects[si].desc.isProxy || !ctx->objects[si].d_nodes)
        return fail(ctx, DPRT_ERR_STATE, "training data can only be generated for an object whose geometry is on this rank");
    if (n > kMaxTraceRays) return fail(ctx, DPRT_ERR_INVALID, "more rays than one launch can index (split the batch)");
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const size_t rb = (size_t)n * sizeof(dprt_ray), hb = (size_t)n * sizeof(dprt_hit), fb = (size_t)n * 5 * sizeof(float), lb = (size_t)n * sizeof(float);
    int r = ensure_io(ctx, rb + hb + fb + lb); if (r) return r;
    char* d = (char*)ctx->d_io;
    CK(cudaMemcpyAsync(d, rays_host, rb, cudaMemcpyHostToDevice, ctx->stream));
    {
        StageScope sc_(ctx, DPRT_STAGE_TRACE_CLOSEST);
        launch_trace_closest(ctx->d_objects + si, 1, ctx->d_textures, ctx->d_matTex, (const dprt_ray*)d, (dprt_hit*)(d + rb), n, ctx->d_queue, ctx->hp.counters, ctx->stream);   // startObj only
        launch_train_features(ctx->d_objects + si, (const dprt_ray*)d, (const dprt_hit*)(d + rb), n, (float*)(d + rb + hb), (float*)(d + rb + hb + fb), ctx->stream);
    }
    ctx->stats.kernel_launches += 2;
    CK(cudaMemcpyAsync(features_host, d + rb + hb, fb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(labels_host, d + rb + hb + fb, lb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    return 0;
}

int dprt_gen_precom_data(dprt_ctx* ctx, int si, const dprt_ray* rays_host, int64_t n, float* features_host, float* labels_host,
                         uint8_t* valid_host) {
    if (!ctx || !rays_host || !features_host || !labels_host || !valid_host || n < 0) return DPRT_ERR_INVALID;
    if (si < 0 || si >= ctx->cfg.sceneSize || !ctx->objects[si].present || ctx->objects[si].desc.isProxy || !ctx->objects[si].d_nodes)
        return fail(ctx, DPRT_ERR_STATE, "training data can only be generated for an object whose geometry is on this rank");
    if (n > kMaxTraceRays) return fail(ctx, DPRT_ERR_INVALID, "more rays than one launch can index (split the batch)");
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const size_t rb = (size_t)n * sizeof(dprt_ray), hb = (size_t)n * sizeof(dprt_hit), fb = (size_t)n * 5 * sizeof(float), lb = (size_t)n * sizeof(float);
    int r = ensure_io(ctx, rb + hb + fb + 2 * lb + (size_t)n + 256); if (r) return r;
    char* d = (char*)ctx->d_io;
    dprt_ray* d_rays = (dprt_ray*)d; dprt_hit* d_hits = (dprt_hit*)(d + rb);
    float* d_feat = (float*)(d + rb + hb); float* d_label = (float*)(d + rb + hb + fb); float* d_ta = (float*)(d + rb + hb + fb + lb);
    uint8_t* d_valid = (uint8_t*)(d + rb + hb + fb + 2 * lb);
    CK(cudaMemcpyAsync(d_rays, rays_host, rb, cudaMemcpyHostToDevice, ctx->stream));
    {
        StageScope sc_(ctx, DPRT_STAGE_TRACE_CLOSEST);
        launch_precom_features(ctx->d_objects + si, d_rays, n, d_feat, d_ta, ctx->stream);                 // proxy AABB (aabbHandle)
        launch_trace_closest(ctx->d_objects + si, 1, ctx->d_textures, ctx->d_matTex, d_rays, d_hits, n, ctx->d_queue, ctx->hp.counters, ctx->stream);   // originHandle, tMax = inf
        launch_precom_labels(ctx->d_objects + si, d_hits, d_ta, n, d_label, d_valid, ctx->stream);
    }
    ctx->stats.kernel_launches += 3;
    CK(cudaMemcpyAsync(features_host, d_feat, fb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(labels_host, d_label, lb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(valid_host, d_valid, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    return 0;
}

int dprt_mlp_infer_device(dprt_ctx* ctx, int si, int kind, const void* x_dev, int64_t n, void* y_dev) {
    if (!ctx || si < 0 || si >= ctx->cfg.sceneSize || !x_dev || !y_dev || n < 0) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const MlpModel* m = kind == 0 ? ctx->objects[si].vis : ctx->objects[si].depth;
    if (!m) return fail(ctx, DPRT_ERR_STATE, "no proxy model uploaded for this scene object");
    if (n == 0) return 0;
    if (mlp_forward(m, (const dprt_half*)x_dev, (dprt_half*)y_dev, n, ctx->stream, ctx->err)) return DPRT_ERR_CUDA;
    ctx->stats.kernel_launches += 1; ctx->stats.nn_queries += n;
    CK(cudaGetLastError());
    return 0;
}

int dprt_mlp_infer(dprt_ctx* ctx, int si, int kind, const dprt_half* x_host, int64_t n, dprt_half* y_host) {
    if (!ctx || !x_host || !y_host || n < 0) return DPRT_ERR_INVALID;
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const size_t xb = ((size_t)n * 5 * sizeof(dprt_half) + 255) & ~(size_t)255, yb = (size_t)n * sizeof(dprt_half);
    int r = ensure_io(ctx, xb + yb + 256); if (r) return r;
    char* d = (char*)ctx->d_io;
    CK(cudaMemcpyAsync(d, x_host, (size_t)n * 5 * sizeof(dprt_half), cudaMemcpyHostToDevice, ctx->stream));
    if ((r = dprt_mlp_infer_device(ctx, si, kind, d, n, d + xb))) return r;
    CK(cudaMemcpyAsync(y_host, d + xb, yb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---- denoiser (denoise.cu, DESIGN.md 3.8) -------------------------------------------------------------------------------
int dprt_denoise_device(dprt_ctx* ctx, const dprt_denoise_params* p, int width, int height, const void* color_dev,
                        const void* albedo_dev, const void* normal_dev, void* out_dev) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (!color_dev || !albedo_dev || !normal_dev || !out_dev) return fail(ctx, DPRT_ERR_INVALID, "dprt_denoise_device: null array");
    dprt_denoise_params q;
    const char* why = nullptr;
    if (denoise_check(p, width, height, &q, &why)) return fail(ctx, DPRT_ERR_INVALID, std::string("dprt_denoise_device: ") + why);
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = denoise_scratch_bytes((int64_t)width * height);
    if (ctx->denoise_bytes < bytes) {
        void* old = ctx->d_denoise;
        ctx->d_denoise = nullptr; ctx->denoise_bytes = 0;
        if (old) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaFree(old)); }
        CK(cudaMalloc(&ctx->d_denoise, bytes));
        ctx->denoise_bytes = bytes;
    }
    launch_denoise(q, width, height, (const float*)color_dev, (const float*)albedo_dev, (const float*)normal_dev, (float*)out_dev,
                   ctx->d_denoise, ctx->stream);
    ctx->stats.kernel_launches += 1 + q.iterations;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int dprt_denoise(dprt_ctx* ctx, const dprt_denoise_params* p, int width, int height, const float* color_host, const float* albedo_host,
                 const float* normal_host, float* out_host) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (!color_host || !albedo_host || !normal_host || !out_host) return fail(ctx, DPRT_ERR_INVALID, "dprt_denoise: null array");
    dprt_denoise_params q;
    const char* why = nullptr;
    if (denoise_check(p, width, height, &q, &why)) return fail(ctx, DPRT_ERR_INVALID, std::string("dprt_denoise: ") + why);
    CK(cudaSetDevice(ctx->device));
    const size_t b = (size_t)width * height * 3 * sizeof(float), bs = (b + 255) & ~(size_t)255;
    int r = ensure_io(ctx, 3 * bs); if (r) return r;
    char* d = (char*)ctx->d_io;
    CK(cudaMemcpyAsync(d, color_host, b, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d + bs, albedo_host, b, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d + 2 * bs, normal_host, b, cudaMemcpyHostToDevice, ctx->stream));
    if ((r = dprt_denoise_device(ctx, &q, width, height, d, d + bs, d + 2 * bs, d))) return r;     // the result over the colour
    CK(cudaMemcpyAsync(out_host, d, b, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int dprt_spec_denoise(const dprt_denoise_params* p, int width, int height, const float* color, const float* albedo, const float* normal,
                      float* out) {
    if (!color || !albedo || !normal || !out) return DPRT_ERR_INVALID;
    dprt_denoise_params q;
    const char* why = nullptr;
    if (denoise_check(p, width, height, &q, &why)) return DPRT_ERR_INVALID;
    return spec_denoise(q, width, height, color, albedo, normal, out);
}

// ---- BVH8 refit (refit.cu, DESIGN.md 3.9) -------------------------------------------------------------------------------
namespace {
// the checks that need no look at the vertices; *out = the chunk
int refit_target(dprt_ctx* ctx, int si, bool has_normals, int64_t ntris, const char* fn, ObjectHost** out) {
    if (si < 0 || si >= ctx->cfg.sceneSize || !ctx->objects[si].present)
        return fail(ctx, DPRT_ERR_INVALID, std::string(fn) + ": no scene object uploaded at this index");
    ObjectHost& o = ctx->objects[si];
    if (o.desc.isProxy || !o.d_nodes) return fail(ctx, DPRT_ERR_INVALID, std::string(fn) + ": the object is not a local chunk");
    if (ntris != o.ntris) return fail(ctx, DPRT_ERR_INVALID, std::string(fn) + ": triangle count differs from the upload's");
    if (has_normals != (o.d_normals != nullptr))
        return fail(ctx, DPRT_ERR_INVALID, std::string(fn) + (has_normals ? ": normals given for a chunk uploaded without them"
                                                                          : ": the chunk was uploaded with normals and none are given"));
    *out = &o;
    return 0;
}
}  // namespace

int dprt_refit_chunk_device(dprt_ctx* ctx, int si, const void* verts9_dev, const void* normals9_dev, int64_t ntris) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (!verts9_dev) return fail(ctx, DPRT_ERR_INVALID, "dprt_refit_chunk_device: null vertex array");
    ObjectHost* o = nullptr;
    int r = refit_target(ctx, si, normals9_dev != nullptr, ntris, "dprt_refit_chunk_device", &o);
    if (r) return r;
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = refit_scratch_bytes(o->nnodes);
    if (ctx->refit_bytes < bytes) {
        void* old = ctx->d_refit;
        ctx->d_refit = nullptr; ctx->refit_bytes = 0;
        CK(cudaStreamSynchronize(ctx->stream));
        if (old) CK(cudaFree(old));
        CK(cudaMalloc(&ctx->d_refit, bytes));
        ctx->refit_bytes = bytes;
    }
    // validate on the device: one reduction, one read-back; nothing is written before it has passed
    const float* v = (const float*)verts9_dev;
    launch_refit_stats(v, ntris, ctx->d_refit, ctx->stream);
    CK(cudaGetLastError());
    RefitStats st;
    CK(cudaMemcpyAsync(&st, ctx->d_refit, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.nonfinite) return fail(ctx, DPRT_ERR_INVALID, "dprt_refit_chunk_device: " + std::to_string(st.nonfinite) + " non-finite coordinates");
    float m = 0.f;
    for (int a = 0; a < 3; a++) {
        if (st.lo[a] < o->desc.aabbMin[a] || st.hi[a] > o->desc.aabbMax[a])
            return fail(ctx, DPRT_ERR_INVALID, "dprt_refit_chunk_device: a vertex lies outside the object's aabbMin / aabbMax");
        m = std::max(m, std::max(std::fabs(st.lo[a]), std::fabs(st.hi[a])));
    }
    if (ctx->aux) CK(cudaStreamSynchronize(ctx->aux));     // the ShadowRay module dprt_render_sample may have left running
    const std::vector<int64_t>& lv = o->mem->levels;
    launch_refit((dprt_bvh8_node*)o->d_nodes, (dprt_bvh8_tri*)o->d_tris, ntris, v, lv.data(), (int)lv.size() - 1, bvh8_chunk_pad(m),
                 ctx->d_refit, ctx->stream);
    CK(cudaGetLastError());
    if (normals9_dev)
        CK(cudaMemcpyAsync(o->d_normals, normals9_dev, (size_t)ntris * 9 * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int dprt_refit_chunk(dprt_ctx* ctx, int si, const float* verts9, const float* normals9, int64_t ntris) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (!verts9) return fail(ctx, DPRT_ERR_INVALID, "dprt_refit_chunk: null vertex array");
    ObjectHost* o = nullptr;
    int r = refit_target(ctx, si, normals9 != nullptr, ntris, "dprt_refit_chunk", &o);
    if (r) return r;
    CK(cudaSetDevice(ctx->device));
    const size_t b = (size_t)ntris * 9 * sizeof(float);
    if ((r = ensure_io(ctx, normals9 ? 2 * b : b))) return r;
    char* d = (char*)ctx->d_io;
    CK(cudaMemcpyAsync(d, verts9, b, cudaMemcpyHostToDevice, ctx->stream));
    if (normals9) CK(cudaMemcpyAsync(d + b, normals9, b, cudaMemcpyHostToDevice, ctx->stream));
    return dprt_refit_chunk_device(ctx, si, d, normals9 ? d + b : nullptr, ntris);
}

int dprt_spec_bvh8_refit(dprt_bvh8_node* nodes, int64_t nnodes, dprt_bvh8_tri* tris, int64_t ntris, const float* verts9) {
    const char* why = nullptr;
    return spec_bvh8_refit(nodes, nnodes, tris, ntris, verts9, &why);
}

int dprt_chunk_bvh8_copy(dprt_ctx* ctx, int si, int64_t* nnodes, int64_t* ntris, dprt_bvh8_node* nodes_out, dprt_bvh8_tri* tris_out) {
    if (!ctx) return DPRT_ERR_INVALID;
    if (si < 0 || si >= ctx->cfg.sceneSize || !ctx->objects[si].present || ctx->objects[si].desc.isProxy || !ctx->objects[si].d_nodes)
        return fail(ctx, DPRT_ERR_INVALID, "dprt_chunk_bvh8_copy: no local chunk at this index");
    const ObjectHost& o = ctx->objects[si];
    if (nnodes) *nnodes = o.nnodes;
    if (ntris) *ntris = o.ntris;
    if (!nodes_out && !tris_out) return 0;
    CK(cudaSetDevice(ctx->device));
    if (nodes_out) CK(cudaMemcpyAsync(nodes_out, o.d_nodes, (size_t)o.nnodes * sizeof(dprt_bvh8_node), cudaMemcpyDeviceToHost, ctx->stream));
    if (tris_out) CK(cudaMemcpyAsync(tris_out, o.d_tris, (size_t)o.ntris * sizeof(dprt_bvh8_tri), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int dprt_device_alloc(dprt_ctx* ctx, size_t bytes, void** dev_ptr) {
    if (!ctx || !dev_ptr) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMalloc(dev_ptr, std::max<size_t>(bytes, 256)));
    ctx->user_allocs.push_back(*dev_ptr);
    return 0;
}
int dprt_device_free(dprt_ctx* ctx, void* dev_ptr) {
    if (!ctx) return DPRT_ERR_INVALID;
    auto it = std::find(ctx->user_allocs.begin(), ctx->user_allocs.end(), dev_ptr);
    if (it == ctx->user_allocs.end()) return DPRT_ERR_INVALID;
    ctx->user_allocs.erase(it);
    CK(cudaSetDevice(ctx->device));
    CK(cudaFree(dev_ptr));
    return 0;
}
int dprt_memcpy_h2d(dprt_ctx* ctx, void* dev, const void* host, size_t bytes) {
    if (!ctx || !dev || !host) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
int dprt_memcpy_d2h(dprt_ctx* ctx, void* host, const void* dev, size_t bytes) {
    if (!ctx || !dev || !host) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
int dprt_timer_start(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    return 0;
}
int dprt_timer_stop(dprt_ctx* ctx, float* ms) {
    if (!ctx || !ms) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    CK(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return 0;
}
int dprt_flush_l2(dprt_ctx* ctx) {
    if (!ctx) return DPRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->d_flush) { ctx->flush_bytes = (size_t)256 << 20; CK(cudaMalloc(&ctx->d_flush, ctx->flush_bytes)); }
    CK(cudaMemsetAsync(ctx->d_flush, 0, ctx->flush_bytes, ctx->stream));
    return 0;
}

}  // extern "C"
