// partition.cu -- single-pass stable multi-bucket partition (sm_100a).
//
// Replaces the reference's per-destination loop of {preKernel, 3x prefixSum, 2x prefixFixup, postKernel}
// (src/cuda/cuda_compaction.cu:8-35,306-439 for paths by targetNode; :140-198,441-617 for NN queries by
// hitAABBID) -- W (or sceneSize) sequential passes of 7 launches each -- with ONE launch:
//   * keys are read once (the last 16 B of a path record / the id words of a query),
//   * in-tile ranks come from warp match/ballot, tile prefixes from a decoupled look-back chain that carries
//     one counter per bucket (lane b of warp 0 owns bucket b),
//   * bucket bases come from the histogram the producing kernel already accumulated (traverse / shadow /
//     secondary), so records are scattered straight to their final, contiguous, bucket-major position.
// Output order is the reference's: bucket-major, original index order inside a bucket, dead entries dropped.
#include <algorithm>
#include <cstdlib>
#include "dprt_internal.cuh"
#include "p2p_exchange.cuh"

namespace dprt {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
// ITEMS records per thread: a tile is kThreads * ITEMS records and kWarps * ITEMS (warp, item) steps in index order.
// 4 for the 64-byte path records; 16 for NN queries, where the key is one byte, nearly all slots are empty and the cost
// is the length of the tile chain, not the bytes.

constexpr uint32_t ST_AGG = 1u << 30, ST_INC = 2u << 30, ST_MASK = 3u << 30, VAL_MASK = ~ST_MASK;
// Tile states are 64-bit words {launch generation, status | value}: a word only counts when its generation is this launch's,
// and tile ids are the running ticket counter minus the tickets of all earlier launches -- so neither the state array nor
// the counter is ever cleared (two cudaMemsetAsync per partition launch gone from the migrate loop).

// Bucket of path record i from its last two words (targetNode, flags): -1 unless it is valid and addressed to one of the W
// ranks; a record that stays on rank `me` and sits at index >= splitL goes to bucket W, which only exists in settled-deque
// mode (B == W + 1; me == -1 otherwise). Reading W, me and splitL through `ops` keeps the early exit a branch: as plain
// arguments, the compiler turns it into selects evaluated for every record.
template <class Ops>
__device__ __forceinline__ int path_bucket(const Ops& ops, uint32_t targetNode, uint32_t flags, int i) {
    const int target = (int)targetNode;
    const bool valid = (flags >> 16) & 0xffu;
    if (!(valid && target >= 0 && target < ops.W)) return -1;
    return (target == ops.me && i >= ops.splitL) ? ops.W : target;
}

struct PathOps {
    static constexpr bool kDirect = false;
    const dprt_path_record* in; dprt_path_record* out; int B; int W; int me; int splitL;
    __device__ __forceinline__ bool skip() const { return false; }
    __device__ __forceinline__ int key(int i) const {
        const uint4 w = reinterpret_cast<const uint4*>(in + i)[3];   // visitedMask, currentNode, targetNode, flags
        return path_bucket(*this, w.z, w.w, i);
    }
    __device__ __forceinline__ void copy(int src, int /*bucket*/, int dst) const {
        const float4* s = reinterpret_cast<const float4*>(in + src);
        float4* d = reinterpret_cast<float4*>(out + dst);
        const float4 a = s[0], b = s[1], c = s[2], e = s[3];
        d[0] = a; d[1] = b; d[2] = c; d[3] = e;
    }
    // staged variant (partition_staged_kernel): key of record i from the last 8 bytes of its staged copy; where bucket b goes
    __device__ __forceinline__ int key_staged(uint2 w, int i) const { return path_bucket(*this, w.x, w.y, i); }
    __device__ __forceinline__ dprt_path_record* dst_base(int /*bucket*/) const { return out; }
};

// Peer-memory exchange (p2p_exchange.cuh): same keys as PathOps in settled-deque mode, but every bucket has its own
// destination pointer, taken from the plan the counts kernel left in device memory -- a peer's receive buffer behind
// NVLink for the travelling buckets, the local settled block for the two self pieces. `dst` is the index inside the bucket.
struct PeerPathOps {
    static constexpr bool kDirect = true;
    const dprt_path_record* in; const P2PPlan* plan; int B; int W; int me; int splitL;
    __device__ __forceinline__ bool skip() const { return *(const volatile int32_t*)&plan->error != 0; }
    __device__ __forceinline__ int key(int i) const {
        const uint4 w = reinterpret_cast<const uint4*>(in + i)[3];
        return path_bucket(*this, w.z, w.w, i);
    }
    __device__ __forceinline__ void copy(int src, int bucket, int dst) const {
        const float4* s = reinterpret_cast<const float4*>(in + src);
        float4* d = reinterpret_cast<float4*>(plan->dst[bucket] + dst);
        const float4 a = s[0], b = s[1], c = s[2], e = s[3];
        d[0] = a; d[1] = b; d[2] = c; d[3] = e;
    }
    __device__ __forceinline__ int key_staged(uint2 w, int i) const { return path_bucket(*this, w.x, w.y, i); }
    __device__ __forceinline__ dprt_path_record* dst_base(int bucket) const { return plan->dst[bucket]; }
};

struct QueryOps {
    static constexpr bool kDirect = false;
    __device__ __forceinline__ bool skip() const { return false; }
    const dprt_nn_query* in; const uint8_t* keys; const dprt_half* fin; dprt_nn_query* out; dprt_half* fout; int B; int insideOnly;
    __device__ __forceinline__ int key(int i) const {
        int id; bool inside;
        if (keys) { const uint32_t k = keys[i]; id = (int)(k & 0x7fu); inside = (k >> 7) != 0u; }   // 1 byte instead of a 48-byte record
        else { id = in[i].hitAABBID; inside = in[i].isInside != 0; }
        if (id < 1 || id > B) return -1;                // preKernelNN: hitAABBID == AABBID (scene index + 1)
        if (insideOnly && !inside) return -1;           // preKernelNN_HIT_INSIDE
        return id - 1;
    }
    __device__ __forceinline__ void copy(int src, int /*bucket*/, int dst) const {
        const float4* s = reinterpret_cast<const float4*>(in + src);
        float4* d = reinterpret_cast<float4*>(out + dst);
        const float4 a = s[0], b = s[1], c = s[2];
        d[0] = a; d[1] = b; d[2] = c;
        const dprt_half* fs = fin + (size_t)src * 5; dprt_half* fd = fout + (size_t)dst * 5;
#pragma unroll
        for (int k = 0; k < 5; k++) fd[k] = fs[k];
    }
};

// Warp 0 of a tile, lane = bucket, once the per-step counts s_cnt[0..kSteps) are in: turns them into exclusive in-tile
// offsets and returns where the tile's first record of the bucket goes. That is the bucket base plus the bucket's records in
// all earlier tiles.
template <class Ops, int kSteps>
__device__ __forceinline__ int tile_bucket_base(int (*s_cnt)[32], int lane, int B, int tile, const int32_t* __restrict__ hist,
                                                int32_t* __restrict__ offsets, unsigned long long* tileState, uint32_t gen) {
    // exclusive scan over the in-tile steps
    int run = 0;
#pragma unroll 8
    for (int s = 0; s < kSteps; s++) { const int c = s_cnt[s][lane]; s_cnt[s][lane] = run; run += c; }
    // bucket bases = exclusive prefix of the histogram (direct mode: every bucket has its own destination, base 0)
    int bucketBase = 0;
    if (!Ops::kDirect) {
        const int h = lane < B ? hist[lane] : 0;
        int incl = h;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        bucketBase = incl - h;
        if (tile == 0) {
            if (lane < B) offsets[lane] = bucketBase;
            if (lane == B - 1) offsets[B] = incl;
        }
    }
    // decoupled look-back, one chain per bucket
    int excl = 0;
    if (lane < B) {
        volatile unsigned long long* st = tileState;
        const unsigned long long g = (unsigned long long)gen << 32;
        if (tile == 0) {
            st[lane] = g | ST_INC | (uint32_t)run;
        } else {
            st[(size_t)tile * 32 + lane] = g | ST_AGG | (uint32_t)run;
            int t = tile - 1;
            for (;;) {
                unsigned long long w;
                do { w = st[(size_t)t * 32 + lane]; } while ((w >> 32) != gen);      // older generations: not written yet
                const uint32_t v = (uint32_t)w;
                excl += (int)(v & VAL_MASK);
                if ((v & ST_MASK) == ST_INC) break;
                t--;
            }
            st[(size_t)tile * 32 + lane] = g | ST_INC | (uint32_t)(excl + run);
        }
    }
    return bucketBase + excl;
}

template <class Ops, int kItems>
__global__ void __launch_bounds__(kThreads) partition_kernel(Ops ops, int n, const int32_t* __restrict__ hist,
                                                              int32_t* __restrict__ offsets, unsigned long long* tileState,
                                                              uint32_t* tileCounter, uint32_t ticketBase, uint32_t gen) {
    constexpr int kTile = kThreads * kItems, kSteps = kWarps * kItems;
    __shared__ int s_tile;
    __shared__ int s_cnt[kSteps][32];
    __shared__ int s_base[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int B = ops.B;

    if (threadIdx.x == 0) s_tile = (int)(atomicAdd(tileCounter, 1u) - ticketBase);   // launch-order tile ids: predecessors are always running
    if (ops.skip()) return;                                      // block-uniform (peer exchange: the plan carries an error); ticket taken
    for (int k = threadIdx.x; k < kSteps * 32; k += kThreads) (&s_cnt[0][0])[k] = 0;
    __syncthreads();
    const int tile = s_tile;

    int key[kItems], rank[kItems];
    const int base = tile * kTile + warp * (32 * kItems);
#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const int idx = base + j * 32 + lane;
        key[j] = idx < n ? ops.key(idx) : -1;
    }
#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const bool v = key[j] >= 0;
        const unsigned m = __ballot_sync(0xffffffffu, v);
        rank[j] = 0;
        if (v) {
            const unsigned peers = __match_any_sync(m, key[j]);
            rank[j] = __popc(peers & ((1u << lane) - 1u));
            if (rank[j] == 0) s_cnt[warp * kItems + j][key[j]] = __popc(peers);
        }
    }
    __syncthreads();

    if (warp == 0) s_base[lane] = tile_bucket_base<Ops, kSteps>(s_cnt, lane, B, tile, hist, offsets, tileState, gen);
    __syncthreads();

#pragma unroll
    for (int j = 0; j < kItems; j++) {
        if (key[j] >= 0) {
            const int idx = base + j * 32 + lane;
            const int dst = s_base[key[j]] + s_cnt[warp * kItems + j][key[j]] + rank[j];
            ops.copy(idx, key[j], dst);
        }
    }
}


// ---- TMA-staged variant for the 64-byte path records -------------------------------------------------------------------
// Same single-pass algorithm (launch-order tile ids, warp match ranks, 32-bucket decoupled look-back), different data
// movement: the tile's 1024 records = 64 KiB arrive in shared memory as ONE bulk copy (cp.async.bulk + mbarrier: every byte
// of the input crosses DRAM once, in full lines, and no thread spends instructions on it); keys are read from the staged
// copy; the scatter runs in 64-byte record units -- four lanes per record, eight records per warp store instruction -- so a
// run of records that stay together (the usual case in a stable partition) leaves the SM as contiguous 512-byte stores,
// to local HBM or to a peer's receive buffer behind NVLink. The per-thread LDG/STG.128 version above stays for the NN queries.

constexpr int kStageTile = 1024;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <class Ops>
__global__ void __launch_bounds__(kThreads) partition_staged_kernel(Ops ops, int n, const int32_t* __restrict__ hist, int32_t* __restrict__ offsets,
                                                                     unsigned long long* tileState, uint32_t* tileCounter, uint32_t ticketBase,
                                                                     uint32_t gen) {
    constexpr int kStageSteps = kStageTile / 32;
    extern __shared__ __align__(128) uint8_t s_stage[];            // kStageTile x 64 B
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ int s_tile;
    __shared__ int s_cnt[kStageSteps][32];
    __shared__ int s_base[32];
    __shared__ uint32_t s_dst[kStageTile];                         // bucket << 27 | index inside the bucket, ~0 = dropped
    __shared__ dprt_path_record* s_ptr[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int B = ops.B;
    constexpr int kItems = kStageTile / kThreads;                  // 4

    if (threadIdx.x == 0) s_tile = (int)(atomicAdd(tileCounter, 1u) - ticketBase);
    if (ops.skip()) return;
    for (int k = threadIdx.x; k < kStageSteps * 32; k += kThreads) (&s_cnt[0][0])[k] = 0;
    if (threadIdx.x < 32) s_ptr[threadIdx.x] = threadIdx.x < B ? ops.dst_base(threadIdx.x) : nullptr;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&s_bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int tile = s_tile;
    const int first = tile * kStageTile;
    const int valid = min(kStageTile, n - first);
    if (threadIdx.x == 0) {
        const uint32_t bytes = (uint32_t)valid * (uint32_t)sizeof(dprt_path_record);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(&s_bar)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(s_stage)),
                     "l"(ops.in + first), "r"(bytes), "r"(smem_addr(&s_bar))
                     : "memory");
    }
    {   // everybody waits for the tile
        uint32_t ok = 0;
        while (!ok) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(ok) : "r"(smem_addr(&s_bar)) : "memory");
        }
    }

    int key[kItems], rank[kItems];
    const int wbase = warp * (32 * kItems);
#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const int r = wbase + j * 32 + lane;
        key[j] = r < valid ? ops.key_staged(*reinterpret_cast<const uint2*>(s_stage + (size_t)r * 64 + 56), first + r) : -1;
    }
#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const bool v = key[j] >= 0;
        const unsigned m = __ballot_sync(0xffffffffu, v);
        rank[j] = 0;
        if (v) {
            const unsigned peers = __match_any_sync(m, key[j]);
            rank[j] = __popc(peers & ((1u << lane) - 1u));
            if (rank[j] == 0) s_cnt[warp * kItems + j][key[j]] = __popc(peers);
        }
    }
    __syncthreads();

    if (warp == 0) s_base[lane] = tile_bucket_base<Ops, kStageSteps>(s_cnt, lane, B, tile, hist, offsets, tileState, gen);
    __syncthreads();

#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const int r = wbase + j * 32 + lane;
        s_dst[r] = key[j] >= 0 ? (((uint32_t)key[j] << 27) | (uint32_t)(s_base[key[j]] + s_cnt[warp * kItems + j][key[j]] + rank[j])) : 0xffffffffu;
    }
    __syncwarp();                                                  // a warp scatters the records it ranked
    // scatter: four lanes per record, eight records per instruction
    const int sub = lane >> 2, part = lane & 3;
#pragma unroll 4
    for (int it = 0; it < (32 * kItems) / 8; it++) {
        const int r = wbase + it * 8 + sub;
        const uint32_t d = s_dst[r];
        if (d != 0xffffffffu) {
            const uint4 v = *reinterpret_cast<const uint4*>(s_stage + (size_t)r * 64 + part * 16);
            reinterpret_cast<uint4*>(s_ptr[d >> 27] + (d & 0x7ffffffu))[part] = v;
        }
    }
}

__global__ void path_hist_kernel(const dprt_path_record* __restrict__ paths, int n, int W, int32_t* hist) {
    __shared__ int sh[32];
    if (threadIdx.x < 32) sh[threadIdx.x] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint4 w = reinterpret_cast<const uint4*>(paths + i)[3];
        const int target = (int)w.z;
        if (((w.w >> 16) & 0xffu) && target >= 0 && target < W) atomicAdd(&sh[target], 1);
    }
    __syncthreads();
    if (threadIdx.x < W && sh[threadIdx.x]) atomicAdd(hist + threadIdx.x, sh[threadIdx.x]);
}

__global__ void query_hist_kernel(const dprt_nn_query* __restrict__ q, int n, int S, int insideOnly, int32_t* hist) {
    __shared__ int sh[32];
    if (threadIdx.x < 32) sh[threadIdx.x] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int id = q[i].hitAABBID;
        if (id >= 1 && id <= S && (!insideOnly || q[i].isInside)) atomicAdd(&sh[id - 1], 1);
    }
    __syncthreads();
    if (threadIdx.x < S && sh[threadIdx.x]) atomicAdd(hist + threadIdx.x, sh[threadIdx.x]);
}

__global__ void empty_offsets_kernel(int32_t* offsets, int B) {
    if (threadIdx.x <= B) offsets[threadIdx.x] = 0;
}

template <class Ops, int kItems>
void run_partition(Ops ops, int n, const int32_t* hist, int32_t* offsets, PartitionScratch& s, cudaStream_t stream) {
    if (n <= 0) { if (!Ops::kDirect) empty_offsets_kernel<<<1, 64, 0, stream>>>(offsets, ops.B); return; }
    constexpr int kTile = kThreads * kItems;
    const int tiles = (n + kTile - 1) / kTile;                 // <= PartitionScratch::maxTiles, which is sized for 1024-record tiles
    s.generation++;
    partition_kernel<Ops, kItems><<<tiles, kThreads, 0, stream>>>(ops, n, hist, offsets, s.tileState, s.tileCounter, s.tickets, s.generation);
    s.tickets += (uint32_t)tiles;                              // every block takes exactly one ticket
}

}  // namespace

void launch_path_histogram(const dprt_path_record* paths, int n, int W, int32_t* hist, cudaStream_t stream) {
    cudaMemsetAsync(hist, 0, 32 * sizeof(int32_t), stream);
    if (n > 0) path_hist_kernel<<<std::min((n + 255) / 256, 148 * 8), 256, 0, stream>>>(paths, n, W, hist);
}

// DPRT_PARTITION_STAGED=1 selects the TMA-staged kernel for the path records. Off by default on the numbers
// (profiles/ab_r2_partition_staged.txt): the kernel itself is 11 % faster (reorder 0.27 -> 0.31 of the HBM roofline), but
// its 64 KiB of shared memory per CTA displace the trace kernels of the other samples in flight (different shared-memory
// carve-out: the SMs have to drain), and the step gets 5 % slower. Read on every launch, so that it can be switched within
// one process.
bool partition_staged() { const char* e = getenv("DPRT_PARTITION_STAGED"); return e && e[0] == '1'; }

template <class Ops>
void run_partition_staged(Ops ops, int n, const int32_t* hist, int32_t* offsets, PartitionScratch& s, cudaStream_t stream) {
    if (n <= 0) { if (!Ops::kDirect) empty_offsets_kernel<<<1, 64, 0, stream>>>(offsets, ops.B); return; }
    static bool once = [] { cudaFuncSetAttribute(partition_staged_kernel<Ops>, cudaFuncAttributeMaxDynamicSharedMemorySize, kStageTile * 64); return true; }();
    (void)once;
    const int tiles = (n + kStageTile - 1) / kStageTile;
    s.generation++;
    partition_staged_kernel<Ops><<<tiles, kThreads, kStageTile * 64, stream>>>(ops, n, hist, offsets, s.tileState, s.tileCounter, s.tickets, s.generation);
    s.tickets += (uint32_t)tiles;
}

void launch_partition_paths(const dprt_path_record* paths, int n, int W, int B, int me, int splitL, const int32_t* hist,
                            dprt_path_record* out, int32_t* offsets, PartitionScratch& s, cudaStream_t stream) {
    PathOps ops{paths, out, B, W, B > W ? me : -1, splitL};
    if (partition_staged()) run_partition_staged<PathOps>(ops, n, hist, offsets, s, stream);
    else run_partition<PathOps, 4>(ops, n, hist, offsets, s, stream);
}

void launch_partition_paths_peer(const dprt_path_record* paths, int n, int W, int me, int splitL, const P2PPlan* plan,
                                 PartitionScratch& s, cudaStream_t stream) {
    PeerPathOps ops{paths, plan, W + 1, W, me, splitL};
    if (partition_staged()) run_partition_staged<PeerPathOps>(ops, n, nullptr, nullptr, s, stream);
    else run_partition<PeerPathOps, 4>(ops, n, nullptr, nullptr, s, stream);
}

cudaError_t partition_preload_kernels() {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, partition_kernel<PeerPathOps, 4>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, partition_kernel<PathOps, 4>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, partition_staged_kernel<PeerPathOps>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, partition_staged_kernel<PathOps>);
    return e;
}

void launch_query_histogram(const dprt_nn_query* q, int n, int S, int insideOnly, int32_t* hist, cudaStream_t stream) {
    cudaMemsetAsync(hist, 0, 32 * sizeof(int32_t), stream);
    if (n > 0) query_hist_kernel<<<std::min((n + 255) / 256, 148 * 8), 256, 0, stream>>>(q, n, S, insideOnly, hist);
}

void launch_partition_queries(const dprt_nn_query* q, const uint8_t* keys, const dprt_half* in, int n, int S, int insideOnly,
                              const int32_t* hist, dprt_nn_query* outQ, dprt_half* outIn, int32_t* offsets,
                              PartitionScratch& s, cudaStream_t stream) {
    QueryOps ops{q, keys, in, outQ, outIn, S, insideOnly};
    if (keys) run_partition<QueryOps, 16>(ops, n, hist, offsets, s, stream);
    else run_partition<QueryOps, 4>(ops, n, hist, offsets, s, stream);
}

}  // namespace dprt
