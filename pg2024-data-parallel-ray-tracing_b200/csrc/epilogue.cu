// epilogue.cu -- proxy-prediction post-processing kernels (sm_100a).
//
//   shadow_occlusion_kernel <- shadowOcclusionFloatTypeKernel  src/cuda/frame_buffer_update.cu:31-72
//   contribution_kernel     <- contributionKernelFloatType     :95-127
//   depth_update_kernel     <- predDepthUpdateKernel           :172-192
//   tmax_kernel             <- tMaxFloatTypeKernel             :222-257
//   target_node_kernel      <- targetNodeKernelFloatType       :259-324
//   image_average_kernel    <- the CPU loop at src/render/renderer.cpp:2031-2043
// All are HBM-bound streaming kernels; grid-stride, one launch each, no device-wide syncs.
#include <algorithm>
#include "dprt_internal.cuh"
#include "dprt_math.cuh"

namespace dprt {

namespace {

constexpr int kBlock = 256;
inline int grid_for(int64_t n) { return (int)std::min<int64_t>((n + kBlock - 1) / kBlock, 148 * 16); }

__global__ void shadow_occlusion_kernel(DevParams p, int size) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < size; i += gridDim.x * blockDim.x) {
        const dprt_nn_query q = p.nnPackedQuery[i];
        if (!q.isValid) continue;
        const size_t slot = (size_t)q.pixelIndex * p.spc + q.shadowPathID;
        p.contribution[slot * 3 + 0] = q.throughput[0];
        p.contribution[slot * 3 + 1] = q.throughput[1];
        p.contribution[slot * 3 + 2] = q.throughput[2];
        const float pv = f16_bits_to_f32(p.pred[i]);
        float flag = pv > 0.5f ? 1.0f : 0.0f;
        if (q.isInside && pv > 0.5f) flag = q.normalizedT;
        p.occlusion[slot * p.mc + q.hitSequence] = flag;
    }
}

// NN = false (proxies off): occlusion and contribution are never written and stay all-zero, so their terms are
// computed from literal zeros (same arithmetic, same bits) instead of being read.
// live != null: the fold runs over the pixels of the paths MainRay just shaded. For any other pixel the shadow planes
// and the contribution terms are +0, and d + (+0) leaves d unchanged bit for bit (d is a sum of non-negative terms
// that starts at +0, so it is never -0): skipping those pixels gives the reference's result.
template <bool NN>
__global__ void contribution_kernel(DevParams p, const int32_t* __restrict__ live, int count) {
    const int N = p.frameBufferSize, spc = p.spc, mc = p.mc;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const int px = live ? live[i] : i;
        if (px < 0) continue;
        float d0 = p.direct[(size_t)px * 3 + 0], d1 = p.direct[(size_t)px * 3 + 1], d2 = p.direct[(size_t)px * 3 + 2];
        for (int s = 0; s < spc; s++) {
            const size_t slot = (size_t)px * spc + s;
            float maxOcc = 0.0f;
            if (NN) for (int j = 0; j < mc; j++) { const float o = p.occlusion[slot * mc + j]; maxOcc = maxOcc > o ? maxOcc : o; }
            const float w = 1.0f - maxOcc;
            const float c0 = NN ? p.contribution[slot * 3 + 0] : 0.0f, c1 = NN ? p.contribution[slot * 3 + 1] : 0.0f,
                        c2 = NN ? p.contribution[slot * 3 + 2] : 0.0f;
            d0 += c0 * w / (float)spc;
            d1 += c1 * w / (float)spc;
            d2 += c2 * w / (float)spc;
        }
        for (int s = 1; s < spc; s++) {
            const size_t pl = ((size_t)N * s + px) * 3;
            d0 += p.direct[pl + 0]; d1 += p.direct[pl + 1]; d2 += p.direct[pl + 2];
        }
        p.direct[(size_t)px * 3 + 0] = d0; p.direct[(size_t)px * 3 + 1] = d1; p.direct[(size_t)px * 3 + 2] = d2;
    }
}

__global__ void reset_planes_kernel(DevParams p, const int32_t* __restrict__ live, int count, int nn) {
    const int N = p.frameBufferSize;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const int px = live[i];
        if (px < 0) continue;
        for (int s = 1; s < p.spc; s++) {
            const size_t pl = ((size_t)N * s + px) * 3;
            p.direct[pl + 0] = 0.0f; p.direct[pl + 1] = 0.0f; p.direct[pl + 2] = 0.0f;
        }
        if (nn) {
            float* oc = p.occlusion + (size_t)px * p.spc * p.mc;
            for (int k = 0; k < p.spc * p.mc; k++) oc[k] = 0.0f;
            float* co = p.contribution + (size_t)px * p.spc * 3;
            for (int k = 0; k < p.spc * 3; k++) co[k] = 0.0f;
        }
    }
}

__global__ void reset_sec_kernel(DevParams p, const int32_t* __restrict__ live, int count) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const int px = live[i];
        if (px < 0) continue;
        float* oc = p.occlusion + (size_t)px * p.mc * 2;
        for (int k = 0; k < p.mc * 2; k++) oc[k] = 0.0f;
    }
}

__global__ void depth_update_kernel(DevParams p, int size) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < size; i += gridDim.x * blockDim.x) {
        const dprt_nn_query q = p.nnPackedQuery[i];
        p.nnQuery[q.pathIndex].normalizedT = f16_bits_to_f32(p.pred[i]) > q.normalizedT ? 0.0f : 1.0f;
    }
}

__global__ void tmax_kernel(DevParams p, int size) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < size; i += gridDim.x * blockDim.x) {
        const dprt_nn_query q = p.nnPackedQuery[i];
        if (!q.isValid) continue;
        const size_t ti = ((size_t)q.pixelIndex * p.mc + q.hitSequence) * 2;
        float v = 0.0f;
        if (f16_bits_to_f32(p.pred[i]) > 0.5f) {
            const float predMax = q.throughput[2] * q.throughput[1] * f16_bits_to_f32(p.pred[(size_t)i + size]);
            const float aabbMax = q.throughput[0];
            if (q.isInside) v = predMax > aabbMax ? 0.0f : (aabbMax - predMax);
            else v = aabbMax + predMax;
        }
        p.occlusion[ti] = v;
        p.occlusion[ti + 1] = (float)q.pathIndex;
    }
}

__global__ void target_node_kernel(DevParams p, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        dprt_path_record* rec = p.paths + i;
        if (!rec->isValid) { if (p.secLive) p.secLive[i] = -1; continue; }
        float tMax = rec->tMax; int currentNode = rec->currentNode;
        const int pixel = rec->pixelIndex;
        if (p.secLive) p.secLive[i] = pixel;
        for (int j = 0; j < p.mc; j++) {
            const size_t ti = ((size_t)pixel * p.mc + j) * 2;
            const float t = p.occlusion[ti];
            if (t < FLT_EPSILON) continue;
            if (tMax > t) { tMax = t; currentNode = (int)p.occlusion[ti + 1]; }
        }
        if (currentNode >= 0) {
            rec->currentNode = currentNode; rec->targetNode = currentNode; rec->isHit = 1; rec->tMax = tMax;
        } else {
            rec->targetNode = p.worldID; rec->tMax = 0.0f; rec->isHit = 0; rec->isValid = 1;
        }
    }
}

__global__ void image_average_kernel(const float* __restrict__ direct, const float* __restrict__ env, float* __restrict__ out,
                                     int n3, float spp) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += gridDim.x * blockDim.x)
        out[i] = (direct[i] + env[i]) / spp;
}

__global__ void aov_average_kernel(const float* __restrict__ sum, float* __restrict__ out, int n3, float spp) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += gridDim.x * blockDim.x) out[i] = sum[i] / spp;
}

}  // namespace

void launch_shadow_occlusion(const DevParams& p, int size, cudaStream_t s) {
    if (size > 0) shadow_occlusion_kernel<<<grid_for(size), kBlock, 0, s>>>(p, size);
}
void launch_contribution(const DevParams& p, const int32_t* live, int liveCount, cudaStream_t s) {
    const int count = live ? liveCount : p.frameBufferSize;
    if (count <= 0) return;
    if (p.proxyMode) contribution_kernel<true><<<grid_for(count), kBlock, 0, s>>>(p, live, count);
    else contribution_kernel<false><<<grid_for(count), kBlock, 0, s>>>(p, live, count);
}
void launch_reset_planes(const DevParams& p, const int32_t* live, int liveCount, int nn, cudaStream_t s) {
    if (liveCount > 0 && (p.spc > 1 || nn)) reset_planes_kernel<<<grid_for(liveCount), kBlock, 0, s>>>(p, live, liveCount, nn);
}
void launch_reset_sec(const DevParams& p, const int32_t* live, int liveCount, cudaStream_t s) {
    if (liveCount > 0) reset_sec_kernel<<<grid_for(liveCount), kBlock, 0, s>>>(p, live, liveCount);
}
void launch_depth_update(const DevParams& p, int size, cudaStream_t s) {
    if (size > 0) depth_update_kernel<<<grid_for(size), kBlock, 0, s>>>(p, size);
}
void launch_tmax(const DevParams& p, int size, cudaStream_t s) {
    if (size > 0) tmax_kernel<<<grid_for(size), kBlock, 0, s>>>(p, size);
}
void launch_target_node(const DevParams& p, int n, cudaStream_t s) {
    if (n > 0) target_node_kernel<<<grid_for(n), kBlock, 0, s>>>(p, n);
}
// samples in flight: the accumulators of a second context of the same rank are added into the first one's
__global__ void accumulate_kernel(float* __restrict__ direct, float* __restrict__ env, const float* __restrict__ direct2,
                                  const float* __restrict__ env2, int n3) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += gridDim.x * blockDim.x) {
        direct[i] += direct2[i];
        env[i] += env2[i];
    }
}
void launch_accumulate(float* direct, float* env, const float* direct2, const float* env2, int n3, cudaStream_t s) {
    if (n3 > 0) accumulate_kernel<<<std::min(grid_for(n3), 148 * 16), kBlock, 0, s>>>(direct, env, direct2, env2, n3);
}
void launch_image_average(const float* direct, const float* env, float* out, int n3, float spp, cudaStream_t s) {
    if (n3 > 0) image_average_kernel<<<grid_for(n3), kBlock, 0, s>>>(direct, env, out, n3, spp);
}
void launch_aov_average(const float* sum, float* out, int n3, float spp, cudaStream_t s) {
    if (n3 > 0) aov_average_kernel<<<grid_for(n3), kBlock, 0, s>>>(sum, out, n3, spp);
}

}  // namespace dprt
