// denoise.cu -- edge-avoiding a-trous wavelet denoiser (Dammertz et al. 2010) on albedo-demodulated colour, guided by the
// first-hit albedo and normal (DESIGN.md 3.8 is the arithmetic specification). Compiled with --fmad=false on the device and
// -ffp-contract=off on the host: dprt_denoise[_device] and dprt_spec_denoise run the same DPRT_HD functions and agree bit
// for bit; tests/denoise_reference.cpp restates the specification independently.
//
// One call = one pack launch (guides packed, colour demodulated) + one launch per iteration (the last one remodulates into
// the output), all on one stream. Per pixel the scratch holds the demodulated colour twice (ping-pong, float4 each) and the
// guides as one float4 {a0, a1, a2, n0} + one float2 {n1, n2}: a tap costs three vector loads.
#include <cmath>
#include <vector>

#include "dprt_internal.cuh"

namespace dprt {
namespace {

constexpr int kTileX = 32, kTileY = 8;     // one block: 32 x 8 pixels, a warp per row of the tile

struct DenoiseK { float kc, kn, ka; };

// the weight constants of iteration i, in binary32: Kc_i = ldexp(1 / (sc sc), 2 i), Kn = 1 / (sn sn), Ka = 1 / (sa sa)
DenoiseK denoise_constants(const dprt_denoise_params& p, int i) {
    DenoiseK k;
    k.kc = std::ldexp(1.0f / (p.sigma_color * p.sigma_color), 2 * i);
    k.kn = 1.0f / (p.sigma_normal * p.sigma_normal);
    k.ka = 1.0f / (p.sigma_albedo * p.sigma_albedo);
    return k;
}

DPRT_HD float demodulate(float c, float a) { return a > 0.0f ? c / a : c; }
DPRT_HD float remodulate(float e, float a) { return a > 0.0f ? e * a : e; }

#ifdef __CUDA_ARCH__
#define DN_LD(p) __ldg(p)
#define DN_UNROLL _Pragma("unroll")
#else
#define DN_LD(p) (*(p))
#define DN_UNROLL
#endif

// Pixel p, colour c, albedo a, normal n -> e (demodulated colour, w unused) and the packed guides.
DPRT_HD void denoise_pack_pixel(const float* c, const float* a, const float* n, int64_t p, float4* e, float4* g0, float2* g1) {
    const float a0 = a[3 * p], a1 = a[3 * p + 1], a2 = a[3 * p + 2];
    e[p] = make_float4(demodulate(c[3 * p], a0), demodulate(c[3 * p + 1], a1), demodulate(c[3 * p + 2], a2), 0.0f);
    g0[p] = make_float4(a0, a1, a2, n[3 * p]);
    g1[p] = make_float2(n[3 * p + 1], n[3 * p + 2]);
}

// One iteration at pixel (x, y) with step s: taps dy = -2..2 (outer), dx = -2..2 (inner) at (x + s dx, y + s dy); taps outside
// the image are skipped. Returns sum(w e_q) / sum(w) per channel.
DPRT_HD float4 atrous_pixel(const float4* __restrict__ e, const float4* __restrict__ g0, const float2* __restrict__ g1, int W, int H,
                            int x, int y, int s, float kc, float kn, float ka) {
    const int p = y * W + x;
    const float4 ep = DN_LD(e + p), gp = DN_LD(g0 + p);
    const float2 hp = DN_LD(g1 + p);
    float sw = 0.0f, s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
    DN_UNROLL
    for (int dy = -2; dy <= 2; dy++) {
        const int qy = y + s * dy;
        if (qy < 0 || qy >= H) continue;
        const float hy = dy == 0 ? 0.375f : (dy == 1 || dy == -1 ? 0.25f : 0.0625f);
        DN_UNROLL
        for (int dx = -2; dx <= 2; dx++) {
            const int qx = x + s * dx;
            if (qx < 0 || qx >= W) continue;
            const float hx = dx == 0 ? 0.375f : (dx == 1 || dx == -1 ? 0.25f : 0.0625f);
            const int q = qy * W + qx;
            const float4 eq = DN_LD(e + q), gq = DN_LD(g0 + q);
            const float2 hq = DN_LD(g1 + q);
            const float c0 = ep.x - eq.x, c1 = ep.y - eq.y, c2 = ep.z - eq.z;
            const float n0 = gp.w - gq.w, n1 = hp.x - hq.x, n2 = hp.y - hq.y;
            const float a0 = gp.x - gq.x, a1 = gp.y - gq.y, a2 = gp.z - gq.z;
            const float dc = (c0 * c0 + c1 * c1) + c2 * c2;
            const float dn = (n0 * n0 + n1 * n1) + n2 * n2;
            const float da = (a0 * a0 + a1 * a1) + a2 * a2;
            const float w = (hx * hy) * det_exp_neg((dc * kc + dn * kn) + da * ka);
            sw = sw + w;
            s0 = s0 + w * eq.x; s1 = s1 + w * eq.y; s2 = s2 + w * eq.z;
        }
    }
    return make_float4(s0 / sw, s1 / sw, s2 / sw, 0.0f);
}

__global__ void __launch_bounds__(256) denoise_pack_kernel(const float* __restrict__ c, const float* __restrict__ a, const float* __restrict__ n,
                                                           int64_t N, float4* __restrict__ e, float4* __restrict__ g0, float2* __restrict__ g1) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < N) denoise_pack_pixel(c, a, n, p, e, g0, g1);
}

// blocks cover the image in kTileX x kTileY tiles, numbered row-major in a 1-D grid (a tall image would exceed gridDim.y)
template <bool LAST>
__global__ void __launch_bounds__(kTileX * kTileY) denoise_atrous_kernel(const float4* __restrict__ e, const float4* __restrict__ g0,
                                                                         const float2* __restrict__ g1, int W, int H, int tilesX, int s,
                                                                         float kc, float kn, float ka, float4* __restrict__ eOut,
                                                                         float* __restrict__ out) {
    const int x = (int)(blockIdx.x % (unsigned)tilesX) * kTileX + threadIdx.x;
    const int y = (int)(blockIdx.x / (unsigned)tilesX) * kTileY + threadIdx.y;
    if (x >= W || y >= H) return;
    const float4 r = atrous_pixel(e, g0, g1, W, H, x, y, s, kc, kn, ka);
    const int64_t p = (int64_t)y * W + x;
    if (LAST) {
        const float4 g = g0[p];
        out[3 * p] = remodulate(r.x, g.x); out[3 * p + 1] = remodulate(r.y, g.y); out[3 * p + 2] = remodulate(r.z, g.z);
    } else {
        eOut[p] = r;
    }
}

struct Planes { float4* e[2]; float4* g0; float2* g1; };

Planes planes(void* base, int64_t N) {
    Planes s;
    float4* f = (float4*)base;
    s.e[0] = f; s.e[1] = f + N; s.g0 = f + 2 * N; s.g1 = (float2*)(f + 3 * N);
    return s;
}

}  // namespace

int denoise_check(const dprt_denoise_params* p, int width, int height, dprt_denoise_params* out, const char** why) {
    dprt_denoise_params d = {DPRT_DENOISE_DEFAULT_ITERATIONS, DPRT_DENOISE_DEFAULT_SIGMA_COLOR, DPRT_DENOISE_DEFAULT_SIGMA_NORMAL,
                             DPRT_DENOISE_DEFAULT_SIGMA_ALBEDO};
    if (p) d = *p;
    *why = nullptr;
    if (width < 1 || height < 1) *why = "width and height must be at least 1";
    else if ((int64_t)width * height > DPRT_DENOISE_MAX_PIXELS) *why = "more than DPRT_DENOISE_MAX_PIXELS pixels";
    else if (d.iterations < 1 || d.iterations > DPRT_DENOISE_MAX_ITERATIONS) *why = "iterations outside 1..10";
    else if (!(std::isfinite(d.sigma_color) && d.sigma_color > 0.0f) || !(std::isfinite(d.sigma_normal) && d.sigma_normal > 0.0f) ||
             !(std::isfinite(d.sigma_albedo) && d.sigma_albedo > 0.0f))
        *why = "every sigma must be finite and > 0";
    else {
        const DenoiseK k = denoise_constants(d, d.iterations - 1);
        auto ok = [](float v) { return std::isfinite(v) && v > 0.0f; };
        if (!ok(k.kc) || !ok(k.kn) || !ok(k.ka)) *why = "a sigma is so small or large that its weight constant is not finite and > 0 in binary32";
    }
    if (*why) return DPRT_ERR_INVALID;
    *out = d;
    return 0;
}

size_t denoise_scratch_bytes(int64_t pixels) { return (size_t)pixels * (3 * sizeof(float4) + sizeof(float2)); }

void launch_denoise(const dprt_denoise_params& p, int width, int height, const float* color, const float* albedo, const float* normal,
                    float* out, void* scratch, cudaStream_t stream) {
    const int64_t N = (int64_t)width * height;
    const Planes s = planes(scratch, N);
    denoise_pack_kernel<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(color, albedo, normal, N, s.e[0], s.g0, s.g1);
    const int tilesX = (width + kTileX - 1) / kTileX, tilesY = (height + kTileY - 1) / kTileY;
    const dim3 block(kTileX, kTileY);
    for (int i = 0; i < p.iterations; i++) {
        const DenoiseK k = denoise_constants(p, i);
        const float4* in = s.e[i & 1];
        if (i + 1 < p.iterations)
            denoise_atrous_kernel<false><<<(unsigned)tilesX * tilesY, block, 0, stream>>>(in, s.g0, s.g1, width, height, tilesX, 1 << i,
                                                                                           k.kc, k.kn, k.ka, s.e[(i + 1) & 1], nullptr);
        else
            denoise_atrous_kernel<true><<<(unsigned)tilesX * tilesY, block, 0, stream>>>(in, s.g0, s.g1, width, height, tilesX, 1 << i,
                                                                                          k.kc, k.kn, k.ka, nullptr, out);
    }
}

// dprt_spec_denoise: the same functions on the host, OpenMP over rows (a pixel's arithmetic does not depend on the thread)
int spec_denoise(const dprt_denoise_params& p, int width, int height, const float* color, const float* albedo, const float* normal, float* out) {
    const int64_t N = (int64_t)width * height;
    std::vector<float4> buf;
    std::vector<float2> g1;
    try { buf.resize(3 * (size_t)N); g1.resize((size_t)N); } catch (const std::bad_alloc&) { return DPRT_ERR_CAPACITY; }
    float4* e[2] = {buf.data(), buf.data() + N};
    float4* g0 = buf.data() + 2 * N;
#pragma omp parallel for schedule(static)
    for (int64_t q = 0; q < N; q++) denoise_pack_pixel(color, albedo, normal, q, e[0], g0, g1.data());
    for (int i = 0; i < p.iterations; i++) {
        const DenoiseK k = denoise_constants(p, i);
        const float4* in = e[i & 1];
        float4* nx = e[(i + 1) & 1];
        const bool last = i + 1 == p.iterations;
#pragma omp parallel for schedule(static)
        for (int y = 0; y < height; y++)
            for (int x = 0; x < width; x++) {
                const float4 r = atrous_pixel(in, g0, g1.data(), width, height, x, y, 1 << i, k.kc, k.kn, k.ka);
                const int64_t q = (int64_t)y * width + x;
                if (last) {
                    out[3 * q] = remodulate(r.x, g0[q].x); out[3 * q + 1] = remodulate(r.y, g0[q].y); out[3 * q + 2] = remodulate(r.z, g0[q].z);
                } else {
                    nx[q] = r;
                }
            }
    }
    return 0;
}

}  // namespace dprt
