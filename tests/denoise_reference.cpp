// CPU reference of the denoiser (DESIGN.md 3.8), restated from the specification in plain C++ for the tests. It shares no
// source with the product: det_exp_neg carries its own copy of the coefficients, and the image is held planar, one float
// array per channel, instead of the product's packed layout. Built with the oracle's flags (-ffp-contract=off, hardware fmaf):
// every operation below is one binary32 add, mul, div or fma in the order the specification gives.
#include <cmath>
#include <cstdint>
#include <vector>

namespace {

float exp_neg(float x) {
    if (!(x < 88.0f)) return 0.0f;
    const float n = std::floor(std::fma(x, 1.44269504088896341f, 0.5f));      // nearest integer to x / ln 2
    const float r = (x + n * -0.693359375f) - n * -2.12194440e-4f;             // x - n ln 2 (two-part ln 2)
    const float y = -r;                                                        // e^-x = 2^-n e^y
    const float y2 = y * y;
    float p = 1.9875691500e-4f;
    p = std::fma(p, y, 1.3981999507e-3f);
    p = std::fma(p, y, 8.3334519073e-3f);
    p = std::fma(p, y, 4.1665795894e-2f);
    p = std::fma(p, y, 1.6666665459e-1f);
    p = std::fma(p, y, 5.0000001201e-1f);
    const float ey = std::fma(p, y2, y) + 1.0f;
    return std::ldexp(ey, -static_cast<int>(n));
}

const float kH[3] = {0.375f, 0.25f, 0.0625f};

}  // namespace

extern "C" {

void ref_exp_neg(const float* x, int64_t n, float* out) {
    for (int64_t i = 0; i < n; i++) out[i] = exp_neg(x[i]);
}

// color / albedo / normal / out: [H][W][3]. Returns 0; the caller validates the parameters.
int ref_denoise(int iterations, float sigma_color, float sigma_normal, float sigma_albedo, int W, int H, const float* color,
                const float* albedo, const float* normal, float* out) {
    const int64_t N = (int64_t)W * H;
    std::vector<float> a[3], nrm[3], e[3], next[3];
    for (int k = 0; k < 3; k++) {
        a[k].resize(N); nrm[k].resize(N); e[k].resize(N); next[k].resize(N);
        for (int64_t p = 0; p < N; p++) {
            a[k][p] = albedo[3 * p + k];
            nrm[k][p] = normal[3 * p + k];
            const float c = color[3 * p + k];
            e[k][p] = a[k][p] > 0.0f ? c / a[k][p] : c;
        }
    }
    const float kn = 1.0f / (sigma_normal * sigma_normal);
    const float ka = 1.0f / (sigma_albedo * sigma_albedo);
    for (int i = 0; i < iterations; i++) {
        const int step = 1 << i;
        const float kc = std::ldexp(1.0f / (sigma_color * sigma_color), 2 * i);
#pragma omp parallel for schedule(dynamic, 4)
        for (int y = 0; y < H; y++) {
            for (int x = 0; x < W; x++) {
                const int64_t p = (int64_t)y * W + x;
                float wsum = 0.0f, esum[3] = {0.0f, 0.0f, 0.0f};
                for (int dy = -2; dy <= 2; dy++) {
                    for (int dx = -2; dx <= 2; dx++) {
                        const int qx = x + step * dx, qy = y + step * dy;
                        if (qx < 0 || qy < 0 || qx >= W || qy >= H) continue;
                        const int64_t q = (int64_t)qy * W + qx;
                        float d[3] = {0.0f, 0.0f, 0.0f};          // colour, normal, albedo distances
                        for (int k = 0; k < 3; k++) {
                            const float dc = e[k][p] - e[k][q], dn = nrm[k][p] - nrm[k][q], da = a[k][p] - a[k][q];
                            d[0] = k == 0 ? dc * dc : d[0] + dc * dc;
                            d[1] = k == 0 ? dn * dn : d[1] + dn * dn;
                            d[2] = k == 0 ? da * da : d[2] + da * da;
                        }
                        const float arg = (d[0] * kc + d[1] * kn) + d[2] * ka;
                        const float w = (kH[dx < 0 ? -dx : dx] * kH[dy < 0 ? -dy : dy]) * exp_neg(arg);
                        wsum = wsum + w;
                        for (int k = 0; k < 3; k++) esum[k] = esum[k] + w * e[k][q];
                    }
                }
                for (int k = 0; k < 3; k++) next[k][p] = esum[k] / wsum;
            }
        }
        for (int k = 0; k < 3; k++) e[k].swap(next[k]);
    }
    for (int64_t p = 0; p < N; p++)
        for (int k = 0; k < 3; k++) out[3 * p + k] = a[k][p] > 0.0f ? e[k][p] * a[k][p] : e[k][p];
    return 0;
}

}  // extern "C"
