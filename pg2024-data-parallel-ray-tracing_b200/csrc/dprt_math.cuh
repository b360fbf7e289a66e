// dprt_math.cuh -- arithmetic specification of the hot path (device side).
//
// Every operation here is written as an explicit sequence of IEEE-754 binary32 operations
// (add, mul, fma, div, sqrt; no contraction: this translation unit is compiled with --fmad=false)
// so that the scalar oracle (oracle/oracle.cpp, built with -ffp-contract=off) reproduces it bit for bit.
// DESIGN.md "Arithmetic specification" is the normative text; both sides implement it independently.
//
// Reference sites restated: optix/random.hpp:31-67 (tea/lcg/rnd), optix/sample.hpp:7-17
// (uniformHemisphere), and the missing moana headers listed in SURVEY.md section 2.4 (Vec3, Frame,
// Camera::generateRay, Triangle::sample, Coordinates::cartesianToSpherical).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <float.h>

#define DPRT_D __device__ __forceinline__
// also compiled for the host: the texture / environment look-ups are exported as dprt_spec_* so that a machine without a GPU
// can compare this very source with the oracle
#define DPRT_HD __host__ __device__ __forceinline__

struct V3 { float x, y, z; };

DPRT_HD V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
DPRT_D V3 v3sub(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
DPRT_D V3 v3add(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
DPRT_D V3 v3mul(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
DPRT_D V3 v3scale(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
DPRT_D V3 v3neg(V3 a) { return v3(-a.x, -a.y, -a.z); }
DPRT_D float v3get(V3 a, int k) { return k == 0 ? a.x : (k == 1 ? a.y : a.z); }
// dot = fma(z,z', fma(y,y', x*x'))
DPRT_D float v3dot(V3 a, V3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
// cross component = fma(a1, b2, -(a2*b1))
DPRT_D V3 v3cross(V3 a, V3 b) {
    return v3(fmaf(a.y, b.z, -(a.z * b.y)), fmaf(a.z, b.x, -(a.x * b.z)), fmaf(a.x, b.y, -(a.y * b.x)));
}
DPRT_D float v3length(V3 a) { return sqrtf(v3dot(a, a)); }
// normalized = v * (1/length)
DPRT_D V3 v3normalized(V3 a) { float inv = 1.0f / v3length(a); return v3scale(a, inv); }
// point on ray = fma(t, d, o)
DPRT_D V3 v3at(V3 o, V3 d, float t) { return v3(fmaf(t, d.x, o.x), fmaf(t, d.y, o.y), fmaf(t, d.z, o.z)); }

// ---- RNG: optix/random.hpp:31-67 (integer arithmetic, exact) ----
DPRT_D uint32_t tea4(uint32_t val0, uint32_t val1) {
    uint32_t v0 = val0, v1 = val1, s0 = 0;
#pragma unroll
    for (int n = 0; n < 4; n++) {
        s0 += 0x9e3779b9u;
        v0 += ((v1 << 4) + 0xa341316cu) ^ (v1 + s0) ^ ((v1 >> 5) + 0xc8013ea4u);
        v1 += ((v0 << 4) + 0xad90777du) ^ (v0 + s0) ^ ((v0 >> 5) + 0x7e95761eu);
    }
    return v0;
}
DPRT_D uint32_t lcg(uint32_t& prev) { prev = 1664525u * prev + 1013904223u; return prev & 0x00FFFFFFu; }
DPRT_D float rnd(uint32_t& prev) { return (float)lcg(prev) / (float)0x01000000; }

// ---- deterministic transcendentals (spec; polynomial coefficients are the Cephes single-precision sets) ----
// sin/cos of 2*pi*x for x in [0,1).
DPRT_D void det_sincos2pi(float x, float* s, float* c) {
    float r = x * 4.0f;                    // exact
    float qf = floorf(r + 0.5f);
    float f = r - qf;                      // in [-0.5, 0.5], exact
    int q = (int)qf & 3;
    float a = f * 1.57079632679489661923f; // angle in [-pi/4, pi/4]
    float z = a * a;
    float sp = fmaf(fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f) * z, a, a);
    float cp = fmaf(fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f), z * z,
                    fmaf(-0.5f, z, 1.0f));
    float ss = (q & 1) ? cp : sp;
    float cc = (q & 1) ? sp : cp;
    if (q == 1 || q == 2) cc = -cc;
    if (q == 2 || q == 3) ss = -ss;
    *s = ss; *c = cc;
}
DPRT_HD float det_asin_poly(float x) {      // |x| <= 0.5
    float z = x * x;
    float p = fmaf(fmaf(fmaf(fmaf(4.2163199048e-2f, z, 2.4181311049e-2f), z, 4.5470025998e-2f), z, 7.4953002686e-2f), z,
                   1.6666752422e-1f);
    return fmaf(p * z, x, x);
}
DPRT_HD float det_acos(float x) {           // x clamped to [-1,1] by the caller
    const float PI = 3.14159265358979323846f, PIO2 = 1.57079632679489661923f;
    if (x > 0.5f) { float s = sqrtf(0.5f * (1.0f - x)); return 2.0f * det_asin_poly(s); }
    if (x < -0.5f) { float s = sqrtf(0.5f * (1.0f + x)); return PI - 2.0f * det_asin_poly(s); }
    return PIO2 - det_asin_poly(x);
}
DPRT_HD float det_atan_pos(float t) {       // t >= 0
    const float PIO2 = 1.57079632679489661923f, PIO4 = 0.78539816339744830962f;
    float y0, x;
    if (t > 2.414213562373095f) { y0 = PIO2; x = -(1.0f / t); }
    else if (t > 0.4142135623730950f) { y0 = PIO4; x = (t - 1.0f) / (t + 1.0f); }
    else { y0 = 0.0f; x = t; }
    float z = x * x;
    float p = fmaf(fmaf(fmaf(8.05374449538e-2f, z, -1.38776856032e-1f), z, 1.99777106478e-1f), z, -3.33329491539e-1f);
    return y0 + fmaf(p * z, x, x);
}
DPRT_HD float det_atan2(float y, float x) {
    const float PI = 3.14159265358979323846f, PIO2 = 1.57079632679489661923f;
    if (x == 0.0f) { if (y > 0.0f) return PIO2; if (y < 0.0f) return -PIO2; return 0.0f; }
    float a = det_atan_pos(fabsf(y) / fabsf(x));
    if (x < 0.0f) a = PI - a;
    return (y < 0.0f) ? -a : a;
}
// e^-x for x >= 0 (the denoiser's edge-stopping weights, DESIGN.md 3.8). x = n ln2 + r with n = floor(x log2(e) + 0.5) and
// r in about [-ln2/2, ln2/2] (Cody-Waite: ln2 = 0.693359375 - 2.12194440e-4, the first part exact in n * 0.693359375);
// e^-r from the Cephes expf polynomial, then ldexpf(., -n). Exactly 1 at 0; 0 when !(x < 88) (NaN included).
// Against exp(): relative error below 1e-7 while the result is normal (x < 87.33), below one subnormal ulp beyond; the
// result is non-increasing in x (tests/test_denoise_cpu.py checks both on a dense grid).
DPRT_HD float det_exp_neg(float x) {
    if (!(x < 88.0f)) return 0.0f;
    const float n = floorf(fmaf(x, 1.44269504088896341f, 0.5f));
    const float y = -((n * -0.693359375f + x) - n * -2.12194440e-4f);
    const float z = y * y;
    const float p = fmaf(fmaf(fmaf(fmaf(fmaf(1.9875691500e-4f, y, 1.3981999507e-3f), y, 8.3334519073e-3f), y, 4.1665795894e-2f), y,
                             1.6666665459e-1f), y, 5.0000001201e-1f);
    return ldexpf(fmaf(p, z, y) + 1.0f, -(int)n);
}
// Coordinates::cartesianToSpherical (+ForTrain, same convention: src/cuda/bvh_intersection.cu:18-26):
// phi = atan2(y,x) wrapped to [0,2pi), theta = acos(clamp(z,-1,1)).
DPRT_HD void det_cartesian_to_spherical(V3 d, float* phi, float* theta) {
    float p = det_atan2(d.y, d.x);
    if (p < 0.0f) p += 6.28318530717958647692f;
    *phi = p;
    *theta = det_acos(fminf(1.0f, fmaxf(-1.0f, d.z)));
}

// ---- Sample::uniformHemisphere: optix/sample.hpp:7-17 ----
DPRT_D V3 uniform_hemisphere(float xi1, float xi2) {
    float z = xi1;
    float r = sqrtf(fmaxf(0.0f, fmaf(-z, z, 1.0f)));
    float s, c; det_sincos2pi(xi2, &s, &c);
    return v3(r * c, r * s, z);
}

// ---- Frame(normal).toWorld: branchless orthonormal basis (Duff et al. 2017) ----
DPRT_D V3 frame_to_world(V3 n, V3 w) {
    float sign = copysignf(1.0f, n.z);
    float a = -1.0f / (sign + n.z);
    float b = n.x * n.y * a;
    V3 s = v3(fmaf(sign * n.x, n.x * a, 1.0f), sign * b, -(sign * n.x));
    V3 t = v3(b, fmaf(n.y, n.y * a, sign), -n.y);
    return v3(fmaf(n.x, w.z, fmaf(t.x, w.y, s.x * w.x)),
              fmaf(n.y, w.z, fmaf(t.y, w.y, s.y * w.x)),
              fmaf(n.z, w.z, fmaf(t.z, w.y, s.z * w.x)));
}
DPRT_D V3 frame_to_local(V3 n, V3 w) {
    float sign = copysignf(1.0f, n.z);
    float a = -1.0f / (sign + n.z);
    float b = n.x * n.y * a;
    V3 s = v3(fmaf(sign * n.x, n.x * a, 1.0f), sign * b, -(sign * n.x));
    V3 t = v3(b, fmaf(n.y, n.y * a, sign), -n.y);
    return v3(v3dot(s, w), v3dot(t, w), v3dot(n, w));
}

// ---- affine world->object (optixTransformPoint/VectorFromWorldToObjectSpace) ----
DPRT_D V3 xform_point(const float* m, V3 p) {
    return v3(fmaf(m[2], p.z, fmaf(m[1], p.y, fmaf(m[0], p.x, m[3]))),
              fmaf(m[6], p.z, fmaf(m[5], p.y, fmaf(m[4], p.x, m[7]))),
              fmaf(m[10], p.z, fmaf(m[9], p.y, fmaf(m[8], p.x, m[11]))));
}
DPRT_D V3 xform_vector(const float* m, V3 v) {
    return v3(fmaf(m[2], v.z, fmaf(m[1], v.y, m[0] * v.x)),
              fmaf(m[6], v.z, fmaf(m[5], v.y, m[4] * v.x)),
              fmaf(m[10], v.z, fmaf(m[9], v.y, m[8] * v.x)));
}

// ---- watertight ray/triangle test (Woop, Benthin, Wald 2013), replaces optixTrace's intersector ----
struct RayShear { int kx, ky, kz; float Sx, Sy, Sz; };

DPRT_D RayShear ray_shear(V3 d) {
    RayShear r;
    int kz = 0; float m = fabsf(d.x);
    if (fabsf(d.y) > m) { kz = 1; m = fabsf(d.y); }
    if (fabsf(d.z) > m) { kz = 2; }
    int kx = kz + 1; if (kx == 3) kx = 0;
    int ky = kx + 1; if (ky == 3) ky = 0;
    float dz = v3get(d, kz);
    if (dz < 0.0f) { int t = kx; kx = ky; ky = t; }
    r.kx = kx; r.ky = ky; r.kz = kz;
    r.Sx = v3get(d, kx) / dz; r.Sy = v3get(d, ky) / dz; r.Sz = 1.0f / dz;
    return r;
}

// Returns true when the triangle is hit with tmin < t < tmax; t and OptiX-style barycentrics
// (alpha = weight of v1, beta = weight of v2) are written on a hit.
DPRT_D bool tri_intersect(const RayShear& rs, V3 o, V3 p0, V3 p1, V3 p2, float tmin, float tmax,
                          float* t_out, float* alpha, float* beta) {
    V3 A = v3sub(p0, o), B = v3sub(p1, o), C = v3sub(p2, o);
    float Akz = v3get(A, rs.kz), Bkz = v3get(B, rs.kz), Ckz = v3get(C, rs.kz);
    float Ax = fmaf(-rs.Sx, Akz, v3get(A, rs.kx)), Ay = fmaf(-rs.Sy, Akz, v3get(A, rs.ky));
    float Bx = fmaf(-rs.Sx, Bkz, v3get(B, rs.kx)), By = fmaf(-rs.Sy, Bkz, v3get(B, rs.ky));
    float Cx = fmaf(-rs.Sx, Ckz, v3get(C, rs.kx)), Cy = fmaf(-rs.Sy, Ckz, v3get(C, rs.ky));
    float U = fmaf(Cx, By, -(Cy * Bx));
    float V = fmaf(Ax, Cy, -(Ay * Cx));
    float W = fmaf(Bx, Ay, -(By * Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    float det = (U + V) + W;
    if (det == 0.0f) return false;
    float Az = rs.Sz * Akz, Bz = rs.Sz * Bkz, Cz = rs.Sz * Ckz;
    float T = fmaf(U, Az, fmaf(V, Bz, W * Cz));
    float t = T / det;
    if (!(t > tmin && t < tmax)) return false;
    *t_out = t; *alpha = V / det; *beta = W / det;
    return true;
}

// ---- proxy AABB test in object space: replaces optixTrace(AS.aabbHandle) + optixIsFrontFaceHit ----
// Front-face hit (ray enters) at t_near, else back-face hit (origin inside) at t_far; tmin < t < tmax.
DPRT_D bool aabb_intersect(V3 ol, V3 dl, const float* mn, const float* mx, float tmin, float tmax,
                           float* t_out, bool* inside) {
    float ix = 1.0f / dl.x, iy = 1.0f / dl.y, iz = 1.0f / dl.z;
    float x0 = (mn[0] - ol.x) * ix, x1 = (mx[0] - ol.x) * ix;
    float y0 = (mn[1] - ol.y) * iy, y1 = (mx[1] - ol.y) * iy;
    float z0 = (mn[2] - ol.z) * iz, z1 = (mx[2] - ol.z) * iz;
    float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
    float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
    if (!(tn <= tf)) return false;
    if (tn > tmin && tn < tmax) { *t_out = tn; *inside = false; return true; }
    if (tf > tmin && tf < tmax) { *t_out = tf; *inside = true; return true; }
    return false;
}

// float -> IEEE binary16, round to nearest even (the reference's __float2half).
DPRT_D uint16_t f32_to_f16_bits(float f) { return __half_as_ushort(__float2half_rn(f)); }
DPRT_D float f16_bits_to_f32(uint16_t h) { return __half2float(__ushort_as_half(h)); }

// ---- textures: albedo / opacity maps and the environment map (real-scene front end) ----
// tex2D<float4>() of kernel.cu:274-279 / :40-44 on a cudaFilterModeLinear, normalised-coordinate texture object
// (renderer.cpp:1700-1710), as binary32 arithmetic instead of the texture unit's 9-bit fixed-point weights, so that the
// oracle reproduces it bit for bit: sample point x = u W - 0.5, texels floor(x) and floor(x) + 1, weights frac(x);
// lerp(a, b, f) = fma(f, b - a, a), first along u in both rows, then along v. u wraps; v wraps (albedo maps: both address
// modes are Wrap in the reference) or clamps (lat-long environment map: theta / pi in [0, 1]).
struct DevTexture { const float4* texels; int32_t width, height; };     // RGBA float texels, row-major, row 0 = v 0

#ifdef __CUDA_ARCH__
#define DPRT_LDG4(p) __ldg(p)
#else
#define DPRT_LDG4(p) (*(p))
#endif

struct TexTap { int i00, i10, i01, i11; float fx, fy; };

DPRT_HD TexTap tex_taps(int W, int H, float u, float v, bool clampV) {
    if (!(fabsf(u) < 1e30f)) u = 0.0f;          // NaN / inf / absurd coordinates: texel (0, 0) side of the map, never UB
    if (!(fabsf(v) < 1e30f)) v = 0.0f;
    u = u - floorf(u);
    v = clampV ? fminf(fmaxf(v, 0.0f), 1.0f) : v - floorf(v);
    const float x = fmaf(u, (float)W, -0.5f), y = fmaf(v, (float)H, -0.5f);
    const float x0f = floorf(x), y0f = floorf(y);
    TexTap t;
    t.fx = x - x0f; t.fy = y - y0f;
    int x0 = (int)x0f, y0 = (int)y0f, x1 = x0 + 1, y1 = y0 + 1;
    if (x0 < 0) x0 += W;
    if (x1 >= W) x1 -= W;
    if (clampV) { if (y0 < 0) y0 = 0; if (y1 > H - 1) y1 = H - 1; }
    else { if (y0 < 0) y0 += H; if (y1 >= H) y1 -= H; }
    t.i00 = y0 * W + x0; t.i10 = y0 * W + x1; t.i01 = y1 * W + x0; t.i11 = y1 * W + x1;
    return t;
}
DPRT_HD float tex_lerp2(float c00, float c10, float c01, float c11, float fx, float fy) {
    const float a = fmaf(fx, c10 - c00, c00), b = fmaf(fx, c11 - c01, c01);
    return fmaf(fy, b - a, a);
}
DPRT_HD float4 tex_bilinear(const DevTexture& T, float u, float v, bool clampV) {
    const TexTap t = tex_taps(T.width, T.height, u, v, clampV);
    const float4 c00 = DPRT_LDG4(T.texels + t.i00), c10 = DPRT_LDG4(T.texels + t.i10), c01 = DPRT_LDG4(T.texels + t.i01), c11 = DPRT_LDG4(T.texels + t.i11);
    float4 r;
    r.x = tex_lerp2(c00.x, c10.x, c01.x, c11.x, t.fx, t.fy);
    r.y = tex_lerp2(c00.y, c10.y, c01.y, c11.y, t.fx, t.fy);
    r.z = tex_lerp2(c00.z, c10.z, c01.z, c11.z, t.fx, t.fy);
    r.w = tex_lerp2(c00.w, c10.w, c01.w, c11.w, t.fx, t.fy);
    return r;
}
// opacity only (the any-hit program reads albedo.w, kernel.cu:349)
DPRT_HD float tex_bilinear_alpha(const DevTexture& T, float u, float v) {
    const TexTap t = tex_taps(T.width, T.height, u, v, false);
    return tex_lerp2(DPRT_LDG4(T.texels + t.i00).w, DPRT_LDG4(T.texels + t.i10).w, DPRT_LDG4(T.texels + t.i01).w, DPRT_LDG4(T.texels + t.i11).w, t.fx, t.fy);
}
// texture coordinate at barycentrics (alpha, beta) = weights of corners 1, 2 (kernel.cu:264-265): gamma t0 + alpha t1 + beta t2
DPRT_HD float tex_interp(float t0, float t1, float t2, float alpha, float beta) {
    const float gamma = 1.0f - alpha - beta;
    return fmaf(beta, t2, fmaf(alpha, t1, gamma * t0));
}
// calculateEnvironmentLighting (kernel.cu:28-48, distributed_traversal_kernel.cu:82-103): lat-long look-up of a direction
DPRT_HD float4 env_map_lookup(const DevTexture& T, float rotationOffset, V3 d) {
    float phi, theta;
    det_cartesian_to_spherical(d, &phi, &theta);
    phi += rotationOffset;
    if (phi > 6.28318530717958647692f) phi -= 6.28318530717958647692f;
    return tex_bilinear(T, phi / 6.28318530717958647692f, theta / 3.14159265358979323846f, true);
}
