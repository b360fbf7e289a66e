// conductor.cuh -- the rough-metal BSDF of bsdfType 2 (DESIGN.md 3.12): Schlick Fresnel, GGX normal distribution, Smith
// height-correlated masking-shadowing, Heitz 2018 visible-normal sampling. Explicit binary32 operations, no contraction
// (--fmad=false on the device, -ffp-contract=off on the host). Compiled for the device (shade_post_kernel) and for the host
// (dprt_spec_conductor_sample / _eval), so that a machine without a GPU compares this very source with the oracle.
// All directions are in the shading frame of the face-forwarded normal (+z).
#pragma once
#include "dprt_math.cuh"

// smallest GGX alpha: keeps D = 1/(pi alpha^2) at the peak finite in binary32 for any roughness > 0
#define DPRT_COND_ALPHA_MIN 1e-3f
// f is 0 where 2 (wi.z A(wo) + wo.z A(wi)) is below this (both cosines below about 1e-27): D / den stays finite
#define DPRT_COND_DEN_MIN 1e-30f

struct CondSample { V3 wi; V3 weight; bool valid; };

// Schlick: F0 + (1 - F0) m^5 per channel, m = 1 - clamp(c, 0, 1)
DPRT_HD V3 cond_fresnel(V3 f0, float c) {
    const float m = 1.0f - fminf(fmaxf(c, 0.0f), 1.0f);
    const float m2 = m * m;
    const float m5 = (m2 * m2) * m;
    return v3(f0.x + (1.0f - f0.x) * m5, f0.y + (1.0f - f0.y) * m5, f0.z + (1.0f - f0.z) * m5);
}
DPRT_HD float cond_alpha(float r) { return fmaxf(r * r, DPRT_COND_ALPHA_MIN); }
// A(w) = |w.z| sqrt(1 + alpha^2 tan^2) = w.z (1 + 2 Lambda(w)) for w.z > 0; finite where Lambda overflows (grazing w)
DPRT_HD float cond_smith_a(float a2, V3 w) { return sqrtf(w.z * w.z + a2 * (w.x * w.x + w.y * w.y)); }

// Next-path direction and throughput factor for roughness r (r == 0: the delta mirror). weight multiplies the throughput;
// !valid (wo.z <= 0 or wi.z <= 0 on the rough lobe) means the path ends with the all-zero record, and wi = weight = 0.
DPRT_HD CondSample cond_sample(V3 f0, float r, V3 wo, float xi1, float xi2) {
    CondSample s;
    if (r == 0.0f) { s.wi = v3(-wo.x, -wo.y, wo.z); s.weight = cond_fresnel(f0, wo.z); s.valid = true; return s; }
    s.wi = v3(0.0f, 0.0f, 0.0f); s.weight = v3(0.0f, 0.0f, 0.0f); s.valid = false;
    if (!(wo.z > 0.0f)) return s;
    const float alpha = cond_alpha(r);
    // Heitz 2018, listing 1: the hemisphere configuration of wo, a point on the projected disk, back to the ellipsoid
    const V3 vh = v3normalized(v3(alpha * wo.x, alpha * wo.y, wo.z));
    const float lensq = vh.x * vh.x + vh.y * vh.y;
    V3 t1 = v3(1.0f, 0.0f, 0.0f);
    if (lensq > 0.0f) { const float inv = 1.0f / sqrtf(lensq); t1 = v3(-vh.y * inv, vh.x * inv, 0.0f); }
    const V3 t2 = v3cross(vh, t1);
    const float rr = sqrtf(xi1);
    float sn, cs; det_sincos2pi(xi2, &sn, &cs);
    const float p1 = rr * cs;
    const float sh = 0.5f * (1.0f + vh.z);
    const float q1 = 1.0f - p1 * p1;
    const float p2 = (1.0f - sh) * sqrtf(fmaxf(0.0f, q1)) + sh * (rr * sn);
    const float pz = sqrtf(fmaxf(0.0f, q1 - p2 * p2));
    const V3 nh = v3(p1 * t1.x + p2 * t2.x + pz * vh.x, p1 * t1.y + p2 * t2.y + pz * vh.y, p1 * t1.z + p2 * t2.z + pz * vh.z);
    const V3 h = v3normalized(v3(alpha * nh.x, alpha * nh.y, fmaxf(0.0f, nh.z)));
    const float woh = v3dot(wo, h);
    const float tw = 2.0f * woh;
    const V3 wi = v3(tw * h.x - wo.x, tw * h.y - wo.y, tw * h.z - wo.z);
    if (!(wi.z > 0.0f)) return s;
    // G2 / G1 = (1 + Lambda(wo)) / (1 + Lambda(wo) + Lambda(wi)) = (wo.z + A(wo)) / (A(wo) + A(wi) wo.z / wi.z)
    const float a2 = alpha * alpha;
    const float ao = cond_smith_a(a2, wo), ai = cond_smith_a(a2, wi);
    const float g = fminf(1.0f, (wo.z + ao) / (ao + ai * (wo.z / wi.z)));
    s.wi = wi; s.weight = v3scale(cond_fresnel(f0, woh), g); s.valid = true;
    return s;
}

// f(wi, wo) = F(wi.h) D(h) G2 / (4 wo.z wi.z), h = normalize(wo + wi); 0 for the mirror (a delta: no light sample reaches it)
// and where a cosine is <= 0. G2 / (4 wo.z wi.z) = 1 / (2 (wi.z A(wo) + wo.z A(wi))) and the GGX denominator
// (alpha^2 - 1) h.z^2 + 1 = (h.x^2 + h.y^2) + alpha^2 h.z^2 (|h| = 1), which loses nothing to cancellation near h.z = 1.
DPRT_HD V3 cond_eval(V3 f0, float r, V3 wo, V3 wi) {
    const V3 zero = v3(0.0f, 0.0f, 0.0f);
    if (r == 0.0f || !(wo.z > 0.0f) || !(wi.z > 0.0f)) return zero;
    const float alpha = cond_alpha(r), a2 = alpha * alpha;
    const V3 h = v3normalized(v3add(wo, wi));
    const float k = (h.x * h.x + h.y * h.y) + a2 * (h.z * h.z);
    const float d = a2 / (3.14159265358979323846f * (k * k));
    const float den = 2.0f * (wi.z * cond_smith_a(a2, wo) + wo.z * cond_smith_a(a2, wi));
    if (!(den > DPRT_COND_DEN_MIN)) return zero;
    return v3scale(cond_fresnel(f0, v3dot(wi, h)), d / den);
}
