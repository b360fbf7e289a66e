// plastic.cuh -- the glossy plastic of bsdfType 3 (DESIGN.md 3.13): a Lambertian base of the material's albedo under a thin
// dielectric coat of IOR 1.5, whose specular lobe is the conductor's GGX lobe (conductor.cuh) at the fixed F0 = 0.04, coupled
// to the base by (1 - F(wo.z)) (1 - F(wi.z)). Explicit binary32 operations, no contraction, compiled for the device
// (shade_post_kernel) and the host (dprt_spec_plastic_sample / _eval) like conductor.cuh. Directions are in the shading frame
// of the face-forwarded normal (+z).
#pragma once
#include "conductor.cuh"

// Schlick F0 of the coat: ((1.5 - 1) / (1.5 + 1))^2, glTF's value for dielectrics
#define DPRT_PLASTIC_F0 0.04f

DPRT_HD V3 plastic_f0() { return v3(DPRT_PLASTIC_F0, DPRT_PLASTIC_F0, DPRT_PLASTIC_F0); }
// the coat's Fresnel: one channel of cond_fresnel at F0 = 0.04 (the three are equal)
DPRT_HD float plastic_fresnel(float c) { return cond_fresnel(plastic_f0(), c).x; }
// probability of the specular lobe, ps = Fs / (Fs + (1 - Fs) y) with y = max(0, Rec. 709 luminance of the albedo): Fs >= 0.04
// keeps it > 0, and it is 1 only where y = 0, where the diffuse term is 0 too
DPRT_HD float plastic_spec_prob(V3 albedo, float fs) {
    const float y = fmaxf(0.0f, (0.2126f * albedo.x + 0.7152f * albedo.y) + 0.0722f * albedo.z);
    return fs / (fs + (1.0f - fs) * y);
}

// Next-path direction and throughput factor, stochastic lobe selection by xi3: the specular lobe with probability ps (the
// conductor's sample at F0 = 0.04, weight / ps; a delta mirror for r == 0), else the diffuse lobe sampled as Lambert samples
// it (uniform hemisphere). !valid (wo.z <= 0, or the specular lobe sampled below the surface) ends the path; wi = weight = 0.
DPRT_HD CondSample plastic_sample(V3 albedo, float r, V3 wo, float xi1, float xi2, float xi3) {
    CondSample s;
    s.wi = v3(0.0f, 0.0f, 0.0f); s.weight = v3(0.0f, 0.0f, 0.0f); s.valid = false;
    if (!(wo.z > 0.0f)) return s;
    const float fs = plastic_fresnel(wo.z);
    const float ps = plastic_spec_prob(albedo, fs);
    if (xi3 < ps) {
        s = cond_sample(plastic_f0(), r, wo, xi1, xi2);
        s.weight = v3(s.weight.x / ps, s.weight.y / ps, s.weight.z / ps);
        return s;
    }
    // xi3 >= ps, so ps < 1 and 1 - ps > 0
    const V3 wi = uniform_hemisphere(xi1, xi2);
    const float k = (((2.0f * wi.z) * (1.0f - fs)) * (1.0f - plastic_fresnel(wi.z))) / (1.0f - ps);
    s.wi = wi; s.weight = v3scale(albedo, k); s.valid = true;
    return s;
}

// f(wi, wo) = cond_eval(0.04, r, wo, wi) + albedo (1 - F(wo.z)) (1 - F(wi.z)) / pi; 0 where a cosine is <= 0. Never a delta:
// at r == 0 the specular term is 0 and the diffuse term still takes the light samples.
DPRT_HD V3 plastic_eval(V3 albedo, float r, V3 wo, V3 wi) {
    if (!(wo.z > 0.0f) || !(wi.z > 0.0f)) return v3(0.0f, 0.0f, 0.0f);
    const V3 spec = cond_eval(plastic_f0(), r, wo, wi);
    const float k = ((1.0f - plastic_fresnel(wo.z)) * (1.0f - plastic_fresnel(wi.z))) / 3.14159265358979323846f;
    return v3add(spec, v3scale(albedo, k));
}
