// plastic_reference.cpp -- CPU reference of the glossy plastic (bsdfType 3, DESIGN.md 3.13), test infrastructure
// (tests/plastic_reference.py compiles it at test time with the oracle's flags).
//
// The conductor reference (tests/conductor_reference.cpp, which carries the oracle and the AOV reference) is included
// unchanged, so worlds that mix conductors and plastics are covered. On top of it, as a restatement of its own:
//   plas_render_sample = cond_render_sample, where every shade is cond_shade (the oracle's shade() and the conductor rule)
//                        followed by the plastic rule for each record whose hit is a bsdfType 3 material: its next record and
//                        its spc shadow slots are recomputed from the record as it was before the shade (same re-trace, albedo
//                        / texel, face-forwarded normal and random numbers, plus a third uniform of the same sequence);
//   plas_sample / plas_eval = the BSDF on its own, for the host compile of plastic.cuh.
// The roughness table is the conductor reference's (cond_set_roughness): the product has one table for both materials.
// Same binary32 operations in the same order as the specification, so every record is comparable bit for bit.
#include "conductor_reference.cpp"

namespace {

// the coat's Schlick Fresnel at F0 = 0.04: 0.04 + (1 - 0.04) m^5, m = 1 - clamp(c, 0, 1)
float coat_fresnel(float c) { return schlick(v3(0.04f, 0.04f, 0.04f), c).x; }
// probability of the specular lobe: Fs / (Fs + (1 - Fs) max(0, Y)), Y the Rec. 709 luminance of the diffuse colour
float spec_probability(V3 kd, float fs) {
    const float lum = (0.2126f * kd.x + 0.7152f * kd.y) + 0.0722f * kd.z;
    const float y = fmaxf(0.0f, lum);
    return fs / (fs + (1.0f - fs) * y);
}
CondOut plastic_sample(V3 kd, float r, V3 wo, float u1, float u2, float u3) {
    CondOut o{v3(0, 0, 0), v3(0, 0, 0), false};
    if (!(wo.z > 0.0f)) return o;
    const float fs = coat_fresnel(wo.z);
    const float ps = spec_probability(kd, fs);
    if (u3 < ps) {                                    // specular: the conductor's lobe at F0 = 0.04, over its probability
        o = conductor_sample(v3(0.04f, 0.04f, 0.04f), r, wo, u1, u2);
        o.weight = v3(o.weight.x / ps, o.weight.y / ps, o.weight.z / ps);
        return o;
    }
    const V3 wi = uniform_hemisphere(u1, u2);         // diffuse: Lambert's sampler, over its probability 1 - ps
    const float w = 2.0f * wi.z;
    const float t = w * (1.0f - fs);
    const float k = (t * (1.0f - coat_fresnel(wi.z))) / (1.0f - ps);
    o.wi = wi; o.weight = scale(kd, k); o.valid = true;
    return o;
}
V3 plastic_eval(V3 kd, float r, V3 wo, V3 wi) {
    if (!(wo.z > 0.0f) || !(wi.z > 0.0f)) return v3(0, 0, 0);
    const V3 s = conductor_eval(v3(0.04f, 0.04f, 0.04f), r, wo, wi);
    const float a = 1.0f - coat_fresnel(wo.z), b = 1.0f - coat_fresnel(wi.z);
    const float k = (a * b) / 3.14159265358979323846f;
    return v3(s.x + kd.x * k, s.y + kd.y * k, s.z + kd.z * k);
}

// the closest-hit program's tail for a plastic: the next path from plastic_sample, the spc light samples with plastic_eval in
// place of albedo / pi (never a delta: the diffuse base takes light at any roughness); light choice and point are shade()'s
void shade_plastic(World& w, Rank& r, int i, const dprt_path_record& path, V3 point, V3 normal, V3 woWorld, V3 kd, float rough,
                   float xi1, float xi2, float xi3) {
    const int n = r.pathSize, spc = w.cfg.shadowPathCount;
    const Frame fr = make_frame(normal);
    const V3 wo = to_local(fr, woWorld);
    const V3 thr = v3(path.throughput[0], path.throughput[1], path.throughput[2]);
    const CondOut ps = plastic_sample(kd, rough, wo, xi1, xi2, xi3);
    dprt_path_record next{};
    if (ps.valid) {
        const V3 nd = normalized(to_world(fr, ps.wi));
        const V3 t = mul(thr, ps.weight);
        next.origin[0] = point.x; next.origin[1] = point.y; next.origin[2] = point.z;
        next.direction[0] = nd.x; next.direction[1] = nd.y; next.direction[2] = nd.z;
        next.tMax = FLT_MAX;
        next.throughput[0] = t.x; next.throughput[1] = t.y; next.throughput[2] = t.z;
        next.pixelIndex = path.pixelIndex; next.shadowPathID = -1; next.visitedMask = 0; next.currentNode = -1; next.targetNode = -1;
        next.isValid = 1;
    }
    r.paths[i] = next;
    for (int s = 0; s < spc; s++) {
        dprt_path_record& slot = r.paths[(size_t)i * spc + s + n];
        slot = dprt_path_record{};
        uint32_t sseed = tea4((uint32_t)(path.pixelIndex * spc + s), (uint32_t)w.sample);
        const float x1 = rnd(sseed), x2 = rnd(sseed), x3 = rnd(sseed);
        const int li = (int)floorf(x1 * (float)w.lights.size());
        const dprt_light_tri& L = w.lights[li];
        const V3 p0 = v3(L.p0[0], L.p0[1], L.p0[2]), p1 = v3(L.p1[0], L.p1[1], L.p1[2]), p2 = v3(L.p2[0], L.p2[1], L.p2[2]);
        const float su = sqrtf(x2);
        const float b0 = 1.0f - su, b1 = x3 * su, b2 = 1.0f - b0 - b1;
        const V3 lp = v3(fmaf(b2, p2.x, fmaf(b1, p1.x, b0 * p0.x)), fmaf(b2, p2.y, fmaf(b1, p1.y, b0 * p0.y)),
                         fmaf(b2, p2.z, fmaf(b1, p1.z, b0 * p0.z)));
        const V3 cr = cross(sub(p1, p0), sub(p2, p0));
        const float crl = length(cr);
        const V3 ln = scale(cr, 1.0f / crl);
        const float areaPDF = (1.0f / (0.5f * crl)) * (1.0f / (float)w.lights.size());
        const V3 ldir = sub(lp, point);
        const V3 wi = normalized(ldir);
        const float stMax = length(ldir);
        const float f1 = fmaxf(0.0f, dot(ln, neg(wi)));
        const float f2 = fmaxf(0.0f, dot(wi, normal));
        const V3 f = plastic_eval(kd, rough, wo, to_local(fr, wi));
        V3 c = mul(mul(v3(L.Le[0], L.Le[1], L.Le[2]), thr), f);
        c = scale(scale(c, f1), f2);
        const float tt = stMax * stMax;
        c = v3(c.x / areaPDF / tt, c.y / areaPDF / tt, c.z / areaPDF / tt);
        slot.origin[0] = point.x; slot.origin[1] = point.y; slot.origin[2] = point.z;
        slot.direction[0] = wi.x; slot.direction[1] = wi.y; slot.direction[2] = wi.z;
        slot.tMax = stMax; slot.throughput[0] = c.x; slot.throughput[1] = c.y; slot.throughput[2] = c.z;
        slot.pixelIndex = path.pixelIndex; slot.shadowPathID = s; slot.visitedMask = 0; slot.currentNode = -1; slot.targetNode = -1;
        slot.isShadowRay = 1; slot.isValid = 1;
    }
}

// cond_shade (the oracle's shade() and the conductor rule), then the plastic rule for every record whose closest hit on this
// rank is a bsdfType 3 material
void plas_shade(World& w, Rank& r, const std::vector<float>* rough) {
    const int n = r.pathSize;
    const std::vector<dprt_path_record> in(r.paths.begin(), r.paths.begin() + n);
    cond_shade(w, r, rough);
#pragma omp parallel for schedule(dynamic, 256)
    for (int i = 0; i < n; i++) {
        const dprt_path_record& path = in[i];
        if (!path.isValid) continue;
        const V3 o = v3(path.origin[0], path.origin[1], path.origin[2]), d = v3(path.direction[0], path.direction[1], path.direction[2]);
        Hit h{}; int hobj = -1; float tMax = FLT_MAX;
        if (!trace_local(w, r.id, o, d, DPRT_EPSILON, tMax, 0u, false, h, hobj)) continue;
        const Object& ob = w.objects[hobj];
        const int matID = ob.mesh.mats[h.prim];
        const dprt_material mat = w.materials[matID];
        if (mat.bsdfType != 3) continue;
        V3 kd = v3(mat.baseColor[0], mat.baseColor[1], mat.baseColor[2]);
        if (!ob.mesh.uvs.empty()) {
            if (const Texture* T = w.texture_of(matID)) {
                float u, v, c[4];
                hit_uv(ob.mesh, h.prim, h.alpha, h.beta, &u, &v);
                T->sample(u, v, false, c);
                kd = v3(c[0], c[1], c[2]);
            }
        }
        const V3 point = at(o, d, h.t);
        const V3 woWorld = neg(d);
        const float* nn = &ob.mesh.normals[9 * (size_t)h.prim];
        const V3 n0 = normalized(v3(nn[0], nn[1], nn[2])), n1 = normalized(v3(nn[3], nn[4], nn[5])), n2 = normalized(v3(nn[6], nn[7], nn[8]));
        const float alpha = h.alpha, beta = h.beta, gamma = 1.0f - alpha - beta;
        V3 normal = v3(fmaf(beta, n2.x, fmaf(alpha, n1.x, gamma * n0.x)), fmaf(beta, n2.y, fmaf(alpha, n1.y, gamma * n0.y)),
                       fmaf(beta, n2.z, fmaf(alpha, n1.z, gamma * n0.z)));
        normal = normalized(normal);
        if (dot(normal, woWorld) < 0.0f) normal = neg(normal);
        // the seed ignores the bounce, as the reference's BSDF sampling does; the third draw chooses the lobe
        uint32_t seed = tea4((uint32_t)path.pixelIndex, (uint32_t)w.sample);
        const float xi1 = rnd(seed), xi2 = rnd(seed), xi3 = rnd(seed);
        const float rr = rough && matID < (int)rough->size() ? (*rough)[matID] : 0.0f;
        shade_plastic(w, r, i, path, point, normal, woWorld, kd, rr, xi1, xi2, xi3);
    }
}

// cond_render_sample with plas_shade in place of cond_shade
void plas_render_sample(World& w, int sample, std::vector<std::vector<float>>* aov, const std::vector<float>* rough) {
    begin_sample(w, sample);
    for (Rank& r : w.ranks) path_gen(w, r);
    for (int bounce = 0; bounce <= w.cfg.bounces; bounce++) {
        if (bounce > 0 && w.cfg.proxyMode) for (Rank& r : w.ranks) { reset_nn(w, r); secondary_module(w, r); }
        for (;;) {
            for (Rank& r : w.ranks) { traverse(w, r); partition(w, r); }
            if (exchange(w)) break;
        }
        for (Rank& r : w.ranks) {
            if (bounce == 0 && aov) add_first_hits(w, r, (*aov)[r.id].data());
            plas_shade(w, r, rough); reset_nn(w, r); shadow_module(w, r);
        }
    }
}

}  // namespace

extern "C" {

int plas_render_sample(void* wp, int sample) {
    World* w = (World*)wp;
    if (!w) return -1;
    auto a = g_aov.find(wp);
    auto r = g_rough.find(wp);
    plas_render_sample(*w, sample, a == g_aov.end() ? nullptr : &a->second, r == g_rough.end() ? nullptr : &r->second);
    return 0;
}

// Renderer::launch: the frame's buffers (colour and guide) cleared, spp samples
int plas_launch(void* wp) {
    World* w = (World*)wp;
    if (!w) return -1;
    orc_reset_frame(wp);
    auto it = g_aov.find(wp);
    if (it != g_aov.end()) for (auto& b : it->second) std::fill(b.begin(), b.end(), 0.f);
    for (int s = 0; s < w->cfg.spp; s++) plas_render_sample(wp, s);
    return 0;
}

// the BSDF on its own, arrays as dprt_spec_plastic_sample / _eval
int plas_sample(const float* kd, const float* r, const float* wo, const float* xi, int64_t n, float* wi, float* weight) {
    for (int64_t i = 0; i < n; i++) {
        const CondOut o = plastic_sample(v3(kd[3 * i], kd[3 * i + 1], kd[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                                         xi[3 * i], xi[3 * i + 1], xi[3 * i + 2]);
        wi[3 * i] = o.wi.x; wi[3 * i + 1] = o.wi.y; wi[3 * i + 2] = o.wi.z;
        weight[3 * i] = o.weight.x; weight[3 * i + 1] = o.weight.y; weight[3 * i + 2] = o.weight.z;
    }
    return 0;
}
int plas_eval(const float* kd, const float* r, const float* wo, const float* wi, int64_t n, float* f) {
    for (int64_t i = 0; i < n; i++) {
        const V3 v = plastic_eval(v3(kd[3 * i], kd[3 * i + 1], kd[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                                  v3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]));
        f[3 * i] = v.x; f[3 * i + 1] = v.y; f[3 * i + 2] = v.z;
    }
    return 0;
}

}  // extern "C"
