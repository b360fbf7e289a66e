// conductor_reference.cpp -- CPU reference of the rough conductor (bsdfType 2, DESIGN.md 3.12), test infrastructure
// (tests/conductor_reference.py compiles it at test time with the oracle's flags).
//
// The oracle (oracle/oracle.cpp) and the AOV reference (tests/aov_reference.cpp) are included unchanged: this translation
// unit exports every orc_* and aov_* entry point and adds the conductor on top of them, as a restatement of its own:
//   cond_render_sample  = aov_render_sample (the oracle's render_sample, guide buffers optional), where every shade is the
//                         oracle's shade() followed by the conductor rule for each record whose hit is a bsdfType 2 material:
//                         its next record and its spc shadow slots are recomputed from the record as it was before shade()
//                         (same re-trace, albedo / texel, face-forwarded normal and random numbers as shade() uses);
//   cond_set_roughness  = dprt_set_material_roughness (per world; materials without an entry have roughness 0);
//   cond_sample / cond_eval = the BSDF on its own, for the host compile of conductor.cuh.
// Same binary32 operations in the same order as the specification, so every record is comparable bit for bit.
#include "aov_reference.cpp"

namespace {

std::map<const void*, std::vector<float>> g_rough;

// Schlick per channel: F0 + (1 - F0) m^5 with m = 1 - clamp(c, 0, 1), m^5 = (m^2 m^2) m
V3 schlick(V3 f0, float c) {
    const float cc = fminf(fmaxf(c, 0.0f), 1.0f);
    const float m = 1.0f - cc, mm = m * m, m5 = (mm * mm) * m;
    V3 f;
    f.x = f0.x + (1.0f - f0.x) * m5;
    f.y = f0.y + (1.0f - f0.y) * m5;
    f.z = f0.z + (1.0f - f0.z) * m5;
    return f;
}
float ggx_alpha(float r) { return fmaxf(r * r, 1e-3f); }
// sqrt(w.z^2 + alpha^2 (w.x^2 + w.y^2)) = w.z (1 + 2 Lambda(w))
float smith_a(float a2, V3 w) {
    const float xy = w.x * w.x + w.y * w.y;
    return sqrtf(w.z * w.z + a2 * xy);
}
struct CondOut { V3 wi, weight; bool valid; };
CondOut conductor_sample(V3 f0, float r, V3 wo, float u1, float u2) {
    CondOut o{v3(0, 0, 0), v3(0, 0, 0), false};
    if (r == 0.0f) {                                   // mirror
        o.wi = v3(-wo.x, -wo.y, wo.z); o.weight = schlick(f0, wo.z); o.valid = true;
        return o;
    }
    if (!(wo.z > 0.0f)) return o;
    const float al = ggx_alpha(r);
    const V3 V = normalized(v3(al * wo.x, al * wo.y, wo.z));           // Heitz 2018 visible normals
    const float l2 = V.x * V.x + V.y * V.y;
    V3 T1 = v3(1.0f, 0.0f, 0.0f);
    if (l2 > 0.0f) { const float k = 1.0f / sqrtf(l2); T1 = v3(-V.y * k, V.x * k, 0.0f); }
    const V3 T2 = cross(V, T1);
    const float rad = sqrtf(u1);
    float sphi, cphi; det_sincos2pi(u2, &sphi, &cphi);
    const float t1 = rad * cphi;
    const float s = 0.5f * (1.0f + V.z);
    const float rest = 1.0f - t1 * t1;
    const float t2 = (1.0f - s) * sqrtf(fmaxf(0.0f, rest)) + s * (rad * sphi);
    const float tz = sqrtf(fmaxf(0.0f, rest - t2 * t2));
    V3 N;
    N.x = t1 * T1.x + t2 * T2.x + tz * V.x;
    N.y = t1 * T1.y + t2 * T2.y + tz * V.y;
    N.z = t1 * T1.z + t2 * T2.z + tz * V.z;
    const V3 m = normalized(v3(al * N.x, al * N.y, fmaxf(0.0f, N.z)));
    const float om = dot(wo, m);
    const V3 wi = sub(scale(m, 2.0f * om), wo);
    if (!(wi.z > 0.0f)) return o;
    const float a2 = al * al, Ao = smith_a(a2, wo), Ai = smith_a(a2, wi);
    const float g2g1 = fminf(1.0f, (wo.z + Ao) / (Ao + Ai * (wo.z / wi.z)));
    o.wi = wi; o.weight = scale(schlick(f0, om), g2g1); o.valid = true;
    return o;
}
V3 conductor_eval(V3 f0, float r, V3 wo, V3 wi) {
    if (r == 0.0f || !(wo.z > 0.0f) || !(wi.z > 0.0f)) return v3(0, 0, 0);
    const float al = ggx_alpha(r), a2 = al * al;
    const V3 m = normalized(v3(wo.x + wi.x, wo.y + wi.y, wo.z + wi.z));
    const float q = (m.x * m.x + m.y * m.y) + a2 * (m.z * m.z);
    const float D = a2 / (3.14159265358979323846f * (q * q));
    const float den = 2.0f * (wi.z * smith_a(a2, wo) + wo.z * smith_a(a2, wi));
    if (!(den > 1e-30f)) return v3(0, 0, 0);
    return scale(schlick(f0, dot(wi, m)), D / den);
}

// the closest-hit program's tail for a conductor: the next path from conductor_sample, the spc light samples with
// conductor_eval in place of albedo / pi; the light choice and point are shade()'s Lambertian ones
void shade_conductor(World& w, Rank& r, int i, const dprt_path_record& path, V3 point, V3 normal, V3 woWorld, V3 f0, float rough,
                     float xi1, float xi2) {
    const int n = r.pathSize, spc = w.cfg.shadowPathCount;
    const Frame fr = make_frame(normal);
    const V3 wo = to_local(fr, woWorld);
    const V3 thr = v3(path.throughput[0], path.throughput[1], path.throughput[2]);
    const CondOut cs = conductor_sample(f0, rough, wo, xi1, xi2);
    dprt_path_record next{};
    if (cs.valid) {
        const V3 nd = normalized(to_world(fr, cs.wi));
        const V3 t = mul(thr, cs.weight);
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
        if (rough == 0.0f) continue;                  // the mirror is a delta lobe: no light samples
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
        const V3 f = conductor_eval(f0, rough, wo, to_local(fr, wi));
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

// shade() of oracle.cpp, then the conductor rule for every record whose closest hit on this rank is a bsdfType 2 material
void cond_shade(World& w, Rank& r, const std::vector<float>* rough) {
    const int n = r.pathSize;
    const std::vector<dprt_path_record> in(r.paths.begin(), r.paths.begin() + n);
    shade(w, r);
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
        if (mat.bsdfType != 2) continue;
        V3 albedo = v3(mat.baseColor[0], mat.baseColor[1], mat.baseColor[2]);
        if (!ob.mesh.uvs.empty()) {
            if (const Texture* T = w.texture_of(matID)) {
                float u, v, c[4];
                hit_uv(ob.mesh, h.prim, h.alpha, h.beta, &u, &v);
                T->sample(u, v, false, c);
                albedo = v3(c[0], c[1], c[2]);
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
        uint32_t seed = tea4((uint32_t)path.pixelIndex, (uint32_t)w.sample);
        const float xi1 = rnd(seed), xi2 = rnd(seed);
        const float rr = rough && matID < (int)rough->size() ? (*rough)[matID] : 0.0f;
        shade_conductor(w, r, i, path, point, normal, woWorld, albedo, rr, xi1, xi2);
    }
}

// aov_render_sample of aov_reference.cpp with cond_shade in place of shade
void cond_render_sample(World& w, int sample, std::vector<std::vector<float>>* aov, const std::vector<float>* rough) {
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
            cond_shade(w, r, rough); reset_nn(w, r); shadow_module(w, r);
        }
    }
}

}  // namespace

extern "C" {

// dprt_set_material_roughness: n in [1, DPRT_MAX_MATERIALS], every entry in [0, 1]; replaces entries [0, n)
int cond_set_roughness(void* wp, const float* roughness, int n) {
    if (!wp || !roughness || n < 1 || n > DPRT_MAX_MATERIALS) return -1;
    for (int i = 0; i < n; i++) if (!(roughness[i] >= 0.0f && roughness[i] <= 1.0f)) return -1;
    std::vector<float>& t = g_rough[wp];
    if ((int)t.size() < n) t.resize(n, 0.0f);
    std::copy(roughness, roughness + n, t.begin());
    return 0;
}
int cond_forget(void* wp) { g_rough.erase(wp); return 0; }

int cond_render_sample(void* wp, int sample) {
    World* w = (World*)wp;
    if (!w) return -1;
    auto a = g_aov.find(wp);
    auto r = g_rough.find(wp);
    cond_render_sample(*w, sample, a == g_aov.end() ? nullptr : &a->second, r == g_rough.end() ? nullptr : &r->second);
    return 0;
}

// Renderer::launch: the frame's buffers (colour and guide) cleared, spp samples
int cond_launch(void* wp) {
    World* w = (World*)wp;
    if (!w) return -1;
    orc_reset_frame(wp);
    auto it = g_aov.find(wp);
    if (it != g_aov.end()) for (auto& b : it->second) std::fill(b.begin(), b.end(), 0.f);
    for (int s = 0; s < w->cfg.spp; s++) cond_render_sample(wp, s);
    return 0;
}

// the BSDF on its own, arrays as dprt_spec_conductor_sample / _eval
int cond_sample(const float* f0, const float* r, const float* wo, const float* xi, int64_t n, float* wi, float* weight) {
    for (int64_t i = 0; i < n; i++) {
        const CondOut o = conductor_sample(v3(f0[3 * i], f0[3 * i + 1], f0[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                                           xi[2 * i], xi[2 * i + 1]);
        wi[3 * i] = o.wi.x; wi[3 * i + 1] = o.wi.y; wi[3 * i + 2] = o.wi.z;
        weight[3 * i] = o.weight.x; weight[3 * i + 1] = o.weight.y; weight[3 * i + 2] = o.weight.z;
    }
    return 0;
}
int cond_eval(const float* f0, const float* r, const float* wo, const float* wi, int64_t n, float* f) {
    for (int64_t i = 0; i < n; i++) {
        const V3 v = conductor_eval(v3(f0[3 * i], f0[3 * i + 1], f0[3 * i + 2]), r[i], v3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]),
                                    v3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]));
        f[3 * i] = v.x; f[3 * i + 1] = v.y; f[3 * i + 2] = v.z;
    }
    return 0;
}

}  // extern "C"
