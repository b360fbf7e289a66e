// aov_reference.cpp -- CPU reference of the first-hit guide buffers (AOVs), test infrastructure (tests/aov_reference.py
// compiles it at test time with the oracle's flags and loads it in place of oracle/liboracle.so).
//
// The oracle (oracle/oracle.cpp) is included unchanged: this translation unit exports every orc_* entry point of
// liboracle.so and adds the AOV rule of DESIGN.md 3.7 on top of it, as a restatement of its own:
//   aov_render_sample   = the oracle's render_sample, with the camera paths' first hits added to the guide buffers
//                         just before the first shade of the sample on every rank;
//   the first hit       = the record's closest hit on the rank that shades it, re-traced exactly as shade() does;
//   albedo              = material baseColor, or the albedo-map texel of a textured material (water too);
//   normal              = interpolated, normalised, face-forwarded shading normal (the one the BSDF is sampled with);
//   a miss adds nothing; frame result = per rank sum / spp, summed over ranks in rank order from +0.
// Same binary32 operations in the same order as shade(), so the per-rank buffers are comparable bit for bit.
#include <map>

#include "../oracle/oracle.cpp"

namespace {

// per world: W buffers of 6N floats (albedo sums 3N, then normal sums 3N); no entry = AOVs off
std::map<const void*, std::vector<std::vector<float>>> g_aov;

void add_first_hits(World& w, Rank& r, float* aov) {
    const int n = r.pathSize;
#pragma omp parallel for schedule(dynamic, 256)
    for (int i = 0; i < n; i++) {                   // at most one record per pixel: no two iterations touch one pixel
        const dprt_path_record& path = r.paths[i];
        if (!path.isValid) continue;
        const V3 o = v3(path.origin[0], path.origin[1], path.origin[2]), d = v3(path.direction[0], path.direction[1], path.direction[2]);
        Hit h{}; int hobj = -1; float tMax = FLT_MAX;
        if (!trace_local(w, r.id, o, d, DPRT_EPSILON, tMax, 0u, false, h, hobj)) continue;
        const Object& ob = w.objects[hobj];
        const dprt_material mat = w.materials[ob.mesh.mats[h.prim]];
        V3 albedo = v3(mat.baseColor[0], mat.baseColor[1], mat.baseColor[2]);
        if (!ob.mesh.uvs.empty()) {
            if (const Texture* T = w.texture_of(ob.mesh.mats[h.prim])) {
                float u, v, c[4];
                hit_uv(ob.mesh, h.prim, h.alpha, h.beta, &u, &v);
                T->sample(u, v, false, c);
                albedo = v3(c[0], c[1], c[2]);
            }
        }
        const float* nn = &ob.mesh.normals[9 * (size_t)h.prim];
        const V3 n0 = normalized(v3(nn[0], nn[1], nn[2])), n1 = normalized(v3(nn[3], nn[4], nn[5])), n2 = normalized(v3(nn[6], nn[7], nn[8]));
        const float alpha = h.alpha, beta = h.beta, gamma = 1.0f - alpha - beta;
        V3 normal = v3(fmaf(beta, n2.x, fmaf(alpha, n1.x, gamma * n0.x)), fmaf(beta, n2.y, fmaf(alpha, n1.y, gamma * n0.y)),
                       fmaf(beta, n2.z, fmaf(alpha, n1.z, gamma * n0.z)));
        normal = normalized(normal);
        if (dot(normal, neg(d)) < 0.0f) normal = neg(normal);
        float* a = aov + 3 * (size_t)path.pixelIndex;
        float* nr = a + 3 * (size_t)w.N;
        a[0] += albedo.x; a[1] += albedo.y; a[2] += albedo.z;
        nr[0] += normal.x; nr[1] += normal.y; nr[2] += normal.z;
    }
}

// render_sample of oracle.cpp, plus the guide buffers at the first shade
void aov_render_sample(World& w, int sample, std::vector<std::vector<float>>* aov) {
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
            shade(w, r); reset_nn(w, r); shadow_module(w, r);
        }
    }
}

}  // namespace

extern "C" {

int aov_enable(void* wp, int enable) {
    World* w = (World*)wp;
    if (!w) return -1;
    if (enable) g_aov[wp].assign(w->W, std::vector<float>(6 * (size_t)w->N, 0.f));
    else g_aov.erase(wp);
    return 0;
}
int aov_forget(void* wp) { g_aov.erase(wp); return 0; }

int aov_render_sample(void* wp, int sample) {
    World* w = (World*)wp;
    if (!w) return -1;
    auto it = g_aov.find(wp);
    aov_render_sample(*w, sample, it == g_aov.end() ? nullptr : &it->second);
    return 0;
}

// Renderer::launch: the frame's buffers (colour and guide) cleared, spp samples
int aov_launch(void* wp) {
    World* w = (World*)wp;
    if (!w) return -1;
    orc_reset_frame(wp);
    auto it = g_aov.find(wp);
    if (it != g_aov.end()) for (auto& b : it->second) std::fill(b.begin(), b.end(), 0.f);
    for (int s = 0; s < w->cfg.spp; s++) aov_render_sample(wp, s);
    return 0;
}

// rank's 6N sums (the layout of DPRT_BUF_AOV)
int aov_buffer(void* wp, int rank, float* out) {
    auto it = g_aov.find(wp);
    World* w = (World*)wp;
    if (it == g_aov.end() || rank < 0 || rank >= w->W) return -1;
    std::memcpy(out, it->second[rank].data(), it->second[rank].size() * sizeof(float));
    return 0;
}

// frame result: sum / spp per rank, summed over ranks in rank order (albedo and normal, 3N floats each)
int aov_reduce(void* wp, float* albedo, float* normal) {
    auto it = g_aov.find(wp);
    if (it == g_aov.end()) return -1;
    World* w = (World*)wp;
    const size_t n3 = (size_t)w->N * 3;
    std::fill(albedo, albedo + n3, 0.f); std::fill(normal, normal + n3, 0.f);
    for (const std::vector<float>& b : it->second)
        for (size_t i = 0; i < n3; i++) {
            albedo[i] += b[i] / (float)w->cfg.spp;
            normal[i] += b[n3 + i] / (float)w->cfg.spp;
        }
    return 0;
}

}  // extern "C"
