// dprt_render.cpp -- the C++ host of the data-parallel path tracer: what Renderer::launch does in the reference
// (src/render/renderer.cpp:1576-2059: one MPI rank per GPU, scene tables, spp x runSample, image average +
// MPI_Reduce, image to disk), written against the C ABI of libdprt.so (include/dprt.h) and nothing else.
//
//   dprt_render --scene scene.dprt --out image.pfm [--spp 4] [--bounces 4] [--proxy 0|1] [--path-gen 0|1]
//               [--world W] [--devices D]   in-process rank group: W chunk owners driven by this thread, owner k on GPU k % D
//               [--nccl-id-file F]     one process per GPU: RANK / WORLD_SIZE / LOCAL_RANK from the environment (the
//                                      launcher of the reference is mpirun; here any launcher that sets them), rank 0
//                                      publishes the NCCL unique id through file F
//
// Scene file (written by pg2024-data-parallel-ray-tracing_b200/scene.py:save_scene; little endian):
//   "DPRTSCN1" | int32 nObjects nMaterials nLights | dprt_camera | dprt_material[nMaterials] | dprt_light_tri[nLights]
//   per object: dprt_object_desc (isProxy ignored) | int64 ntris | float verts[9 ntris] | float normals[9 ntris]
//               | int32 mats[ntris] | int64 visBytes | vis blob | int64 depthBytes | depth blob   (proxy MLP weights, may be 0)
// Real-scene variant (real_scene.py:save_scene_v2; the front end of SURVEY.md 8f row 3 -- textures, cut-outs, environment map):
//   "DPRTSCN2" | int32 nObjects nMaterials nLights nTextures | dprt_camera | dprt_material[nMaterials] | int32 matTex[nMaterials]
//   | dprt_light_tri[nLights] | per texture: int32 slot width height | float rgba[4 w h]   (params.albedoTextures, renderer.cpp:1621-1721)
//   | int32 envWidth envHeight (0 0 = analytic sky) | float rotationOffset | float rgba[4 w h]   (params.envLightTexture, :1851)
//   per object: dprt_object_desc | int64 ntris | int32 hasUv | verts | normals | float uv[6 ntris] if hasUv | mats | vis blob | depth blob
//   (instanced / indexed meshes arrive flattened: the file is written after dprt_flatten_instances)
// Rough conductors and glossy plastics (real_scene.py:save_scene_v2 when the scene has a roughness table; DESIGN.md 3.12, 3.13):
//   "DPRTSCN3" | the DPRTSCN2 layout after its magic | float roughness[nMaterials]   (dprt_set_material_roughness)
//               [--frames F] [--camera-move dx,dy,dz] [--camera-target x,y,z] [--light-move dx,dy,dz] [--light-start dx,dy,dz]
//                                      the frame loop of launch() (renderer.cpp:1938-2059): per frame the first two lights move by
//                                      -light-move (after a one-off +light-start, LIGHT_MOVE :1941-1966) and the camera origin by
//                                      +camera-move (CAMERA_MOVE :1968-1983; re-aimed at --camera-target when given, else translated);
//                                      frame f is written as <f><name> like std::to_string(cframe) + exrFilename (:2055-2058)
//               [--aov 1]              also the first-hit guide buffers a denoiser takes beside the colour (dprt_enable_aov on every
//                                      context, samples in flight included): <name>.albedo.<ext> and <name>.normal.<ext>, e.g.
//                                      --out img.exr writes img.albedo.exr and img.normal.exr (<f>img.albedo.exr per frame f)
//               [--gpu-build 1]        build the own chunks' BVH8s on the GPU (dprt_build_chunk) instead of on the host; the
//                                      image is the same bit for bit
//               [--denoise 1]          also the frame filtered by dprt_denoise (default parameters) with those guide buffers (turned
//                                      on for it as --aov 1 does, but written only with --aov 1): <name>.denoised.<ext>
//   dprt_render --convert in.pfm out.exr     no GPU: re-encode an image (the reference's Image::save writes EXR)
//
// Output on the root rank: OpenEXR (uncompressed scanlines, float32 B/G/R) when the name ends in .exr, else PFM (RGB float32,
// bottom-up as the format demands); one JSON line of statistics per frame on stdout.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "dprt.h"

namespace {

struct Object {
    dprt_object_desc desc;
    int64_t ntris = 0;
    std::vector<float> verts, normals, uvs;          // uvs: 6 per triangle, empty = no texture coordinates
    std::vector<int32_t> mats;
    std::vector<char> vis, depth;
};
struct Texture { int32_t slot = 0, w = 0, h = 0; std::vector<float> rgba; };
struct Scene {
    dprt_camera cam;
    std::vector<dprt_material> materials;
    std::vector<int32_t> matTex;                     // texture slot per material (-1 = none); empty for DPRTSCN1 files
    std::vector<float> roughness;                    // per material (bsdfType 2 and 3); empty unless DPRTSCN3
    std::vector<dprt_light_tri> lights;
    std::vector<Texture> textures;
    Texture env; float envRotation = 0.f;            // env.w == 0: analytic sky
    std::vector<Object> objects;
};

bool read_exact(FILE* f, void* p, size_t n) { return n == 0 || fread(p, 1, n, f) == n; }

bool read_texels(FILE* f, Texture& t) {
    if (t.w < 1 || t.h < 1 || (int64_t)t.w * t.h > (int64_t(1) << 28)) return false;
    t.rgba.resize(4 * (size_t)t.w * t.h);
    return read_exact(f, t.rgba.data(), t.rgba.size() * 4);
}

bool load_scene(const std::string& path, Scene& sc, std::string& err) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) { err = "cannot open " + path; return false; }
    char magic[8]; int32_t hdr[4] = {0, 0, 0, 0};
    bool ok = read_exact(f, magic, 8);
    const bool v3 = ok && std::memcmp(magic, "DPRTSCN3", 8) == 0;
    const bool v2 = ok && (v3 || std::memcmp(magic, "DPRTSCN2", 8) == 0);
    ok = ok && (v2 || std::memcmp(magic, "DPRTSCN1", 8) == 0) && read_exact(f, hdr, v2 ? 16 : 12);
    if (ok) ok = hdr[0] >= 1 && hdr[0] <= 32 && hdr[1] >= 1 && hdr[1] <= DPRT_MAX_MATERIALS && hdr[2] >= 1 && hdr[2] <= DPRT_MAX_LIGHTS &&
                 hdr[3] >= 0 && hdr[3] <= DPRT_MAX_TEXTURES;
    if (ok) {
        sc.materials.resize(hdr[1]); sc.lights.resize(hdr[2]); sc.objects.resize(hdr[0]);
        ok = read_exact(f, &sc.cam, sizeof(sc.cam)) && read_exact(f, sc.materials.data(), sizeof(dprt_material) * hdr[1]);
        if (ok && v2) { sc.matTex.resize(hdr[1]); ok = read_exact(f, sc.matTex.data(), 4 * (size_t)hdr[1]); }
        ok = ok && read_exact(f, sc.lights.data(), sizeof(dprt_light_tri) * hdr[2]);
    }
    if (ok && v2) {
        sc.textures.resize(hdr[3]);
        for (Texture& t : sc.textures) {
            int32_t th[3];
            ok = ok && read_exact(f, th, 12);
            if (!ok) break;
            t.slot = th[0]; t.w = th[1]; t.h = th[2];
            ok = t.slot >= 0 && t.slot < DPRT_MAX_TEXTURES && read_texels(f, t);
        }
        int32_t eh[2] = {0, 0};
        ok = ok && read_exact(f, eh, 8) && read_exact(f, &sc.envRotation, 4);
        if (ok && (eh[0] != 0 || eh[1] != 0)) { sc.env.w = eh[0]; sc.env.h = eh[1]; ok = read_texels(f, sc.env); }
    }
    for (size_t k = 0; ok && k < sc.objects.size(); k++) {
        Object& o = sc.objects[k];
        int32_t hasUv = 0;
        ok = read_exact(f, &o.desc, sizeof(o.desc)) && read_exact(f, &o.ntris, 8) && o.ntris >= 0 && o.ntris < (int64_t(1) << 27);
        if (ok && v2) ok = read_exact(f, &hasUv, 4);
        if (!ok) break;
        o.verts.resize(9 * (size_t)o.ntris); o.normals.resize(9 * (size_t)o.ntris); o.mats.resize((size_t)o.ntris);
        if (hasUv) o.uvs.resize(6 * (size_t)o.ntris);
        int64_t vb = 0, db = 0;
        ok = read_exact(f, o.verts.data(), o.verts.size() * 4) && read_exact(f, o.normals.data(), o.normals.size() * 4) &&
             read_exact(f, o.uvs.data(), o.uvs.size() * 4) &&
             read_exact(f, o.mats.data(), o.mats.size() * 4) && read_exact(f, &vb, 8) && vb >= 0 && vb < (int64_t(1) << 30);
        if (ok) { o.vis.resize((size_t)vb); ok = read_exact(f, o.vis.data(), (size_t)vb) && read_exact(f, &db, 8) && db >= 0 && db < (int64_t(1) << 30); }
        if (ok) { o.depth.resize((size_t)db); ok = read_exact(f, o.depth.data(), (size_t)db); }
    }
    if (ok && v3) { sc.roughness.resize(sc.materials.size()); ok = read_exact(f, sc.roughness.data(), 4 * sc.roughness.size()); }
    fclose(f);
    if (!ok) err = "malformed scene file " + path;
    return ok;
}

bool write_pfm(const std::string& path, const float* rgb, int w, int h) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    fprintf(f, "PF\n%d %d\n-1.0\n", w, h);
    for (int row = h - 1; row >= 0; row--) fwrite(rgb + (size_t)row * w * 3, sizeof(float), (size_t)w * 3, f);
    fclose(f);
    return true;
}

// Minimal OpenEXR 2 writer: single-part scanline file, NO_COMPRESSION, three FLOAT channels (stored alphabetically: B, G, R),
// increasing-Y line order. What Image::save(width, height, pixels, exrFilename) produces in the reference (renderer.cpp:2055-2058).
bool write_exr(const std::string& path, const float* rgb, int w, int h) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    std::vector<char> hd;
    auto put = [&](const void* p, size_t n) { hd.insert(hd.end(), (const char*)p, (const char*)p + n); };
    auto puts0 = [&](const char* s) { put(s, std::strlen(s) + 1); };
    auto i32 = [&](int32_t v) { put(&v, 4); };
    auto f32 = [&](float v) { put(&v, 4); };
    const uint32_t magic = 20000630u, version = 2u;
    put(&magic, 4); put(&version, 4);
    puts0("channels"); puts0("chlist"); i32(3 * (2 + 16) + 1);
    for (const char* c : {"B", "G", "R"}) { puts0(c); i32(2 /* FLOAT */); const char z[4] = {0, 0, 0, 0}; put(z, 4); i32(1); i32(1); }
    { const char z = 0; put(&z, 1); }
    puts0("compression"); puts0("compression"); i32(1); { const char c = 0; put(&c, 1); }
    puts0("dataWindow"); puts0("box2i"); i32(16); i32(0); i32(0); i32(w - 1); i32(h - 1);
    puts0("displayWindow"); puts0("box2i"); i32(16); i32(0); i32(0); i32(w - 1); i32(h - 1);
    puts0("lineOrder"); puts0("lineOrder"); i32(1); { const char c = 0; put(&c, 1); }
    puts0("pixelAspectRatio"); puts0("float"); i32(4); f32(1.0f);
    puts0("screenWindowCenter"); puts0("v2f"); i32(8); f32(0.0f); f32(0.0f);
    puts0("screenWindowWidth"); puts0("float"); i32(4); f32(1.0f);
    { const char z = 0; put(&z, 1); }
    const uint64_t rowBytes = 8 + (uint64_t)w * 12;
    uint64_t off = hd.size() + (uint64_t)h * 8;
    for (int y = 0; y < h; y++) { put(&off, 8); off += rowBytes; }
    bool ok = fwrite(hd.data(), 1, hd.size(), f) == hd.size();
    std::vector<float> row((size_t)w * 3);
    for (int y = 0; y < h && ok; y++) {
        const float* src = rgb + (size_t)y * w * 3;
        for (int x = 0; x < w; x++) { row[x] = src[3 * x + 2]; row[(size_t)w + x] = src[3 * x + 1]; row[2 * (size_t)w + x] = src[3 * x]; }
        const int32_t yy = y, bytes = (int32_t)(w * 12);
        ok = fwrite(&yy, 4, 1, f) == 1 && fwrite(&bytes, 4, 1, f) == 1 && fwrite(row.data(), 4, row.size(), f) == row.size();
    }
    fclose(f);
    return ok;
}

bool read_pfm(const std::string& path, std::vector<float>& rgb, int& w, int& h) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    char tag[3] = {0}; float scale = 0.f;
    bool ok = fscanf(f, "%2s %d %d %f", tag, &w, &h, &scale) == 4 && std::strcmp(tag, "PF") == 0 && w > 0 && h > 0 && scale < 0.f;
    if (ok) { fgetc(f); rgb.resize((size_t)w * h * 3); }
    for (int row = h - 1; ok && row >= 0; row--) ok = fread(rgb.data() + (size_t)row * w * 3, sizeof(float), (size_t)w * 3, f) == (size_t)w * 3;
    fclose(f);
    return ok;
}

bool ends_with(const std::string& s, const char* suf) { const size_t n = std::strlen(suf); return s.size() >= n && s.compare(s.size() - n, n, suf) == 0; }
bool write_image(const std::string& path, const float* rgb, int w, int h) { return ends_with(path, ".exr") ? write_exr(path, rgb, w, h) : write_pfm(path, rgb, w, h); }

// "<stem>.<tag><ext>": the guide buffer `tag` of the image `path` (img.exr -> img.albedo.exr; no extension: img -> img.albedo)
std::string aov_name(const std::string& path, const char* tag) {
    const size_t slash = path.find_last_of('/'), dot = path.find_last_of('.');
    if (dot == std::string::npos || (slash != std::string::npos && dot < slash)) return path + "." + tag;
    return path.substr(0, dot) + "." + tag + path.substr(dot);
}

// "<dir>/<frame><name>" like std::to_string(cframe) + exrFilename (renderer.cpp:2058)
std::string frame_name(const std::string& path, int frame, int frames) {
    if (frames <= 1) return path;
    const size_t slash = path.find_last_of('/');
    const std::string dir = slash == std::string::npos ? "" : path.substr(0, slash + 1);
    return dir + std::to_string(frame) + (slash == std::string::npos ? path : path.substr(slash + 1));
}

bool parse3(const char* s, float v[3]) { return s && std::sscanf(s, "%f,%f,%f", v, v + 1, v + 2) == 3; }

// camera.m_origin += move; camera.updateTransformMatrix() (renderer.cpp:1968-1983). With a target the basis is re-aimed (the
// lengths of U and V carry the field of view and the aspect ratio); without one the camera is translated.
void move_camera(dprt_camera& c, const float move[3], const float* target) {
    for (int a = 0; a < 3; a++) c.origin[a] = c.origin[a] + move[a];
    if (!target) return;
    auto len = [](const double* v) { return std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); };
    const double U0[3] = {c.U[0], c.U[1], c.U[2]}, V0[3] = {c.V[0], c.V[1], c.V[2]};
    const double lu = len(U0), lv = len(V0);
    double w[3] = {(double)target[0] - c.origin[0], (double)target[1] - c.origin[1], (double)target[2] - c.origin[2]};
    const double lw = len(w); for (double& x : w) x /= lw;
    const double up[3] = {c.V[0] / lv, c.V[1] / lv, c.V[2] / lv};
    double u[3] = {w[1] * up[2] - w[2] * up[1], w[2] * up[0] - w[0] * up[2], w[0] * up[1] - w[1] * up[0]};
    const double lu2 = len(u); for (double& x : u) x /= lu2;
    const double v[3] = {u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0]};
    for (int a = 0; a < 3; a++) { c.U[a] = (float)(u[a] * lu); c.V[a] = (float)(v[a] * lv); c.W[a] = (float)w[a]; }
}

// the AccelerationStructure table of one rank (renderer.cpp:1812-1842): own objects as geometry, the others as proxies.
// gpuBuild: own objects' BVH8s are built on the GPU (dprt_build_chunk) instead of on the host
int upload_scene(dprt_ctx* ctx, const Scene& sc, int rank, bool gpuBuild) {
    int r;
    for (size_t k = 0; k < sc.objects.size(); k++) {
        const Object& o = sc.objects[k];
        dprt_object_desc d = o.desc;
        if (o.desc.nodeID == rank) {
            d.isProxy = 0;
            const float* uv = o.uvs.empty() ? nullptr : o.uvs.data();
            if ((r = gpuBuild ? dprt_build_chunk(ctx, (int)k, &d, o.verts.data(), o.normals.data(), uv, o.mats.data(), o.ntris)
                              : dprt_upload_chunk_uv(ctx, (int)k, &d, o.verts.data(), o.normals.data(), uv, o.mats.data(), o.ntris))) return r;
        } else {
            d.isProxy = 1;
            if ((r = dprt_upload_proxy(ctx, (int)k, &d, o.vis.empty() ? nullptr : o.vis.data(), o.vis.size(),
                                       o.depth.empty() ? nullptr : o.depth.data(), o.depth.size()))) return r;
        }
    }
    if ((r = dprt_set_materials(ctx, sc.materials.data(), (int)sc.materials.size()))) return r;
    // albedo / opacity maps, texture slot per material, environment map (renderer.cpp:1621-1721, :1851)
    for (const Texture& t : sc.textures) if ((r = dprt_set_texture(ctx, t.slot, t.rgba.data(), t.w, t.h))) return r;
    if (!sc.matTex.empty() && (r = dprt_set_material_textures(ctx, sc.matTex.data(), (int)sc.matTex.size()))) return r;
    if (!sc.roughness.empty() && (r = dprt_set_material_roughness(ctx, sc.roughness.data(), (int)sc.roughness.size()))) return r;
    if (sc.env.w > 0 && (r = dprt_set_env_map(ctx, sc.env.rgba.data(), sc.env.w, sc.env.h, sc.envRotation))) return r;
    if ((r = dprt_set_lights(ctx, sc.lights.data(), (int)sc.lights.size()))) return r;
    return dprt_set_camera(ctx, &sc.cam);
}

int die(const char* what, dprt_ctx* ctx, int rc) {
    fprintf(stderr, "dprt_render: %s failed (%d): %s\n", what, rc, dprt_last_error(ctx));
    return 1;
}

// Samples in flight (dprt.h): `extra` contexts adopt `ctx`'s scene; context j renders samples j, j + K, ... from its own thread,
// then everything is accumulated into `ctx`. K = 1: the plain sample loop of Renderer::launch (renderer.cpp:1993-2022).
int render_samples(dprt_ctx* ctx, std::vector<dprt_ctx*>& extra, int spp, const char** what, dprt_ctx** failed) {
    const int K = 1 + (int)extra.size();
    std::vector<dprt_ctx*> all{ctx};
    all.insert(all.end(), extra.begin(), extra.end());
    std::vector<int> rc(K, 0);
    auto work = [&](int j) {
        for (int s = j; s < spp && !rc[j]; s += K) rc[j] = dprt_render_sample(all[j], s);
    };
    std::vector<std::thread> th;
    for (int j = 1; j < K; j++) th.emplace_back(work, j);
    work(0);
    for (auto& t : th) t.join();
    for (int j = 0; j < K; j++) if (rc[j]) { *what = "dprt_render_sample"; *failed = all[j]; return rc[j]; }
    for (int j = 1; j < K; j++) {
        const int r = dprt_accumulate_from(ctx, all[j]);
        if (r) { *what = "dprt_accumulate_from"; *failed = ctx; return r; }
    }
    return 0;
}

const char* arg(int argc, char** argv, const char* name, const char* dflt) {
    for (int i = 1; i + 1 < argc; i++) if (!std::strcmp(argv[i], name)) return argv[i + 1];
    return dflt;
}

}  // namespace

int main(int argc, char** argv) {
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);       // before the first CUDA call: one hardware queue per stream (--inflight)
    if (argc == 4 && !std::strcmp(argv[1], "--convert")) {            // no GPU involved
        std::vector<float> rgb; int w = 0, h = 0;
        if (!read_pfm(argv[2], rgb, w, h)) { fprintf(stderr, "dprt_render: cannot read PFM %s\n", argv[2]); return 1; }
        if (!write_image(argv[3], rgb.data(), w, h)) { fprintf(stderr, "dprt_render: cannot write %s\n", argv[3]); return 1; }
        return 0;
    }
    const std::string scenePath = arg(argc, argv, "--scene", ""), outPath = arg(argc, argv, "--out", "");
    if (scenePath.empty()) {
        fprintf(stderr, "usage: dprt_render --scene S.dprt [--out image.pfm] [--spp n] [--bounces n] [--proxy 0|1] [--path-gen 0|1] "
                        "[--inflight K] [--world W | --nccl-id-file F] [--frames F] [--camera-move x,y,z] [--camera-target x,y,z] "
                        "[--light-move x,y,z] [--light-start x,y,z] [--aov 0|1] [--denoise 0|1] [--gpu-build 0|1]\n       dprt_render --convert in.pfm out.exr\n");
        return 2;
    }
    Scene sc; std::string err;
    if (!load_scene(scenePath, sc, err)) { fprintf(stderr, "dprt_render: %s\n", err.c_str()); return 1; }
    const char* idFile = arg(argc, argv, "--nccl-id-file", nullptr);
    int world = std::atoi(arg(argc, argv, "--world", "0"));
    int rank = 0, local = 0;
    if (idFile) {
        rank = std::atoi(getenv("RANK") ? getenv("RANK") : "0");
        world = std::atoi(getenv("WORLD_SIZE") ? getenv("WORLD_SIZE") : "1");
        local = std::atoi(getenv("LOCAL_RANK") ? getenv("LOCAL_RANK") : "0");
    }
    int owners = 0;
    for (const Object& o : sc.objects) owners = o.desc.nodeID + 1 > owners ? o.desc.nodeID + 1 : owners;
    if (world <= 0) world = owners;
    if (world != owners) { fprintf(stderr, "dprt_render: scene has %d chunk owners, world is %d\n", owners, world); return 1; }

    dprt_config cfg; std::memset(&cfg, 0, sizeof(cfg));
    cfg.width = sc.cam.width; cfg.height = sc.cam.height;
    cfg.spp = std::atoi(arg(argc, argv, "--spp", "1"));
    cfg.bounces = std::atoi(arg(argc, argv, "--bounces", "4"));
    cfg.shadowPathCount = DPRT_DEFAULT_SHADOW_PATH_COUNT; cfg.maxCount = DPRT_DEFAULT_MAX_COUNT;   // renderer.cpp:1602-1603
    cfg.sceneSize = (int)sc.objects.size();
    cfg.proxyMode = std::atoi(arg(argc, argv, "--proxy", "0"));
    cfg.pathGenMode = std::atoi(arg(argc, argv, "--path-gen", world > 1 ? "1" : "0"));
    cfg.mlpDtype = std::atoi(arg(argc, argv, "--mlp-dtype", "1"));
    cfg.envColor[0] = 0.6f; cfg.envColor[1] = 0.7f; cfg.envColor[2] = 0.9f;
    const size_t N = (size_t)cfg.width * cfg.height;
    std::vector<float> image(3 * N);
    const bool gpuBuild = std::atoi(arg(argc, argv, "--gpu-build", "0")) != 0;
    const bool aov = std::atoi(arg(argc, argv, "--aov", "0")) != 0;
    const bool denoise = std::atoi(arg(argc, argv, "--denoise", "0")) != 0;
    const bool guides = aov || denoise;                                 // the denoiser filters with the guide buffers
    std::vector<float> albedo(guides ? 3 * N : 0), normal(guides ? 3 * N : 0), denoised(denoise ? 3 * N : 0);
    std::vector<dprt_ctx*> ctxs, extra;
    int inflight = std::atoi(arg(argc, argv, "--inflight", "1"));      // samples in flight per rank
    if (inflight < 1) inflight = 1;
    if (inflight > cfg.spp) inflight = cfg.spp;
    int r;
    // frame loop of launch() (renderer.cpp:1938-2059)
    const int frames = std::max(1, std::atoi(arg(argc, argv, "--frames", "1")));
    float camMove[3] = {0, 0, 0}, camTarget[3], lightMove[3] = {0, 0, 0}, lightStart[3] = {0, 0, 0};
    const bool haveCamMove = parse3(arg(argc, argv, "--camera-move", nullptr), camMove);
    const bool haveTarget = parse3(arg(argc, argv, "--camera-target", nullptr), camTarget);
    const bool haveLightMove = parse3(arg(argc, argv, "--light-move", nullptr), lightMove);
    parse3(arg(argc, argv, "--light-start", nullptr), lightStart);
    // per frame: LIGHT_MOVE (:1941-1966) then CAMERA_MOVE (:1968-1983), uploaded to every context of this process
    auto advance_frame = [&](int frame, const std::vector<dprt_ctx*>& all) -> int {
        if (haveLightMove) {
            const size_t nl = std::min<size_t>(2, sc.lights.size());
            for (size_t i = 0; i < nl; i++) {
                dprt_light_tri& L = sc.lights[i];
                for (int a = 0; a < 3; a++) {
                    if (frame == 0) { L.p0[a] = L.p0[a] + lightStart[a]; L.p1[a] = L.p1[a] + lightStart[a]; L.p2[a] = L.p2[a] + lightStart[a]; }
                    L.p0[a] = L.p0[a] - lightMove[a]; L.p1[a] = L.p1[a] - lightMove[a]; L.p2[a] = L.p2[a] - lightMove[a];
                }
            }
        }
        if (haveCamMove) move_camera(sc.cam, camMove, haveTarget ? camTarget : nullptr);
        for (dprt_ctx* c : all) {
            int rr;
            if (haveLightMove && (rr = dprt_set_lights(c, sc.lights.data(), (int)sc.lights.size()))) return rr;
            if (haveCamMove && (rr = dprt_set_camera(c, &sc.cam))) return rr;
        }
        return 0;
    };
    auto save_frame = [&](int frame) -> bool {
        if (rank != 0 || outPath.empty()) return true;
        const std::string name = frame_name(outPath, frame, frames);
        bool ok = write_image(name, image.data(), cfg.width, cfg.height);
        if (ok && aov) {
            ok = write_image(frame_name(aov_name(outPath, "albedo"), frame, frames), albedo.data(), cfg.width, cfg.height) &&
                 write_image(frame_name(aov_name(outPath, "normal"), frame, frames), normal.data(), cfg.width, cfg.height);
        }
        if (ok && denoise) ok = write_image(frame_name(aov_name(outPath, "denoised"), frame, frames), denoised.data(), cfg.width, cfg.height);
        if (!ok) fprintf(stderr, "dprt_render: cannot write %s, its guide buffers or its denoised image\n", name.c_str());
        return ok;
    };
    auto enable_aov = [&](const std::vector<dprt_ctx*>& all) -> int {
        int rr = 0;
        for (dprt_ctx* c : all) if (guides && (rr = dprt_enable_aov(c, 1))) return rr;
        return 0;
    };
    // K - 1 more contexts of this rank on the same communicator, sharing the uploaded scene (collective across ranks)
    auto make_inflight = [&](dprt_ctx* ctx) -> int {
        if (world > 1 && !dprt_p2p_enabled(ctx)) return 0;          // the NCCL fallback exchange needs the communicator to itself
        for (int j = 1; j < inflight; j++) {
            dprt_ctx* c = nullptr;
            int rr = dprt_create_shared(&cfg, ctx, &c);
            if (rr) return rr;
            extra.push_back(c);
            if ((rr = dprt_adopt_scene(c, ctx))) return rr;
            if ((rr = dprt_reset_frame(c))) return rr;
        }
        return 0;
    };

    if (idFile && world > 1) {
        // ---- one process per GPU (the reference's deployment) ----
        char id[128];
        if (rank == 0) {
            if ((r = dprt_get_unique_id(id))) return die("dprt_get_unique_id", nullptr, r);
            const std::string tmp = std::string(idFile) + ".tmp";
            FILE* f = fopen(tmp.c_str(), "wb");
            if (!f || fwrite(id, 1, 128, f) != 128) { fprintf(stderr, "dprt_render: cannot write %s\n", tmp.c_str()); return 1; }
            fclose(f);
            std::rename(tmp.c_str(), idFile);
        } else {
            bool got = false;
            for (int tries = 0; tries < 6000 && !got; tries++) {
                FILE* f = fopen(idFile, "rb");
                if (f) { got = fread(id, 1, 128, f) == 128; fclose(f); }
                if (!got) std::this_thread::sleep_for(std::chrono::milliseconds(10));
            }
            if (!got) { fprintf(stderr, "dprt_render: rank %d never saw %s\n", rank, idFile); return 1; }
        }
        dprt_ctx* ctx = nullptr;
        if ((r = dprt_create(&cfg, rank, world, local, id, &ctx))) return die("dprt_create", nullptr, r);
        ctxs.push_back(ctx);
        if ((r = upload_scene(ctx, sc, rank, gpuBuild))) return die("scene upload", ctx, r);
        if ((r = make_inflight(ctx))) return die("samples in flight", nullptr, r);
        std::vector<dprt_ctx*> all{ctx};
        all.insert(all.end(), extra.begin(), extra.end());
        if ((r = enable_aov(all))) return die("dprt_enable_aov", ctx, r);
        for (int frame = 0; frame < frames; frame++) {
            if ((r = advance_frame(frame, all))) return die("frame setup", ctx, r);
            const auto t0 = std::chrono::steady_clock::now();
            for (dprt_ctx* c : all) if ((r = dprt_reset_frame(c))) return die("dprt_reset_frame", c, r);
            { const char* what = ""; dprt_ctx* bad = ctx; if ((r = render_samples(ctx, extra, cfg.spp, &what, &bad))) return die(what, bad, r); }
            if ((r = dprt_reduce_image(ctx, 0, rank == 0 ? image.data() : nullptr))) return die("dprt_reduce_image", ctx, r);
            if (guides && (r = dprt_reduce_aov(ctx, 0, rank == 0 ? albedo.data() : nullptr, rank == 0 ? normal.data() : nullptr)))
                return die("dprt_reduce_aov", ctx, r);
            if (denoise && rank == 0 && (r = dprt_denoise(ctx, nullptr, cfg.width, cfg.height, image.data(), albedo.data(), normal.data(), denoised.data())))
                return die("dprt_denoise", ctx, r);
            const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            dprt_stats st; dprt_get_stats(ctx, &st);
            printf("{\"frame\": %d, \"rank\": %d, \"world\": %d, \"seconds\": %.6f, \"rays_walked\": %lld, \"paths_sent_offrank\": %lld, \"exchange_iters\": %lld}\n",
                   frame, rank, world, sec, (long long)st.rays_walked, (long long)st.paths_sent_offrank, (long long)st.exchange_iters);
            if (!save_frame(frame)) return 1;
        }
    } else {
        // ---- in-process rank group (or a single rank) ----
        int ndev = std::atoi(arg(argc, argv, "--devices", "1"));      // chunk owner k runs on GPU k % ndev
        if (ndev < 1) ndev = 1;
        ctxs.resize(world, nullptr);
        for (int k = 0; k < world; k++) {
            if ((r = dprt_create(&cfg, k, world, k % ndev, nullptr, &ctxs[k]))) return die("dprt_create", nullptr, r);
            if ((r = upload_scene(ctxs[k], sc, k, gpuBuild))) return die("scene upload", ctxs[k], r);
        }
        if (world == 1 && (r = make_inflight(ctxs[0]))) return die("samples in flight", nullptr, r);
        std::vector<dprt_ctx*> all(ctxs);
        all.insert(all.end(), extra.begin(), extra.end());
        if ((r = enable_aov(all))) return die("dprt_enable_aov", ctxs[0], r);
        for (int frame = 0; frame < frames; frame++) {
            if ((r = advance_frame(frame, all))) return die("frame setup", ctxs[0], r);
            const auto t0 = std::chrono::steady_clock::now();
            for (dprt_ctx* c : all) if ((r = dprt_reset_frame(c))) return die("dprt_reset_frame", c, r);
            if (world == 1) {
                const char* what = ""; dprt_ctx* bad = ctxs[0];
                if ((r = render_samples(ctxs[0], extra, cfg.spp, &what, &bad))) return die(what, bad, r);
            } else {
                for (int s = 0; s < cfg.spp; s++)
                    if ((r = dprt_render_sample_group(ctxs.data(), world, s))) return die("dprt_render_sample_group", ctxs[0], r);
            }
            r = world == 1 ? dprt_reduce_image(ctxs[0], 0, image.data()) : dprt_reduce_image_group(ctxs.data(), world, 0, image.data());
            if (r) return die("dprt_reduce_image", ctxs[0], r);
            if (guides) {
                r = world == 1 ? dprt_reduce_aov(ctxs[0], 0, albedo.data(), normal.data())
                               : dprt_reduce_aov_group(ctxs.data(), world, 0, albedo.data(), normal.data());
                if (r) return die("dprt_reduce_aov", ctxs[0], r);
            }
            if (denoise && (r = dprt_denoise(ctxs[0], nullptr, cfg.width, cfg.height, image.data(), albedo.data(), normal.data(), denoised.data())))
                return die("dprt_denoise", ctxs[0], r);
            const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            long long walked = 0, sent = 0;
            for (int k = 0; k < world; k++) { dprt_stats st; dprt_get_stats(ctxs[k], &st); walked += st.rays_walked; sent += st.paths_sent_offrank; }
            printf("{\"frame\": %d, \"rank\": 0, \"world\": %d, \"seconds\": %.6f, \"rays_walked\": %lld, \"paths_sent_offrank\": %lld}\n", frame, world, sec, walked, sent);
            if (!save_frame(frame)) return 1;
        }
    }
    for (dprt_ctx* c : extra) dprt_destroy(c);         // borrowers before the owner of the scene and the communicator
    for (dprt_ctx* c : ctxs) dprt_destroy(c);
    return 0;
}
